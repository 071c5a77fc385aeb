// Shared helpers for libstegan_b200 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/stegan_b200.h"

namespace stg {

void set_cuda_error(cudaError_t e, const char* where);

#define STG_CUDA_CHECK(expr)                                   \
  do {                                                         \
    cudaError_t _e = (expr);                                   \
    if (_e != cudaSuccess) {                                   \
      ::stg::set_cuda_error(_e, #expr);                        \
      return STG_ECUDA;                                        \
    }                                                          \
  } while (0)

extern unsigned long long g_launch_count;  // kernels launched by this library (process-wide)
extern double g_ingest_bytes;              // debug accounting: shared-memory ingest (TMA loads) planned by the tcgen05 launches since the last reset
extern int g_sm_limit;                     // SMs the persistent tcgen05 kernels may occupy (0 = all), stg_set_sm_limit
#define STG_LAUNCH_CHECK()                 \
  do {                                     \
    ++::stg::g_launch_count;               \
    STG_CUDA_CHECK(cudaGetLastError());    \
  } while (0)

using bf16 = __nv_bfloat16;

__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(bf16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f<bf16>(float v) { return __float2bfloat16_rn(v); }

// 4 consecutive elements, 4-element aligned.
__device__ __forceinline__ void ld4(const float* p, float (&o)[4]) {
  float4 v = *reinterpret_cast<const float4*>(p);
  o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
}
__device__ __forceinline__ void ld4(const bf16* p, float (&o)[4]) {
  uint2 v = *reinterpret_cast<const uint2*>(p);
  __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&v.x);
  __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&v.y);
  o[0] = __low2float(a); o[1] = __high2float(a); o[2] = __low2float(b); o[3] = __high2float(b);
}
__device__ __forceinline__ void st4(float* p, const float (&v)[4]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
__device__ __forceinline__ void st4(bf16* p, const float (&v)[4]) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]);
  __nv_bfloat162 b = __floats2bfloat162_rn(v[2], v[3]);
  uint2 u;
  u.x = *reinterpret_cast<uint32_t*>(&a);
  u.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = u;
}

__device__ __forceinline__ float act_apply(int act, float v) {
  switch (act) {
    case STG_ACT_RELU: return v > 0.f ? v : 0.f;
    case STG_ACT_LEAKY: return v > 0.f ? v : 0.1f * v;
    case STG_ACT_TANH: return tanhf(v);
    default: return v;
  }
}
// derivative of the activation expressed through its OUTPUT m
__device__ __forceinline__ float act_grad_from_output(int mode, float m) {
  switch (mode) {
    case STG_ACT_RELU: return m > 0.f ? 1.f : 0.f;
    case STG_ACT_LEAKY: return m > 0.f ? 1.f : 0.1f;
    case STG_ACT_TANH: return 1.f - m * m;
    default: return 1.f;
  }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// block-wide sum; `red` is >= 32 floats of shared memory; result valid in every thread
__device__ __forceinline__ float block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float r = (lane < nw) ? red[lane] : 0.f;
  r = warp_sum(r);
  return r;
}

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// engines.  valid_units / rows_per_unit: the per-sample length mask of stg_conv_masked (nullptr: none)
int conv_simt(const StgConv* d, cudaStream_t s, const int32_t* valid_units = nullptr, int rows_per_unit = 1);
int conv_tc(const StgConv* d, cudaStream_t s, const int32_t* valid_units = nullptr, int rows_per_unit = 1);
int conv_tc_plan(const StgConv* d, int* out);   // host-only: the plan conv_tc would launch (16 ints, see stg_debug_conv_plan)
bool conv_tc_supported(const StgConv* d);
int wgrad_simt(const StgWgrad* d, cudaStream_t s);
int wgrad_tc(const StgWgrad* d, cudaStream_t s);
bool wgrad_tc_supported(const StgWgrad* d);
int tc_pack_groups(int c_in, int c_out, int groups);
bool conv_c1_supported(const StgConv* d);
int conv_c1(const StgConv* d, cudaStream_t s);
bool wgrad_c1_supported(const StgWgrad* d);
int wgrad_c1(const StgWgrad* d, cudaStream_t s);
void conv_tc_set_trace(long long* buf);
void wgrad_tc_layout(const StgWgrad* d, int* ld, int* span);

}  // namespace stg
