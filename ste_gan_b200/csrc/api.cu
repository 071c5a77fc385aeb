// extern "C" entry points that dispatch between the engines, plus diagnostics.
#include <string.h>

#include <string>

#include "common.cuh"

namespace stg {

static thread_local std::string g_last_error;
unsigned long long g_launch_count = 0;
double g_ingest_bytes = 0.0;
int g_sm_limit = 0;   // stg_set_sm_limit: SMs the persistent tcgen05 kernels may occupy (0 = all)

void set_cuda_error(cudaError_t e, const char* where) {
  g_last_error = std::string(cudaGetErrorName(e)) + ": " + cudaGetErrorString(e) + " at " + where;
}

int colsum(const void* dy, int dtype, int64_t rows, int C, float* out, cudaStream_t s);

static int validate_conv(const StgConv* d) {
  if (!d || !d->src || !d->w) return STG_EINVAL;
  if (d->dtype != STG_F32 && d->dtype != STG_BF16) return STG_EINVAL;
  if (d->n_samples < 1 || d->phases < 1 || d->t_src < 1 || d->t_dst < 1) return STG_EINVAL;
  if (d->groups < 1 || d->c_src % d->groups || d->c_dst % d->groups) return STG_EINVAL;
  if (d->k < 1 || d->dilation < 1 || d->stride < 1 || d->pad < 0) return STG_EINVAL;
  if (d->post_shift < 0 || d->post_shift > 1) return STG_EINVAL;
  if (d->dup_rows && d->pair_sum) return STG_EINVAL;
  if (!d->y_raw && !d->y_act) return STG_EINVAL;
  if (d->w_fwd_pack && !d->transposed) return STG_EINVAL;
  return STG_OK;
}

}  // namespace stg

using namespace stg;

extern "C" int stg_conv(const StgConv* d, stg_stream_t stream) {
  int r = validate_conv(d);
  if (r) return r;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  switch (d->engine) {
    case STG_ENGINE_SIMT: return d->w_fwd_pack ? STG_EUNSUPPORTED : conv_simt(d, s);
    case STG_ENGINE_TCGEN05: return conv_tc(d, s);
    case STG_ENGINE_AUTO:
      if (conv_c1_supported(d)) return conv_c1(d, s);   // 1-channel logits layers: matrix-vector kernels
      if (conv_tc_supported(d)) return conv_tc(d, s);
      return d->w_fwd_pack ? STG_EUNSUPPORTED : conv_simt(d, s);
    default: return STG_EINVAL;
  }
}

/* stg_conv with per-sample length masks (forward only; the matvec engine is never chosen) */
extern "C" int stg_conv_masked(const StgConv* d, const int32_t* valid_units, int32_t rows_per_unit, stg_stream_t stream) {
  int r = validate_conv(d);
  if (r) return r;
  if (!valid_units || rows_per_unit < 1 || d->transposed || d->pair_sum || d->phases != 1) return STG_EINVAL;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  switch (d->engine) {
    case STG_ENGINE_SIMT: return conv_simt(d, s, valid_units, rows_per_unit);
    case STG_ENGINE_TCGEN05: return conv_tc(d, s, valid_units, rows_per_unit);
    case STG_ENGINE_AUTO:
      return conv_tc_supported(d) ? conv_tc(d, s, valid_units, rows_per_unit) : conv_simt(d, s, valid_units, rows_per_unit);
    default: return STG_EINVAL;
  }
}

/* which engine a call will run on: STG_ENGINE_SIMT, STG_ENGINE_TCGEN05 or STG_ENGINE_MATVEC */
extern "C" int stg_conv_route(const StgConv* d) {
  if (!d || validate_conv(d) != STG_OK) return STG_EINVAL;
  if (d->engine == STG_ENGINE_SIMT) return STG_ENGINE_SIMT;
  if (d->engine == STG_ENGINE_TCGEN05) return STG_ENGINE_TCGEN05;
  if (conv_c1_supported(d)) return STG_ENGINE_MATVEC;
  return conv_tc_supported(d) ? STG_ENGINE_TCGEN05 : STG_ENGINE_SIMT;
}
extern "C" int stg_wgrad_route(const StgWgrad* d) {
  if (!d) return STG_EINVAL;
  if (d->engine == STG_ENGINE_SIMT) return STG_ENGINE_SIMT;
  if (d->engine == STG_ENGINE_TCGEN05) return STG_ENGINE_TCGEN05;
  if (wgrad_c1_supported(d)) return STG_ENGINE_MATVEC;
  return wgrad_tc_supported(d) ? STG_ENGINE_TCGEN05 : STG_ENGINE_SIMT;
}
extern "C" int stg_conv_tc_supported(const StgConv* d) { return (d && validate_conv(d) == STG_OK && conv_tc_supported(d)) ? 1 : 0; }
extern "C" int stg_tc_pack_groups(int c_in, int c_out, int groups) {
  if (groups < 1 || c_in % groups || c_out % groups) return groups;
  return tc_pack_groups(c_in, c_out, groups);
}
extern "C" int stg_wgrad_tc_supported(const StgWgrad* d) { return (d && wgrad_tc_supported(d)) ? 1 : 0; }

extern "C" int stg_conv_wgrad(const StgWgrad* d, stg_stream_t stream) {
  if (!d || !d->x || !d->dy) return STG_EINVAL;
  if (d->dtype != STG_F32 && d->dtype != STG_BF16) return STG_EINVAL;
  if (d->groups < 1 || d->c_in % d->groups || d->c_out % d->groups) return STG_EINVAL;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int r = STG_OK;
  if (d->dw) {
    // the tcgen05 engine folds the bias gradient into the same kernel (one extra MMA against an all-ones operand)
    if (d->engine == STG_ENGINE_AUTO && wgrad_c1_supported(d)) return wgrad_c1(d, s);   // incl. the bias gradient
    if (d->engine == STG_ENGINE_TCGEN05) return wgrad_tc(d, s);
    if (d->engine == STG_ENGINE_AUTO && wgrad_tc_supported(d)) return wgrad_tc(d, s);
    if (d->engine == STG_ENGINE_AUTO || d->engine == STG_ENGINE_SIMT) r = wgrad_simt(d, s);
    else r = STG_EINVAL;
    if (r) return r;
  }
  if (d->dbias) r = colsum(d->dy, d->dtype, (int64_t)d->n_samples * d->phases * d->t_out, d->c_out, d->dbias, s);
  return r;
}

extern "C" int stg_wgrad_layout(const StgWgrad* d, int* ld, int* span) {
  if (!d || !ld || !span || d->groups < 1 || d->c_in % d->groups) return STG_EINVAL;
  const bool tc = d->engine == STG_ENGINE_TCGEN05 ||
                  (d->engine == STG_ENGINE_AUTO && !wgrad_c1_supported(d) && wgrad_tc_supported(d));
  if (tc) { wgrad_tc_layout(d, ld, span); return STG_OK; }
  *span = d->c_in / d->groups;
  *ld = d->k * *span;
  return STG_OK;
}

extern "C" const char* stg_strerror(int code) {
  switch (code) {
    case STG_OK: return "ok";
    case STG_EINVAL: return "invalid argument or unsupported shape";
    case STG_ECUDA: return "CUDA error";
    case STG_EUNSUPPORTED: return "shape not supported by the requested engine";
    default: return "unknown error";
  }
}
extern "C" const char* stg_last_cuda_error(void) { return g_last_error.c_str(); }
extern "C" int stg_version(void) { return 100; }
extern "C" unsigned long long stg_launch_count(void) { return g_launch_count; }
extern "C" void stg_set_sm_limit(int n) { g_sm_limit = n > 0 ? n : 0; }
/* debug: bytes the tcgen05 launches since the last reset were planned to pull into shared memory through TMA */
extern "C" double stg_debug_ingest_bytes(int reset) { const double v = g_ingest_bytes; if (reset) g_ingest_bytes = 0.0; return v; }

/* debug, host-only: the launch plan of the tcgen05 convolution engine for a descriptor (pointers only need to be non-NULL) */
extern "C" int stg_debug_conv_plan(const StgConv* d, int* out) {
  if (!out) return STG_EINVAL;
  const int r = validate_conv(d);
  if (r != STG_OK) return r;
  return conv_tc_plan(d, out);
}

/* debug: device buffer of 1 + 3*4000 int64 receiving a timeline of CTA 0 of every following stg_conv tcgen05 launch */
extern "C" int stg_debug_set_trace(void* buf) { conv_tc_set_trace(static_cast<long long*>(buf)); return STG_OK; }
