// tcgen05 weight-gradient kernel, bf16 in / fp32 accumulate.
//
//   dw[co][j][ci] += sum_{sample n, row r} dy[n][r][co] * x[n][r*stride + j*dilation - pad][ci]
//
// GEMM view: M = 128 output channels (TMEM lanes), N = BNW input channels per tap (TMEM
// columns, one accumulator block per tap), K = time rows in chunks of 64.  The
// contraction index (time) is the slow axis of the channels-last tensors, so both
// operands are MN-major: a TMA box of (64 channels x 64 rows) lands in shared memory as
// 64 rows of 128 B with 128-byte swizzle, which is exactly the canonical MN-major SW128
// UMMA layout ((8,n),(8,k)):((1,LBO),(8,SBO)) with LBO = bytes between 64-channel boxes
// and SBO = 1024.  Zero padding / dilation / sample boundaries again come from TMA
// out-of-bounds fill.  Split-K over (sample, row-chunk) pairs.
//
// Epilogue: the fp32 accumulator tile is staged through shared memory in 128 x 32 sub-tiles
// (128-byte swizzle) and added into the gradient with TMA REDUCE (cp.reduce.async.bulk.tensor
// .add.f32): one bulk L2 reduction per sub-tile instead of 4096 scalar atomics whose lanes
// are a whole gradient row apart.  The bias gradient (column sums of dy) rides along as one
// extra 16-column MMA per K step against an all-ones B operand.
//
// Grouped convolutions: the 128 output channels of a tile only meet the input channels of
// their own groups - a span of ci_span channels; the MMA computes the dense 128 x ci_span
// product and the gradient is written in the "span" layout dw[co][j][ci_span] whose
// off-diagonal entries are ignored by the fold backward (stg_wgrad_layout).
#include <string.h>

#include "tc_common.cuh"

namespace stg {
namespace {

using namespace tc;

constexpr int RK = 64;                 // time rows per K chunk
constexpr int BOX_BYTES = RK * 128;    // one (64 ch x 64 rows) box
constexpr int MAX_STAGES = 6;
constexpr int BIAS_COLS = 32;          // TMEM columns reserved for the bias accumulator (16 used)
constexpr int STAGE_TILE = 128 * 32 * 4;  // one fp32 128 x 32 epilogue sub-tile

struct WgTcP {
  int phases, t_out, c_in, c_out, k, stride;
  int cin_g, cout_g, ci_span, x_tiles;  // groups: channels per group, input-channel span of one 128-row co tile
  int n_taps, tap_groups, bnw, nbox_b, stages, tmem_cols;
  int chunks_per_sample, total_chunks, chunks_per_split;
  int bias_tg;                          // tap group whose x-tile-0 CTAs also accumulate the bias gradient (-1: none)
  // x window (stride 1): the taps of a group read row-shifted views (tap * dilation rows further down) of ONE
  // TMA-loaded window of 64 + (n_taps-1)*dilation rows per 64-channel box, instead of one 64-row tile per tap
  int win, win_rows, wb_bytes, dilation;
  int tap_off[STG_MAX_TAPS];
  float* dbias;
};

__device__ __forceinline__ void tma_reduce_add_3d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

__global__ void __launch_bounds__(192, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmX,
                const __grid_constant__ CUtensorMap tmD, const WgTcP p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int a_bytes = 2 * BOX_BYTES;
  const int b_bytes = p.nbox_b * BOX_BYTES;  // per tap
  const int stage_bytes = a_bytes + (p.win ? p.nbox_b * p.wb_bytes : p.n_taps * b_bytes);
  const uint32_t epi_base = smem_base + p.stages * stage_bytes;      // 2 x STAGE_TILE staging + BOX_BYTES of ones
  const uint32_t ones_base = epi_base + 2 * STAGE_TILE;
  const uint32_t bar_base = ones_base + BOX_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (MAX_STAGES + s); };
  const uint32_t tmem_full_bar = bar_base + 8u * (2 * MAX_STAGES);
  const uint32_t tmem_slot = bar_base + 8u * (2 * MAX_STAGES + 1);

  // broadcast from lane 0: the compiler can prove the warp index (hence every role branch) warp-uniform, so the
  // single-issuer instructions (TMA, tcgen05.mma / commit) take their operands straight from uniform registers
  // instead of a per-instruction ELECT + R2UR "waterfall"
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int co_tile = blockIdx.y / p.tap_groups, tg = blockIdx.y - co_tile * p.tap_groups;
  const int co0 = co_tile * 128;
  const int span0 = (co0 / p.cout_g) * p.cin_g;   // first input channel this co tile meets
  const int ci0 = span0 + blockIdx.x * p.bnw;
  const int tap0 = tg * p.n_taps;
  const int ntap = min(p.n_taps, p.k - tap0);
  const int q0 = blockIdx.z * p.chunks_per_split, q1 = min(p.total_chunks, q0 + p.chunks_per_split);
  const bool do_bias = p.dbias != nullptr && tg == p.bias_tg && blockIdx.x == 0;

  pdl_trigger();
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmY);
    prefetch_tmap(&tmX);
    prefetch_tmap(&tmD);
    for (int s = 0; s < p.stages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols); tmem_relinquish(); }
  if (do_bias) {  // all-ones B operand (any layout of ones is ones; shared memory only)
    for (int i = threadIdx.x; i < BOX_BYTES / 4; i += blockDim.x)
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(ones_base + 4u * i), "r"(0x3F803F80u) : "memory");
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();      // prologue above overlapped the previous kernel; global memory is only touched from here on
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  const uint32_t bias_tmem = tmem_base + (uint32_t)(p.n_taps * p.bnw);

  if (warp == 0) {
    // ===== TMA producer: warp-uniform loop, elected issue, coordinates advance by increments (see conv_tc.cu) =====
    const uint32_t tx_bytes = (uint32_t)(a_bytes + (p.win ? p.nbox_b * p.win_rows * 128 : ntap * b_bytes));
    int s = 0; uint32_t phs = 0;
    const int n0 = q0 / p.chunks_per_sample;
    int rc = q0 - n0 * p.chunks_per_sample, b = n0 / p.phases, ph = n0 - b * p.phases;
    for (int q = q0; q < q1; ++q) {
      const int r0 = rc * RK;
      mbar_wait(empty_bar(s), phs ^ 1);
      mbar_expect_tx_el(full_bar(s), tx_bytes);
      const uint32_t a_dst = smem_base + (uint32_t)(s * stage_bytes);
      tma_load_4d_el(a_dst, &tmY, full_bar(s), co0, r0, ph, b);
      tma_load_4d_el(a_dst + BOX_BYTES, &tmY, full_bar(s), co0 + 64, r0, ph, b);
      if (p.win) {
#pragma unroll 1
        for (int bx = 0; bx < p.nbox_b; ++bx)
          tma_load_4d_el(a_dst + a_bytes + bx * p.wb_bytes, &tmX, full_bar(s), ci0 + bx * 64, r0 + p.tap_off[tap0], ph, b);
      } else {
#pragma unroll 1
        for (int tl = 0; tl < ntap; ++tl)
#pragma unroll 1
          for (int bx = 0; bx < p.nbox_b; ++bx)
            tma_load_4d_el(a_dst + a_bytes + tl * b_bytes + bx * BOX_BYTES, &tmX, full_bar(s), ci0 + bx * 64,
                           r0 * p.stride + p.tap_off[tap0 + tl], ph, b);
      }
      if (++s == p.stages) { s = 0; phs ^= 1u; }
      if (++rc == p.chunks_per_sample) { rc = 0; if (++ph == p.phases) { ph = 0; ++b; } }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: warp-uniform loop, elected issue, descriptors advance by adds =====
    const uint32_t idesc = idesc_bf16_f32(128, p.bnw, 1, 1);
    const uint32_t idesc_b = idesc_bf16_f32(128, 16, 1, 1);
    const uint64_t ones_desc = smem_desc_mnmajor_sw128(ones_base, BOX_BYTES, 1024);
    const uint64_t adesc0 = smem_desc_mnmajor_sw128(smem_base, BOX_BYTES, 1024);
    const uint64_t bdesc0 = smem_desc_mnmajor_sw128(smem_base + a_bytes, p.win ? (uint32_t)p.wb_bytes : (uint32_t)BOX_BYTES, 1024);
    const uint32_t dstep = (uint32_t)stage_bytes >> 4;                                      // next stage (address field units of 16 B)
    const uint32_t tstep = p.win ? (uint32_t)(p.dilation * 128) >> 4 : (uint32_t)b_bytes >> 4;  // next tap: window row shift / next tile
    int s = 0; uint32_t phs = 0;
    for (int q = q0; q < q1; ++q) {
      mbar_wait(full_bar(s), phs);
      tc_fence_after();
      const uint64_t ad = adesc0 + (uint64_t)((uint32_t)s * dstep), bd0 = bdesc0 + (uint64_t)((uint32_t)s * dstep);
      const uint32_t acc0 = q > q0 ? 1u : 0u;
#pragma unroll 1
      for (int tl = 0; tl < ntap; ++tl) {
        const uint64_t bd = bd0 + (uint64_t)((uint32_t)tl * tstep);
#pragma unroll
        for (int ks = 0; ks < RK / 16; ++ks)  // 16 rows = 2048 B further along K
          umma_bf16_el(tmem_base + (uint32_t)(tl * p.bnw), ad + (uint64_t)(ks * 128), bd + (uint64_t)(ks * 128), idesc,
                       ks > 0 ? 1u : acc0);
      }
      if (do_bias) {
#pragma unroll
        for (int ks = 0; ks < RK / 16; ++ks)
          umma_bf16_el(bias_tmem, ad + (uint64_t)(ks * 128), ones_desc + (uint64_t)(ks * 128), idesc_b, ks > 0 ? 1u : acc0);
      }
      umma_commit_el(empty_bar(s));
      if (q == q1 - 1) umma_commit_el(tmem_full_bar);
      if (++s == p.stages) { s = 0; phs ^= 1u; }
    }
  } else {
    // ===== epilogue: TMEM -> swizzled smem sub-tiles -> TMA reduce-add into dw =====
    const int sub = warp & 3;
    const int row = sub * 32 + lane;   // output channel co0 + row
    mbar_wait(tmem_full_bar, 0);
    tc_fence_after();
    const uint32_t t_lane = tmem_base + ((uint32_t)(sub * 32) << 16);
    int buf = 0, issued = 0;
    const int ci_lim = min(p.bnw, p.ci_span - (int)blockIdx.x * p.bnw);  // valid columns of this x tile
    for (int tl = 0; tl < ntap; ++tl) {
      for (int c = 0; c < ci_lim; c += 32) {
        // wait until the TMA reduce that last read this staging buffer is done reading it
        if (issued >= 2) { if (threadIdx.x == 64) bulk_wait_read<1>(); epi_bar_sync(); }
        const uint32_t dst = epi_base + buf * STAGE_TILE + (uint32_t)row * 128u;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float v[16];
          tmem_ld16(t_lane + (uint32_t)(tl * p.bnw + c + 16 * h), v);
#pragma unroll
          for (int j = 0; j < 4; ++j) {  // 16-byte chunk (4*h + j) of the row goes to position chunk ^ (row & 7)
            const uint32_t a = dst + (uint32_t)((((4 * h + j) ^ (row & 7)) & 7) << 4);
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v[4 * j]), "f"(v[4 * j + 1]),
                         "f"(v[4 * j + 2]), "f"(v[4 * j + 3]) : "memory");
          }
        }
        fence_proxy_async();
        epi_bar_sync();
        if (threadIdx.x == 64) {
          tma_reduce_add_3d(&tmD, epi_base + buf * STAGE_TILE, (int)blockIdx.x * p.bnw + c, tap0 + tl, co0);
          bulk_commit();
        }
        buf ^= 1; ++issued;
      }
    }
    if (do_bias) {
      float v[16];
      tmem_ld16(t_lane + (uint32_t)(p.n_taps * p.bnw), v);
      if (co0 + row < p.c_out) atomicAdd(p.dbias + co0 + row, v[0]);
    }
    if (threadIdx.x == 64) bulk_wait_read<0>();   // reductions have read their staging tiles; they complete by the end of the grid
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

int make_tmap_f32_sw128(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                        const uint32_t* box) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) { set_cuda_error(cudaErrorNotSupported, "cuTensorMapEncodeTiled entry point"); return STG_ECUDA; }
  cuuint64_t gd[5]; cuuint64_t gs[4]; cuuint32_t bx[5]; cuuint32_t es[5];
  for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) gs[i] = strides_bytes[i];
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_cuda_error(cudaErrorInvalidValue, "cuTensorMapEncodeTiled(f32) failed"); return STG_ECUDA; }
  return STG_OK;
}

int span_of(const StgWgrad* d) {
  if (d->groups == 1) return d->c_in;
  const int cin_g = d->c_in / d->groups, cout_g = d->c_out / d->groups;
  return cout_g >= 128 ? cin_g : (128 / cout_g) * cin_g;
}

}  // namespace

bool wgrad_tc_supported(const StgWgrad* d) {
  if (d->dtype != STG_BF16) return false;
  if (d->k < 1 || d->k > STG_MAX_TAPS) return false;
  if ((d->c_in % 8) || (d->c_out % 8)) return false;
  if (d->stride > 4) return false;
  if (d->c_out < 32) return false;  // 1- and 8-channel outputs: CUDA-core engine
  if (d->groups > 1) {
    const int cout_g = d->c_out / d->groups;
    if (cout_g < 128 ? (128 % cout_g) : (cout_g % 128)) return false;  // co tiles aligned to group boundaries
  }
  if (span_of(d) % 4) return false;  // 16-byte rows of the fp32 gradient for the TMA reduction
  return true;
}

// Layout of dw the engine writes: element (co, j, ci_local) at co*ld + j*span + goff(co) + ci_local with
// goff(co) = ((co / cout_g) % (128 / cout_g)) * cin_g when cout_g < 128, else 0.
void wgrad_tc_layout(const StgWgrad* d, int* ld, int* span) {
  *span = span_of(d);
  *ld = d->k * *span;
}

int wgrad_tc(const StgWgrad* d, cudaStream_t s) {
  if (!wgrad_tc_supported(d)) return STG_EUNSUPPORTED;
  WgTcP p;
  p.phases = d->phases; p.t_out = d->t_out; p.c_in = d->c_in; p.c_out = d->c_out; p.k = d->k; p.stride = d->stride;
  p.cin_g = d->c_in / d->groups; p.cout_g = d->c_out / d->groups;
  p.ci_span = span_of(d);
  p.bnw = p.ci_span > 64 ? 128 : 64;
  p.x_tiles = ceil_div(p.ci_span, p.bnw);
  p.nbox_b = p.bnw / 64;
  const int epi_bytes = 2 * STAGE_TILE + BOX_BYTES;
  const int smem_budget = 200 * 1024 - epi_bytes;
  int taps = (512 - BIAS_COLS) / p.bnw;         // TMEM columns, bias block after the taps
  while (taps > 1 && (2 * BOX_BYTES + taps * p.nbox_b * BOX_BYTES) * 2 > smem_budget) --taps;  // >= 2 stages
  if (taps > d->k) taps = d->k;
  p.n_taps = taps;
  p.tap_groups = ceil_div(d->k, taps);
  p.bias_tg = p.tap_groups - 1;                 // the last tap group has the fewest taps
  p.tmem_cols = 32;
  while (p.tmem_cols < taps * p.bnw + BIAS_COLS) p.tmem_cols *= 2;
  for (int j = 0; j < d->k; ++j) p.tap_off[j] = j * d->dilation - d->pad;
  p.dilation = d->dilation;
  p.win_rows = RK + (taps - 1) * d->dilation;
  p.win = (d->stride == 1 && taps > 1 && p.win_rows <= 256) ? 1 : 0;
  p.wb_bytes = ceil_div(p.win_rows * 128, 1024) * 1024;
  const int stage_bytes = 2 * BOX_BYTES + (p.win ? p.nbox_b * p.wb_bytes : taps * p.nbox_b * BOX_BYTES);
  int stages = smem_budget / stage_bytes;
  if (stages > MAX_STAGES) stages = MAX_STAGES;
  p.chunks_per_sample = ceil_div(d->t_out, RK);
  p.total_chunks = d->n_samples * d->phases * p.chunks_per_sample;
  const int gx = p.x_tiles, gy = ceil_div(d->c_out, 128) * p.tap_groups;
  // split-K factor: as many splits as still fit ONE wave (one CTA per SM: ~200 KB of shared memory each) - rounding up
  // (180 CTAs for 36 tiles) put a second, nearly empty wave behind the first
  static const int n_sm = [] { int d = 0, n = 148; if (cudaGetDevice(&d) == cudaSuccess) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, d); return n > 0 ? n : 148; }();
  const int sms = (g_sm_limit > 0 && g_sm_limit < n_sm) ? g_sm_limit : n_sm;
  int want = sms / (gx * gy);
  if (want < 1) want = 1;
  if (want > p.total_chunks) want = p.total_chunks;
  p.chunks_per_split = ceil_div(p.total_chunks, want);
  const int nsplit = ceil_div(p.total_chunks, p.chunks_per_split);
  if (stages > p.chunks_per_split) stages = p.chunks_per_split;
  if (stages < 1) stages = 1;
  p.stages = stages;
  p.dbias = d->dbias;
  const size_t smem = (size_t)stages * stage_bytes + epi_bytes + 1024 + 8 * (2 * MAX_STAGES + 2);

  CUtensorMap tmY, tmX, tmD;
  {
    const uint64_t C = d->c_out, P = d->phases, T = d->t_out, B = d->n_samples;
    const uint64_t dims[4] = {C, T, P, B};
    const uint64_t strides[3] = {P * C * 2, C * 2, T * P * C * 2};
    const uint32_t box[4] = {64, RK, 1, 1};
    int r = make_tmap_bf16(&tmY, d->dy, 4, dims, strides, box, nullptr);
    if (r) return r;
  }
  {
    const uint64_t C = d->c_in, P = d->phases, T = d->t_in, B = d->n_samples;
    const uint64_t dims[4] = {C, T, P, B};
    const uint64_t strides[3] = {P * C * 2, C * 2, T * P * C * 2};
    const uint32_t box[4] = {64, (uint32_t)(p.win ? p.win_rows : RK * d->stride), 1, 1};
    const uint32_t es[4] = {1, (uint32_t)d->stride, 1, 1};
    int r = make_tmap_bf16(&tmX, d->x, 4, dims, strides, box, es);
    if (r) return r;
  }
  {
    const uint64_t W = p.ci_span, K = d->k, M = d->c_out;
    const uint64_t dims[3] = {W, K, M};
    const uint64_t strides[2] = {W * 4, K * W * 4};
    const uint32_t box[3] = {32, 1, 128};
    int r = make_tmap_f32_sw128(&tmD, d->dw, 3, dims, strides, box);
    if (r) return r;
  }
  static bool attr_set = false;
  if (!attr_set) {
    STG_CUDA_CHECK(cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    attr_set = true;
  }
  dim3 grid(gx, gy, nsplit);
  g_ingest_bytes += (double)gx * gy * nsplit * p.chunks_per_split * stage_bytes;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = dim3(192); cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[1];
  cfg.attrs = at; cfg.numAttrs = tc_launch_attrs(at);
  STG_CUDA_CHECK(cudaLaunchKernelEx(&cfg, wgrad_tc_kernel, tmY, tmX, tmD, p));
  STG_LAUNCH_CHECK();
  return STG_OK;
}

}  // namespace stg
