// tcgen05 implicit-GEMM convolution (forward and data-gradient), bf16 in / fp32 accumulate.
//
// GEMM view (channels-last activations):   D[t][c_dst] = sum_taps sum_{c_src} A_tap[t][c_src] * W_tap[c_dst][c_src]
//   M = 128 output rows of one sample           -> TMEM lanes
//   N = BN <= 256 output channels               -> TMEM columns
//   K = 64-channel chunks, one per (tap, chunk) -> one pipeline stage each
// A tiles come straight from the activation tensor by TMA: the row coordinate is
// h0*stride + tap_offset, may be negative or run past the sample and is zero-filled by
// the TMA unit, which implements zero padding, dilation and per-sample boundaries with
// no im2col buffer.  Period views (DiscriminatorP's [B,C,T/p,p] Conv2d) are a 4-D tensor map
// (C, phase, h, B) and a tile packs ALL p phases of 128/p consecutive h rows, so the M tile stays full
// however short T/p is and its output rows are contiguous in memory.
// W tiles come from the packed [k][c_dst][c_src/g] weights.  Both operands are K-major
// with 128-byte swizzle.
//
// PERSISTENT kernel: one CTA per SM walks the tile list (column tile fastest, so CTAs that run
// together share A rows in L2).  Warp 0 = TMA producer, warp 1 = TMEM alloc + single-thread
// tcgen05.mma issuer, the rest = epilogue.  The shared-memory ring runs continuously across tiles; the
// accumulator is DOUBLE-BUFFERED in TMEM (2 x 256 columns), so the epilogue of tile i overlaps the MMAs
// of tile i+1.
//
// Two epilogues (bias, pair-sum, add_pre, activation-derivative mask, residual add, activation, row
// duplication are fused in both):
//   STAGED  (bf16 outputs, c_dst % 8 == 0, no residue classes): 4 warps.  Epilogue operands are TMA-loaded
//           into 128 x 32 shared-memory sub-tiles two sub-tiles ahead, results are written to swizzled
//           shared memory and leave with TMA stores - no thread touches global memory, so the LSU only
//           sees conflict-free 16-byte shared accesses (row-per-thread global accesses cost one
//           wavefront per 16 bytes and made the epilogue, not the MMAs, the critical path).
//   DIRECT  (fp32 outputs, 1-channel logits, strided data-gradients): 8 warps, row-per-thread global
//           loads/stores with the next chunk's operands prefetched.
#include <string.h>

#include "tc_common.cuh"

namespace stg {

namespace {

using namespace tc;

constexpr int TM = 128;        // rows per CTA tile
constexpr int KC = 64;         // channels per K chunk (128 B of bf16)
constexpr int MAX_STAGES = 8;
constexpr int ACC_COLS = 256;  // TMEM column distance between the two accumulator buffers (TcP::acc_cols; 128 when two CTAs share an SM)
constexpr int SUB = 32;        // staged epilogue: columns per sub-tile (64-byte rows, SWIZZLE_64B)
constexpr int SLOT = TM * SUB * 2;  // bytes of one 128 x 32 bf16 sub-tile
constexpr int MAX_RES = 8;     // residues of a strided data-gradient (= stride)

struct TcEpi {
  int rows, c_dst, post_shift, mask_mode, act, dup_rows, out_f32, pair_sum;  // rows: output rows per sample (all phases)
  int n_in, n_out, has_pre, has_mask, has_post, has_raw, has_act;            // staged: slot bookkeeping
  int in_sh;                    // staged: the epilogue-operand ring holds 1 << in_sh sub-tiles (2, 4 or 8) in flight
  float act_slope, mask_slope;  // act(v) = max(v, act_slope*v) ; act'(m) = m > 0 ? 1 : mask_slope   (none 1, relu 0, leaky 0.1)
  const float* bias;
  const bf16 *add_pre, *mask, *add_post;
  void* y_raw;
  void* y_act;
  const int32_t* valid_units;   // stg_conv_masked: accumulator rows >= valid_units[b] * rows_per_unit are written as 0 (nullptr: no mask)
  int rows_per_unit;
};

// Per-group / per-tap tables, read with warp-uniform indices (uniform constant loads) by the producer / MMA warps.
struct TapTables {
  short g_off[STG_MAX_TAPS];   // source-row offset of the group's window (its rows start at h0*stride + g_off)
  short tap_shift[STG_MAX_TAPS];   // h-row shift of the tap inside its group's window
  unsigned char g_tfirst[STG_MAX_TAPS], g_ntaps[STG_MAX_TAPS];  // taps of group g: [g_tfirst, g_tfirst + g_ntaps)
  unsigned char tap_w[STG_MAX_TAPS];  // tap index into the packed weights
};

struct TcP {
  int phases, t_dst, stride, k_chunks, bn, stages, a_boxes, tmem_cols;
  int acc_cols, out_ring;  // TMEM distance between the two accumulator buffers; depth of the staged epilogue's output ring (3, or 2 when two CTAs share an SM)
  int pack, nh, mrows;     // phases packed per tile, h rows per tile, used accumulator rows = nh * pack
  int cs_g, cd_g;          // source / destination channels per (packed) group
  int n_res, tiles_m;      // output-row residues (1 unless transposed && stride > 1), row tiles per residue
  int tiles_n, n_tiles;    // column tiles, total tiles = B * n_res * tiles_m * tiles_n
  int n_samples;           // a row-class tail tile may gather rows past the last sample (zero-filled loads, clipped stores)
  // Row classes (staged, stride-1, single-phase kernels): T rows per sample rarely fill whole 128-row tiles (T = 100 /
  // 200 / 400: 78 %).  The rows of a sample are cut into 128-row tiles plus a binary tail (64 / 32 / 16 / 8 rows), and a
  // tail tile gathers the SAME seg-row slice of 128 / seg consecutive samples with one (C, seg rows, samples) TMA box -
  // loads, epilogue operands and stores alike.  Class c: cls_seg rows per sample starting at row cls_h0, cls_tps tiles
  // per sample (full tiles) or 0 (tail: one tile per 128 / seg samples); row tiles [cls_mt0[c], cls_mt0[c+1]).
  int n_cls, cls_mt0[5], cls_seg[4], cls_h0[4], cls_tps[4];
  // Tap groups ("A windows"): the taps of one group read row-shifted views of ONE TMA-loaded window of
  // nh + max_shift h rows (UMMA descriptors take any row offset into a 128B-swizzled tile - the swizzle is a
  // function of the shared-memory address, tools/rowshift_probe.py), so a k-tap conv loads its activations
  // once per group instead of once per tap.  One pipeline stage = (group, 64-channel chunk).
  int hb, a_bytes, max_ntaps;  // h rows per A box, bytes reserved for the window (1024-aligned), taps per stage slot
  int b_mn;                    // data-gradient: W tiles are [64 co rows][64 ci] boxes of the FORWARD pack (MN-major B operand);
                               // 2 = all bn/64 boxes of a tile come from ONE 4-D TMA box (c_dst/g % 64 == 0)
  // Compact groups (grouped convs whose groups have 16 / 32 / 64 source channels; K-major W only).  A 64-channel K chunk of
  // the activations holds cu_fpc = 64 / cu_k whole groups ("units") side by side; the W tile of a stage is the COMPACT
  // [cu_fpc * cu_n rows][cu_k] block of the pack (rows of 32 / 64 / 128 bytes, loaded with the matching swizzle), and
  // every unit gets its own MMA chain - N = cu_n, A descriptor advanced to the unit's channels inside the swizzle atom,
  // accumulator columns (chunk * cu_fpc + q) * cu_n.  Nothing is multiplied by the zeros of a block-diagonal weight
  // tile any more and the W bytes per stage shrink by 64 / cu_k (hardware check: tools/group_mma_probe.py).
  int cu_k, cu_n, cu_fpc;      // cu_k == 0: off
  int res_gfirst[MAX_RES + 1]; // groups of residue r: [res_gfirst[r], res_gfirst[r+1])
  TapTables tt;
  long long* trace;            // debug timeline (stg_debug_set_trace) or nullptr
  TcEpi e;
};

constexpr int MAX_STAGED_RES = 4;   // residue classes the staged epilogue has tensor maps for
// Epilogue tensors as 4-D maps (C, phase, h, B) - per residue class of a strided data-gradient: class r holds the
// rows h = h'*s + r, i.e. base + r rows, h stride s rows, extent ceil((T - r)/s) - and y_act as (C, dup, h, B).
struct EpiMaps {   // index: residue class (strided data-gradients) or row class (see TcP::n_cls) - never both
  CUtensorMap pre[MAX_STAGED_RES], mask[MAX_STAGED_RES], raw[MAX_STAGED_RES], post[MAX_STAGED_RES], act[MAX_STAGED_RES];
};
struct TmA4 { CUtensorMap m[4]; };   // activation map per row class

__device__ __forceinline__ void unpack8(const uint4& q, float* o) {
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&w[i]);
    o[2 * i] = __low2float(h);
    o[2 * i + 1] = __high2float(h);
  }
}
__device__ __forceinline__ uint4 pack8(const float* v) {
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    w[i] = *reinterpret_cast<uint32_t*>(&h);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ void ld16(const bf16* p, float (&o)[16]) {
  unpack8(*reinterpret_cast<const uint4*>(p), o);
  unpack8(*reinterpret_cast<const uint4*>(p + 8), o + 8);
}
__device__ __forceinline__ void st16(bf16* p, const float (&v)[16]) {
  *reinterpret_cast<uint4*>(p) = pack8(v);
  *reinterpret_cast<uint4*>(p + 8) = pack8(v + 8);
}
__device__ __forceinline__ void st16f(float* p, const float (&v)[16]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) *reinterpret_cast<float4*>(p + 4 * i) = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
}
__device__ __forceinline__ uint4 lds128(uint32_t a) {
  uint4 q;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(q.x), "=r"(q.y), "=r"(q.z), "=r"(q.w) : "r"(a) : "memory");
  return q;
}
__device__ __forceinline__ void sts128(uint32_t a, const uint4& q) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(q.x), "r"(q.y), "r"(q.z), "r"(q.w) : "memory");
}
// Branch-free activation forms keep the unrolled epilogue small enough for the instruction cache (a per-element
// switch with tanhf inlined 32x made the epilogue body ~50 KB and instruction-fetch bound).
__device__ __forceinline__ float fast_tanh(float x) {
  const float t = __expf(-2.f * fabsf(x));
  return copysignf(__fdividef(1.f - t, 1.f + t), x);
}
__device__ __forceinline__ float act_fast(const TcEpi& e, float v) {
  return e.act == STG_ACT_TANH ? fast_tanh(v) : fmaxf(v, e.act_slope * v);
}
__device__ __forceinline__ float dact_fast(const TcEpi& e, float m) {
  return e.mask_mode == STG_ACT_TANH ? 1.f - m * m : (m > 0.f ? 1.f : e.mask_slope);
}
// byte offset of 16-byte chunk j (0..3) of row r inside a SWIZZLE_64B sub-tile
__device__ __forceinline__ uint32_t sw64(int r, int j) { return (uint32_t)(r * 64 + ((j ^ ((r >> 1) & 3)) << 4)); }

// debug timeline of CTA 0: each role thread appends (tag, value, globaltimer) triples to its own region of the
// buffer (plain stores, no atomics: the probe must not perturb what it measures).  Regions of 1300 events:
// 0 producer (tag 1 tile start), 1 MMA issuer (2 tile start, 3 tile issued), 2 epilogue leader (10 tile start,
// 11 accumulator ready, 20..24 sub-tile phases, 12 sub-tile done).  Empty slots keep tag 0.
struct Tracer {
  long long* base; int n;
  __device__ __forceinline__ Tracer(long long* tr, int region) : base(tr && blockIdx.x == 0 ? tr + 1 + 3 * 1300 * region : nullptr), n(0) {}
  __device__ __forceinline__ void ev(int tag, int val) {
    if (base == nullptr || n >= 1300) return;
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    base[3 * n] = tag; base[3 * n + 1] = val; base[3 * n + 2] = t; ++n;
  }
};

// life-cycle events of CTA 0 (entry / set-up done / dependency released / exit), appended across launches through the
// counter in trace[0] so that back-to-back launches show their period and overlap
__device__ __forceinline__ void life_ev(long long* tr, int tag) {
  if (tr == nullptr || blockIdx.x != 0 || threadIdx.x != 0) return;
  long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  const int slot = (int)atomicAdd(reinterpret_cast<unsigned long long*>(tr), 1ull);
  if (slot < 1300) { long long* b = tr + 1 + 3 * 1300 * 3 + 3 * slot; b[0] = tag; b[1] = slot; b[2] = t; }
}

// ---------------------------------------------------------------------------------------------- tiles
struct Tile {
  int b, res, h0, col0, ch0, wcol0, g0, n_iters, cls;
};
__device__ __forceinline__ Tile decode_tile(const TcP& p, int t) {
  Tile x;
  const int tn = t % p.tiles_n; int u = t / p.tiles_n;
  int tm;
  // strided data-gradient: output rows h = h' * n_res + res are produced per residue class `res` from the
  // taps j with (res + pad - j*dilation) % stride == 0, as a stride-1 correlation over h'
  if (p.n_cls > 1) {
    int c = 0;
    while (c + 1 < p.n_cls && u >= p.cls_mt0[c + 1]) ++c;
    const int idx = u - p.cls_mt0[c];
    x.cls = c; x.res = 0;
    if (p.cls_tps[c] > 0) { x.b = idx / p.cls_tps[c]; tm = idx - x.b * p.cls_tps[c]; }
    else { x.b = idx * (TM / p.cls_seg[c]); tm = 0; }
    x.h0 = p.cls_h0[c] + tm * TM;
    x.col0 = tn * p.bn;
    x.ch0 = (x.col0 / p.cd_g) * p.cs_g;
    x.wcol0 = x.col0 % p.cd_g;
    x.g0 = p.res_gfirst[0];
    x.n_iters = (p.res_gfirst[1] - x.g0) * p.k_chunks;
    return x;
  } else {
    tm = u % p.tiles_m; u /= p.tiles_m;
    x.res = u % p.n_res; x.b = u / p.n_res;
  }
  x.cls = 0;
  x.h0 = tm * p.nh;
  x.col0 = tn * p.bn;
  x.ch0 = (x.col0 / p.cd_g) * p.cs_g;  // first source channel of this column tile's group
  x.wcol0 = x.col0 % p.cd_g;           // column offset inside the group (forward-pack W coordinates)
  x.g0 = p.res_gfirst[x.res];
  x.n_iters = (p.res_gfirst[x.res + 1] - x.g0) * p.k_chunks;
  return x;
}
// accumulator row m of a tile -> flat output row of the sample (before pair_sum), or -1
__device__ __forceinline__ int out_row(const TcP& p, const Tile& x, int m) {
  if (m >= p.mrows || x.b >= p.n_samples) return -1;
  const int hl = m / p.pack, ph = m - hl * p.pack;
  const int h = (x.h0 + hl) * p.n_res + x.res;
  return h < p.t_dst ? h * p.phases + ph : -1;
}

// stg_conv_masked: does output row `row` of sample b (before dup_rows) lie inside the sample's valid length?  Called after
// pdl_wait (valid_units may be written by the previous kernel of the stream).
__device__ __forceinline__ bool row_kept(const TcEpi& e, int b, int row) {
  return (int64_t)row < (int64_t)max(e.valid_units[b], 0) * e.rows_per_unit;
}

// ---------------------------------------------------------------------------------------------- direct epilogue
struct EpiIn {
  float pre[16], mk[16], post[16];
};
__device__ __forceinline__ void epi_load(const TcEpi& e, int b, int row, int col, bool row_ok, EpiIn& in) {
  if (!row_ok || col >= e.c_dst) return;
  const int ncols = min(16, e.c_dst - col);
  const bool vec = (ncols == 16) && ((e.c_dst & 7) == 0);
  const int64_t off = ((int64_t)b * e.rows + row) * e.c_dst + col;
  if (e.add_pre) {
    if (vec) ld16(e.add_pre + off, in.pre); else for (int i = 0; i < 16; ++i) in.pre[i] = i < ncols ? to_f(e.add_pre[off + i]) : 0.f;
  }
  if (e.mask) {
    if (vec) ld16(e.mask + off, in.mk); else for (int i = 0; i < 16; ++i) in.mk[i] = i < ncols ? to_f(e.mask[off + i]) : 0.f;
  }
  if (e.add_post) {
    const int64_t o2 = ((int64_t)b * (e.rows >> e.post_shift) + (row >> e.post_shift)) * e.c_dst + col;
    if (vec) ld16(e.add_post + o2, in.post); else for (int i = 0; i < 16; ++i) in.post[i] = i < ncols ? to_f(e.add_post[o2 + i]) : 0.f;
  }
}
// v: accumulator (+bias, pair-summed) of one output row, 16 channels
// keep == false (length mask): the row is written as 0 - a select, so NaN in the padded rows of add_post never reaches it
__device__ __forceinline__ void epi_store(const TcEpi& e, int b, int row, int col, float (&v)[16], const EpiIn& in, bool keep) {
  const int64_t off = ((int64_t)b * e.rows + row) * e.c_dst + col;
  const int ncols = min(16, e.c_dst - col);
  const bool vec = (ncols == 16) && ((e.c_dst & 7) == 0);
  if (e.add_pre) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] += in.pre[i];
  }
  if (e.mask) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] *= dact_fast(e, in.mk[i]);
  }
  if (e.add_post) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] += in.post[i];
  }
  if (!keep) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = 0.f;
  }
  if (e.y_raw) {
    if (e.out_f32) {
      float* p = static_cast<float*>(e.y_raw) + off;
      if (vec) st16f(p, v); else for (int i = 0; i < ncols; ++i) p[i] = v[i];
    } else {
      bf16* p = static_cast<bf16*>(e.y_raw) + off;
      if (vec) st16(p, v); else for (int i = 0; i < ncols; ++i) p[i] = __float2bfloat16_rn(v[i]);
    }
  }
  if (e.y_act) {
    float a[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = act_fast(e, v[i]);
    const int64_t o0 = e.dup_rows ? ((int64_t)b * 2 * e.rows + 2 * row) * e.c_dst + col : off;
    if (e.out_f32) {
      float* p0 = static_cast<float*>(e.y_act) + o0;
      if (vec) st16f(p0, a); else for (int i = 0; i < ncols; ++i) p0[i] = a[i];
      if (e.dup_rows) { float* p1 = p0 + e.c_dst; if (vec) st16f(p1, a); else for (int i = 0; i < ncols; ++i) p1[i] = a[i]; }
    } else {
      bf16* p0 = static_cast<bf16*>(e.y_act) + o0;
      if (vec) st16(p0, a); else for (int i = 0; i < ncols; ++i) p0[i] = __float2bfloat16_rn(a[i]);
      if (e.dup_rows) { bf16* p1 = p0 + e.c_dst; if (vec) st16(p1, a); else for (int i = 0; i < ncols; ++i) p1[i] = __float2bfloat16_rn(a[i]); }
    }
  }
}

// ---------------------------------------------------------------------------------------------- kernel
// kMask: stg_conv_masked (per-sample length masks in both epilogues); the unmasked instances compile without them
template <bool kStaged, bool kMask>
__global__ void __launch_bounds__(kStaged ? 384 : 352, kStaged ? 2 : 1)
conv_tc_kernel(const __grid_constant__ TmA4 tmA4, const __grid_constant__ CUtensorMap tmW,
               const __grid_constant__ EpiMaps em, const TcP p) {
  constexpr int EPI_WARPS = 8;   // warps that read the accumulator (arrivals on tmem_empty)
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment for SWIZZLE_128B tiles
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  // B tile bytes per tap (compact groups: only the rows of the chunk's units)
  const int b_bytes = p.cu_k ? p.cu_fpc * p.cu_n * p.cu_k * 2 : p.bn * KC * 2;
  const int stage_bytes = p.a_bytes + p.max_ntaps * b_bytes;
  const TcEpi& e = p.e;
  const int tile0 = (int)blockIdx.x, tstep = (int)gridDim.x;
  const uint32_t epi_base = smem_base + p.stages * stage_bytes;           // staged: (n_in << in_sh) + 3 n_out slots + bias
  const uint32_t bias_base = epi_base + (kStaged ? ((e.n_in << e.in_sh) + p.out_ring * e.n_out) * SLOT : 0);
  const uint32_t bar_base = bias_base + (kStaged ? 2048 : 0);   // one bias copy per epilogue team
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (MAX_STAGES + s); };
  auto tmem_full_bar = [&](int a) { return bar_base + 8u * (2 * MAX_STAGES + a); };
  auto tmem_empty_bar = [&](int a) { return bar_base + 8u * (2 * MAX_STAGES + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * MAX_STAGES + 4);
  auto in_bar = [&](int a) { return bar_base + 8u * (2 * MAX_STAGES + 6 + a); };   // a < 8

  // broadcast from lane 0: the compiler can prove the warp index (hence every role branch) warp-uniform, so the
  // single-issuer instructions (TMA, tcgen05.mma / commit) take their operands straight from uniform registers
  // instead of a per-instruction ELECT + R2UR "waterfall" (MMA issue: 410 -> 82 clk per stage)
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;

  life_ev(p.trace, 30);
  pdl_trigger();   // the next kernel of the stream may start its prologue now (it still waits for this grid to complete)
  if (warp == 0 && lane == 0) {
    for (int c = 0; c < p.n_cls; ++c) prefetch_tmap(&tmA4.m[c]);
    prefetch_tmap(&tmW);
    for (int s = 0; s < p.stages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tmem_full_bar(a), 1); mbar_init(tmem_empty_bar(a), EPI_WARPS); }
    for (int a = 0; a < 8; ++a) mbar_init(in_bar(a), 1);
    fence_barrier_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  life_ev(p.trace, 31);
  pdl_wait();      // everything above overlapped the previous kernel's tail; no global memory is touched before this line
  life_ev(p.trace, 32);
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  // Two producer warps: warp 0 loads the A (activation) boxes and posts the stage's expect_tx, the LAST warp of the CTA
  // loads the W boxes of the same stage onto the same barrier (its complete_tx may land before the expect_tx - both
  // belong to the same barrier phase, which cannot complete before warp 0's arrival).  One warp issuing both spent
  // ~240 clk per stage on issue alone, more than the MMAs of a narrow (bn <= 128) stage.
  constexpr int WPROD = kStaged ? 11 : 10;
  if ((warp == 0 || warp == WPROD) && p.max_ntaps == 1) {
    const bool do_a = warp == 0;
    // ===== TMA producers, one tap per stage (the common case) =====
    // Warp-uniform control flow: every lane runs the loop, lane 0's instructions take effect.  The loop body is
    // kept to a wait, an expect_tx and the TMA issues - ring position and coordinates advance by increments (the
    // div/mod + table look-ups of the first version cost the issuing thread ~900 clk per stage, more than the
    // stage's MMAs).
    const bool lead = lane == 0;
    Tracer trc(lead && do_a ? p.trace : nullptr, 0);
    const uint32_t a_box_bytes = (uint32_t)(p.hb * p.pack * KC * 2);
    const uint32_t tx_bytes = (uint32_t)p.a_boxes * a_box_bytes + (uint32_t)b_bytes;
    const int row_step = p.hb * p.stride;
    int s = 0; uint32_t phs = 0;   // ring position, continuous across tiles
#ifdef STG_PROF_LOOP
    long long prof[4] = {0, 0, 0, 0};   // clocks in: empty wait | expect_tx + A loads | W loads + advance ; stages
#endif
    for (int t = tile0; t < p.n_tiles; t += tstep) {
      const Tile x = decode_tile(p, t);
      trc.ev(1, t);
      const int n_groups = p.res_gfirst[x.res + 1] - x.g0;
      // W coordinate of the tile along the destination-channel axis
      const int wc = p.b_mn == 0 ? x.col0 : p.b_mn == 2 ? x.wcol0 / 64 : x.wcol0;
      for (int gi = 0; gi < n_groups; ++gi) {
        const int g = x.g0 + gi;
        const int row0 = x.h0 * p.stride + p.tt.g_off[g];
        const int tap = p.tt.tap_w[g];
        for (int chunk = 0; chunk < p.k_chunks; ++chunk) {
#ifdef STG_PROF_LOOP
          const long long pc0 = clock64();
#endif
          mbar_wait(empty_bar(s), phs ^ 1);
          trc.ev(4, chunk);
#ifdef STG_PROF_LOOP
          const long long pc1 = clock64();
#endif
          const uint32_t a_dst = smem_base + (uint32_t)(s * stage_bytes);
          const uint32_t fb = full_bar(s);
          const int c0 = x.ch0 + chunk * KC;
          if (do_a) {
            mbar_expect_tx_el(fb, tx_bytes);
#pragma unroll 1
            for (int bx = 0; bx < p.a_boxes; ++bx)
              tma_load_4d_el(a_dst + bx * a_box_bytes, &tmA4.m[x.cls], fb, c0, 0, row0 + bx * row_step, x.b);
          }
#ifdef STG_PROF_LOOP
          const long long pc2 = clock64();
#endif
          if (do_a) {
          } else if (p.cu_k) {       // compact groups: [cu_fpc * cu_n rows][cu_k] block of the units of this chunk
            tma_load_3d_el(a_dst + p.a_bytes, &tmW, fb, 0, x.col0 + chunk * p.cu_fpc * p.cu_n, tap);
          } else if (p.b_mn == 0) {
            tma_load_3d_el(a_dst + p.a_bytes, &tmW, fb, chunk * KC, wc, tap);
          } else if (p.b_mn == 2) {  // forward pack seen as (64, co row, ci/64, tap): one box = the whole [bn/64][64][64] tile
            tma_load_4d_el(a_dst + p.a_bytes, &tmW, fb, 0, c0, wc, tap);
          } else {  // forward pack [k][c_src][c_dst/g]: bn/64 boxes of (64 destination channels x 64 source-channel rows)
#pragma unroll 1
            for (int nb = 0; nb < p.bn / 64; ++nb)
              tma_load_3d_el(a_dst + p.a_bytes + nb * 8192, &tmW, fb, wc + nb * 64, c0, tap);
          }
          if (++s == p.stages) { s = 0; phs ^= 1u; }
#ifdef STG_PROF_LOOP
          const long long pc3 = clock64();
          prof[0] += pc1 - pc0; prof[1] += pc2 - pc1; prof[2] += pc3 - pc2; prof[3] += 1;
#endif
        }
      }
    }
#ifdef STG_PROF_LOOP
    if (lead && do_a && p.trace && blockIdx.x == 0) for (int i = 0; i < 4; ++i) p.trace[1 + 3 * 5200 + i] = prof[i];
#endif
  } else if (warp == 1 && p.max_ntaps == 1) {
    // ===== MMA issuer, one tap per stage (warp-uniform control flow) =====
    const bool lead = lane == 0;
    const uint32_t idesc = idesc_bf16_f32(TM, p.bn, 0, p.b_mn ? 1 : 0);
    const uint32_t idesc_u = idesc_bf16_f32(TM, p.cu_k ? p.cu_n : p.bn, 0, 0);   // compact groups: N = one unit's columns
    // ... K steps per unit = 1 << cu_ks, B descriptor without its start address, start-address step between units
    const int cu_ks = p.cu_k == 16 ? 0 : (p.cu_k == 32 ? 1 : 2), cu_km = (1 << cu_ks) - 1;
    const uint64_t cu_bhi = smem_desc_kmajor_narrow(0, p.cu_k ? p.cu_k * 2 : 128);
    const int cu_bq = (p.cu_n * p.cu_k * 2) >> 4;
    Tracer trc(lead ? p.trace : nullptr, 1);
    // descriptors of stage 0; a stage further on adds stage_bytes >> 4 to the 14-bit start-address field (no carry:
    // every operand address is below 256 KB)
    const uint64_t adesc0 = smem_desc_kmajor_sw128(smem_base);
    const uint64_t bdesc0 = p.b_mn ? smem_desc_mnmajor_sw128(smem_base + p.a_bytes, 8192, 1024) : smem_desc_kmajor_sw128(smem_base + p.a_bytes);
    const uint32_t dstep = (uint32_t)stage_bytes >> 4;
    const uint32_t bstep = p.b_mn ? 128u : 2u;   // 16 K elements further: +32 B inside the K-major atom / 16 rows (2048 B) of the MN-major tile
    int s = 0, acc_i = 0; uint32_t phs = 0;
#ifdef STG_PROF_LOOP
    long long mprof[3] = {0, 0, 0};     // clocks in: full wait | MMA issue + commits ; stages
#endif
    for (int t = tile0; t < p.n_tiles; t += tstep) {
      const Tile x = decode_tile(p, t);
      if (x.n_iters == 0) continue;
      const int as = acc_i & 1, aph = (acc_i >> 1) & 1;
      mbar_wait(tmem_empty_bar(as), aph ^ 1);  // epilogue(s) have drained this accumulator buffer
      tc_fence_after();
      trc.ev(2, t);
      const uint32_t d_tmem = tmem_base + (uint32_t)(as * p.acc_cols);
      int cu_chunk = 0;
      for (int it = 0; it < x.n_iters; ++it) {
#ifdef STG_PROF_LOOP
        const long long mc0 = clock64();
#endif
        mbar_wait(full_bar(s), phs);
        tc_fence_after();
        trc.ev(5, it);
#ifdef STG_PROF_LOOP
        const long long mc1 = clock64();
#endif
        const uint64_t ad = adesc0 + (uint64_t)((uint32_t)s * dstep), bd = bdesc0 + (uint64_t)((uint32_t)s * dstep);
        if (p.cu_k) {
          // compact groups: one MMA chain per unit of this chunk (see TcP::cu_k); `it` walks (tap group, chunk) with the
          // chunk fastest, so a unit's columns are first written while it < k_chunks.  A chunk is always 4 K steps:
          // step i belongs to unit q = i >> cu_ks, K step i & (kpu - 1) of that unit.
          const uint32_t dcol = d_tmem + (uint32_t)(cu_chunk * p.cu_fpc * p.cu_n);
          if (++cu_chunk == p.k_chunks) cu_chunk = 0;
          const uint64_t bu = cu_bhi | (uint64_t)(((smem_base + (uint32_t)(s * stage_bytes) + (uint32_t)p.a_bytes) >> 4) & 0x3FFFu);
          const uint32_t acc0 = it >= p.k_chunks ? 1u : 0u;
#pragma unroll
          for (int i = 0; i < KC / 16; ++i) {
            const int q = i >> cu_ks, ks = i & cu_km;
            umma_bf16_el(dcol + (uint32_t)(q * p.cu_n), ad + 2 * i, bu + (uint64_t)(q * cu_bq + 2 * ks), idesc_u, (acc0 | (uint32_t)(ks > 0)));
          }
        } else {
#pragma unroll
          for (int ks = 0; ks < KC / 16; ++ks)
            umma_bf16_el(d_tmem, ad + 2 * ks, bd + bstep * ks, idesc, (it > 0 || ks > 0) ? 1u : 0u);
        }
        umma_commit_el(empty_bar(s));
        if (it == x.n_iters - 1) umma_commit_el(tmem_full_bar(as));
        if (++s == p.stages) { s = 0; phs ^= 1u; }
#ifdef STG_PROF_LOOP
        const long long mc2 = clock64();
        mprof[0] += mc1 - mc0; mprof[1] += mc2 - mc1; mprof[2] += 1;
#endif
      }
      trc.ev(3, t);
      ++acc_i;
    }
#ifdef STG_PROF_LOOP
    if (lead && p.trace && blockIdx.x == 0) for (int i = 0; i < 3; ++i) p.trace[1 + 3 * 5200 + 8 + i] = mprof[i];
#endif
  } else if (warp == 0 || warp == WPROD) {
    // ===== TMA producers, tap windows (warp 0: A window + expect_tx, last warp: the W tiles of the group's taps) =====
    const bool do_a = warp == 0;
    int s = 0; uint32_t phs = 0;
    for (int t = tile0; t < p.n_tiles; t += tstep) {
      const Tile x = decode_tile(p, t);
      const int n_groups = p.res_gfirst[x.res + 1] - x.g0;
      for (int gi = 0; gi < n_groups; ++gi) {
       const int g = x.g0 + gi;
       const int nt = p.tt.g_ntaps[g], t0 = p.tt.g_tfirst[g];
       for (int chunk = 0; chunk < p.k_chunks; ++chunk) {
        mbar_wait(empty_bar(s), phs ^ 1);
        const uint32_t a_dst = smem_base + s * stage_bytes;
        if (do_a) {
          mbar_expect_tx_el(full_bar(s), (uint32_t)(p.a_boxes * p.hb * p.pack * KC * 2 + nt * b_bytes));
#pragma unroll 1
          for (int bx = 0; bx < p.a_boxes; ++bx)
            tma_load_4d_el(a_dst + bx * p.hb * p.pack * KC * 2, &tmA4.m[0], full_bar(s), x.ch0 + chunk * KC, 0,
                           (x.h0 + bx * p.hb) * p.stride + p.tt.g_off[g], x.b);
        }
#pragma unroll 1
        for (int tl = 0; tl < (do_a ? 0 : nt); ++tl) {
          if (p.cu_k) {
            tma_load_3d_el(a_dst + p.a_bytes + tl * b_bytes, &tmW, full_bar(s), 0, x.col0 + chunk * p.cu_fpc * p.cu_n,
                           p.tt.tap_w[t0 + tl]);
          } else if (!p.b_mn) {
            tma_load_3d_el(a_dst + p.a_bytes + tl * b_bytes, &tmW, full_bar(s), chunk * KC, x.col0, p.tt.tap_w[t0 + tl]);
          } else if (p.b_mn == 2) {
            tma_load_4d_el(a_dst + p.a_bytes + tl * b_bytes, &tmW, full_bar(s), 0, x.ch0 + chunk * KC, x.wcol0 / 64,
                           p.tt.tap_w[t0 + tl]);
          } else {
#pragma unroll 1
            for (int nb = 0; nb < p.bn / 64; ++nb)
              tma_load_3d_el(a_dst + p.a_bytes + tl * b_bytes + nb * 8192, &tmW, full_bar(s), x.wcol0 + nb * 64,
                             x.ch0 + chunk * KC, p.tt.tap_w[t0 + tl]);
          }
        }
        if (++s == p.stages) { s = 0; phs ^= 1u; }
       }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer, tap windows (warp-uniform control flow) =====
    const uint32_t idesc = idesc_bf16_f32(TM, p.bn, 0, p.b_mn ? 1 : 0);
    const uint32_t idesc_u = idesc_bf16_f32(TM, p.cu_k ? p.cu_n : p.bn, 0, 0);
    const int cu_ks = p.cu_k == 16 ? 0 : (p.cu_k == 32 ? 1 : 2), cu_km = (1 << cu_ks) - 1;
    const uint64_t cu_bhi = smem_desc_kmajor_narrow(0, p.cu_k ? p.cu_k * 2 : 128);
    const int cu_bq = (p.cu_n * p.cu_k * 2) >> 4;
    int s = 0, acc_i = 0; uint32_t phs = 0;
    for (int t = tile0; t < p.n_tiles; t += tstep) {
      const Tile x = decode_tile(p, t);
      if (x.n_iters == 0) continue;
      const int as = acc_i & 1, aph = (acc_i >> 1) & 1;
      mbar_wait(tmem_empty_bar(as), aph ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(as * p.acc_cols);
      int g = x.g0, chunk = 0;
      for (int it = 0; it < x.n_iters; ++it) {
        const int nt = p.tt.g_ntaps[g], t0 = p.tt.g_tfirst[g];
        mbar_wait(full_bar(s), phs);
        tc_fence_after();
        const uint32_t a_addr = smem_base + s * stage_bytes;
#pragma unroll 1
        for (int tl = 0; tl < nt; ++tl) {
          // tap = the same window, `tap_shift` h rows (x pack phase rows of 128 B) further down
          const uint64_t adesc = smem_desc_kmajor_sw128(a_addr + (uint32_t)(p.tt.tap_shift[t0 + tl] * p.pack * KC * 2));
          const uint32_t b_addr = a_addr + p.a_bytes + tl * b_bytes;
          if (p.cu_k) {   // compact groups: one MMA chain per unit of this chunk (see TcP::cu_k and the one-tap issuer)
            const uint32_t dcol = d_tmem + (uint32_t)(chunk * p.cu_fpc * p.cu_n);
            const uint64_t bu = cu_bhi | (uint64_t)((b_addr >> 4) & 0x3FFFu);
            const uint32_t acc0 = (it >= p.k_chunks || tl > 0) ? 1u : 0u;
#pragma unroll
            for (int i = 0; i < KC / 16; ++i) {
              const int q = i >> cu_ks, ks = i & cu_km;
              umma_bf16_el(dcol + (uint32_t)(q * p.cu_n), adesc + 2 * i, bu + (uint64_t)(q * cu_bq + 2 * ks), idesc_u, (acc0 | (uint32_t)(ks > 0)));
            }
            continue;
          }
          const uint64_t bdesc = p.b_mn ? smem_desc_mnmajor_sw128(b_addr, 8192, 1024) : smem_desc_kmajor_sw128(b_addr);
          const uint64_t bstep = p.b_mn ? 128 : 2;
#pragma unroll
          for (int ks = 0; ks < KC / 16; ++ks)
            umma_bf16_el(d_tmem, adesc + 2 * ks, bdesc + bstep * ks, idesc, (it > 0 || tl > 0 || ks > 0) ? 1u : 0u);
        }
        umma_commit_el(empty_bar(s));
        if (it == x.n_iters - 1) umma_commit_el(tmem_full_bar(as));
        if (++s == p.stages) { s = 0; phs ^= 1u; }
        if (++chunk == p.k_chunks) { chunk = 0; ++g; }
      }
      ++acc_i;
    }
  } else if constexpr (kStaged) {
    // ===== staged epilogue: TMEM -> registers -> swizzled smem sub-tiles -> TMA store =====
    // warps 2..5 and 6..9: two math TEAMS of 128 threads (one accumulator row per thread; sub-tile q belongs to team
    // q & 1, so every SM sub-partition has two epilogue warps to interleave - one team took ~930 clk per sub-tile,
    // instruction-latency-bound); warp 10: epilogue DMA (all TMA loads / stores of the epilogue, so their issue cost
    // stays off the math warps' critical path).
    // Hand-shake per sub-tile q through named barriers (160 = the 128 math threads of q's team + 32 DMA threads):
    //   FULL[q%3]  math arrives after writing the output slots (which implies it has consumed the input slots)
    //   FREE[q%3]  DMA arrives once the stores that last read output buffer q%3 (sub-tile q-3) have drained
    const int n_sub = p.bn / SUB;
    const int in_mask = (1 << e.in_sh) - 1;
    auto ring = [&](int q) { return p.out_ring == 2 ? (q & 1) : q % 3; };   // output-ring slot of sub-tile q
    auto in_slot = [&](int buf, int i) { return epi_base + (uint32_t)((buf * e.n_in + i) * SLOT); };
    auto out_slot = [&](int buf, int o) { return epi_base + (uint32_t)(((e.n_in << e.in_sh) + buf * e.n_out + o) * SLOT); };  // buf: q % 3
    auto bar_full = [&](int b3) { return 2 + b3; };
    auto bar_free = [&](int b3) { return 5 + b3; };
    const int my_tiles = (p.n_tiles - tile0 + tstep - 1) / tstep;
    const int q_total = my_tiles * n_sub;
    if (warp == 10) {
      // ----- epilogue DMA warp: warp-uniform control flow, elected issue (see the producer warp) -----
      if (lane == 0) {
        for (int r = 0; r < max(p.n_res, p.n_cls); ++r) {
          prefetch_tmap(&em.pre[r]); prefetch_tmap(&em.mask[r]); prefetch_tmap(&em.raw[r]);
          if (r < p.n_cls) { prefetch_tmap(&em.post[r]); prefetch_tmap(&em.act[r]); }
        }
      }
      const int rows_in = e.pair_sum ? 64 : p.mrows;                     // rows of a pre/mask/output box
      const uint32_t in_bytes = (uint32_t)((e.has_pre + e.has_mask) * rows_in * SUB * 2 + e.has_post * (rows_in >> e.post_shift) * SUB * 2);
      const int rsh = e.pair_sum ? 1 : 0;
      // iterator over (tile, sub-tile) pairs for the operand loads, which run 1 << in_sh sub-tiles ahead of the math (a load
      // takes 0.6-0.8 us to land, a team turns a sub-tile around in ~0.25 us: two in flight left the math waiting)
      int ld_t = tile0, ld_s = 0, ld_q = 0;
      Tile lx = decode_tile(p, ld_t < p.n_tiles ? ld_t : tile0);
      auto issue_loads = [&]() {
        if (e.n_in == 0 || ld_t >= p.n_tiles) return;
        const int buf = ld_q & in_mask;
        const int col = lx.col0 + ld_s * SUB;
        const int r0 = lx.h0 >> rsh;                                     // first h row of the tile in its residue class
        mbar_expect_tx_el(in_bar(buf), in_bytes);
        int i = 0;
        const int mv = lx.res + lx.cls;                                  // map variant: residue class or row class
        if (e.has_pre) tma_load_4d_el(in_slot(buf, i++), &em.pre[mv], in_bar(buf), col, 0, r0, lx.b);
        if (e.has_mask) tma_load_4d_el(in_slot(buf, i++), &em.mask[mv], in_bar(buf), col, 0, r0, lx.b);
        if (e.has_post) tma_load_4d_el(in_slot(buf, i++), &em.post[lx.cls], in_bar(buf), col, 0, r0 >> e.post_shift, lx.b);
        ++ld_q;
        if (++ld_s == n_sub) {
          ld_s = 0; ld_t += tstep;
          if (ld_t < p.n_tiles) lx = decode_tile(p, ld_t);
        }
      };
      for (int i = 0; i <= in_mask; ++i) issue_loads();
      int q = 0;
      for (int t = tile0; t < p.n_tiles; t += tstep) {
        const Tile x = decode_tile(p, t);
        const int r0_out = x.h0 >> rsh;
        for (int s = 0; s < n_sub; ++s, ++q) {
          const int obuf = ring(q);
          asm volatile("bar.sync %0, 160;" ::"r"(bar_full(obuf)) : "memory");   // output slots written, input slots consumed
          const int col = x.col0 + s * SUB;
          int o = 0;
          if (e.has_raw) tma_store_4d_el(&em.raw[x.res + x.cls], out_slot(obuf, o++), col, 0, r0_out, x.b);
          if (e.has_act) {
            tma_store_4d_el(&em.act[x.cls], out_slot(obuf, o), col, 0, r0_out, x.b);
            if (e.dup_rows) tma_store_4d_el(&em.act[x.cls], out_slot(obuf, o), col, 1, r0_out, x.b);
          }
          bulk_commit_el();
          issue_loads();                         // operands of sub-tile q + (1 << in_sh) into the input slots just consumed
          bulk_wait_read_el<1>();                // stores of sub-tile q-1 have read their slots -> its buffer is free
          __syncwarp();
          // ... which sub-tile q - 1 + out_ring will write
          if (q >= 1 && q - 1 + p.out_ring < q_total) asm volatile("bar.arrive %0, 160;" ::"r"(bar_free(ring(q - 1))) : "memory");
        }
      }
      bulk_wait_read_el<0>();   // the stores have READ their shared-memory slots; their global writes complete by the end of the grid
    } else {
      // ----- math warps -----
      const int team = (warp - 2) >> 2;                 // 0 / 1: takes the sub-tiles with q & 1 == team
      const int et = (int)(threadIdx.x - 64) & 127;     // thread of the team
      const int sub = warp & 3;            // TMEM sub-partition this warp may read
      const int m = sub * 32 + lane;       // accumulator row
      const uint32_t my_bias = bias_base + (uint32_t)team * 1024u;
      const int bias_bar = team ? 8 : 1;   // named barrier of the team (ids 2..7: FULL / FREE)
      Tracer trc(threadIdx.x == 64 ? p.trace : nullptr, 2);
      int acc_i = 0, qbase = 0;
      for (int t = tile0; t < p.n_tiles; t += tstep) {
        const Tile x = decode_tile(p, t);
        const int as = acc_i & 1, aph = (acc_i >> 1) & 1;
        trc.ev(10, t);
        // length mask: my row is (x.b, x.h0 + m), or in a row-class tail tile, which stacks seg-row slices of 128 / seg
        // samples, (x.b + m / seg, x.h0 + m % seg).  Rows past the sample or the batch are clipped by the TMA stores.
        // The select runs only in warps that hold a masked row (warp-uniform branch): the epilogue is issue-bound, and
        // most tiles of a padded batch lie wholly inside their samples.
        bool keep = true, warp_masked = false;
        if constexpr (kMask) {
          int mb = x.b, mh = x.h0 + m;
          if (p.n_cls > 1 && p.cls_tps[x.cls] == 0) { const int seg = p.cls_seg[x.cls]; mb += m / seg; mh = x.h0 + m % seg; }
          keep = mb < p.n_samples && row_kept(e, mb, mh);
          warp_masked = __any_sync(0xffffffffu, !keep);
        }
        // bias of this column tile -> smem (nobody reads the previous tile's bias any more: every thread has
        // passed its FULL arrive of the last sub-tile, which comes after its bias reads ... of ITS OWN rows only,
        // hence the 128-thread barrier below also orders the overwrite against slower warps)
        if (e.bias) {
          asm volatile("bar.sync %0, 128;" ::"r"(bias_bar) : "memory");
          for (int c = et; c < p.bn; c += 128) {
            const int col = x.col0 + c;
            const float bv = col < e.c_dst ? e.bias[col] : 0.f;
            asm volatile("st.shared.f32 [%0], %1;" ::"r"(my_bias + 4u * c), "f"(bv) : "memory");
          }
          asm volatile("bar.sync %0, 128;" ::"r"(bias_bar) : "memory");
        }
        if (x.n_iters > 0) {
          mbar_wait(tmem_full_bar(as), aph);
          tc_fence_after();
        }
        trc.ev(11, t);
        const uint32_t t_addr = tmem_base + ((uint32_t)(sub * 32) << 16) + (uint32_t)(as * p.acc_cols);
        const int r_in = e.pair_sum ? (m >> 1) : m;      // my row inside pre / mask / output sub-tiles
        const bool writer = !e.pair_sum || (lane & 1) == 0;
        // last sub-tile of this tile that belongs to my team (-1: none - possible only for one-sub-tile tiles)
        const int last_s = (((qbase + n_sub - 1) & 1) == team) ? n_sub - 1 : n_sub - 2;
        if (last_s < 0 && x.n_iters > 0) {   // nothing to read: hand the buffer back (after tmem_full, so the arrival lands in this tile's phase)
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tmem_empty_bar(as));
        }
#pragma unroll 1
        for (int s = (qbase & 1) == team ? 0 : 1; s < n_sub; s += 2) {
          const int q = qbase + s;
          const int buf = q & in_mask;
          float v[32];
          if (x.n_iters > 0) {
            tmem_ld16(t_addr + (uint32_t)(s * SUB), *reinterpret_cast<float(*)[16]>(&v[0]));
            tmem_ld16(t_addr + (uint32_t)(s * SUB + 16), *reinterpret_cast<float(*)[16]>(&v[16]));
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = 0.f;
          }
          if (s == last_s && x.n_iters > 0) {  // my team's part of the accumulator is read: hand the TMEM buffer back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tmem_empty_bar(as));
          }
          if (e.bias) {
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              float4 bq;
              asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(bq.x), "=f"(bq.y), "=f"(bq.z), "=f"(bq.w)
                           : "r"(my_bias + 4u * (s * SUB + i)) : "memory");
              v[i] += bq.x; v[i + 1] += bq.y; v[i + 2] += bq.z; v[i + 3] += bq.w;
            }
          }
          if (e.pair_sum) {
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], 1);
          }
          trc.ev(20, s);
          if (e.n_in > 0) {
            mbar_wait(in_bar(buf), (q >> e.in_sh) & 1);
            trc.ev(21, s);
            int i = 0;
            if (e.has_pre) {
              const uint32_t sl = in_slot(buf, i++);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                float t8[8]; unpack8(lds128(sl + sw64(r_in, j)), t8);
#pragma unroll
                for (int u = 0; u < 8; ++u) v[8 * j + u] += t8[u];
              }
            }
            if (e.has_mask) {
              const uint32_t sl = in_slot(buf, i++);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                float t8[8]; unpack8(lds128(sl + sw64(r_in, j)), t8);
#pragma unroll
                for (int u = 0; u < 8; ++u) v[8 * j + u] *= (t8[u] > 0.f ? 1.f : e.mask_slope);
              }
            }
            if (e.has_post) {
              const uint32_t sl = in_slot(buf, i++);
              const int rp = r_in >> e.post_shift;
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                float t8[8]; unpack8(lds128(sl + sw64(rp, j)), t8);
#pragma unroll
                for (int u = 0; u < 8; ++u) v[8 * j + u] += t8[u];
              }
            }
          }
          const int obuf = ring(q);
          if (q >= p.out_ring) asm volatile("bar.sync %0, 160;" ::"r"(bar_free(obuf)) : "memory");  // stores of sub-tile q - out_ring drained
          trc.ev(23, s);
          if (warp_masked) {
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = keep ? v[i] : 0.f;
          }
          if (writer) {
            int o = 0;
            if (e.has_raw) {
              const uint32_t sl = out_slot(obuf, o++);
#pragma unroll
              for (int j = 0; j < 4; ++j) sts128(sl + sw64(r_in, j), pack8(&v[8 * j]));
            }
            if (e.has_act) {
              const uint32_t sl = out_slot(obuf, o++);
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], e.act_slope * v[i]);
#pragma unroll
              for (int j = 0; j < 4; ++j) sts128(sl + sw64(r_in, j), pack8(&v[8 * j]));
            }
          }
          fence_proxy_async();
          asm volatile("bar.arrive %0, 160;" ::"r"(bar_full(obuf)) : "memory");
          trc.ev(12, s);
        }
        qbase += n_sub;
        if (x.n_iters > 0) ++acc_i;
      }
    }
  } else {
    // ===== direct epilogue =====
    const int ew = warp - 2;
    const int sub = warp & 3;        // TMEM sub-partition this warp may read
    const int half = ew >> 2;        // column half of the tile
    // columns of this warp: chunks of 16, split between the two warps of a sub-partition
    const int n_chunks = p.bn / 16;
    const int c_lo = (half == 0) ? 0 : (n_chunks + 1) / 2, c_hi = (half == 0) ? (n_chunks + 1) / 2 : n_chunks;
    int acc_i = 0;
    for (int t = tile0; t < p.n_tiles; t += tstep) {
      const Tile x = decode_tile(p, t);
      const int as = acc_i & 1, aph = (acc_i >> 1) & 1;
      const int arow = out_row(p, x, sub * 32 + lane);  // output row of this thread (before pair_sum)
      const bool row_ok = arow >= 0 && (!e.pair_sum || (lane & 1) == 0);
      const int orow = e.pair_sum ? (arow >> 1) : arow;
      const bool keep = !kMask || (row_ok && row_kept(e, x.b, orow));
      EpiIn inA, inB;
      if (c_lo < c_hi) epi_load(e, x.b, orow, x.col0 + c_lo * 16, row_ok, inA);
      if (x.n_iters > 0) {
        mbar_wait(tmem_full_bar(as), aph);
        tc_fence_after();
      }
      const uint32_t t_addr = tmem_base + ((uint32_t)(sub * 32) << 16) + (uint32_t)(as * p.acc_cols);
      auto process = [&](int c, const EpiIn& in) {
        float v[16];
        if (x.n_iters > 0) {
          tmem_ld16(t_addr + (uint32_t)(c * 16), v);
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = 0.f;
        }
        const int col = x.col0 + c * 16;
        if (col >= e.c_dst) return;  // warp-uniform
        if (e.bias) {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] += (col + i < e.c_dst) ? e.bias[col + i] : 0.f;
        }
        if (e.pair_sum) {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], 1);
        }
        if (row_ok) epi_store(e, x.b, orow, col, v, in, keep);
      };
#pragma unroll 1
      for (int c = c_lo; c < c_hi; c += 2) {
        if (c + 1 < c_hi) epi_load(e, x.b, orow, x.col0 + (c + 1) * 16, row_ok, inB);
        process(c, inA);
        if (c + 1 < c_hi) {
          if (c + 2 < c_hi) epi_load(e, x.b, orow, x.col0 + (c + 2) * 16, row_ok, inA);
          process(c + 1, inB);
        }
      }
      if (x.n_iters > 0) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tmem_empty_bar(as));
        ++acc_i;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  life_ev(p.trace, 33);
}

}  // namespace

PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(ptr);
  }
  return fn;
}

int make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box, const uint32_t* elem_strides, int swizzle_bytes) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) { set_cuda_error(cudaErrorNotSupported, "cuTensorMapEncodeTiled entry point"); return STG_ECUDA; }
  cuuint64_t gd[5]; cuuint64_t gs[4]; cuuint32_t bx[5]; cuuint32_t es[5];
  for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; es[i] = elem_strides ? elem_strides[i] : 1; }
  for (int i = 0; i + 1 < rank; ++i) gs[i] = strides_bytes[i];
  const CUtensorMapSwizzle sw = swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                              : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B;
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_cuda_error(cudaErrorInvalidValue, "cuTensorMapEncodeTiled failed");
    return STG_ECUDA;
  }
  return STG_OK;
}

static int sm_count() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n < 1)
      n = 148;
  }
  return (g_sm_limit > 0 && g_sm_limit < n) ? g_sm_limit : n;   // stg_set_sm_limit: leave SMs to a concurrent communicator
}

// Cost model for the column-tile width.  One CTA per SM walks ceil(tiles / SMs) tiles; a tile's main loop costs
// n_stages x (max(2 bn, 200) + 60) clk (the MMAs of a 64-deep stage against the producers' issue floor), epilogues hide
// behind the next tile's main loop except the last one (bn / 32 sub-tiles of ~200 clk with two teams).  Picks the
// multiple of `step` dividing cd_g with the smallest makespan (0: none divides); ties go to the wider tile.
static int pick_bn_model(int cd_g, int groups, int64_t row_tiles, int n_stages, int step) {
  int best = 0;
  double best_t = 0;
  for (int bn = 256; bn >= step; bn -= step) {
    if (cd_g % bn) continue;
    const int64_t tiles = row_tiles * (cd_g / bn) * groups;
    const double waves = (double)((tiles + sm_count() - 1) / sm_count());
    const double mma = 2.0 * bn > 200.0 ? 2.0 * bn : 200.0;
    const double stage = mma + 60.0;   // + barrier round trip / commit latency per stage
    const double epi = (bn / 32.0) * 200.0;
    const double t = waves * n_stages * stage + epi;
    if (best == 0 || t < best_t * 0.999) { best = bn; best_t = t; }
  }
  return best;
}

static int pick_bn(int cd_g, int groups, int64_t row_tiles, int n_stages) {
  if (groups == 1 && (cd_g % 16) != 0) return cd_g <= 16 ? 16 : (cd_g <= 128 ? ((cd_g + 15) / 16) * 16 : 128);
  const int b = pick_bn_model(cd_g, groups, row_tiles, n_stages, 32);   // multiples of 32: staged-epilogue sub-tiles
  if (b > 0) return b;
  // no multiple of 32 divides cd_g (cd_g = 16 mod 32): the widest dividing multiple of 16, narrower (down to 128) while
  // the launch has fewer than min_tiles tiles
  constexpr int min_tiles = 128;
  int best = 0;
  for (int bn = 256; bn >= 16; bn -= 16) {
    if (cd_g % bn) continue;
    if (best != 0 && bn < 128) break;              // narrower than 128 only when nothing wider divides
    best = bn;
    if (row_tiles * (cd_g / bn) * groups >= min_tiles) break;
  }
  return best;
}

// data-gradient column tiles are whole 64-channel boxes of the forward pack
static int pick_bn_mn(int cd_g, int groups, int64_t row_tiles, int n_stages) {
  if (cd_g % 64 != 0) return groups == 1 ? (cd_g <= 64 ? 64 : 128) : 0;
  return pick_bn_model(cd_g, groups, row_tiles, n_stages, 64);   // 64 divides cd_g: never 0
}

// Row classes of a sample of t_dst rows (TcP::n_cls): whole 128-row tiles, then a binary tail (64 / 32 / 16 / 8 rows) whose
// tiles gather the same row slice of 128 / seg samples; at most 4 classes - the last one covers whatever is left.
// seg: rows per sample, h0: first row, tps: tiles per sample (0: one tile per 128 / seg samples).
struct RowCls { int seg, h0, tps; };
static int row_classes(int t_dst, RowCls* rc) {
  int n = 0;
  const int full = t_dst / TM;
  int r = t_dst % TM, h = full * TM;
  if (full > 0) rc[n++] = RowCls{TM, 0, full};
  while (r > 0) {
    int seg = 8;
    while (seg * 2 <= r) seg *= 2;                               // largest power of two <= r (at least 8)
    if (n == 3 || r < 8) { seg = 8; while (seg < r) seg *= 2; }  // last slot: one class covers what is left
    rc[n++] = seg >= TM ? RowCls{TM, h, 1} : RowCls{seg, h, 0};
    h += seg; r -= seg < r ? seg : r;
  }
  return n;
}
int debug_row_classes(int t_dst, int* out) {   // out[3 * c + {0, 1, 2}] = seg, h0, tps
  RowCls rc[4];
  const int n = row_classes(t_dst, rc);
  for (int c = 0; c < n; ++c) { out[3 * c] = rc[c].seg; out[3 * c + 1] = rc[c].h0; out[3 * c + 2] = rc[c].tps; }
  return n;
}

static void tile_geometry(const StgConv* d, int* pack, int* nh, int* n_res, int* tiles_m) {
  *pack = d->phases;
  *nh = TM / d->phases;
  *n_res = (d->transposed && d->stride > 1) ? d->stride : 1;
  *tiles_m = ceil_div(ceil_div(d->t_dst, *n_res), *nh);
}

// Compact groups (TcP::cu_k): groups of ku in {16, 32, 64} source channels and nu % 16 == 0 destination channels.  A CTA
// tile covers f groups, the smallest divisor of `groups` that makes whole 64-channel K chunks on the source side and whole
// 64-column blocks on the destination side (the geometry the block-diagonal packs had); 0 = not possible.
static int compact_merge(int ku, int nu, int groups) {
  if ((ku != 16 && ku != 32 && ku != 64) || (nu % 16) != 0) return 0;
  for (int f = 1; f <= groups; ++f) {
    if (groups % f) continue;
    if ((ku * f) % KC == 0 && (nu * f) % KC == 0) return nu * f <= 256 ? f : 0;
  }
  return 0;
}

bool conv_tc_supported(const StgConv* d) {
  if (d->dtype != STG_BF16) return false;
  if (d->k > STG_MAX_TAPS || d->k < 1) return false;
  if ((d->c_src % 8) != 0) return false;                 // 16-byte global strides for TMA
  if (d->phases > 64) return false;
  if (d->groups > 1) {
    if (((d->c_dst / d->groups) % 16) != 0) return false;
    if ((d->c_src / d->groups) % KC) {                   // narrow groups: compact-group path (K-major W only)
      if (d->transposed && d->w_fwd_pack) return false;
      if (compact_merge(d->c_src / d->groups, d->c_dst / d->groups, d->groups) == 0) return false;
    } else if (d->transposed && !d->w_fwd_pack && d->c_src / d->groups != KC) {
      return false;                                      // K-major data-gradient packs of wide groups: not needed, not built
    }
  }
  // data-gradients read the forward pack as an MN-major B operand (w_fwd_pack) or - grouped convs - a K-major
  // data-gradient pack wd [k][c_in][c_out/g] through the same code path as a forward convolution
  if (d->transposed && !d->w_fwd_pack && d->groups == 1) return false;
  if (d->transposed && ((d->c_dst / d->groups) % 8) != 0) return false;
  if (d->transposed && d->w_fwd_pack && d->groups > 1 && ((d->c_dst / d->groups) % 64) != 0) return false;
  if (d->transposed && d->stride > MAX_RES) return false;
  if (d->transposed && d->stride > 1 && d->pair_sum) return false;
  if (!d->transposed && d->stride > 4) return false;
  if (!d->transposed && d->stride > 2 && d->phases > 1 && (TM / d->phases) * d->stride > 256) return false;
  if ((d->pair_sum || d->dup_rows || d->post_shift) && d->phases != 1) return false;
  if (d->pair_sum && (d->t_dst & 1)) return false;
  if (d->add_pre == nullptr && d->mask == nullptr && d->add_post == nullptr && d->y_raw == nullptr && d->y_act == nullptr)
    return false;
  return true;
}

int tc_pack_groups(int c_in, int c_out, int groups) {
  if (groups <= 1) return 1;
  const int cin_g = c_in / groups, cout_g = c_out / groups;
  // Units of the compact-group path: the smallest merge m | groups whose merged group has 16 / 32 / 64 (or a multiple of 64)
  // channels on BOTH sides - the forward conv contracts over the input side, the data-gradient over the output side, and
  // an MMA K step is 16 channels.  The packs are block-diagonal only inside a unit (m > 1: groups of 8 channels).
  auto side_ok = [](int c) { return c == 16 || c == 32 || (c % KC) == 0; };
  for (int m = 1; m <= groups; ++m) {
    if (groups % m) continue;
    if (side_ok(cin_g * m) && side_ok(cout_g * m)) return groups / m;
  }
  return groups;
}

// tensor map of an epilogue operand / output for residue class `res` of `n_res`: [B][T][P][C] seen as
// (C, P, h', B) with h = h'*n_res + res; box = (32, pack, box_h, 1).  `dup`: y_act as [B][T][2][C] -> (C, 2, h, B).
static int epi_map(CUtensorMap* m, const void* base, int C, int P, int T, int B, int res, int n_res, int pack, int box_h,
                   bool dup, int box_b = 1) {
  if (dup) {
    const uint64_t dims[4] = {(uint64_t)C, 2, (uint64_t)T, (uint64_t)B};
    const uint64_t strides[3] = {(uint64_t)C * 2, (uint64_t)C * 4, (uint64_t)T * C * 4};
    const uint32_t box[4] = {SUB, 1, (uint32_t)box_h, (uint32_t)box_b};
    return make_tmap_bf16(m, base, 4, dims, strides, box, nullptr, 64);
  }
  const int h_ext = (T - res + n_res - 1) / n_res;
  const uint64_t dims[4] = {(uint64_t)C, (uint64_t)P, (uint64_t)h_ext, (uint64_t)B};
  const uint64_t strides[3] = {(uint64_t)C * 2, (uint64_t)n_res * P * C * 2, (uint64_t)T * P * C * 2};
  const uint32_t box[4] = {SUB, (uint32_t)pack, (uint32_t)box_h, (uint32_t)box_b};
  const bf16* b0 = static_cast<const bf16*>(base) + (int64_t)res * P * C;
  return make_tmap_bf16(m, b0, 4, dims, strides, box, nullptr, 64);
}

static long long* g_trace = nullptr;
void conv_tc_set_trace(long long* buf) { g_trace = buf; }
static int* g_plan_out = nullptr;   // stg_debug_conv_plan: conv_tc() fills this with its plan and returns before touching the device
int conv_tc_plan(const StgConv* d, int* out) {
  g_plan_out = out;
  const int r = conv_tc(d, nullptr);
  g_plan_out = nullptr;
  return r;
}

int conv_tc(const StgConv* d, cudaStream_t s, const int32_t* valid_units, int rows_per_unit) {
  if (!conv_tc_supported(d)) return STG_EUNSUPPORTED;
  TcP p;
  p.trace = g_trace;
  p.phases = d->phases; p.t_dst = d->t_dst; p.stride = d->transposed ? 1 : d->stride;
  p.cs_g = d->c_src / d->groups; p.cd_g = d->c_dst / d->groups;
  int tile_groups = d->groups;     // groups as the tile walk sees them
  p.cu_k = p.cu_n = p.cu_fpc = 0;
  if (d->groups > 1 && (p.cs_g % KC) != 0) {   // compact groups: a tile covers f units (see TcP::cu_k)
    const int f = compact_merge(p.cs_g, p.cd_g, d->groups);
    if (f == 0) return STG_EUNSUPPORTED;
    p.cu_k = p.cs_g; p.cu_n = p.cd_g; p.cu_fpc = KC / p.cs_g;
    p.cs_g *= f; p.cd_g *= f; tile_groups = d->groups / f;
  }
  p.k_chunks = ceil_div(p.cs_g, KC);
  tile_geometry(d, &p.pack, &p.nh, &p.n_res, &p.tiles_m);
  p.mrows = p.nh * p.pack;
  p.b_mn = (d->transposed && d->w_fwd_pack) ? 1 : 0;
  // stages of one tile: taps (of one residue class) x 64-channel chunks
  const int n_stages_est = ceil_div(d->k, p.n_res) * p.k_chunks;
  p.bn = p.cu_k ? p.cd_g   // compact groups: a column tile is the whole merged group
       : p.b_mn ? pick_bn_mn(p.cd_g, tile_groups, (int64_t)d->n_samples * p.n_res * p.tiles_m, n_stages_est)
                : pick_bn(p.cd_g, tile_groups, (int64_t)d->n_samples * p.n_res * p.tiles_m, n_stages_est);
  if (p.bn <= 0) return STG_EUNSUPPORTED;
  p.tmem_cols = 512;  // two accumulator buffers ACC_COLS apart
  // ---- taps per residue class, as (source offset, weight index)
  struct Tap { int off, w; };
  Tap taps[MAX_RES][STG_MAX_TAPS]; int ntap[MAX_RES];
  if (p.n_res > 1) {
    for (int r = 0; r < p.n_res; ++r) {
      ntap[r] = 0;
      for (int j = 0; j < d->k; ++j) {
        const int num = r + d->pad - j * d->dilation;
        if (((num % d->stride) + d->stride) % d->stride != 0) continue;
        taps[r][ntap[r]++] = Tap{(num >= 0) ? num / d->stride : -((-num) / d->stride), j};  // exact division
      }
    }
  } else {
    ntap[0] = d->k;
    for (int j = 0; j < d->k; ++j) taps[0][j] = Tap{d->transposed ? (d->pad - j * d->dilation) : (j * d->dilation - d->pad), j};
  }
  TcEpi& e = p.e;
  const int rows_per_phase = d->pair_sum ? d->t_dst / 2 : d->t_dst;
  e.rows = rows_per_phase * d->phases; e.c_dst = d->c_dst;
  e.post_shift = d->post_shift; e.mask_mode = d->mask_mode; e.act = d->act; e.dup_rows = d->dup_rows;
  e.out_f32 = d->out_f32; e.pair_sum = d->pair_sum; e.bias = d->bias;
  e.add_pre = static_cast<const bf16*>(d->add_pre); e.mask = static_cast<const bf16*>(d->mask);
  e.add_post = static_cast<const bf16*>(d->add_post); e.y_raw = d->y_raw; e.y_act = d->y_act;
  e.has_pre = d->add_pre != nullptr; e.has_mask = d->mask != nullptr; e.has_post = d->add_post != nullptr;
  e.has_raw = d->y_raw != nullptr; e.has_act = d->y_act != nullptr;
  e.valid_units = valid_units; e.rows_per_unit = rows_per_unit;
  e.n_in = e.has_pre + e.has_mask + e.has_post; e.n_out = e.has_raw + e.has_act;
  e.act_slope = d->act == STG_ACT_RELU ? 0.f : (d->act == STG_ACT_LEAKY ? 0.1f : 1.f);
  e.mask_slope = d->mask_mode == STG_ACT_RELU ? 0.f : (d->mask_mode == STG_ACT_LEAKY ? 0.1f : 1.f);
  const bool staged = !d->out_f32 && d->act != STG_ACT_TANH && d->mask_mode != STG_ACT_TANH && (d->c_dst % 8) == 0 &&
                      p.n_res <= MAX_STAGED_RES && (p.n_res == 1 || (!d->add_post && !d->y_act)) && (p.bn % SUB) == 0 &&
                      (!d->post_shift || (rows_per_phase % 2) == 0);

  // ---- row classes (see TcP::n_cls): 128-row tiles + a binary tail whose tiles gather several samples
  RowCls rc[4];
  int n_rc = 0;
  int64_t cls_tiles = 0;
  if (staged && d->phases == 1 && p.n_res == 1 && d->stride == 1) {
    n_rc = row_classes(d->t_dst, rc);
    for (int c = 0; c < n_rc; ++c)
      cls_tiles += rc[c].tps > 0 ? (int64_t)d->n_samples * rc[c].tps : ceil_div(d->n_samples, TM / rc[c].seg);
    const int64_t classic = (int64_t)d->n_samples * p.tiles_m;
    if (n_rc < 2 || cls_tiles >= classic) n_rc = 0;
    if (n_rc) {   // the column tile is chosen for the new tile count
      const int bn2 = p.cu_k ? p.cd_g : p.b_mn ? pick_bn_mn(p.cd_g, tile_groups, cls_tiles, n_stages_est) : pick_bn(p.cd_g, tile_groups, cls_tiles, n_stages_est);
      if (bn2 > 0 && (bn2 % SUB) == 0) p.bn = bn2; else n_rc = 0;
    }
  }

  // ---- tap groups (A windows) and pipeline depth.  Taps of a group must lie on one row lattice of the strided
  // A box (same offset mod stride) and close enough for the window to fit its boxes; candidates: <= ng taps per
  // group, pick the ng with the least shared-memory ingest per tile among those that leave >= 3 (else 2) stages.
  p.n_samples = d->n_samples;
  const int b_bytes = p.cu_k ? p.cu_fpc * p.cu_n * p.cu_k * 2 : p.bn * KC * 2;
  // epilogue-operand ring: as deep as a column tile has sub-tiles (<= 8) while the main loop keeps >= 4 stages of the
  // one-tap-per-stage plan (or all the stages a tile has), else 4, else 2
  // shared memory for main-loop stages + epilogue staging (the launch adds ~1.5 KB of alignment slack, barriers and tap tables;
  // the SM gives one CTA 227 KB)
  constexpr int smem_budget = 224 * 1024;
  e.in_sh = 1;
  if (staged && e.n_in > 0) {
    const int stage1 = TM * KC * 2 + (p.cu_k ? p.cu_fpc * p.cu_n * p.cu_k * 2 : p.bn * KC * 2);
    const int want = n_stages_est < 4 ? n_stages_est : 4;
    for (int sh = 3; sh >= 2; --sh) {
      if ((1 << (sh - 1)) >= p.bn / SUB) continue;                       // the ring need not exceed the tile
      const int epi = ((e.n_in << sh) + 3 * e.n_out) * SLOT + 2048;
      if ((smem_budget - epi) / stage1 >= want) { e.in_sh = sh; break; }
    }
  }
  int epi_bytes = staged ? ((e.n_in << e.in_sh) + 3 * e.n_out) * SLOT + 2048 : 0;
  int avail = smem_budget - epi_bytes;
  // Two CTAs per SM: the staged single-CTA kernel fits twice on an SM when a CTA stays below ~113 KB of shared memory and
  // 256 TMEM columns (bn <= 128: two accumulator buffers 128 columns apart; epilogue rings two deep).  Measured
  // (tools/conv_bench.py, profiles/r2_occ2_conv_bench.txt): the halved pipelines cost the dense layers 5-35 % (the bytes
  // in flight per SM stay the same, the rings get shallower), but the issue-bound data-gradients of the compact-group layers
  // gain 10-25 % (two issuing threads per SM) and grouped layers whose tiles hold few rows (1024 channels in 16 groups,
  // T = 25: 256 mostly empty tiles) run in one wave instead of two (2.0x).  So: those two classes only.
  const bool occ2_class = (p.cu_k != 0 && d->transposed) || (tile_groups > 1 && p.cu_k == 0 && p.bn <= 64);
  bool occ2 = false;
  if (occ2_class && staged && p.bn <= 128) {
    const int epi2 = ((e.n_in << 1) + 2 * e.n_out) * SLOT + 2048;
    const int avail2 = 110 * 1024 - epi2;
    if (avail2 / (TM * KC * 2 + b_bytes) >= 2) { occ2 = true; e.in_sh = 1; epi_bytes = epi2; avail = avail2; }
  }
  p.out_ring = occ2 ? 2 : 3; p.acc_cols = occ2 ? 128 : ACC_COLS; p.tmem_cols = occ2 ? 256 : 512;
  struct Plan { int ng, stages, hb, a_boxes, a_bytes, n_groups; long long traffic; bool ok; };
  auto build = [&](int ng, TcP* out) {
    Plan pl{ng, 0, 0, 0, 0, 0, 0, false};
    int n_groups = 0, n_taps_out = 0, max_shift = 0;
    for (int r = 0; r < p.n_res; ++r) {
      if (out) out->res_gfirst[r] = n_groups;
      bool used[STG_MAX_TAPS] = {false};
      for (int i = 0; i < ntap[r]; ++i) {
        if (used[i]) continue;
        // new group seeded by tap i: later taps of the same lattice, sorted by offset implicitly (offsets are monotone in j)
        int lo = taps[r][i].off, members[STG_MAX_TAPS], nm = 0;
        for (int j2 = i; j2 < ntap[r] && nm < ng; ++j2) {
          if (used[j2]) continue;
          const int diff = taps[r][j2].off - taps[r][i].off;
          if (diff % p.stride != 0) continue;
          int new_lo = taps[r][j2].off < lo ? taps[r][j2].off : lo, hi = taps[r][i].off;
          for (int q = 0; q < nm; ++q) { const int o = taps[r][members[q]].off; if (o > hi) hi = o; if (o < new_lo) new_lo = o; }
          if (taps[r][j2].off > hi) hi = taps[r][j2].off;
          if ((hi - new_lo) / p.stride > 128) continue;   // window would not fit
          members[nm++] = j2; used[j2] = true; lo = new_lo;
        }
        for (int q = 0; q < nm; ++q) {
          const int sh = (taps[r][members[q]].off - lo) / p.stride;
          if (sh > max_shift) max_shift = sh;
          if (out) { out->tt.tap_shift[n_taps_out] = (short)sh; out->tt.tap_w[n_taps_out] = (unsigned char)taps[r][members[q]].w; }
          ++n_taps_out;
        }
        if (out) { out->tt.g_off[n_groups] = (short)lo; out->tt.g_tfirst[n_groups] = (unsigned char)(n_taps_out - nm); out->tt.g_ntaps[n_groups] = (unsigned char)nm; }
        ++n_groups;
      }
    }
    if (out) out->res_gfirst[p.n_res] = n_groups;
    // window boxes: a_boxes boxes of hb h rows (hb * stride <= 256; box starts on 8-row swizzle boundaries)
    const int win_h = p.nh + max_shift;
    int a_boxes = ceil_div(win_h * p.stride, 256), hb = ceil_div(win_h, a_boxes);
    if (a_boxes > 1) {
      const int align = 8 / (p.pack >= 8 ? 8 : (8 % p.pack == 0 ? p.pack : 1));   // hb * pack % 8 == 0
      hb = ceil_div(hb, align) * align;
      if ((hb * p.pack) % 8 != 0) return pl;
      while (hb * p.stride > 256) { ++a_boxes; hb = ceil_div(ceil_div(win_h, a_boxes), align) * align; }
    }
    if (hb * p.stride > 256 || p.pack > 256) return pl;
    int a_rows = a_boxes * hb * p.pack;
    if (a_rows < TM + max_shift * p.pack) a_rows = TM + max_shift * p.pack;   // the MMA always reads 128 rows from the shift
    pl.hb = hb; pl.a_boxes = a_boxes; pl.a_bytes = ceil_div(a_rows * KC * 2, 1024) * 1024; pl.n_groups = n_groups;
    const int stage_bytes = pl.a_bytes + ng * b_bytes;
    pl.stages = avail / stage_bytes;
    if (pl.stages > MAX_STAGES) pl.stages = MAX_STAGES;
    pl.traffic = (long long)n_groups * (a_boxes * hb * p.pack * KC * 2) + (long long)n_taps_out * b_bytes;
    pl.ok = pl.stages >= 2;
    return pl;
  };
  Plan best{0, 0, 0, 0, 0, 0, 0, false};
  const long long base_traffic = build(1, nullptr).traffic;
  const int cands[] = {1, 2, 3, 4, 5, 6, 8, 10};
  for (int ci = 0; ci < 8; ++ci) {
    const int ng = cands[ci];
    if (ng > d->k && ng != 1) continue;
    Plan pl = build(ng, nullptr);
    if (!pl.ok) continue;
    if (!best.ok) { best = pl; continue; }           // ng = 1 comes first: the baseline
    // a window plan replaces the one-tap-per-stage baseline only if it still pipelines (>= 3 stages) and moves
    // at least 35 % fewer bytes: for k = 3 the saving is ~25 % and the coarser stages cost more than that
    if (pl.stages >= 3 && pl.traffic * 100 <= base_traffic * 65 && pl.traffic < best.traffic) best = pl;
  }
  if (!best.ok) return STG_EUNSUPPORTED;
  if (n_rc && best.ng != 1) n_rc = 0;   // tap windows load (128 + shift)-row boxes of one sample: classic tiles
  p.n_cls = n_rc ? n_rc : 1;
  p.cls_mt0[0] = 0;
  for (int c = 0; c < p.n_cls; ++c) {
    p.cls_seg[c] = n_rc ? rc[c].seg : TM; p.cls_h0[c] = n_rc ? rc[c].h0 : 0; p.cls_tps[c] = n_rc ? rc[c].tps : p.tiles_m;
    p.cls_mt0[c + 1] = p.cls_mt0[c] + (n_rc ? (rc[c].tps > 0 ? d->n_samples * rc[c].tps : ceil_div(d->n_samples, TM / rc[c].seg)) : 0);
  }
  build(best.ng, &p);
  p.hb = best.hb; p.a_boxes = best.a_boxes; p.a_bytes = best.a_bytes; p.max_ntaps = best.ng; p.stages = best.stages;
  const int stage_bytes = p.a_bytes + p.max_ntaps * b_bytes;
  const size_t smem = (size_t)p.stages * stage_bytes + epi_bytes + 1024 /*align slack*/ + 8 * (2 * MAX_STAGES + 16) + sizeof(TapTables) + 16;
  if (g_plan_out) {   // host-only query (no tensor maps, no launch): see stg_debug_conv_plan in include/stegan_b200.h
    const int tiles_n = ceil_div(d->c_dst, p.bn);
    const int64_t nt = n_rc ? (int64_t)p.cls_mt0[p.n_cls] * tiles_n : (int64_t)d->n_samples * p.n_res * p.tiles_m * tiles_n;
    const int64_t slots = (occ2 ? 2 : 1) * sm_count();
    int* o = g_plan_out;
    o[0] = p.bn; o[1] = staged; o[2] = p.max_ntaps; o[3] = p.stages; o[4] = (int)smem; o[5] = occ2; o[6] = p.n_cls;
    o[7] = (int)nt; o[8] = (int)(nt < slots ? nt : slots); o[9] = p.cu_k; o[10] = p.k_chunks; o[11] = p.tmem_cols;
    o[12] = staged && e.n_in > 0 ? 1 << e.in_sh : 0; o[13] = p.out_ring; o[14] = p.n_res;
    return STG_OK;
  }

  CUtensorMap tmW;
  TmA4 tmA;
  EpiMaps em;
  memset(&em, 0, sizeof(em));
  memset(&tmA, 0, sizeof(tmA));
  for (int c = 0; c < p.n_cls; ++c) {
    const uint64_t C = d->c_src, P = d->phases, T = d->t_src, B = d->n_samples;
    const uint64_t dims[4] = {C, P, T, B};
    const uint64_t strides[3] = {C * 2, P * C * 2, T * P * C * 2};
    // row class c: seg rows of TM / seg consecutive samples (classic tiles: hb rows of one sample)
    const uint32_t box_h = n_rc ? (uint32_t)rc[c].seg : (uint32_t)(p.hb * p.stride);
    const uint32_t box_b = n_rc && rc[c].tps == 0 ? (uint32_t)(TM / rc[c].seg) : 1u;
    const uint32_t box[4] = {(uint32_t)KC, (uint32_t)p.pack, box_h, box_b};
    const uint32_t es[4] = {1, 1, (uint32_t)p.stride, 1};
    int r = make_tmap_bf16(&tmA.m[c], d->src, 4, dims, strides, box, es);
    if (r) return r;
  }
  if (p.cu_k) {
    // compact pack [k][c_dst][cu_k]: rows of 32 / 64 / 128 bytes, box = the rows of one chunk's units, matching swizzle
    const uint64_t C = p.cu_k, N = d->c_dst, K = d->k;
    const uint64_t dims[3] = {C, N, K};
    const uint64_t strides[2] = {C * 2, N * C * 2};
    const uint32_t box[3] = {(uint32_t)p.cu_k, (uint32_t)(p.cu_fpc * p.cu_n), 1};
    int r = make_tmap_bf16(&tmW, d->w, 3, dims, strides, box, nullptr, p.cu_k * 2);
    if (r) return r;
  } else if (!p.b_mn) {
    const uint64_t C = p.cs_g, N = d->c_dst, K = d->k;
    const uint64_t dims[3] = {C, N, K};
    const uint64_t strides[2] = {C * 2, N * C * 2};
    const uint32_t box[3] = {(uint32_t)KC, (uint32_t)p.bn, 1};
    int r = make_tmap_bf16(&tmW, d->w, 3, dims, strides, box, nullptr);
    if (r) return r;
  } else if (p.cd_g % 64 == 0) {
    // forward pack [k][c_src][cd_g] seen as (64 inner, source-channel row, cd_g/64, tap): ONE box delivers the whole
    // MN-major tile [bn/64][64 rows][64] (one TMA instruction per stage instead of bn/64 - each costs ~0.12 us to issue)
    p.b_mn = 2;
    const uint64_t N = p.cd_g, R = d->c_src, K = d->k;
    const uint64_t dims[4] = {64, R, N / 64, K};
    const uint64_t strides[3] = {N * 2, 128, R * N * 2};
    const uint32_t box[4] = {64, (uint32_t)KC, (uint32_t)(p.bn / 64), 1};
    int r = make_tmap_bf16(&tmW, d->w, 4, dims, strides, box, nullptr);
    if (r) return r;
  } else {  // (destination channel within group, source channel row, tap); bn/64 boxes per tile, partial last box zero-filled
    const uint64_t N = p.cd_g, R = d->c_src, K = d->k;
    const uint64_t dims[3] = {N, R, K};
    const uint64_t strides[2] = {N * 2, R * N * 2};
    const uint32_t box[3] = {64, (uint32_t)KC, 1};
    int r = make_tmap_bf16(&tmW, d->w, 3, dims, strides, box, nullptr);
    if (r) return r;
  }
  if (staged) {
    const int box_h = d->pair_sum ? 64 : p.nh;          // h rows of one box (x pack phases = rows of the sub-tile)
    const int t_rows = rows_per_phase;                  // output rows per phase (after pair_sum)
    int r = 0;
    for (int res = 0; res < (n_rc ? 0 : p.n_res); ++res) {
      if (e.has_pre) r |= epi_map(&em.pre[res], d->add_pre, d->c_dst, d->phases, t_rows, d->n_samples, res, p.n_res, p.pack, box_h, false);
      if (e.has_mask) r |= epi_map(&em.mask[res], d->mask, d->c_dst, d->phases, t_rows, d->n_samples, res, p.n_res, p.pack, box_h, false);
      if (e.has_raw) r |= epi_map(&em.raw[res], d->y_raw, d->c_dst, d->phases, t_rows, d->n_samples, res, p.n_res, p.pack, box_h, false);
    }
    if (!n_rc) {
      if (e.has_post) r |= epi_map(&em.post[0], d->add_post, d->c_dst, d->phases, t_rows >> d->post_shift, d->n_samples, 0, 1, p.pack, box_h >> d->post_shift, false);
      if (e.has_act) r |= epi_map(&em.act[0], d->y_act, d->c_dst, d->phases, t_rows, d->n_samples, 0, 1, p.pack, box_h, d->dup_rows != 0);
    }
    for (int c = 0; c < n_rc; ++c) {   // row classes: boxes of (seg [/ 2] rows) x (TM / seg samples)
      const int bh = d->pair_sum ? rc[c].seg / 2 : rc[c].seg, bb = rc[c].tps == 0 ? TM / rc[c].seg : 1;
      if (e.has_pre) r |= epi_map(&em.pre[c], d->add_pre, d->c_dst, 1, t_rows, d->n_samples, 0, 1, 1, bh, false, bb);
      if (e.has_mask) r |= epi_map(&em.mask[c], d->mask, d->c_dst, 1, t_rows, d->n_samples, 0, 1, 1, bh, false, bb);
      if (e.has_raw) r |= epi_map(&em.raw[c], d->y_raw, d->c_dst, 1, t_rows, d->n_samples, 0, 1, 1, bh, false, bb);
      if (e.has_post) r |= epi_map(&em.post[c], d->add_post, d->c_dst, 1, t_rows >> d->post_shift, d->n_samples, 0, 1, 1, bh >> d->post_shift, false, bb);
      if (e.has_act) r |= epi_map(&em.act[c], d->y_act, d->c_dst, 1, t_rows, d->n_samples, 0, 1, 1, bh, d->dup_rows != 0, bb);
    }
    if (r) return STG_ECUDA;
  }
  using Kernel = decltype(&conv_tc_kernel<true, false>);
  // [kStaged][kMask]
  static const Kernel kernels[2][2] = {{conv_tc_kernel<false, false>, conv_tc_kernel<false, true>},
                                       {conv_tc_kernel<true, false>, conv_tc_kernel<true, true>}};
  static bool attr_set = false;
  if (!attr_set) {
    for (int i = 0; i < 4; ++i) {
      const Kernel k = kernels[i >> 1][i & 1];
      STG_CUDA_CHECK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      if (i >> 1)   // staged kernels: two may share an SM
        STG_CUDA_CHECK(cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    }
    attr_set = true;
  }
  const bool masked = valid_units != nullptr;
  p.tiles_n = ceil_div(d->c_dst, p.bn);
  const int64_t n_tiles = n_rc ? (int64_t)p.cls_mt0[p.n_cls] * p.tiles_n : (int64_t)d->n_samples * p.n_res * p.tiles_m * p.tiles_n;
  if (n_tiles > 0x7fffffff) return STG_EINVAL;
  p.n_tiles = (int)n_tiles;
  g_ingest_bytes += (double)n_tiles * ((double)best.traffic * p.k_chunks / p.n_res + (staged ? (double)e.n_in * p.mrows * p.bn * 2 : 0.0));
  const int slots = (occ2 ? 2 : 1) * sm_count();
  const int grid = p.n_tiles < slots ? p.n_tiles : slots;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(staged ? 384 : 352); cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[1];
  cfg.attrs = at; cfg.numAttrs = tc_launch_attrs(at);
  STG_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernels[staged][masked], tmA, tmW, em, p));
  STG_LAUNCH_CHECK();
  return STG_OK;
}

}  // namespace stg
