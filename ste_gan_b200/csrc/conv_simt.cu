// CUDA-core (FFMA) implicit-GEMM convolution: the fp32 validation engine and the
// engine for shapes the tcgen05 path does not take (tiny channel counts).
// Handles stride / dilation / groups / period views, forward and data-gradient
// (StgConv), and the weight gradient (StgWgrad).  fp32 accumulation always.
#include "common.cuh"

namespace stg {

namespace {

constexpr int BM = 64, BN = 64, BK = 16, LDS = 68;  // LDS: padded leading dim (floats)

struct EpiP {
  int phases, t_out, c_dst, post_shift, mask_mode, act, dup_rows, out_f32, pair_sum;
  const float* bias;
  const void *add_pre, *mask, *add_post;
  void *y_raw, *y_act;
  const int32_t* valid_units;   // stg_conv_masked: rows >= valid_units[b] * rows_per_unit are written as 0 (nullptr: no mask)
  int rows_per_unit;
};

// Writes up to 4 consecutive channels of one output row.
template <typename T, bool kMask>
__device__ __forceinline__ void epilogue_row(const EpiP& e, int b, int ph, int row, int col, int ncols, float (&v)[4]) {
  const int64_t pitch = (int64_t)e.phases * e.c_dst;
  const int64_t off = ((int64_t)b * e.t_out + row) * pitch + (int64_t)ph * e.c_dst + col;
  const bool vec = (ncols == 4) && ((e.c_dst & 3) == 0);
  float pre[4] = {0, 0, 0, 0}, mk[4], post[4] = {0, 0, 0, 0};
  if (e.add_pre) {
    const T* p = static_cast<const T*>(e.add_pre) + off;
    if (vec) ld4(p, pre); else for (int i = 0; i < ncols; ++i) pre[i] = to_f(p[i]);
  }
  if (e.mask) {
    const T* p = static_cast<const T*>(e.mask) + off;
    if (vec) ld4(p, mk); else for (int i = 0; i < ncols; ++i) mk[i] = to_f(p[i]);
  }
  if (e.add_post) {
    const int t_post = e.t_out >> e.post_shift;
    const int64_t o2 = ((int64_t)b * t_post + (row >> e.post_shift)) * pitch + (int64_t)ph * e.c_dst + col;
    const T* p = static_cast<const T*>(e.add_post) + o2;
    if (vec) ld4(p, post); else for (int i = 0; i < ncols; ++i) post[i] = to_f(p[i]);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float x = v[i] + pre[i];
    if (e.mask) x *= act_grad_from_output(e.mask_mode, mk[i]);
    v[i] = x + post[i];
  }
  if constexpr (kMask) {   // a select, not a product: NaN in the padded rows of add_post cannot leak into a masked row
    const bool keep = (int64_t)row < (int64_t)max(e.valid_units[b], 0) * e.rows_per_unit;
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = keep ? v[i] : 0.f;
  }
  if (e.y_raw) {
    if (e.out_f32) {
      float* p = static_cast<float*>(e.y_raw) + off;
      if (vec) st4(p, v); else for (int i = 0; i < ncols; ++i) p[i] = v[i];
    } else {
      T* p = static_cast<T*>(e.y_raw) + off;
      if (vec) st4(p, v); else for (int i = 0; i < ncols; ++i) p[i] = from_f<T>(v[i]);
    }
  }
  if (e.y_act) {
    float a[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = act_apply(e.act, v[i]);
    const int64_t o0 = e.dup_rows ? ((int64_t)b * 2 * e.t_out + 2 * row) * pitch + (int64_t)ph * e.c_dst + col : off;
    if (e.out_f32) {
      float* p0 = static_cast<float*>(e.y_act) + o0;
      if (vec) st4(p0, a); else for (int i = 0; i < ncols; ++i) p0[i] = a[i];
      if (e.dup_rows) { float* p1 = p0 + pitch; if (vec) st4(p1, a); else for (int i = 0; i < ncols; ++i) p1[i] = a[i]; }
    } else {
      T* p0 = static_cast<T*>(e.y_act) + o0;
      if (vec) st4(p0, a); else for (int i = 0; i < ncols; ++i) p0[i] = from_f<T>(a[i]);
      if (e.dup_rows) { T* p1 = p0 + pitch; if (vec) st4(p1, a); else for (int i = 0; i < ncols; ++i) p1[i] = from_f<T>(a[i]); }
    }
  }
}

struct ConvP {
  int n_vs, phases, t_src, t_dst, c_src, c_dst, groups, k, dilation, stride, pad, transposed;
  int csrc_g, cdst_g, tiles_per_group;
  const void *src, *w;
  EpiP e;
};

// kMask: stg_conv_masked (per-sample length masks in the epilogue); the unmasked instances compile without them
template <typename T, bool kMask>
__global__ void __launch_bounds__(256) conv_simt_kernel(const ConvP p) {
  __shared__ __align__(16) float As[BK][LDS];
  __shared__ __align__(16) float Bs[BK][LDS];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int n = blockIdx.z, b = n / p.phases, ph = n % p.phases;
  const int r0 = blockIdx.x * BM;
  const int gi = blockIdx.y / p.tiles_per_group;
  const int cl0 = (blockIdx.y % p.tiles_per_group) * BN;  // column offset inside the group
  const int col0 = gi * p.cdst_g + cl0;
  const int K = p.k * p.csrc_g;
  const T* src = static_cast<const T*>(p.src);
  const T* w = static_cast<const T*>(p.w);
  const int64_t src_pitch = (int64_t)p.phases * p.c_src;
  const int64_t src_base = (int64_t)b * p.t_src * src_pitch + (int64_t)ph * p.c_src + (int64_t)gi * p.csrc_g;

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const int lrow = tid >> 2, lk = (tid & 3) * 4;
  const int drow = r0 + lrow;
  const bool vec4 = (p.csrc_g & 3) == 0;
  const bool col_ok = (cl0 + lrow) < p.cdst_g;

  for (int k0 = 0; k0 < K; k0 += BK) {
    const int kg = k0 + lk;
    float a[4] = {0, 0, 0, 0}, bb[4] = {0, 0, 0, 0};
    if (vec4) {
      if (kg < K) {
        const int j = kg / p.csrc_g, q = kg - j * p.csrc_g;
        int srow;
        bool ok = drow < p.t_dst;
        if (!p.transposed) {
          srow = drow * p.stride + j * p.dilation - p.pad;
        } else {
          const int num = drow + p.pad - j * p.dilation;
          srow = num / p.stride;
          ok = ok && (num >= 0) && (srow * p.stride == num);
        }
        ok = ok && srow >= 0 && srow < p.t_src;
        if (ok) ld4(src + src_base + (int64_t)srow * src_pitch + q, a);
        if (col_ok) ld4(w + ((int64_t)j * p.c_dst + col0 + lrow) * p.csrc_g + q, bb);
      }
    } else {
      // channel counts that are not a multiple of 4 (C = 1 logits): element-wise gather
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int ke = kg + i;
        if (ke >= K) break;
        const int j = ke / p.csrc_g, q = ke - j * p.csrc_g;
        int srow;
        bool ok = drow < p.t_dst;
        if (!p.transposed) {
          srow = drow * p.stride + j * p.dilation - p.pad;
        } else {
          const int num = drow + p.pad - j * p.dilation;
          srow = num / p.stride;
          ok = ok && (num >= 0) && (srow * p.stride == num);
        }
        ok = ok && srow >= 0 && srow < p.t_src;
        if (ok) a[i] = to_f(src[src_base + (int64_t)srow * src_pitch + q]);
        if (col_ok) bb[i] = to_f(w[((int64_t)j * p.c_dst + col0 + lrow) * p.csrc_g + q]);
      }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) { As[lk + i][lrow] = a[i]; Bs[lk + i][lrow] = bb[i]; }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 av = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float ar[4] = {av.x, av.y, av.z, av.w}, br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
    }
  }

  const int cl = cl0 + tx * 4;
  if (cl >= p.cdst_g) return;
  const int ncols = min(4, p.cdst_g - cl);
  const int col = gi * p.cdst_g + cl;
  float bias[4] = {0, 0, 0, 0};
  if (p.e.bias) for (int i = 0; i < ncols; ++i) bias[i] = p.e.bias[col + i];
  if (p.e.pair_sum) {
#pragma unroll
    for (int i = 0; i < 4; i += 2) {
      const int row = r0 + ty * 4 + i;  // accumulator row (even)
      if (row + 1 < p.t_dst + 1 && row < p.t_dst) {
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = acc[i][j] + acc[i + 1][j] + 2.f * bias[j];
        epilogue_row<T, kMask>(p.e, b, ph, row >> 1, col, ncols, v);
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int row = r0 + ty * 4 + i;
      if (row < p.t_dst) {
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = acc[i][j] + bias[j];
        epilogue_row<T, kMask>(p.e, b, ph, row, col, ncols, v);
      }
    }
  }
}

// ---------------------------------------------------------------- wgrad
struct WgP {
  int n_vs, phases, t_in, t_out, c_in, c_out, groups, k, dilation, stride, pad;
  int cin_g, cout_g, tiles_per_group, rows_per_split;
  int64_t total_rows;
  const void *x, *dy;
  float* dw;
};

template <typename T>
__global__ void __launch_bounds__(256) wgrad_simt_kernel(const WgP p) {
  __shared__ __align__(16) float As[BK][LDS];  // dy  [row][co]
  __shared__ __align__(16) float Bs[BK][LDS];  // x   [row][kk]
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int KK = p.k * p.cin_g;
  const int kk0 = blockIdx.x * BN;
  const int gi = blockIdx.y / p.tiles_per_group;
  const int cl0 = (blockIdx.y % p.tiles_per_group) * BM;
  const int co0 = gi * p.cout_g + cl0;
  const T* x = static_cast<const T*>(p.x);
  const T* dy = static_cast<const T*>(p.dy);
  const int64_t x_pitch = (int64_t)p.phases * p.c_in, y_pitch = (int64_t)p.phases * p.c_out;

  const int64_t row_begin = (int64_t)blockIdx.z * p.rows_per_split;
  const int64_t row_end = min(p.total_rows, row_begin + (int64_t)p.rows_per_split);

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const int lrow = tid >> 4, lc = (tid & 15) * 4;
  // decode this thread's (tap, channel) once: it does not change over the row loop
  const int kg = kk0 + lc;
  const bool kk_ok = kg < KK;
  const int tj = kk_ok ? kg / p.cin_g : 0;
  const int tq = kk_ok ? kg - tj * p.cin_g : 0;
  const bool co_ok = (cl0 + lc) < p.cout_g;
  const int co_n = co_ok ? min(4, p.cout_g - (cl0 + lc)) : 0;

  for (int64_t rr = row_begin; rr < row_end; rr += BK) {
    const int64_t r = rr + lrow;
    float a[4] = {0, 0, 0, 0}, bb[4] = {0, 0, 0, 0};
    if (r < row_end) {
      const int n = (int)(r / p.t_out), to = (int)(r - (int64_t)n * p.t_out);
      const int b = n / p.phases, ph = n - b * p.phases;
      if (co_ok) {
        const T* ptr = dy + ((int64_t)b * p.t_out + to) * y_pitch + (int64_t)ph * p.c_out + co0 + lc;
        if (co_n == 4 && (p.c_out & 3) == 0) ld4(ptr, a);
        else for (int i = 0; i < co_n; ++i) a[i] = to_f(ptr[i]);
      }
      if (kk_ok) {
        const int xr = to * p.stride + tj * p.dilation - p.pad;
        if (xr >= 0 && xr < p.t_in)
          ld4(x + ((int64_t)b * p.t_in + xr) * x_pitch + (int64_t)ph * p.c_in + (int64_t)gi * p.cin_g + tq, bb);
      }
    }
    __syncthreads();
    *reinterpret_cast<float4*>(&As[lrow][lc]) = make_float4(a[0], a[1], a[2], a[3]);
    *reinterpret_cast<float4*>(&Bs[lrow][lc]) = make_float4(bb[0], bb[1], bb[2], bb[3]);
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 av = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float ar[4] = {av.x, av.y, av.z, av.w}, br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int cl = cl0 + ty * 4 + i;
    if (cl >= p.cout_g) continue;
    const int co = gi * p.cout_g + cl;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int kq = kk0 + tx * 4 + j;
      if (kq < KK) atomicAdd(p.dw + (int64_t)co * KK + kq, acc[i][j]);
    }
  }
}

// Column sums (bias gradient): out[c] += sum_r dy[r][c].  Generic path for C that is not a multiple of the vector width.
template <typename T>
__global__ void __launch_bounds__(256) colsum_kernel(const T* __restrict__ dy, int64_t rows, int C, int rows_per_block,
                                                     float* __restrict__ out) {
  __shared__ float red[32];
  const int64_t rb = (int64_t)blockIdx.x * rows_per_block, re = min(rows, rb + rows_per_block);
  for (int c = 0; c < C; ++c) {
    float s = 0.f;
    for (int64_t r = rb + threadIdx.x; r < re; r += 256) s += to_f(dy[r * C + c]);
    s = block_sum(s, red);
    if (threadIdx.x == 0) atomicAdd(out + c, s);
  }
}

// Vectorised path: a thread owns VEC consecutive channels (16-byte loads) and walks rows with stride `lanes`;
// the block reduces its row lanes in shared memory and issues C atomics.  HBM/L2-bound: dy is read once.
template <typename T, int VEC>
__global__ void __launch_bounds__(256) colsum_vec_kernel(const T* __restrict__ dy, int64_t rows, int C, int rows_per_block,
                                                         float* __restrict__ out) {
  __shared__ float red[256 * VEC];
  const int cg = C / VEC, lanes = 256 / cg;
  const int rl = threadIdx.x / cg, c = threadIdx.x - rl * cg;
  const int64_t rb = (int64_t)blockIdx.x * rows_per_block, re = min(rows, rb + rows_per_block);
  float acc[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) acc[i] = 0.f;
  if (rl < lanes) {
    for (int64_t r = rb + rl; r < re; r += lanes) {
      const T* p = dy + r * C + c * VEC;
      if constexpr (VEC == 8) {
        float a[4], b[4];
        const uint4 q = *reinterpret_cast<const uint4*>(p);
        const uint2 lo = make_uint2(q.x, q.y), hi = make_uint2(q.z, q.w);
        ld4(reinterpret_cast<const bf16*>(&lo), a); ld4(reinterpret_cast<const bf16*>(&hi), b);
#pragma unroll
        for (int i = 0; i < 4; ++i) { acc[i] += a[i]; acc[4 + i] += b[i]; }
      } else {
        float a[4];
        ld4(p, a);
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[i] += a[i];
      }
    }
  }
#pragma unroll
  for (int i = 0; i < VEC; ++i) red[threadIdx.x * VEC + i] = acc[i];
  __syncthreads();
  int s = 1;
  while (s < lanes) s <<= 1;
  for (s >>= 1; s > 0; s >>= 1) {
    if (rl < s && rl + s < lanes) {
#pragma unroll
      for (int i = 0; i < VEC; ++i) red[threadIdx.x * VEC + i] += red[(threadIdx.x + s * cg) * VEC + i];
    }
    __syncthreads();
  }
  if (rl == 0) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) atomicAdd(out + c * VEC + i, red[threadIdx.x * VEC + i]);
  }
}

}  // namespace

int conv_simt(const StgConv* d, cudaStream_t s, const int32_t* valid_units, int rows_per_unit) {
  ConvP p;
  p.n_vs = d->n_samples * d->phases; p.phases = d->phases; p.t_src = d->t_src; p.t_dst = d->t_dst;
  p.c_src = d->c_src; p.c_dst = d->c_dst; p.groups = d->groups; p.k = d->k; p.dilation = d->dilation;
  p.stride = d->stride; p.pad = d->pad; p.transposed = d->transposed;
  p.csrc_g = d->c_src / d->groups; p.cdst_g = d->c_dst / d->groups;
  p.tiles_per_group = ceil_div(p.cdst_g, BN);
  p.src = d->src; p.w = d->w;
  if (d->pair_sum && (d->t_dst & 1)) return STG_EINVAL;
  EpiP& e = p.e;
  e.phases = d->phases; e.t_out = d->pair_sum ? d->t_dst / 2 : d->t_dst; e.c_dst = d->c_dst;
  e.post_shift = d->post_shift; e.mask_mode = d->mask_mode; e.act = d->act; e.dup_rows = d->dup_rows;
  e.out_f32 = d->out_f32; e.pair_sum = d->pair_sum; e.bias = d->bias; e.add_pre = d->add_pre; e.mask = d->mask;
  e.add_post = d->add_post; e.y_raw = d->y_raw; e.y_act = d->y_act;
  e.valid_units = valid_units; e.rows_per_unit = rows_per_unit;
  dim3 grid(ceil_div(d->t_dst, BM), d->groups * p.tiles_per_group, p.n_vs);
  if (grid.z > 65535 || grid.y > 65535) return STG_EINVAL;
  const bool masked = valid_units != nullptr;
  if (d->dtype == STG_F32) (masked ? conv_simt_kernel<float, true> : conv_simt_kernel<float, false>)<<<grid, 256, 0, s>>>(p);
  else (masked ? conv_simt_kernel<bf16, true> : conv_simt_kernel<bf16, false>)<<<grid, 256, 0, s>>>(p);
  STG_LAUNCH_CHECK();
  return STG_OK;
}

int wgrad_simt(const StgWgrad* d, cudaStream_t s) {
  WgP p;
  p.n_vs = d->n_samples * d->phases; p.phases = d->phases; p.t_in = d->t_in; p.t_out = d->t_out;
  p.c_in = d->c_in; p.c_out = d->c_out; p.groups = d->groups; p.k = d->k; p.dilation = d->dilation;
  p.stride = d->stride; p.pad = d->pad;
  p.cin_g = d->c_in / d->groups; p.cout_g = d->c_out / d->groups;
  if ((p.cin_g & 3) != 0) return STG_EINVAL;
  p.tiles_per_group = ceil_div(p.cout_g, BM);
  p.total_rows = (int64_t)p.n_vs * d->t_out;
  p.x = d->x; p.dy = d->dy; p.dw = d->dw;
  const int gx = ceil_div(d->k * p.cin_g, BN), gy = d->groups * p.tiles_per_group;
  // aim for ~4 waves of CTAs; each split at least 64 rows
  int64_t want = ceil_div64(148 * 4, (int64_t)gx * gy);
  int64_t max_splits = ceil_div64(p.total_rows, 64);
  int64_t nsplit = want < 1 ? 1 : (want > max_splits ? max_splits : want);
  if (nsplit > 65535) nsplit = 65535;
  p.rows_per_split = (int)(ceil_div64(ceil_div64(p.total_rows, nsplit), BK) * BK);
  nsplit = ceil_div64(p.total_rows, p.rows_per_split);
  dim3 grid(gx, gy, (unsigned)nsplit);
  if (d->dw) {
    if (d->dtype == STG_F32) wgrad_simt_kernel<float><<<grid, 256, 0, s>>>(p);
    else wgrad_simt_kernel<bf16><<<grid, 256, 0, s>>>(p);
    STG_LAUNCH_CHECK();
  }
  return STG_OK;
}

int colsum(const void* dy, int dtype, int64_t rows, int C, float* out, cudaStream_t s) {
  const int vec = dtype == STG_F32 ? 4 : 8;
  if (C % vec == 0 && C / vec <= 256) {
    const int lanes = 256 / (C / vec);
    int64_t rpb = ceil_div64(rows, 148 * 4);
    if (rpb < 4 * lanes) rpb = 4 * lanes;
    const int blocks = (int)ceil_div64(rows, rpb);
    if (dtype == STG_F32) colsum_vec_kernel<float, 4><<<blocks, 256, 0, s>>>(static_cast<const float*>(dy), rows, C, (int)rpb, out);
    else colsum_vec_kernel<bf16, 8><<<blocks, 256, 0, s>>>(static_cast<const bf16*>(dy), rows, C, (int)rpb, out);
  } else {
    int64_t rpb = ceil_div64(rows, 148 * 2);
    if (rpb < 1024) rpb = 1024;
    const int blocks = (int)ceil_div64(rows, rpb);
    if (dtype == STG_F32) colsum_kernel<float><<<blocks, 256, 0, s>>>(static_cast<const float*>(dy), rows, C, (int)rpb, out);
    else colsum_kernel<bf16><<<blocks, 256, 0, s>>>(static_cast<const bf16*>(dy), rows, C, (int)rpb, out);
  }
  STG_LAUNCH_CHECK();
  return STG_OK;
}

}  // namespace stg
