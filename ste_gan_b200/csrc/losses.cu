// Loss kernels: multi-resolution time-domain feature loss (fwd + bwd) and its per-utterance scores on length-masked
// batches (fwd), LSGAN MSE-to-constant and feature-matching L1 reductions (fwd + bwd).  HBM-bound; vectorised loads where
// the layout allows, warp-shuffle + one atomic per block reductions (fixed-order, atomic-free for the per-utterance
// scores), fp32 arithmetic throughout.
#include "common.cuh"

namespace stg {
namespace {

__device__ __forceinline__ int reflect(int t, int T_) {
  t = t < 0 ? -t : t;
  return t >= T_ ? 2 * (T_ - 1) - t : t;
}
__device__ __forceinline__ float sgn(float d) { return (float)((d > 0.f) - (d < 0.f)); }

// low = avg(avg(x)) (window 2*half+1, 9 in the reference) with reflect padding at each stage; hi = |x - low|
// (time_domain_loss.py:51-60)
__global__ void td_filter_kernel(const float* __restrict__ x, int T_, int C, int64_t total, int half, float* __restrict__ low,
                                 float* __restrict__ hi) {
  const float iw = 1.f / (float)(2 * half + 1);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const int64_t bt = i / C;
    const int t = (int)(bt % T_);
    const float* xs = x + (bt - t) * C + c;  // sample base, channel c; element t at xs[t*C]
    float s2 = 0.f;
    for (int a = -half; a <= half; ++a) {
      const int u = reflect(t + a, T_);
      float s1 = 0.f;
      for (int q = -half; q <= half; ++q) s1 += xs[(int64_t)reflect(u + q, T_) * C];
      s2 += s1 * iw;
    }
    const float lw = s2 * iw;
    low[i] = lw;
    hi[i] = fabsf(xs[(int64_t)t * C] - lw);
  }
}

struct TdRes { int win, shift, frames, start0; };   // start0: first sample of frame 0 (-win/2 with padded windowing, else 0)

// one thread per (b, f, c): 4 features of real and generated, L1, optional scatter of d/dlow, d/dhi
__global__ void __launch_bounds__(256) td_feature_kernel(const float* __restrict__ low_r, const float* __restrict__ hi_r,
                                                         const float* __restrict__ low_g, const float* __restrict__ hi_g,
                                                         int B, int T_, int C, TdRes r, float* __restrict__ loss_slot,
                                                         float gscale_host, const float* __restrict__ gscale_dev,
                                                         float* __restrict__ dlow, float* __restrict__ dhi) {
  __shared__ float red[32];
  const float gscale = gscale_dev ? *gscale_dev : gscale_host;   // upstream gradient of this resolution's loss
  const int64_t total = (int64_t)B * r.frames * C;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const float inv_n = 1.f / (float)(total * 4);
  float acc = 0.f;
  if (i < total) {
    const int c = (int)(i % C);
    const int64_t bf = i / C;
    const int f = (int)(bf % r.frames), b = (int)(bf / r.frames);
    const int64_t base = (int64_t)b * T_ * C + c;
    const int start = f * r.shift + r.start0;
    float ml_r = 0, pl_r = 0, ph_r = 0, mh_r = 0, ml_g = 0, pl_g = 0, ph_g = 0, mh_g = 0;
    for (int j = 0; j < r.win; ++j) {
      const int64_t o = base + (int64_t)reflect(start + j, T_) * C;
      const float a = low_r[o], h = hi_r[o], a2 = low_g[o], h2 = hi_g[o];
      ml_r += a; pl_r = fmaf(a, a, pl_r); ph_r = fmaf(h, h, ph_r); mh_r += h;
      ml_g += a2; pl_g = fmaf(a2, a2, pl_g); ph_g = fmaf(h2, h2, ph_g); mh_g += h2;
    }
    const float iw = 1.f / (float)r.win;
    const float d0 = (ml_g - ml_r) * iw, d1 = pl_g - pl_r, d2 = ph_g - ph_r, d3 = (mh_g - mh_r) * iw;
    acc = fabsf(d0) + fabsf(d1) + fabsf(d2) + fabsf(d3);
    if (dlow) {
      const float s0 = sgn(d0) * inv_n * gscale * iw, s1 = sgn(d1) * inv_n * gscale * 2.f;
      const float s2 = sgn(d2) * inv_n * gscale * 2.f, s3 = sgn(d3) * inv_n * gscale * iw;
      for (int j = 0; j < r.win; ++j) {
        const int64_t o = base + (int64_t)reflect(start + j, T_) * C;
        atomicAdd(dlow + o, s0 + s1 * low_g[o]);
        atomicAdd(dhi + o, s3 + s2 * hi_g[o]);
      }
    }
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) atomicAdd(loss_slot, acc * inv_n);
}

// z = dlow - dhi*sgn(x-low) (in place over dlow) ; dx += dhi*sgn(x-low)
__global__ void td_bwd_split_kernel(const float* __restrict__ x, const float* __restrict__ low, float* __restrict__ dlow,
                                    const float* __restrict__ dhi, int64_t total, float* __restrict__ dx) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const float d = dhi[i] * sgn(x[i] - low[i]);
    dlow[i] -= d;
    dx[i] += d;
  }
}
// transpose of the reflect-padded (2*half+1)-tap mean: out[reflect(t+a)] += z[t]/window
__global__ void td_avg9_t_kernel(const float* __restrict__ z, int T_, int C, int64_t total, int half, float* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const int64_t bt = i / C;
    const int t = (int)(bt % T_);
    const int64_t base = (bt - t) * C + c;
    const float v = z[i] / (float)(2 * half + 1);
    for (int a = -half; a <= half; ++a) atomicAdd(out + base + (int64_t)reflect(t + a, T_) * C, v);
  }
}

template <typename T, typename TD>
__global__ void __launch_bounds__(256) mse_const_kernel(const T* __restrict__ x, int64_t n, float target,
                                                        float* __restrict__ slot, float gcoef, TD* __restrict__ dx) {
  __shared__ float red[32];
  float acc = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float d = to_f(x[i]) - target;
    acc = fmaf(d, d, acc);
    if (dx) dx[i] = from_f<TD>(gcoef * d);
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0 && slot) atomicAdd(slot, acc / (float)n);
}

template <typename T>
__global__ void __launch_bounds__(256) l1_mean_kernel(const T* __restrict__ a, const T* __restrict__ b, int64_t n4,
                                                      int64_t n, float* __restrict__ slot, float gcoef, T* __restrict__ da) {
  __shared__ float red[32];
  float acc = 0.f;
  // vector body (4 elements / thread / iteration)
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float va[4], vb[4], g[4];
    ld4(a + 4 * i, va);
    ld4(b + 4 * i, vb);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float d = va[q] - vb[q];
      acc += fabsf(d);
      g[q] = gcoef * sgn(d);
    }
    if (da) st4(da + 4 * i, g);
  }
  // scalar tail
  for (int64_t i = 4 * n4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float d = to_f(a[i]) - to_f(b[i]);
    acc += fabsf(d);
    if (da) da[i] = from_f<T>(gcoef * sgn(d));
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0 && slot) atomicAdd(slot, acc / (float)n);
}

// ---- multi-tensor forms (the feature-matching / LSGAN terms are 27 + 24 tiny tensors per step): the item table
// travels BY VALUE in the kernel parameters, so the launch is CUDA-graph capturable with no device-side table.
struct L1Table { StgL1Item it[STG_MAX_LOSS_ITEMS]; int block0[STG_MAX_LOSS_ITEMS + 1]; int n; };
struct MseTable { StgMseItem it[STG_MAX_LOSS_ITEMS]; int block0[STG_MAX_LOSS_ITEMS + 1]; int n; };

template <typename Tab>
__device__ __forceinline__ int item_of_block(const Tab& t, int blk) {
  int i = 0;
  while (i + 1 < t.n && t.block0[i + 1] <= blk) ++i;
  return i;
}

template <typename T>
__global__ void __launch_bounds__(256) l1_mean_multi_kernel(const L1Table tab, float* __restrict__ slot, float grad_scale) {
  __shared__ float red[32];
  const int i = item_of_block(tab, blockIdx.x);
  const StgL1Item d = tab.it[i];
  const int lb = blockIdx.x - tab.block0[i], nb = tab.block0[i + 1] - tab.block0[i];
  const T* a = static_cast<const T*>(d.a); const T* b = static_cast<const T*>(d.b); T* da = static_cast<T*>(d.da);
  const int64_t n = d.n;
  const bool al = ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(da)) & 15) == 0;
  const int64_t n4 = al ? n / 4 : 0;
  const float gcoef = grad_scale / (float)n;
  float acc = 0.f;
  for (int64_t j = (int64_t)lb * 256 + threadIdx.x; j < n4; j += (int64_t)nb * 256) {
    float va[4], vb[4], g[4];
    ld4(a + 4 * j, va);
    ld4(b + 4 * j, vb);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float df = va[q] - vb[q];
      acc += fabsf(df);
      g[q] = gcoef * sgn(df);
    }
    if (da) st4(da + 4 * j, g);
  }
  for (int64_t j = 4 * n4 + (int64_t)lb * 256 + threadIdx.x; j < n; j += (int64_t)nb * 256) {
    const float df = to_f(a[j]) - to_f(b[j]);
    acc += fabsf(df);
    if (da) da[j] = from_f<T>(gcoef * sgn(df));
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0 && slot) atomicAdd(slot, acc / (float)n);
}

template <typename T, typename TD>
__global__ void __launch_bounds__(256) mse_const_multi_kernel(const MseTable tab, float* __restrict__ slots, float grad_scale) {
  __shared__ float red[32];
  const int i = item_of_block(tab, blockIdx.x);
  const StgMseItem d = tab.it[i];
  const int lb = blockIdx.x - tab.block0[i], nb = tab.block0[i + 1] - tab.block0[i];
  const T* x = static_cast<const T*>(d.x); TD* dx = static_cast<TD*>(d.dx);
  const float gcoef = grad_scale * 2.f / (float)d.n;
  float acc = 0.f;
  for (int64_t j = (int64_t)lb * 256 + threadIdx.x; j < d.n; j += (int64_t)nb * 256) {
    const float df = to_f(x[j]) - d.target;
    acc = fmaf(df, df, acc);
    if (dx) dx[j] = from_f<TD>(gcoef * df);
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0 && slots) atomicAdd(slots + d.slot, acc / (float)d.n);
}

// reflect-padded moving average over the last axis of [rows][T]
__global__ void average_filter_kernel(const float* __restrict__ x, int64_t rows, int T_, int window, int pad, int To,
                                      float* __restrict__ out) {
  const int64_t total = rows * To;
  const int half = pad ? window / 2 : 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / To;
    const int t = (int)(i - r * To);
    float s = 0.f;
    for (int j = 0; j < window; ++j) s += x[r * T_ + reflect(t - half + j, T_)];
    out[i] = s / (float)window;
  }
}

// framed mean and power of one signal: one thread per (b, f, c)   (time_domain_loss.py:35-49)
__global__ void frame_stats_kernel(const float* __restrict__ x, int B, int T_, int C, TdRes r, float* __restrict__ mean,
                                   float* __restrict__ power, int out_stride, int mean_off, int power_off) {
  const int64_t total = (int64_t)B * r.frames * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const int64_t bf = i / C;
    const int f = (int)(bf % r.frames), b = (int)(bf / r.frames);
    const int64_t base = (int64_t)b * T_ * C + c;
    const int start = f * r.shift + r.start0;
    float m = 0.f, p = 0.f;
    for (int j = 0; j < r.win; ++j) {
      const float a = x[base + (int64_t)reflect(start + j, T_) * C];
      m += a; p = fmaf(a, a, p);
    }
    if (mean) mean[i * out_stride + mean_off] = m / (float)r.win;
    if (power) power[i * out_stride + power_off] = p;
  }
}
// Tensor.unfold(1, win, shift) of the (reflect-padded) signal: out[b][f][c][j]   (time_domain_loss.py:35-41)
__global__ void window_signal_kernel(const float* __restrict__ x, int B, int T_, int C, TdRes r, float* __restrict__ out) {
  const int64_t total = (int64_t)B * r.frames * C * r.win;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int j = (int)(i % r.win);
    int64_t q = i / r.win;
    const int c = (int)(q % C); q /= C;
    const int f = (int)(q % r.frames), b = (int)(q / r.frames);
    out[i] = x[((int64_t)b * T_ + reflect(f * r.shift + r.start0 + j, T_)) * C + c];
  }
}

// ---- per-utterance scores of a padded batch (stg_td_scores).  Sample b holds n_b rows and no row >= n_b of either input is
// read: the filter reflects at n_b and the frames are those of an n_b-row signal.  The features of (b, resolution i) are summed
// in chunks of TS_ITEMS (frame, channel) items, one CTA per chunk, then the chunks in order by one thread: fixed-order sums
// without atomics, so a sample's value does not depend on the batch, on T or on the replay.
constexpr int TS_ITEMS = 256;    // (frame, channel) items per chunk = threads per CTA
struct TdResSet { TdRes r[8]; };

__device__ __forceinline__ int ts_rows(const int32_t* valid_units, int b, int rows_per_unit, int T_) {
  return min(max(valid_units[b], 0), T_ / rows_per_unit) * rows_per_unit;
}
// frames of an n-row signal, 0 where the reference's reflect padding (or unfold) raises: n <= avg_window / 2, n <= win / 2
// with padded windows, or fewer rows than one window
__device__ __forceinline__ int ts_frames(int n, int half, const TdRes& r) {
  const int p = -r.start0;
  if (n <= half || p >= n) return 0;
  const int padded = n + 2 * p;
  return padded < r.win ? 0 : (padded - r.win) / r.shift + 1;
}

// low = avg(avg(x)), hi = |x - low| of both inputs (filt = low_r | hi_r | low_g | hi_g, [B][T][C] each); rows >= n_b of filt
// are left as they are
__global__ void td_filter_masked_kernel(const float* __restrict__ x_real, const float* __restrict__ x_gen, int T_, int C,
                                        int64_t n, const int32_t* __restrict__ valid_units, int rows_per_unit, int half,
                                        float* __restrict__ filt) {
  const float iw = 1.f / (float)(2 * half + 1);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < 2 * n; i += (int64_t)gridDim.x * blockDim.x) {
    const int gen = i >= n;
    const int64_t e = gen ? i - n : i;
    const int c = (int)(e % C);
    const int64_t bt = e / C;
    const int t = (int)(bt % T_);
    const int nb = ts_rows(valid_units, (int)(bt / T_), rows_per_unit, T_);
    if (t >= nb || nb <= half) continue;
    const float* xs = (gen ? x_gen : x_real) + (bt - t) * C + c;
    float s2 = 0.f;
    for (int a = -half; a <= half; ++a) {
      const int u = reflect(t + a, nb);
      float s1 = 0.f;
      for (int q = -half; q <= half; ++q) s1 += xs[(int64_t)reflect(u + q, nb) * C];
      s2 += s1 * iw;
    }
    const float lw = s2 * iw;
    float* low = filt + 2 * gen * n;
    low[e] = lw;
    low[n + e] = fabsf(xs[(int64_t)t * C] - lw);
  }
}

// grid (chunk, b, i): partial[(b * n_res + i) * chunks + chunk] = sum over this chunk's items of the 4 feature L1 terms
__global__ void __launch_bounds__(TS_ITEMS) td_score_partial_kernel(const float* __restrict__ filt, int T_, int C, int64_t n,
                                                                      const int32_t* __restrict__ valid_units, int rows_per_unit,
                                                                      int half, const __grid_constant__ TdResSet rs, int chunks,
                                                                      float* __restrict__ partial) {
  __shared__ float red[32];
  const int chunk = blockIdx.x, b = blockIdx.y, i = blockIdx.z;
  const TdRes& r = rs.r[i];
  const int nb = ts_rows(valid_units, b, rows_per_unit, T_);
  const int64_t items = (int64_t)ts_frames(nb, half, r) * C;
  if ((int64_t)chunk * TS_ITEMS >= items) return;                   // uniform over the CTA
  const float *low_r = filt, *hi_r = filt + n, *low_g = filt + 2 * n, *hi_g = filt + 3 * n;
  const float iw = 1.f / (float)r.win;
  const int64_t j = (int64_t)chunk * TS_ITEMS + threadIdx.x;
  float acc = 0.f;
  if (j < items) {
    const int c = (int)(j % C), f = (int)(j / C);
    const int64_t base = (int64_t)b * T_ * C + c;
    const int start = f * r.shift + r.start0;
    float ml_r = 0, pl_r = 0, ph_r = 0, mh_r = 0, ml_g = 0, pl_g = 0, ph_g = 0, mh_g = 0;
    for (int q = 0; q < r.win; ++q) {
      const int64_t o = base + (int64_t)reflect(start + q, nb) * C;
      const float a = low_r[o], h = hi_r[o], a2 = low_g[o], h2 = hi_g[o];
      ml_r += a; pl_r = fmaf(a, a, pl_r); ph_r = fmaf(h, h, ph_r); mh_r += h;
      ml_g += a2; pl_g = fmaf(a2, a2, pl_g); ph_g = fmaf(h2, h2, ph_g); mh_g += h2;
    }
    acc = fabsf((ml_g - ml_r) * iw) + fabsf(pl_g - pl_r) + fabsf(ph_g - ph_r) + fabsf((mh_g - mh_r) * iw);
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) partial[((int64_t)b * gridDim.z + i) * chunks + chunk] = acc;
}

// one thread per (b, i): the chunks in order, over F_b * C * 4 features; NaN where the sample has no frames
__global__ void td_score_finish_kernel(const float* __restrict__ partial, const int32_t* __restrict__ valid_units,
                                       int rows_per_unit, int T_, int C, int half, TdResSet rs, int B, int n_res, int chunks,
                                       float* __restrict__ out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= B * n_res) return;
  const int64_t items = (int64_t)ts_frames(ts_rows(valid_units, k / n_res, rows_per_unit, T_), half, rs.r[k % n_res]) * C;
  if (items == 0) { out[k] = __int_as_float(0x7fffffff); return; }
  float s = 0.f;
  for (int64_t q = 0; q * TS_ITEMS < items; ++q) s += partial[(int64_t)k * chunks + q];
  out[k] = s / (float)(items * 4);
}

inline int grid_for(int64_t n, int per_thread = 1) {
  int64_t b = ceil_div64(n, 256 * (int64_t)per_thread);
  const int64_t cap = 148 * 8;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace
}  // namespace stg

using namespace stg;
#define S_ static_cast<cudaStream_t>(stream)

static bool td_res(int T, int win, int shift, int pad_windows, TdRes* r) {
  if (win < 1 || shift < 1) return false;
  const int padded = pad_windows ? T + 2 * (win / 2) : T;
  if (padded < win || (pad_windows && win / 2 >= T)) return false;   // reflect padding needs pad < T
  r->win = win; r->shift = shift; r->start0 = pad_windows ? -(win / 2) : 0;
  r->frames = (padded - win) / shift + 1;
  return true;
}

extern "C" int stg_td_loss_ex(const float* x_real, const float* x_gen, int B, int T, int C, int n_res, const int* wins,
                              const int* shifts, int pad_windows, int avg_window, float* losses,
                              const float* grad_scale, const float* grad_scale_dev, float* dx_gen, float* scratch,
                              stg_stream_t stream) {
  if (!x_real || !x_gen || !losses || !scratch || !wins || !shifts || n_res < 1 || n_res > 8) return STG_EINVAL;
  if (avg_window < 1 || (avg_window & 1) == 0 || avg_window / 2 >= T) return STG_EINVAL;
  if (dx_gen && !grad_scale && !grad_scale_dev) return STG_EINVAL;
  TdRes rs[8];
  for (int i = 0; i < n_res; ++i) if (!td_res(T, wins[i], shifts[i], pad_windows, &rs[i])) return STG_EINVAL;
  const int half = avg_window / 2;
  const int64_t n = (int64_t)B * T * C;
  float *low_r = scratch, *hi_r = scratch + n, *low_g = scratch + 2 * n, *hi_g = scratch + 3 * n;
  float *dlow = scratch + 4 * n, *dhi = scratch + 5 * n;
  td_filter_kernel<<<grid_for(n), 256, 0, S_>>>(x_real, T, C, n, half, low_r, hi_r);
  STG_LAUNCH_CHECK();
  td_filter_kernel<<<grid_for(n), 256, 0, S_>>>(x_gen, T, C, n, half, low_g, hi_g);
  STG_LAUNCH_CHECK();
  STG_CUDA_CHECK(cudaMemsetAsync(losses, 0, n_res * sizeof(float), S_));
  if (dx_gen) STG_CUDA_CHECK(cudaMemsetAsync(dlow, 0, 2 * n * sizeof(float), S_));
  for (int i = 0; i < n_res; ++i) {
    const int64_t total = (int64_t)B * rs[i].frames * C;
    td_feature_kernel<<<(int)ceil_div64(total, 256), 256, 0, S_>>>(
        low_r, hi_r, low_g, hi_g, B, T, C, rs[i], losses + i, (dx_gen && grad_scale) ? grad_scale[i] : 0.f,
        (dx_gen && grad_scale_dev) ? grad_scale_dev + i : nullptr, dx_gen ? dlow : nullptr, dhi);
    STG_LAUNCH_CHECK();
  }
  if (dx_gen) {
    td_bwd_split_kernel<<<grid_for(n), 256, 0, S_>>>(x_gen, low_g, dlow, dhi, n, dx_gen);
    STG_LAUNCH_CHECK();
    STG_CUDA_CHECK(cudaMemsetAsync(dhi, 0, n * sizeof(float), S_));
    td_avg9_t_kernel<<<grid_for(n), 256, 0, S_>>>(dlow, T, C, n, half, dhi);  // dhi <- A^T z
    STG_LAUNCH_CHECK();
    td_avg9_t_kernel<<<grid_for(n), 256, 0, S_>>>(dhi, T, C, n, half, dx_gen);  // dx += A^T A^T z
    STG_LAUNCH_CHECK();
  }
  return STG_OK;
}

extern "C" int stg_td_loss(const float* x_real, const float* x_gen, int B, int T, int C, float* losses,
                           const float* grad_scale, float* dx_gen, float* scratch, stg_stream_t stream) {
  const int wins[3] = {20, 51, 80}, shifts[3] = {8, 13, 16};  // time_domain_loss.py:88-93
  return stg_td_loss_ex(x_real, x_gen, B, T, C, 3, wins, shifts, 1, 9, losses, grad_scale, nullptr, dx_gen, scratch, stream);
}

extern "C" int stg_td_scores(const float* x_real, const float* x_gen, int B, int T, int C, const int32_t* valid_units,
                             int32_t rows_per_unit, int n_res, const int* wins, const int* shifts, int pad_windows,
                             int avg_window, float* out, float* scratch, stg_stream_t stream) {
  if (!x_real || !x_gen || !valid_units || !wins || !shifts || !out || !scratch) return STG_EINVAL;
  if (B < 1 || T < 1 || C < 1 || n_res < 1 || n_res > 8 || avg_window < 1 || (avg_window & 1) == 0) return STG_EINVAL;
  if (rows_per_unit < 1 || T % rows_per_unit != 0) return STG_EINVAL;
  if (B > 65535) return STG_EUNSUPPORTED;                           // grid y
  TdResSet rs;
  int64_t chunks = 1;                                               // of the longest sample (n_b = T) at any resolution
  for (int i = 0; i < n_res; ++i) {
    if (wins[i] < 1 || shifts[i] < 1) return STG_EINVAL;
    const int p = pad_windows ? wins[i] / 2 : 0;
    rs.r[i] = TdRes{wins[i], shifts[i], 0, -p};
    const int64_t padded = (int64_t)T + 2 * p;
    const int64_t frames = padded < wins[i] ? 0 : (padded - wins[i]) / shifts[i] + 1;
    const int64_t ch = ceil_div64(frames * C, TS_ITEMS);
    if (ch > chunks) chunks = ch;
  }
  const int half = avg_window / 2;
  const int64_t n = (int64_t)B * T * C;
  float* partial = scratch + 4 * n;       // [B][n_res][chunks]: chunks <= ceil((T + 1) * C / TS_ITEMS), since frames <= T + 1
  td_filter_masked_kernel<<<grid_for(2 * n), 256, 0, S_>>>(x_real, x_gen, T, C, n, valid_units, rows_per_unit, half, scratch);
  STG_LAUNCH_CHECK();
  td_score_partial_kernel<<<dim3((unsigned)chunks, B, n_res), TS_ITEMS, 0, S_>>>(scratch, T, C, n, valid_units, rows_per_unit,
                                                                                   half, rs, (int)chunks, partial);
  STG_LAUNCH_CHECK();
  td_score_finish_kernel<<<(B * n_res + 127) / 128, 128, 0, S_>>>(partial, valid_units, rows_per_unit, T, C, half, rs, B, n_res,
                                                                   (int)chunks, out);
  STG_LAUNCH_CHECK();
  return STG_OK;
}

extern "C" int stg_td_features(const float* x, int B, int T, int C, int win, int shift, int pad_windows, int avg_window,
                               float* feats, float* scratch, stg_stream_t stream) {
  TdRes r;
  if (!x || !feats || !scratch || !td_res(T, win, shift, pad_windows, &r)) return STG_EINVAL;
  if (avg_window < 1 || (avg_window & 1) == 0 || avg_window / 2 >= T) return STG_EINVAL;
  const int64_t n = (int64_t)B * T * C, total = (int64_t)B * r.frames * C;
  float *low = scratch, *hi = scratch + n;
  td_filter_kernel<<<grid_for(n), 256, 0, S_>>>(x, T, C, n, avg_window / 2, low, hi);
  STG_LAUNCH_CHECK();
  // stacked on the last axis: [mean(low), power(low), power(hi), mean(hi)]   (time_domain_loss.py:62-67)
  frame_stats_kernel<<<grid_for(total), 256, 0, S_>>>(low, B, T, C, r, feats, feats, 4, 0, 1);
  STG_LAUNCH_CHECK();
  frame_stats_kernel<<<grid_for(total), 256, 0, S_>>>(hi, B, T, C, r, feats, feats, 4, 3, 2);
  STG_LAUNCH_CHECK();
  return STG_OK;
}

extern "C" int stg_frame_stats(const float* x, int B, int T, int C, int win, int shift, int pad_windows, float* mean,
                               float* power, stg_stream_t stream) {
  TdRes r;
  if (!x || (!mean && !power) || !td_res(T, win, shift, pad_windows, &r)) return STG_EINVAL;
  frame_stats_kernel<<<grid_for((int64_t)B * r.frames * C), 256, 0, S_>>>(x, B, T, C, r, mean, power, 1, 0, 0);
  STG_LAUNCH_CHECK();
  return STG_OK;
}

extern "C" int stg_window_signal(const float* x, int B, int T, int C, int win, int shift, int pad_windows, float* out,
                                 stg_stream_t stream) {
  TdRes r;
  if (!x || !out || !td_res(T, win, shift, pad_windows, &r)) return STG_EINVAL;
  window_signal_kernel<<<grid_for((int64_t)B * r.frames * C * win), 256, 0, S_>>>(x, B, T, C, r, out);
  STG_LAUNCH_CHECK();
  return STG_OK;
}

extern "C" int stg_average_filter(const float* x, int64_t rows, int T, int window, int pad, float* out, stg_stream_t stream) {
  if (!x || !out || window < 1 || window > T) return STG_EINVAL;
  const int To = pad ? T : T - window + 1;
  average_filter_kernel<<<grid_for(rows * To), 256, 0, S_>>>(x, rows, T, window, pad, To, out);
  STG_LAUNCH_CHECK();
  return STG_OK;
}

extern "C" int stg_mse_const(const void* x, int dtype, int64_t n, float target, float* out_slot, float grad_scale,
                             void* dx, int dx_dtype, stg_stream_t stream) {
  if (!x || n < 1) return STG_EINVAL;
  const float gcoef = grad_scale * 2.f / (float)n;
  const int g = grid_for(n);
  if (dtype == STG_F32 && dx_dtype == STG_F32) mse_const_kernel<float, float><<<g, 256, 0, S_>>>((const float*)x, n, target, out_slot, gcoef, (float*)dx);
  else if (dtype == STG_F32) mse_const_kernel<float, bf16><<<g, 256, 0, S_>>>((const float*)x, n, target, out_slot, gcoef, (bf16*)dx);
  else if (dx_dtype == STG_F32) mse_const_kernel<bf16, float><<<g, 256, 0, S_>>>((const bf16*)x, n, target, out_slot, gcoef, (float*)dx);
  else mse_const_kernel<bf16, bf16><<<g, 256, 0, S_>>>((const bf16*)x, n, target, out_slot, gcoef, (bf16*)dx);
  STG_LAUNCH_CHECK();
  return STG_OK;
}

extern "C" int stg_l1_mean(const void* a, const void* b, int dtype, int64_t n, float* out_slot, float grad_scale,
                           void* da, stg_stream_t stream) {
  if (!a || !b || n < 1) return STG_EINVAL;
  const float gcoef = grad_scale / (float)n;
  const bool al = ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(da)) & 15) == 0;
  const int64_t n4 = al ? n / 4 : 0;
  if (dtype == STG_F32) l1_mean_kernel<float><<<grid_for(n, 4), 256, 0, S_>>>((const float*)a, (const float*)b, n4, n, out_slot, gcoef, (float*)da);
  else l1_mean_kernel<bf16><<<grid_for(n, 4), 256, 0, S_>>>((const bf16*)a, (const bf16*)b, n4, n, out_slot, gcoef, (bf16*)da);
  STG_LAUNCH_CHECK();
  return STG_OK;
}

extern "C" int stg_l1_mean_multi(const StgL1Item* items, int n_items, int dtype, float* out_slot, float grad_scale,
                                 stg_stream_t stream) {
  if (!items || n_items < 1 || n_items > STG_MAX_LOSS_ITEMS) return STG_EINVAL;
  L1Table t;
  t.n = n_items;
  int blocks = 0;
  for (int i = 0; i < n_items; ++i) {
    if (!items[i].a || !items[i].b || items[i].n < 1) return STG_EINVAL;
    t.it[i] = items[i];
    t.block0[i] = blocks;
    int64_t b = ceil_div64(items[i].n, 256 * 4 * 4);   // ~4 vector iterations per thread
    blocks += (int)(b < 1 ? 1 : (b > 148 ? 148 : b));
  }
  t.block0[n_items] = blocks;
  if (dtype == STG_F32) l1_mean_multi_kernel<float><<<blocks, 256, 0, S_>>>(t, out_slot, grad_scale);
  else if (dtype == STG_BF16) l1_mean_multi_kernel<bf16><<<blocks, 256, 0, S_>>>(t, out_slot, grad_scale);
  else return STG_EINVAL;
  STG_LAUNCH_CHECK();
  return STG_OK;
}

extern "C" int stg_mse_const_multi(const StgMseItem* items, int n_items, int x_dtype, int dx_dtype, float* slots,
                                   float grad_scale, stg_stream_t stream) {
  if (!items || n_items < 1 || n_items > STG_MAX_LOSS_ITEMS) return STG_EINVAL;
  MseTable t;
  t.n = n_items;
  int blocks = 0;
  for (int i = 0; i < n_items; ++i) {
    if (!items[i].x || items[i].n < 1) return STG_EINVAL;
    t.it[i] = items[i];
    t.block0[i] = blocks;
    int64_t b = ceil_div64(items[i].n, 256 * 4);
    blocks += (int)(b < 1 ? 1 : (b > 64 ? 64 : b));
  }
  t.block0[n_items] = blocks;
  if (x_dtype == STG_F32 && dx_dtype == STG_F32) mse_const_multi_kernel<float, float><<<blocks, 256, 0, S_>>>(t, slots, grad_scale);
  else if (x_dtype == STG_F32) mse_const_multi_kernel<float, bf16><<<blocks, 256, 0, S_>>>(t, slots, grad_scale);
  else if (dx_dtype == STG_F32) mse_const_multi_kernel<bf16, float><<<blocks, 256, 0, S_>>>(t, slots, grad_scale);
  else mse_const_multi_kernel<bf16, bf16><<<blocks, 256, 0, S_>>>(t, slots, grad_scale);
  STG_LAUNCH_CHECK();
  return STG_OK;
}
