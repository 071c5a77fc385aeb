// Kernels of the frozen EMG encoder's perceptual losses (SURVEY.md 8f rank 1; ste_gan/models/emg_encoder.py:36-88,
// ste_gan/layers/transformer.py:63-306, ste_gan/losses/emg_encoder_loss.py:56-84) that are not convolutions / GEMMs:
//   * LayerNorm forward / input-gradient (post-norm transformer layers, transformer.py:54-60)
//   * multi-head self-attention with per-head learned relative positional logits, forward and input-gradient
//     (transformer.py:87-113 + LearnedRelativePositionalEmbedding, unmasked, :163-306), fp32 arithmetic: one CTA per
//     (sample, head) with the operands in shared memory where they fit (the train step's T/16 = 100-128 frames at head dim
//     96), and band-tiled kernels for any sequence length
//   * speech-unit (mean pairwise L2 distance, eps 1e-6) and phoneme (cross-entropy) losses with their gradients
// The projections (q/k/v, output, feed-forward, w_raw_in / w_out / w_aux) and the strided ResBlocks with their eval-mode
// BatchNorm folded into weights and bias run on the tcgen05 convolution engine as k = 1 / k = 3 convs (passes_encoder.py).
// The encoder is frozen (emg_encoder_loss.py:61): only the gradient w.r.t. the EMG input exists.
#include "common.cuh"

namespace stg {
namespace {

__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max_f(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---------------------------------------------------------------------------------------------- LayerNorm
// one warp per row; stats[row] = (mean, rstd)
template <typename T>
__global__ void __launch_bounds__(256) layernorm_fwd_kernel(const T* __restrict__ x, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, int rows, int D, float eps,
                                                            T* __restrict__ y, float* __restrict__ stats) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const T* xr = x + (int64_t)row * D;
  float s = 0.f;
  for (int i = lane; i < D; i += 32) s += to_f(xr[i]);
  const float mean = warp_sum_f(s) / (float)D;
  float v = 0.f;
  for (int i = lane; i < D; i += 32) { const float d = to_f(xr[i]) - mean; v = fmaf(d, d, v); }
  const float rstd = rsqrtf(warp_sum_f(v) / (float)D + eps);
  T* yr = y + (int64_t)row * D;
  for (int i = lane; i < D; i += 32) yr[i] = from_f<T>((to_f(xr[i]) - mean) * rstd * gamma[i] + beta[i]);
  if (lane == 0 && stats) { stats[2 * row] = mean; stats[2 * row + 1] = rstd; }
}

// dx = rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dy * gamma,  xhat = (x - mean) * rstd      (+ add, if given)
template <typename T>
__global__ void __launch_bounds__(256) layernorm_bwd_kernel(const T* __restrict__ dy, const T* __restrict__ x,
                                                            const float* __restrict__ stats, const float* __restrict__ gamma,
                                                            int rows, int D, T* __restrict__ dx) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float mean = stats[2 * row], rstd = stats[2 * row + 1];
  const T* xr = x + (int64_t)row * D;
  const T* gr = dy + (int64_t)row * D;
  float s1 = 0.f, s2 = 0.f;
  for (int i = lane; i < D; i += 32) {
    const float g = to_f(gr[i]) * gamma[i], xh = (to_f(xr[i]) - mean) * rstd;
    s1 += g; s2 = fmaf(g, xh, s2);
  }
  s1 = warp_sum_f(s1) / (float)D; s2 = warp_sum_f(s2) / (float)D;
  T* o = dx + (int64_t)row * D;
  for (int i = lane; i < D; i += 32) {
    const float g = to_f(gr[i]) * gamma[i], xh = (to_f(xr[i]) - mean) * rstd;
    o[i] = from_f<T>(rstd * (g - s1 - xh * s2));
  }
}

// ---------------------------------------------------------------------------------------------- attention
// qkv [B][L][3*H*d] (q | k | v, each head-major), emb [H][2M-1][d] fp32, probs [B][H][L][L] fp32, o [B][L][H*d].
// logit(i, j) = q_i . k_j * scale + (|j - i| < M ? q_i . emb[h][j - i + M - 1] : -1e8)            (transformer.py:100-108,262-268)
struct AttnP { int B, L, H, d, M; float scale; };

template <typename T>
__device__ __forceinline__ void load_rows(const T* __restrict__ base, int64_t row_stride, int L, int d, int ds, float* __restrict__ dst) {
  for (int i = threadIdx.x; i < L * d; i += blockDim.x) {
    const int r = i / d, c = i - r * d;
    dst[r * ds + c] = to_f(base[(int64_t)r * row_stride + c]);
  }
}
__device__ __forceinline__ float dot4(const float4& a, const float4& b, float acc) {
  return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, fmaf(a.w, b.w, acc))));
}
__device__ __forceinline__ void axpy4(float s, const float4& v, float4& acc) {
  acc.x = fmaf(s, v.x, acc.x); acc.y = fmaf(s, v.y, acc.y); acc.z = fmaf(s, v.z, acc.z); acc.w = fmaf(s, v.w, acc.w);
}
template <typename T>
__device__ __forceinline__ void store4(T* p, const float4& v, float s) {
  p[0] = from_f<T>(v.x * s); p[1] = from_f<T>(v.y * s); p[2] = from_f<T>(v.z * s); p[3] = from_f<T>(v.w * s);
}

// Operand rows in shared memory are ds = d + 4 floats long: 16-byte aligned, and for d = 96 (ds = 100 = 4 mod 32 banks) the
// LDS.128 of 8 lanes that read 8 different rows hit 32 different banks.  Every product is register-blocked over AR = 4 rows of
// the side that is NOT spread over the lanes: a K / V / E / Q / dO row costs a lane one LDS.128 (4 shared-memory wavefronts)
// and is then used against 4 broadcast rows (1 wavefront each), i.e. 16 FMAs per ~8 wavefronts instead of 4 per ~9.
// History at B = 16, L = 100, d = 96 (per layer): scalar dots 203 us forward / 568 us backward -> float4 dots, 16 warps 115 / 241
// -> 4-row blocks: see DESIGN.md section 3.5.
constexpr int AR = 4;

// Key-length masks (kMask, stg_relattn_fwd_masked / stg_relattn_band_fwd_masked): sample b holds Lb = clamp(lengths[b], 0, L)
// rows.  Lb replaces L in every bound of the arithmetic (L stays the memory stride), so a kept row runs the loops, lanes and
// summation order of the same kernel at (B = 1, L = Lb) and is bit-identical to it; padded K / V rows are skipped, never
// multiplied by a zero probability (0 * NaN = NaN).  Query rows >= Lb get o = 0 and an all-zero probability row.
template <bool kMask>
__device__ __forceinline__ int valid_len(const int32_t* __restrict__ lengths, int b, int L) {
  if constexpr (kMask) return min(max(lengths[b], 0), L);
  return L;
}

// shared memory (floats): K [L][ds] | V [L][ds] | per warp: q [AR][d] + logits/probs [AR][Lp] + positional logits [AR][Lt]
// (d % 4 == 0, Lp = roundup4(L), Lt = roundup4(L + AR)); the head's embedding rows are read through L1.
template <typename T, bool kMask>
__global__ void __launch_bounds__(512, 1) relattn_fwd_kernel(const T* __restrict__ qkv, const float* __restrict__ emb, AttnP p,
                                                          T* __restrict__ o, float* __restrict__ probs,
                                                          const int32_t* __restrict__ lengths) {
  extern __shared__ __align__(16) float sm[];
  const int b = blockIdx.x / p.H, h = blockIdx.x - b * p.H;
  const int L = valid_len<kMask>(lengths, b, p.L), d = p.d, ds = d + 4, d4 = d >> 2, M = p.M, HD = p.H * d;
  const int Ls = p.L, Lp = (Ls + 3) & ~3, Lt = (Ls + AR + 3) & ~3;     // L: rows of the sample; Ls: rows in memory
  float* Ks = sm; float* Vs = Ks + L * ds; float* wsc = Vs + L * ds;
  const int nw = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* qs = wsc + warp * (AR * d + AR * Lp + AR * Lt); float* lg = qs + AR * d; float* ts = lg + AR * Lp;
  const float* Eh = emb + (int64_t)h * (2 * M - 1) * d;
  const T* base = qkv + (int64_t)b * Ls * 3 * HD + h * d;
  load_rows(base + HD, 3 * HD, L, d, ds, Ks);
  load_rows(base + 2 * HD, 3 * HD, L, d, ds, Vs);
  __syncthreads();
  if constexpr (kMask) {                                          // rows / keys past the sample's end: exactly 0
    for (int i = warp; i < Ls; i += nw) {
      float* pr = probs + (((int64_t)b * p.H + h) * Ls + i) * Ls;
      for (int j = (i < L ? L : 0) + lane; j < Ls; j += 32) pr[j] = 0.f;
      if (i >= L)
        for (int c = lane; c < d; c += 32) o[((int64_t)b * Ls + i) * HD + h * d + c] = from_f<T>(0.f);
    }
  }
  for (int ib = warp * AR; ib < L; ib += nw * AR) {
    const int nr = min(AR, L - ib);
    for (int x = lane; x < AR * d; x += 32) {
      const int r = x / d, c = x - r * d;
      qs[x] = r < nr ? to_f(base[(int64_t)(ib + r) * 3 * HD + c]) : 0.f;
    }
    __syncwarp();
    const float4* q4 = reinterpret_cast<const float4*>(qs);
    for (int j = lane; j < L; j += 32) {                          // q . k
      const float4* k4 = reinterpret_cast<const float4*>(Ks + j * ds);
      float acc[AR] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
      for (int c = 0; c < d4; ++c) {
        const float4 k = k4[c];
#pragma unroll
        for (int r = 0; r < AR; ++r) acc[r] = dot4(q4[r * d4 + c], k, acc[r]);
      }
#pragma unroll
      for (int r = 0; r < AR; ++r) lg[r * Lp + j] = acc[r] * p.scale;
    }
    // q . emb[rel] for every relative position the block can meet: rel = mi - (ib + AR - 1), i.e. j - i = rel for row i = ib + r
    // at j = mi - (AR - 1) + r
    for (int mi = lane; mi < L + AR - 1; mi += 32) {
      const int rel = mi - (ib + AR - 1);
      const bool in = rel > -M && rel < M;
      float acc[AR] = {0.f, 0.f, 0.f, 0.f};
      if (in) {
        const float4* e4 = reinterpret_cast<const float4*>(Eh + (int64_t)(rel + M - 1) * d);
#pragma unroll 2
        for (int c = 0; c < d4; ++c) {
          const float4 e = e4[c];
#pragma unroll
          for (int r = 0; r < AR; ++r) acc[r] = dot4(q4[r * d4 + c], e, acc[r]);
        }
      }
#pragma unroll
      for (int r = 0; r < AR; ++r) ts[r * Lt + mi] = in ? acc[r] : -1e8f;
    }
    __syncwarp();
    for (int r = 0; r < nr; ++r) {                                // softmax of row ib + r
      float* row = lg + r * Lp;
      const float* tr = ts + r * Lt + (AR - 1 - r);               // tr[j] = positional logit of (ib + r, j)
      float mx = -INFINITY;
      for (int j = lane; j < L; j += 32) { const float v = row[j] + tr[j]; row[j] = v; mx = fmaxf(mx, v); }
      mx = warp_max_f(mx);
      float sum = 0.f;
      for (int j = lane; j < L; j += 32) { const float e = __expf(row[j] - mx); row[j] = e; sum += e; }
      sum = warp_sum_f(sum);
      const float inv = 1.f / sum;
      float* pr = probs + (((int64_t)b * p.H + h) * Ls + ib + r) * Ls;
      for (int j = lane; j < L; j += 32) { const float pv = row[j] * inv; row[j] = pv; pr[j] = pv; }
    }
    __syncwarp();
    for (int c = lane; c < d4; c += 32) {                         // probs . v, 4 output channels per lane
      float4 acc[AR];
#pragma unroll
      for (int r = 0; r < AR; ++r) acc[r] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 2
      for (int j = 0; j < L; ++j) {
        const float4 v = *reinterpret_cast<const float4*>(Vs + j * ds + 4 * c);
#pragma unroll
        for (int r = 0; r < AR; ++r) axpy4(lg[r * Lp + j], v, acc[r]);
      }
      for (int r = 0; r < nr; ++r) store4(o + ((int64_t)b * Ls + ib + r) * HD + h * d + 4 * c, acc[r], 1.f);
    }
    __syncwarp();
  }
}

// shared memory (floats): Q | K | V | dO [L][ds] each | Dr [Lp] | per warp: dS block [AR][Lp]   (embedding rows through L1)
template <typename T>
__global__ void __launch_bounds__(512, 1) relattn_bwd_kernel(const T* __restrict__ qkv, const float* __restrict__ emb,
                                                          const float* __restrict__ probs, const T* __restrict__ dout, AttnP p,
                                                          T* __restrict__ dqkv) {
  extern __shared__ __align__(16) float sm[];
  const int b = blockIdx.x / p.H, h = blockIdx.x - b * p.H;
  const int L = p.L, d = p.d, ds = d + 4, d4 = d >> 2, M = p.M, HD = p.H * d, Lp = (L + 3) & ~3;
  float* Qs = sm; float* Ks = Qs + L * ds; float* Vs = Ks + L * ds; float* Gs = Vs + L * ds;
  float* Dr = Gs + L * ds; float* wsc = Dr + Lp;
  const float* Eh = emb + (int64_t)h * (2 * M - 1) * d;
  const int nw = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* dS = wsc + warp * AR * Lp;
  const T* base = qkv + (int64_t)b * L * 3 * HD + h * d;
  load_rows(base, 3 * HD, L, d, ds, Qs);
  load_rows(base + HD, 3 * HD, L, d, ds, Ks);
  load_rows(base + 2 * HD, 3 * HD, L, d, ds, Vs);
  load_rows(dout + (int64_t)b * L * HD + h * d, HD, L, d, ds, Gs);
  __syncthreads();
  const float* P = probs + ((int64_t)b * p.H + h) * L * L;
  T* dbase = dqkv + (int64_t)b * L * 3 * HD + h * d;
  // pass 1, a warp per block of AR query rows: dP_ij = dO_i . V_j ; D_i = sum_j dP_ij P_ij ; dS_ij = P_ij (dP_ij - D_i) ;
  //                                             dq_i = sum_j dS_ij (scale K_j + E[j - i])
  for (int ib = warp * AR; ib < L; ib += nw * AR) {
    const int nr = min(AR, L - ib);
    float dsum[AR] = {0.f, 0.f, 0.f, 0.f};
    for (int j = lane; j < L; j += 32) {
      const float4* v4 = reinterpret_cast<const float4*>(Vs + j * ds);
      float acc[AR] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
      for (int c = 0; c < d4; ++c) {
        const float4 v = v4[c];
#pragma unroll
        for (int r = 0; r < AR; ++r)
          acc[r] = dot4(*reinterpret_cast<const float4*>(Gs + min(ib + r, L - 1) * ds + 4 * c), v, acc[r]);
      }
#pragma unroll
      for (int r = 0; r < AR; ++r) {
        dS[r * Lp + j] = acc[r];
        if (r < nr) dsum[r] = fmaf(acc[r], P[(int64_t)(ib + r) * L + j], dsum[r]);
      }
    }
#pragma unroll
    for (int r = 0; r < AR; ++r) dsum[r] = warp_sum_f(dsum[r]);
    if (lane == 0)
      for (int r = 0; r < nr; ++r) Dr[ib + r] = dsum[r];
    for (int j = lane; j < L; j += 32)
#pragma unroll
      for (int r = 0; r < AR; ++r) dS[r * Lp + j] = r < nr ? P[(int64_t)(ib + r) * L + j] * (dS[r * Lp + j] - dsum[r]) : 0.f;
    __syncwarp();
    for (int c = lane; c < d4; c += 32) {
      float4 ak[AR], ae[AR];
#pragma unroll
      for (int r = 0; r < AR; ++r) { ak[r] = make_float4(0.f, 0.f, 0.f, 0.f); ae[r] = ak[r]; }
#pragma unroll 2
      for (int j = 0; j < L; ++j) {
        const float4 k = *reinterpret_cast<const float4*>(Ks + j * ds + 4 * c);
#pragma unroll
        for (int r = 0; r < AR; ++r) axpy4(dS[r * Lp + j], k, ak[r]);
      }
      for (int mi = 0; mi < L + AR - 1; ++mi) {                  // relative position rel meets row ib + r at j = mi - (AR - 1) + r
        const int rel = mi - (ib + AR - 1);
        if (rel <= -M || rel >= M) continue;
        const float4 e = *reinterpret_cast<const float4*>(Eh + (int64_t)(rel + M - 1) * d + 4 * c);
#pragma unroll
        for (int r = 0; r < AR; ++r) {
          const int j = mi - (AR - 1) + r;
          if (j >= 0 && j < L) axpy4(dS[r * Lp + j], e, ae[r]);
        }
      }
      for (int r = 0; r < nr; ++r) {
        float4 q = ak[r];
        q.x = q.x * p.scale + ae[r].x; q.y = q.y * p.scale + ae[r].y; q.z = q.z * p.scale + ae[r].z; q.w = q.w * p.scale + ae[r].w;
        store4(dbase + (int64_t)(ib + r) * 3 * HD + 4 * c, q, 1.f);
      }
    }
    __syncwarp();
  }
  __syncthreads();
  // pass 2, a warp per block of AR key rows: dS_ij recomputed from D_i ; dk_j = scale sum_i dS_ij q_i ; dv_j = sum_i P_ij dO_i
  for (int jb = warp * AR; jb < L; jb += nw * AR) {
    const int nr = min(AR, L - jb);
    for (int i = lane; i < L; i += 32) {
      const float4* g4 = reinterpret_cast<const float4*>(Gs + i * ds);
      float acc[AR] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
      for (int c = 0; c < d4; ++c) {
        const float4 g = g4[c];
#pragma unroll
        for (int r = 0; r < AR; ++r)
          acc[r] = dot4(g, *reinterpret_cast<const float4*>(Vs + min(jb + r, L - 1) * ds + 4 * c), acc[r]);
      }
      const float di = Dr[i];
#pragma unroll
      for (int r = 0; r < AR; ++r) dS[r * Lp + i] = r < nr ? P[(int64_t)i * L + jb + r] * (acc[r] - di) : 0.f;
    }
    __syncwarp();
    for (int c = lane; c < d4; c += 32) {
      float4 dk[AR], dv[AR];
#pragma unroll
      for (int r = 0; r < AR; ++r) { dk[r] = make_float4(0.f, 0.f, 0.f, 0.f); dv[r] = dk[r]; }
#pragma unroll 2
      for (int i = 0; i < L; ++i) {
        const float4 q = *reinterpret_cast<const float4*>(Qs + i * ds + 4 * c);
        const float4 g = *reinterpret_cast<const float4*>(Gs + i * ds + 4 * c);
#pragma unroll
        for (int r = 0; r < AR; ++r) {
          axpy4(dS[r * Lp + i], q, dk[r]);
          axpy4(r < nr ? P[(int64_t)i * L + jb + r] : 0.f, g, dv[r]);
        }
      }
      for (int r = 0; r < nr; ++r) {
        store4(dbase + (int64_t)(jb + r) * 3 * HD + HD + 4 * c, dk[r], p.scale);
        store4(dbase + (int64_t)(jb + r) * 3 * HD + 2 * HD + 4 * c, dv[r], 1.f);
      }
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------- band-tiled attention (any L)
// Out-of-band logits are -1e8, so exp(-1e8 - max) is exactly 0 in fp32 and the softmax over the band j in [i-M+1, i+M-1] n [0, L)
// IS the softmax over the row.  Probabilities are kept in band layout probs_band [B][H][L][W], W = 2M - 1: entry (i, w) is
// P(i, j = i + w - (M - 1)), exactly 0 where that j lies outside [0, L).
// One CTA per (query or key tile of BQT rows, head, sample); every warp owns one block of AR rows r0 .. r0 + AR - 1 and meets the
// partner rows r0 - M + 1 + s, slot s in [0, U), U = W + AR - 1.  Row r of a query block meets slot s at band entry w = s - r, row r
// of a key block at w = W - 1 - (s - r); either is in the band when 0 <= s - r < W.  The partner rows of the whole tile pass through
// shared memory in chunks of BKC rows, so shared memory depends on d and M only.  The arithmetic is the dense kernels', term for term.
constexpr int BNW = 8, BQT = BNW * AR, BKC = 64, BAND_D_MAX = 128, BAND_M_MAX = 256;
struct BandP { int L, H, d, M, W, U, Up; float scale; };

struct BandTile {               // the indices one warp of a band kernel works with
  int b, h, r0, nr, s0, lo, hi;
  int64_t bh;
  __device__ BandTile(const BandP& p) {
    b = blockIdx.z; h = blockIdx.y; bh = (int64_t)b * p.H + h;
    const int t0 = blockIdx.x * BQT;
    r0 = t0 + (threadIdx.x >> 5) * AR;
    nr = max(0, min(AR, p.L - r0));                      // rows of this warp's block inside [0, L) (0: the warp only syncs)
    s0 = r0 - p.M + 1;                                   // partner row of slot 0
    lo = max(0, t0 - p.M + 1); hi = min(p.L, t0 + BQT + p.M - 1);   // partner rows of the whole tile
  }
};

// this warp's AR rows (zero past row L - 1) of a [L][stride] operand -> dst [AR][d]
template <typename T>
__device__ __forceinline__ void load_block(const T* __restrict__ base, int64_t stride, int r0, int nr, int d, float* __restrict__ dst) {
  for (int x = threadIdx.x & 31; x < AR * d; x += 32) {
    const int r = x / d, c = x - r * d;
    dst[x] = r < nr ? to_f(base[(int64_t)(r0 + r) * stride + c]) : 0.f;
  }
  __syncwarp();
}

// shared memory (floats): partner chunk [BKC][ds] | per warp: q [AR][d] + logits/probs [AR][Up]      (embedding rows through L1)
template <typename T, bool kMask>
__global__ void __launch_bounds__(BNW * 32) relattn_band_fwd_kernel(const T* __restrict__ qkv, const float* __restrict__ emb,
                                                                    BandP p, T* __restrict__ o, float* __restrict__ probs,
                                                                    const int32_t* __restrict__ lengths) {
  extern __shared__ __align__(16) float sm[];
  const int L = valid_len<kMask>(lengths, blockIdx.z, p.L), Ls = p.L;  // L: rows of the sample; Ls: rows in memory
  BandTile t(p);
  if constexpr (kMask) {                                          // L replaces p.L in both bounds of the tile
    t.nr = max(0, min(AR, L - t.r0));
    t.hi = min(L, (int)blockIdx.x * BQT + BQT + p.M - 1);
  }
  const int d = p.d, ds = d + 4, d4 = d >> 2, M = p.M, W = p.W, U = p.U, Up = p.Up, HD = p.H * d;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nr = t.nr, s0 = t.s0;
  float* Cs = sm;
  float* qs = Cs + BKC * ds + warp * (AR * d + AR * Up); float* lg = qs + AR * d;
  const float* Eh = emb + (int64_t)t.h * W * d;
  const T* base = qkv + (int64_t)t.b * Ls * 3 * HD + t.h * d;
  if constexpr (kMask) {                                          // this warp's rows in [L, Ls): o = 0, probabilities 0
    for (int r = nr; r < min(AR, Ls - t.r0); ++r) {
      float* pr = probs + (t.bh * Ls + t.r0 + r) * W;
      for (int w = lane; w < W; w += 32) pr[w] = 0.f;
      for (int c = lane; c < d; c += 32) o[((int64_t)t.b * Ls + t.r0 + r) * HD + t.h * d + c] = from_f<T>(0.f);
    }
  }
  load_block(base, 3 * HD, t.r0, nr, d, qs);
  for (int x = lane; x < AR * Up; x += 32) lg[x] = 0.f;                 // every slot defined before the += below
  __syncwarp();
  const float4* q4 = reinterpret_cast<const float4*>(qs);
  for (int w = lane; w < W && nr > 0; w += 32) {                  // positional logits lg[r][w + r] = q_r . emb[w]
    const float4* e4 = reinterpret_cast<const float4*>(Eh + (int64_t)w * d);
    float acc[AR] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
    for (int c = 0; c < d4; ++c) {
      const float4 e = e4[c];
#pragma unroll
      for (int r = 0; r < AR; ++r) acc[r] = dot4(q4[r * d4 + c], e, acc[r]);
    }
#pragma unroll
    for (int r = 0; r < AR; ++r) lg[r * Up + w + r] = acc[r];
  }
  for (int c0 = t.lo; c0 < t.hi; c0 += BKC) {                     // + scale * q . k, key chunk by key chunk
    const int n = min(BKC, t.hi - c0);
    __syncthreads();
    load_rows(base + HD + (int64_t)c0 * 3 * HD, 3 * HD, n, d, ds, Cs);
    __syncthreads();
    if (nr == 0) continue;
    for (int j = max(c0, s0) + lane; j < min(c0 + n, s0 + U); j += 32) {
      const float4* k4 = reinterpret_cast<const float4*>(Cs + (j - c0) * ds);
      float acc[AR] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
      for (int c = 0; c < d4; ++c) {
        const float4 k = k4[c];
#pragma unroll
        for (int r = 0; r < AR; ++r) acc[r] = dot4(q4[r * d4 + c], k, acc[r]);
      }
#pragma unroll
      for (int r = 0; r < AR; ++r) lg[r * Up + j - s0] = __fmul_rn(acc[r], p.scale) + lg[r * Up + j - s0];   // slots off row r's
    }                                                                                                    // band: dropped below
  }
  __syncwarp();
  for (int r = 0; r < nr; ++r) {                                  // softmax of row i over its band
    float* row = lg + r * Up + r;                                 // row[w] = logit of band entry w
    const int i = t.r0 + r;
    float mx = -INFINITY;
    for (int w = lane; w < W; w += 32) {
      const int j = i + w - (M - 1);
      if (j >= 0 && j < L) mx = fmaxf(mx, row[w]);
    }
    mx = warp_max_f(mx);
    float sum = 0.f;
    for (int w = lane; w < W; w += 32) {
      const int j = i + w - (M - 1);
      const float e = j >= 0 && j < L ? __expf(row[w] - mx) : 0.f;
      row[w] = e; sum += e;
    }
    sum = warp_sum_f(sum);
    const float inv = 1.f / sum;
    float* pr = probs + (t.bh * Ls + i) * W;
    for (int w = lane; w < W; w += 32) { const float pv = row[w] * inv; row[w] = pv; pr[w] = pv; }
    for (int s = lane; s < U; s += 32)
      if (s < r || s >= r + W) lg[r * Up + s] = 0.f;
  }
  __syncwarp();
  float4 acc[AR];                                                 // probs . v, 4 output channels per lane (d <= 128)
#pragma unroll
  for (int r = 0; r < AR; ++r) acc[r] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int c0 = t.lo; c0 < t.hi; c0 += BKC) {
    const int n = min(BKC, t.hi - c0);
    __syncthreads();
    load_rows(base + 2 * HD + (int64_t)c0 * 3 * HD, 3 * HD, n, d, ds, Cs);
    __syncthreads();
    if (nr == 0 || lane >= d4) continue;
#pragma unroll 2
    for (int j = max(c0, s0); j < min(c0 + n, s0 + U); ++j) {
      const float4 v = *reinterpret_cast<const float4*>(Cs + (j - c0) * ds + 4 * lane);
#pragma unroll
      for (int r = 0; r < AR; ++r) axpy4(lg[r * Up + j - s0], v, acc[r]);
    }
  }
  if (lane < d4)
    for (int r = 0; r < nr; ++r) store4(o + ((int64_t)t.b * Ls + t.r0 + r) * HD + t.h * d + 4 * lane, acc[r], 1.f);
}

// Backward, query side: dP_ij = dO_i . v_j ; D_i = sum_j dP_ij P_ij (-> Dsc [B][H][L]) ; dS_ij = P_ij (dP_ij - D_i) ;
// dq_i = sum_j dS_ij (scale k_j + emb[w]).   shared memory (floats): chunk [BKC][ds] | per warp: dO [AR][d] + dP / dS [AR][Up]
template <typename T>
__global__ void __launch_bounds__(BNW * 32) relattn_band_bwd_q_kernel(const T* __restrict__ qkv, const float* __restrict__ emb,
                                                                      const float* __restrict__ probs, const T* __restrict__ dout,
                                                                      BandP p, T* __restrict__ dqkv, float* __restrict__ Dsc) {
  extern __shared__ __align__(16) float sm[];
  const BandTile t(p);
  const int L = p.L, d = p.d, ds = d + 4, d4 = d >> 2, M = p.M, W = p.W, U = p.U, Up = p.Up, HD = p.H * d;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nr = t.nr, s0 = t.s0;
  float* Cs = sm;
  float* gs = Cs + BKC * ds + warp * (AR * d + AR * Up); float* dS = gs + AR * d;
  const float* Eh = emb + (int64_t)t.h * W * d;
  const T* base = qkv + (int64_t)t.b * L * 3 * HD + t.h * d;
  load_block(dout + (int64_t)t.b * L * HD + t.h * d, HD, t.r0, nr, d, gs);
  for (int x = lane; x < AR * Up; x += 32) dS[x] = 0.f;                 // slots outside the window stay defined
  __syncwarp();
  const float4* g4 = reinterpret_cast<const float4*>(gs);
  for (int c0 = t.lo; c0 < t.hi; c0 += BKC) {                     // dP, value chunk by value chunk
    const int n = min(BKC, t.hi - c0);
    __syncthreads();
    load_rows(base + 2 * HD + (int64_t)c0 * 3 * HD, 3 * HD, n, d, ds, Cs);
    __syncthreads();
    if (nr == 0) continue;
    for (int j = max(c0, s0) + lane; j < min(c0 + n, s0 + U); j += 32) {
      const float4* v4 = reinterpret_cast<const float4*>(Cs + (j - c0) * ds);
      float acc[AR] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
      for (int c = 0; c < d4; ++c) {
        const float4 v = v4[c];
#pragma unroll
        for (int r = 0; r < AR; ++r) acc[r] = dot4(g4[r * d4 + c], v, acc[r]);
      }
#pragma unroll
      for (int r = 0; r < AR; ++r) dS[r * Up + j - s0] = acc[r];
    }
  }
  __syncwarp();
  for (int r = 0; r < nr; ++r) {
    const int i = t.r0 + r;
    const float* pr = probs + (t.bh * L + i) * W;
    float dsum = 0.f;
    for (int w = lane; w < W; w += 32) {
      const int j = i + w - (M - 1);
      if (j >= 0 && j < L) dsum = fmaf(dS[r * Up + w + r], pr[w], dsum);
    }
    dsum = warp_sum_f(dsum);
    if (lane == 0) Dsc[t.bh * L + i] = dsum;
    for (int s = lane; s < U; s += 32) {
      const int w = s - r, j = s0 + s;
      dS[r * Up + s] = w >= 0 && w < W && j >= 0 && j < L ? pr[w] * (dS[r * Up + s] - dsum) : 0.f;
    }
  }
  __syncwarp();
  float4 ak[AR], ae[AR];
#pragma unroll
  for (int r = 0; r < AR; ++r) { ak[r] = make_float4(0.f, 0.f, 0.f, 0.f); ae[r] = ak[r]; }
  if (nr > 0 && lane < d4)
    for (int w = 0; w < W; ++w) {                                 // band entry w of row r is slot w + r
      const float4 e = *reinterpret_cast<const float4*>(Eh + (int64_t)w * d + 4 * lane);
#pragma unroll
      for (int r = 0; r < AR; ++r) axpy4(dS[r * Up + w + r], e, ae[r]);
    }
  for (int c0 = t.lo; c0 < t.hi; c0 += BKC) {                     // + sum_j dS_ij k_j, key chunk by key chunk
    const int n = min(BKC, t.hi - c0);
    __syncthreads();
    load_rows(base + HD + (int64_t)c0 * 3 * HD, 3 * HD, n, d, ds, Cs);
    __syncthreads();
    if (nr == 0 || lane >= d4) continue;
#pragma unroll 2
    for (int j = max(c0, s0); j < min(c0 + n, s0 + U); ++j) {
      const float4 k = *reinterpret_cast<const float4*>(Cs + (j - c0) * ds + 4 * lane);
#pragma unroll
      for (int r = 0; r < AR; ++r) axpy4(dS[r * Up + j - s0], k, ak[r]);
    }
  }
  if (lane < d4)
    for (int r = 0; r < nr; ++r) {
      float4 q = ak[r];
      q.x = q.x * p.scale + ae[r].x; q.y = q.y * p.scale + ae[r].y; q.z = q.z * p.scale + ae[r].z; q.w = q.w * p.scale + ae[r].w;
      store4(dqkv + ((int64_t)t.b * L + t.r0 + r) * 3 * HD + t.h * d + 4 * lane, q, 1.f);
    }
}

// Backward, key side (after the query side has written D): dS_ij = P_ij (dO_i . v_j - D_i) ; dk_j = scale sum_i dS_ij q_i ;
// dv_j = sum_i P_ij dO_i.   shared memory (floats): chunk [BKC][ds] | per warp: v [AR][d] + dS [AR][Up] + P [AR][Up]
template <typename T>
__global__ void __launch_bounds__(BNW * 32) relattn_band_bwd_kv_kernel(const T* __restrict__ qkv, const float* __restrict__ probs,
                                                                       const T* __restrict__ dout, const float* __restrict__ Dsc,
                                                                       BandP p, T* __restrict__ dqkv) {
  extern __shared__ __align__(16) float sm[];
  const BandTile t(p);
  const int L = p.L, d = p.d, ds = d + 4, d4 = d >> 2, W = p.W, U = p.U, Up = p.Up, HD = p.H * d;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nr = t.nr, s0 = t.s0;
  float* Cs = sm;
  float* vs = Cs + BKC * ds + warp * (AR * d + 2 * AR * Up); float* dS = vs + AR * d; float* Pk = dS + AR * Up;
  const T* base = qkv + (int64_t)t.b * L * 3 * HD + t.h * d;
  load_block(base + 2 * HD, 3 * HD, t.r0, nr, d, vs);
  const float4* v4 = reinterpret_cast<const float4*>(vs);
  float4 dk[AR], dv[AR];
#pragma unroll
  for (int r = 0; r < AR; ++r) { dk[r] = make_float4(0.f, 0.f, 0.f, 0.f); dv[r] = dk[r]; }
  for (int c0 = t.lo; c0 < t.hi; c0 += BKC) {                     // dS and P of this chunk of queries, then dv
    const int n = min(BKC, t.hi - c0);
    __syncthreads();
    load_rows(dout + (int64_t)t.b * L * HD + t.h * d + (int64_t)c0 * HD, HD, n, d, ds, Cs);
    __syncthreads();
    if (nr == 0) continue;
    const int i_lo = max(c0, s0), i_hi = min(c0 + n, s0 + U);
    for (int i = i_lo + lane; i < i_hi; i += 32) {
      const float4* g4 = reinterpret_cast<const float4*>(Cs + (i - c0) * ds);
      float acc[AR] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
      for (int c = 0; c < d4; ++c) {
        const float4 g = g4[c];
#pragma unroll
        for (int r = 0; r < AR; ++r) acc[r] = dot4(g, v4[r * d4 + c], acc[r]);
      }
      const float* pr = probs + (t.bh * L + i) * W;
      const float di = Dsc[t.bh * L + i];
      const int s = i - s0;
#pragma unroll
      for (int r = 0; r < AR; ++r) {
        const int w = W - 1 - (s - r);
        const float pv = r < nr && w >= 0 && w < W ? pr[w] : 0.f;
        Pk[r * Up + s] = pv;
        dS[r * Up + s] = pv * (acc[r] - di);
      }
    }
    __syncwarp();
    if (lane < d4) {
#pragma unroll 2
      for (int i = i_lo; i < i_hi; ++i) {
        const float4 g = *reinterpret_cast<const float4*>(Cs + (i - c0) * ds + 4 * lane);
#pragma unroll
        for (int r = 0; r < AR; ++r) axpy4(Pk[r * Up + i - s0], g, dv[r]);
      }
    }
  }
  for (int c0 = t.lo; c0 < t.hi; c0 += BKC) {                     // dk, query chunk by query chunk
    const int n = min(BKC, t.hi - c0);
    __syncthreads();
    load_rows(base + (int64_t)c0 * 3 * HD, 3 * HD, n, d, ds, Cs);
    __syncthreads();
    if (nr == 0 || lane >= d4) continue;
#pragma unroll 2
    for (int i = max(c0, s0); i < min(c0 + n, s0 + U); ++i) {
      const float4 q = *reinterpret_cast<const float4*>(Cs + (i - c0) * ds + 4 * lane);
#pragma unroll
      for (int r = 0; r < AR; ++r) axpy4(dS[r * Up + i - s0], q, dk[r]);
    }
  }
  if (lane < d4)
    for (int r = 0; r < nr; ++r) {
      store4(dqkv + ((int64_t)t.b * L + t.r0 + r) * 3 * HD + HD + t.h * d + 4 * lane, dk[r], p.scale);
      store4(dqkv + ((int64_t)t.b * L + t.r0 + r) * 3 * HD + 2 * HD + t.h * d + 4 * lane, dv[r], 1.f);
    }
}

// ---------------------------------------------------------------------------------------------- losses
// one warp per (b, t) row.  slots[0] += mean_r || tgt_r - pred_r + 1e-6 ||_2          (F.pairwise_distance, eps 1e-6)
//                           slots[1] += mean_r -log softmax(logits_r)[target_r]       (F.cross_entropy)
// d_units = gs[0] * d slots[0] / d pred ; d_logits = gs[1] * d slots[1] / d logits
template <typename T>
__global__ void __launch_bounds__(256) encoder_loss_kernel(const float* __restrict__ pred, const float* __restrict__ tgt,
                                                           const float* __restrict__ logits, const int64_t* __restrict__ ph,
                                                           int N, int Du, int P, float* __restrict__ slots, float gs_u, float gs_p,
                                                           T* __restrict__ d_units, T* __restrict__ d_logits) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= N) return;
  const float inv_n = 1.f / (float)N;
  const float* pr = pred + (int64_t)r * Du; const float* tr = tgt + (int64_t)r * Du;
  float ss = 0.f;
  for (int i = lane; i < Du; i += 32) { const float df = tr[i] - pr[i] + 1e-6f; ss = fmaf(df, df, ss); }
  ss = warp_sum_f(ss);
  const float nrm = sqrtf(ss);
  if (d_units) {
    const float c = nrm > 0.f ? -gs_u * inv_n / nrm : 0.f;
    for (int i = lane; i < Du; i += 32) d_units[(int64_t)r * Du + i] = from_f<T>(c * (tr[i] - pr[i] + 1e-6f));
  }
  const float* lr = logits + (int64_t)r * P;
  float mx = -INFINITY;
  for (int i = lane; i < P; i += 32) mx = fmaxf(mx, lr[i]);
  mx = warp_max_f(mx);
  float se = 0.f;
  for (int i = lane; i < P; i += 32) se += __expf(lr[i] - mx);
  se = warp_sum_f(se);
  const int t = (int)ph[r];
  const float lse = mx + __logf(se);
  if (d_logits)
    for (int i = lane; i < P; i += 32)
      d_logits[(int64_t)r * P + i] = from_f<T>(gs_p * inv_n * (__expf(lr[i] - lse) - (i == t ? 1.f : 0.f)));
  if (lane == 0) {
    atomicAdd(slots, nrm * inv_n);
    atomicAdd(slots + 1, (lse - lr[t]) * inv_n);
  }
}

// Per-utterance scores (stg_encoder_scores): one CTA of SC_W warps per sample b over its n_b = clamp(lengths[b], 0, T) rows;
// warp w takes rows w, w + SC_W, ...  sums[b] = (sum_r ||tgt_r - pred_r + 1e-6||_2, sum_r CE_r); counts[b] = (rows, argmax ==
// target, target == silence, both and target != silence).  Per-warp partial sums in a fixed row order, then a fixed-order sum
// over the warps: no atomics, so replays are bit-identical.  A target outside [0, P) is not read through: its CE is NaN.
constexpr int SC_W = 8;
__global__ void __launch_bounds__(SC_W * 32) encoder_scores_kernel(const float* __restrict__ pred, const float* __restrict__ tgt,
                                                                   const float* __restrict__ logits, const int64_t* __restrict__ ph,
                                                                   const int32_t* __restrict__ lengths, int T, int Du, int P,
                                                                   int silence, float* __restrict__ sums, int32_t* __restrict__ counts) {
  __shared__ float s_sum[SC_W][2];
  __shared__ int s_cnt[SC_W][3];
  const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = min(max(lengths[b], 0), T);
  float su = 0.f, ce = 0.f;
  int correct = 0, sil = 0, correct_ns = 0;
  for (int t = warp; t < n; t += SC_W) {
    const int64_t row = (int64_t)b * T + t;
    const float* pr = pred + row * Du; const float* tr = tgt + row * Du;
    float ss = 0.f;
    for (int i = lane; i < Du; i += 32) { const float df = tr[i] - pr[i] + 1e-6f; ss = fmaf(df, df, ss); }
    su += sqrtf(warp_sum_f(ss));
    const float* lr = logits + row * P;
    float mx = -INFINITY;
    int arg = P;
    for (int i = lane; i < P; i += 32)
      if (lr[i] > mx || arg == P) { mx = lr[i]; arg = i; }                   // first maximum of this lane's entries
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {                                      // first maximum of the row (torch.argmax)
      const float m2 = __shfl_xor_sync(0xffffffffu, mx, o);
      const int a2 = __shfl_xor_sync(0xffffffffu, arg, o);
      if (m2 > mx || (m2 == mx && a2 < arg)) { mx = m2; arg = a2; }
    }
    float se = 0.f;
    for (int i = lane; i < P; i += 32) se += __expf(lr[i] - mx);
    se = warp_sum_f(se);
    const int64_t k = ph[row];
    const bool in = k >= 0 && k < P;
    ce += in ? mx + __logf(se) - lr[in ? k : 0] : __int_as_float(0x7fffffff);
    correct += arg == k;
    sil += k == silence;
    correct_ns += arg == k && k != silence;
  }
  if (lane == 0) {
    s_sum[warp][0] = su; s_sum[warp][1] = ce;
    s_cnt[warp][0] = correct; s_cnt[warp][1] = sil; s_cnt[warp][2] = correct_ns;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, c = 0.f;
    int k0 = 0, k1 = 0, k2 = 0;
    for (int w = 0; w < SC_W; ++w) { a += s_sum[w][0]; c += s_sum[w][1]; k0 += s_cnt[w][0]; k1 += s_cnt[w][1]; k2 += s_cnt[w][2]; }
    sums[2 * b] = a; sums[2 * b + 1] = c;
    counts[4 * b] = n; counts[4 * b + 1] = k0; counts[4 * b + 2] = k1; counts[4 * b + 3] = k2;
  }
}

}  // namespace
}  // namespace stg

using namespace stg;
#define S_ static_cast<cudaStream_t>(stream)

extern "C" int stg_layernorm_fwd(const void* x, int dtype, const float* gamma, const float* beta, int rows, int D, float eps,
                                 void* y, float* stats, stg_stream_t stream) {
  if (!x || !gamma || !beta || !y || rows < 1 || D < 1) return STG_EINVAL;
  const int blocks = (rows + 7) / 8;
  if (dtype == STG_F32) layernorm_fwd_kernel<float><<<blocks, 256, 0, S_>>>((const float*)x, gamma, beta, rows, D, eps, (float*)y, stats);
  else if (dtype == STG_BF16) layernorm_fwd_kernel<bf16><<<blocks, 256, 0, S_>>>((const bf16*)x, gamma, beta, rows, D, eps, (bf16*)y, stats);
  else return STG_EINVAL;
  STG_LAUNCH_CHECK();
  return STG_OK;
}

extern "C" int stg_layernorm_bwd(const void* dy, const void* x, int dtype, const float* stats, const float* gamma, int rows, int D,
                                 void* dx, stg_stream_t stream) {
  if (!dy || !x || !stats || !gamma || !dx || rows < 1 || D < 1) return STG_EINVAL;
  const int blocks = (rows + 7) / 8;
  if (dtype == STG_F32) layernorm_bwd_kernel<float><<<blocks, 256, 0, S_>>>((const float*)dy, (const float*)x, stats, gamma, rows, D, (float*)dx);
  else if (dtype == STG_BF16) layernorm_bwd_kernel<bf16><<<blocks, 256, 0, S_>>>((const bf16*)dy, (const bf16*)x, stats, gamma, rows, D, (bf16*)dx);
  else return STG_EINVAL;
  STG_LAUNCH_CHECK();
  return STG_OK;
}

static size_t attn_smem(int L, int d, int n_tiles, int per_warp, int extra, int n_warps) {
  const int ds = d + 4;
  return sizeof(float) * ((size_t)n_tiles * L * ds + extra + (size_t)n_warps * per_warp);
}
constexpr size_t ATTN_SMEM_MAX = 226 * 1024;

// Shared memory of the dense (one CTA per head) kernels at (L, d), with the warps they then run: 16 when the per-warp scratch
// fits beside the operand tiles, else 8.  0: the sequence is too long for them.  (Far past the limits of L and d: no int
// overflow below.)
static size_t dense_fwd_smem(int L, int d, int* nw) {
  if (L > (1 << 16) || d > 4096) return 0;
  const int Lp = (L + 3) & ~3;
  const int Lt = (L + 4 + 3) & ~3, pw = 4 * d + 4 * Lp + 4 * Lt;      // per-warp scratch (AR = 4 rows)
  *nw = 16;
  size_t smem = attn_smem(L, d, 2, pw, 0, *nw);
  if (smem > ATTN_SMEM_MAX) { *nw = 8; smem = attn_smem(L, d, 2, pw, 0, *nw); }
  return smem > ATTN_SMEM_MAX ? 0 : smem;
}
static size_t dense_bwd_smem(int L, int d, int* nw) {
  if (L > (1 << 16) || d > 4096) return 0;
  const int Lp = (L + 3) & ~3;
  *nw = 16;
  size_t smem = attn_smem(L, d, 4, 4 * Lp, Lp, *nw);
  if (smem > ATTN_SMEM_MAX) { *nw = 8; smem = attn_smem(L, d, 4, 4 * Lp, Lp, *nw); }
  return smem > ATTN_SMEM_MAX ? 0 : smem;
}

extern "C" int stg_relattn_dense_supported(int L, int d, int need_bwd) {
  int nw;
  if (L < 1 || d < 4 || (d & 3)) return 0;
  return dense_fwd_smem(L, d, &nw) != 0 && (!need_bwd || dense_bwd_smem(L, d, &nw) != 0);
}

template <typename T, bool kMask>
static int dense_fwd(const T* qkv, const float* emb, const AttnP& p, int nw, size_t smem, T* o, float* probs,
                     const int32_t* lengths, cudaStream_t s) {
  STG_CUDA_CHECK(cudaFuncSetAttribute(relattn_fwd_kernel<T, kMask>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  relattn_fwd_kernel<T, kMask><<<p.B * p.H, 32 * nw, smem, s>>>(qkv, emb, p, o, probs, lengths);
  STG_LAUNCH_CHECK();
  return STG_OK;
}

template <bool kMask>
static int relattn_fwd_any(const void* qkv, int dtype, const float* emb, int B, int L, int H, int d, int max_rel, float scale,
                           void* o, float* probs, const int32_t* lengths, cudaStream_t s) {
  if (!qkv || !emb || !o || !probs || B < 1 || L < 1 || H < 1 || d < 4 || (d & 3) || max_rel < 1) return STG_EINVAL;
  int nw;
  const size_t smem = dense_fwd_smem(L, d, &nw);
  if (!smem) return STG_EUNSUPPORTED;                   // sequence too long for the one-CTA-per-head kernel: stg_relattn_band_fwd
  if (dtype != STG_F32 && dtype != STG_BF16) return STG_EINVAL;
  AttnP p{B, L, H, d, max_rel, scale};
  if (dtype == STG_F32) return dense_fwd<float, kMask>((const float*)qkv, emb, p, nw, smem, (float*)o, probs, lengths, s);
  return dense_fwd<bf16, kMask>((const bf16*)qkv, emb, p, nw, smem, (bf16*)o, probs, lengths, s);
}

extern "C" int stg_relattn_fwd(const void* qkv, int dtype, const float* emb, int B, int L, int H, int d, int max_rel, float scale,
                               void* o, float* probs, stg_stream_t stream) {
  return relattn_fwd_any<false>(qkv, dtype, emb, B, L, H, d, max_rel, scale, o, probs, nullptr, S_);
}

extern "C" int stg_relattn_fwd_masked(const void* qkv, int dtype, const float* emb, int B, int L, int H, int d, int max_rel,
                                      float scale, void* o, float* probs, const int32_t* lengths, stg_stream_t stream) {
  if (!lengths) return STG_EINVAL;
  return relattn_fwd_any<true>(qkv, dtype, emb, B, L, H, d, max_rel, scale, o, probs, lengths, S_);
}

extern "C" int stg_relattn_bwd(const void* qkv, int dtype, const float* emb, const float* probs, const void* dout, int B, int L,
                               int H, int d, int max_rel, float scale, void* dqkv, stg_stream_t stream) {
  if (!qkv || !emb || !probs || !dout || !dqkv || B < 1 || L < 1 || H < 1 || d < 4 || (d & 3) || max_rel < 1) return STG_EINVAL;
  int nw;
  const size_t smem = dense_bwd_smem(L, d, &nw);
  if (!smem) return STG_EUNSUPPORTED;
  AttnP p{B, L, H, d, max_rel, scale};
  if (dtype == STG_F32) {
    STG_CUDA_CHECK(cudaFuncSetAttribute(relattn_bwd_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    relattn_bwd_kernel<float><<<B * H, 32 * nw, smem, S_>>>((const float*)qkv, emb, probs, (const float*)dout, p, (float*)dqkv);
  } else if (dtype == STG_BF16) {
    STG_CUDA_CHECK(cudaFuncSetAttribute(relattn_bwd_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    relattn_bwd_kernel<bf16><<<B * H, 32 * nw, smem, S_>>>((const bf16*)qkv, emb, probs, (const bf16*)dout, p, (bf16*)dqkv);
  } else return STG_EINVAL;
  STG_LAUNCH_CHECK();
  return STG_OK;
}

// Band kernels: argument checks, then the bounds of the kernels (d <= 128: one float4 of channels per lane; the grid's y / z
// dimensions).  The sequence length is not bounded.  Shared memory depends on d and max_rel only: <= 182 KB at the bounds.
static int band_params(int B, int L, int H, int d, int max_rel, float scale, BandP* p, dim3* grid) {
  if (B < 1 || L < 1 || H < 1 || d < 4 || (d & 3) || max_rel < 1) return STG_EINVAL;
  if (d > BAND_D_MAX || max_rel > BAND_M_MAX || B > 65535 || H > 65535) return STG_EUNSUPPORTED;
  const int W = 2 * max_rel - 1, U = W + AR - 1;
  *p = BandP{L, H, d, max_rel, W, U, (U + 3) & ~3, scale};
  *grid = dim3((unsigned)((L + BQT - 1) / BQT), (unsigned)H, (unsigned)B);
  return STG_OK;
}
static size_t band_smem(const BandP& p, int per_warp_rows) {
  return sizeof(float) * ((size_t)BKC * (p.d + 4) + (size_t)BNW * (AR * p.d + per_warp_rows * AR * p.Up));
}

template <typename T, bool kMask>
static int band_fwd(const T* qkv, const float* emb, const BandP& p, dim3 grid, T* o, float* probs, const int32_t* lengths,
                    cudaStream_t s) {
  const size_t smem = band_smem(p, 1);
  STG_CUDA_CHECK(cudaFuncSetAttribute(relattn_band_fwd_kernel<T, kMask>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  relattn_band_fwd_kernel<T, kMask><<<grid, BNW * 32, smem, s>>>(qkv, emb, p, o, probs, lengths);
  STG_LAUNCH_CHECK();
  return STG_OK;
}

template <typename T>
static int band_bwd(const T* qkv, const float* emb, const float* probs, const T* dout, const BandP& p, dim3 grid, T* dqkv,
                    float* scratch, cudaStream_t s) {
  const size_t sq = band_smem(p, 1), skv = band_smem(p, 2);
  STG_CUDA_CHECK(cudaFuncSetAttribute(relattn_band_bwd_q_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sq));
  STG_CUDA_CHECK(cudaFuncSetAttribute(relattn_band_bwd_kv_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)skv));
  relattn_band_bwd_q_kernel<T><<<grid, BNW * 32, sq, s>>>(qkv, emb, probs, dout, p, dqkv, scratch);
  STG_LAUNCH_CHECK();
  relattn_band_bwd_kv_kernel<T><<<grid, BNW * 32, skv, s>>>(qkv, probs, dout, scratch, p, dqkv);
  STG_LAUNCH_CHECK();
  return STG_OK;
}

template <bool kMask>
static int band_fwd_any(const void* qkv, int dtype, const float* emb, int B, int L, int H, int d, int max_rel, float scale, void* o,
                        float* probs_band, const int32_t* lengths, cudaStream_t s) {
  if (!qkv || !emb || !o || !probs_band || (dtype != STG_F32 && dtype != STG_BF16)) return STG_EINVAL;
  BandP p; dim3 grid;
  if (const int rc = band_params(B, L, H, d, max_rel, scale, &p, &grid)) return rc;
  if (dtype == STG_F32) return band_fwd<float, kMask>((const float*)qkv, emb, p, grid, (float*)o, probs_band, lengths, s);
  return band_fwd<bf16, kMask>((const bf16*)qkv, emb, p, grid, (bf16*)o, probs_band, lengths, s);
}

extern "C" int stg_relattn_band_fwd(const void* qkv, int dtype, const float* emb, int B, int L, int H, int d, int max_rel,
                                    float scale, void* o, float* probs_band, stg_stream_t stream) {
  return band_fwd_any<false>(qkv, dtype, emb, B, L, H, d, max_rel, scale, o, probs_band, nullptr, S_);
}

extern "C" int stg_relattn_band_fwd_masked(const void* qkv, int dtype, const float* emb, int B, int L, int H, int d, int max_rel,
                                           float scale, void* o, float* probs_band, const int32_t* lengths, stg_stream_t stream) {
  if (!lengths) return STG_EINVAL;
  return band_fwd_any<true>(qkv, dtype, emb, B, L, H, d, max_rel, scale, o, probs_band, lengths, S_);
}

extern "C" int stg_relattn_band_bwd(const void* qkv, int dtype, const float* emb, const float* probs_band, const void* dout, int B,
                                    int L, int H, int d, int max_rel, float scale, void* dqkv, float* scratch, stg_stream_t stream) {
  if (!qkv || !emb || !probs_band || !dout || !dqkv || !scratch || (dtype != STG_F32 && dtype != STG_BF16)) return STG_EINVAL;
  BandP p; dim3 grid;
  if (const int rc = band_params(B, L, H, d, max_rel, scale, &p, &grid)) return rc;
  if (dtype == STG_F32)
    return band_bwd((const float*)qkv, emb, probs_band, (const float*)dout, p, grid, (float*)dqkv, scratch, S_);
  return band_bwd((const bf16*)qkv, emb, probs_band, (const bf16*)dout, p, grid, (bf16*)dqkv, scratch, S_);
}

extern "C" int stg_encoder_losses(const float* unit_pred, const float* unit_target, const float* phoneme_logits,
                                  const int64_t* phoneme_target, int N, int Du, int P, float* slots, float gs_units, float gs_phonemes,
                                  void* d_units, void* d_logits, int grad_dtype, stg_stream_t stream) {
  if (!unit_pred || !unit_target || !phoneme_logits || !phoneme_target || !slots || N < 1 || Du < 1 || P < 1) return STG_EINVAL;
  const int blocks = (N + 7) / 8;
  if (grad_dtype == STG_F32) encoder_loss_kernel<float><<<blocks, 256, 0, S_>>>(unit_pred, unit_target, phoneme_logits, phoneme_target, N, Du, P, slots, gs_units, gs_phonemes, (float*)d_units, (float*)d_logits);
  else if (grad_dtype == STG_BF16) encoder_loss_kernel<bf16><<<blocks, 256, 0, S_>>>(unit_pred, unit_target, phoneme_logits, phoneme_target, N, Du, P, slots, gs_units, gs_phonemes, (bf16*)d_units, (bf16*)d_logits);
  else return STG_EINVAL;
  STG_LAUNCH_CHECK();
  return STG_OK;
}

extern "C" int stg_encoder_scores(const float* unit_pred, const float* unit_target, const float* phoneme_logits,
                                  const int64_t* phoneme_target, const int32_t* lengths, int B, int T, int Du, int P,
                                  int silence_index, float* sums, int32_t* counts, stg_stream_t stream) {
  if (!unit_pred || !unit_target || !phoneme_logits || !phoneme_target || !lengths || !sums || !counts) return STG_EINVAL;
  if (B < 1 || T < 1 || Du < 1 || P < 1 || B > (1 << 30)) return STG_EINVAL;
  encoder_scores_kernel<<<B, SC_W * 32, 0, S_>>>(unit_pred, unit_target, phoneme_logits, phoneme_target, lengths, T, Du, P,
                                                 silence_index, sums, counts);
  STG_LAUNCH_CHECK();
  return STG_OK;
}
