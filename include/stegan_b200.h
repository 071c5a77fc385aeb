/*
 * stegan_b200.h - C ABI of libstegan_b200.so: hand-written sm_100a kernels for the
 * STE-GAN hot path (generator + discriminator stacks + TD / LSGAN / feature-matching
 * losses, forward and backward).
 *
 * The reference (scheck-k/ste-gan) is 100 % Python and defines no FFI of its own: on
 * this path it dispatches into PyTorch (torch==2.0.1 + cuDNN 8.5, requirements.txt:51,97).
 * Each entry point below therefore cites the reference *call site* whose library
 * dispatch it replaces.  Plain pointers + sizes only; no torch types.  The caller
 * (PyTorch on the host side) owns every buffer; the library allocates nothing
 * persistent and never frees caller memory.  Every function enqueues work on
 * `stream` and returns 0, or a negative STG_E* code (see stg_strerror); the host
 * wrapper turns non-zero into a Python exception.  There is no CPU fallback.
 *
 * Layout convention: activations are CHANNELS-LAST, [B][T][C] with C contiguous
 * (the reference is [B][C][T]; the host wrapper converts at the module boundary).
 * A "period view" (DiscriminatorP's [B,C,T/p,p] Conv2d with (k,1) kernels,
 * models/discriminator.py:34-43,84-93) is the same memory addressed as B*p virtual
 * samples whose rows are p*C elements apart: `phases = p`.
 */
#ifndef STEGAN_B200_H_
#define STEGAN_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* stg_stream_t; /* cudaStream_t */

enum { STG_F32 = 0, STG_BF16 = 1 };
enum { STG_ACT_NONE = 0, STG_ACT_RELU = 1, STG_ACT_LEAKY = 2, STG_ACT_TANH = 3 };
enum {
  STG_OK = 0,
  STG_EINVAL = -1,      /* bad argument / unsupported shape */
  STG_ECUDA = -2,       /* CUDA runtime error (see stg_last_cuda_error) */
  STG_EUNSUPPORTED = -3 /* shape not supported by the requested engine */
};
enum { STG_ENGINE_AUTO = 0, STG_ENGINE_SIMT = 1, STG_ENGINE_TCGEN05 = 2, STG_ENGINE_MATVEC = 3 /* routing result only */ };

#define STG_MAX_TAPS 48

/*
 * One convolution-shaped contraction, used for forward, data-gradient and (with
 * stg_conv_wgrad) weight-gradient:
 *
 *   acc[n][r][c] = sum_{j<k} sum_{q<c_src/groups} src[n][row(r,j)][g(c)*c_src/groups + q] * w[j][c][q]
 *     forward   : row(r,j) = r*stride + j*dilation - pad
 *     transposed: row(r,j) = (r + pad - j*dilation) / stride  (tap skipped unless divisible)
 *   v = acc + bias[c]
 *   if pair_sum : v[r'] = v[2r'] + v[2r'+1]                 (backward of nearest-upsample x2)
 *   v = (v + add_pre[r][c]) * dact(mask[r][c]) + add_post[r >> post_shift][c]
 *   y_raw[r][c] = v ;  y_act[r (and 2r,2r+1 if dup_rows)][c] = act(v)
 *
 * Replaces: nn.Conv1d / nn.Conv2d((k,1)) dispatch at layers/conv.py:16-17,89-101 with the
 * elementwise neighbours of layers/conv.py:38-84 (ReLU, nn.Upsample, residual sums),
 * models/generator.py:133-137,160 (ReLU, tanh) and models/discriminator.py:40,64,90,116
 * (leaky_relu 0.1) fused in; `transposed` is the autograd conv backward-data of the same.
 */
typedef struct StgConv {
  int32_t dtype;      /* STG_F32 | STG_BF16 : storage type of src, w, add_*, mask, y_*; accumulation is fp32 */
  int32_t engine;     /* STG_ENGINE_* */
  int32_t n_samples;  /* B */
  int32_t phases;     /* period p (virtual samples = B*p), 1 for plain conv1d */
  int32_t t_src;      /* rows per virtual sample of src */
  int32_t t_dst;      /* rows per virtual sample of the accumulator (before pair_sum) */
  int32_t c_src;      /* channels of src (total) */
  int32_t c_dst;      /* channels of dst (total) */
  int32_t groups;
  int32_t k, dilation, stride, pad;
  int32_t transposed; /* 0 forward, 1 data-gradient */
  int32_t pair_sum;   /* 1: sum accumulator rows 2r,2r+1 -> output row r */
  int32_t post_shift; /* add_post row index = r >> post_shift */
  int32_t mask_mode;  /* STG_ACT_* whose derivative (as a function of its OUTPUT) multiplies v */
  int32_t act;        /* STG_ACT_* applied for y_act */
  int32_t dup_rows;   /* 1: y_act row r is written to rows 2r and 2r+1 (nearest-upsample x2) */
  int32_t out_f32;    /* 1: y_raw and y_act are float32 regardless of dtype */
  int32_t w_fwd_pack; /* transposed only: `w` is the FORWARD pack wf [k][c_out][c_in/groups] (= [k][c_src][c_dst/groups]);
                         the tcgen05 engine reads it as an MN-major operand, so no second (data-gradient) pack is needed.
                         The CUDA-core engine needs the data-gradient pack wd (w_fwd_pack = 0). */
  const void* src;
  const void* w;        /* packed [k][c_dst][c_src/groups] (see stg_weightnorm_fold), or the forward pack if w_fwd_pack */
  const float* bias;    /* [c_dst] or NULL */
  const void* add_pre;  /* [B][rows][c_dst] or NULL */
  const void* mask;     /* [B][rows][c_dst] or NULL */
  const void* add_post; /* [B][rows >> post_shift][c_dst] or NULL */
  void* y_raw;          /* or NULL */
  void* y_act;          /* or NULL */
} StgConv;

int stg_conv(const StgConv* d, stg_stream_t stream);

/*
 * stg_conv with per-sample length masks in the epilogue, for batches of utterances zero-padded to a common length:
 * accumulator row r of sample b is kept iff r < valid_units[b] * rows_per_unit; every other row is written as 0 to
 * y_raw and y_act (both 2r and 2r+1 when dup_rows).  The zero is a select, so whatever the padded rows of add_post or
 * src hold - NaN included - a masked output row is exactly 0.  When every layer of a stack masks its outputs, each
 * convolution reads zeros past a sample's end, which is the zero padding of that sample run on its own.
 * valid_units: DEVICE array of n_samples ints, read at execution time (a captured graph serves any length mix);
 * negative values count as 0, values past t_dst mask nothing.  Forward only: STG_EINVAL when valid_units is NULL,
 * rows_per_unit < 1, or the call is transposed, pair_sum or phases != 1.  Same engines and launch plan as stg_conv
 * (tcgen05 when stg_conv_tc_supported, otherwise the CUDA-core engine; never the 1-channel matvec kernels).
 */
int stg_conv_masked(const StgConv* d, const int32_t* valid_units, int32_t rows_per_unit, stg_stream_t stream);

/*
 * Weight gradient: dw[c][j][q] += sum_{n,r} dy[n][r][c] * x[n][r*stride + j*dilation - pad][g(c)*cin_g + q]
 * dw is float32 [c_out][k][c_in/groups] and is ACCUMULATED into (caller zeroes it).
 * Replaces the autograd conv backward-weight of the call sites listed for StgConv.
 */
typedef struct StgWgrad {
  int32_t dtype, engine;
  int32_t n_samples, phases, t_in, t_out, c_in, c_out, groups, k, dilation, stride, pad;
  const void* x;   /* [B][t_in*phases][c_in]  */
  const void* dy;  /* [B][t_out*phases][c_out] */
  float* dw;       /* [c_out][k][c_in/groups] */
  float* dbias;    /* [c_out] accumulated column sums of dy, or NULL */
} StgWgrad;

int stg_conv_wgrad(const StgWgrad* d, stg_stream_t stream);
/* Layout of dw the selected engine writes for this contraction: element (co, j, ci) at co*ld + j*span + goff(co) + ci.
 * CUDA-core engine and ungrouped convs: span = c_in/groups, ld = k*span, goff = 0 (compact).  tcgen05 engine on a
 * grouped conv: span = the input channels a 128-row output-channel tile meets ((128/cout_g)*cin_g, or cin_g when
 * cout_g >= 128), goff(co) = ((co/cout_g) % (128/cout_g))*cin_g; entries outside a row's own group are scratch.
 * dw must hold c_out*ld floats. */
int stg_wgrad_layout(const StgWgrad* d, int* ld, int* span);

/*
 * weight_norm (torch.nn.utils.weight_norm, dim 0; layers/conv.py:16-17,92,99):
 *   w = g * v / ||v||  per output channel; v is the torch layout [c_out][c_in/groups][k].
 * Emits the forward pack wf [k][c_out][c_in/pack_groups] and the data-gradient pack
 * wd [k][c_in][c_out/pack_groups] in `dtype`, and scale[c_out] = g/||v|| (fp32) for the backward.
 * pack_groups (0 = groups) divides groups: the packs then describe the same convolution with only
 * pack_groups groups whose per-group matrices are block-diagonal - this widens narrow groups to the
 * 64-channel K chunks of the tcgen05 engine (see stg_tc_pack_groups); pass the same number as
 * StgConv.groups.  flags & STG_PACK_UNFOLD (groups == 1): taps and channels form one K axis of
 * Kp = roundup8(k*c_in) elements, wf [c_out][Kp], wd [Kp][c_out] - the operand layouts of a 1-tap
 * convolution over stg_unfold rows (tiny-channel first layers).
 */
enum { STG_PACK_UNFOLD = 1 };
int stg_weightnorm_fold(const float* v, const float* g, int c_out, int cin_g, int k, int groups, int pack_groups,
                        int flags, int dtype, void* wf, void* wd, float* scale, stg_stream_t stream);
/* dw fp32 in the layout reported by stg_wgrad_layout: element (co, j, ci) at co*dw_ld + j*dw_span + goff(co) + ci
 * (dw_span 0 = cin_g, dw_ld 0 = k*dw_span: the compact [c_out][k][cin_g]) -> dv (torch layout) and dg;
 * ACCUMULATES into dv/dg when accumulate != 0. */
int stg_weightnorm_fold_bwd(const float* dw, int dw_ld, int dw_span, const float* v, const float* g, int c_out, int cin_g,
                            int k, int groups, float* dv, float* dg, int accumulate, stg_stream_t stream);

/*
 * spectral_norm (legacy torch.nn.utils.spectral_norm, layers/conv.py:94,101): when
 * `training`, one power iteration updating u[c_out], v[cin_g*k] in place (eps 1e-12), then
 * sigma = u^T W v, packs of W/sigma as above.  `sigma_out[0]` receives sigma.
 * scratch: float[c_out + cin_g*k + 8].  u_used / v_used (optional, [c_out] / [cin_g*k]): copies of the u, v THIS forward used,
 * for its backward (the module's buffers move on with the next forward's power iteration).
 */
int stg_spectralnorm_fold(const float* w_orig, float* u, float* v, int c_out, int cin_g, int k, int groups,
                          int pack_groups, int flags, int training, int dtype, void* wf, void* wd, float* sigma_out,
                          float* scratch, float* u_used, float* v_used, stg_stream_t stream);
/* d w_orig = dw/sigma - (sum(dw .* w_orig)/sigma^2) u v^T ; u, v, sigma are the values used by that forward. */
int stg_spectralnorm_fold_bwd(const float* dw, int dw_ld, int dw_span, const float* w_orig, const float* u, const float* v,
                              const float* sigma, int c_out, int cin_g, int k, int groups, float* dw_orig, int accumulate,
                              float* scratch, stg_stream_t stream);
/*
 * Multi-tensor forms: ONE launch sequence for all weight-normed convs of a network (45 in G, 31 in small D; the
 * per-layer calls above are launch-bound).  `items` is a DEVICE array of n_items entries ordered by row0 / tile0:
 *   row0  = running sum of c_out (one block per output channel), total_rows = its end value
 *   tile0 = running sum of pack tiles: k * pack_groups * ceil(c_out/pg/32) * ceil(c_in/pg/32), or for
 *           STG_PACK_UNFOLD ceil(c_out/32) * ceil(roundup8(k*c_in)/32); total_tiles = its end value
 * total_tiles <= 0 selects the row form (a warp per output-channel row, forward packs only); -total_tiles is then the
 * number of transposition blocks that build the K-major data-gradient packs wd of the grouped convs from their forward
 * packs: an item with wd != NULL has k * pg blocks, tile0 = running block count (items without wd: no blocks).
 * stg_weightnorm_fold_multi fills wf / wd / scale of every item; stg_weightnorm_fold_bwd_multi turns every
 * item's dw (layout dw_ld / dw_span, see stg_wgrad_layout) into dv / dg.
 */
typedef struct StgFoldItem {
  const float* v;      /* [c_out][cin_g][k] */
  const float* g;      /* [c_out] */
  void* wf;
  void* wd;            /* or NULL */
  float* scale;        /* [c_out] */
  const float* dw;     /* backward only */
  float* dv;
  float* dg;
  int32_t c_out, cin_g, k, groups, pg, flags, dw_ld, dw_span;
  int32_t row0, tile0;
} StgFoldItem;
int stg_weightnorm_fold_multi(const StgFoldItem* items, int n_items, int total_rows, int total_tiles, int dtype,
                              stg_stream_t stream);
int stg_weightnorm_fold_bwd_multi(const StgFoldItem* items, int n_items, int total_rows, int accumulate,
                                  stg_stream_t stream);
/* The same for the table rows [row_base, row_base + n_rows) only (rows = output channels, numbered through the items in
 * table order): the fold-backward of ONE gradient bucket, so that the data-parallel all-reduce of that bucket can start
 * while the backward pass of the layers in front of it is still running. */
int stg_weightnorm_fold_bwd_range(const StgFoldItem* items, int n_items, int row_base, int n_rows, int accumulate,
                                  stg_stream_t stream);

/* Number of groups the tcgen05 engine wants the packs of a (c_in, c_out, groups) convolution in (== groups
 * when no widening is needed or possible). */
int stg_tc_pack_groups(int c_in, int c_out, int groups);

/*
 * im2col rows for tiny-channel first layers (C_in = 8: models/discriminator.py:26,55,77,104): src [B][t_src*phases][C]
 * in `dtype` -> out [B][t_dst*phases][Kp], out[b][t*phases+ph][j*C + c] = src[b][(t*stride + j*dilation - pad)*phases + ph][c]
 * (0 outside the sample or for j*C + c >= k*C), Kp = roundup8(k*C).  stg_unfold_bwd is the adjoint:
 * dsrc (float32, ACCUMULATED) [B][t_src*phases][C] from dout [B][t_dst*phases][Kp] in `dtype`.
 */
int stg_unfold(const void* src, int dtype, int B, int phases, int t_src, int t_dst, int C, int k, int dilation, int stride,
               int pad, void* out, stg_stream_t stream);
int stg_unfold_bwd(const void* dout, int dtype, int B, int phases, int t_src, int t_dst, int C, int k, int dilation,
                   int stride, int pad, float* dsrc, stg_stream_t stream);

/* First layer of a period stack, fused (models/discriminator.py:26,36,77,86): reflect-pad right to a multiple of `period`,
 * [B,C,T/p,p] view, Conv2d(C -> c_out, (k,1), stride (stride,1), padding (pad,0)), bias, LeakyReLU(slope), from the fp32
 * input x [B][T][C] to the bf16 channels-last map y [B][H_out*period][c_out].  wf: the STG_PACK_UNFOLD forward pack
 * [c_out][roundup8(k*C)] in bf16.  Same values as stg_unfold + stg_conv on the tensor engine (bf16 operands, fp32 sums). */
int stg_period_first_layer(const float* x, const void* wf, const float* bias, int B, int T, int C, int period, int c_out,
                           int k, int stride, int pad, float slope, void* y, stg_stream_t stream);

/* models/generator.py:143-146,154: x0[b][t] = concat(units[b][t][0:d_units], emb[ids[b]][0:d_emb]) in `dtype`. */
int stg_embed_concat(const float* units, const float* emb, const int64_t* ids, int B, int T, int d_units, int d_emb,
                     int dtype, void* x0, stg_stream_t stream);
/* backward of the embedding branch: demb[ids[b]] += sum_t dx0[b][t][d_units:] (dx0 in `dtype`). */
int stg_embed_concat_bwd(const void* dx0, const int64_t* ids, int B, int T, int d_units, int d_emb, int dtype,
                         float* demb, stg_stream_t stream);

/*
 * Discriminator input preparation (models/discriminator.py:36,86 reflect pad right by p - T%p;
 * :140,153 AvgPool1d(4,2,1), count_include_pad).  x is float32 [B][T][C].
 */
int stg_reflect_pad_right(const float* x, int B, int T, int C, int T_pad, int dtype, void* out, stg_stream_t stream);
int stg_reflect_pad_right_bwd(const void* dout, int B, int T, int C, int T_pad, int dtype, float* dx, stg_stream_t stream);
int stg_avgpool4(const float* x, int B, int T, int C, float* out, stg_stream_t stream);           /* out [B][T/2][C] */
int stg_avgpool4_bwd(const float* dout, int B, int T, int C, float* dx, stg_stream_t stream);     /* dx += */
int stg_cast(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n, stg_stream_t stream);
/* out = dy * act'(y), the derivative expressed through the activation OUTPUT y (tanh of models/generator.py:160);
 * dy, y float32, out in `dtype`. */
int stg_act_bwd(const float* dy, const float* y, int mode, int64_t n, int dtype, void* out, stg_stream_t stream);
/* out[r (dup: 2r and 2r+1)] = relu(src[r]) over rows of C elements: the ReLU -> nn.Upsample(2) prologue of a GBlock used
 * on its own (layers/conv.py:38-40); inside the models the previous convolution's epilogue produces it. */
int stg_relu_rows(const void* src, int dtype, int64_t rows, int C, int dup, void* out, stg_stream_t stream);
/* out[r] = in[2r] + in[2r+1] over rows of C elements (backward of nearest-upsample x2). */
int stg_pair_sum_rows(const void* in, int64_t rows_out, int C, int dtype, void* out, stg_stream_t stream);
int stg_axpy_f32(float* y, const void* x, int x_dtype, float alpha, int64_t n, stg_stream_t stream); /* y += alpha*x */

/*
 * Multi-resolution time-domain feature loss (losses/time_domain_loss.py:13-107,
 * layers/average_filter.py:10-28).  x_real, x_gen float32 [B][T][C].  Writes
 * losses[0..2] (one per (win,shift) in {(20,8),(51,13),(80,16)}) and, if dx_gen != NULL,
 * ACCUMULATES sum_i grad_scale[i] * d losses[i] / d x_gen into dx_gen (grad_scale: 3 host floats).
 * scratch: float[ 6*B*T*C + 3 ].
 */
int stg_td_loss(const float* x_real, const float* x_gen, int B, int T, int C, float* losses, const float* grad_scale,
                float* dx_gen, float* scratch, stg_stream_t stream);
/* The same loss for ANY list of (win, shift) resolutions (n_res <= 8), with or without the reflect-padded windowing
 * (TimeDomainFeatureLoss.apply_padding_windowing) and any odd average-filter window - the constructor arguments of
 * losses/time_domain_loss.py:20-33.  The upstream gradients come from the host array grad_scale[n_res] or, when
 * grad_scale_dev != NULL, from a DEVICE array read at execution time (no host synchronisation inside autograd). */
int stg_td_loss_ex(const float* x_real, const float* x_gen, int B, int T, int C, int n_res, const int* wins,
                   const int* shifts, int pad_windows, int avg_window, float* losses, const float* grad_scale,
                   const float* grad_scale_dev, float* dx_gen, float* scratch, stg_stream_t stream);
/* Per-utterance TimeDomainFeatureLoss of a padded batch, forward only.  Sample b holds n_b = clamp(valid_units[b], 0,
 * T / rows_per_unit) * rows_per_unit rows (valid_units: DEVICE int32 [B], read at execution time, so a captured graph serves
 * any length mix - the convention of stg_conv_masked).  out[b][i] (float32 [B][n_res]) = TimeDomainFeatureLoss(wins[i],
 * shifts[i], pad_windows, avg_window).time_domain_loss(x_real[b, :n_b], x_gen[b, :n_b]): the filter reflects at n_b and the
 * L1 mean runs over the F_b * C * 4 features of an n_b-row signal.  No row >= n_b of either input is read (NaN there cannot
 * reach a kept value).  Where the reference's reflect padding raises (n_b <= avg_window / 2, or n_b <= win / 2 with padded
 * windows; zero-length samples included) or n_b is shorter than one window, out[b][i] is NaN.  Fixed-order sums without
 * atomics: a sample's value is bit-identical to the same call at B = 1, T = n_b, and across replays.
 * scratch: float[4*B*T*C + 8*B*ceil((T+1)*C/256)]; rows >= n_b of its filtered copies are neither written nor read.
 * STG_EINVAL (before any CUDA call): a NULL pointer, B, T or C < 1, n_res outside [1, 8], a win or shift < 1, an even or
 * non-positive avg_window, rows_per_unit < 1, T % rows_per_unit != 0.  STG_EUNSUPPORTED: B > 65535. */
int stg_td_scores(const float* x_real, const float* x_gen, int B, int T, int C, const int32_t* valid_units,
                  int32_t rows_per_unit, int n_res, const int* wins, const int* shifts, int pad_windows, int avg_window,
                  float* out, float* scratch, stg_stream_t stream);
/* TimeDomainFeatureLoss.calculate_time_domain_features (time_domain_loss.py:57-68): x [B][T][C] -> feats [B][F][C][4] =
 * [mean(low), sum(low^2), sum(hi^2), mean(hi)] per frame, low = avg(avg(x)), hi = |x - low|.  scratch: float[2*B*T*C]. */
int stg_td_features(const float* x, int B, int T, int C, int win, int shift, int pad_windows, int avg_window,
                    float* feats, float* scratch, stg_stream_t stream);
/* frame_means / frame_power (time_domain_loss.py:43-49): mean and sum of squares per frame, [B][F][C] each (either may
 * be NULL); window_signal (time_domain_loss.py:35-41): the frames themselves, out [B][F][C][win]. */
int stg_frame_stats(const float* x, int B, int T, int C, int win, int shift, int pad_windows, float* mean, float* power,
                    stg_stream_t stream);
int stg_window_signal(const float* x, int B, int T, int C, int win, int shift, int pad_windows, float* out,
                      stg_stream_t stream);
/* AverageFilter (layers/average_filter.py:10-28) on `rows` independent series of length T (float32):
 * reflect pad window/2 (if pad) then mean over `window`, stride 1. */
int stg_average_filter(const float* x, int64_t rows, int T, int window, int pad, float* out, stg_stream_t stream);

/*
 * LSGAN terms (ste_gan/train.py:192-196,209-211): out[slot] += mean((x - target)^2);
 * if dx != NULL, dx = grad_scale * 2 (x - target) / n   (written, `dx_dtype`).
 */
int stg_mse_const(const void* x, int dtype, int64_t n, float target, float* out_slot, float grad_scale, void* dx,
                  int dx_dtype, stg_stream_t stream);
/*
 * Feature matching (ste_gan/train.py:257-264): out[slot] += mean(|a - b|); if da != NULL,
 * da = grad_scale * sign(a - b) / n (written, `dtype`).
 */
int stg_l1_mean(const void* a, const void* b, int dtype, int64_t n, float* out_slot, float grad_scale, void* da,
                stg_stream_t stream);

/* Multi-tensor forms of the two above (27 feature-map pairs / 2 x 8 logits tensors per train step): one launch,
 * `items` is a HOST array (<= STG_MAX_LOSS_ITEMS) copied by value into the kernel parameters.
 *   l1 : out_slot[0] += sum_i mean|a_i - b_i| ; da_i = grad_scale * sign(a_i - b_i) / n_i
 *   mse: slots[slot_i] += mean((x_i - target_i)^2) ; dx_i = grad_scale * 2 (x_i - target_i) / n_i */
#define STG_MAX_LOSS_ITEMS 32
typedef struct StgL1Item { const void* a; const void* b; void* da; int64_t n; } StgL1Item;
typedef struct StgMseItem { const void* x; void* dx; int64_t n; float target; int32_t slot; } StgMseItem;
int stg_l1_mean_multi(const StgL1Item* items, int n_items, int dtype, float* out_slot, float grad_scale, stg_stream_t stream);
int stg_mse_const_multi(const StgMseItem* items, int n_items, int x_dtype, int dx_dtype, float* slots, float grad_scale,
                        stg_stream_t stream);

/*
 * EMG-encoder perceptual losses (SURVEY.md 8f rank 1): the pieces of the frozen encoder that are not convolutions / GEMMs.
 * The encoder is frozen (losses/emg_encoder_loss.py:61), so only input gradients exist.
 *
 * nn.LayerNorm over the last axis (layers/transformer.py:37-38,56,59): x, y [rows][D] in `dtype`; stats [rows][2] = (mean,
 * rstd) for the backward, which returns d/dx from dy, the PRE-norm input x and the stats.
 */
int stg_layernorm_fwd(const void* x, int dtype, const float* gamma, const float* beta, int rows, int D, float eps, void* y,
                      float* stats, stg_stream_t stream);
int stg_layernorm_bwd(const void* dy, const void* x, int dtype, const float* stats, const float* gamma, int rows, int D,
                      void* dx, stg_stream_t stream);
/*
 * MultiHeadAttention with LearnedRelativePositionalEmbedding (layers/transformer.py:87-113,163-306; unmasked, per-head
 * embeddings added to the keys): qkv [B][L][3*H*d] = (q | k | v), each [H][d] per row, in `dtype`; emb [H][2*max_rel-1][d]
 * float32; logit(i,j) = scale * q_i.k_j + (|j-i| < max_rel ? q_i.emb[h][j-i+max_rel-1] : -1e8); probs [B][H][L][L] float32
 * (softmax, kept for the backward); o [B][L][H*d] = probs * v.  The backward returns dqkv from dout = d/do.
 * One CTA per (sample, head) with its operands in shared memory, so L is bounded (STG_EUNSUPPORTED beyond):
 * stg_relattn_dense_supported tells which (L, d) these two calls take; stg_relattn_band_fwd/bwd take any L.
 */
int stg_relattn_fwd(const void* qkv, int dtype, const float* emb, int B, int L, int H, int d, int max_rel, float scale, void* o,
                    float* probs, stg_stream_t stream);
int stg_relattn_bwd(const void* qkv, int dtype, const float* emb, const float* probs, const void* dout, int B, int L, int H,
                    int d, int max_rel, float scale, void* dqkv, stg_stream_t stream);
/* Host-only, no GPU: 1 if stg_relattn_fwd (and, when need_bwd, stg_relattn_bwd) takes (L, d) - the smem rule those calls use
 * (d = 96: forward up to L = 206, backward up to 133). */
int stg_relattn_dense_supported(int L, int d, int need_bwd);
/*
 * The same attention at any sequence length, tiled over the band |j - i| < max_rel (out-of-band probabilities are exactly 0 in
 * fp32, so this is the same softmax), in the same fp32 arithmetic.  probs_band [B][H][L][2*max_rel-1] float32: entry (i, w) =
 * P(i, j = i + w - (max_rel - 1)), exactly 0 where that j lies outside [0, L).  The backward runs in two launches without atomics
 * (deterministic); scratch [B][H][L] float32 is caller-owned.  STG_EINVAL: a NULL pointer, d % 4 != 0, L < 1, max_rel < 1, an
 * unknown dtype.  STG_EUNSUPPORTED: d > 128, max_rel > 256, B or H > 65535.  L is not bounded.
 */
int stg_relattn_band_fwd(const void* qkv, int dtype, const float* emb, int B, int L, int H, int d, int max_rel, float scale,
                         void* o, float* probs_band, stg_stream_t stream);
int stg_relattn_band_bwd(const void* qkv, int dtype, const float* emb, const float* probs_band, const void* dout, int B, int L,
                         int H, int d, int max_rel, float scale, void* dqkv, float* scratch, stg_stream_t stream);
/*
 * The two forwards with per-sample key-length masks, for batches of utterances padded to a common length L: sample b holds
 * Lb = lengths[b] rows (a DEVICE array of B ints, read at execution time, so a captured graph serves any length mix; negative
 * counts as 0, more than L as L).  Lb replaces L in every bound of the kernel, so each row i < Lb is bit-identical to the same
 * call at B = 1, L = Lb; rows i >= Lb of o and of the probabilities are 0, and so are the probabilities of keys j >= Lb.  Padded
 * q / k / v rows are never read into a kept row, NaN included.  L stays the row stride of qkv, o and the probabilities.
 * Forward only.  STG_EINVAL on a NULL `lengths`, otherwise the arguments and return codes of the unmasked calls.
 */
int stg_relattn_fwd_masked(const void* qkv, int dtype, const float* emb, int B, int L, int H, int d, int max_rel, float scale,
                           void* o, float* probs, const int32_t* lengths, stg_stream_t stream);
int stg_relattn_band_fwd_masked(const void* qkv, int dtype, const float* emb, int B, int L, int H, int d, int max_rel, float scale,
                                void* o, float* probs_band, const int32_t* lengths, stg_stream_t stream);
/*
 * EMGEncoderLoss (losses/emg_encoder_loss.py:63-84) over N = B*T rows: slots[0] += mean_r ||target_r - pred_r + 1e-6||_2
 * (F.pairwise_distance), slots[1] += mean_r cross_entropy(logits_r, phoneme_r); d_units / d_logits (`grad_dtype`, may be
 * NULL) = gs_units * d slots[0] / d pred and gs_phonemes * d slots[1] / d logits.
 */
int stg_encoder_losses(const float* unit_pred, const float* unit_target, const float* phoneme_logits,
                       const int64_t* phoneme_target, int N, int Du, int P, float* slots, float gs_units, float gs_phonemes,
                       void* d_units, void* d_logits, int grad_dtype, stg_stream_t stream);
/*
 * EMGEncoderLoss per utterance of a padded batch (losses/emg_encoder_loss.py:19-84): unit_pred / unit_target [B][T][Du],
 * phoneme_logits [B][T][P] float32, phoneme_target [B][T] int64; sample b holds n = clamp(lengths[b], 0, T) frames (DEVICE
 * int32 [B]) and rows t >= n are never read.  sums [B][2] = (sum_t ||target_t - pred_t + 1e-6||_2, sum_t cross_entropy_t);
 * counts [B][4] int32 = (n, argmax_t == target_t, target_t == silence_index, both of those and target_t != silence_index);
 * argmax takes the first maximum, as torch.argmax.  A target outside [0, P) makes that utterance's cross-entropy sum NaN.
 * Fixed-order reductions without atomics: replays are bit-identical.  STG_EINVAL: a NULL pointer, B, T, Du or P < 1.
 */
int stg_encoder_scores(const float* unit_pred, const float* unit_target, const float* phoneme_logits,
                       const int64_t* phoneme_target, const int32_t* lengths, int B, int T, int Du, int P, int silence_index,
                       float* sums, int32_t* counts, stg_stream_t stream);

/* torch.optim.AdamW (ste_gan/constants.py:57; train.py:80-81,199,267) over one flat fp32 buffer.
 * step_count is a device int64 (incremented by the kernel) so the update is CUDA-graph capturable.
 * lr_dev (device float[1], or NULL to use the host value `lr`): the learning rate is read on the device at execution
 * time, so the reference's per-epoch ExponentialLR(.999) (train.py:98-104,470-472) changes it between replays of a
 * captured graph.
 * enable (device int32[1], or NULL = always): when *enable == 0 the whole update - step counter included - is skipped;
 * after an executed update the flag is cleared.  This lets ONE captured graph hold "apply the previous step's generator
 * gradient, if there is one" at its head (where it overlaps work that does not depend on the generator).
 * flags & STG_ADAMW_KEEP_STEP: do not increment step_count - the update of a SLICE of a network whose first slice already
 * counted this optimiser step (gradient buckets are updated one by one, each right behind its all-reduce). */
enum { STG_ADAMW_KEEP_STEP = 1 };
int stg_adamw(float* p, const float* g, float* m, float* v, int64_t n, float lr, const float* lr_dev, float beta1,
              float beta2, float eps, float weight_decay, int64_t* step_count, float grad_scale, int32_t* enable,
              int flags, stg_stream_t stream);

/* diagnostics */
const char* stg_strerror(int code);
const char* stg_last_cuda_error(void);
int stg_version(void);
/* number of CUDA kernels this library has launched in this process (bench.py's gpu_launches) */
unsigned long long stg_launch_count(void);
/* Upper bound on the SMs the persistent tcgen05 kernels occupy from now on (0 = all).  The data-parallel trainer lowers
 * it while it captures the graphs that run beside a gradient all-reduce, so that the communicator's CTAs find free SMs. */
void stg_set_sm_limit(int n_sms);
/* 1 if the tcgen05 engine can take this contraction (shape/alignment rules in DESIGN.md), else 0. */
int stg_conv_tc_supported(const StgConv* d);
int stg_wgrad_tc_supported(const StgWgrad* d);
/* engine a call will run on (STG_ENGINE_SIMT / _TCGEN05 / _MATVEC: the 1-channel logits kernels) */
int stg_conv_route(const StgConv* d);
int stg_wgrad_route(const StgWgrad* d);
/* debug: device buffer of 1 + 3*4000 int64 that receives a (tag, value, globaltimer ns) timeline of CTA 0 of every
 * following tcgen05 stg_conv launch (NULL switches it off). */
int stg_debug_set_trace(void* buf);
/* debug hardware probe (csrc/debug_probe.cu): one 128x64x64 MMA whose A operand starts `shift` rows into a TMA-loaded
 * [rows_a][64] bf16 tile, descriptor base-offset field = base_off; out = float [128][64]. */
int stg_debug_rowshift(const void* x, const void* w, int rows_a, int shift, int base_off, float* out, stg_stream_t stream);
/* debug hardware probe (csrc/debug_probe.cu): the per-group MMAs of a grouped convolution - A [128][64] bf16 with 64/cin_g
 * groups side by side on K, W compact [(64/cin_g)*cout_g][cin_g] loaded with a 32- / 64- / 128-byte swizzle, one N = cout_g
 * MMA chain per group into its own accumulator columns; out = float [128][(64/cin_g)*cout_g]. */
int stg_debug_group_mma(const void* x, const void* w, int cin_g, int cout_g, float* out, stg_stream_t stream);
/* Host-only diagnostic: row classes of the tcgen05 convolution for t_dst output rows per sample (128-row tiles + binary
 * tail tiles that gather one row slice of several samples).  out[3c..3c+2] = rows per sample, first row, tiles per sample
 * (0: one tile per 128/rows samples); returns the number of classes (<= 4).  No GPU needed. */
int stg_debug_row_classes(int t_dst, int* out);
/* debug hardware probe (csrc/debug_probe.cu): bytes per clock one SM ingests through TMA while `grid` SMs pull
 * [box_rows][64] bf16 boxes of an L2-resident buffer [n_rows][64] at once, from disjoint rows (mode 0) or all from the same
 * rows (mode 1), through a `stages`-deep ring; clk[cta] = clocks for n_iters boxes. */
int stg_debug_tma_bw(const void* buf, long long n_rows, int box_rows, int n_iters, int mode, int stages, int grid, long long* clk,
                     stg_stream_t stream);
/* Host-only diagnostic: the plan the tcgen05 convolution engine would launch for `d` (only the geometry is read; pointers
 * just need to be non-NULL where the call would use them).  out[15] = { column tile bn, staged epilogue, taps per stage (tap
 * window), main-loop stages, dynamic shared memory bytes, two CTAs per SM, row classes, tiles, grid, compact-group K (0: none),
 * 64-channel chunks per tap, TMEM columns, epilogue-operand ring depth (0: no operands), output ring depth, output-row
 * residue classes }.  STG_EUNSUPPORTED when the engine does not take the shape.  No GPU needed. */
int stg_debug_conv_plan(const StgConv* d, int* out);
/* debug accounting (host side): bytes the tcgen05 launches since the last reset were planned to pull into shared memory
 * through TMA (main-loop operands + epilogue operands). */
double stg_debug_ingest_bytes(int reset);

#ifdef __cplusplus
}
#endif
#endif /* STEGAN_B200_H_ */
