"""Fused forward / input-gradient pass of the FROZEN EMG encoder and its two perceptual losses (SURVEY.md 8f rank 1).

Reference: EMGEncoderTransformer.forward in eval mode (ste_gan/models/emg_encoder.py:71-88), ResBlock
(layers/conv.py:106-132), TransformerEncoderLayer / MultiHeadAttention with learned relative positional logits
(layers/transformer.py:45-113,163-306), EMGEncoderLoss (losses/emg_encoder_loss.py:56-84), called from the generator step at
ste_gan/train.py:219-230.

What runs where (channels-last [B, T, C] activations, bf16 production / fp32 validation, like the GAN passes):
  * The encoder is frozen, so its operands are packed ONCE (EncoderPlan): every eval-mode BatchNorm is folded into the
    weights and bias of the conv in front of it (y = (conv(x) + b - mean) * gamma / sqrt(var + eps) + beta), the per-head
    q / k / v projections become ONE 768 -> 2304 GEMM and the per-head output projection one 768 -> 768 GEMM.
  * Convs and GEMMs = k = 3 / k = 1 launches of the tcgen05 convolution engine with their neighbours in the epilogue: ReLU,
    the ResBlock sum (add_post), the transformer residuals (add_post), ReLU derivatives as masks read from the saved
    outputs.  The 8-channel first block runs as 1-tap convs over im2col rows like the discriminators' first layers.
  * LayerNorm, attention (+ relative positional logits + softmax) and the two losses: csrc/encoder.cu.
Only the gradient w.r.t. the EMG input is produced - no weight gradients exist for a frozen network.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Tuple

import torch

from . import ops
from .ops import ACT_NONE, ACT_RELU
from .passes import Folded, _dgrad, _fwd, unfold_input

Tensor = torch.Tensor
BN_EPS, LN_EPS = 1e-5, 1e-5


class FrozenConv:
    """The attributes passes._fwd / _dgrad read from a conv module, for a frozen (pre-folded) weight."""
    norm, groups, dilation = "frozen", 1, 1

    def __init__(self, c_in: int, c_out: int, k: int, stride: int, pad: int, bias: Tensor):
        self.in_channels, self.out_channels, self.kernel, self.stride, self.pad = c_in, c_out, k, stride, pad
        self.bias = bias            # fp32 [c_out]; `.data` of a plain tensor is the tensor itself

    def t_out(self, t_in: int) -> int:
        return (t_in + 2 * self.pad - (self.kernel - 1) - 1) // self.stride + 1


def _pack(w: Tensor, b: Tensor, stride: int, pad: int, dtype: torch.dtype) -> Folded:
    """torch conv weight [c_out, c_in, k] (fp32, already final) -> packed operands of the convolution engines.  One-time host-side
    setup of a frozen network (plain tensor permutes), not on the step's hot path."""
    c_out, c_in, k = w.shape
    mod = FrozenConv(c_in, c_out, k, stride, pad, b.contiguous().float())
    unf = c_in < 16 and c_out >= 32          # tiny-channel first block: one K axis of (tap, channel), see passes.pack_mode
    if unf:
        kp = ops.round_up8(k * c_in)
        wf = torch.zeros(c_out, kp, device=w.device, dtype=torch.float32)
        wf[:, :k * c_in] = w.permute(0, 2, 1).reshape(c_out, k * c_in)          # q = j * c_in + c
        return Folded(mod, wf.to(dtype).contiguous(), wf.t().to(dtype).contiguous(), dtype, unfold=True, kp=kp)
    wf = w.permute(2, 0, 1).contiguous().to(dtype)                              # [k][c_out][c_in]
    wd = w.permute(2, 1, 0).contiguous().to(dtype) if dtype != torch.bfloat16 else None     # [k][c_in][c_out] (CUDA-core engine)
    return Folded(mod, wf, wd, dtype)


def _bn_fold(conv, bn) -> Tuple[Tensor, Tensor]:
    """eval-mode BatchNorm1d folded into the conv in front of it (conv.py:111-118)."""
    scale = bn.weight.data / torch.sqrt(bn.running_var + BN_EPS)
    return conv.weight.data * scale[:, None, None], (conv.bias.data - bn.running_mean) * scale + bn.bias.data


@dataclass
class _Layer:
    qkv: Folded
    out: Folded
    l1: Folded
    l2: Folded
    emb: Tensor
    g1: Tensor
    b1: Tensor
    g2: Tensor
    b2: Tensor
    n_head: int
    max_rel: int


class EncoderPlan:
    def __init__(self, enc, dtype: torch.dtype):
        self.dtype = dtype
        self.device = enc.w_out.weight.device
        if self.device.type != "cuda":
            raise RuntimeError("EMG encoder: move the module to a CUDA device first (there is no CPU path)")
        lin = lambda m: _pack(m.weight.data[:, :, None], m.bias.data, 1, 0, dtype)
        self.blocks = []
        for blk in enc.conv_blocks:
            c1 = _pack(*_bn_fold(blk.conv1, blk.bn1), blk.stride, 1, dtype)
            c2 = _pack(*_bn_fold(blk.conv2, blk.bn2), 1, 1, dtype)
            res = _pack(*_bn_fold(blk.residual_path, blk.res_norm), blk.stride, 0, dtype) if blk.residual_path is not None else None
            self.blocks.append((c1, c2, res))
        self.frame_rows = 1                 # EMG rows per encoder frame: the product of the ResBlock strides (16)
        for c1, _, _ in self.blocks:
            self.frame_rows *= c1.mod.stride
        self.w_in = lin(enc.w_raw_in)
        self.layers: List[_Layer] = []
        for lyr in enc.transformer.layers:
            a = lyr.self_attn
            H, D, d = a.w_q.shape
            # q / k / v of all heads as one [3*H*d, D] weight: row (which, h, a) = w_which[h, :, a]      (transformer.py:96-98)
            w_qkv = torch.cat([w.data.permute(0, 2, 1).reshape(H * d, D) for w in (a.w_q, a.w_k, a.w_v)], 0)
            # out[f] = sum_{h,a} o[h,a] w_o[h,a,f]                                                       (transformer.py:112)
            w_o = a.w_o.data.reshape(H * d, D).t()
            zeros = lambda n: torch.zeros(n, device=self.device)
            self.layers.append(_Layer(
                qkv=_pack(w_qkv[:, :, None], zeros(3 * H * d), 1, 0, dtype), out=_pack(w_o[:, :, None], zeros(D), 1, 0, dtype),
                l1=lin(lyr.linear1), l2=lin(lyr.linear2),
                emb=a.relative_positional.embeddings.data[..., 0].contiguous().float(),
                g1=lyr.norm1.weight.data.float().contiguous(), b1=lyr.norm1.bias.data.float().contiguous(),
                g2=lyr.norm2.weight.data.float().contiguous(), b2=lyr.norm2.bias.data.float().contiguous(),
                n_head=H, max_rel=a.relative_positional.max_relative_pos))
        self.w_out, self.w_aux = lin(enc.w_out), lin(enc.w_aux)


@dataclass
class EncCtx:
    B: int
    T: int
    blocks: list
    y_last: Tensor
    t_last: int
    layers: list
    x_final: Tensor


def _src(f: Folded, x: Tensor, B: int, t: int) -> Tensor:
    return unfold_input(f, x, B, t) if f.unfold else x


def encoder_forward(plan: EncoderPlan, emg: Tensor, need_ctx: bool = True, lengths: Optional[Tensor] = None):
    """emg fp32 [B, T, C] -> (speech-unit prediction fp32 [B, T/16, 256], phoneme logits fp32 [B, T/16, P], ctx).
    lengths (int32 [B] on the device, frames; forward only): sample b is an utterance of lengths[b] frames (16 * lengths[b]
    EMG rows) padded to T / 16 frames with anything, NaN included.  Rows [0, lengths[b]) of both heads are what the utterance
    gives on its own, the rows after them are 0.  Why output masks alone make this exact: every conv writes 0 at its rows
    past the sample's end (rates of 8, 4, 2, 1 rows per frame after blocks 1-4), so each conv reads 0 there, which is the
    zero padding the utterance gets alone.  Only conv2 of a ResBlock (k = 3, pad 1, stride 1) reads a row past the end, and
    that row is conv1's masked output.  The stride-2 convs on even lengths read rows <= 2o + 1 (k = 3, pad 1) or 2o (k = 1)
    for a kept output row o: all inside the sample.  The transformer is row-local except attention, which skips the padded
    keys (stg_relattn_fwd_masked); the padded rows of the LayerNorm outputs hold beta, but no kept row reads them."""
    if lengths is not None:
        if need_ctx:
            raise ValueError("encoder_forward: length masks are forward-only (need_ctx=True with lengths)")
        if emg.shape[1] % plan.frame_rows != 0:
            raise ValueError(f"encoder_forward: with lengths, T = {emg.shape[1]} must be a multiple of {plan.frame_rows} "
                             "(EMG rows per frame)")
    dt = plan.dtype
    x = emg.contiguous().float()
    B, T, _ = x.shape
    h_in, t = ops.cast(x, dt), T
    rate = plan.frame_rows                  # rows per frame of the current activations
    saved_blocks = []
    for (c1, c2, res) in plan.blocks:
        m = dict(lengths=lengths, rate=rate // c1.mod.stride)
        _, h, t1 = _fwd(c1, _src(c1, h_in, B, t), B, t, act=ACT_RELU, want_act=True, **m)      # relu(bn1(conv1 x))
        if res is not None:
            r, _, _ = _fwd(res, _src(res, h_in, B, t), B, t, want_raw=True, **m)                # res_norm(residual_path x)
        else:
            r = h_in
        _, y, _ = _fwd(c2, h, B, t1, act=ACT_RELU, want_act=True, add_post=r, **m)              # relu(bn2(conv2 h) + res)
        saved_blocks.append(dict(x_in=h_in, h=h, y=y, t_in=t, t_out=t1))
        h_in, t, rate = y, t1, m["rate"]
    L = t
    m = dict(lengths=lengths, rate=rate)
    xl, _, _ = _fwd(plan.w_in, h_in, B, L, want_raw=True, **m)                                  # emg_encoder.py:80
    saved_layers = []
    for ly in plan.layers:
        qkv, _, _ = _fwd(ly.qkv, xl, B, L, want_raw=True, **m)
        # the one-CTA-per-head kernels where they take L (for the backward too, when it follows), the band-tiled ones beyond
        band = not ops.relattn_dense_supported(L, qkv.shape[-1] // (3 * ly.n_head), need_ctx)
        o, probs = (ops.relattn_band_fwd if band else ops.relattn_fwd)(qkv, ly.emb, ly.n_head, ly.max_rel, lengths=lengths)
        pre1, _, _ = _fwd(ly.out, o, B, L, want_raw=True, add_post=xl, **m)                     # src + attn        (transformer.py:54-55)
        x1, st1 = ops.layernorm(pre1, ly.g1, ly.b1, LN_EPS)                                     # norm1             (:56)
        _, hff, _ = _fwd(ly.l1, x1, B, L, act=ACT_RELU, want_act=True, **m)                     # relu(linear1)     (:57)
        pre2, _, _ = _fwd(ly.l2, hff, B, L, want_raw=True, add_post=x1, **m)                    # src + linear2     (:57-58)
        x2, st2 = ops.layernorm(pre2, ly.g2, ly.b2, LN_EPS)                                     # norm2             (:59)
        saved_layers.append(dict(qkv=qkv, probs=probs, band=band, pre1=pre1, st1=st1, hff=hff, pre2=pre2, st2=st2))
        xl = x2
    units, _, _ = _fwd(plan.w_out, xl, B, L, want_raw=True, out_f32=True, **m)                  # emg_encoder.py:88
    logits, _, _ = _fwd(plan.w_aux, xl, B, L, want_raw=True, out_f32=True, **m)
    ctx = EncCtx(B=B, T=T, blocks=saved_blocks, y_last=h_in, t_last=L, layers=saved_layers, x_final=xl) if need_ctx else None
    return units, logits, ctx


def encoder_backward(plan: EncoderPlan, ctx: EncCtx, d_units: Optional[Tensor], d_logits: Optional[Tensor]) -> Tensor:
    """Gradient w.r.t. the EMG input (fp32 [B, T, C]) from the gradients w.r.t. the two heads (`plan.dtype`, either may be None)."""
    dt, B, L = plan.dtype, ctx.B, ctx.t_last
    dx = None
    if d_units is not None:
        dx = _dgrad(plan.w_out, d_units.contiguous().to(dt), B, L, L)
    if d_logits is not None:
        dx = _dgrad(plan.w_aux, d_logits.contiguous().to(dt), B, L, L, add_post=dx)
    for ly, s in zip(reversed(plan.layers), reversed(ctx.layers)):
        dpre2 = ops.layernorm_bwd(dx, s["pre2"], s["st2"], ly.g2)
        dh = _dgrad(ly.l2, dpre2, B, L, L, mask=s["hff"], mask_mode=ACT_RELU)
        dx1 = _dgrad(ly.l1, dh, B, L, L, add_post=dpre2)
        dpre1 = ops.layernorm_bwd(dx1, s["pre1"], s["st1"], ly.g1)
        do = _dgrad(ly.out, dpre1, B, L, L)
        dqkv = (ops.relattn_band_bwd if s["band"] else ops.relattn_bwd)(s["qkv"], ly.emb, s["probs"], do, ly.n_head, ly.max_rel)
        dx = _dgrad(ly.qkv, dqkv, B, L, L, add_post=dpre1)
    # w_raw_in, then the ReLU of the last ResBlock (its saved output is the mask)
    dz = _dgrad(plan.w_in, dx, B, L, L, mask=ctx.y_last, mask_mode=ACT_RELU)
    n = len(plan.blocks)
    for i in reversed(range(n)):
        c1, c2, res = plan.blocks[i]
        s = ctx.blocks[i]
        t_in, t_out = s["t_in"], s["t_out"]
        dh = _dgrad(c2, dz, B, t_out, t_out, mask=s["h"], mask_mode=ACT_RELU)          # through bn2 / conv2 and the inner ReLU
        if c1.unfold:                                                                 # first block: fp32 gradient of the 8-channel input
            dxa = _dgrad(c1, dh, B, t_out, t_in, out_f32=True)
            if res is not None:
                ops.axpy_f32(dxa, _dgrad(res, dz, B, t_out, t_in, out_f32=True), 1.0)
            else:
                ops.axpy_f32(dxa, dz, 1.0)
            return dxa
        dxa = _dgrad(c1, dh, B, t_out, t_in)
        # + residual branch, then the ReLU of the block in front (whose output is this block's input)
        if res is not None:
            dz = _dgrad(res, dz, B, t_out, t_in, add_pre=dxa, mask=s["x_in"] if i > 0 else None,
                        mask_mode=ACT_RELU if i > 0 else ACT_NONE)
        else:
            raise NotImplementedError("identity residual (stride 1, equal channels) does not occur in the encoder (emg_encoder.py:50-53)")
    return ops.cast(dz, torch.float32)


def encoder_losses(plan: EncoderPlan, emg: Tensor, unit_target: Tensor, phoneme_target: Tensor, slots: Tensor,
                   w_units: float = 1.0, w_phonemes: float = 1.0, want_grad: bool = True,
                   use_units: bool = True, use_phonemes: bool = True):
    """EMGEncoderLoss.forward (emg_encoder_loss.py:69-84) + the gradient of  w_units * su_loss + w_phonemes * phoneme_loss
    w.r.t. the EMG signal (train.py:219-230).  slots[0] += su_loss, slots[1] += phoneme_loss.
    Returns (d/d emg fp32 | None, units, logits)."""
    units, logits, ctx = encoder_forward(plan, emg, need_ctx=want_grad)
    du, dl = ops.encoder_losses(units, unit_target.contiguous().float(), logits, phoneme_target.contiguous().to(torch.int64), slots,
                                w_units if use_units else 0.0, w_phonemes if use_phonemes else 0.0,
                                plan.dtype if want_grad else None)
    if not want_grad:
        return None, units, logits
    return encoder_backward(plan, ctx, du if use_units else None, dl if use_phonemes else None), units, logits


def encoder_scores(plan: EncoderPlan, emg: Tensor, unit_target: Tensor, phoneme_target: Tensor, lengths: Tensor):
    """EMGEncoderLoss per utterance of a padded batch, forward only: emg fp32 [B, T, C], unit_target [B, T/16, Du],
    phoneme_target [B, T/16], lengths int32 [B] on the device (frames).  Returns the device tensors (sums fp32 [B, 2],
    counts int32 [B, 4]) of ops.encoder_scores; rows past an utterance's end are never read."""
    from .models.emg_encoder import SILENCE_PHONEME_INDEX
    units, logits, _ = encoder_forward(plan, emg, need_ctx=False, lengths=lengths)
    return ops.encoder_scores(units, unit_target.contiguous().float(), logits, phoneme_target.contiguous().to(torch.int64),
                              lengths, SILENCE_PHONEME_INDEX)
