"""Whole-network forward / backward passes over the C-ABI kernels.

This is the host side of the hot path: explicit (autograd-free) forward and backward
schedules for the generator (models/generator.py:140-162 + layers/conv.py:82-84 of the
reference) and the discriminator stacks (models/discriminator.py), in channels-last
layout, with every elementwise neighbour of a convolution folded into that convolution's
epilogue (see include/stegan_b200.h, StgConv).  torch.autograd.Function wrappers in
ste_gan_b200/autograd.py expose the same passes to `loss.backward()` users.

Gradient flow conventions
  * activations / activation-gradients: `dtype` (bf16 or fp32) channels-last [B, T(*p), C]
  * parameter gradients: fp32, ACCUMULATED into `param.grad` (allocated on first use)
  * weight gradients are first produced in the packed [c_out][k][cin_g] layout by the
    wgrad engines and then pulled back through the weight_norm / spectral_norm fold.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import ops
from .ops import ACT_LEAKY, ACT_NONE, ACT_RELU, ACT_TANH

Tensor = torch.Tensor


# --------------------------------------------------------------------------------------
# folded (re-parametrised + packed) weights
# --------------------------------------------------------------------------------------
@dataclass
class Folded:
    mod: torch.nn.Module
    wf: Tensor
    wd: Optional[Tensor]
    dtype: torch.dtype
    scale: Optional[Tensor] = None          # weight-norm: g/||v||
    u: Optional[Tensor] = None              # spectral-norm: u, v, sigma used by THIS forward
    v: Optional[Tensor] = None
    sigma: Optional[Tensor] = None
    pg: int = 1                             # groups of the packed operands (narrow groups merged for tcgen05)
    unfold: bool = False                    # tiny-channel first layer: 1-tap conv over im2col rows
    kp: int = 0                             # ... whose K axis has kp = roundup8(k * c_in) elements


def _w3(t: Tensor) -> Tensor:
    """[c_out, cin_g, k] or [c_out, cin_g, k, 1] -> 3-D view."""
    return t.view(t.shape[0], t.shape[1], t.shape[2])


def pack_mode(mod, dtype: torch.dtype) -> Tuple[int, bool]:
    """(pack groups, unfold?) of a conv module in this precision.  fp32 (CUDA-core validation engine) keeps the
    reference's own grouping; bf16 widens narrow groups to the tensor engine's 64-channel K chunks and turns
    the C_in = 8 first layers (discriminator.py:26,55,77,104) into 1-tap convs over im2col rows."""
    if mod.groups == 1 and mod.kernel == 1 and mod.in_channels % 8 != 0 and mod.out_channels >= 32:
        return 1, True      # e.g. the MFCC generator's 89 -> 768 input conv: channels zero-padded to a multiple of 8
    if dtype != torch.bfloat16:
        return mod.groups, False
    if mod.groups == 1 and mod.in_channels < 16 and mod.in_channels * mod.kernel <= 256 and mod.out_channels >= 32:
        return 1, True
    return ops.tc_pack_groups(mod.in_channels, mod.out_channels, mod.groups), False


def fold(mod, dtype: torch.dtype, training: bool = True, want_dgrad: bool = True,
         persist: Optional[Dict[int, "Folded"]] = None) -> Folded:
    """Re-parametrise one conv module into the packed operand layouts (one fold = one
    power iteration for spectral-norm layers in training mode, as in the reference's
    forward pre-hook).  `persist` keeps the weight-norm packs of a module in the same
    buffers across calls (fixed addresses, so CUDA graphs that read them stay valid)."""
    pg, unf = pack_mode(mod, dtype)
    kp = ops.round_up8(mod.kernel * mod.in_channels) if unf else 0
    # bf16 data-gradients read the forward pack - except grouped convs, whose tensor-engine data-gradient wants the
    # K-major pack wd [k][c_in][c_out/pg] (compact groups, conv_tc.cu)
    want_dgrad = want_dgrad and (dtype != torch.bfloat16 or mod.groups > 1)
    if mod.norm == "weight_norm":
        prev = persist.get(id(mod)) if persist is not None else None
        out = (prev.wf, prev.wd, prev.scale) if prev is not None and prev.dtype == dtype and prev.wd is not None else None
        wf, wd, scale = ops.weightnorm_fold(_w3(mod.weight_v.data), mod.weight_g.data, mod.groups, dtype,
                                            want_dgrad or persist is not None, out=out, pack_groups=pg, unfold=unf)
        f = Folded(mod, wf, wd, dtype, scale=scale, pg=pg, unfold=unf, kp=kp)
        if persist is not None:
            persist[id(mod)] = f
        return f
    wf, wd, sigma, u_used, v_used = ops.spectralnorm_fold(_w3(mod.weight_orig.data), mod.weight_u, mod.weight_v, mod.groups,
                                                          training, dtype, want_dgrad, pack_groups=pg, unfold=unf, keep_uv=True)
    return Folded(mod, wf, wd, dtype, u=u_used, v=v_used, sigma=sigma, pg=pg, unfold=unf, kp=kp)


def _grad_of(p: torch.nn.Parameter) -> Tensor:
    if p.grad is None:
        p.grad = torch.zeros_like(p, memory_format=torch.contiguous_format)
    return p.grad


def dw_layout(f: Folded) -> Tuple[int, int, int]:
    """(floats, ld, span) of the packed weight-gradient buffer of this conv (ops.wgrad_layout); cached per fold mode."""
    m = f.mod
    key = (f.dtype, f.unfold, ops._engine_override)
    cache = m.__dict__.setdefault("_stg_dw_layout", {})
    if key not in cache:
        if f.unfold:                        # im2col layers: rows are kp long, (tap, channel) order = packed order
            ld, span = f.kp, m.in_channels
        else:
            ld, span = ops.wgrad_layout(f.dtype, c_in=m.in_channels, c_out=m.out_channels, k=m.kernel, groups=m.groups,
                                        stride=m.stride)
        cache[key] = (m.out_channels * ld, ld, span)
    return cache[key]


def fold_backward(f: Folded, dw: Tensor) -> None:
    m = f.mod
    _, ld, span = dw_layout(f)
    if m.norm == "weight_norm":
        ops.weightnorm_fold_bwd(dw, _w3(m.weight_v.data), m.weight_g.data, _grad_of(m.weight_v), _grad_of(m.weight_g), True,
                                dw_ld=ld, dw_span=span, groups=m.groups)
    else:
        ops.spectralnorm_fold_bwd(dw, _w3(m.weight_orig.data), f.u, f.v, f.sigma, _grad_of(m.weight_orig), True,
                                  dw_ld=ld, dw_span=span, groups=m.groups)


class _Workspace:
    """Zero-initialised fp32 arena for packed weight gradients (one memset per pass)."""
    deferred = False    # weight-norm fold backward runs per layer, right after its wgrad

    def __init__(self, folds: Sequence["Folded"], device):
        n = sum(dw_layout(f)[0] for f in folds)
        self.buf = torch.zeros(n, device=device, dtype=torch.float32)
        self.off = 0

    def take(self, f: "Folded") -> Tensor:
        n = dw_layout(f)[0]
        t = self.buf[self.off:self.off + n]
        self.off += n
        return t


class FoldPlan:
    """Everything the weight-normed convs of ONE network need, at fixed device addresses: packed operands
    (wf, wd, scale), the fp32 weight-gradient arena, and the device table that lets one launch fold / un-fold all
    of them (stg_weightnorm_fold_multi / _bwd_multi).  Create it AFTER the parameters and gradients have been
    re-homed into their flat buffers (trainer.FlatParams): the table stores raw pointers to them.
    Spectral-norm convs keep their per-forward fold (one power iteration each); they only get gradient scratch here."""
    deferred = True     # weight-norm fold backward runs once per phase: backward()
    wgrad_stream = None  # while set (async_wgrads), _wgrad launches on a side stream, ordered after its operands
    _keep: list = []

    def async_wgrads(self, stream) -> None:
        """From now until join_wgrads(), weight-gradient kernels go to a side stream: a conv's wgrad and dgrad both
        consume dy and are independent, so the backward critical path becomes the dgrad chain alone.
        `stream`: one CUDA stream, or a dict {id of a compute stream (.cuda_stream): its side stream} when several
        branches run backward passes concurrently (wgrads launched from a stream that is not in the dict stay inline)."""
        self.wgrad_stream, self._keep = stream, []

    def side_for_current(self):
        ws = self.wgrad_stream
        if isinstance(ws, dict):
            return ws.get(torch.cuda.current_stream().cuda_stream)
        return ws

    def join_wgrads_of(self, compute_streams) -> None:
        """Make the current stream wait for the weight-gradient side streams of these compute streams only (one backward
        branch is through while others still run); the mapping and the kept operands stay until join_wgrads()."""
        ws = self.wgrad_stream
        if not isinstance(ws, dict):
            return
        for cs in compute_streams:
            st = ws.get(cs.cuda_stream)
            if st is not None:
                ev = torch.cuda.Event()
                ev.record(st)
                torch.cuda.current_stream().wait_event(ev)

    def join_wgrads(self) -> None:
        ws = self.wgrad_stream
        for st in (ws.values() if isinstance(ws, dict) else ([ws] if ws is not None else [])):
            ev = torch.cuda.Event()
            ev.record(st)
            torch.cuda.current_stream().wait_event(ev)
        self.wgrad_stream, self._keep = None, []     # operands were kept alive until the side streams were joined

    def __init__(self, convs: Sequence, dtype: torch.dtype):
        from . import _lib
        self.dtype = dtype
        self.need_wd = dtype != torch.bfloat16     # bf16: data-gradients read the forward pack (tcgen05, MN-major operand) ...
        need_wd = lambda m: self.need_wd or m.groups > 1   # ... except grouped convs (K-major wd, compact groups)
        self.wn = [c for c in convs if c.norm == "weight_norm"]
        dev = self.wn[0].bias.device
        self.device = dev
        self.folds: Dict[int, Folded] = {}
        esz = 2 if dtype == torch.bfloat16 else 4
        metas, n_pack, n_scale, n_dw = [], 0, 0, 0
        for m in self.wn:
            pg, unf = pack_mode(m, dtype)
            cin_g = m.in_channels // m.groups
            sf, sd = ops._pack_shapes(m.out_channels, cin_g, m.kernel, m.groups, pg, unf)
            nf = sf[0] * sf[1] * (sf[2] if len(sf) > 2 else 1)
            nf_al = (nf + 63) // 64 * 64                       # 128-byte aligned packs (TMA base addresses)
            metas.append((m, pg, unf, sf, sd, nf, nf_al))
            n_pack += (2 if need_wd(m) else 1) * nf_al; n_scale += (m.out_channels + 3) // 4 * 4
        self._packs = torch.zeros(n_pack, device=dev, dtype=dtype)
        self._scales = torch.zeros(n_scale, device=dev, dtype=torch.float32)
        po = so = 0
        for (m, pg, unf, sf, sd, nf, nf_al) in metas:
            wf = self._packs[po:po + nf].view(sf); po += nf_al
            wd = None
            if need_wd(m):
                wd = self._packs[po:po + nf].view(sd); po += nf_al
            scale = self._scales[so:so + m.out_channels]; so += (m.out_channels + 3) // 4 * 4
            kp = ops.round_up8(m.kernel * m.in_channels) if unf else 0
            self.folds[id(m)] = Folded(m, wf, wd, dtype, scale=scale, pg=pg, unfold=unf, kp=kp)
        # gradient arena (weight-norm convs only; fixed slices)
        self._dw_off = {}
        for m in self.wn:
            n = dw_layout(self.folds[id(m)])[0]
            self._dw_off[id(m)] = (n_dw, n); n_dw += (n + 3) // 4 * 4
        self.arena = torch.zeros(n_dw, device=dev, dtype=torch.float32)
        # device table
        items, row0, tile0 = [], 0, 0
        for m in self.wn:
            f = self.folds[id(m)]
            cin_g = m.in_channels // m.groups
            _, ld, span = dw_layout(f)
            off, n = self._dw_off[id(m)]
            gv, gg = _grad_of(m.weight_v), _grad_of(m.weight_g)
            items.append(_lib.StgFoldItem(
                v=m.weight_v.data.data_ptr(), g=m.weight_g.data.data_ptr(), wf=f.wf.data_ptr(), wd=f.wd.data_ptr() if f.wd is not None else None,
                scale=f.scale.data_ptr(), dw=self.arena[off:off + n].data_ptr(), dv=gv.data_ptr(), dg=gg.data_ptr(),
                c_out=m.out_channels, cin_g=cin_g, k=m.kernel, groups=m.groups, pg=f.pg,
                flags=_lib.PACK_UNFOLD if f.unfold else 0, dw_ld=ld, dw_span=span, row0=row0, tile0=tile0))
            row0 += m.out_channels
            if not self.need_wd:          # row form: tile0 counts the wd transposition blocks of the grouped convs
                tile0 += m.kernel * f.pg if f.wd is not None else 0
            elif f.unfold:
                tile0 += -(-m.out_channels // 32) * -(-f.kp // 32)
            else:
                tile0 += m.kernel * f.pg * -(-(m.out_channels // f.pg) // 32) * -(-(m.in_channels // f.pg) // 32)
        self.n_items, self.total_rows, self.total_tiles = len(items), row0, (tile0 if self.need_wd else -tile0)
        self.item_row0 = [it.row0 for it in items] + [row0]      # table row of each item's first output channel
        self.table = ops.fold_table(items, dev)
        self._ptrs = [(p.data_ptr(), p.grad.data_ptr()) for m in self.wn for p in (m.weight_v, m.weight_g)]

    def _check_ptrs(self) -> None:
        cur = [(p.data_ptr(), p.grad.data_ptr() if p.grad is not None else 0) for m in self.wn for p in (m.weight_v, m.weight_g)]
        if cur != self._ptrs:
            raise RuntimeError("FoldPlan: parameter / gradient storage moved after the plan was built")

    def fold(self) -> Dict[int, Folded]:
        """Re-parametrise every weight-normed conv from the current weights (2 launches)."""
        self._check_ptrs()
        ops.weightnorm_fold_multi(self.table, self.n_items, self.total_rows, self.total_tiles, self.dtype)
        return self.folds

    # -- gradient arena (the _Workspace interface of _wgrad) -------------------------------------------
    def zero(self) -> None:
        self.arena.zero_()

    def take(self, f: Folded) -> Tensor:
        ent = self._dw_off.get(id(f.mod))
        if ent is None:                                   # spectral-norm conv: scratch per use
            return torch.zeros(dw_layout(f)[0], device=self.device, dtype=torch.float32)
        return self.arena[ent[0]:ent[0] + ent[1]]

    def backward(self, accumulate: bool = True) -> None:
        """dv, dg (+)= fold-backward of everything accumulated in the arena since zero() (1 launch).  accumulate=False
        overwrites: for a caller that knows this is the only contribution to these gradients since they were zeroed
        (the fused train step) it saves re-reading every dv."""
        self._check_ptrs()
        ops.weightnorm_fold_bwd_multi(self.table, self.n_items, self.total_rows, accumulate)


    def backward_range(self, item_lo: int, item_hi: int, accumulate: bool = True) -> None:
        """backward() for the weight-normed convs [item_lo, item_hi) of the plan only (one gradient bucket)."""
        self._check_ptrs()
        r0, r1 = self.item_row0[item_lo], self.item_row0[item_hi]
        if r1 > r0:
            ops.weightnorm_fold_bwd_range(self.table, self.n_items, r0, r1 - r0, accumulate)


def unfold_input(f: Folded, src: Tensor, B: int, t_src: int, phases: int = 1) -> Tensor:
    """im2col rows of a tiny-channel first layer's input (what _fwd / _wgrad of an `unfold` layer consume)."""
    m = f.mod
    return ops.unfold(src, n_samples=B, phases=phases, t_src=t_src, t_dst=m.t_out(t_src), channels=m.in_channels,
                      k=m.kernel, dilation=m.dilation, stride=m.stride, pad=m.pad)


def _fwd(f: Folded, src: Tensor, B: int, t_src: int, *, phases: int = 1, act: int = ACT_NONE, want_raw: bool = False,
         want_act: bool = False, dup: bool = False, add_post: Optional[Tensor] = None, post_shift: int = 0,
         out_f32: bool = False, lengths: Optional[Tensor] = None, rate: int = 1) -> Tuple[Optional[Tensor], Optional[Tensor], int]:
    """One conv forward.  For an `unfold` layer `src` is the im2col tensor from unfold_input().
    lengths (int32 [B] frames, optional): output rows >= rate * lengths[b] of sample b are written as 0."""
    m = f.mod
    t_dst = m.t_out(t_src)
    odt = torch.float32 if out_f32 else f.dtype
    y_raw = torch.empty((B, t_dst * phases, m.out_channels), device=src.device, dtype=odt) if want_raw else None
    y_act = torch.empty((B, t_dst * phases * (2 if dup else 1), m.out_channels), device=src.device, dtype=odt) if want_act else None
    if f.unfold:
        ops.conv(src, f.wf, n_samples=B, phases=phases, t_src=t_dst, t_dst=t_dst, c_src=f.kp, c_dst=m.out_channels, k=1,
                 bias=m.bias.data, act=act, dup_rows=dup, add_post=add_post, post_shift=post_shift, y_raw=y_raw, y_act=y_act,
                 valid_units=lengths, rows_per_unit=rate)
    else:
        ops.conv(src, f.wf, n_samples=B, phases=phases, t_src=t_src, t_dst=t_dst, c_src=m.in_channels, c_dst=m.out_channels,
                 groups=f.pg, k=m.kernel, dilation=m.dilation, stride=m.stride, pad=m.pad, bias=m.bias.data, act=act,
                 dup_rows=dup, add_post=add_post, post_shift=post_shift, y_raw=y_raw, y_act=y_act, acct_groups=m.groups,
                 valid_units=lengths, rows_per_unit=rate)
    return y_raw, y_act, t_dst


def _dgrad(f: Folded, dy: Tensor, B: int, t_dy: int, t_x: int, *, phases: int = 1, mask: Optional[Tensor] = None,
           mask_mode: int = ACT_NONE, add_pre: Optional[Tensor] = None, add_post: Optional[Tensor] = None,
           pair_sum: bool = False, out_f32: bool = False) -> Tensor:
    m = f.mod
    if f.unfold:
        # gradient w.r.t. the im2col rows, then its adjoint back onto the [B, t_x*phases, C_in] input (fp32)
        assert mask is None and add_pre is None and add_post is None and not pair_sum
        du = torch.empty((B, t_dy * phases, f.kp), device=dy.device, dtype=f.dtype)
        fwd_pack = f.dtype == torch.bfloat16
        ops.conv(dy, f.wf if fwd_pack else f.wd, n_samples=B, phases=phases, t_src=t_dy, t_dst=t_dy, c_src=m.out_channels,
                 c_dst=f.kp, k=1, transposed=True, y_raw=du, w_fwd_pack=fwd_pack)
        dx = torch.zeros((B, t_x * phases, m.in_channels), device=dy.device, dtype=torch.float32)
        ops.unfold_bwd(du, dx, n_samples=B, phases=phases, t_src=t_x, t_dst=t_dy, channels=m.in_channels, k=m.kernel,
                       dilation=m.dilation, stride=m.stride, pad=m.pad)
        return dx if out_f32 else ops.cast(dx, f.dtype)
    rows = t_x // 2 if pair_sum else t_x
    dx = torch.empty((B, rows * phases, m.in_channels), device=dy.device, dtype=torch.float32 if out_f32 else f.dtype)
    # bf16 (tensor engine / logits matvec): data-gradients read the FORWARD pack - grouped convs the K-major wd pack;
    # fp32 (CUDA-core engine): the wd pack
    fwd_pack = f.dtype == torch.bfloat16 and not (m.groups > 1 and f.wd is not None)
    ops.conv(dy, f.wf if fwd_pack else f.wd, n_samples=B, phases=phases, t_src=t_dy, t_dst=t_x, c_src=m.out_channels,
             c_dst=m.in_channels, groups=f.pg, k=m.kernel, dilation=m.dilation, stride=m.stride, pad=m.pad, transposed=True,
             pair_sum=pair_sum, mask=mask, mask_mode=mask_mode, add_pre=add_pre, add_post=add_post, y_raw=dx,
             w_fwd_pack=fwd_pack, acct_groups=m.groups)
    return dx


def _wgrad(f: Folded, x: Tensor, dy: Tensor, B: int, t_x: int, t_dy: int, ws: _Workspace, phases: int = 1) -> None:
    """Weight + bias gradient of one conv.  For an `unfold` layer `x` is the im2col tensor from unfold_input()."""
    m = f.mod
    side = ws.side_for_current() if getattr(ws, "wgrad_stream", None) is not None else None
    if side is not None:
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())       # dy (and x) are ready at this point of the current stream
        side.wait_event(ev)
        ws._keep.append((x, dy))                     # the current stream must not recycle them before the join
        with torch.cuda.stream(side):
            _wgrad_here(f, x, dy, B, t_x, t_dy, ws, phases)
        return
    _wgrad_here(f, x, dy, B, t_x, t_dy, ws, phases)


def _wgrad_here(f: Folded, x: Tensor, dy: Tensor, B: int, t_x: int, t_dy: int, ws, phases: int) -> None:
    m = f.mod
    dw = ws.take(f)
    if f.unfold:
        ops.wgrad(x, dy, dw, _grad_of(m.bias), n_samples=B, phases=phases, t_in=t_dy, t_out=t_dy, c_in=f.kp,
                  c_out=m.out_channels, k=1)
    else:
        ops.wgrad(x, dy, dw, _grad_of(m.bias), n_samples=B, phases=phases, t_in=t_x, t_out=t_dy, c_in=m.in_channels,
                  c_out=m.out_channels, groups=m.groups, k=m.kernel, dilation=m.dilation, stride=m.stride, pad=m.pad)
    if not (ws.deferred and m.norm == "weight_norm"):
        fold_backward(f, dw)


# --------------------------------------------------------------------------------------
# generator
# --------------------------------------------------------------------------------------
def generator_convs(model) -> List:
    convs = [model.gblocks[0]]
    for blk in list(model.gblocks)[1:]:
        c = blk.convs()
        convs += [c["c1"], c["c2"], c["res"], c["c3"], c["c4"]]
    convs.append(model.last_conv[1])
    return convs


def gblock_fwd(blk, folds: Dict[int, Folded], x_raw: Tensor, x_act: Tensor, B: int, t: int, *, want_raw: bool,
               want_act: bool, dup_next: bool, side=None, lengths: Optional[Tensor] = None, rate: int = 1):
    """GBlock.forward (layers/conv.py:82-84) on channels-last tensors.
    x_raw [B,t,C_in]: block input; x_act [B,t*up,C_in]: relu(x) with rows duplicated when the block upsamples.
    lengths (optional): frames per sample, the input having `rate` rows per frame; every output row past a sample's
    end is written as 0.
    Returns (y_raw|None, relu(y) (rows duplicated if dup_next)|None, saved)."""
    c = blk.convs()
    up = blk.upsample
    t_hi = t * up
    lo = dict(lengths=lengths, rate=rate)
    hi = dict(lengths=lengths, rate=rate * up)
    # conv1: ReLU -> [Up] -> conv(d1) -> ReLU -> conv(d3);  res1: [Up] -> conv(k1) on the raw input   (conv.py:38-56,83)
    # the residual 1x1 conv is independent of conv1's first conv: optionally on a side stream
    (r, _, _), (_, a1, _) = fork_join(
        side, lambda: _fwd(folds[id(c["res"])], x_raw, B, t, want_raw=True, **lo),     # 1x1 commutes with nearest upsampling
        lambda: _fwd(folds[id(c["c1"])], x_act, B, t_hi, act=ACT_RELU, want_act=True, **hi))
    h_raw, h_act, _ = _fwd(folds[id(c["c2"])], a1, B, t_hi, act=ACT_RELU, want_raw=True, want_act=True,
                           add_post=r, post_shift=1 if up > 1 else 0, **hi)
    # conv2: ReLU -> conv(d9) -> ReLU -> conv(d27);  y = h + conv2(h)                                (conv.py:61-75,84)
    _, a3, _ = _fwd(folds[id(c["c3"])], h_act, B, t_hi, act=ACT_RELU, want_act=True, **hi)
    y_raw, y_act, _ = _fwd(folds[id(c["c4"])], a3, B, t_hi, act=ACT_RELU, want_raw=want_raw, want_act=want_act,
                           add_post=h_raw, dup=dup_next, **hi)
    saved = dict(x_raw=x_raw, x_act=x_act, a1=a1, h_act=h_act, a3=a3, t_lo=t, t_hi=t_hi, up=up)
    return y_raw, y_act, saved


def gblock_bwd(blk, folds: Dict[int, Folded], s: dict, dy: Tensor, B: int, ws: _Workspace, out_f32: bool = False,
               side=None) -> Tensor:
    """Backward of gblock_fwd: dy = d/d(y raw) [B,t_hi,C_out] -> d/d(x raw) [B,t_lo,C_in]; accumulates weight grads."""
    c = blk.convs()
    t_lo, t_hi, up = s["t_lo"], s["t_hi"], s["up"]
    f1, f2, fr, f3, f4 = (folds[id(c[k])] for k in ("c1", "c2", "res", "c3", "c4"))
    # y = h + conv_d27(relu(conv_d9(relu h)))
    _wgrad(f4, s["a3"], dy, B, t_hi, t_hi, ws)
    da3 = _dgrad(f4, dy, B, t_hi, t_hi, mask=s["a3"], mask_mode=ACT_RELU)
    _wgrad(f3, s["h_act"], da3, B, t_hi, t_hi, ws)
    dh = _dgrad(f3, da3, B, t_hi, t_hi, mask=s["h_act"], mask_mode=ACT_RELU, add_post=dy)
    # h = conv_d3(relu(conv_d1(up(relu x)))) + up(res1(x))
    _wgrad(f2, s["a1"], dh, B, t_hi, t_hi, ws)

    def res_branch():           # gradient through up(res1(x)): independent of the conv1 chain until their sum
        dr = dh if up == 1 else ops.pair_sum_rows(dh, B * t_lo, fr.mod.out_channels).view(B, t_lo, -1)
        _wgrad(fr, s["x_raw"], dr, B, t_lo, t_lo, ws)
        return _dgrad(fr, dr, B, t_lo, t_lo), dr

    (dx_res, dr), da1 = fork_join(side, res_branch, lambda: _dgrad(f2, dh, B, t_hi, t_hi, mask=s["a1"], mask_mode=ACT_RELU))
    _wgrad(f1, s["x_act"], da1, B, t_hi, t_hi, ws)
    return _dgrad(f1, da1, B, t_hi, t_hi, pair_sum=up > 1, mask=s["x_raw"], mask_mode=ACT_RELU, add_post=dx_res,
                  out_f32=out_f32)


def fold_generator(model, dtype: torch.dtype, want_dgrad: bool = True, plan: Optional[FoldPlan] = None) -> Dict[int, Folded]:
    if plan is not None:
        return plan.fold()
    return {id(c): fold(c, dtype, want_dgrad=want_dgrad) for c in generator_convs(model)}


@dataclass
class GenCtx:
    B: int = 0
    T: int = 0
    dtype: torch.dtype = torch.float32
    folds: Dict[int, Folded] = field(default_factory=dict)
    x0: Optional[Tensor] = None
    ids: List[Optional[Tensor]] = field(default_factory=list)
    emb_dims: List[int] = field(default_factory=list)
    blocks: List[dict] = field(default_factory=list)
    y_last_act: Optional[Tensor] = None
    x_pred: Optional[Tensor] = None


def generator_forward(model, speech_units: Tensor, session_ids: Optional[Tensor], speaking_mode_ids: Optional[Tensor],
                      dtype: torch.dtype, need_ctx: bool, folds: Optional[Dict[int, Folded]] = None, side=None,
                      lengths: Optional[Tensor] = None):
    """EMGGeneratorGanTTS.forward (generator.py:140-162).  Returns (x_pred fp32 [B,16T,C], ctx|None).
    lengths (int32 [B] on the device, frames; forward only): sample b is an utterance of lengths[b] frames zero-padded
    to T.  Every convolution writes 0 past its sample's end, so rows [0, r*lengths[b]) of x_pred[b] are what the
    utterance gives on its own (r = output rows per frame) and the rows after it are 0, whatever the padded units hold."""
    if need_ctx and lengths is not None:
        raise ValueError("generator_forward: length masks are forward-only (need_ctx=True with lengths)")
    su = speech_units.contiguous().float()
    B, T, du = su.shape
    if folds is None:
        folds = fold_generator(model, dtype, want_dgrad=need_ctx)
    # units ++ session embedding ++ speaking-mode embedding  (generator.py:143-151)
    tables, ids = [], []
    if model.use_session_embeddings:
        tables.append(model.session_embeddings.weight); ids.append(session_ids.to(torch.int64).contiguous())
    if model.use_speaking_mode_embedding:
        tables.append(model.speaking_mode_embeddings.weight); ids.append(speaking_mode_ids.to(torch.int64).contiguous())
    if len(tables) == 0:
        x0 = ops.cast(su, dtype)
    elif len(tables) == 1:
        x0 = ops.embed_concat(su, tables[0].data, ids[0], dtype)
    else:  # two tables: concatenate in two steps (fp32 intermediate)
        tmp = ops.embed_concat(su, tables[0].data, ids[0], torch.float32)
        x0 = ops.embed_concat(tmp, tables[1].data, ids[1], dtype)
    blocks = list(model.gblocks)[1:]
    ups = [b.upsample for b in blocks]
    for u in ups:
        if u not in (1, 2):
            raise ValueError("GBlock upsample must be 1 or 2 on this path")
    # gblocks.0 (1x1): raw output feeds res1 of the first GBlock, relu(.) feeds its conv1 (duplicated rows = Upsample)
    f0 = folds[id(model.gblocks[0])]
    if f0.unfold:                 # input channels not a multiple of 8 (MFCC variant): zero-padded rows for the tensor engine
        x0 = unfold_input(f0, x0, B, T)
    x_raw, x_act, t = _fwd(f0, x0, B, T, act=ACT_RELU, want_raw=True, want_act=True, dup=ups[0] > 1, lengths=lengths)
    saved = []
    rate = 1                      # rows per unit frame of the current activations
    for i, blk in enumerate(blocks):
        last = i + 1 == len(blocks)
        nxt_dup = (not last) and ups[i + 1] > 1
        y_raw, y_act, s = gblock_fwd(blk, folds, x_raw, x_act, B, t, want_raw=not last, want_act=True, dup_next=nxt_dup,
                                     side=side, lengths=lengths, rate=rate)
        if need_ctx:
            saved.append(s)
        x_raw, x_act, t = y_raw, y_act, s["t_hi"]
        rate *= s["up"]
    # last_conv: ReLU -> conv(k3) ; tanh after the channel-last transpose (generator.py:133-137,157-160)
    _, x_pred, _ = _fwd(folds[id(model.last_conv[1])], x_act, B, t, act=ACT_TANH, want_act=True, out_f32=True,
                        lengths=lengths, rate=rate)
    if not need_ctx:
        return x_pred, None
    ctx = GenCtx(B=B, T=T, dtype=dtype, folds=folds, x0=x0, ids=ids, emb_dims=[tb.shape[1] for tb in tables],
                 blocks=saved, y_last_act=x_act, x_pred=x_pred)
    ctx.tables = tables
    ctx.d_units = du
    ctx.t_out = t
    return x_pred, ctx


class GenBackward:
    """Backward of generator_forward in resumable pieces, back to front: __init__ (tanh', last_conv), blocks(lo, hi)
    (GBlocks hi-1 ... lo), finish() (gblocks.0, embeddings).  With a FoldPlan, bucket(item_lo, item_hi) completes one
    gradient BUCKET: it waits for the bucket's weight-gradient kernels and runs the weight-norm backward of just those
    convs, after which the bucket's slice of the flat gradient is final - the data-parallel all-reduce of that slice
    can run while the layers in front of it are still in their backward pass."""

    def __init__(self, model, ctx: GenCtx, dx_pred: Tensor, plan: Optional[FoldPlan] = None, side=None, res_side=None,
                 overwrite_grads: bool = False):
        self.model, self.ctx, self.plan, self.side, self.res_side = model, ctx, plan, side, res_side
        self.accumulate = not overwrite_grads
        B, dtype, folds = ctx.B, ctx.dtype, ctx.folds
        if plan is not None:
            plan.zero()
            self.ws = plan
            if side is not None:
                plan.async_wgrads(side)             # `side`: extra stream for the weight-gradient kernels
        else:
            self.ws = _Workspace([folds[id(c)] for c in generator_convs(model)], dx_pred.device)
        self.gblocks = list(model.gblocks)[1:]
        t = ctx.t_out
        # tanh' from the output, then last_conv
        dpre = ops.act_bwd(dx_pred.contiguous(), ctx.x_pred, ACT_TANH, dtype)
        f = folds[id(model.last_conv[1])]
        _wgrad(f, ctx.y_last_act, dpre, B, t, t, self.ws)
        self.dy = _dgrad(f, dpre, B, t, t, mask=ctx.y_last_act, mask_mode=ACT_RELU)        # d(y8 raw)

    def blocks(self, lo: int, hi: int) -> None:
        for i in reversed(range(lo, hi)):
            self.dy = gblock_bwd(self.gblocks[i], self.ctx.folds, self.ctx.blocks[i], self.dy, self.ctx.B, self.ws, side=self.res_side)

    def finish(self) -> None:
        model, ctx, dy, B = self.model, self.ctx, self.dy, self.ctx.B
        # gblocks.0 and the embeddings
        f0 = ctx.folds[id(model.gblocks[0])]
        _wgrad(f0, ctx.x0, dy, B, ctx.T, ctx.T, self.ws)
        if ctx.tables:
            dx0 = _dgrad(f0, dy, B, ctx.T, ctx.T)
            off = ctx.d_units
            if len(ctx.tables) == 1:
                ops.embed_concat_bwd(dx0, ctx.ids[0], off, _grad_of(ctx.tables[0]))
            else:
                d0, d1 = ctx.emb_dims
                # [units | emb0 | emb1]: slice copies keep the kernel's contiguous-tail contract
                ops.embed_concat_bwd(dx0[:, :, :off + d0].contiguous(), ctx.ids[0], off, _grad_of(ctx.tables[0]))
                ops.embed_concat_bwd(dx0, ctx.ids[1], off + d0, _grad_of(ctx.tables[1]))
        self.dy = None

    def bucket(self, item_lo: int, item_hi: int, last: bool = False) -> None:
        """Convs [item_lo, item_hi) of generator_convs(model) are done: make their gradients final."""
        plan = self.plan
        if plan is None:
            return
        plan.join_wgrads()
        plan.backward_range(item_lo, item_hi, accumulate=self.accumulate)
        if not last and self.side is not None:
            plan.async_wgrads(self.side)


def generator_backward(model, ctx: GenCtx, dx_pred: Tensor, plan: Optional[FoldPlan] = None, side=None,
                       res_side=None, overwrite_grads: bool = False) -> None:
    """Backward of generator_forward: accumulates into the .grad of every generator parameter.
    dx_pred: fp32 [B, 16T, C] gradient w.r.t. the tanh output.  With a FoldPlan the packed weight gradients go to
    its arena and the weight-norm backward of all convs is one launch at the end."""
    gb = GenBackward(model, ctx, dx_pred, plan, side, res_side, overwrite_grads)
    gb.blocks(0, len(gb.gblocks))
    gb.finish()
    if plan is not None:
        plan.join_wgrads()
        plan.backward(accumulate=not overwrite_grads)


def fork_many(streams: Sequence["torch.cuda.Stream"], fns: Sequence) -> None:
    """Run fns[0] on the current stream and fns[1 + i] on streams[i], all ordered after everything enqueued so far; the
    current stream then waits for every side stream (same contract as fork_join, results through closures)."""
    cur = torch.cuda.current_stream()
    ev = torch.cuda.Event()
    ev.record(cur)
    for st, fn in zip(streams, fns[1:]):
        st.wait_event(ev)
        with torch.cuda.stream(st):
            fn()
    fns[0]()
    for st in streams[:len(fns) - 1]:
        e2 = torch.cuda.Event()
        e2.record(st)
        cur.wait_event(e2)


def fork_join(side: Optional["torch.cuda.Stream"], fn_side, fn_main):
    """Run fn_side on `side` and fn_main on the current stream, both ordered after everything enqueued so far;
    returns (fn_side(), fn_main()) once the current stream has been made to wait for `side`.  Works under CUDA
    graph capture (the side stream joins the capture through the fork event).  Callers keep every tensor the two
    functions create referenced until their own phase ends; together with the fork ordering this keeps the caching
    allocator's per-stream pools from recycling a block that the other stream still uses."""
    if side is None:
        return fn_side(), fn_main()
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream())
    side.wait_event(ev)
    with torch.cuda.stream(side):
        ra = fn_side()
    rb = fn_main()
    ev2 = torch.cuda.Event()
    ev2.record(side)
    torch.cuda.current_stream().wait_event(ev2)
    return ra, rb


# --------------------------------------------------------------------------------------
# discriminators
# --------------------------------------------------------------------------------------
def disc_subnets(model) -> List[Tuple[str, object]]:
    return [("P", d) for d in model.multi_pooled_disc] + [("S", d) for d in model.multi_scale_disc]


def discriminator_convs(model) -> List:
    out = []
    for _, d in disc_subnets(model):
        out += list(d.layers) + [d.output]
    return out


def fold_discriminator(model, dtype: torch.dtype, training: bool = True, want_dgrad: bool = True,
                       reuse: Optional[Dict[int, Folded]] = None,
                       persist: Optional[Dict[int, Folded]] = None,
                       plan: Optional[FoldPlan] = None, refold: bool = True, sn_streams=None) -> Dict[int, Folded]:
    """Fold every discriminator conv.  Weight-norm folds depend on the weights only and may be
    reused between forwards (`reuse`); spectral-norm layers are ALWAYS re-folded because every
    training-mode forward of the reference runs one more power iteration (conv.py:94,101)."""
    if plan is not None:
        # weight-norm convs: one multi-tensor launch (when the weights changed); spectral-norm convs one by one - each
        # is a chain of ~7 small dependent kernels (power iteration, sigma, pack), so with `sn_streams` the layers'
        # chains run side by side (and beside the multi-tensor launch) instead of back to back.  The same layer
        # always goes to the same stream: its next power iteration is ordered behind this one.
        sn = [c for c in discriminator_convs(model) if c.norm != "weight_norm"]
        if sn_streams and sn:
            cur = torch.cuda.current_stream()
            ev = torch.cuda.Event()
            ev.record(cur)
            out = dict(plan.fold() if refold else plan.folds)
            used = []
            for i, c in enumerate(sn):
                st = sn_streams[i % len(sn_streams)]
                if st not in used:
                    st.wait_event(ev)
                    used.append(st)
                with torch.cuda.stream(st):
                    out[id(c)] = fold(c, dtype, training=training, want_dgrad=want_dgrad)
            for st in used:
                e2 = torch.cuda.Event()
                e2.record(st)
                cur.wait_event(e2)
            return out
        out = dict(plan.fold() if refold else plan.folds)
        for c in sn:
            out[id(c)] = fold(c, dtype, training=training, want_dgrad=want_dgrad)
        return out
    out = {}
    for c in discriminator_convs(model):
        if reuse is not None and c.norm == "weight_norm" and id(c) in reuse:
            out[id(c)] = reuse[id(c)]
        else:
            out[id(c)] = fold(c, dtype, training=training, want_dgrad=want_dgrad, persist=persist)
    return out


@dataclass
class DiscCtx:
    B: int = 0
    T: int = 0
    C: int = 0
    dtype: torch.dtype = torch.float32
    folds: Dict[int, Folded] = field(default_factory=dict)
    subs: List[dict] = field(default_factory=list)


def _heavy_split(subs: Sequence) -> Tuple[List[int], List[int]]:
    """Indices of the sub-discriminators that go to the side stream / stay on the current one: the first (full-rate)
    scale discriminator is about half of the work of a pass, everything else is the other half."""
    heavy = [i for i, (kind, _) in enumerate(subs) if kind == "S"][:1]
    return heavy, [i for i in range(len(subs)) if i not in heavy]


def discriminator_forward(model, x: Tensor, dtype: torch.dtype, folds: Dict[int, Folded], side=None,
                          subset: Optional[Sequence[int]] = None, spread: Optional[Sequence] = None):
    """DiscriminatorSmall.forward / Discriminator.forward (discriminator.py:144-155,180-191).
    x: fp32 [B,T,C].  Returns (results, ctx): results[d] = channels-last feature maps
    [B, H*p, C_j] in `dtype` with the fp32 logits last.  `side`: optional extra CUDA stream; the sub-discriminators
    are independent, so the full-rate scale discriminator runs there while the others run on the current stream.
    `subset`: run only these sub-discriminators (indices into disc_subnets); the other entries stay None.
    `spread`: extra CUDA streams; the (independent) sub-discriminators are dealt round-robin to the current stream and
    these - each stack is a chain of ~6 small dependent launches, five of them back to back was the longest branch."""
    x = x.contiguous().float()
    B, T, Cc = x.shape
    ctx = DiscCtx(B=B, T=T, C=Cc, dtype=dtype, folds=folds)
    subs = disc_subnets(model)
    # multi-scale inputs: fp32, AvgPool1d(4,2,1) between (and after) the scales (discriminator.py:153)
    wanted = set(range(len(subs)) if subset is None else subset)
    last_scale = max([i for i in wanted if subs[i][0] == "S"], default=-1)
    scale_in, xs = {}, x
    for i, (kind, d) in enumerate(subs):
        if kind == "S":
            scale_in[i] = xs
            if subset is None or i < last_scale:      # (the reference also pools once more after the last scale)
                xs = ops.avgpool4(xs)
    results: List = [None] * len(subs)
    sub_ctx: List = [None] * len(subs)

    def run(idx: List[int]) -> None:
        for i in idx:
            kind, d = subs[i]
            fused0 = False
            if kind == "P":
                p = d.period
                t_pad = T + (p - T % p)          # reflect pad is always >= 1 (discriminator.py:36,86)
                phases, t = p, t_pad // p
                l0, f0_ = d.layers[0], folds[id(d.layers[0])]
                # bf16: pad + period view + first conv + LeakyReLU in ONE launch from the fp32 input (K = k*C <= 40);
                # the im2col rows that the first layer's weight gradient wants are rebuilt in the backward pass
                fused0 = (f0_.unfold and dtype == torch.bfloat16 and l0.groups == 1 and l0.dilation == 1 and
                          l0.out_channels % 8 == 0 and t_pad - T < T)
                src = None if fused0 else ops.reflect_pad_right(x, t_pad, dtype)
            else:
                src = ops.cast(scale_in[i], dtype)
                phases, t = 1, scale_in[i].shape[1]
            f0 = folds[id(d.layers[0])]
            if f0.unfold and not fused0:          # im2col rows replace the raw input (kept for the first layer's wgrad)
                src = unfold_input(f0, src, B, t, phases)
            sub = dict(kind=kind, phases=phases, inputs=[src], ts=[t], t_in0=scale_in[i].shape[1] if kind == "S" else T, mod=d)
            fmaps = []
            h = src
            layers = list(d.layers)
            if fused0:
                l0 = layers[0]
                h, t = ops.period_first_layer(x, f0.wf, l0.bias.data, period=phases, c_out=l0.out_channels, k=l0.kernel,
                                              stride=l0.stride, pad=l0.pad, slope=0.1)
                fmaps.append(h); sub["inputs"].append(h); sub["ts"].append(t)
                sub["x0"] = x                     # inputs[0] (None) is rebuilt from this by first_layer_input()
                layers = layers[1:]
            for layer in layers:
                _, h, t = _fwd(folds[id(layer)], h, B, t, phases=phases, act=ACT_LEAKY, want_act=True)
                fmaps.append(h); sub["inputs"].append(h); sub["ts"].append(t)
            logits, _, t = _fwd(folds[id(d.output)], h, B, t, phases=phases, want_raw=True, out_f32=True)
            sub["ts"].append(t)
            fmaps.append(logits)
            if kind == "S":
                sub["x_scale"] = scale_in[i]
            results[i], sub_ctx[i] = fmaps, sub

    heavy, rest = _heavy_split(subs)
    heavy, rest = [i for i in heavy if i in wanted], [i for i in rest if i in wanted]
    if spread:
        todo = heavy + rest
        lanes = [todo[j::len(spread) + 1] for j in range(len(spread) + 1)]
        fork_many(list(spread), [(lambda idx=idx: run(idx)) for idx in lanes if idx])
    elif side is not None and heavy and rest:
        fork_join(side, lambda: run(heavy), lambda: run(rest))
    else:
        run(heavy + rest)
    ctx.subs = sub_ctx
    ctx.keep = (scale_in, xs)
    return results, ctx


def first_layer_input(sub: dict, f: Folded, B: int, dtype: torch.dtype) -> Tensor:
    """The im2col rows of a period stack's first layer when the forward ran it fused (inputs[0] is None): reflect pad +
    unfold of the saved fp32 input - in the backward pass, off the forward's critical path."""
    x, p, t = sub["x0"], sub["phases"], sub["ts"][0]
    src = ops.reflect_pad_right(x, t * p, dtype)
    return unfold_input(f, src, B, t, p)


def split_disc_batch(results: List, ctx: DiscCtx, idx: Sequence[int], n_first: int):
    """A forward over the concatenation [first n_first samples | rest] for the sub-discriminators `idx` ->
    (feature maps of the first part, of the second part, per-sub contexts of the first part for a backward through
    it).  Everything returned is a contiguous leading / trailing slice of the batched tensors (no copies)."""
    res_a: List = [None] * len(results)
    res_b: List = [None] * len(results)
    sub_a: List = [None] * len(results)
    for i in idx:
        res_a[i] = [fm[:n_first] for fm in results[i]]
        res_b[i] = [fm[n_first:] for fm in results[i]]
        sub = dict(ctx.subs[i])
        sub["inputs"] = [t[:n_first] if t is not None else None for t in sub["inputs"]]
        if "x0" in sub:
            sub["x0"] = sub["x0"][:n_first]
        if "x_scale" in sub:
            sub["x_scale"] = sub["x_scale"][:n_first]
        sub_a[i] = sub
    return res_a, res_b, sub_a


def discriminator_backward(model, ctx: DiscCtx, dlogits: Sequence[Optional[Tensor]],
                           dfmaps: Optional[Sequence[Sequence[Optional[Tensor]]]] = None, want_input_grad: bool = False,
                           want_weight_grad: bool = True, plan: Optional[FoldPlan] = None, side=None,
                           spread: Optional[Sequence] = None) -> Optional[Tensor]:
    """Backward through one discriminator forward.
    dlogits[d]: gradient w.r.t. the logits of sub-discriminator d (`dtype`, same shape) or None;
    dfmaps[d][j]: gradient w.r.t. feature map j (`dtype`) or None.
    Returns d/dx fp32 [B,T,C] when want_input_grad.  `side`: optional extra stream for the full-rate scale
    discriminator (see discriminator_forward)."""
    B, T, Cc, dtype, folds = ctx.B, ctx.T, ctx.C, ctx.dtype, ctx.folds
    dev = next(sub for sub in ctx.subs if sub is not None)["inputs"][1].device
    if plan is not None and want_weight_grad:
        ws = plan                                 # caller zeroes the arena and runs plan.backward() after its passes
    else:
        ws = _Workspace([folds[id(c)] for c in discriminator_convs(model)], dev) if want_weight_grad else None
        if ws is not None:
            side = None                           # the bump allocator of _Workspace is not safe across branches
    dx = torch.zeros((B, T, Cc), device=dev, dtype=torch.float32) if want_input_grad else None
    n_sub = len(ctx.subs)
    scale_grad: List = [None] * n_sub             # d/d x_scale of the scale discriminators

    def run(idx: List[int]) -> None:
        for di in idx:
            sub = ctx.subs[di]
            if sub is None:                         # a forward with `subset`: this sub-discriminator ran elsewhere
                continue
            d, phases, inputs, ts = sub["mod"], sub["phases"], sub["inputs"], sub["ts"]
            convs = list(d.layers) + [d.output]
            g = dlogits[di]
            fm_g = dfmaps[di] if dfmaps is not None else None
            if g is None and (fm_g is None or all(t is None for t in fm_g)):
                continue
            if g is None:
                g = torch.zeros((B, ts[-1] * phases, 1), device=dev, dtype=dtype)
            dxin = None
            for j in reversed(range(len(convs))):
                f = folds[id(convs[j])]
                if want_weight_grad:
                    xin = inputs[j] if inputs[j] is not None else first_layer_input(sub, f, B, dtype)
                    _wgrad(f, xin, g, B, ts[j], ts[j + 1], ws, phases=phases)
                if j == 0:
                    if want_input_grad:
                        dxin = _dgrad(f, g, B, ts[1], ts[0], phases=phases, out_f32=True)
                    break
                g = _dgrad(f, g, B, ts[j + 1], ts[j], phases=phases, mask=inputs[j], mask_mode=ACT_LEAKY,
                           add_pre=fm_g[j - 1] if fm_g is not None else None)
            if want_input_grad:
                if sub["kind"] == "P":
                    ops.reflect_pad_right_bwd(dxin, T, dx)      # period discriminators all run in the same branch
                else:
                    scale_grad[di] = dxin

    heavy, rest = _heavy_split([(sub["kind"] if sub is not None else "-", None) for sub in ctx.subs])
    if spread and (plan is not None or not want_weight_grad):   # (a _Workspace bump allocator is not safe across branches)
        # the stacks are independent (reflect_pad_right_bwd adds into dx atomically): the full-rate scale stack on
        # `side` when given, the others dealt round-robin over the current stream and `spread`
        h_here = [i for i in heavy if ctx.subs[i] is not None] if side is not None else []
        todo = [i for i in range(n_sub) if ctx.subs[i] is not None and i not in h_here]
        lanes = [l for l in (todo[j::len(spread) + 1] for j in range(len(spread) + 1)) if l]
        fns = [(lambda idx=idx: run(idx)) for idx in lanes] or [lambda: None]
        streams = list(spread)[:len(fns) - 1]
        if h_here:
            fns.append(lambda: run(h_here)); streams.append(side)
        fork_many(streams, fns)
    elif side is not None and heavy and any(ctx.subs[i] is not None for i in rest):
        fork_join(side, lambda: run(heavy), lambda: run(rest))
    else:
        run(list(range(n_sub)))
    if want_input_grad:
        # x_s(i+1) = avgpool(x_s(i)): fold the chain from the coarsest scale back to the input
        carry = None
        for di in reversed([i for i, sub in enumerate(ctx.subs) if sub is not None and sub["kind"] == "S"]):
            t_in, cur = ctx.subs[di]["t_in0"], scale_grad[di]
            if carry is not None:
                if cur is None:
                    cur = torch.zeros((B, t_in, Cc), device=dev, dtype=torch.float32)
                ops.avgpool4_bwd(carry, t_in, cur)
            carry = cur
        if carry is not None:
            ops.axpy_f32(dx, carry, 1.0)
    return dx


# --------------------------------------------------------------------------------------
# layout helpers + per-layer drop-in forwards (reference layouts)
# --------------------------------------------------------------------------------------
def to_reference_layout(fm: Tensor, kind: str, phases: int) -> Tensor:
    """channels-last [B, H*p, C] -> the reference's [B,C,H,p] (period) or [B,C,T] (scale) view."""
    B, HP, Cc = fm.shape
    if kind == "P":
        return fm.view(B, HP // phases, phases, Cc).permute(0, 3, 1, 2)
    return fm.transpose(1, 2)


def single_conv_forward(mod, x: Tensor) -> Tensor:
    from .autograd import SingleConvFn
    return SingleConvFn.apply(mod, x, *[p for p in mod.parameters()])


def gblock_forward_torch_layout(blk, x: Tensor) -> Tensor:
    from .autograd import GBlockFn
    return GBlockFn.apply(blk, x, *[p for p in blk.parameters()])

