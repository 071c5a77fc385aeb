"""Host-side wrappers: torch tensors in, C-ABI calls out (raw pointers + current stream).

PyTorch is used for device memory and streams only.  Every wrapper checks buffer sizes
before handing raw pointers to the library (an out-of-bounds write on the device is a
fault, not an exception).  No CPU fallback exists: tensors must live on a CUDA device.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import (ACT_LEAKY, ACT_NONE, ACT_RELU, ACT_TANH, BF16, ENGINE_AUTO, ENGINE_SIMT, ENGINE_TCGEN05, F32,
                   StgConv, StgWgrad, check)

Tensor = torch.Tensor
_engine_override: Optional[int] = None  # tests force an engine through this
profile = None  # bench.py sets this to a list: every conv / wgrad launch is then bracketed by CUDA events
flop_log = None  # bench.py sets this to a list: every conv / wgrad launch appends its ALGORITHMIC flops / bytes (no events:
                 # safe under CUDA-graph capture, where it records exactly the launches the timed graphs replay)


def set_engine(engine: Optional[int]) -> None:
    global _engine_override
    _engine_override = engine


def code_of(dtype: torch.dtype) -> int:
    if dtype == torch.float32:
        return F32
    if dtype == torch.bfloat16:
        return BF16
    raise TypeError(f"unsupported dtype {dtype}")


def _ptr(t: Optional[Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _need(t: Optional[Tensor], numel: int, dtype: Optional[torch.dtype], name: str) -> None:
    if t is None:
        return
    if not t.is_cuda:
        raise _lib.StgError(f"{name}: expected a CUDA tensor (there is no CPU fallback)")
    if not t.is_contiguous():
        raise _lib.StgError(f"{name}: expected a contiguous tensor")
    if dtype is not None and t.dtype != dtype:
        raise _lib.StgError(f"{name}: expected {dtype}, got {t.dtype}")
    if t.numel() < numel:
        raise _lib.StgError(f"{name}: buffer too small ({t.numel()} < {numel})")


def conv(src: Tensor, w: Tensor, *, n_samples: int, t_src: int, t_dst: int, c_src: int, c_dst: int, k: int,
         phases: int = 1, groups: int = 1, dilation: int = 1, stride: int = 1, pad: int = 0, transposed: bool = False,
         pair_sum: bool = False, post_shift: int = 0, mask: Optional[Tensor] = None, mask_mode: int = ACT_NONE,
         act: int = ACT_NONE, dup_rows: bool = False, bias: Optional[Tensor] = None, add_pre: Optional[Tensor] = None,
         add_post: Optional[Tensor] = None, y_raw: Optional[Tensor] = None, y_act: Optional[Tensor] = None,
         engine: int = ENGINE_AUTO, w_fwd_pack: bool = False, acct_groups: Optional[int] = None,
         valid_units: Optional[Tensor] = None, rows_per_unit: int = 1) -> None:
    """One StgConv launch (see include/stegan_b200.h for the exact contraction + epilogue).
    w_fwd_pack (transposed only): `w` is the forward pack wf - what the tcgen05 engine wants for data-gradients.
    acct_groups: the MODULE's group count when `groups` is a (merged) pack-group count - only used to account the
    algorithmic FLOPs of the launch (block-diagonal packs run redundant MMAs that are not work).
    valid_units (int32 [n_samples] on the device): stg_conv_masked - output rows >= valid_units[b] * rows_per_unit of
    sample b are written as 0 (forward only)."""
    dt = src.dtype
    nv = n_samples * phases
    t_out = t_dst // 2 if pair_sum else t_dst
    _need(src, nv * t_src * c_src, None, "src")
    _need(w, k * c_dst * (c_src // groups), dt, "w")
    _need(bias, c_dst, torch.float32, "bias")
    _need(add_pre, nv * t_out * c_dst, dt, "add_pre")
    _need(mask, nv * t_out * c_dst, dt, "mask")
    _need(add_post, nv * (t_out >> post_shift) * c_dst, dt, "add_post")
    outs = [t for t in (y_raw, y_act) if t is not None]
    out_f32 = dt != torch.float32 and len(outs) > 0 and all(t.dtype == torch.float32 for t in outs)
    odt = torch.float32 if out_f32 else dt
    _need(y_raw, nv * t_out * c_dst, odt, "y_raw")
    _need(y_act, nv * t_out * c_dst * (2 if dup_rows else 1), odt, "y_act")
    _need(valid_units, n_samples, torch.int32, "valid_units")
    d = StgConv(dtype=code_of(dt), engine=_engine_override if _engine_override is not None else engine,
                n_samples=n_samples, phases=phases, t_src=t_src, t_dst=t_dst, c_src=c_src, c_dst=c_dst, groups=groups,
                k=k, dilation=dilation, stride=stride, pad=pad, transposed=int(transposed), pair_sum=int(pair_sum),
                post_shift=post_shift, mask_mode=mask_mode, act=act, dup_rows=int(dup_rows), out_f32=int(out_f32),
                w_fwd_pack=int(w_fwd_pack), src=_ptr(src), w=_ptr(w), bias=_ptr(bias), add_pre=_ptr(add_pre), mask=_ptr(mask),
                add_post=_ptr(add_post), y_raw=_ptr(y_raw), y_act=_ptr(y_act))
    lib = _lib.load()

    def launch():
        if valid_units is None:
            check(lib.stg_conv(C.byref(d), _stream()), "stg_conv")
        else:
            check(lib.stg_conv_masked(C.byref(d), _ptr(valid_units), rows_per_unit, _stream()), "stg_conv_masked")

    if profile is None and flop_log is None:
        launch()
        return
    if valid_units is None:
        route = {1: "simt", 2: "tcgen05", 3: "matvec"}[lib.stg_conv_route(C.byref(d))]
    else:   # stg_conv_masked never takes the matvec engine
        eng = d.engine if d.engine != ENGINE_AUTO else (ENGINE_TCGEN05 if lib.stg_conv_tc_supported(C.byref(d)) else ENGINE_SIMT)
        route = "tcgen05" if eng == ENGINE_TCGEN05 else "simt"
    ag = acct_groups if acct_groups is not None else groups
    flops = 2.0 * nv * t_src * c_src * k * (c_dst // ag) if transposed else 2.0 * nv * t_dst * c_dst * k * (c_src // ag)
    esz = 2 if dt == torch.bfloat16 else 4
    nbytes = esz * (nv * t_src * c_src + k * c_dst * (c_src // ag)) + sum(
        t.numel() * t.element_size() for t in (add_pre, mask, add_post, y_raw, y_act) if t is not None)
    rec = dict(kind=("dgrad" if transposed else "fwd"), engine=route, flops=flops, bytes=nbytes,
               shape=(n_samples, phases, t_src, t_dst, c_src, c_dst, k, dilation, stride, ag))
    if flop_log is not None:
        flop_log.append(rec)
    if profile is None:
        launch()
        return
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    launch()
    e1.record()
    rec["ingest"] = _ingest(lib)
    # a record replays as fn(desc, *args, stream)
    fn, args = ("stg_conv", ()) if valid_units is None else ("stg_conv_masked", (_ptr(valid_units), rows_per_unit))
    profile.append(dict(rec, events=(e0, e1), desc=d, fn=fn, args=args,
                        keep=(src, w, bias, add_pre, mask, add_post, y_raw, y_act, valid_units)))


def _ingest(lib) -> float:
    """Bytes the launch just issued was planned to pull into shared memory (debug accounting of the tcgen05 engines)."""
    return float(lib.stg_debug_ingest_bytes(1))


def conv_tc_supported(**kw) -> bool:
    d = StgConv(**kw)
    return bool(_lib.load().stg_conv_tc_supported(C.byref(d)))


def wgrad_layout(dtype: torch.dtype, *, c_in: int, c_out: int, k: int, groups: int = 1, stride: int = 1,
                 engine: int = ENGINE_AUTO) -> tuple:
    """(ld, span) of the gradient buffer the selected engine writes (include/stegan_b200.h, stg_wgrad_layout)."""
    d = StgWgrad(dtype=code_of(dtype), engine=_engine_override if _engine_override is not None else engine, n_samples=1,
                 phases=1, t_in=1, t_out=1, c_in=c_in, c_out=c_out, groups=groups, k=k, dilation=1, stride=stride, pad=0)
    ld, span = C.c_int(0), C.c_int(0)
    check(_lib.load().stg_wgrad_layout(C.byref(d), C.byref(ld), C.byref(span)), "stg_wgrad_layout")
    return ld.value, span.value


def wgrad(x: Tensor, dy: Tensor, dw: Optional[Tensor], dbias: Optional[Tensor], *, n_samples: int, t_in: int,
          t_out: int, c_in: int, c_out: int, k: int, phases: int = 1, groups: int = 1, dilation: int = 1,
          stride: int = 1, pad: int = 0, engine: int = ENGINE_AUTO) -> None:
    """dw (layout: wgrad_layout) += ..., dbias[c_out] += column sums of dy (fp32, accumulated)."""
    nv = n_samples * phases
    _need(x, nv * t_in * c_in, None, "x")
    _need(dy, nv * t_out * c_out, x.dtype, "dy")
    if dw is not None:
        ld, _ = wgrad_layout(x.dtype, c_in=c_in, c_out=c_out, k=k, groups=groups, stride=stride, engine=engine)
        _need(dw, c_out * ld, torch.float32, "dw")
    _need(dbias, c_out, torch.float32, "dbias")
    d = StgWgrad(dtype=code_of(x.dtype), engine=_engine_override if _engine_override is not None else engine,
                 n_samples=n_samples, phases=phases, t_in=t_in, t_out=t_out, c_in=c_in, c_out=c_out, groups=groups,
                 k=k, dilation=dilation, stride=stride, pad=pad, x=_ptr(x), dy=_ptr(dy), dw=_ptr(dw), dbias=_ptr(dbias))
    lib = _lib.load()
    if profile is None and flop_log is None:
        check(lib.stg_conv_wgrad(C.byref(d), _stream()), "stg_conv_wgrad")
        return
    route = {1: "simt", 2: "tcgen05", 3: "matvec"}[lib.stg_wgrad_route(C.byref(d))]
    esz = 2 if x.dtype == torch.bfloat16 else 4
    rec = dict(kind="wgrad", engine=route, flops=2.0 * nv * t_out * c_out * k * (c_in // groups),
               bytes=esz * nv * (t_in * c_in + t_out * c_out) + 4 * c_out * k * (c_in // groups),
               shape=(n_samples, phases, t_in, t_out, c_in, c_out, k, dilation, stride, groups))
    if flop_log is not None:
        flop_log.append(rec)
    if profile is None:
        check(lib.stg_conv_wgrad(C.byref(d), _stream()), "stg_conv_wgrad")
        return
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    check(lib.stg_conv_wgrad(C.byref(d), _stream()), "stg_conv_wgrad")
    e1.record()
    rec["ingest"] = _ingest(lib)
    profile.append(dict(rec, events=(e0, e1), desc=d, fn="stg_conv_wgrad", keep=(x, dy, dw, dbias)))


def tc_pack_groups(c_in: int, c_out: int, groups: int) -> int:
    """Group count the tcgen05 engine wants the packs in (narrow groups merged into block-diagonal ones)."""
    return int(_lib.load().stg_tc_pack_groups(c_in, c_out, groups))


def round_up8(n: int) -> int:
    return (n + 7) // 8 * 8


def _pack_shapes(c_out: int, cin_g: int, k: int, groups: int, pack_groups: int, unfold: bool):
    if unfold:
        kp = round_up8(k * cin_g)
        return (c_out, kp), (kp, c_out)
    c_in = cin_g * groups
    return (k, c_out, c_in // pack_groups), (k, c_in, c_out // pack_groups)


def weightnorm_fold(v: Tensor, g: Tensor, groups: int, dtype: torch.dtype, want_dgrad: bool = True, out=None,
                    pack_groups: Optional[int] = None, unfold: bool = False):
    """v [c_out, cin_g, k(,1)], g [c_out,1,1(,1)] -> (wf [k,c_out,c_in/pg], wd [k,c_in,c_out/pg] | None, scale [c_out]);
    unfold: wf [c_out,Kp], wd [Kp,c_out] (see include/stegan_b200.h).
    `out` = (wf, wd, scale) re-uses persistent buffers (fixed addresses for CUDA-graph replay)."""
    c_out, cin_g, k = v.shape[0], v.shape[1], v.shape[2]
    pg = groups if pack_groups is None else pack_groups
    sf, sd = _pack_shapes(c_out, cin_g, k, groups, pg, unfold)
    nf = sf[0] * sf[1] * (sf[2] if len(sf) > 2 else 1)
    _need(v, c_out * cin_g * k, torch.float32, "v"); _need(g, c_out, torch.float32, "g")
    if out is not None:
        wf, wd, scale = out
        _need(wf, nf, dtype, "wf"); _need(wd, nf, dtype, "wd"); _need(scale, c_out, torch.float32, "scale")
    else:
        wf = torch.empty(sf, device=v.device, dtype=dtype)
        wd = torch.empty(sd, device=v.device, dtype=dtype) if want_dgrad else None
        scale = torch.empty((c_out,), device=v.device, dtype=torch.float32)
    check(_lib.load().stg_weightnorm_fold(_ptr(v), _ptr(g), c_out, cin_g, k, groups, pg, _lib.PACK_UNFOLD if unfold else 0,
                                          code_of(dtype), _ptr(wf), _ptr(wd), _ptr(scale), _stream()), "stg_weightnorm_fold")
    return wf, wd, scale


def weightnorm_fold_bwd(dw: Tensor, v: Tensor, g: Tensor, dv: Tensor, dg: Tensor, accumulate: bool, dw_ld: int = 0,
                        dw_span: int = 0, groups: int = 1) -> None:
    """dw in the layout of `wgrad_layout` (defaults: compact [c_out][k][cin_g])."""
    c_out, cin_g, k = v.shape[0], v.shape[1], v.shape[2]
    _need(dw, c_out * max(dw_ld, max(dw_span, cin_g) * k), torch.float32, "dw"); _need(dv, c_out * cin_g * k, torch.float32, "dv")
    _need(dg, c_out, torch.float32, "dg")
    check(_lib.load().stg_weightnorm_fold_bwd(_ptr(dw), dw_ld, dw_span, _ptr(v), _ptr(g), c_out, cin_g, k, groups, _ptr(dv),
                                              _ptr(dg), int(accumulate), _stream()), "stg_weightnorm_fold_bwd")


def spectralnorm_fold(w_orig: Tensor, u: Tensor, v: Tensor, groups: int, training: bool, dtype: torch.dtype,
                      want_dgrad: bool = True, pack_groups: Optional[int] = None, unfold: bool = False, keep_uv: bool = False):
    """In-place power iteration on u, v when training.  Returns (wf, wd, sigma[1]) - with keep_uv also copies of the u, v this
    forward used (written by the same kernels), for its backward."""
    c_out, cin_g, k = w_orig.shape[0], w_orig.shape[1], w_orig.shape[2]
    n = cin_g * k
    pg = groups if pack_groups is None else pack_groups
    sf, sd = _pack_shapes(c_out, cin_g, k, groups, pg, unfold)
    _need(w_orig, c_out * n, torch.float32, "w_orig"); _need(u, c_out, torch.float32, "u"); _need(v, n, torch.float32, "v")
    wf = torch.empty(sf, device=u.device, dtype=dtype)
    wd = torch.empty(sd, device=u.device, dtype=dtype) if want_dgrad else None
    sigma = torch.empty((1,), device=u.device, dtype=torch.float32)
    scratch = torch.empty((c_out + n + 8,), device=u.device, dtype=torch.float32)
    u_used = torch.empty_like(u) if keep_uv else None
    v_used = torch.empty_like(v) if keep_uv else None
    check(_lib.load().stg_spectralnorm_fold(_ptr(w_orig), _ptr(u), _ptr(v), c_out, cin_g, k, groups, pg,
                                            _lib.PACK_UNFOLD if unfold else 0, int(training), code_of(dtype), _ptr(wf),
                                            _ptr(wd), _ptr(sigma), _ptr(scratch), _ptr(u_used), _ptr(v_used), _stream()),
          "stg_spectralnorm_fold")
    if keep_uv:
        return wf, wd, sigma, u_used, v_used
    return wf, wd, sigma


def spectralnorm_fold_bwd(dw: Tensor, w_orig: Tensor, u: Tensor, v: Tensor, sigma: Tensor, dw_orig: Tensor,
                          accumulate: bool, dw_ld: int = 0, dw_span: int = 0, groups: int = 1) -> None:
    c_out, cin_g, k = w_orig.shape[0], w_orig.shape[1], w_orig.shape[2]
    _need(dw, c_out * max(dw_ld, max(dw_span, cin_g) * k), torch.float32, "dw"); _need(dw_orig, c_out * cin_g * k, torch.float32, "dw_orig")
    scratch = torch.empty((8,), device=u.device, dtype=torch.float32)
    check(_lib.load().stg_spectralnorm_fold_bwd(_ptr(dw), dw_ld, dw_span, _ptr(w_orig), _ptr(u), _ptr(v), _ptr(sigma), c_out,
                                                cin_g, k, groups, _ptr(dw_orig), int(accumulate), _ptr(scratch), _stream()),
          "stg_spectralnorm_fold_bwd")


def fold_table(items: list, device) -> Tensor:
    """Device-resident StgFoldItem table (uint8 tensor) from a list of _lib.StgFoldItem."""
    arr = (_lib.StgFoldItem * len(items))(*items)
    return torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(device)


def weightnorm_fold_multi(table: Tensor, n_items: int, total_rows: int, total_tiles: int, dtype: torch.dtype) -> None:
    check(_lib.load().stg_weightnorm_fold_multi(_ptr(table), n_items, total_rows, total_tiles, code_of(dtype), _stream()),
          "stg_weightnorm_fold_multi")


def weightnorm_fold_bwd_multi(table: Tensor, n_items: int, total_rows: int, accumulate: bool = True) -> None:
    check(_lib.load().stg_weightnorm_fold_bwd_multi(_ptr(table), n_items, total_rows, int(accumulate), _stream()),
          "stg_weightnorm_fold_bwd_multi")


def weightnorm_fold_bwd_range(table: Tensor, n_items: int, row_base: int, n_rows: int, accumulate: bool = True) -> None:
    check(_lib.load().stg_weightnorm_fold_bwd_range(_ptr(table), n_items, row_base, n_rows, int(accumulate), _stream()),
          "stg_weightnorm_fold_bwd_range")


def unfold(src: Tensor, *, n_samples: int, phases: int, t_src: int, t_dst: int, channels: int, k: int, dilation: int,
           stride: int, pad: int) -> Tensor:
    """im2col rows [B, t_dst*phases, roundup8(k*C)] of a channels-last (period-view) tensor, same dtype."""
    _need(src, n_samples * phases * t_src * channels, None, "src")
    out = torch.empty((n_samples, t_dst * phases, round_up8(k * channels)), device=src.device, dtype=src.dtype)
    check(_lib.load().stg_unfold(_ptr(src), code_of(src.dtype), n_samples, phases, t_src, t_dst, channels, k, dilation,
                                 stride, pad, _ptr(out), _stream()), "stg_unfold")
    return out


def unfold_bwd(dout: Tensor, dsrc: Tensor, *, n_samples: int, phases: int, t_src: int, t_dst: int, channels: int, k: int,
               dilation: int, stride: int, pad: int) -> None:
    """dsrc (fp32 [B, t_src*phases, C]) += adjoint of `unfold` applied to dout."""
    _need(dout, n_samples * phases * t_dst * round_up8(k * channels), None, "dout")
    _need(dsrc, n_samples * phases * t_src * channels, torch.float32, "dsrc")
    check(_lib.load().stg_unfold_bwd(_ptr(dout), code_of(dout.dtype), n_samples, phases, t_src, t_dst, channels, k,
                                     dilation, stride, pad, _ptr(dsrc), _stream()), "stg_unfold_bwd")


def period_first_layer(x: Tensor, wf: Tensor, bias: Optional[Tensor], *, period: int, c_out: int, k: int, stride: int, pad: int,
                       slope: float = 0.1) -> Tuple[Tensor, int]:
    """Fused first layer of a period stack: fp32 x [B,T,C] -> (bf16 [B, H_out*period, c_out], H_out)."""
    B, T, Cc = x.shape
    _need(x, B * T * Cc, torch.float32, "x")
    t_pad = T + (period - T % period)
    h_out = (t_pad // period + 2 * pad - (k - 1) - 1) // stride + 1
    _need(wf, c_out * round_up8(k * Cc), torch.bfloat16, "wf")
    y = torch.empty((B, h_out * period, c_out), device=x.device, dtype=torch.bfloat16)
    check(_lib.load().stg_period_first_layer(_ptr(x), _ptr(wf), _ptr(bias), B, T, Cc, period, c_out, k, stride, pad, float(slope),
                                             _ptr(y), _stream()), "stg_period_first_layer")
    return y, h_out


def embed_concat(units: Tensor, emb: Optional[Tensor], ids: Optional[Tensor], dtype: torch.dtype) -> Tensor:
    B, T, du = units.shape
    de = 0 if emb is None else emb.shape[1]
    _need(units, B * T * du, torch.float32, "units")
    if emb is not None:
        _need(emb, emb.shape[0] * de, torch.float32, "emb"); _need(ids, B, torch.int64, "ids")
    x0 = torch.empty((B, T, du + de), device=units.device, dtype=dtype)
    check(_lib.load().stg_embed_concat(_ptr(units), _ptr(emb), _ptr(ids), B, T, du, de, code_of(dtype), _ptr(x0),
                                       _stream()), "stg_embed_concat")
    return x0


def embed_concat_bwd(dx0: Tensor, ids: Tensor, d_units: int, demb: Tensor) -> None:
    B, T, Cc = dx0.shape
    de = Cc - d_units
    _need(ids, B, torch.int64, "ids"); _need(demb, de, torch.float32, "demb")
    check(_lib.load().stg_embed_concat_bwd(_ptr(dx0), _ptr(ids), B, T, d_units, de, code_of(dx0.dtype), _ptr(demb),
                                           _stream()), "stg_embed_concat_bwd")


def reflect_pad_right(x: Tensor, t_pad: int, dtype: torch.dtype) -> Tensor:
    B, T, Cc = x.shape
    _need(x, B * T * Cc, torch.float32, "x")
    out = torch.empty((B, t_pad, Cc), device=x.device, dtype=dtype)
    check(_lib.load().stg_reflect_pad_right(_ptr(x), B, T, Cc, t_pad, code_of(dtype), _ptr(out), _stream()),
          "stg_reflect_pad_right")
    return out


def reflect_pad_right_bwd(dout: Tensor, T: int, dx: Tensor) -> None:
    B, t_pad, Cc = dout.shape
    _need(dx, B * T * Cc, torch.float32, "dx"); _need(dout, B * t_pad * Cc, None, "dout")
    check(_lib.load().stg_reflect_pad_right_bwd(_ptr(dout), B, T, Cc, t_pad, code_of(dout.dtype), _ptr(dx), _stream()),
          "stg_reflect_pad_right_bwd")


def avgpool4(x: Tensor) -> Tensor:
    B, T, Cc = x.shape
    _need(x, B * T * Cc, torch.float32, "x")
    out = torch.empty((B, (T + 2 - 4) // 2 + 1, Cc), device=x.device, dtype=torch.float32)
    check(_lib.load().stg_avgpool4(_ptr(x), B, T, Cc, _ptr(out), _stream()), "stg_avgpool4")
    return out


def avgpool4_bwd(dout: Tensor, T: int, dx: Tensor) -> None:
    B, To, Cc = dout.shape
    _need(dout, B * To * Cc, torch.float32, "dout"); _need(dx, B * T * Cc, torch.float32, "dx")
    check(_lib.load().stg_avgpool4_bwd(_ptr(dout), B, T, Cc, _ptr(dx), _stream()), "stg_avgpool4_bwd")


def cast(src: Tensor, dtype: torch.dtype) -> Tensor:
    _need(src, src.numel(), None, "src")
    dst = torch.empty(src.shape, device=src.device, dtype=dtype)
    check(_lib.load().stg_cast(_ptr(src), code_of(src.dtype), _ptr(dst), code_of(dtype), src.numel(), _stream()), "stg_cast")
    return dst


def act_bwd(dy: Tensor, y: Tensor, mode: int, dtype: torch.dtype) -> Tensor:
    """out = dy * act'(y) with the derivative expressed through the activation OUTPUT y (both fp32)."""
    _need(dy, y.numel(), torch.float32, "dy"); _need(y, y.numel(), torch.float32, "y")
    out = torch.empty(y.shape, device=y.device, dtype=dtype)
    check(_lib.load().stg_act_bwd(_ptr(dy), _ptr(y), mode, y.numel(), code_of(dtype), _ptr(out), _stream()), "stg_act_bwd")
    return out


def average_filter(x: Tensor, window: int, pad: bool) -> Tensor:
    """AverageFilter.forward on [B, C, T] fp32 (layers/average_filter.py:22-28)."""
    xc = x.contiguous().float()
    rows, T = xc.numel() // xc.shape[-1], xc.shape[-1]
    t_out = T if pad else T - window + 1
    out = torch.empty(xc.shape[:-1] + (t_out,), device=x.device, dtype=torch.float32)
    check(_lib.load().stg_average_filter(_ptr(xc), rows, T, window, int(pad), _ptr(out), _stream()), "stg_average_filter")
    return out


def relu_rows(x: Tensor, dup: bool) -> Tensor:
    """[B, T, C] -> relu(x) with every row written twice when `dup` ([B, 2T, C])."""
    B, T, Cc = x.shape
    _need(x, B * T * Cc, None, "x")
    out = torch.empty((B, T * (2 if dup else 1), Cc), device=x.device, dtype=x.dtype)
    check(_lib.load().stg_relu_rows(_ptr(x), code_of(x.dtype), B * T, Cc, int(dup), _ptr(out), _stream()), "stg_relu_rows")
    return out


def pair_sum_rows(x: Tensor, rows_out: int, Cc: int) -> Tensor:
    _need(x, 2 * rows_out * Cc, None, "x")
    out = torch.empty((rows_out, Cc), device=x.device, dtype=x.dtype)
    check(_lib.load().stg_pair_sum_rows(_ptr(x), rows_out, Cc, code_of(x.dtype), _ptr(out), _stream()), "stg_pair_sum_rows")
    return out


def axpy_f32(y: Tensor, x: Tensor, alpha: float) -> None:
    _need(y, x.numel(), torch.float32, "y"); _need(x, x.numel(), None, "x")
    check(_lib.load().stg_axpy_f32(_ptr(y), _ptr(x), code_of(x.dtype), float(alpha), x.numel(), _stream()), "stg_axpy_f32")


def td_loss(x_real: Tensor, x_gen: Tensor, losses: Tensor, grad_scale=None, dx_gen: Optional[Tensor] = None) -> None:
    """losses[0:3] <- the three resolutions; dx_gen += sum_i grad_scale[i] * d loss_i / d x_gen when given."""
    B, T, Cc = x_gen.shape
    n = B * T * Cc
    _need(x_real, n, torch.float32, "x_real"); _need(x_gen, n, torch.float32, "x_gen")
    _need(losses, 3, torch.float32, "losses"); _need(dx_gen, n, torch.float32, "dx_gen")
    scratch = torch.empty((6 * n + 8,), device=x_gen.device, dtype=torch.float32)
    gs = (C.c_float * 3)(*([0.0] * 3 if grad_scale is None else [float(g) for g in grad_scale]))
    check(_lib.load().stg_td_loss(_ptr(x_real), _ptr(x_gen), B, T, Cc, _ptr(losses), gs, _ptr(dx_gen),
                                  _ptr(scratch), _stream()), "stg_td_loss")


def n_frames(T: int, win: int, shift: int, pad: bool) -> int:
    return ((T + 2 * (win // 2) if pad else T) - win) // shift + 1


def td_loss_ex(x_real: Tensor, x_gen: Tensor, resolutions, losses: Tensor, *, pad_windows: bool = True, avg_window: int = 9,
               grad_scale=None, dx_gen: Optional[Tensor] = None) -> None:
    """stg_td_loss for any [(win, shift)] list.  grad_scale: None (no backward), a list of host floats, or a DEVICE
    fp32[n_res] tensor (read when the kernels run - no host synchronisation)."""
    B, T, Cc = x_gen.shape
    n, nr = B * T * Cc, len(resolutions)
    _need(x_real, n, torch.float32, "x_real"); _need(x_gen, n, torch.float32, "x_gen")
    _need(losses, nr, torch.float32, "losses"); _need(dx_gen, n, torch.float32, "dx_gen")
    scratch = torch.empty((6 * n + 8,), device=x_gen.device, dtype=torch.float32)
    wins = (C.c_int * nr)(*[int(w) for w, _ in resolutions]); shifts = (C.c_int * nr)(*[int(s_) for _, s_ in resolutions])
    gs_host, gs_dev = None, None
    if isinstance(grad_scale, torch.Tensor):
        _need(grad_scale, nr, torch.float32, "grad_scale")
        gs_dev = grad_scale
    elif grad_scale is not None:
        gs_host = (C.c_float * nr)(*[float(g) for g in grad_scale])
    check(_lib.load().stg_td_loss_ex(_ptr(x_real), _ptr(x_gen), B, T, Cc, nr, wins, shifts, int(pad_windows), int(avg_window),
                                     _ptr(losses), gs_host, _ptr(gs_dev), _ptr(dx_gen), _ptr(scratch), _stream()), "stg_td_loss_ex")


def td_scores(x_real: Tensor, x_gen: Tensor, lengths: Tensor, rate: int, resolutions=None, pad_windows: bool = True,
              avg_window: int = 9) -> Tensor:
    """Per-utterance time-domain feature losses of a padded batch (stg_td_scores): x_real / x_gen fp32 [B, T, C], lengths
    int32 [B] on the device (units of `rate` rows; sample b holds rate * lengths[b] rows, rows past them are never read) ->
    fp32 [B, n_res], entry (b, i) = TimeDomainFeatureLoss(win_i, shift_i, pad_windows, avg_window).time_domain_loss on
    sample b alone; NaN where the reference's reflect padding would raise.  resolutions: [(win, shift)], by default the
    three of MultiTimeDomainFeatureLoss."""
    if resolutions is None:
        from .losses.time_domain_loss import _RES as resolutions
    B, T, Cc = x_gen.shape
    n, nr = B * T * Cc, len(resolutions)
    _need(x_real, n, torch.float32, "x_real"); _need(x_gen, n, torch.float32, "x_gen"); _need(lengths, B, torch.int32, "lengths")
    out = torch.empty((B, nr), device=x_gen.device, dtype=torch.float32)
    scratch = torch.empty((4 * n + 8 * B * (((T + 1) * Cc + 255) // 256),), device=x_gen.device, dtype=torch.float32)
    wins = (C.c_int * nr)(*[int(w) for w, _ in resolutions]); shifts = (C.c_int * nr)(*[int(s_) for _, s_ in resolutions])
    check(_lib.load().stg_td_scores(_ptr(x_real), _ptr(x_gen), B, T, Cc, _ptr(lengths), int(rate), nr, wins, shifts,
                                    int(pad_windows), int(avg_window), _ptr(out), _ptr(scratch), _stream()), "stg_td_scores")
    return out


def td_features(x: Tensor, win: int, shift: int, pad_windows: bool = True, avg_window: int = 9) -> Tensor:
    """[B,T,C] fp32 -> [B,F,C,4] time-domain features (time_domain_loss.py:57-68)."""
    x = x.contiguous().float()
    B, T, Cc = x.shape
    _need(x, B * T * Cc, torch.float32, "x")
    out = torch.empty((B, n_frames(T, win, shift, pad_windows), Cc, 4), device=x.device, dtype=torch.float32)
    scratch = torch.empty((2 * B * T * Cc,), device=x.device, dtype=torch.float32)
    check(_lib.load().stg_td_features(_ptr(x), B, T, Cc, win, shift, int(pad_windows), avg_window, _ptr(out), _ptr(scratch),
                                      _stream()), "stg_td_features")
    return out


def frame_stats(x: Tensor, win: int, shift: int, pad_windows: bool, want_mean: bool, want_power: bool):
    x = x.contiguous().float()
    B, T, Cc = x.shape
    _need(x, B * T * Cc, torch.float32, "x")
    F_ = n_frames(T, win, shift, pad_windows)
    mean = torch.empty((B, F_, Cc), device=x.device, dtype=torch.float32) if want_mean else None
    power = torch.empty((B, F_, Cc), device=x.device, dtype=torch.float32) if want_power else None
    check(_lib.load().stg_frame_stats(_ptr(x), B, T, Cc, win, shift, int(pad_windows), _ptr(mean), _ptr(power), _stream()),
          "stg_frame_stats")
    return mean, power


def window_signal(x: Tensor, win: int, shift: int, pad_windows: bool) -> Tensor:
    x = x.contiguous().float()
    B, T, Cc = x.shape
    _need(x, B * T * Cc, torch.float32, "x")
    out = torch.empty((B, n_frames(T, win, shift, pad_windows), Cc, win), device=x.device, dtype=torch.float32)
    check(_lib.load().stg_window_signal(_ptr(x), B, T, Cc, win, shift, int(pad_windows), _ptr(out), _stream()), "stg_window_signal")
    return out


def mse_const(x: Tensor, target: float, out_slot: Optional[Tensor], grad_scale: float = 0.0, dx: Optional[Tensor] = None) -> None:
    _need(x, x.numel(), None, "x"); _need(dx, x.numel(), None, "dx"); _need(out_slot, 1, torch.float32, "out_slot")
    check(_lib.load().stg_mse_const(_ptr(x), code_of(x.dtype), x.numel(), float(target), _ptr(out_slot), float(grad_scale),
                                    _ptr(dx), code_of(dx.dtype) if dx is not None else 0, _stream()), "stg_mse_const")


def l1_mean(a: Tensor, b: Tensor, out_slot: Optional[Tensor], grad_scale: float = 0.0, da: Optional[Tensor] = None) -> None:
    _need(a, a.numel(), None, "a"); _need(b, a.numel(), a.dtype, "b"); _need(da, a.numel(), a.dtype, "da")
    _need(out_slot, 1, torch.float32, "out_slot")
    check(_lib.load().stg_l1_mean(_ptr(a), _ptr(b), code_of(a.dtype), a.numel(), _ptr(out_slot), float(grad_scale), _ptr(da),
                                  _stream()), "stg_l1_mean")


def l1_mean_multi(pairs, out_slot: Tensor, grad_scale: float, want_grad: bool = True):
    """Feature matching over a list of (a, b) tensor pairs in one launch per 32 pairs:
    out_slot[0] += sum_i mean|a_i - b_i|; returns [da_i] (= grad_scale * sign(a_i - b_i) / n_i) or None."""
    _need(out_slot, 1, torch.float32, "out_slot")
    das = []
    lib = _lib.load()
    for lo in range(0, len(pairs), _lib.MAX_LOSS_ITEMS):
        chunk = pairs[lo:lo + _lib.MAX_LOSS_ITEMS]
        items = (_lib.StgL1Item * len(chunk))()
        for i, (a, b) in enumerate(chunk):
            _need(a, a.numel(), None, "a"); _need(b, a.numel(), a.dtype, "b")
            if a.dtype != chunk[0][0].dtype:
                raise _lib.StgError("l1_mean_multi: mixed dtypes")
            da = torch.empty_like(a) if want_grad else None
            das.append(da)
            items[i] = _lib.StgL1Item(_ptr(a), _ptr(b), _ptr(da), a.numel())
        check(lib.stg_l1_mean_multi(items, len(chunk), code_of(chunk[0][0].dtype), _ptr(out_slot), float(grad_scale), _stream()),
              "stg_l1_mean_multi")
    return das if want_grad else None


def mse_const_multi(xs, targets, slots: Tensor, slot_idx, grad_scale: float, dx_dtype: torch.dtype, outs=None):
    """LSGAN terms over a list of logits tensors in one launch: slots[slot_idx[i]] += mean((x_i - target_i)^2);
    returns [dx_i] in `dx_dtype` (written into outs[i] where given: contiguous, same element count)."""
    n = len(xs)
    if n > _lib.MAX_LOSS_ITEMS:
        raise _lib.StgError("mse_const_multi: too many tensors")
    items = (_lib.StgMseItem * n)()
    dxs = []
    for i, x in enumerate(xs):
        _need(x, x.numel(), xs[0].dtype, "x")
        if outs is not None and outs[i] is not None:
            dx = outs[i]
            _need(dx, x.numel(), dx_dtype, "out")
        else:
            dx = torch.empty(x.shape, device=x.device, dtype=dx_dtype)
        dxs.append(dx)
        items[i] = _lib.StgMseItem(_ptr(x), _ptr(dx), x.numel(), float(targets[i]), int(slot_idx[i]))
    check(_lib.load().stg_mse_const_multi(items, n, code_of(xs[0].dtype), code_of(dx_dtype), _ptr(slots), float(grad_scale),
                                          _stream()), "stg_mse_const_multi")
    return dxs


def adamw(p: Tensor, g: Tensor, m: Tensor, v: Tensor, step: Tensor, lr, beta1: float = 0.8, beta2: float = 0.99,
          eps: float = 1e-8, weight_decay: float = 0.01, grad_scale: float = 1.0, enable: Optional[Tensor] = None,
          keep_step: bool = False) -> None:
    """lr: a Python float, or a device fp32[1] tensor read by the kernel when it RUNS (graph-safe schedules).
    enable: optional device int32[1]; 0 skips the update (step counter included), an executed update clears it.
    keep_step: do not increment `step` (a later slice of a network whose first slice counted this optimiser step)."""
    _need(enable, 1, torch.int32, "enable")
    n = p.numel()
    lr_dev = None
    if isinstance(lr, torch.Tensor):
        _need(lr, 1, torch.float32, "lr")
        lr_dev, lr = lr, 0.0
    for t, nm in ((p, "p"), (g, "g"), (m, "m"), (v, "v")):
        _need(t, n, torch.float32, nm)
    _need(step, 1, torch.int64, "step")
    check(_lib.load().stg_adamw(_ptr(p), _ptr(g), _ptr(m), _ptr(v), n, float(lr), _ptr(lr_dev), beta1, beta2, eps, weight_decay,
                                _ptr(step), grad_scale, _ptr(enable), int(keep_step), _stream()), "stg_adamw")


# ---- EMG-encoder perceptual losses (SURVEY.md 8f rank 1)
def layernorm(x: Tensor, gamma: Tensor, beta: Tensor, eps: float = 1e-5) -> Tuple[Tensor, Tensor]:
    """nn.LayerNorm over the last axis of a contiguous [..., D] tensor -> (y, stats [rows, 2] = mean, rstd)."""
    D = x.shape[-1]
    rows = x.numel() // D
    _need(x, rows * D, None, "x"); _need(gamma, D, torch.float32, "gamma"); _need(beta, D, torch.float32, "beta")
    y = torch.empty_like(x)
    stats = torch.empty((rows, 2), device=x.device, dtype=torch.float32)
    check(_lib.load().stg_layernorm_fwd(_ptr(x), code_of(x.dtype), _ptr(gamma), _ptr(beta), rows, D, float(eps), _ptr(y), _ptr(stats),
                                        _stream()), "stg_layernorm_fwd")
    return y, stats


def layernorm_bwd(dy: Tensor, x: Tensor, stats: Tensor, gamma: Tensor) -> Tensor:
    D = x.shape[-1]
    rows = x.numel() // D
    _need(dy, rows * D, x.dtype, "dy"); _need(x, rows * D, None, "x"); _need(stats, rows * 2, torch.float32, "stats")
    dx = torch.empty_like(x)
    check(_lib.load().stg_layernorm_bwd(_ptr(dy), _ptr(x), code_of(x.dtype), _ptr(stats), _ptr(gamma), rows, D, _ptr(dx), _stream()),
          "stg_layernorm_bwd")
    return dx


def relattn_fwd(qkv: Tensor, emb: Tensor, n_head: int, max_rel: int, lengths: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """qkv [B, L, 3*H*d] -> (o [B, L, H*d], probs fp32 [B, H, L, L]); emb fp32 [H, 2*max_rel-1, d].
    lengths (int32 [B] on the device): stg_relattn_fwd_masked - sample b attends over its first lengths[b] rows only, its
    rows past them are 0."""
    B, L, C3 = qkv.shape
    d = C3 // (3 * n_head)
    _need(qkv, B * L * C3, None, "qkv"); _need(emb, n_head * (2 * max_rel - 1) * d, torch.float32, "emb")
    _need(lengths, B, torch.int32, "lengths")
    o = torch.empty((B, L, n_head * d), device=qkv.device, dtype=qkv.dtype)
    probs = torch.empty((B, n_head, L, L), device=qkv.device, dtype=torch.float32)
    args = (_ptr(qkv), code_of(qkv.dtype), _ptr(emb), B, L, n_head, d, max_rel, float(d) ** -0.5, _ptr(o), _ptr(probs))
    if lengths is None:
        check(_lib.load().stg_relattn_fwd(*args, _stream()), "stg_relattn_fwd")
    else:
        check(_lib.load().stg_relattn_fwd_masked(*args, _ptr(lengths), _stream()), "stg_relattn_fwd_masked")
    return o, probs


def relattn_bwd(qkv: Tensor, emb: Tensor, probs: Tensor, dout: Tensor, n_head: int, max_rel: int) -> Tensor:
    B, L, C3 = qkv.shape
    d = C3 // (3 * n_head)
    _need(qkv, B * L * C3, None, "qkv"); _need(dout, B * L * n_head * d, qkv.dtype, "dout")
    _need(probs, B * n_head * L * L, torch.float32, "probs")
    dqkv = torch.empty_like(qkv)
    check(_lib.load().stg_relattn_bwd(_ptr(qkv), code_of(qkv.dtype), _ptr(emb), _ptr(probs), _ptr(dout), B, L, n_head, d, max_rel,
                                      float(d) ** -0.5, _ptr(dqkv), _stream()), "stg_relattn_bwd")
    return dqkv


def relattn_dense_supported(L: int, d: int, need_bwd: bool) -> bool:
    """Whether relattn_fwd (and, with need_bwd, relattn_bwd) take sequence length L at head dim d (host-only query)."""
    return bool(_lib.load().stg_relattn_dense_supported(int(L), int(d), int(bool(need_bwd))))


def relattn_band_fwd(qkv: Tensor, emb: Tensor, n_head: int, max_rel: int,
                     lengths: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """relattn_fwd at any L -> (o [B, L, H*d], probs_band fp32 [B, H, L, 2*max_rel-1]): entry (i, w) is the probability of key
    j = i + w - (max_rel - 1), 0 where that j is outside [0, L).  lengths: as relattn_fwd (stg_relattn_band_fwd_masked)."""
    B, L, C3 = qkv.shape
    d = C3 // (3 * n_head)
    _need(qkv, B * L * C3, None, "qkv"); _need(emb, n_head * (2 * max_rel - 1) * d, torch.float32, "emb")
    _need(lengths, B, torch.int32, "lengths")
    o = torch.empty((B, L, n_head * d), device=qkv.device, dtype=qkv.dtype)
    probs = torch.empty((B, n_head, L, 2 * max_rel - 1), device=qkv.device, dtype=torch.float32)
    args = (_ptr(qkv), code_of(qkv.dtype), _ptr(emb), B, L, n_head, d, max_rel, float(d) ** -0.5, _ptr(o), _ptr(probs))
    if lengths is None:
        check(_lib.load().stg_relattn_band_fwd(*args, _stream()), "stg_relattn_band_fwd")
    else:
        check(_lib.load().stg_relattn_band_fwd_masked(*args, _ptr(lengths), _stream()), "stg_relattn_band_fwd_masked")
    return o, probs


def relattn_band_bwd(qkv: Tensor, emb: Tensor, probs: Tensor, dout: Tensor, n_head: int, max_rel: int) -> Tensor:
    """Input gradient of relattn_band_fwd from its band-layout probabilities."""
    B, L, C3 = qkv.shape
    d = C3 // (3 * n_head)
    _need(qkv, B * L * C3, None, "qkv"); _need(dout, B * L * n_head * d, qkv.dtype, "dout")
    _need(emb, n_head * (2 * max_rel - 1) * d, torch.float32, "emb")
    _need(probs, B * n_head * L * (2 * max_rel - 1), torch.float32, "probs")
    dqkv = torch.empty_like(qkv)
    scratch = torch.empty((B, n_head, L), device=qkv.device, dtype=torch.float32)
    check(_lib.load().stg_relattn_band_bwd(_ptr(qkv), code_of(qkv.dtype), _ptr(emb), _ptr(probs), _ptr(dout), B, L, n_head, d,
                                           max_rel, float(d) ** -0.5, _ptr(dqkv), _ptr(scratch), _stream()), "stg_relattn_band_bwd")
    return dqkv


def encoder_losses(unit_pred: Tensor, unit_target: Tensor, logits: Tensor, phoneme_target: Tensor, slots: Tensor,
                   gs_units: float = 0.0, gs_phonemes: float = 0.0, grad_dtype: Optional[torch.dtype] = None):
    """slots[0] += speech-unit loss, slots[1] += phoneme loss; returns (d_units, d_logits) in grad_dtype (None: no gradients)."""
    N, Du = unit_pred.numel() // unit_pred.shape[-1], unit_pred.shape[-1]
    P_ = logits.shape[-1]
    _need(unit_pred, N * Du, torch.float32, "unit_pred"); _need(unit_target, N * Du, torch.float32, "unit_target")
    _need(logits, N * P_, torch.float32, "logits"); _need(phoneme_target, N, torch.int64, "phoneme_target")
    _need(slots, 2, torch.float32, "slots")
    du = torch.empty(unit_pred.shape, device=unit_pred.device, dtype=grad_dtype) if grad_dtype is not None else None
    dl = torch.empty(logits.shape, device=logits.device, dtype=grad_dtype) if grad_dtype is not None else None
    check(_lib.load().stg_encoder_losses(_ptr(unit_pred), _ptr(unit_target), _ptr(logits), _ptr(phoneme_target), N, Du, P_, _ptr(slots),
                                         float(gs_units), float(gs_phonemes), _ptr(du), _ptr(dl),
                                         code_of(grad_dtype) if grad_dtype is not None else F32, _stream()), "stg_encoder_losses")
    return du, dl


def encoder_scores(unit_pred: Tensor, unit_target: Tensor, logits: Tensor, phoneme_target: Tensor, lengths: Tensor,
                   silence_index: int) -> Tuple[Tensor, Tensor]:
    """Per-utterance EMGEncoderLoss of a padded batch (stg_encoder_scores): unit_pred / unit_target fp32 [B, T, Du], logits fp32
    [B, T, P], phoneme_target int64 [B, T], lengths int32 [B] (frames; rows past them are never read) ->
    (sums fp32 [B, 2] = (sum of unit distances, sum of cross-entropies), counts int32 [B, 4] = (frames, correct phones,
    silence phones, correct non-silence phones))."""
    B, T, Du = unit_pred.shape
    P_ = logits.shape[-1]
    _need(unit_pred, B * T * Du, torch.float32, "unit_pred"); _need(unit_target, B * T * Du, torch.float32, "unit_target")
    _need(logits, B * T * P_, torch.float32, "logits"); _need(phoneme_target, B * T, torch.int64, "phoneme_target")
    _need(lengths, B, torch.int32, "lengths")
    sums = torch.empty((B, 2), device=unit_pred.device, dtype=torch.float32)
    counts = torch.empty((B, 4), device=unit_pred.device, dtype=torch.int32)
    check(_lib.load().stg_encoder_scores(_ptr(unit_pred), _ptr(unit_target), _ptr(logits), _ptr(phoneme_target), _ptr(lengths),
                                         B, T, Du, P_, int(silence_index), _ptr(sums), _ptr(counts), _stream()),
          "stg_encoder_scores")
    return sums, counts
