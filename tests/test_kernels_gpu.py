"""Kernel-level parity (GPU): every conv engine through the C ABI against a CPU fp64 conv.

fp32 (CUDA-core engine): relative L2 <= 1e-5.  bf16 tcgen05 engine: inputs are rounded to
bf16 on the host first and the accumulator is read back as fp32, so the only difference
from the fp64 reference is the fp32 accumulation order: relative L2 <= 1e-4 (2e-2 is the
north_star tolerance for bf16 *storage*, checked in the model-level tests).
"""
import pytest
import torch
import torch.nn.functional as F

from tests.refconv import conv_ref, expand_groups, pack_dgrad, pack_fwd, rel_l2, to_virtual, from_virtual, unfold_ref

pytestmark = pytest.mark.gpu

# name, B, phases, T, c_in, c_out, k, dil, stride, pad, groups
CASES = [
    ("g_k3d1", 2, 1, 100, 64, 128, 3, 1, 1, 1, 1),
    ("g_k3d27", 2, 1, 100, 128, 64, 3, 27, 1, 27, 1),
    ("g_k3d9_192", 2, 1, 300, 192, 192, 3, 9, 1, 9, 1),
    ("g_k1_320", 2, 1, 37, 320, 64, 1, 1, 1, 0, 1),
    ("g_k3_768", 1, 1, 100, 768, 384, 3, 3, 1, 3, 1),
    ("s_k15_c8", 2, 1, 200, 8, 128, 15, 1, 1, 7, 1),
    ("s_k37_g4", 2, 1, 200, 128, 256, 37, 1, 2, 18, 4),
    ("s_k37_g16", 2, 1, 100, 256, 512, 37, 1, 2, 18, 16),
    ("s_k41_s4_g16", 1, 1, 128, 256, 512, 41, 1, 4, 20, 16),
    ("s_k5", 1, 1, 50, 512, 128, 5, 1, 1, 2, 1),
    ("s_out", 2, 1, 50, 128, 1, 3, 1, 1, 1, 1),
    ("p3_l1", 2, 3, 67, 8, 32, 3, 1, 1, 2, 1),
    ("p3_l2", 2, 3, 69, 32, 256, 3, 1, 3, 2, 1),
    ("p2_l3", 2, 2, 140, 256, 128, 3, 1, 3, 2, 1),
    ("p5_k5s3", 2, 5, 40, 32, 128, 5, 1, 3, 2, 1),
    ("last", 2, 1, 160, 192, 8, 3, 1, 1, 1, 1),
    ("s_k41_s2_g4_full", 2, 1, 150, 128, 128, 41, 1, 2, 20, 4),
    ("s_k41_g16_full", 1, 1, 60, 1024, 1024, 41, 1, 1, 20, 16),
    ("s_k37_s2_big", 2, 1, 530, 128, 256, 37, 1, 2, 18, 4),
    ("g_k3_c48", 2, 1, 100, 64, 48, 3, 1, 1, 1, 1),      # c_out = 16 mod 32: no multiple of 32 divides it (tcgen05 bn 48)
]


def t_out_of(T, k, d, s, pad):
    return (T + 2 * pad - d * (k - 1) - 1) // s + 1


def make_case(case, seed=0):
    name, B, p, T, ci, co, k, d, s, pad, g = case
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T * p, ci, generator=gen)
    w = torch.randn(co, ci // g, k, generator=gen) / (ci // g * k) ** 0.5
    bias = torch.randn(co, generator=gen)
    To = t_out_of(T, k, d, s, pad)
    dy = torch.randn(B, To * p, co, generator=gen)
    return x, w, bias, dy, To


def _pack_groups(ops, case, engine):
    """tcgen05 engine: the pack groups are the UNITS of the compact-group path (groups of fewer than 16 channels are merged
    into block-diagonal units; everything else keeps the module's own groups)."""
    name, B, p, T, ci, co, k, d, s, pad, g = case
    return ops.tc_pack_groups(ci, co, g) if engine == ops.ENGINE_TCGEN05 else g


def run_fwd(ops, case, dtype, engine, x, w, bias, To):
    name, B, p, T, ci, co, k, d, s, pad, g = case
    dev = "cuda"
    xd = x.to(dev, dtype)
    pg = _pack_groups(ops, case, engine)
    wf = pack_fwd(expand_groups(w, g, pg)).to(dev, dtype)
    g = pg
    y = torch.empty(B, To * p, co, device=dev, dtype=torch.float32)
    ya = torch.empty(B, To * p, co, device=dev, dtype=torch.float32)
    ops.conv(xd, wf, n_samples=B, phases=p, t_src=T, t_dst=To, c_src=ci, c_dst=co, groups=g, k=k, dilation=d,
             stride=s, pad=pad, bias=bias.to(dev), act=ops.ACT_LEAKY, y_raw=y, y_act=ya, engine=engine)
    torch.cuda.synchronize()
    return y.cpu(), ya.float().cpu()


def run_dgrad(ops, case, dtype, engine, dy, w, To):
    name, B, p, T, ci, co, k, d, s, pad, g = case
    dev = "cuda"
    pg = _pack_groups(ops, case, engine)
    # the tensor engine reads the forward pack as an MN-major operand - grouped convs the K-major data-gradient pack
    fwd_pack = engine == ops.ENGINE_TCGEN05 and g == 1
    we = expand_groups(w, g, pg)
    wd = (pack_fwd(we) if fwd_pack else pack_dgrad(we, pg)).to(dev, dtype)
    g = pg
    dx = torch.empty(B, T * p, ci, device=dev, dtype=torch.float32)
    ops.conv(dy.to(dev, dtype), wd, n_samples=B, phases=p, t_src=To, t_dst=T, c_src=co, c_dst=ci, groups=g, k=k,
             dilation=d, stride=s, pad=pad, transposed=True, y_raw=dx, engine=engine, w_fwd_pack=fwd_pack)
    torch.cuda.synchronize()
    return dx.cpu()


def run_wgrad(ops, case, dtype, engine, x, dy, To):
    name, B, p, T, ci, co, k, d, s, pad, g = case
    dev = "cuda"
    ld, span = ops.wgrad_layout(dtype, c_in=ci, c_out=co, k=k, groups=g, stride=s, engine=engine)
    dw = torch.zeros(co * ld, device=dev)
    db = torch.zeros(co, device=dev)
    ops.wgrad(x.to(dev, dtype), dy.to(dev, dtype), dw, db, n_samples=B, phases=p, t_in=T, t_out=To, c_in=ci, c_out=co,
              groups=g, k=k, dilation=d, stride=s, pad=pad, engine=engine)
    torch.cuda.synchronize()
    # element (co, j, ci) at co*ld + j*span + goff(co) + ci  (include/stegan_b200.h, stg_wgrad_layout)
    cin_g, cout_g = ci // g, co // g
    dwv = dw.cpu().view(co, k, span)
    out = torch.empty(co, k, cin_g)
    for c in range(co):
        goff = 0 if (span == cin_g or cout_g >= 128) else ((c // cout_g) % (128 // cout_g)) * cin_g
        out[c] = dwv[c, :, goff:goff + cin_g]
    return out, db.cpu()


def reference(case, x, w, bias, dy):
    name, B, p, T, ci, co, k, d, s, pad, g = case
    xr = x.double().requires_grad_(True)
    wr = w.double().requires_grad_(True)
    y = conv_ref(xr, wr, bias, phases=p, stride=s, dilation=d, pad=pad, groups=g)
    gx, gw = torch.autograd.grad(y, [xr, wr], dy.double())
    return y.detach(), gx, gw.permute(0, 2, 1).contiguous(), dy.double().sum(dim=(0, 1))  # gw -> [co][k][cin_g]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_simt_f32(case):
    from ste_gan_b200 import ops
    x, w, bias, dy, To = make_case(case)
    y_ref, gx_ref, gw_ref, gb_ref = reference(case, x, w, bias, dy)
    y, ya = run_fwd(ops, case, torch.float32, ops.ENGINE_SIMT, x, w, bias, To)
    assert rel_l2(y, y_ref) < 1e-5
    assert rel_l2(ya, F.leaky_relu(y_ref, 0.1)) < 1e-5
    dx = run_dgrad(ops, case, torch.float32, ops.ENGINE_SIMT, dy, w, To)
    assert rel_l2(dx, gx_ref) < 1e-5
    dw, db = run_wgrad(ops, case, torch.float32, ops.ENGINE_SIMT, x, dy, To)
    assert rel_l2(dw, gw_ref) < 1e-5
    assert rel_l2(db, gb_ref) < 1e-5


def _bf(t):
    return t.to(torch.bfloat16).float()


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_simt_bf16(case):
    from ste_gan_b200 import ops
    x, w, bias, dy, To = make_case(case, seed=1)
    x, w, dy = _bf(x), _bf(w), _bf(dy)
    y_ref, gx_ref, gw_ref, gb_ref = reference(case, x, w, bias, dy)
    y, ya = run_fwd(ops, case, torch.bfloat16, ops.ENGINE_SIMT, x, w, bias, To)
    assert rel_l2(y, y_ref) < 1e-4
    assert rel_l2(ya, F.leaky_relu(y_ref, 0.1)) < 1e-2
    assert rel_l2(run_dgrad(ops, case, torch.bfloat16, ops.ENGINE_SIMT, dy, w, To), gx_ref) < 1e-4
    dw, db = run_wgrad(ops, case, torch.bfloat16, ops.ENGINE_SIMT, x, dy, To)
    assert rel_l2(dw, gw_ref) < 1e-4 and rel_l2(db, gb_ref) < 1e-4


def _tc_conv_desc(ops, case, transposed):
    name, B, p, T, ci, co, k, d, s, pad, g = case
    grouped = g > 1
    g = ops.tc_pack_groups(ci, co, g)
    To = t_out_of(T, k, d, s, pad)
    if transposed:
        return dict(dtype=1, engine=2, n_samples=B, phases=p, t_src=To, t_dst=T, c_src=co, c_dst=ci, groups=g, k=k,
                    dilation=d, stride=s, pad=pad, transposed=1, w_fwd_pack=0 if grouped else 1, src=1, w=1, y_raw=1)
    return dict(dtype=1, engine=2, n_samples=B, phases=p, t_src=T, t_dst=To, c_src=ci, c_dst=co, groups=g, k=k,
                dilation=d, stride=s, pad=pad, transposed=0, src=1, w=1, y_raw=1)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_tcgen05_fwd(case):
    from ste_gan_b200 import ops
    if not ops.conv_tc_supported(**_tc_conv_desc(ops, case, False)):
        pytest.skip("shape not taken by the tcgen05 engine")
    x, w, bias, dy, To = make_case(case, seed=2)
    x, w = _bf(x), _bf(w)
    y_ref = conv_ref(x, w, bias, phases=case[2], stride=case[8], dilation=case[7], pad=case[9], groups=case[10])
    y, ya = run_fwd(ops, case, torch.bfloat16, ops.ENGINE_TCGEN05, x, w, bias, To)
    assert rel_l2(y, y_ref) < 1e-4
    assert rel_l2(ya, F.leaky_relu(y_ref, 0.1)) < 1e-2


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_tcgen05_dgrad(case):
    from ste_gan_b200 import ops
    if not ops.conv_tc_supported(**_tc_conv_desc(ops, case, True)):
        pytest.skip("shape not taken by the tcgen05 engine")
    x, w, bias, dy, To = make_case(case, seed=3)
    w, dy = _bf(w), _bf(dy)
    _, gx_ref, _, _ = reference(case, x, w, bias, dy)
    assert rel_l2(run_dgrad(ops, case, torch.bfloat16, ops.ENGINE_TCGEN05, dy, w, To), gx_ref) < 1e-4


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_tcgen05_wgrad(case):
    from ste_gan_b200 import ops, _lib
    import ctypes as C
    name, B, p, T, ci, co, k, d, s, pad, g = case
    To = t_out_of(T, k, d, s, pad)
    wd = _lib.StgWgrad(dtype=1, engine=2, n_samples=B, phases=p, t_in=T, t_out=To, c_in=ci, c_out=co, groups=g, k=k,
                       dilation=d, stride=s, pad=pad)
    if not _lib.load().stg_wgrad_tc_supported(C.byref(wd)):
        pytest.skip("shape not taken by the tcgen05 engine")
    x, w, bias, dy, To = make_case(case, seed=4)
    x, dy = _bf(x), _bf(dy)
    _, _, gw_ref, gb_ref = reference(case, x, w, bias, dy)
    dw, db = run_wgrad(ops, case, torch.bfloat16, ops.ENGINE_TCGEN05, x, dy, To)
    assert rel_l2(dw, gw_ref) < 1e-4
    assert rel_l2(db, gb_ref) < 1e-4


@pytest.mark.parametrize("geom", [(2, 1, 50, 128, 3), (2, 3, 61, 512, 3), (3, 11, 18, 512, 3), (2, 1, 100, 1024, 3), (2, 2, 37, 1024, 5)],
                         ids=["s_c128", "p3_c512", "p11_c512", "s_c1024", "p2_k5"])
def test_logits_layer_kernels(geom):
    """C -> 1 `output` layers (matrix-vector kernels picked by ENGINE_AUTO): forward, masked data-gradient with the
    feature-matching term added, weight + bias gradient."""
    from ste_gan_b200 import ops
    B, p, T, ci, k = geom
    pad = (k - 1) // 2
    case = ("o", B, p, T, ci, 1, k, 1, 1, pad, 1)
    x, w, bias, dy, To = make_case(case, seed=12)
    x, w, dy = _bf(x), _bf(w), _bf(dy)
    y_ref, gx_ref, gw_ref, gb_ref = reference(case, x, w, bias, dy)
    dev, bf = "cuda", torch.bfloat16
    y = torch.empty(B, To * p, 1, device=dev, dtype=torch.float32)
    ops.conv(x.to(dev, bf), pack_fwd(w).to(dev, bf), n_samples=B, phases=p, t_src=T, t_dst=To, c_src=ci, c_dst=1, k=k,
             pad=pad, bias=bias.to(dev), y_raw=y)
    assert rel_l2(y.cpu(), y_ref) < 1e-4
    gen = torch.Generator().manual_seed(5)
    m = _bf(torch.randn(B, T * p, ci, generator=gen)); pre = _bf(torch.randn(B, T * p, ci, generator=gen) * 0.1)
    dx = torch.empty(B, T * p, ci, device=dev, dtype=bf)
    ops.conv(dy.to(dev, bf), pack_fwd(w).to(dev, bf), n_samples=B, phases=p, t_src=To, t_dst=T, c_src=1, c_dst=ci, k=k,
             pad=pad, transposed=True, mask=m.to(dev, bf), mask_mode=ops.ACT_LEAKY, add_pre=pre.to(dev, bf), y_raw=dx,
             w_fwd_pack=True)
    ref = (gx_ref + pre.double()) * torch.where(m > 0, 1.0, 0.1).double()
    assert rel_l2(dx.float().cpu(), ref) < 4e-3        # bf16 output rounding
    dw = torch.zeros(1, k, ci, device=dev); db = torch.zeros(1, device=dev)
    ops.wgrad(x.to(dev, bf), dy.to(dev, bf), dw, db, n_samples=B, phases=p, t_in=T, t_out=To, c_in=ci, c_out=1, k=k, pad=pad)
    assert rel_l2(dw.cpu(), gw_ref) < 1e-4 and rel_l2(db.cpu(), gb_ref) < 1e-4


@pytest.mark.parametrize("engine_dtype", [("simt", torch.float32), ("simt", torch.bfloat16), ("tc", torch.bfloat16)],
                         ids=["simt-f32", "simt-bf16", "tc-bf16"])
def test_fused_epilogue(engine_dtype):
    """pair_sum + add_pre + mask + add_post(shifted) on a data-gradient, and dup_rows + residual on a forward."""
    from ste_gan_b200 import ops
    eng, dtype = engine_dtype
    engine = ops.ENGINE_SIMT if eng == "simt" else ops.ENGINE_TCGEN05
    tol = 1e-5 if dtype == torch.float32 else 2e-2
    dev = "cuda"
    gen = torch.Generator().manual_seed(11)
    B, T, ci, co, k, d = 2, 96, 64, 128, 3, 3
    q = (lambda t: t) if dtype == torch.float32 else _bf
    x = q(torch.randn(B, T, ci, generator=gen)); w = q(torch.randn(co, ci, k, generator=gen) / 14)
    bias = torch.randn(co, generator=gen)
    res = q(torch.randn(B, T // 2, co, generator=gen))
    # forward: y = conv(x) + bias + res[t>>1]; y_act = relu(y) duplicated
    y = torch.empty(B, T, co, device=dev, dtype=dtype); ya = torch.empty(B, 2 * T, co, device=dev, dtype=dtype)
    ops.conv(x.to(dev, dtype), pack_fwd(w).to(dev, dtype), n_samples=B, t_src=T, t_dst=T, c_src=ci, c_dst=co, k=k,
             dilation=d, pad=d, bias=bias.to(dev), add_post=res.to(dev, dtype), post_shift=1, act=ops.ACT_RELU,
             dup_rows=True, y_raw=y, y_act=ya, engine=engine)
    y_ref = conv_ref(x, w, bias, dilation=d, pad=d) + res.double().repeat_interleave(2, dim=1)
    assert rel_l2(y.float().cpu(), y_ref) < tol
    assert rel_l2(ya.float().cpu(), F.relu(y_ref).repeat_interleave(2, dim=1)) < tol
    # data-gradient with pair-sum: dx[t] = (g[2t] + g[2t+1] + pre[t]) * relu'(m[t]) + post[t]
    dy = q(torch.randn(B, T, co, generator=gen))
    pre = q(torch.randn(B, T // 2, ci, generator=gen)); post = q(torch.randn(B, T // 2, ci, generator=gen))
    m = q(torch.randn(B, T // 2, ci, generator=gen))
    dx = torch.empty(B, T // 2, ci, device=dev, dtype=dtype)
    tc = eng == "tc"
    ops.conv(dy.to(dev, dtype), (pack_fwd(w) if tc else pack_dgrad(w, 1)).to(dev, dtype), n_samples=B, t_src=T, t_dst=T,
             c_src=co, c_dst=ci, k=k, dilation=d, pad=d, transposed=True, pair_sum=True, add_pre=pre.to(dev, dtype),
             mask=m.to(dev, dtype), mask_mode=ops.ACT_RELU, add_post=post.to(dev, dtype), y_raw=dx, engine=engine,
             w_fwd_pack=tc)
    xr = x.double().requires_grad_(True)
    (g,) = torch.autograd.grad(conv_ref(xr, w, None, dilation=d, pad=d), xr, dy.double())
    ref = (g[:, 0::2] + g[:, 1::2] + pre.double()) * (m.double() > 0) + post.double()
    assert rel_l2(dx.float().cpu(), ref) < tol


# ---------------------------------------------------------------------------------------------
# weight-norm / spectral-norm folds, input preparation and loss reductions against torch (CPU, fp64)
# ---------------------------------------------------------------------------------------------
FOLD_CASES = [(128, 8, 15, 1), (256, 32, 37, 4), (512, 16, 37, 16), (1024, 512, 5, 1), (1, 512, 3, 1), (768, 320, 1, 1)]


@pytest.mark.parametrize("shape", FOLD_CASES, ids=[str(s) for s in FOLD_CASES])
def test_weightnorm_fold_fwd_bwd(shape):
    from ste_gan_b200 import ops
    co, cg, k, groups = shape
    gen = torch.Generator().manual_seed(co + k)
    v = torch.randn(co, cg, k, generator=gen); g = torch.rand(co, 1, 1, generator=gen) + 0.5
    dwp = torch.randn(co, k, cg, generator=gen)               # packed-layout upstream gradient
    vd, gd = v.double().requires_grad_(True), g.double().requires_grad_(True)
    w = vd * (gd / vd.norm(2, dim=(1, 2), keepdim=True))
    gv, gg = torch.autograd.grad(w, [vd, gd], dwp.double().permute(0, 2, 1))
    wf, wd, scale = ops.weightnorm_fold(v.cuda(), g.cuda(), groups, torch.float32)
    assert rel_l2(wf.cpu(), pack_fwd(w.detach())) < 1e-6
    assert rel_l2(wd.cpu(), pack_dgrad(w.detach(), groups)) < 1e-6
    dv = torch.zeros(co, cg, k, device="cuda"); dg = torch.zeros(co, device="cuda")
    ops.weightnorm_fold_bwd(dwp.cuda(), v.cuda(), g.cuda(), dv, dg, True)
    assert rel_l2(dv.cpu(), gv) < 1e-5 and rel_l2(dg.cpu(), gg.flatten()) < 1e-5


@pytest.mark.parametrize("shape", [(256, 32, 37, 4), (512, 16, 37, 16), (256, 8, 41, 16), (1024, 64, 41, 16)],
                         ids=["g4", "g16", "g16_c8", "g16_c64"])
def test_fold_pack_groups(shape):
    """Pack groups of the tensor engine = the units of the compact-group path: groups keep their own 16 / 32 / 64-channel
    packs, groups of 8 channels are merged pairwise into block-diagonal units; forward and K-major data-gradient packs."""
    from ste_gan_b200 import ops
    co, cg, k, groups = shape
    gen = torch.Generator().manual_seed(co + k)
    v = torch.randn(co, cg, k, generator=gen); g = torch.rand(co, 1, 1, generator=gen) + 0.5
    w = v * (g / v.norm(2, dim=(1, 2), keepdim=True))
    pg = ops.tc_pack_groups(cg * groups, co, groups)
    unit_in, unit_out = cg * groups // pg, co // pg
    assert groups % pg == 0 and unit_in == max(cg, 16) and (unit_out in (16, 32) or unit_out % 64 == 0)
    wf, wd, _ = ops.weightnorm_fold(v.cuda(), g.cuda(), groups, torch.bfloat16, pack_groups=pg)
    we = expand_groups(w, groups, pg)
    for mine, ref in ((wf, pack_fwd(we)), (wd, pack_dgrad(we, pg))):
        mine = mine.float().cpu()
        assert mine.shape == ref.shape and rel_l2(mine, ref) < 4e-3               # bf16 rounding of the packs
        assert torch.equal(mine == 0, ref == 0)                                     # exact block-diagonal structure


@pytest.mark.parametrize("geom", [(2, 1, 200, 8, 128, 15, 1, 1, 7), (2, 3, 67, 8, 32, 3, 1, 1, 2), (2, 5, 41, 8, 32, 5, 1, 3, 2)],
                         ids=["s_k15", "p3_k3", "p5_k5s3"])
def test_unfold_first_layer(geom):
    """C_in = 8 first layers as a 1-tap conv over im2col rows: unfold, unfolded packs, fwd / wgrad / input gradient."""
    from ste_gan_b200 import ops
    B, p, T, ci, co, k, d, s, pad = geom
    case = ("u", B, p, T, ci, co, k, d, s, pad, 1)
    x, w, bias, dy, To = make_case(case, seed=7)
    x, w, dy = _bf(x), _bf(w), _bf(dy)
    y_ref, gx_ref, gw_ref, _ = reference(case, x, w, bias, dy)
    xu = ops.unfold(x.cuda().to(torch.bfloat16), n_samples=B, phases=p, t_src=T, t_dst=To, channels=ci, k=k, dilation=d,
                    stride=s, pad=pad)
    assert torch.equal(xu.float().cpu(), unfold_ref(x, phases=p, k=k, dilation=d, stride=s, pad=pad, t_out=To))
    kp = xu.shape[-1]
    g1 = torch.ones(co, 1, 1)
    wf, wd, _ = ops.weightnorm_fold(w.cuda(), w.norm(2, dim=(1, 2), keepdim=True).cuda(), 1, torch.bfloat16, unfold=True)
    assert wf.shape == (co, kp) and wd.shape == (kp, co)
    y = torch.empty(B, To * p, co, device="cuda", dtype=torch.float32)
    ops.conv(xu, wf, n_samples=B, phases=p, t_src=To, t_dst=To, c_src=kp, c_dst=co, k=1, bias=bias.cuda(), y_raw=y)
    assert rel_l2(y.cpu(), y_ref) < 5e-3          # weights re-rounded to bf16 by the fold
    dw = torch.zeros(co, kp, device="cuda")
    ops.wgrad(xu, dy.cuda().to(torch.bfloat16), dw, None, n_samples=B, phases=p, t_in=To, t_out=To, c_in=kp, c_out=co, k=1)
    assert rel_l2(dw[:, :k * ci].reshape(co, k, ci).cpu(), gw_ref) < 1e-4
    du = torch.empty(B, To * p, kp, device="cuda", dtype=torch.bfloat16)
    ops.conv(dy.cuda().to(torch.bfloat16), wf, n_samples=B, phases=p, t_src=To, t_dst=To, c_src=co, c_dst=kp, k=1,
             transposed=True, y_raw=du, w_fwd_pack=True)
    dx = torch.zeros(B, T * p, ci, device="cuda")
    ops.unfold_bwd(du, dx, n_samples=B, phases=p, t_src=T, t_dst=To, channels=ci, k=k, dilation=d, stride=s, pad=pad)
    assert rel_l2(dx.cpu(), gx_ref) < 1e-2        # du is stored in bf16


@pytest.mark.parametrize("shape", FOLD_CASES[:4], ids=[str(s) for s in FOLD_CASES[:4]])
@pytest.mark.parametrize("training", [True, False])
def test_spectralnorm_fold_fwd_bwd(shape, training):
    from oracle import ste_gan_oracle as O
    from ste_gan_b200 import ops
    co, cg, k, groups = shape
    gen = torch.Generator().manual_seed(co * 3 + k)
    w0 = torch.randn(co, cg, k, generator=gen) / (cg * k) ** 0.5
    u = torch.nn.functional.normalize(torch.randn(co, generator=gen), dim=0)
    v = torch.nn.functional.normalize(torch.randn(cg * k, generator=gen), dim=0)
    dwp = torch.randn(co, k, cg, generator=gen)
    wd_, ud, vd = w0.double().requires_grad_(True), u.double().clone(), v.double().clone()
    w = O.spectral_norm_weight(wd_, ud, vd, training)         # updates ud, vd in place when training
    (gw,) = torch.autograd.grad(w, wd_, dwp.double().permute(0, 2, 1))
    uc, vc = u.cuda(), v.cuda()
    wf, wdp, sigma = ops.spectralnorm_fold(w0.cuda(), uc, vc, groups, training, torch.float32)
    assert rel_l2(uc.cpu(), ud) < 1e-5 and rel_l2(vc.cpu(), vd) < 1e-5
    assert rel_l2(wf.cpu(), pack_fwd(w.detach())) < 1e-5
    assert rel_l2(wdp.cpu(), pack_dgrad(w.detach(), groups)) < 1e-5
    dW = torch.zeros(co, cg, k, device="cuda")
    ops.spectralnorm_fold_bwd(dwp.cuda(), w0.cuda(), uc, vc, sigma, dW, True)
    assert rel_l2(dW.cpu(), gw) < 1e-5


def test_disc_input_prep_and_reductions():
    from ste_gan_b200 import ops
    gen = torch.Generator().manual_seed(9)
    x = torch.randn(3, 101, 8, generator=gen)
    for p in (2, 3, 5, 7, 11):
        tp = 101 + (p - 101 % p)
        ref = F.pad(x.transpose(1, 2), (0, tp - 101), "reflect").transpose(1, 2)
        out = ops.reflect_pad_right(x.cuda(), tp, torch.float32)
        assert torch.equal(out.cpu(), ref)
        g = torch.randn(3, tp, 8, generator=gen)
        xr = x.clone().requires_grad_(True)
        (gx,) = torch.autograd.grad(F.pad(xr.transpose(1, 2), (0, tp - 101), "reflect").transpose(1, 2), xr, g)
        dx = torch.zeros(3, 101, 8, device="cuda")
        ops.reflect_pad_right_bwd(g.cuda(), 101, dx)
        assert rel_l2(dx.cpu(), gx) < 1e-6
    for T in (100, 101):
        xx = torch.randn(2, T, 8, generator=gen)
        xr = xx.clone().requires_grad_(True)
        ref = F.avg_pool1d(xr.transpose(1, 2), 4, 2, 1).transpose(1, 2)
        out = ops.avgpool4(xx.cuda())
        assert rel_l2(out.cpu(), ref) < 1e-6
        g = torch.randn(ref.shape, generator=gen)
        (gx,) = torch.autograd.grad(ref, xr, g)
        dx = torch.zeros(2, T, 8, device="cuda")
        ops.avgpool4_bwd(g.cuda(), T, dx)
        assert rel_l2(dx.cpu(), gx) < 1e-6
    a, b = torch.randn(5, 333, generator=gen), torch.randn(5, 333, generator=gen)
    slot = torch.zeros(2, device="cuda"); da = torch.empty(5, 333, device="cuda"); dl = torch.empty(5, 333, device="cuda")
    ops.l1_mean(a.cuda(), b.cuda(), slot[0:1], 7.0, da)
    ops.mse_const(a.cuda(), 1.0, slot[1:2], 1.0, dl)
    assert abs(slot[0].item() - F.l1_loss(a, b).item()) < 1e-6
    assert abs(slot[1].item() - F.mse_loss(a, torch.ones_like(a)).item()) < 1e-6
    assert rel_l2(da.cpu(), 7.0 * torch.sign(a - b) / a.numel()) < 1e-6
    assert rel_l2(dl.cpu(), 2.0 * (a - 1.0) / a.numel()) < 1e-6


def test_multi_tensor_losses():
    """One-launch feature matching / LSGAN over lists of tensors against torch."""
    from ste_gan_b200 import ops
    gen = torch.Generator().manual_seed(21)
    shapes = [(2, 77, 32), (2, 300, 8), (1, 5, 1024), (3, 33, 1)] * 9          # 36 pairs -> two launches
    pairs = [(torch.randn(sh, generator=gen), torch.randn(sh, generator=gen)) for sh in shapes]
    slot = torch.zeros(3, device="cuda")
    das = ops.l1_mean_multi([(a.cuda().bfloat16(), b.cuda().bfloat16()) for a, b in pairs], slot[2:3], 7.0)
    ref = sum(F.l1_loss(a.bfloat16().float(), b.bfloat16().float()).item() for a, b in pairs)
    assert abs(slot[2].item() - ref) < 1e-4 * ref
    for (a, b), da in zip(pairs, das):
        d = a.bfloat16().float() - b.bfloat16().float()
        assert rel_l2(da.float().cpu(), (7.0 * torch.sign(d) / a.numel()).bfloat16().float()) < 1e-6
    xs = [torch.randn(2, 50 + i, 1, generator=gen) for i in range(16)]
    tg = [0.0] * 8 + [1.0] * 8
    dxs = ops.mse_const_multi([x.cuda() for x in xs], tg, slot, [0] * 8 + [1] * 8, 1.0, torch.bfloat16)
    assert abs(slot[0].item() - sum(F.mse_loss(x, torch.zeros_like(x)).item() for x in xs[:8])) < 1e-5
    assert abs(slot[1].item() - sum(F.mse_loss(x, torch.ones_like(x)).item() for x in xs[8:])) < 1e-5
    for x, t, dx in zip(xs, tg, dxs):
        assert rel_l2(dx.float().cpu(), 2.0 * (x - t) / x.numel()) < 4e-3


def test_adamw_matches_torch():
    from ste_gan_b200 import ops
    gen = torch.Generator().manual_seed(4)
    p0 = torch.randn(10007, generator=gen)
    pr = p0.clone().requires_grad_(True)
    opt = torch.optim.AdamW([pr], lr=2e-4, betas=(0.8, 0.99))
    p, m, v = p0.cuda(), torch.zeros(10007, device="cuda"), torch.zeros(10007, device="cuda")
    step = torch.zeros(1, device="cuda", dtype=torch.int64)
    for i in range(5):
        g = torch.randn(10007, generator=gen)
        pr.grad = g.clone(); opt.step()
        ops.adamw(p, g.cuda(), m, v, step, 2e-4)
    assert int(step.item()) == 5
    assert rel_l2(p.cpu(), pr.detach()) < 1e-6


@pytest.mark.parametrize("geom", [(2, 1600, 2, 3, 1, 2), (3, 1601, 11, 3, 1, 2), (2, 640, 5, 5, 3, 2)], ids=["p2", "p11_odd", "p5_k5s3"])
def test_period_first_layer_fused(geom):
    """stg_period_first_layer (reflect pad + period view + conv + bias + LeakyReLU in one launch) against an fp64
    F.pad(reflect) + Conv2d on bf16-rounded operands."""
    from ste_gan_b200 import ops
    B, T, p, k, s, pad = geom
    C, co = 8, 32
    gen = torch.Generator().manual_seed(11)
    x = torch.randn(B, T, C, generator=gen)
    w = torch.randn(co, C, k, generator=gen) / (C * k) ** 0.5
    bias = torch.randn(co, generator=gen)
    Kp = (k * C + 7) // 8 * 8
    wf = torch.zeros(co, Kp)
    wf[:, :k * C] = w.permute(0, 2, 1).reshape(co, k * C)           # q = j*C + c
    y, h_out = ops.period_first_layer(x.cuda(), wf.cuda().bfloat16(), bias.cuda(), period=p, c_out=co, k=k, stride=s, pad=pad)
    xb, wb = x.bfloat16().double(), w.bfloat16().double()
    t_pad = T + (p - T % p)
    xp = F.pad(xb.transpose(1, 2), (0, t_pad - T), mode="reflect")   # [B,C,t_pad]
    x4 = xp.view(B, C, t_pad // p, p)
    ref = F.leaky_relu(F.conv2d(x4, wb.unsqueeze(-1), bias.double(), stride=(s, 1), padding=(pad, 0)), 0.1)   # [B,co,Ho,p]
    assert ref.shape[2] == h_out
    ref = ref.permute(0, 2, 3, 1).reshape(B, h_out * p, co)
    assert rel_l2(y.float().cpu(), ref) < 5e-3      # bf16 output rounding
