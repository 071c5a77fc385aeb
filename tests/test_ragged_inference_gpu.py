"""Padded batches with per-sample length masks (GPU): stg_conv_masked on both convolution engines, the masked generator
forward against each utterance run alone and against the oracle, and serve_batched against serve.

Tolerances: a masked row is exactly 0 and a kept row is bit-identical to the unmasked call (the mask is a select in the
epilogue); a masked batch against the same utterance alone: rel-L2 1e-6 (fp32) / 1e-2 (bf16, other tile shapes); against
the oracle: 1e-4 / 2e-2 (BASELINE.json north_star)."""
import pytest
import torch

from oracle import ste_gan_oracle as O
from tests.refconv import pack_fwd

pytestmark = pytest.mark.gpu
SELF_TOL = {"fp32": 1e-6, "bf16": 1e-2}
ORACLE_TOL = {"fp32": 1e-4, "bf16": 2e-2}
NAN = float("nan")


def _limits(T):
    """valid rows per sample: tile and sub-tile edges, the sample's end, past it, and a negative count"""
    return [0, 1, 7, 8, 9, 63, 64, 65, 127, 128, 129, T - 1, T, T + 5, -3]


# name, T, c_in, c_out, k, dilation, dup_rows, post_shift (None: no add_post), act, bias, NaN in masked rows of src / add_post
CASES = [
    ("T100_k1_nan", 100, 64, 128, 1, 1, False, 0, "relu", True, True),
    ("T400_dup_post1", 400, 64, 128, 3, 3, True, 1, "relu", True, False),
    ("T400_k1_post1_nan", 400, 128, 64, 1, 1, True, 1, "relu", False, True),
    ("T1500_d9", 1500, 128, 128, 3, 9, False, None, "relu", True, False),
    ("T3000_post0", 3000, 64, 64, 3, 27, False, 0, "relu", True, False),
    ("T1500_tanh_f32", 1500, 128, 8, 3, 1, False, None, "tanh", True, False),
    ("T3000_cdst12", 3000, 64, 12, 3, 1, False, None, "relu", True, False),
    ("T400_cdst12_dup_post1", 400, 64, 12, 3, 1, True, 1, "relu", True, False),
    ("T896_k1_post0_nan", 896, 128, 128, 1, 1, False, 0, "relu", True, True),
    ("T1024_k1_tanh_dup_nan", 1024, 128, 128, 1, 1, True, None, "tanh", True, True),
]
# expected tcgen05 plan per case: staged (1) or direct (0) epilogue
PLANS = {"T100_k1_nan": 1, "T400_dup_post1": 1, "T400_k1_post1_nan": 1, "T1500_d9": 1, "T3000_post0": 1, "T1500_tanh_f32": 0,
         "T3000_cdst12": 0, "T400_cdst12_dup_post1": 0, "T896_k1_post0_nan": 1, "T1024_k1_tanh_dup_nan": 0}


def _run(ops, engine, dtype, case, x, w, bias, post, lens=None, rpu=1):
    name, T, ci, co, k, d, dup, post_shift, act, _, _ = case
    B = x.shape[0]
    tanh = act == "tanh"
    odt = torch.float32 if tanh else dtype
    y = None if tanh else torch.full((B, T, co), 7.0, device="cuda", dtype=odt)
    ya = torch.full((B, T * (2 if dup else 1), co), 7.0, device="cuda", dtype=odt)
    lib = ops._lib.load()
    n0 = lib.stg_launch_count()
    ops.conv(x, w, n_samples=B, t_src=T, t_dst=T, c_src=ci, c_dst=co, k=k, dilation=d, pad=d * (k // 2), bias=bias,
             add_post=post, post_shift=post_shift or 0, act=ops.ACT_TANH if tanh else ops.ACT_RELU, dup_rows=dup,
             y_raw=y, y_act=ya, engine=engine, valid_units=lens, rows_per_unit=rpu)
    torch.cuda.synchronize()
    return y, ya, lib.stg_launch_count() - n0


@pytest.mark.parametrize("rpu", [1, 4], ids=["rows", "units4"])
@pytest.mark.parametrize("eng", ["simt_fp32", "tcgen05_bf16"])
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_conv_masked_equals_masked_unmasked_output(case, eng, rpu):
    from ste_gan_b200 import ops
    name, T, ci, co, k, d, dup, post_shift, act, has_bias, nan = case
    dtype = torch.float32 if eng == "simt_fp32" else torch.bfloat16
    engine = ops.ENGINE_SIMT if eng == "simt_fp32" else ops.ENGINE_TCGEN05
    # rpu = 4: limits rounded up to whole units (the negative count stays negative)
    units = [v if v < 0 else -(-v // rpu) for v in _limits(T)]
    lim = torch.tensor([max(u, 0) * rpu for u in units])
    B = len(units)
    gen = torch.Generator().manual_seed(sum(map(ord, name)))
    x = torch.randn(B, T, ci, generator=gen)
    w = pack_fwd(torch.randn(co, ci, k, generator=gen) / (ci * k) ** 0.5)
    bias = torch.randn(co, generator=gen) if has_bias else None
    post = torch.randn(B, T >> post_shift, co, generator=gen) if post_shift is not None else None
    if engine == ops.ENGINE_TCGEN05:
        d_desc = dict(dtype=1, engine=2, n_samples=B, phases=1, t_src=T, t_dst=T, c_src=ci, c_dst=co, groups=1, k=k,
                      dilation=d, stride=1, pad=d * (k // 2), src=1, w=1, y_act=1)
        assert ops.conv_tc_supported(**d_desc), name
    dev = lambda t: None if t is None else t.to("cuda", dtype).contiguous()   # noqa: E731
    y0, ya0, n_plain = _run(ops, engine, dtype, case, dev(x), dev(w), None if bias is None else bias.cuda(), dev(post))
    if nan:   # garbage the masked rows of the operands a kept row never reads (k = 1: its own input row; post: row >> shift)
        for b in range(B):
            x[b, lim[b]:] = NAN
            if post is not None:
                post[b, -(-int(lim[b]) // (1 << post_shift)):] = NAN
    lens = torch.tensor(units, dtype=torch.int32, device="cuda")
    y, ya, n_masked = _run(ops, engine, dtype, case, dev(x), dev(w), None if bias is None else bias.cuda(), dev(post), lens, rpu)
    assert n_masked == n_plain == 1                                     # same launch plan: no extra kernels
    rows = torch.arange(T, device="cuda")
    keep = rows[None, :] < lim.cuda()[:, None]                          # [B, T]
    if y is not None:
        assert torch.equal(y, torch.where(keep[..., None], y0, torch.zeros_like(y0))), name
    keep_a = keep.repeat_interleave(2, dim=1) if dup else keep
    assert torch.equal(ya, torch.where(keep_a[..., None], ya0, torch.zeros_like(ya0))), name
    assert not torch.isnan(ya).any()


def test_conv_masked_rejects_backward_shapes():
    """Length masks are forward-only: transposed, pair-summed and period-view calls are refused."""
    from ste_gan_b200 import ops
    from ste_gan_b200._lib import StgError
    B, T, c = 2, 64, 64
    x = torch.randn(B, 2 * T, c, device="cuda", dtype=torch.bfloat16)
    w = torch.randn(3, c, c, device="cuda", dtype=torch.bfloat16)
    y = torch.empty(B, 2 * T, c, device="cuda", dtype=torch.bfloat16)
    lens = torch.tensor([10, 20], dtype=torch.int32, device="cuda")
    for kw in (dict(transposed=True, w_fwd_pack=True), dict(transposed=True, t_dst=2 * T, pair_sum=True), dict(phases=2)):
        args = dict(n_samples=B, t_src=T, t_dst=T, c_src=c, c_dst=c, k=3, pad=1, y_raw=y, valid_units=lens)
        args.update(kw)
        with pytest.raises(StgError):
            ops.conv(x, w, **args)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_conv_masked_epilogue_plans(case):
    """The tcgen05 cases above reach both masked kernel instances: staged and direct epilogues.  The masked call launches
    the plan of the same unmasked descriptor."""
    import ctypes as C
    from ste_gan_b200 import _lib
    name, T, ci, co, k, d, dup, post_shift, act, has_bias, _ = case
    tanh = act == "tanh"
    desc = _lib.StgConv(dtype=1, engine=2, n_samples=len(_limits(T)), phases=1, t_src=T, t_dst=T, c_src=ci, c_dst=co, groups=1,
                        k=k, dilation=d, stride=1, pad=d * (k // 2), post_shift=post_shift or 0, act=3 if tanh else 1,
                        dup_rows=int(dup), out_f32=int(tanh), src=1, w=1, bias=1 if has_bias else None,
                        add_post=None if post_shift is None else 1, y_raw=None if tanh else 1, y_act=1)
    out = (C.c_int * 15)()
    assert _lib.load().stg_debug_conv_plan(C.byref(desc), out) == 0
    assert out[1] == PLANS[name], (name, list(out))


# ---------------------------------------------------------------------------------------------
# model level
# ---------------------------------------------------------------------------------------------
LENS = [1500, 1137, 640, 37, 1]
VARIANTS = {   # name: (constructor args, unit_dim, feature type, speaking modes, rows per frame)
    "units": (dict(speech_feature_type="SPEECH_UNITS", speech_feature_size=256), 256, "SPEECH_UNITS", False, 16),
    "mfcc": (dict(speech_feature_type="MFCCS", speech_feature_size=25, channels=256), 25, "MFCCS", False, 8),
    "modes": (dict(speech_feature_type="SPEECH_UNITS", speech_feature_size=256, channels=256,
                   use_speaking_mode_embedding=True), 256, "SPEECH_UNITS", True, 16),
}
_ORACLE = {}


def _generator(variant):
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    kw, *_ = VARIANTS[variant]
    kw = dict(kw)
    torch.manual_seed(0)
    return EMGGeneratorGanTTS(kw.pop("speech_feature_type"), kw.pop("speech_feature_size"), 17, 8, **kw)


def _batch(variant):
    _, du, _, modes, _ = VARIANTS[variant]
    su, sess, _ = O.synthetic_batch(len(LENS), max(LENS), seed=7, unit_dim=du)
    for b, L in enumerate(LENS):
        su[b, L:] = NAN                                                  # padded units never reach a kept row
    mode = torch.tensor([0, 1, 2, 1, 0]) if modes else None
    return su, sess, mode


def _oracle(variant, g):
    if variant not in _ORACLE:
        su, sess, mode = _batch(variant)
        sd = {k: v.detach().cpu().clone() for k, v in g.state_dict().items()}
        with torch.no_grad():
            _ORACLE[variant] = [O.generator_forward(sd, su[b:b + 1, :L], sess[b:b + 1], None if mode is None else mode[b:b + 1],
                                                    speech_feature_type=VARIANTS[variant][2])[0] for b, L in enumerate(LENS)]
    return _ORACLE[variant]


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_masked_generator_equals_each_utterance_alone(variant, prec):
    from ste_gan_b200.inference import UtteranceGenerator
    g = _generator(variant).cuda()
    r = VARIANTS[variant][4]
    su, sess, mode = _batch(variant)
    cu = lambda t: None if t is None else t.cuda()                       # noqa: E731
    ug = UtteranceGenerator(g, prec)
    lens = torch.tensor(LENS, dtype=torch.int32)
    y = ug.generate(su.cuda(), sess.cuda(), cu(mode), lengths=lens.cuda())
    assert y.shape == (len(LENS), r * max(LENS), 8)
    refs = _oracle(variant, g)
    for b, L in enumerate(LENS):
        alone = ug.generate(su[b:b + 1, :L].cuda(), sess[b:b + 1].cuda(), None if mode is None else mode[b:b + 1].cuda())[0]
        assert alone.shape == (r * L, 8)
        assert O.rel_l2(y[b, :r * L], alone) <= SELF_TOL[prec], (b, L)
        assert O.rel_l2(y[b, :r * L], refs[b]) <= ORACLE_TOL[prec], (b, L)
        assert torch.count_nonzero(y[b, r * L:]) == 0, (b, L)
    # the captured graph: one masked graph per (batch, frames) shape serves every length mix
    yg = ug.generate_graph(su, sess, mode, lengths=lens).clone()
    assert O.rel_l2(yg, y) <= SELF_TOL[prec] and not torch.isnan(yg).any()
    perm = list(reversed(range(len(LENS))))
    yp = ug.generate_graph(su[perm], sess[perm], None if mode is None else mode[perm], lengths=lens[perm])
    assert O.rel_l2(yp, y[perm]) <= SELF_TOL[prec]
    assert len(ug._graphs) == 1 and (len(LENS), max(LENS), True) in ug._graphs


def test_masked_generator_rejects_backward():
    from ste_gan_b200 import passes
    g = _generator("mfcc").cuda()
    su, sess, _ = O.synthetic_batch(2, 20, unit_dim=25)
    with pytest.raises(ValueError):
        passes.generator_forward(g, su.cuda(), sess.cuda(), None, torch.float32, True,
                                 lengths=torch.tensor([20, 10], dtype=torch.int32, device="cuda"))


# ---------------------------------------------------------------------------------------------
# serving
# ---------------------------------------------------------------------------------------------
SERVE_LENS = [1, 16, 17, 37, 100, 112, 113, 128, 129, 150, 200, 224, 225, 256, 300, 320, 333, 400, 448, 500, 512, 530, 600, 640]


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_serve_batched_matches_serve(prec):
    """~24 utterances over 13 buckets, 1 frame and bucket edges (16, 112, 128, 224, 256, 320, 448, 512, 640) included."""
    from ste_gan_b200.inference import UtteranceGenerator, plan_batches
    g = _generator("units").cuda()
    gen = torch.Generator().manual_seed(3)
    utts = [(torch.randn(L, 256, generator=gen), torch.randint(0, 17, (), generator=gen)) for L in SERVE_LENS]
    assert len({T for T, _ in plan_batches(SERVE_LENS)}) >= 10
    ref = UtteranceGenerator(g, prec).serve(utts)
    ug = UtteranceGenerator(g, prec, max_graphs=3)
    out = ug.serve_batched(utts, max_batch=4)
    assert sorted(out) == list(range(len(utts)))
    for i, L in enumerate(SERVE_LENS):
        assert out[i].device.type == "cpu" and out[i].shape == ref[i].shape == (16 * L, 8), i
        assert O.rel_l2(out[i], ref[i]) <= SELF_TOL[prec], (i, L)
    assert len(ug._graphs) <= 3
    shards = [ug.serve_batched(utts, rank=r, world=2, max_batch=4) for r in range(2)]
    assert sorted(list(shards[0]) + list(shards[1])) == list(range(len(utts)))    # every index exactly once
    for s in shards:
        for i, y in s.items():
            assert torch.equal(y, out[i]), i
    assert len(ug._graphs) <= 3
