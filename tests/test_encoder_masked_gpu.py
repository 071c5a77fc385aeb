"""Padded batches through the frozen EMG encoder (GPU): masked convolutions at the encoder's strided shapes, the key-length
masked attention kernels, the masked encoder forward against each utterance alone and against the oracle, the per-utterance
score kernel, and UtteranceGenerator.validate_batched.

Tolerances as in test_ragged_inference_gpu.py: a masked row is exactly 0 and a kept row of one kernel is bit-identical to the
same kernel on that sample alone; a masked batch against the same utterance alone: rel-L2 1e-6 (fp32) / 1e-2 (bf16, other tile
shapes); against the oracle: 1e-4 / 2e-2."""
import pytest
import torch
import torch.nn.functional as F

from oracle import emg_encoder_oracle as E
from oracle import ste_gan_oracle as O

pytestmark = pytest.mark.gpu
SELF_TOL = {"fp32": 1e-6, "bf16": 1e-2}
ORACLE_TOL = {"fp32": 1e-4, "bf16": 2e-2}
DT = {"fp32": torch.float32, "bf16": torch.bfloat16}
NAN = float("nan")
M = 100


def _enc_masks(ctx):
    cl = lambda t: t.float().cpu().transpose(1, 2) > 0                  # noqa: E731
    return dict(blocks=[(cl(s["h"]), cl(s["y"])) for s in ctx.blocks], layers=[s["hff"].float().cpu() > 0 for s in ctx.layers])


def _tiny_encoder():
    from ste_gan_b200.models.emg_encoder import EMGEncoderTransformer
    enc = EMGEncoderTransformer(8, 256, 48, **E.TINY_ENCODER)
    sd = {k: (v.float() if v.is_floating_point() else v) for k, v in E.tiny_encoder_state(EMGEncoderTransformer).items()}
    enc.load_state_dict(sd)
    return enc.eval(), sd


def _full_size_encoder():
    """768-d, 8 heads of 96, random init with non-trivial BatchNorm statistics (as test_encoder_full_size_vs_oracle)."""
    from ste_gan_b200.models.emg_encoder import EMGEncoderTransformer
    torch.manual_seed(0)
    enc = EMGEncoderTransformer(8, 256, 48).eval()
    g = torch.Generator().manual_seed(5)
    for mod in enc.modules():
        if isinstance(mod, torch.nn.BatchNorm1d):
            mod.running_mean.normal_(0, 0.3, generator=g); mod.running_var.uniform_(0.5, 1.5, generator=g)
            mod.weight.data.uniform_(0.5, 1.5, generator=g); mod.bias.data.normal_(0, 0.2, generator=g)
    return enc, {k: v.detach().clone() for k, v in enc.state_dict().items()}


# ---------------------------------------------------------------------------------------------
# masked convolutions at the encoder's shapes
# ---------------------------------------------------------------------------------------------
# name, c_in, c_out, k, stride, pad, output frames, output rows per frame: conv1 of a ResBlock, its residual_path, and the
# 8-channel first block (conv1 and residual) through im2col rows
CONV_CASES = [("conv1_k3s2", 128, 256, 3, 2, 1, 150, 4), ("res_k1s2", 128, 256, 1, 2, 0, 150, 4),
              ("conv1_k3s2_r1", 256, 128, 3, 2, 1, 300, 1), ("unfold_k3s2", 8, 128, 3, 2, 1, 100, 8),
              ("unfold_k1s2", 8, 128, 1, 2, 0, 100, 8)]


@pytest.mark.parametrize("eng", ["simt_fp32", "tcgen05_bf16"])
@pytest.mark.parametrize("case", CONV_CASES, ids=[c[0] for c in CONV_CASES])
def test_masked_conv_at_encoder_shapes(case, eng):
    from ste_gan_b200 import ops, passes_encoder as pe
    from ste_gan_b200.passes import _fwd
    name, ci, co, k, s, pad, nf, rate = case
    dtype = torch.float32 if eng == "simt_fp32" else torch.bfloat16
    gen = torch.Generator().manual_seed(sum(map(ord, name)))
    f = pe._pack(torch.randn(co, ci, k, generator=gen).cuda() / (ci * k) ** 0.5, torch.randn(co, generator=gen).cuda(), s, pad, dtype)
    assert f.unfold == name.startswith("unfold")
    t_in, t_out = nf * rate * s, nf * rate
    units = [0, 1, 7, 8, 31, 32, 50, nf - 1, nf, nf + 5, -3]
    B = len(units)
    x = torch.randn(B, t_in, ci, generator=gen)
    lib = ops._lib.load()

    def run(x, lens):
        xd = ops.cast(x.cuda(), dtype) if dtype != torch.float32 else x.cuda()
        src = pe._src(f, xd, B, t_in)
        n0 = lib.stg_launch_count()
        y, ya, t = _fwd(f, src, B, t_in, act=ops.ACT_RELU, want_raw=True, want_act=True, lengths=lens, rate=rate)
        torch.cuda.synchronize()
        assert t == t_out
        return y, ya, lib.stg_launch_count() - n0

    ops.set_engine(ops.ENGINE_SIMT if eng == "simt_fp32" else ops.ENGINE_TCGEN05)
    try:
        y0, ya0, n_plain = run(x, None)
        for b, u in enumerate(units):                                   # input rows no kept output row reads
            x[b, s * rate * max(u, 0):] = NAN
        y, ya, n_masked = run(x, torch.tensor(units, dtype=torch.int32, device="cuda"))
    finally:
        ops.set_engine(None)
    assert n_masked == n_plain == 1
    lim = torch.tensor([max(u, 0) * rate for u in units], device="cuda")
    keep = (torch.arange(t_out, device="cuda")[None, :] < lim[:, None])[..., None]
    assert torch.equal(y, torch.where(keep, y0, torch.zeros_like(y0))), name
    assert torch.equal(ya, torch.where(keep, ya0, torch.zeros_like(ya0))), name
    assert not torch.isnan(y).any() and not torch.isnan(ya).any()


# ---------------------------------------------------------------------------------------------
# masked attention
# ---------------------------------------------------------------------------------------------
def _attn_reference(qkv, emb, H):
    B, L, C3 = qkv.shape
    d = C3 // (3 * H)
    q, k, v = (t.view(B, L, H, d).permute(0, 2, 1, 3) for t in qkv.double().split(H * d, dim=-1))
    logits = torch.einsum("bhqa,bhka->bhqk", q, k) / d ** 0.5 + E.relative_logits(q, emb.double())
    probs = torch.softmax(logits, -1)
    return probs, torch.einsum("bhqk,bhka->bhqa", probs, v).permute(0, 2, 1, 3).reshape(B, L, H * d)


ATTN_GEOMS = [("band", 111), ("band", 257), ("dense", 111), ("dense", 206)]


@pytest.mark.parametrize("d", [4, 96])
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("geom", ATTN_GEOMS, ids=[f"{k}_L{L}" for k, L in ATTN_GEOMS])
def test_masked_attention(geom, prec, d):
    from ste_gan_b200 import ops
    kind, L = geom
    H = 2
    fn = ops.relattn_band_fwd if kind == "band" else ops.relattn_fwd
    lens = [0, 1, 31, 32, 99, 100, L - 1, L, L + 5, -3]
    B = len(lens)
    gen = torch.Generator().manual_seed(L + d)
    qkv = torch.randn(B, L, 3 * H * d, generator=gen)
    if prec == "bf16":
        qkv = qkv.to(torch.bfloat16).float()
    emb = (torch.randn(H, 2 * M - 1, d, generator=gen) * d ** -0.5).cuda()
    clean = qkv.clone()
    for b, n in enumerate(lens):
        qkv[b, max(n, 0):] = NAN                                        # padded q / k / v rows
    o, p = fn(qkv.cuda().to(DT[prec]), emb, H, M, lengths=torch.tensor(lens, dtype=torch.int32, device="cuda"))
    assert not torch.isnan(o).any() and not torch.isnan(p).any()
    W = 2 * M - 1
    for b, n in enumerate(lens):
        n = min(max(n, 0), L)
        assert torch.count_nonzero(o[b, n:]) == 0 and torch.count_nonzero(p[b, :, n:]) == 0, (b, n)
        if n == 0:
            continue
        if kind == "dense":
            assert torch.count_nonzero(p[b, :, :n, n:]) == 0, (b, n)
        else:                                                           # band entries whose key j = i + w - (M - 1) >= n
            j = torch.arange(n, device="cuda")[:, None] + torch.arange(W, device="cuda")[None, :] - (M - 1)
            assert torch.count_nonzero(p[b, :, :n][:, j >= n]) == 0, (b, n)
        o1, p1 = fn(clean[b:b + 1, :n].cuda().to(DT[prec]), emb, H, M)  # the same kernel on this sample alone
        assert torch.equal(o[b, :n], o1[0]), (b, n)
        assert torch.equal(p[b, :, :n, :n] if kind == "dense" else p[b, :, :n], p1[0]), (b, n)
        probs_ref, o_ref = _attn_reference(clean[b:b + 1, :n], emb.cpu(), H)
        tol = 2e-5 if prec == "fp32" else 6e-3
        assert O.rel_l2(o[b, :n], o_ref[0]) < tol, (b, n)


# ---------------------------------------------------------------------------------------------
# masked encoder forward
# ---------------------------------------------------------------------------------------------
ENC_LENS = {"tiny": [1500, 1137, 100, 99, 37, 1, 0], "full": [1500, 250, 99, 1]}


def _encoder(which):
    return _tiny_encoder() if which == "tiny" else _full_size_encoder()


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("which", ["tiny", "full"])
def test_masked_encoder_forward(which, prec):
    from ste_gan_b200 import passes_encoder as pe
    enc, sd = _encoder(which)
    plan = enc.cuda().plan(DT[prec])
    lens = ENC_LENS[which]
    Lmax = max(lens)
    g = torch.Generator().manual_seed(len(lens) + Lmax)
    x = torch.tanh(torch.randn(len(lens), 16 * Lmax, 8, generator=g))
    for b, n in enumerate(lens):
        x[b, 16 * n:] = NAN
    units, logits, ctx = pe.encoder_forward(plan, x.cuda(), need_ctx=False, lengths=torch.tensor(lens, dtype=torch.int32).cuda())
    assert ctx is None and units.shape == (len(lens), Lmax, 256) and logits.shape == (len(lens), Lmax, 48)
    f64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    for b, n in enumerate(lens):
        assert torch.count_nonzero(units[b, n:]) == 0 and torch.count_nonzero(logits[b, n:]) == 0, (b, n)
        if n == 0:
            continue
        xa = x[b:b + 1, :16 * n]
        u1, l1, _ = pe.encoder_forward(plan, xa.cuda(), need_ctx=False)
        assert O.rel_l2(units[b, :n], u1[0]) <= SELF_TOL[prec] and O.rel_l2(logits[b, :n], l1[0]) <= SELF_TOL[prec], (b, n)
        if which == "full" and n > 300 and prec == "bf16":
            continue                        # (the fp64 oracle of the full-size encoder on a 30 s utterance once, in fp32)
        _, _, ctx1 = pe.encoder_forward(plan, xa.cuda(), need_ctx=True)     # the ReLU sign patterns of this utterance
        with torch.no_grad():
            ur, lr = E.emg_encoder_forward(f64, xa.double(), _enc_masks(ctx1))
        assert O.rel_l2(units[b, :n], ur[0]) <= ORACLE_TOL[prec] and O.rel_l2(logits[b, :n], lr[0]) <= ORACLE_TOL[prec], (b, n)


# ---------------------------------------------------------------------------------------------
# scores
# ---------------------------------------------------------------------------------------------
def _score_reference(up, ut, lg, ph, n, sil=47):
    up, ut, lg, ph = up[:n].double(), ut[:n].double(), lg[:n].double(), ph[:n]
    am = lg.argmax(-1)
    return (float(F.pairwise_distance(ut, up, eps=1e-6).sum()), float(F.cross_entropy(lg, ph, reduction="sum")),
            [n, int((am == ph).sum()), int((ph == sil).sum()), int(((am == ph) & (ph != sil)).sum())])


def test_encoder_scores_kernel():
    """Against torch per utterance; ties in the logits (the first maximum wins), a zero-length row, a length past T, rows
    past the end that hold NaN and targets out of range, and a kept target out of range (its cross-entropy sum is NaN)."""
    from ste_gan_b200 import ops
    lens = [100, 37, 1, 0, 150, -4, 64]
    B, T, Du, P = len(lens), 100, 256, 48
    g = torch.Generator().manual_seed(21)
    up, ut = torch.randn(B, T, Du, generator=g), torch.randn(B, T, Du, generator=g)
    lg = torch.randn(B, T, P, generator=g) * 3
    ph = torch.randint(0, P, (B, T), generator=g)
    ph[:, ::7] = 47                                                     # silence
    lg[:, ::3, 5] = 30.0; lg[:, ::3, 9] = 30.0                          # ties: argmax = 5
    ph[:, ::6] = 9
    ph[:, 3::6] = 5
    for b, n in enumerate(lens):
        n = min(max(n, 0), T)
        up[b, n:] = NAN; lg[b, n:] = NAN; ph[b, n:] = 1000
    ph[6, 10] = P                                                       # kept, out of range
    dl = torch.tensor(lens, dtype=torch.int32, device="cuda")
    args = (up.cuda(), ut.cuda(), lg.cuda(), ph.cuda(), dl, 47)
    sums, counts = ops.encoder_scores(*args)
    sums2, counts2 = ops.encoder_scores(*args)
    assert torch.equal(sums.view(torch.int32), sums2.view(torch.int32)) and torch.equal(counts, counts2)   # bit-identical
    for b, n in enumerate(lens):
        n = min(max(n, 0), T)
        if b == 6:
            assert torch.isnan(sums[b, 1])
            ph6 = ph[b].clone(); ph6[10] = 0
            su, _, cnt = _score_reference(up[b], ut[b], lg[b], ph6, n)
            cnt[1] -= int(lg[b, 10].argmax() == 0); cnt[3] -= int(lg[b, 10].argmax() == 0)
        else:
            su, ce, cnt = _score_reference(up[b], ut[b], lg[b], ph[b], n)
            assert abs(float(sums[b, 1]) - ce) <= 1e-5 * max(1.0, abs(ce)), b
        assert abs(float(sums[b, 0]) - su) <= 1e-5 * max(1.0, abs(su)), b
        assert counts[b].tolist() == cnt, (b, counts[b].tolist(), cnt)
    assert counts[3].tolist() == [0, 0, 0, 0] and sums[3].tolist() == [0.0, 0.0]


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_encoder_scores_equal_the_loss_module_per_utterance(prec):
    import ste_gan_b200
    from ste_gan_b200 import passes_encoder as pe
    from ste_gan_b200.inference import EncoderScore
    from ste_gan_b200.losses.emg_encoder_loss import EMGEncoderLoss
    enc, _ = _tiny_encoder()
    enc = enc.cuda()
    lens = [300, 120, 99, 1, 0]
    B, T = len(lens), max(lens)
    g = torch.Generator().manual_seed(4)
    x = torch.tanh(torch.randn(B, 16 * T, 8, generator=g))
    ut, ph = torch.randn(B, T, 256, generator=g), torch.randint(0, 48, (B, T), generator=g)
    for b, n in enumerate(lens):
        x[b, 16 * n:] = NAN; ut[b, n:] = NAN; ph[b, n:] = -7
    dl = torch.tensor(lens, dtype=torch.int32, device="cuda")
    sums, counts = pe.encoder_scores(enc.plan(DT[prec]), x.cuda(), ut.cuda(), ph.cuda(), dl)
    loss = EMGEncoderLoss(enc)
    for b, n in enumerate(lens):
        sc = EncoderScore(float(sums[b, 0]), float(sums[b, 1]), *counts[b].tolist())
        if n == 0:
            assert sc == EncoderScore(0.0, 0.0, 0, 0, 0, 0)
            continue
        with torch.no_grad(), ste_gan_b200.precision(prec):
            out = loss(x[b:b + 1, :16 * n].cuda(), ut[b:b + 1, :n].cuda(), ph[b:b + 1, :n].cuda())
        tol = ORACLE_TOL[prec]
        assert abs(sc.speech_unit_loss - float(out.speech_unit_loss)) <= tol * float(out.speech_unit_loss), b
        assert abs(sc.phoneme_loss - float(out.phoneme_loss)) <= tol * float(out.phoneme_loss), b
        assert sc.num_phones == out.num_phones == n and sc.num_silence_phones == out.num_silence_phones
        if prec == "fp32":
            assert (sc.num_correct_phones, sc.num_correct_phones_no_silence) == \
                (out.num_correct_phones, out.num_correct_phones_no_silence), b


# ---------------------------------------------------------------------------------------------
# validate_batched
# ---------------------------------------------------------------------------------------------
VAL_LENS = [1, 16, 17, 37, 99, 100, 112, 113, 150, 224, 225, 300]


def _validation_set():
    g = torch.Generator().manual_seed(9)
    return [(torch.randn(n, 256, generator=g), torch.randint(0, 17, (), generator=g), torch.randn(n, 256, generator=g),
             torch.randint(0, 48, (n,), generator=g)) for n in VAL_LENS]


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_validate_batched(prec):
    from ste_gan_b200.inference import UtteranceGenerator, aggregate_scores, plan_batches
    from ste_gan_b200.losses.emg_encoder_loss import EMGEncoderLoss
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    import ste_gan_b200
    torch.manual_seed(0)
    gen = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8).cuda()
    enc, _ = _tiny_encoder()
    enc = enc.cuda()
    utts = _validation_set()
    n_buckets = len({T for T, _ in plan_batches(VAL_LENS, 4)})
    ug = UtteranceGenerator(gen, prec, max_graphs=32, emg_encoder=enc)
    captures = []
    real_capture = ug._capture_validate
    ug._capture_validate = lambda *a: (captures.append(a), real_capture(*a))
    scores = ug.validate_batched(utts, max_batch=4)
    assert sorted(scores) == list(range(len(utts)))
    assert len(captures) == n_buckets                                   # one graph per bucket
    # each score equals EMGEncoderLoss on that utterance's serve_batched EMG alone
    emg = UtteranceGenerator(gen, prec).serve_batched([(u[0], u[1]) for u in utts], max_batch=4)
    loss = EMGEncoderLoss(enc)
    for i, (_, _, ut, ph) in enumerate(utts):
        with torch.no_grad(), ste_gan_b200.precision(prec):
            out = loss(emg[i][None].cuda(), ut[None].cuda(), ph[None].cuda())
        sc = scores[i]
        assert sc.num_phones == VAL_LENS[i] and sc.num_silence_phones == out.num_silence_phones
        assert abs(sc.speech_unit_loss - float(out.speech_unit_loss)) <= ORACLE_TOL[prec] * float(out.speech_unit_loss), i
        assert abs(sc.phoneme_loss - float(out.phoneme_loss)) <= ORACLE_TOL[prec] * float(out.phoneme_loss), i
        if prec == "fp32":
            assert (sc.num_correct_phones, sc.num_correct_phones_no_silence) == \
                (out.num_correct_phones, out.num_correct_phones_no_silence), i
    # a second call replays the graphs; two ranks' shards are the union of one rank's dict
    again = ug.validate_batched(utts, max_batch=4)
    assert len(captures) == n_buckets and again == scores
    shards = [ug.validate_batched(utts, rank=r, world=2, max_batch=4) for r in range(2)]
    assert len(captures) == n_buckets
    assert sorted(list(shards[0]) + list(shards[1])) == list(range(len(utts)))
    assert {**shards[0], **shards[1]} == scores
    assert aggregate_scores(list(shards[0].values()) + list(shards[1].values())) == aggregate_scores(scores.values())
    # refold() drops the validation graphs: the next call captures again
    ug.refold()
    assert not ug._graphs
    ug.validate_batched(utts[:1], max_batch=4)
    assert len(captures) == n_buckets + 1


def test_validate_batched_needs_an_encoder():
    from ste_gan_b200.inference import UtteranceGenerator
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    torch.manual_seed(0)
    ug = UtteranceGenerator(EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8, channels=128).cuda(), "bf16")
    with pytest.raises(ValueError, match="emg_encoder"):
        ug.validate_batched(_validation_set()[:2])


def test_masked_encoder_forward_rejects_backward_on_the_device():
    from ste_gan_b200 import passes_encoder as pe
    enc, _ = _tiny_encoder()
    plan = enc.cuda().plan(torch.float32)
    with pytest.raises(ValueError):
        pe.encoder_forward(plan, torch.zeros(2, 160, 8, device="cuda"), need_ctx=True,
                           lengths=torch.tensor([10, 3], dtype=torch.int32, device="cuda"))
