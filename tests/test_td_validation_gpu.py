"""Time-domain validation of padded batches (GPU): the per-utterance score kernel stg_td_scores against the fp64 oracle, the loss
modules and itself; UtteranceGenerator.validate_batched(real_emg=...) against the per-utterance modules; speaking-mode
generators in serve_batched / validate_batched.

Tolerances: the kernel against the fp64 oracle and the modules 1e-5 relative; validate_batched against the modules on the
serve_batched EMG 1e-4 (fp32) / 2e-2 (bf16); a masked batch against each utterance alone: rel-L2 1e-6 (fp32) / 1e-2 (bf16),
as test_ragged_inference_gpu.py."""
import pytest
import torch

from oracle import ste_gan_oracle as O

pytestmark = pytest.mark.gpu
NAN = float("nan")
SELF_TOL = {"fp32": 1e-6, "bf16": 1e-2}
TD_TOL = {"fp32": 1e-4, "bf16": 2e-2}
DEFAULT = [(20, 8), (51, 13), (80, 16)]


def _legal(n, win, pad, avg):
    """The reference's F.pad(..., 'reflect') and unfold take an n-row signal."""
    return n > avg // 2 and (n > win // 2 if pad else n >= win)


def _bits(t):
    return t.contiguous().view(torch.int32)


def _rel(a, b):
    return abs(a - b) / max(abs(b), 1e-30)


# (resolutions, pad_windows, avg_window, rows per unit)
KERNEL_CASES = {"default": (DEFAULT, True, 9, 4), "nondefault_avg5": ([(33, 5), (20, 8)], True, 5, 4),
                "unpadded": (DEFAULT, False, 9, 8), "unpadded_avg5": ([(51, 13)], False, 5, 2)}


def _kernel_lengths(res, pad, avg, rate, Tu):
    """Units: full, the shortest legal for every resolution, one unit above it, zero, negative, past T, and lengths legal for
    some resolutions only."""
    legal_all = next(u for u in range(Tu + 1) if all(_legal(rate * u, w, pad, avg) for w, _ in res))
    return [Tu, legal_all, legal_all + 1, 0, -3, Tu + 5, legal_all - 1, 1, Tu // 2 + 1, 7]


@pytest.mark.parametrize("case", list(KERNEL_CASES), ids=list(KERNEL_CASES))
def test_td_scores_kernel(case):
    from ste_gan_b200 import ops
    from ste_gan_b200.losses.time_domain_loss import TimeDomainFeatureLoss
    res, pad, avg, rate = KERNEL_CASES[case]
    Tu = 60
    T = rate * Tu
    units = _kernel_lengths(res, pad, avg, rate, Tu)
    B = len(units)
    g = torch.Generator().manual_seed(len(case))
    xr, xg = torch.randn(B, T, 8, generator=g), torch.randn(B, T, 8, generator=g) * 0.7 + 0.1
    clean_r, clean_g = xr.clone(), xg.clone()
    rows = [rate * min(max(u, 0), Tu) for u in units]
    for b, n in enumerate(rows):
        xr[b, n:] = NAN; xg[b, n:] = NAN                                # padded rows are never read
    lens = torch.tensor(units, dtype=torch.int32, device="cuda")
    out = ops.td_scores(xr.cuda(), xg.cuda(), lens, rate, res, pad, avg)
    assert out.shape == (B, len(res))
    again = ops.td_scores(xr.cuda(), xg.cuda(), lens, rate, res, pad, avg)
    assert torch.equal(_bits(out), _bits(again))
    n_kept = 0
    for b, n in enumerate(rows):
        alone = None
        if n > 0:                                                       # the same call at B = 1, T = n_b
            alone = ops.td_scores(clean_r[b:b + 1, :n].cuda(), clean_g[b:b + 1, :n].cuda(),
                                  torch.tensor([n // rate], dtype=torch.int32, device="cuda"), rate, res, pad, avg)
            assert torch.equal(_bits(out[b]), _bits(alone[0])), (case, b, n)
        for i, (w, s) in enumerate(res):
            v = float(out[b, i])
            if not _legal(n, w, pad, avg):
                assert v != v, (case, b, n, w)                          # NaN
                continue
            n_kept += 1
            ref = float(O.td_loss(clean_r[b:b + 1, :n].double(), clean_g[b:b + 1, :n].double(), w, s, pad, avg))
            assert _rel(v, ref) <= 1e-5, (case, b, n, w, v, ref)
            mod = TimeDomainFeatureLoss(8, w, s, pad, avg)                  # the module through stg_td_loss_ex
            with torch.no_grad():
                m = float(mod(clean_r[b:b + 1, :n].cuda(), clean_g[b:b + 1, :n].cuda()))
            assert _rel(v, m) <= 1e-5, (case, b, n, w, v, m)
    assert n_kept >= 5 * len(res)


def test_td_scores_equal_the_multi_resolution_module_and_replay_bit_identically():
    from ste_gan_b200 import ops
    from ste_gan_b200.losses.time_domain_loss import MultiTimeDomainFeatureLoss
    units = [1500, 1137, 3, 0, 640, 37]
    B, T = len(units), 16 * max(units)
    g = torch.Generator().manual_seed(11)
    xr, xg = torch.randn(B, T, 8, generator=g).cuda(), torch.tanh(torch.randn(B, T, 8, generator=g)).cuda()
    lens = torch.tensor(units, dtype=torch.int32, device="cuda")
    eager = ops.td_scores(xr, xg, lens, 16)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.td_scores(xr, xg, lens, 16)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = ops.td_scores(xr, xg, lens, 16)
    graph.replay()
    first = captured.clone()
    graph.replay()
    assert torch.equal(_bits(first), _bits(captured)) and torch.equal(_bits(first), _bits(eager))
    mod = MultiTimeDomainFeatureLoss(8)
    for b, u in enumerate(units):
        if u == 0:
            assert torch.isnan(eager[b]).all()
            continue
        with torch.no_grad():
            total, parts = mod.time_domain_loss(xr[b:b + 1, :16 * u], xg[b:b + 1, :16 * u])
        for i in range(3):
            assert _rel(float(eager[b, i]), float(parts[i])) <= 1e-5, (b, u, i)
        assert _rel(float(eager[b].sum()), float(total)) <= 1e-5, (b, u)


# ---------------------------------------------------------------------------------------------
# validate_batched(real_emg=...)
# ---------------------------------------------------------------------------------------------
VAL_LENS = [3, 16, 17, 37, 99, 100, 112, 113, 150, 224, 225, 300]


def _tiny_encoder():
    from oracle import emg_encoder_oracle as E
    from ste_gan_b200.models.emg_encoder import EMGEncoderTransformer
    enc = EMGEncoderTransformer(8, 256, 48, **E.TINY_ENCODER)
    enc.load_state_dict({k: (v.float() if v.is_floating_point() else v)
                         for k, v in E.tiny_encoder_state(EMGEncoderTransformer).items()})
    return enc.eval().cuda()


def _validation_set(lens, D=256, r=16, seed=9):
    g = torch.Generator().manual_seed(seed)
    utts = [(torch.randn(n, D, generator=g), torch.randint(0, 17, (), generator=g), torch.randn(n, 256, generator=g),
             torch.randint(0, 48, (n,), generator=g)) for n in lens]
    real = [torch.tanh(torch.randn(r * n, 8, generator=g)) for n in lens]
    return utts, real


def _module_td(real, emg):
    from ste_gan_b200.losses.time_domain_loss import MultiTimeDomainFeatureLoss
    with torch.no_grad():
        _, parts = MultiTimeDomainFeatureLoss(8).time_domain_loss(real[None].cuda(), emg[None].cuda())
    return [float(p) for p in parts]


def _counting(ug):
    captures = []
    real_capture = ug._capture_validate
    ug._capture_validate = lambda *a: (captures.append(a), real_capture(*a))
    return captures


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_validate_batched_with_real_emg(prec):
    from ste_gan_b200.inference import (TdScore, UtteranceGenerator, ValidationScore, aggregate_td, plan_batches)
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    torch.manual_seed(0)
    gen = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8).cuda()
    utts, real = _validation_set(VAL_LENS)
    n_buckets = len({T for T, _ in plan_batches(VAL_LENS, 4)})
    ug = UtteranceGenerator(gen, prec, max_graphs=32, emg_encoder=_tiny_encoder())
    captures = _counting(ug)
    scores = ug.validate_batched(utts, max_batch=4, real_emg=real)
    assert sorted(scores) == list(range(len(utts))) and len(captures) == n_buckets
    emg = UtteranceGenerator(gen, prec).serve_batched([u[:2] for u in utts], max_batch=4)
    for i in range(len(utts)):
        sc = scores[i]
        assert isinstance(sc, ValidationScore) and isinstance(sc.td, TdScore) and len(sc.td.values) == 3
        ref = _module_td(real[i], emg[i])
        for v, m in zip(sc.td.values, ref):
            assert _rel(v, m) <= TD_TOL[prec], (i, v, m)
        assert _rel(sc.td.loss, sum(ref)) <= TD_TOL[prec], i
    # the encoder scores are those of validate_batched without real_emg
    enc_only = ug.validate_batched(utts, max_batch=4)
    assert len(captures) == 2 * n_buckets                               # a graph of its own per bucket
    assert {i: sc.encoder for i, sc in scores.items()} == enc_only
    # a second call replays without recapturing; two ranks' shards are the union of one rank's dict
    again = ug.validate_batched(utts, max_batch=4, real_emg=real)
    assert len(captures) == 2 * n_buckets and again == scores
    shards = [ug.validate_batched(utts, rank=r, world=2, max_batch=4, real_emg=real) for r in range(2)]
    assert len(captures) == 2 * n_buckets
    assert sorted(list(shards[0]) + list(shards[1])) == list(range(len(utts)))
    assert {**shards[0], **shards[1]} == scores
    assert aggregate_td(sc.td for s in shards for sc in s.values()) == aggregate_td(sc.td for sc in scores.values())
    # refold() drops the graphs: the next call captures again
    ug.refold()
    assert not ug._graphs
    ug.validate_batched(utts[:1], max_batch=4, real_emg=real[:1])
    assert len(captures) == 2 * n_buckets + 1
    # an engine without an encoder: (units, session_id) items, the same time-domain values
    bare = UtteranceGenerator(gen, prec, max_graphs=32)
    td_only = bare.validate_batched([u[:2] for u in utts], max_batch=4, real_emg=real)
    assert all(td_only[i].encoder is None and td_only[i].td == scores[i].td for i in scores)


def test_validate_batched_mfcc_generator():
    from ste_gan_b200.inference import UtteranceGenerator
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    torch.manual_seed(0)
    gen = EMGGeneratorGanTTS("MFCCS", 25, 17, 8, channels=256).cuda()
    lens = [6, 7, 40, 99, 130]
    utts, real = _validation_set(lens, D=25, r=8, seed=3)
    ug = UtteranceGenerator(gen, "fp32")
    assert ug.rows_per_frame == 8
    scores = ug.validate_batched([u[:2] for u in utts], max_batch=4, real_emg=real)
    emg = ug.serve_batched([u[:2] for u in utts], max_batch=4)
    for i in range(len(lens)):
        assert emg[i].shape == (8 * lens[i], 8)
        for v, m in zip(scores[i].td.values, _module_td(real[i], emg[i])):
            assert _rel(v, m) <= TD_TOL["fp32"], (i, v, m)


# ---------------------------------------------------------------------------------------------
# speaking modes
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_speaking_mode_generator_in_batches(prec):
    from ste_gan_b200.inference import UtteranceGenerator
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    torch.manual_seed(0)
    gen = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8, use_speaking_mode_embedding=True, channels=256).cuda()
    lens = [3, 37, 40, 100, 113, 150]
    modes = [0, 1, 2, 1, 2, 0]
    utts, real = _validation_set(lens, seed=5)
    units = [u[:2] for u in utts]
    ug = UtteranceGenerator(gen, prec, max_graphs=32)
    out = ug.serve_batched(units, max_batch=4, speaking_mode_ids=modes)
    for i, (su, sid) in enumerate(units):
        alone = ug.generate_graph(su[None], sid.reshape(1), torch.tensor([modes[i]]))[0].cpu()
        assert out[i].shape == alone.shape == (16 * lens[i], 8)
        assert O.rel_l2(out[i], alone) <= SELF_TOL[prec], (i, modes[i])
    other = ug.serve_batched(units, max_batch=4, speaking_mode_ids=[(m + 1) % 3 for m in modes])
    assert all(not torch.equal(other[i], out[i]) for i in range(len(lens)))    # the ids reach the embedding
    scores = ug.validate_batched(units, max_batch=4, real_emg=real, speaking_mode_ids=modes)
    for i in range(len(lens)):
        for v, m in zip(scores[i].td.values, _module_td(real[i], out[i])):
            assert _rel(v, m) <= TD_TOL[prec], (i, v, m)
    enc = UtteranceGenerator(gen, prec, max_graphs=32, emg_encoder=_tiny_encoder())
    with_enc = enc.validate_batched(utts, max_batch=4, speaking_mode_ids=modes)
    assert sorted(with_enc) == list(range(len(lens))) and all(with_enc[i].num_phones == lens[i] for i in with_enc)
