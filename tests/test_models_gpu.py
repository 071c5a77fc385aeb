"""Model-level parity (GPU): drop-in modules and the fused train step against the CPU oracle
(oracle/ste_gan_oracle.py, pinned to the reference by tests/golden/*) and against the
committed golden fixtures.

Tolerances (BASELINE.json north_star): relative L2 <= 1e-4 in the fp32 validation mode,
<= 2e-2 in bf16.
"""
import os

import pytest
import torch

from oracle import ste_gan_oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
TOL = {"fp32": 1e-4, "bf16": 2e-2}


def seeded(ctor, seed=0):
    torch.manual_seed(seed)
    return ctor()


def cpu_sd(mod):
    return {k: v.detach().cpu().clone() for k, v in mod.state_dict().items()}


@pytest.fixture(scope="module")
def nets():
    from ste_gan_b200.models.discriminator import DiscriminatorSmall
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    g = seeded(lambda: EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8))
    d = seeded(lambda: DiscriminatorSmall(8))
    return g, d


def test_init_matches_reference_checksums(nets):
    """Seed-0 initialisation is bit-identical to the reference modules (fixture from oracle/make_golden.py)."""
    init = torch.load(os.path.join(GOLD, "init_checksums.pt"))
    for name, mod in (("generator", nets[0]), ("disc_small", nets[1])):
        sd = mod.state_dict()
        assert list(sd.keys()) == list(init[name].keys())
        for k, ref in init[name].items():
            t = sd[k].detach().double().flatten()
            assert list(sd[k].shape) == ref["shape"]
            assert abs(t.sum().item() - ref["sum"]) <= 1e-9 * max(1.0, ref["abssum"]), k
            assert torch.equal(t[ref["idx"]].float(), ref["samples"]), k


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_generator_tiny_golden(prec):
    """channels=64 generator with the reference's stored weights, input and output."""
    import ste_gan_b200
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    fx = torch.load(os.path.join(GOLD, "generator_tiny.pt"))
    g = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8, channels=fx["channels"])
    g.load_state_dict(fx["state_dict"])
    g.cuda()
    with ste_gan_b200.precision(prec):
        y = g.generate(fx["speech_units"].cuda(), fx["session_ids"].cuda(), torch.zeros(2, dtype=torch.long).cuda())
    assert y.shape == fx["output"].shape
    assert O.rel_l2(y, fx["output"]) < TOL[prec]


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_generator_full_vs_oracle(nets, prec):
    import ste_gan_b200
    g = nets[0].cuda()
    su, sess, _ = O.synthetic_batch(2, 100, seed=1)
    with torch.no_grad():
        ref = O.generator_forward(cpu_sd(g), su, sess)
    with ste_gan_b200.precision(prec):
        y = g.generate(su.cuda(), sess.cuda(), torch.zeros(2, dtype=torch.long).cuda())
    assert O.rel_l2(y, ref) < TOL[prec]
    if prec == "fp32":   # configs[0] golden: B=1 T=100 seed-0 weights
        fx = torch.load(os.path.join(GOLD, "train_step_b1.pt"))
        su1, sess1, _ = O.synthetic_batch(1, 100, seed=0)
        with ste_gan_b200.precision("fp32"):
            y1 = g.generate(su1.cuda(), sess1.cuda(), torch.zeros(1, dtype=torch.long).cuda())
        assert O.rel_l2(y1, fx["x_pred"]) < 1e-4


@pytest.mark.parametrize("small", [True, False], ids=["small", "full"])
def test_discriminator_golden_two_forwards(small):
    """Two consecutive training forwards (pins the per-forward spectral-norm power iteration)."""
    import ste_gan_b200
    from ste_gan_b200.models.discriminator import Discriminator, DiscriminatorSmall
    fx = torch.load(os.path.join(GOLD, "disc_small.pt" if small else "disc_full.pt"))
    d = seeded(lambda: (DiscriminatorSmall if small else Discriminator)(8)).cuda()
    assert d.discriminator_names == fx["names"]
    x = fx["x"].cuda()
    with ste_gan_b200.precision("fp32"):
        for p in range(2):
            with torch.no_grad():
                res = d(x)
            for fms, refs in zip(res, fx["passes"][p]):
                assert len(fms) == len(refs)
                for fm, ref in zip(fms, refs):
                    assert list(fm.shape) == ref["shape"]
                    t = fm.detach().double().cpu().contiguous().flatten()
                    assert abs(t.norm().item() - ref["l2"]) <= 1e-4 * max(ref["l2"], 1e-3)
                    assert (t[ref["idx"]].float() - ref["samples"]).norm() <= 2e-4 * max(ref["samples"].norm().item(), 1e-3)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_discriminator_vs_oracle(nets, prec):
    import ste_gan_b200
    d = seeded(lambda: type(nets[1])(8)).cuda()
    sd = cpu_sd(d)
    _, _, x = O.synthetic_batch(2, 100, seed=2)
    with torch.no_grad():
        ref = O.discriminator_forward(sd, x, small=True, training=True)
    with ste_gan_b200.precision(prec), torch.no_grad():
        res = d(x.cuda())
    worst = max(O.rel_l2(a, b) for fa, fb in zip(res, ref) for a, b in zip(fa, fb))
    assert worst < TOL[prec], worst
    # spectral-norm buffers advanced identically
    for k in ("multi_scale_disc.0.layers.3.weight_u", "multi_scale_disc.0.layers.0.weight_v"):
        assert O.rel_l2(d.state_dict()[k], sd[k]) < 1e-4


def test_td_loss_golden():
    from ste_gan_b200.losses.time_domain_loss import MultiTimeDomainFeatureLoss
    fx = torch.load(os.path.join(GOLD, "td_loss.pt"))
    mtd = MultiTimeDomainFeatureLoss(8)
    xg = fx["x_gen"].cuda().requires_grad_(True)
    loss, parts = mtd.time_domain_loss(fx["x_real"].cuda(), xg)
    for a, b in zip(parts, fx["parts"]):
        assert abs(float(a) - float(b)) <= 1e-5 * abs(float(b))
    assert abs(float(loss) - float(fx["loss"])) <= 1e-5 * abs(float(fx["loss"]))
    loss.backward()
    assert O.rel_l2(xg.grad, fx["grad_x_gen"]) < 1e-4
    # forward(x_real, x_generated) argument order (time_domain_loss.py:105-107)
    assert abs(float(mtd(fx["x_real"].cuda(), fx["x_gen"].cuda())) - float(fx["loss"])) <= 1e-5 * abs(float(fx["loss"]))


def _fresh_nets(small=True):
    from ste_gan_b200.models.discriminator import Discriminator, DiscriminatorSmall
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    g = seeded(lambda: EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8))
    d = seeded(lambda: (DiscriminatorSmall if small else Discriminator)(8))
    return g, d


def _flat_rel_l2(mine: dict, ref: dict) -> float:
    """relative L2 of the whole gradient of a network (the flat vector the optimiser / all-reduce consume)."""
    num = sum(float((mine[k].double() - ref[k].double()).pow(2).sum()) for k in ref)
    den = sum(float(ref[k].double().pow(2).sum()) for k in ref)
    return (num / den) ** 0.5


# LeakyReLU / ReLU have a discontinuous derivative: a pre-activation that is zero to within the arithmetic's
# rounding gets the other slope ("sign flip") and changes the gradient of everything upstream of it by a
# finite amount (tools/sn_probe.py, tools/grad_probe.py: ONE flipped element out of 4.1e5 moves a first-layer
# weight gradient by 1.7e-3 in fp32; in bf16 ~0.25 % of the elements flip).  Round 1 loosened the bound for
# tensors behind a flip; now the ORACLE is made flip-aware instead: its backward takes the sign pattern of every
# ReLU / LeakyReLU from the CUDA path's own saved activations (oracle._ActWithMask), so both differentiate the
# same piecewise-linear branch and EVERY gradient tensor is held to the north_star tolerance (1e-4 / 2e-2).
def disc_masks(fmaps, d):
    """sign patterns of a CUDA discriminator pass (channels-last feature maps) in the reference layout"""
    from ste_gan_b200 import passes
    out = []
    for (kind, sub), fm in zip(passes.disc_subnets(d), fmaps):
        out.append([passes.to_reference_layout(a.float().cpu(), kind, getattr(sub, "period", 1)) > 0 for a in fm[:-1]])
    return out


def gen_masks(gctx):
    """sign patterns of the generator's ReLU inputs from the saved (post-ReLU) activations of its forward"""
    cl = lambda t: t.float().cpu().transpose(1, 2) > 0
    out = []
    for s in gctx.blocks:
        xa = s["x_act"][:, ::2] if s["up"] > 1 else s["x_act"]       # rows are duplicated where the block upsamples
        out.append([cl(xa), cl(s["a1"]), cl(s["h_act"]), cl(s["a3"])])
    out.append(cl(gctx.y_last_act))
    return out


def run_step_vs_oracle(g, d, batch, prec, small=True, speaking_mode_ids=None, speech_feature_type="SPEECH_UNITS", encoder=None):
    """One fused train step against the flip-aware oracle: G output, every feature map of the three discriminator
    passes that carry gradients, every loss term, and the gradient of EVERY parameter tensor of G and D."""
    from ste_gan_b200 import passes
    from ste_gan_b200.trainer import GanTrainer
    sd_g, sd_d = cpu_sd(g), cpu_sd(d)
    su, sess, x_real = batch
    tol = TOL[prec]
    enc_arg = None
    if encoder is not None:                       # (frozen EMG encoder module in eval mode, phoneme targets [B, frames])
        enc_mod, ph = encoder
        enc_sd = {k: (v.detach().cpu().double() if v.is_floating_point() else v.detach().cpu().clone()) for k, v in enc_mod.state_dict().items()}
        enc_arg = dict(sd=enc_sd, phoneme_targets=ph, w_su=1.0, w_ph=1.0)
    tr = GanTrainer(g.cuda(), d.cuda(), precision=prec, emg_encoder=enc_mod.cuda() if encoder is not None else None)
    if encoder is not None:
        tr._cur_ph = ph.cuda()
    mode = speaking_mode_ids.cuda() if speaking_mode_ids is not None else None
    tr._phase_d(su.cuda(), sess.cuda(), mode, x_real.cuda())
    gd = {n: p.grad.detach().cpu().clone() for n, p in d.named_parameters()}
    fm_fake_det, fm_real = tr._last_d_fmaps[:2]
    tr._phase_g(x_real.cuda(), update_d=False)
    fm_fake = tr._last_g_fmaps[0]
    masks = dict(g=gen_masks(tr._last_gctx), d_fake_det=disc_masks(fm_fake_det, d), d_real=disc_masks(fm_real, d),
                 d_fake=disc_masks(fm_fake, d))
    if encoder is not None:                       # the encoder's ReLU sign patterns on THIS x_pred (a second forward of the frozen net)
        from ste_gan_b200 import passes_encoder as pe
        from tests.test_encoder_gpu import _enc_masks
        masks["encoder"] = _enc_masks(pe.encoder_forward(tr._enc_plan, tr.x_pred)[2])
    # the oracle is evaluated in float64: both the reference (fp32) and this library approximate the same function
    f64 = lambda sd: {k: v.double() for k, v in sd.items()}
    ref = O.losses_and_grads(f64(sd_g), f64(sd_d), su.double(), sess, x_real.double(), small=small, masks=masks,
                             speaking_mode_ids=speaking_mode_ids, speech_feature_type=speech_feature_type, encoder=enc_arg)
    assert O.rel_l2(tr.x_pred, ref["x_pred"]) < tol
    subs = passes.disc_subnets(d)
    n_flip = 0
    for mine, theirs in ((fm_fake_det, ref["d_fake_det"]), (fm_real, ref["d_real"]), (fm_fake, ref["d_fake"])):
        for di, (fm_m, fm_o) in enumerate(zip(mine, theirs)):
            kind, sub = subs[di]
            for j, (a, b) in enumerate(zip(fm_m, fm_o)):
                a = passes.to_reference_layout(a.float().cpu(), kind, getattr(sub, "period", 1))
                assert O.rel_l2(a, b) < tol, (di, j)
                if j + 1 < len(fm_m):
                    n_flip += int(((a > 0) != (b > 0)).sum())
    L = tr.losses()
    for k in ("loss_d", "loss_adv", "loss_fm", "loss_td", "loss_g"):
        assert abs(L[k] - float(ref[k])) <= tol * max(1.0, abs(float(ref[k]))), (k, L[k], float(ref[k]))
    gg = {n: p.grad.detach().cpu() for n, p in g.named_parameters()}
    flat_d, flat_g = _flat_rel_l2(gd, ref["grad_d"]), _flat_rel_l2(gg, ref["grad_g"])
    bad = {k: O.rel_l2(gd[k], ref["grad_d"][k]) for k in gd}
    bad_g = {k: O.rel_l2(gg[k], ref["grad_g"][k]) for k in gg}
    print(f"[{prec} B={su.shape[0]}] grad_d flat {flat_d:.3e} worst {max(bad.values()):.3e} ({max(bad, key=bad.get)}); "
          f"grad_g flat {flat_g:.3e} worst {max(bad_g.values()):.3e} ({max(bad_g, key=bad_g.get)}); "
          f"discriminator activations whose sign differs from the unmasked oracle forward: {n_flip}")
    assert flat_d < tol and flat_g < tol
    # EVERY parameter tensor at the north_star tolerance.  A 1-element parameter (weight_g / bias of the 1-channel logits
    # convs) has no relative L2 of its own - it is ONE number, a sum of signed terms that can cancel to any degree
    # (d weight_g = sum_t dlogit_t (logit_t - b) / g) - so it is held to the tolerance jointly with the other parameters
    # of its conv: the relative L2 of the conv's concatenated gradient [bias | weight_g | weight_v].
    for grads, refs in ((gd, ref["grad_d"]), (gg, ref["grad_g"])):
        for k in grads:
            if grads[k].numel() > 1:
                e = O.rel_l2(grads[k], refs[k])
            else:
                sib = [q for q in grads if q.rsplit(".", 1)[0] == k.rsplit(".", 1)[0]]
                e = _flat_rel_l2({q: grads[q] for q in sib}, {q: refs[q] for q in sib})
            assert e < tol, (k, e)
    return tr, ref


@pytest.mark.parametrize("batch", [2, 16], ids=["B2", "B16"])
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_train_step_losses_and_grads_vs_oracle(prec, batch):
    """One fused train step at T=100 - B=2 and the BENCHMARKED configuration B=16 (BASELINE.json configs[1]; the
    batched [fake | real] discriminator stacks then run 32 samples) - against the flip-aware oracle, every tensor held
    to 1e-4 (fp32) / 2e-2 (bf16)."""
    g, d = _fresh_nets()
    run_step_vs_oracle(g, d, O.synthetic_batch(batch, 100, seed=3), prec)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_speaking_mode_embedding_train_step(prec):
    """use_speaking_mode_embedding=True (generator.py:104-107,148-151): 256 + 64 + 64 = 384 input channels, two
    embedding tables, both with gradients."""
    from ste_gan_b200.models.discriminator import DiscriminatorSmall
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    g = seeded(lambda: EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8, use_speaking_mode_embedding=True, channels=256))
    d = seeded(lambda: DiscriminatorSmall(8))
    su, sess, x_real = O.synthetic_batch(3, 40, seed=12)
    mode = torch.tensor([2, 0, 1])
    tr, ref = run_step_vs_oracle(g, d, (su, sess, x_real), prec, speaking_mode_ids=mode)
    assert "speaking_mode_embeddings.weight" in ref["grad_g"]


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_mfcc_generator_variant(prec):
    """speech_feature_type = MFCCS (generator.py:116,178-179): 25-d input (+64 embedding = 89 channels, not a multiple
    of 8 - zero-padded rows on the tensor engine), no upsampling in GBlock 6 -> 8T output samples.  Forward vs the oracle
    and one fused train step (losses + flat gradients)."""
    import ste_gan_b200
    from ste_gan_b200.models.discriminator import DiscriminatorSmall
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    from ste_gan_b200.trainer import GanTrainer
    g = seeded(lambda: EMGGeneratorGanTTS("MFCCS", 25, 17, 8, channels=256))
    d = seeded(lambda: DiscriminatorSmall(8))
    su, sess, x_real = O.synthetic_batch(2, 100, seed=6, unit_dim=25, hop=8)
    assert x_real.shape[1] == 800
    tr, _ = run_step_vs_oracle(g, d, (su, sess, x_real), prec, speech_feature_type="MFCCS")
    assert tr.x_pred.shape == (2, 800, 8)


def test_full_discriminator_train_step_bf16():
    """The full CARGAN `Discriminator` (discriminator.py:158-191: k=41 stride-4 grouped scale stacks, (5,1)/(3,1)
    period stacks) through one fused train step in the tensor-core mode, against the oracle."""
    from ste_gan_b200.trainer import GanTrainer
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    g = seeded(lambda: EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8, channels=128))
    _, d = _fresh_nets(small=False)
    run_step_vs_oracle(g, d, O.synthetic_batch(2, 64, seed=8), "bf16", small=False)


def test_autograd_dropin_matches_fused_step():
    """The reference-style loop (modules + loss.backward()) gives the same gradients as the fused trainer (fp32)."""
    import torch.nn.functional as F
    import ste_gan_b200
    from ste_gan_b200.losses.time_domain_loss import MultiTimeDomainFeatureLoss
    from ste_gan_b200.trainer import GanTrainer
    su, sess, x_real = (t.cuda() for t in O.synthetic_batch(2, 100, seed=4))
    g1, d1 = _fresh_nets()
    tr = GanTrainer(g1.cuda(), d1.cuda(), precision="fp32")
    tr._phase_d(su, sess, None, x_real)
    gd_ref = {n: p.grad.detach().clone() for n, p in d1.named_parameters()}
    tr._phase_g(x_real, update_d=False)
    g2, d2 = _fresh_nets()
    g2.cuda(); d2.cuda()
    mtd = MultiTimeDomainFeatureLoss(8)
    with ste_gan_b200.precision("fp32"):
        x_pred = g2(su, sess, torch.zeros(2, dtype=torch.long).cuda())                 # train.py:182
        D_fake_det, D_real = d2(x_pred.detach()), d2(x_real)                          # :190-191
        loss_D = sum(F.mse_loss(s[-1], torch.zeros_like(s[-1])) for s in D_fake_det) + \
            sum(F.mse_loss(s[-1], torch.ones_like(s[-1])) for s in D_real)
        loss_D.backward()                                                              # :198
        for n, p in d2.named_parameters():
            assert O.rel_l2(p.grad, gd_ref[n]) < 1e-4, n
        d2.zero_grad()
        D_fake, D_real = d2(x_pred), d2(x_real)                                        # :206-207
        loss_G = sum(F.mse_loss(s[-1], torch.ones_like(s[-1])) for s in D_fake) + 15.0 * mtd(x_real, x_pred)
        for i in range(len(D_fake)):
            for j in range(len(D_fake[i]) - 1):
                loss_G = loss_G + 7.0 * F.l1_loss(D_fake[i][j], D_real[i][j].detach())  # :259-263
        loss_G.backward()                                                              # :266
    assert abs(float(loss_G) - tr.losses()["loss_g"]) <= 1e-4 * abs(float(loss_G))
    for (n, p), (_, q) in zip(g2.named_parameters(), g1.named_parameters()):
        assert O.rel_l2(p.grad, q.grad) < 1e-4, n


def test_multi_step_matches_oracle_trainer():
    """Three full steps (D update between the phases, AdamW on both nets) track the oracle's loss trajectory."""
    from ste_gan_b200.trainer import GanTrainer
    g, d = _fresh_nets()
    ot = O.OracleTrainer(cpu_sd(g), cpu_sd(d), small=True)
    tr = GanTrainer(g.cuda(), d.cuda(), precision="fp32")
    for step in range(3):
        su, sess, x_real = O.synthetic_batch(2, 100, seed=10 + step)
        ref = ot.step(su, sess, x_real)
        tr.step(su.cuda(), sess.cuda(), x_real.cuda())
        L = tr.losses()
        for k in ("loss_d", "loss_g", "loss_fm", "loss_td"):
            assert abs(L[k] - ref[k]) <= 2e-3 * max(1.0, abs(ref[k])), (step, k, L[k], ref[k])
    # parameters after 3 optimiser steps
    worst = max(O.rel_l2(p, ot.g[n]) for n, p in g.named_parameters())
    assert worst < 1e-3, worst


def test_cuda_graph_step_matches_eager():
    from ste_gan_b200.trainer import GanTrainer
    su, sess, x_real = (t.cuda() for t in O.synthetic_batch(2, 100, seed=5))
    g1, d1 = _fresh_nets(); g2, d2 = _fresh_nets()
    t1 = GanTrainer(g1.cuda(), d1.cuda(), precision="bf16")
    t2 = GanTrainer(g2.cuda(), d2.cuda(), precision="bf16")
    t2.capture(2, 100)               # (its warm-up steps leave no trace in the training state: see the test below)
    for _ in range(2):
        t1.step(su, sess, x_real)
        t2.step_graph(su, sess, x_real)
    a, b = t1.losses(), t2.losses()
    for k in a:
        assert abs(a[k] - b[k]) <= 2e-2 * max(1.0, abs(a[k])), (k, a[k], b[k])
    # the replay defers the last generator optimiser step: flush(), then the parameters agree as well
    assert t2._fused is not None and t2._pending_host      # the default capture: ONE graph per step, generator update pending
    t2.flush()
    # Tolerance: the weight-gradient reductions (TMA reduce-add, atomics) are order-nondeterministic, and AdamW's first
    # steps turn noise-level gradients into +-lr updates, so two runs of the SAME schedule differ by ~1e-3 here; a lost
    # optimiser step would be ~7e-3 (lr / |w|).
    assert O.rel_l2(t2.G.flat, t1.G.flat) < 3e-3 and O.rel_l2(t2.D.flat, t1.D.flat) < 3e-3


def test_cuda_graph_step_three_buckets_matches_eager():
    """The three-bucket generator backward under capture - AdamW per bucket on the communication stream (keep_step for
    all but the first), the last bucket deferred behind the device flag - against the eager one-bucket step."""
    from ste_gan_b200.trainer import GanTrainer
    su, sess, x_real = (t.cuda() for t in O.synthetic_batch(2, 100, seed=7))
    g1, d1 = _fresh_nets(); g2, d2 = _fresh_nets()
    t1 = GanTrainer(g1.cuda(), d1.cuda(), precision="bf16")                    # one gradient bucket (no data-parallel group)
    t2 = GanTrainer(g2.cuda(), d2.cuda(), precision="bf16", grad_buckets=3)    # the three-bucket generator backward
    assert len(t1.g_buckets) == 1 and len(t2.g_buckets) == 3
    t2.capture(2, 100)
    for _ in range(3):
        t1.step(su, sess, x_real)
        t2.step_graph(su, sess, x_real)
    t2.flush()
    a, b = t1.losses(), t2.losses()
    for k in a:
        assert abs(a[k] - b[k]) <= 2e-2 * max(1.0, abs(a[k])), (k, a[k], b[k])
    assert O.rel_l2(t2.G.flat, t1.G.flat) < 3e-3 and O.rel_l2(t2.D.flat, t1.D.flat) < 3e-3      # (see above)


def _state_of(tr):
    return [t.clone() for fp in (tr.G, tr.D) for t in (fp.flat, fp.m, fp.v, fp.step)] + [b.clone() for b in tr._sn_buffers()]


def test_capture_preserves_training_state():
    """capture() warms up with two real steps on zero inputs; parameters, AdamW moments, step counters and the
    spectral-norm u / v must come out of it bit-identical (resume-then-capture is safe; ADVICE r1)."""
    from ste_gan_b200.trainer import GanTrainer
    batch = [t.cuda() for t in O.synthetic_batch(2, 64, seed=31)]
    g, d = _fresh_nets()
    tr = GanTrainer(g.cuda(), d.cuda(), precision="bf16")
    tr.step(*batch)
    before = _state_of(tr)
    tr.capture(2, 64)
    torch.cuda.synchronize()
    for a, b in zip(before, _state_of(tr)):
        assert torch.equal(a, b)
    assert int(tr.G.step) == 1 and int(tr.D.step) == 1


def test_learning_rate_is_read_on_the_device_under_graphs():
    """`trainer.lr = x` after capture() reaches the AdamW kernels inside the replayed graphs (ExponentialLR per epoch,
    train.py:470-472; lr restored by load_latest_checkpoint).  lr = 0 with weight decay off the table (decay = 1 - lr*wd)
    must freeze both networks exactly; restoring it must move them again."""
    from ste_gan_b200.trainer import GanTrainer
    batch = [t.cuda() for t in O.synthetic_batch(2, 64, seed=32)]
    g, d = _fresh_nets()
    tr = GanTrainer(g.cuda(), d.cuda(), precision="bf16")
    tr.capture(2, 64)
    tr.step_graph(*batch); tr.flush()
    tr.lr = 0.0
    g0, d0 = tr.G.flat.clone(), tr.D.flat.clone()
    tr.step_graph(*batch); tr.flush()
    assert torch.equal(tr.G.flat, g0) and torch.equal(tr.D.flat, d0)
    assert tr.scheduler_step(0.5) == 0.0
    tr.lr = 2e-4
    assert abs(tr.scheduler_step(0.999) - 2e-4 * 0.999) < 1e-12 and abs(float(tr.lr_dev) - 2e-4 * 0.999) < 1e-10
    tr.step_graph(*batch); tr.flush()
    assert not torch.equal(tr.G.flat, g0) and not torch.equal(tr.D.flat, d0)


def test_adamw_graph_replay_follows_exponential_lr():
    """The fused AdamW kernel with a device-resident lr, captured ONCE and replayed over two 'epochs' of three steps,
    against torch.optim.AdamW + ExponentialLR(gamma) (train.py:80-81,98-104,470-472; constants.py:57)."""
    from ste_gan_b200 import ops
    gen = torch.Generator().manual_seed(9)
    n, gamma = 4096, 0.9
    p0 = torch.randn(n, generator=gen)
    grads = [torch.randn(n, generator=gen) for _ in range(6)]
    ref_p = torch.nn.Parameter(p0.clone())
    opt = torch.optim.AdamW([ref_p], lr=2e-4, betas=(0.8, 0.99))
    sched = torch.optim.lr_scheduler.ExponentialLR(opt, gamma=gamma)
    p, g = p0.clone().cuda(), torch.zeros(n).cuda()
    m, v = torch.zeros(n).cuda(), torch.zeros(n).cuda()
    step = torch.zeros(1, dtype=torch.int64).cuda()
    lr = torch.full((1,), 2e-4).cuda()
    side = torch.cuda.Stream(); side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.adamw(p, g, m, v, step, lr)           # warm-up launch, undone below
    torch.cuda.current_stream().wait_stream(side); torch.cuda.synchronize()
    p.copy_(p0); m.zero_(); v.zero_(); step.zero_()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ops.adamw(p, g, m, v, step, lr)
    for epoch in range(2):
        for i in range(3):
            g.copy_(grads[3 * epoch + i]); graph.replay()
            ref_p.grad = grads[3 * epoch + i].clone(); opt.step()
        sched.step()
        lr.fill_(sched.get_last_lr()[0])
    assert int(step) == 6 and O.rel_l2(p, ref_p) < 1e-6


def test_checkpoint_resume_into_captured_graphs(tmp_path):
    """capture -> load_latest_checkpoint -> step_graph runs on the LOADED weights (the discriminator packs are re-packed
    eagerly by the load: a captured phase-D graph would otherwise reuse the packs of the pre-load weights; ADVICE r1)."""
    from ste_gan_b200.trainer import GanTrainer
    batch = [t.cuda() for t in O.synthetic_batch(2, 64, seed=33)]
    g1, d1 = _fresh_nets(); g2, d2 = _fresh_nets(); g3, d3 = _fresh_nets()
    t1 = GanTrainer(g1.cuda(), d1.cuda(), precision="bf16")
    for _ in range(3):
        t1.step(*batch)
    t1.lr = 1.5e-4
    t1.save_checkpoint(tmp_path, steps=3, epoch=1)
    t2 = GanTrainer(g2.cuda(), d2.cuda(), precision="bf16")      # graphs captured BEFORE the load
    t2.capture(2, 64)
    assert t2.load_latest_checkpoint(tmp_path) == (1, 3) and t2.lr == 1.5e-4
    t3 = GanTrainer(g3.cuda(), d3.cuda(), precision="bf16")      # eager reference from the same checkpoint
    t3.load_latest_checkpoint(tmp_path)
    t2.step_graph(*batch); t2.flush()
    t3.step(*batch)
    a, b = t2.losses(), t3.losses()
    for k in a:
        assert abs(a[k] - b[k]) <= 2e-2 * max(1.0, abs(a[k])), (k, a[k], b[k])
    assert O.rel_l2(t2.G.flat, t3.G.flat) < 3e-3 and O.rel_l2(t2.D.flat, t3.D.flat) < 3e-3
    assert int(t2.G.step) == 4 and int(t2.D.step) == 4


def test_no_cpu_fallback():
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    g = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8, channels=64)
    su, sess, _ = O.synthetic_batch(1, 8)
    with pytest.raises(RuntimeError):
        g(su, sess, torch.zeros(1, dtype=torch.long))


def test_checkpoint_round_trip_through_reference_format(tmp_path):
    """save_checkpoint writes the reference's netG- / netD- / checkpoint-{steps:08d}.pt triple (train.py:421-436) with the
    optimiser state as torch.optim.AdamW state_dicts; a fresh trainer resumes from it (utils/common.py:23-61) with
    identical parameters, moments and step counters, and the next step gives the same losses."""
    from ste_gan_b200.trainer import GanTrainer
    batch = [t.cuda() for t in O.synthetic_batch(2, 64, seed=21)]
    g1, d1 = _fresh_nets(); g2, d2 = _fresh_nets()
    t1 = GanTrainer(g1.cuda(), d1.cuda(), precision="fp32")
    for _ in range(2):
        t1.step(*batch)
    t1.save_checkpoint(tmp_path, steps=2, epoch=1)
    assert sorted(f.name for f in tmp_path.iterdir()) == ["checkpoint-00000002.pt", "netD-00000002.pt", "netG-00000002.pt"]
    ck = torch.load(tmp_path / "checkpoint-00000002.pt")
    assert set(ck) == {"epoch", "steps", "optG", "optD"} and float(ck["optG"]["state"][0]["step"]) == 2.0
    # the reference's own optimiser class loads it
    ref_opt = torch.optim.AdamW([torch.nn.Parameter(torch.zeros(p.shape)) for p in g1.parameters()], lr=1.0)
    ref_opt.load_state_dict(ck["optG"])
    t2 = GanTrainer(g2.cuda(), d2.cuda(), precision="fp32")
    t2.step(*[torch.zeros_like(b) for b in batch])            # (state that the load must overwrite)
    assert t2.load_latest_checkpoint(tmp_path) == (1, 2)
    for a, b in ((t1.G, t2.G), (t1.D, t2.D)):
        assert torch.equal(a.flat, b.flat) and torch.equal(a.m, b.m) and torch.equal(a.v, b.v) and int(a.step) == int(b.step)
    for k, v in d1.state_dict().items():                      # buffers too (spectral-norm u / v)
        assert torch.equal(v, d2.state_dict()[k]), k
    t1.step(*batch); t2.step(*batch)
    a, b = t1.losses(), t2.losses()
    for k in a:
        assert abs(a[k] - b[k]) <= 1e-4 * max(1.0, abs(a[k])), (k, a[k], b[k])


@pytest.mark.parametrize("batch", [1, 4], ids=["B1", "B4"])
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_generate_30s_utterance_vs_oracle(nets, prec, batch):
    """BASELINE.json configs[3], the BENCHMARKED inference shape: 1500 unit frames -> 24000 x 8 EMG samples (row classes,
    tile counts and the column-tile choice all change with T), batch 1 and the batch-4 throughput mode; the module
    path (`generate`) and - in bf16 - the serving engine's CUDA-graph replay that bench.py times."""
    import ste_gan_b200
    from ste_gan_b200.inference import UtteranceGenerator
    g = nets[0].cuda()
    su, sess, _ = O.synthetic_batch(batch, 1500, seed=30 + batch)
    with torch.no_grad():
        ref = O.generator_forward(cpu_sd(g), su, sess)
    assert ref.shape == (batch, 24000, 8)
    with ste_gan_b200.precision(prec):
        y = g.generate(su.cuda(), sess.cuda(), torch.zeros(batch, dtype=torch.long).cuda())
    assert y.shape == ref.shape and O.rel_l2(y, ref) < TOL[prec]
    worst = max(O.rel_l2(y[b], ref[b]) for b in range(batch))          # per utterance, not only in aggregate
    assert worst < TOL[prec], worst
    ug = UtteranceGenerator(g, prec)
    for _ in range(2):                                                   # capture, then a replay
        y2 = ug.generate_graph(su.pin_memory(), sess.pin_memory())
    assert O.rel_l2(y2, ref) < TOL[prec]


def test_generate_from_data_dict(nets):
    """EMGGenerator.generate_from_data_dict (generator.py:52-75): a dataset item (2-D units, scalar ids) -> [16T, C] on the
    CPU; a batched item keeps its batch dimension."""
    import ste_gan_b200
    from ste_gan_b200.constants import DataType
    g = nets[0].cuda()
    su, sess, _ = O.synthetic_batch(1, 37, seed=41)
    item = {DataType.SPEECH_UNITS: su[0], DataType.SESSION_INDEX: sess[0], DataType.SPEAKING_MODE_INDEX: torch.tensor(0)}
    with torch.no_grad():
        ref = O.generator_forward(cpu_sd(g), su, sess)
    with ste_gan_b200.precision("fp32"):
        y = g.generate_from_data_dict(item, torch.device("cuda"))
    assert y.device.type == "cpu" and y.shape == (37 * 16, 8)
    assert O.rel_l2(y, ref[0]) < 1e-4
    batched = {DataType.SPEECH_UNITS: su, DataType.SESSION_INDEX: sess, DataType.SPEAKING_MODE_INDEX: torch.zeros(1, dtype=torch.long)}
    with ste_gan_b200.precision("fp32"):
        yb = g.generate_from_data_dict(batched, torch.device("cuda"))
    assert yb.shape == (37 * 16, 8) and O.rel_l2(yb, ref[0]) < 1e-4     # squeeze(0) of a batch of one (generator.py:75)


@pytest.mark.parametrize("window,pad", [(9, True), (5, True), (9, False)])
def test_average_filter_module(window, pad):
    """AverageFilter (layers/average_filter.py:10-28): reflect pad window//2 + AvgPool1d(window, stride 1)."""
    import torch.nn.functional as F
    from ste_gan_b200.layers.average_filter import AverageFilter
    x = torch.randn(3, 8, 203, generator=torch.Generator().manual_seed(5))
    af = AverageFilter(8, window, pad_signal=pad)
    y = af(x.cuda())
    ref = O.average_filter(x, window) if pad else F.avg_pool1d(x, kernel_size=window, stride=1)
    assert y.shape == ref.shape and O.rel_l2(y, ref) < 1e-6
    with pytest.raises(RuntimeError):
        af(x)                                                            # no CPU path


def test_data_parallel_matches_single_process():
    """N ranks through the bucketed graph step == one process on the global batch (tools/dp_check.py under
    torchrun, 2 GPUs, fp32).  Skipped on single-GPU boxes; the log of the last multi-GPU run is kept under profiles/."""
    import subprocess, sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(29600 + os.getpid() % 300), os.path.join(root, "tools", "dp_check.py")],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0 and "dp_check ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.parametrize("win,shift,pad,aw", [(21, 8, True, 9), (30, 10, False, 9), (16, 4, True, 5)])
def test_time_domain_feature_loss_any_setting(win, shift, pad, aw):
    """TimeDomainFeatureLoss with constructor settings OTHER than the three of the multi-resolution loss (the class
    default is (21, 8), time_domain_loss.py:20-33) and every helper method of the reference class
    (time_domain_loss.py:35-68), against the oracle."""
    from ste_gan_b200.losses.time_domain_loss import TimeDomainFeatureLoss
    gen = torch.Generator().manual_seed(win)
    xr, xg = torch.tanh(torch.randn(3, 400, 8, generator=gen)), torch.tanh(torch.randn(3, 400, 8, generator=gen))
    td = TimeDomainFeatureLoss(8, win, shift, apply_padding_windowing=pad, average_filter_window_size=aw)
    xg_c = xg.cuda().requires_grad_(True)
    loss = td.time_domain_loss(xr.cuda(), xg_c)
    (3.0 * loss).backward()
    xg_o = xg.double().requires_grad_(True)
    ref = O.td_loss(xr.double(), xg_o, win, shift, pad, aw)
    (3.0 * ref).backward()
    assert abs(float(loss) - float(ref)) <= 1e-5 * abs(float(ref))
    assert O.rel_l2(xg_c.grad, xg_o.grad) < 1e-4
    feats = td.calculate_time_domain_features(xg.cuda())
    ref_f = O.td_features(xg.double(), win, shift, pad, aw)
    assert feats.shape == ref_f.shape and O.rel_l2(feats, ref_f) < 1e-5
    ws = O.window_signal(xg, win, shift, pad)
    assert torch.equal(td.window_signal(xg.cuda()).cpu(), ws)                   # a gather: bit-exact
    assert O.rel_l2(td.frame_means(xg.cuda()), ws.double().mean(-1)) < 1e-6
    assert O.rel_l2(td.frame_power(xg.cuda()), (ws.double() ** 2).sum(-1)) < 1e-6
    low = O.average_filter(O.average_filter(xg.double().transpose(1, 2), aw), aw).transpose(1, 2)
    assert O.rel_l2(td.double_average(xg.cuda()), low) < 1e-6


def test_disc_losses_step_matches_reference_port():
    """GanTrainer.disc_losses_step (BASELINE.json configs[4]: D stacks + TD + FM + LSGAN isolated, fwd + bwd incl. the D AdamW
    step) against the same sequence on the CPU (baseline/ref_runner.PortTrainer = the oracle's functions): the gradient w.r.t.
    the fake batch that phase G hands to the generator, small and full discriminator, fp32."""
    from baseline import ref_runner as R
    from ste_gan_b200.trainer import GanTrainer
    for small in (True, False):
        g, d = _fresh_nets(small=small)
        gen = torch.Generator().manual_seed(40)
        x_pred = torch.tanh(torch.randn(2, 1024, 8, generator=gen))
        _, _, x_real = O.synthetic_batch(2, 64, seed=41)
        ref = R.PortTrainer("cpu", small=small)
        dx_ref = ref.disc_losses_step(x_pred, x_real)
        tr = GanTrainer(g.cuda(), d.cuda(), precision="fp32")
        dx = tr.disc_losses_step(x_pred.cuda(), x_real.cuda())
        # (the D AdamW step between the phases turns noise-level gradient elements into +-lr updates: 1e-3, not 1e-4)
        assert O.rel_l2(dx, dx_ref) < 1e-3, (small, O.rel_l2(dx, dx_ref))
        assert int(tr.D.step) == 1 and int(tr.G.step) == 0


def test_utterance_generator_graph_cache_and_speaking_mode():
    """The serving engine: LRU-bounded per-shape graph cache, speaking-mode ids through the captured graph, flush of a
    trainer's pending generator update before the weights are packed (ADVICE r1)."""
    import ste_gan_b200
    from ste_gan_b200.inference import UtteranceGenerator
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    g = seeded(lambda: EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8, use_speaking_mode_embedding=True, channels=64)).cuda()
    ug = UtteranceGenerator(g, "fp32", max_graphs=2)
    outs = {}
    for T in (20, 24, 28, 20):
        su, sess, _ = O.synthetic_batch(1, T, seed=T)
        mode = torch.tensor([T % 3])
        y = ug.generate_graph(su.cuda(), sess.cuda(), mode.cuda()).clone()
        with torch.no_grad():
            ref = O.generator_forward(cpu_sd(g), su, sess, mode)
        assert O.rel_l2(y, ref) < 1e-4, T
        outs[T] = y
    assert len(ug._graphs) == 2 and (1, 20) in ug._graphs and (1, 28) in ug._graphs      # (1, 24) was the least recently used
    with pytest.raises(ValueError):
        ug.generate_graph(*[t.cuda() for t in O.synthetic_batch(1, 20, seed=1)[:2]])     # speaking-mode ids are required
