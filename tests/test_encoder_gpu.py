"""EMG-encoder perceptual losses (SURVEY.md 8f rank 1) on the GPU against the CPU oracle (oracle/emg_encoder_oracle.py, pinned
to the reference by tests/golden/emg_encoder_tiny.pt) and against that fixture itself.

Tolerances as everywhere: relative L2 <= 1e-4 in the fp32 validation mode, <= 2e-2 in bf16.
"""
import os

import pytest
import torch
import torch.nn.functional as F

from oracle import emg_encoder_oracle as E
from oracle import ste_gan_oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
TOL = {"fp32": 1e-4, "bf16": 2e-2}
DT = {"fp32": torch.float32, "bf16": torch.bfloat16}


def _tiny_encoder():
    from ste_gan_b200.models.emg_encoder import EMGEncoderTransformer
    fx = torch.load(os.path.join(GOLD, "emg_encoder_tiny.pt"))
    for i, case in enumerate(fx["cases"]):
        case["x"], case["unit_target"], case["phoneme_target"] = E.tiny_case_inputs(i)
    enc = EMGEncoderTransformer(8, 256, 48, **E.TINY_ENCODER)
    sd = {k: (v.float() if v.is_floating_point() else v) for k, v in E.tiny_encoder_state(EMGEncoderTransformer).items()}
    enc.load_state_dict(sd)
    return enc.eval(), sd, fx


def test_encoder_init_matches_reference_checksums():
    """Seed-0 initialisation of the drop-in EMGEncoderTransformer is bit-identical to the reference's, key order included
    (fixture from oracle/make_golden.py)."""
    from ste_gan_b200.models.emg_encoder import EMGEncoderTransformer
    init = torch.load(os.path.join(GOLD, "emg_encoder_init.pt"))
    torch.manual_seed(0)
    sd = EMGEncoderTransformer(8, 256, 48, model_size=32, num_extra_res_blocks=3, num_transformer_layers=2).state_dict()
    assert list(sd.keys()) == list(init.keys())
    for k, ref in init.items():
        t = sd[k].detach().double().flatten()
        assert abs(t.sum().item() - ref["sum"]) <= 1e-9 * max(1.0, ref["abssum"]), k
        assert torch.equal(t[ref["idx"]].float(), ref["samples"]), k


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_layernorm_kernels(prec):
    from ste_gan_b200 import ops
    gen = torch.Generator().manual_seed(1)
    x = torch.randn(3, 50, 768, generator=gen) * 2 + 0.5
    g, b = torch.rand(768, generator=gen) + 0.5, torch.randn(768, generator=gen)
    dy = torch.randn(3, 50, 768, generator=gen)
    q = (lambda t: t.to(torch.bfloat16).float()) if prec == "bf16" else (lambda t: t)
    x, dy = q(x), q(dy)
    xr = x.double().requires_grad_(True)
    yr = F.layer_norm(xr, (768,), g.double(), b.double(), 1e-5)
    (dxr,) = torch.autograd.grad(yr, xr, dy.double())
    y, st = ops.layernorm(x.cuda().to(DT[prec]), g.cuda(), b.cuda())
    dx = ops.layernorm_bwd(dy.cuda().to(DT[prec]), x.cuda().to(DT[prec]), st, g.cuda())
    tol = 1e-5 if prec == "fp32" else 4e-3        # (bf16: output rounding only - the arithmetic is fp32)
    assert O.rel_l2(y, yr) < tol and O.rel_l2(dx, dxr) < tol


@pytest.mark.parametrize("geom", [(2, 25, 8, 4), (1, 111, 8, 4), (2, 100, 8, 96), (1, 128, 8, 96)], ids=["L25", "L111", "L100_d96", "L128_d96"])
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_relative_attention_kernels(prec, geom):
    """softmax(q.k/sqrt(d) + relative positional logits) v and its input gradient; L = 111 / 128 exceed the 100 relative positions
    (logits beyond the table get -1e8, transformer.py:262-268)."""
    from ste_gan_b200 import ops
    B, L, H, d = geom
    gen = torch.Generator().manual_seed(L + d)
    qkv = torch.randn(B, L, 3 * H * d, generator=gen)
    emb = torch.randn(H, 199, d, generator=gen) * d ** -0.5
    do = torch.randn(B, L, H * d, generator=gen)
    if prec == "bf16":
        qkv, do = qkv.to(torch.bfloat16).float(), do.to(torch.bfloat16).float()
    qr = qkv.double().requires_grad_(True)
    q, k, v = (t.view(B, L, H, d).permute(0, 2, 1, 3) for t in qr.split(H * d, dim=-1))
    logits = torch.einsum("bhqa,bhka->bhqk", q, k) / d ** 0.5 + E.relative_logits(q, emb.double())
    probs = torch.softmax(logits, -1)
    o_ref = torch.einsum("bhqk,bhka->bhqa", probs, v).permute(0, 2, 1, 3).reshape(B, L, H * d)
    (dq_ref,) = torch.autograd.grad(o_ref, qr, do.double())
    o, p = ops.relattn_fwd(qkv.cuda().to(DT[prec]), emb.cuda(), H, 100)
    dqkv = ops.relattn_bwd(qkv.cuda().to(DT[prec]), emb.cuda(), p, do.cuda().to(DT[prec]), H, 100)
    tol = 2e-5 if prec == "fp32" else 6e-3
    assert O.rel_l2(p, probs) < tol and O.rel_l2(o, o_ref) < tol and O.rel_l2(dqkv, dq_ref) < tol


def test_encoder_loss_kernel():
    from ste_gan_b200 import ops
    gen = torch.Generator().manual_seed(3)
    up, ut = torch.randn(4, 25, 256, generator=gen), torch.randn(4, 25, 256, generator=gen)
    lg, ph = torch.randn(4, 25, 48, generator=gen) * 3, torch.randint(0, 48, (4, 25), generator=gen)
    upr, lgr = up.double().requires_grad_(True), lg.double().requires_grad_(True)
    su, ce = E.encoder_losses(upr, lgr, ut.double(), ph)
    gu, gl = torch.autograd.grad(0.7 * su + 1.3 * ce, [upr, lgr])
    slots = torch.zeros(2, device="cuda")
    du, dl = ops.encoder_losses(up.cuda(), ut.cuda(), lg.cuda(), ph.cuda(), slots, 0.7, 1.3, torch.float32)
    assert abs(float(slots[0]) - float(su)) < 1e-5 * float(su) and abs(float(slots[1]) - float(ce)) < 1e-5 * float(ce)
    assert O.rel_l2(du, gu) < 1e-5 and O.rel_l2(dl, gl) < 1e-5


def _enc_masks(ctx):
    cl = lambda t: t.float().cpu().transpose(1, 2) > 0
    return dict(blocks=[(cl(s["h"]), cl(s["y"])) for s in ctx.blocks], layers=[s["hff"].float().cpu() > 0 for s in ctx.layers])


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_encoder_tiny_golden(prec):
    """The reference's own outputs (fixture): both heads, both losses and the gradient of their sum w.r.t. the EMG input, for a
    25-frame batch of two and a 111-frame utterance (> 100 relative positions)."""
    import ste_gan_b200
    from ste_gan_b200.losses.emg_encoder_loss import EMGEncoderLoss
    enc, sd, fx = _tiny_encoder()
    loss_mod = EMGEncoderLoss(enc.cuda())
    tol = TOL[prec]
    for case in fx["cases"]:
        x = case["x"].cuda().requires_grad_(True)
        with ste_gan_b200.precision(prec):
            out = loss_mod(x, case["unit_target"].cuda(), case["phoneme_target"].cuda())
            (out.speech_unit_loss + out.phoneme_loss).backward()
        assert O.rel_l2(out.speech_unit_pred, case["units"]) < tol and O.rel_l2(out.phoneme_pred, case["phonemes"]) < tol
        assert abs(float(out.speech_unit_loss) - float(case["unit_loss"])) <= tol * float(case["unit_loss"])
        assert abs(float(out.phoneme_loss) - float(case["phoneme_loss"])) <= tol * float(case["phoneme_loss"])
        if prec == "fp32":
            assert O.rel_l2(x.grad, case["dx"]) < tol
        assert out.num_phones == case["phoneme_target"].numel()
        assert out.num_correct_phones == int((case["phonemes"].argmax(-1) == case["phoneme_target"]).sum()) or prec == "bf16"
    # bf16: the input gradient against the flip-aware oracle (the ReLU sign patterns of THIS forward, see test_models_gpu.py)
    from ste_gan_b200 import passes_encoder as pe
    case = fx["cases"][0]
    plan = enc.plan(DT[prec])
    slots = torch.zeros(2, device="cuda")
    dx, units, logits = pe.encoder_losses(plan, case["x"].cuda(), case["unit_target"].cuda(), case["phoneme_target"].cuda(), slots)
    _, _, ctx = pe.encoder_forward(plan, case["x"].cuda())
    xr = case["x"].double().requires_grad_(True)
    f64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    u, l_ = E.emg_encoder_forward(f64, xr, _enc_masks(ctx))
    su, ce = E.encoder_losses(u, l_, case["unit_target"].double(), case["phoneme_target"])
    (dx_ref,) = torch.autograd.grad(su + ce, xr)
    assert O.rel_l2(dx, dx_ref) < tol


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_encoder_full_size_vs_oracle(prec):
    """The configuration of the train step (configs/emg_encoder/conv_transformer.yaml: 768-d, 4 ResBlocks, 6 layers, 8 heads of 96)
    with random-init weights (no checkpoint ships with the reference) and non-trivial BatchNorm statistics, B = 2, 1600 EMG samples
    -> 100 frames: heads, losses, input gradient."""
    from ste_gan_b200 import passes_encoder as pe
    from ste_gan_b200.models.emg_encoder import EMGEncoderTransformer
    torch.manual_seed(0)
    enc = EMGEncoderTransformer(8, 256, 48).eval()
    g = torch.Generator().manual_seed(5)
    for mod in enc.modules():
        if isinstance(mod, torch.nn.BatchNorm1d):
            mod.running_mean.normal_(0, 0.3, generator=g); mod.running_var.uniform_(0.5, 1.5, generator=g)
            mod.weight.data.uniform_(0.5, 1.5, generator=g); mod.bias.data.normal_(0, 0.2, generator=g)
    sd = {k: v.detach().clone() for k, v in enc.state_dict().items()}
    x = torch.tanh(torch.randn(2, 1600, 8, generator=g))
    ut, ph = torch.randn(2, 100, 256, generator=g), torch.randint(0, 48, (2, 100), generator=g)
    plan = enc.cuda().plan(DT[prec])
    slots = torch.zeros(2, device="cuda")
    dx, units, logits = pe.encoder_losses(plan, x.cuda(), ut.cuda(), ph.cuda(), slots, 1.0, 1.0)
    _, _, ctx = pe.encoder_forward(plan, x.cuda())
    xr = x.double().requires_grad_(True)
    f64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    u, l_ = E.emg_encoder_forward(f64, xr, _enc_masks(ctx))
    su, ce = E.encoder_losses(u, l_, ut.double(), ph)
    (dx_ref,) = torch.autograd.grad(su + ce, xr)
    tol = TOL[prec]
    assert O.rel_l2(units, u) < tol and O.rel_l2(logits, l_) < tol
    assert abs(float(slots[0]) - float(su)) <= tol * float(su) and abs(float(slots[1]) - float(ce)) <= tol * float(ce)
    assert O.rel_l2(dx, dx_ref) < tol
    with pytest.raises(RuntimeError):
        enc.train()(x.cuda())                      # only the frozen eval-mode encoder is on this path


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_train_step_with_encoder_losses(prec):
    """The generator step WITH the two perceptual losses (train.py:219-230) through GanTrainer, against the oracle: loss values
    and the gradient of every generator parameter (the discriminator gradients do not depend on them)."""
    from tests.test_models_gpu import _fresh_nets, run_step_vs_oracle
    from ste_gan_b200.models.emg_encoder import EMGEncoderTransformer
    torch.manual_seed(0)
    enc = EMGEncoderTransformer(8, 256, 48, model_size=128, num_extra_res_blocks=3, num_transformer_layers=2).eval()
    g, d = _fresh_nets()
    su, sess, x_real = O.synthetic_batch(2, 100, seed=13)
    ph = torch.randint(0, 48, (2, 100), generator=torch.Generator().manual_seed(14))
    tr, ref = run_step_vs_oracle(g, d, (su, sess, x_real), prec, encoder=(enc, ph))
    L = tr.losses()
    tol = TOL[prec]
    for k in ("loss_speech_unit", "loss_phoneme"):
        assert abs(L[k] - float(ref[k])) <= tol * max(1.0, abs(float(ref[k]))), (k, L[k], float(ref[k]))


def test_encoder_losses_in_captured_graph():
    """step_graph with the encoder losses (static phoneme-target buffer) follows the eager step."""
    from tests.test_models_gpu import _fresh_nets
    from ste_gan_b200.models.emg_encoder import EMGEncoderTransformer
    from ste_gan_b200.trainer import GanTrainer
    su, sess, x_real = (t.cuda() for t in O.synthetic_batch(2, 64, seed=15))
    ph = torch.randint(0, 48, (2, 64), generator=torch.Generator().manual_seed(16)).cuda()
    trainers = []
    for _ in range(2):
        torch.manual_seed(0)
        enc = EMGEncoderTransformer(8, 256, 48, model_size=128, num_transformer_layers=2).eval().cuda()
        g, d = _fresh_nets()
        trainers.append(GanTrainer(g.cuda(), d.cuda(), precision="bf16", emg_encoder=enc))
    t1, t2 = trainers
    t2.capture(2, 64)
    for _ in range(2):
        t1.step(su, sess, x_real, phoneme_targets=ph)
        t2.step_graph(su, sess, x_real, phoneme_targets=ph)
    t2.flush()
    a, b = t1.losses(), t2.losses()
    for k in a:
        assert abs(a[k] - b[k]) <= 2e-2 * max(1.0, abs(a[k])), (k, a[k], b[k])
    assert a["loss_speech_unit"] > 0 and a["loss_phoneme"] > 0
    assert O.rel_l2(t2.G.flat, t1.G.flat) < 3e-3
    with pytest.raises(ValueError):
        t2.step_graph(su, sess, x_real)
