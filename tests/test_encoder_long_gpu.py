"""The frozen EMG encoder past the sequence lengths of the one-CTA-per-head attention kernels: the band-tiled attention kernels
against an fp64 reference and against the dense kernels, then the encoder, its drop-in loss module and the train step at lengths
only the band kernels take.

Tolerances as everywhere: relative L2 <= 1e-4 in the fp32 validation mode, <= 2e-2 in bf16 (kernels alone: 2e-5 / 6e-3).
"""
import pytest
import torch

from oracle import emg_encoder_oracle as E
from oracle import ste_gan_oracle as O
from tests.test_encoder_gpu import DT, TOL, _enc_masks, _tiny_encoder

pytestmark = pytest.mark.gpu
M = 100


def _attn_case(B, L, H, d, prec, seed):
    gen = torch.Generator().manual_seed(seed)
    qkv = torch.randn(B, L, 3 * H * d, generator=gen)
    emb = torch.randn(H, 2 * M - 1, d, generator=gen) * d ** -0.5
    do = torch.randn(B, L, H * d, generator=gen)
    if prec == "bf16":
        qkv, do = qkv.to(torch.bfloat16).float(), do.to(torch.bfloat16).float()
    return qkv, emb, do


def _reference(qkv, emb, do, H):
    """fp64 einsum restatement (the formula of test_relative_attention_kernels): probs [B,H,L,L], o, d/dqkv."""
    B, L, C3 = qkv.shape
    d = C3 // (3 * H)
    qr = qkv.double().requires_grad_(True)
    q, k, v = (t.view(B, L, H, d).permute(0, 2, 1, 3) for t in qr.split(H * d, dim=-1))
    logits = torch.einsum("bhqa,bhka->bhqk", q, k) / d ** 0.5 + E.relative_logits(q, emb.double())
    probs = torch.softmax(logits, -1)
    o = torch.einsum("bhqk,bhka->bhqa", probs, v).permute(0, 2, 1, 3).reshape(B, L, H * d)
    (dq,) = torch.autograd.grad(o, qr, do.double())
    return probs.detach(), o.detach(), dq


def band_to_dense(pb: torch.Tensor) -> torch.Tensor:
    """probs_band [B,H,L,2M-1] -> [B,H,L,L]; asserts that the entries whose key lies outside [0, L) are exactly 0."""
    pb = pb.float().cpu()
    B, H, L, W = pb.shape
    i, w = torch.arange(L)[:, None], torch.arange(W)[None, :]
    j = i + w - (M - 1)
    ok = (j >= 0) & (j < L)
    assert torch.all(pb[:, :, ~ok] == 0)
    dense = torch.zeros(B, H, L, L)
    dense[:, :, i.expand(L, W)[ok], j[ok]] = pb[:, :, ok]
    return dense


GEOMS = [(2, L, 2, d) for d in (4, 96) for L in (1, 25, 99, 100, 101, 111, 257)] + [(1, 600, 4, 16), (1, 1500, 2, 96)]


@pytest.mark.parametrize("geom", GEOMS, ids=[f"B{b}_L{l}_H{h}_d{d}" for b, l, h, d in GEOMS])
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_band_attention_vs_fp64(prec, geom):
    """o, the input gradient and the band-layout probabilities against fp64; L = 1 / < M / < one 32-row tile / a partly empty
    last tile / many tiles."""
    from ste_gan_b200 import ops
    B, L, H, d = geom
    qkv, emb, do = _attn_case(B, L, H, d, prec, seed=L + d)
    probs, o_ref, dq_ref = _reference(qkv, emb, do, H)
    dev = lambda t: t.cuda().to(DT[prec])
    o, pb = ops.relattn_band_fwd(dev(qkv), emb.cuda(), H, M)
    assert pb.shape == (B, H, L, 2 * M - 1)
    dqkv = ops.relattn_band_bwd(dev(qkv), emb.cuda(), pb, dev(do), H, M)
    tol = 2e-5 if prec == "fp32" else 6e-3
    assert O.rel_l2(band_to_dense(pb), probs) < tol
    assert O.rel_l2(o, o_ref) < tol and O.rel_l2(dqkv, dq_ref) < tol


@pytest.mark.parametrize("L", [25, 100, 128])
def test_band_equals_dense(L):
    """Where both kernels run, they compute the same thing: only the order of the softmax and D sums differs."""
    from ste_gan_b200 import ops
    B, H, d = 2, 8, 96
    qkv, emb, do = (t.cuda() for t in _attn_case(B, L, H, d, "fp32", seed=7 * L))
    emb = emb.cuda()
    o_d, p_d = ops.relattn_fwd(qkv, emb, H, M)
    dq_d = ops.relattn_bwd(qkv, emb, p_d, do, H, M)
    o_b, p_b = ops.relattn_band_fwd(qkv, emb, H, M)
    dq_b = ops.relattn_band_bwd(qkv, emb, p_b, do, H, M)
    assert O.rel_l2(band_to_dense(p_b), p_d) <= 1e-6
    assert O.rel_l2(o_b, o_d) <= 1e-6 and O.rel_l2(dq_b, dq_d) <= 1e-6


def test_band_backward_is_deterministic():
    from ste_gan_b200 import ops
    qkv, emb, do = (t.cuda().to(torch.bfloat16) for t in _attn_case(4, 700, 8, 96, "bf16", seed=11))
    emb = emb.float()
    o1, p1 = ops.relattn_band_fwd(qkv, emb, 8, M)
    o2, p2 = ops.relattn_band_fwd(qkv, emb, 8, M)
    g1 = ops.relattn_band_bwd(qkv, emb, p1, do, 8, M)
    g2 = ops.relattn_band_bwd(qkv, emb, p2, do, 8, M)
    assert torch.equal(o1, o2) and torch.equal(p1, p2) and torch.equal(g1, g2)


def _check_vs_oracle(plan, sd, x, ut, ph, prec):
    """heads, both losses and the input gradient of their sum against the fp64 oracle with the ReLU sign patterns of this forward;
    every attention layer must have run on the band kernels."""
    from ste_gan_b200 import passes_encoder as pe
    slots = torch.zeros(2, device="cuda")
    dx, units, logits = pe.encoder_losses(plan, x.cuda(), ut.cuda(), ph.cuda(), slots, 1.0, 1.0)
    _, _, ctx = pe.encoder_forward(plan, x.cuda())
    assert all(s["band"] for s in ctx.layers)
    xr = x.double().requires_grad_(True)
    f64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    u, l_ = E.emg_encoder_forward(f64, xr, _enc_masks(ctx))
    su, ce = E.encoder_losses(u, l_, ut.double(), ph)
    (dx_ref,) = torch.autograd.grad(su + ce, xr)
    tol = TOL[prec]
    assert O.rel_l2(units, u) < tol and O.rel_l2(logits, l_) < tol
    assert abs(float(slots[0]) - float(su)) <= tol * float(su) and abs(float(slots[1]) - float(ce)) <= tol * float(ce)
    assert O.rel_l2(dx, dx_ref) < tol


@pytest.mark.parametrize("shape", [(1, 24000), (2, 16000)], ids=["1x1500frames", "2x1000frames"])
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_tiny_encoder_long_vs_oracle(prec, shape):
    """The tiny fixture encoder (head dim 4: the dense forward stops at 720 frames) on a 30 s utterance and a batch of 20 s ones."""
    enc, sd, _ = _tiny_encoder()
    B, T = shape
    g = torch.Generator().manual_seed(T + B)
    x = torch.tanh(torch.randn(B, T, 8, generator=g))
    ut, ph = torch.randn(B, T // 16, 256, generator=g), torch.randint(0, 48, (B, T // 16), generator=g)
    _check_vs_oracle(enc.cuda().plan(DT[prec]), sd, x, ut, ph, prec)


def _full_size_encoder(**kw):
    """768-d, 8 heads of 96, random init with non-trivial BatchNorm statistics (as test_encoder_full_size_vs_oracle)."""
    from ste_gan_b200.models.emg_encoder import EMGEncoderTransformer
    torch.manual_seed(0)
    enc = EMGEncoderTransformer(8, 256, 48, **kw).eval()
    g = torch.Generator().manual_seed(5)
    for mod in enc.modules():
        if isinstance(mod, torch.nn.BatchNorm1d):
            mod.running_mean.normal_(0, 0.3, generator=g); mod.running_var.uniform_(0.5, 1.5, generator=g)
            mod.weight.data.uniform_(0.5, 1.5, generator=g); mod.bias.data.normal_(0, 0.2, generator=g)
    return enc


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_full_size_encoder_300_frames_vs_oracle(prec):
    """4800 EMG samples = 300 frames: past both dense kernels at head dim 96 (206 forward, 133 backward)."""
    enc = _full_size_encoder()
    sd = {k: v.detach().clone() for k, v in enc.state_dict().items()}
    g = torch.Generator().manual_seed(6)
    x = torch.tanh(torch.randn(1, 4800, 8, generator=g))
    ut, ph = torch.randn(1, 300, 256, generator=g), torch.randint(0, 48, (1, 300), generator=g)
    _check_vs_oracle(enc.cuda().plan(DT[prec]), sd, x, ut, ph, prec)


def test_loss_module_on_a_30s_utterance():
    """EMGEncoderLoss through autograd on one 24000-sample utterance, full-size encoder, bf16."""
    import ste_gan_b200
    from ste_gan_b200.losses.emg_encoder_loss import EMGEncoderLoss
    enc = _full_size_encoder().cuda()
    g = torch.Generator().manual_seed(8)
    x = torch.tanh(torch.randn(1, 24000, 8, generator=g)).cuda().requires_grad_(True)
    ut, ph = torch.randn(1, 1500, 256, generator=g).cuda(), torch.randint(0, 48, (1, 1500), generator=g).cuda()
    with ste_gan_b200.precision("bf16"):
        out = EMGEncoderLoss(enc)(x, ut, ph)
        (out.speech_unit_loss + out.phoneme_loss).backward()
        with torch.no_grad():
            units, logits = enc(x)
    assert out.speech_unit_pred.shape == (1, 1500, 256) and out.phoneme_pred.shape == (1, 1500, 48)
    assert torch.isfinite(x.grad).all() and float(x.grad.abs().sum()) > 0
    assert torch.isfinite(out.speech_unit_loss) and torch.isfinite(out.phoneme_loss)
    assert O.rel_l2(units, out.speech_unit_pred) < 1e-6 and O.rel_l2(logits, out.phoneme_pred) < 1e-6


def _one_layer_encoder():
    from ste_gan_b200.models.emg_encoder import EMGEncoderTransformer
    torch.manual_seed(0)
    return EMGEncoderTransformer(8, 256, 48, num_transformer_layers=1).eval()


def _assert_band_route(trainer, x):
    """The trainer's encoder pass at the shape of x (with the context its backward needs) runs on the band kernels."""
    from ste_gan_b200 import passes_encoder as pe
    _, _, ctx = pe.encoder_forward(trainer._enc_plan, x.cuda())
    assert ctx.layers and all(s["band"] for s in ctx.layers)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_train_step_with_encoder_losses_past_133_frames(prec):
    """GanTrainer with the encoder losses at 144 frames (2304 EMG samples): head dim 96, longer than the dense backward takes."""
    from tests.test_models_gpu import _fresh_nets, run_step_vs_oracle
    enc = _one_layer_encoder()
    g, d = _fresh_nets()
    su, sess, x_real = O.synthetic_batch(2, 144, seed=17)
    ph = torch.randint(0, 48, (2, 144), generator=torch.Generator().manual_seed(18))
    tr, ref = run_step_vs_oracle(g, d, (su, sess, x_real), prec, encoder=(enc, ph))
    _assert_band_route(tr, x_real)
    L = tr.losses()
    tol = TOL[prec]
    for k in ("loss_speech_unit", "loss_phoneme"):
        assert abs(L[k] - float(ref[k])) <= tol * max(1.0, abs(float(ref[k]))), (k, L[k], float(ref[k]))


def test_encoder_losses_in_captured_graph_past_133_frames():
    """capture(2, 144) + step_graph follows the eager step."""
    from tests.test_models_gpu import _fresh_nets
    from ste_gan_b200.trainer import GanTrainer
    su, sess, x_real = (t.cuda() for t in O.synthetic_batch(2, 144, seed=19))
    ph = torch.randint(0, 48, (2, 144), generator=torch.Generator().manual_seed(20)).cuda()
    trainers = []
    for _ in range(2):
        enc = _one_layer_encoder().cuda()
        g, d = _fresh_nets()
        trainers.append(GanTrainer(g.cuda(), d.cuda(), precision="bf16", emg_encoder=enc))
    t1, t2 = trainers
    t2.capture(2, 144)
    _assert_band_route(t1, x_real)
    for _ in range(2):
        t1.step(su, sess, x_real, phoneme_targets=ph)
        t2.step_graph(su, sess, x_real, phoneme_targets=ph)
    t2.flush()
    a, b = t1.losses(), t2.losses()
    for k in a:
        assert abs(a[k] - b[k]) <= 2e-2 * max(1.0, abs(a[k])), (k, a[k], b[k])
    assert a["loss_speech_unit"] > 0 and a["loss_phoneme"] > 0
    assert O.rel_l2(t2.G.flat, t1.G.flat) < 3e-3
