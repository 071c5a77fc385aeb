"""CPU: the oracle (oracle/ste_gan_oracle.py) against the committed golden fixtures produced from the
UNMODIFIED reference modules (oracle/make_golden.py), and against the live reference when the
environment variable STE_GAN_REFERENCE names a checkout of the original STE-GAN (the directory that
holds its `ste_gan` package)."""
import os
import sys
import types

import pytest
import torch

from oracle import ste_gan_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")
REF = os.environ.get("STE_GAN_REFERENCE", "")
HAVE_REF = bool(REF) and os.path.isdir(os.path.join(REF, "ste_gan"))


def _seed0_state_dicts():
    """Seed-0 weights through the drop-in modules (bit-identical to the reference init, see
    test_host_cpu.py::test_init_matches_golden_checksums)."""
    from ste_gan_b200.models.discriminator import Discriminator, DiscriminatorSmall
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    torch.manual_seed(0); g = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8)
    torch.manual_seed(0); ds = DiscriminatorSmall(8)
    torch.manual_seed(0); df = Discriminator(8)
    sd = lambda m: {k: v.detach().clone() for k, v in m.state_dict().items()}
    return sd(g), sd(ds), sd(df)


def test_generator_tiny_golden():
    fx = torch.load(os.path.join(GOLD, "generator_tiny.pt"))
    y = O.generator_forward(fx["state_dict"], fx["speech_units"], fx["session_ids"])
    assert y.shape == fx["output"].shape
    assert O.rel_l2(y, fx["output"]) < 1e-6


def test_td_loss_golden():
    fx = torch.load(os.path.join(GOLD, "td_loss.pt"))
    xg = fx["x_gen"].clone().requires_grad_(True)
    loss, parts = O.multi_td_loss(fx["x_real"], xg)
    assert abs(float(loss) - float(fx["loss"])) < 1e-6 * abs(float(fx["loss"]))
    for a, b in zip(parts, fx["parts"]):
        assert abs(float(a) - float(b)) < 1e-6 * abs(float(b))
    (g,) = torch.autograd.grad(loss, xg)
    assert O.rel_l2(g, fx["grad_x_gen"]) < 1e-6
    for (w, s), ref in zip(O.TD_RESOLUTIONS, fx["feats_real"]):
        assert O.rel_l2(O.td_features(fx["x_real"], w, s), ref) < 1e-6


@pytest.mark.parametrize("small", [True, False], ids=["small", "full"])
def test_discriminator_golden_two_forwards(small):
    fx = torch.load(os.path.join(GOLD, "disc_small.pt" if small else "disc_full.pt"))
    _, sds, sdf = _seed0_state_dicts()
    sd = sds if small else sdf
    for p in range(2):
        with torch.no_grad():
            res = O.discriminator_forward(sd, fx["x"], small=small, training=True)
        for fms, refs in zip(res, fx["passes"][p]):
            assert len(fms) == len(refs)
            for fm, ref in zip(fms, refs):
                assert list(fm.shape) == ref["shape"]
                t = fm.double().contiguous().flatten()
                assert abs(t.norm().item() - ref["l2"]) <= 1e-5 * max(ref["l2"], 1e-6)
                assert torch.allclose(t[ref["idx"]].float(), ref["samples"], rtol=1e-4, atol=1e-6)


def test_train_step_b1_golden():
    """BASELINE.json configs[0]: G + small D fwd/bwd, batch 1, 100 frames, on CPU."""
    fx = torch.load(os.path.join(GOLD, "train_step_b1.pt"))
    sd_g, sd_d, _ = _seed0_state_dicts()
    su, sess, x_real = O.synthetic_batch(1, 100, seed=0)
    o = O.losses_and_grads(sd_g, sd_d, su, sess, x_real, small=True)
    for k in ("loss_d", "loss_g", "loss_adv", "loss_td", "loss_fm"):
        assert abs(float(o[k]) - float(fx[k])) <= 1e-5 * max(1.0, abs(float(fx[k]))), k
    assert O.rel_l2(o["x_pred"], fx["x_pred"]) < 1e-6
    assert O.rel_l2(o["grad_x_pred"], fx["grad_x_pred"]) < 1e-4
    for name, grads in (("grad_g", o["grad_g"]), ("grad_d", o["grad_d"])):
        for k, ref in fx[name].items():
            t = grads[k].double().flatten()
            assert abs(t.norm().item() - ref["l2"]) <= 2e-4 * max(ref["l2"], 1e-9), (name, k)


@pytest.mark.skipif(not HAVE_REF, reason="STE_GAN_REFERENCE does not name a checkout of the original STE-GAN")
def test_oracle_vs_live_reference():
    m = types.ModuleType("omegaconf"); m.OmegaConf = object; m.DictConfig = dict
    sys.modules.setdefault("omegaconf", m)
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import warnings
    warnings.filterwarnings("ignore")
    from ste_gan.models.discriminator import DiscriminatorSmall
    from ste_gan.models.generator import EMGGeneratorGanTTS
    torch.manual_seed(3); g = EMGGeneratorGanTTS("MFCCS", 25, 17, 8, channels=64, use_speaking_mode_embedding=True)
    gen = torch.Generator().manual_seed(1)
    x = torch.randn(2, 10, 25, generator=gen); sess = torch.tensor([3, 16]); mode = torch.tensor([0, 2])
    with torch.no_grad():
        y = g(x, sess, mode)
    sd = {k: v.detach().clone() for k, v in g.state_dict().items()}
    assert O.rel_l2(O.generator_forward(sd, x, sess, mode, "MFCCS"), y) < 1e-6
    torch.manual_seed(4); d = DiscriminatorSmall(8); d.eval()
    xs = torch.tanh(torch.randn(1, 330, 8, generator=gen))
    sdd = {k: v.detach().clone() for k, v in d.state_dict().items()}
    with torch.no_grad():
        ref = d(xs)
        got = O.discriminator_forward(sdd, xs, small=True, training=False)
    assert max(O.rel_l2(a, b) for fa, fb in zip(got, ref) for a, b in zip(fa, fb)) < 1e-5


def test_emg_encoder_oracle_matches_reference_fixture():
    """SURVEY.md 8f rank 1 (no CUDA path yet - this pins the oracle for it): the frozen EMG encoder's forward, the
    speech-unit / phoneme losses taken through it and the gradient of their sum w.r.t. the EMG input, against the
    reference modules' outputs (25 frames, and 111 frames > the 100-frame relative-position range)."""
    from oracle import emg_encoder_oracle as E
    from ste_gan_b200.models.emg_encoder import EMGEncoderTransformer
    fx = torch.load(os.path.join(GOLD, "emg_encoder_tiny.pt"))
    # the halves the reference ran on, drawn from their seeds (bit-identical: the drop-in initialises as the reference does)
    sd = {k: v.double() for k, v in E.tiny_encoder_state(EMGEncoderTransformer).items()}
    for i, case in enumerate(fx["cases"]):
        case["x"], case["unit_target"], case["phoneme_target"] = E.tiny_case_inputs(i)
        x = case["x"].double().requires_grad_(True)
        units, phon = E.emg_encoder_forward(sd, x)
        assert list(units.shape) == list(case["units"].shape) and list(phon.shape) == list(case["phonemes"].shape)
        assert O.rel_l2(units, case["units"]) < 1e-5 and O.rel_l2(phon, case["phonemes"]) < 1e-5
        ul, ce = E.encoder_losses(units, phon, case["unit_target"].double(), case["phoneme_target"])
        assert abs(float(ul) - float(case["unit_loss"])) < 1e-5 * float(case["unit_loss"])
        assert abs(float(ce) - float(case["phoneme_loss"])) < 1e-5 * float(case["phoneme_loss"])
        (dx,) = torch.autograd.grad(ul + ce, x)
        assert O.rel_l2(dx, case["dx"]) < 1e-4
