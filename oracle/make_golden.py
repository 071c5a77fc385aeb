"""Generate tests/golden/*.pt by running the UNMODIFIED reference modules.

Needs a checkout of the original STE-GAN (the directory that holds its `ste_gan` package):
    STE_GAN_REFERENCE=<checkout> python oracle/make_golden.py
The reference imports `omegaconf` (absent here) for type annotations only, so a
3-line in-memory stub is installed first (SURVEY.md 8c).  Nothing from the
reference is copied; only its *outputs* on seeded inputs are stored.

Fixtures (all fp32, seed 0):
  init_checksums.pt   per-key checksums of the seed-0 random init of G, small D and
                      full D - pins that the drop-in modules initialise identically,
                      so the large weights never need to be committed.
  generator_tiny.pt   channels=64 generator: full state_dict + inputs + output.
  td_loss.pt          inputs + features + the three loss values.
  disc_small.pt / disc_full.pt   seed-0 discriminators on a seeded input: per-fmap
                      shape, checksum and strided samples (two consecutive training
                      forwards, so the spectral-norm power iteration is pinned).
  train_step_b1.pt    BASELINE.json configs[0]: G + small D fwd/bwd, B=1, T=100:
                      losses, G output, per-parameter gradient norms and samples.
  emg_encoder_init.pt per-key checksums of the seed-0 initialisation of that encoder (pins the drop-in module's init).
  emg_encoder_tiny.pt (SURVEY.md 8f rank 1) a model_size=32, 2-layer EMG encoder in eval
                      mode on two inputs (25 and 111 frames): both outputs, the speech-unit and
                      phoneme losses and the gradient of their sum w.r.t. the EMG input.  Its
                      weights and inputs are drawn from seeds (oracle/emg_encoder_oracle.py,
                      tiny_encoder_state / tiny_case_inputs), not stored.
"""
import os
import sys
import types
import warnings

import torch

warnings.filterwarnings("ignore")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
m = types.ModuleType("omegaconf"); m.OmegaConf = object; m.DictConfig = dict
sys.modules["omegaconf"] = m
sys.path.insert(0, os.environ["STE_GAN_REFERENCE"])

import torch.nn.functional as F  # noqa: E402
from ste_gan.losses.time_domain_loss import MultiTimeDomainFeatureLoss  # noqa: E402
from ste_gan.models.discriminator import Discriminator, DiscriminatorSmall  # noqa: E402
from ste_gan.models.generator import EMGGeneratorGanTTS  # noqa: E402

from oracle import ste_gan_oracle as O  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
os.makedirs(OUT, exist_ok=True)
torch.set_num_threads(os.cpu_count())


def checksum(t: torch.Tensor):
    t = t.detach().double().flatten()
    n = t.numel()
    idx = torch.linspace(0, n - 1, min(n, 16)).long()
    return dict(shape=list(t.shape) if False else None, numel=n, sum=t.sum().item(), abssum=t.abs().sum().item(),
                l2=t.norm().item(), samples=t[idx].float().clone(), idx=idx)


def tensor_summary(t: torch.Tensor):
    c = checksum(t)
    c["shape"] = list(t.shape)
    return c


def seeded(ctor, seed=0):
    torch.manual_seed(seed)
    return ctor()


def main():
    # ---- init checksums -------------------------------------------------
    g = seeded(lambda: EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8))
    ds = seeded(lambda: DiscriminatorSmall(8))
    df = seeded(lambda: Discriminator(8))
    gm = seeded(lambda: EMGGeneratorGanTTS("MFCCS", 25, 17, 8))
    init = {name: {k: tensor_summary(v) for k, v in mod.state_dict().items()}
            for name, mod in [("generator", g), ("disc_small", ds), ("disc_full", df), ("generator_mfcc", gm)]}
    init["param_order"] = {name: [n for n, _ in mod.named_parameters()]
                           for name, mod in [("generator", g), ("disc_small", ds), ("disc_full", df)]}
    torch.save(init, os.path.join(OUT, "init_checksums.pt"))

    # ---- tiny generator with stored weights ----------------------------
    gt = seeded(lambda: EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8, channels=64), seed=1)
    su, sess, _ = O.synthetic_batch(2, 12, seed=3)
    with torch.no_grad():
        y = gt(su, sess, torch.zeros(2, dtype=torch.long))
    sd = {k: v.detach().clone() for k, v in gt.state_dict().items()}
    assert O.rel_l2(O.generator_forward(sd, su, sess), y) < 1e-6
    torch.save(dict(state_dict=sd, speech_units=su, session_ids=sess, output=y, channels=64),
               os.path.join(OUT, "generator_tiny.pt"))

    # ---- TD loss ---------------------------------------------------------
    gen = torch.Generator().manual_seed(5)
    xr = torch.tanh(torch.randn(2, 160, 8, generator=gen))
    xg = torch.tanh(torch.randn(2, 160, 8, generator=gen)).requires_grad_(True)
    mtd = MultiTimeDomainFeatureLoss(8)
    loss, parts = mtd.time_domain_loss(xr, xg)
    (grad,) = torch.autograd.grad(loss, xg)
    feats = [l.calculate_time_domain_features(xr).detach() for l in mtd.time_domain_losses]
    torch.save(dict(x_real=xr, x_gen=xg.detach(), loss=loss.detach(), parts=[p.detach() for p in parts],
                    grad_x_gen=grad, feats_real=feats), os.path.join(OUT, "td_loss.pt"))
    ol, op = O.multi_td_loss(xr, xg.detach())
    assert abs(float(ol) - float(loss)) < 1e-6, (float(ol), float(loss))

    # ---- discriminators: two consecutive training forwards ---------------
    for name, mod, small in [("disc_small", ds, True), ("disc_full", df, False)]:
        gen = torch.Generator().manual_seed(7)
        x = torch.tanh(torch.randn(2, 400, 8, generator=gen))
        sd0 = {k: v.detach().clone() for k, v in mod.state_dict().items()}
        passes = []
        for _ in range(2):
            with torch.no_grad():
                res = mod(x)
            passes.append([[tensor_summary(f) for f in fm] for fm in res])
        # oracle agreement (functional restatement, same two forwards)
        sdo = {k: v.clone() for k, v in sd0.items()}
        for p in range(2):
            with torch.no_grad():
                ores = O.discriminator_forward(sdo, x, small=small, training=True)
            for a, b in zip(ores, passes[p]):
                for fa, fb in zip(a, b):
                    assert list(fa.shape) == fb["shape"]
                    assert abs(fa.double().sum().item() - fb["sum"]) <= 1e-4 * max(1.0, fb["abssum"]), name
        torch.save(dict(x=x, passes=passes, names=mod.discriminator_names), os.path.join(OUT, f"{name}.pt"))

    # ---- configs[0]: B=1 T=100 G + small D fwd/bwd ------------------------
    g = seeded(lambda: EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8))
    ds = seeded(lambda: DiscriminatorSmall(8))
    sd_g = {k: v.detach().clone() for k, v in g.state_dict().items()}
    sd_d = {k: v.detach().clone() for k, v in ds.state_dict().items()}
    su, sess, x_real = O.synthetic_batch(1, 100, seed=0)
    mtd = MultiTimeDomainFeatureLoss(8)
    g.train(); ds.train()
    x_pred = g(su, sess, torch.zeros(1, dtype=torch.long))
    d_fake_det = ds(x_pred.detach()); d_real = ds(x_real)
    loss_d = 0
    for sc in d_fake_det:
        loss_d = loss_d + F.mse_loss(sc[-1], torch.zeros_like(sc[-1]))
    for sc in d_real:
        loss_d = loss_d + F.mse_loss(sc[-1], torch.ones_like(sc[-1]))
    ds.zero_grad(); loss_d.backward()
    grad_d = {n: p.grad.detach().clone() for n, p in ds.named_parameters()}
    ds.zero_grad()
    d_fake = ds(x_pred); d_real = ds(x_real)
    loss_adv = 0
    for sc in d_fake:
        loss_adv = loss_adv + F.mse_loss(sc[-1], torch.ones_like(sc[-1]))
    td = mtd(x_real, x_pred)
    fm = 0
    for i in range(len(d_fake)):
        for j in range(len(d_fake[i]) - 1):
            fm = fm + F.l1_loss(d_fake[i][j], d_real[i][j].detach())
    loss_g = loss_adv + 15.0 * td + 7.0 * fm
    x_pred.retain_grad()
    loss_g.backward()
    grad_g = {n: p.grad.detach().clone() for n, p in g.named_parameters()}
    ref = dict(loss_d=loss_d.detach(), loss_g=loss_g.detach(), loss_adv=loss_adv.detach(), loss_td=td.detach(),
               loss_fm=fm.detach(), x_pred=x_pred.detach().clone(), grad_x_pred=x_pred.grad.detach().clone(),
               grad_g={k: tensor_summary(v) for k, v in grad_g.items()},
               grad_d={k: tensor_summary(v) for k, v in grad_d.items()},
               d_fake_det=[[tensor_summary(f) for f in fm_] for fm_ in d_fake_det])
    torch.save(ref, os.path.join(OUT, "train_step_b1.pt"))
    # oracle agreement on the same step (no D update between the phases, as above)
    o = O.losses_and_grads(sd_g, sd_d, su, sess, x_real, small=True)
    for k in ("loss_d", "loss_g", "loss_adv", "loss_td", "loss_fm"):
        assert abs(float(o[k]) - float(ref[k])) <= 1e-5 * max(1.0, abs(float(ref[k]))), (k, float(o[k]), float(ref[k]))
    assert O.rel_l2(o["x_pred"], ref["x_pred"]) < 1e-6
    worst = max(O.rel_l2(o["grad_g"][k], grad_g[k]) for k in grad_g)
    worst_d = max(O.rel_l2(o["grad_d"][k], grad_d[k]) for k in grad_d)
    print("oracle vs reference: worst grad_g rel-L2 %.3e, worst grad_d rel-L2 %.3e" % (worst, worst_d))
    assert worst < 1e-4 and worst_d < 1e-4
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


def emg_encoder_fixture():
    """SURVEY.md 8f rank 1: the frozen EMG encoder (eval mode) and the two losses taken through it, from the reference
    modules (ste_gan/models/emg_encoder.py, ste_gan/losses/emg_encoder_loss.py).  torch 2.11's nn.TransformerEncoder
    .forward rejects the reference's custom layer (it reads self_attn.batch_first; the reference pins torch 2.0.1), so
    the encoder's own layers are applied one after the other - exactly what 2.0.1 does for a mask-free stack."""
    from ste_gan.models.emg_encoder import EMGEncoderTransformer
    from oracle import emg_encoder_oracle as E
    torch.manual_seed(0)
    enc = EMGEncoderTransformer(8, 256, 48, **E.TINY_ENCODER).eval()
    # seed-0 initialisation checksums (key order included): pins that the drop-in module consumes the RNG identically
    torch.save({k: tensor_summary(v.float()) for k, v in enc.state_dict().items()}, os.path.join(OUT, "emg_encoder_init.pt"))
    enc.load_state_dict(E.tiny_encoder_state(EMGEncoderTransformer))     # fp16-grid weights, non-trivial BatchNorm statistics

    def fwd(x):
        h = enc.conv_blocks(x.transpose(1, 2)).transpose(1, 2)
        h = enc.w_raw_in(h).transpose(0, 1)
        for layer in enc.transformer.layers:
            h = layer(h)
        h = h.transpose(0, 1)
        return enc.w_out(h), enc.w_aux(h)

    cases = []
    for i in range(len(E.TINY_CASE_SHAPES)):
        x, tgt, ph = E.tiny_case_inputs(i)
        x.requires_grad_(True)
        units, phon = fwd(x)
        unit_loss = F.pairwise_distance(tgt.reshape(-1, 256), units.reshape(-1, 256)).mean()     # emg_encoder_loss.py:63-67
        ce = F.cross_entropy(phon.transpose(1, 2), ph)                                           # :80-83
        (dx,) = torch.autograd.grad(unit_loss + ce, x)
        cases.append(dict(units=units.detach(), phonemes=phon.detach(), unit_loss=unit_loss.detach(), phoneme_loss=ce.detach(),
                          dx=dx))
    torch.save(dict(cases=cases), os.path.join(OUT, "emg_encoder_tiny.pt"))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "emg_encoder":     # only the fixture of the section-8f row
        emg_encoder_fixture()
    else:
        main()
        emg_encoder_fixture()
