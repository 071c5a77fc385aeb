"""Per-shape conv / wgrad times of one eager GAN train step at the bench configuration (configs[1]: batch 16, 100 unit
frames, bf16, DiscriminatorSmall), or of one GanTrainer.disc_losses_step (configs[4]) with `disc`:
    python tools/step_shapes.py [rows]
    python tools/step_shapes.py disc [small|full] [batch]
Each distinct launch is also replayed alone on the chip (its own descriptor and buffers, CUDA events)."""
import os, sys, collections
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from ste_gan_b200 import ops
from ste_gan_b200.models.discriminator import Discriminator, DiscriminatorSmall
from ste_gan_b200.models.generator import EMGGeneratorGanTTS
from ste_gan_b200.synthetic import synthetic_batch
from ste_gan_b200.trainer import GanTrainer
args = sys.argv[1:]
if args[:1] == ["disc"]:
    family = args[1] if len(args) > 1 else "full"
    B = int(args[2]) if len(args) > 2 else 16
    rows, title = 28, f"configs[4] {family} B={B} discriminator + losses"
    torch.manual_seed(0); g = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8, channels=64).cuda()
    torch.manual_seed(0); d = (DiscriminatorSmall if family == "small" else Discriminator)(8).cuda()
    tr = GanTrainer(g, d, precision="bf16")
    x_real = synthetic_batch(B, 100, seed=11)[2].cuda()
    x_pred = torch.tanh(torch.randn(B, 1600, 8, generator=torch.Generator().manual_seed(12))).cuda()
    run = lambda: tr.disc_losses_step(x_pred, x_real)
else:
    rows, title = int(args[0]) if args else 200, "configs[1] train step"
    torch.manual_seed(0); g = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8).cuda()
    torch.manual_seed(0); d = DiscriminatorSmall(8).cuda()
    tr = GanTrainer(g, d, precision="bf16")
    batch = [t.cuda() for t in synthetic_batch(16, 100, seed=0)]
    run = lambda: tr.step(*batch)
for _ in range(3):
    run()
torch.cuda.synchronize()
ops.profile = []
torch.cuda._sleep(int(0.06 * 1.9e9))
run()
torch.cuda.synchronize()
prof, ops.profile = ops.profile, None
import ctypes as C
from ste_gan_b200 import _lib
lib = _lib.load()
REPS = 10


def replay_us(p):
    """The launch replayed REPS times back to back inside one CUDA graph (its own descriptor and buffers)."""
    fn = getattr(lib, p["fn"])
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st):
            for _ in range(REPS):
                fn(C.byref(p["desc"]), C.c_void_p(st.cuda_stream))
        g.replay(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st); g.replay(); e1.record(st); torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / REPS


agg = collections.OrderedDict()
for p in prof:
    k = (p["kind"], p["engine"], p["shape"])
    first = k not in agg
    a = agg.setdefault(k, [0, 0.0, 0.0, 0.0, 0.0])
    a[4] += p.get("ingest", 0.0)
    a[0] += 1; a[1] += p["events"][0].elapsed_time(p["events"][1]) * 1e3; a[2] += p["flops"]
    if first:
        a[3] = replay_us(p)
tot = sum(a[1] for a in agg.values())
print(f"{title}: {len(prof)} conv/wgrad launches, {tot:.0f} us (events around each launch inside the step), "
      f"{sum(a[2] for a in agg.values()) / 1e9:.1f} GFLOP")
print(f"back-to-back graph replay of each distinct launch x its count: {sum(a[0] * a[3] for a in agg.values()):.0f} us")
print(f"planned shared-memory ingest of the tcgen05 launches: {sum(a[4] for a in agg.values()) / 1e9:.2f} GB per step")
print("kind  engine  (B, phases, t_src, t_dst, c_src, c_dst, k, dil, stride, groups)   n  in_step_us(avg)  replay_us  n*replay  TFLOP/s(replay)  ingest MB/launch  B/clk/SM(replay)")
for (kind, eng, shape), (n, us, fl, rp, ing) in sorted(agg.items(), key=lambda kv: -kv[1][0] * kv[1][3])[:rows]:
    print(f"{kind:5s} {eng:7s} {str(shape):58s} {n:3d} {us / n:9.1f} {rp:9.1f} {n * rp:9.1f} {fl / n / rp / 1e6:8.1f} {ing / n / 1e6:9.1f} {ing / n / (rp * 1965 * 148):8.1f}")
