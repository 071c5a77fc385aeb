"""Data-parallel correctness check (GPU, 2+ ranks): N ranks x B samples through the bucketed graph step vs ONE
process on the global batch (eager step, no exchange).  fp32 validation mode, 2 optimiser steps.
    torchrun --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/dp_check.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist
from oracle import ste_gan_oracle as O
from ste_gan_b200.dist import init_from_env
from ste_gan_b200.models.discriminator import DiscriminatorSmall
from ste_gan_b200.models.generator import EMGGeneratorGanTTS
from ste_gan_b200.trainer import GanTrainer

rank, world, local = init_from_env("nccl")
dev = torch.device("cuda", local)
B, T, STEPS = 2, 64, 2


def nets():
    torch.manual_seed(0); g = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8, channels=128).to(dev)
    torch.manual_seed(0); d = DiscriminatorSmall(8).to(dev)
    return g, d


batches = [O.synthetic_batch(B * world, T, seed=100 + s) for s in range(STEPS)]
tr = GanTrainer(*nets(), precision="fp32")
assert tr.reducer.enabled and len(tr.g_buckets) == 3
tr.capture(B, T)                     # (its warm-up steps leave no trace in the training state)
for su, sess, xr in batches:
    sl = slice(rank * B, (rank + 1) * B)
    tr.step_graph(su[sl].to(dev), sess[sl].to(dev), xr[sl].to(dev))
tr.flush()
torch.cuda.synchronize()
if rank == 0:
    ref = GanTrainer(*nets(), precision="fp32", data_parallel=False)          # single process, global batch
    for su, sess, xr in batches:
        ref.step(su.to(dev), sess.to(dev), xr.to(dev))
    torch.cuda.synchronize()
    eg, ed = O.rel_l2(tr.G.flat, ref.G.flat), O.rel_l2(tr.D.flat, ref.D.flat)
    print(f"dp_check: world {world}, rel-L2 of the parameters after {STEPS} steps vs one process on the global batch: G {eg:.3e}  D {ed:.3e}")
    assert eg < 3e-3 and ed < 3e-3, (eg, ed)
    print("dp_check ok")
dist.barrier()
dist.destroy_process_group()
