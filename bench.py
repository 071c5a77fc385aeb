#!/usr/bin/env python
"""bench.py - STE-GAN hot-path benchmark (BASELINE.json: GAN train samples/s, configs[1]).

    python bench.py --gpus N --steps K --warmup W [--repeats R] [--impl reference] [--torch-compile] [--no-cpu-baseline]
                    [--quick] [--dump-outputs DIR]
    (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

One "step" = one full GAN train step (train.py:165-268 without the encoder losses) on a synthetic batch of 16 samples
per GPU, 100 unit frames -> 1600x8 EMG samples, bf16 tensor-core mode, weak scaling (per-GPU batch fixed).  Prints ONE
JSON line (rank 0).  Inputs and initial weights come from fixed seeds: the same arguments give the same inputs.

  value     whole-job samples/s with inputs resident in HBM, CUDA-graph replay, device-timed; K timed steps in all, split
            into R timed regions (default 1, each bracketed by barrier + synchronize); the MEDIAN of their ms per step is
            reported
  --dump-outputs DIR  after those K steps: the loss slots, the generated batch and a fixed sample of the updated weights
            of the last step, as DIR/<name>.npy (float32), for comparing the outputs of two builds (two runs of one build
            differ by rounding noise that grows with the number of steps: DESIGN.md section 8)
  e2e       the same through GanTrainer.step_graph() with pinned HOST inputs (H2D inside the timed region) and a host
            read of the loss slots every step
  parity_gate  BEFORE any timing: the first graph step's losses against the CPU reference arm on the same batch and
            seed-0 weights (2e-2, the bf16 tolerance); the run aborts when they disagree
  roofline  dominant kernel (tcgen05 implicit-GEMM conv): ALGORITHMIC FLOPs of the launches recorded while the timed
            graphs were captured (module groups, not pack groups) / the kernel's busy time in a CUPTI timeline of replays
            of the SAME graphs (torch.profiler, outside the timed regions) vs MEASURED_PEAKS.json; `alone` = the same
            launches replayed one shape at a time, 10x back to back in a CUDA graph of their own; `hbm` = the HBM-bound kernels
  cpu_baseline  the reference's own modules (baseline/_ref, kind "reference"; the oracle port otherwise) on the host cores
  inference / disc_losses / context.torch_gpu  BASELINE.json configs[3], configs[4] and the same reference step on the
            B200 through torch + cuDNN (BASELINE.md section 5)
  --impl reference  times the CPU reference arm alone (rank 0), same metric / unit / config
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH_PER_GPU, FRAMES, UNIT_DIM, HOP, CHANNELS = 16, 100, 256, 16, 8
STEP_GFLOP_PER_SAMPLE = 94.7          # SURVEY.md 8(d): G 41.42 + D fwd 4x5.919 + D bwd 2x11.84 + D dgrad 5.92
INFER_FRAMES = 1500                   # configs[3]: 30 s utterances
G_FWD_GFLOP_PER_FRAME = 13.807 / 100  # SURVEY.md 8(d)
# configs[4], GFLOP per sample of one disc_losses step: D fwd x4 + D bwd (dgrad + wgrad) x2 + D dgrad x1 = 9 forward-equivalents
DISC_GFLOP_PER_SAMPLE = {"small": 9 * 5.919, "full": 9 * 3.509}
DISC_BATCHES = (16, 32, 64, 128, 256)
GATE_TOL = 2e-2


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(tflops=float(d["bf16_tflops_sustained"]), burst=float(d["bf16_tflops"]), hbm=float(d["hbm_gbs"]),
                    source="measured (MEASURED_PEAKS.json: sustained bf16 TFLOP/s, copy GB/s)")
    return dict(tflops=1400.0, burst=1590.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill(); out, _ = self.proc.communicate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def config_dict(world: int):
    return {"workload": "STE-GAN base train step (G + DiscriminatorSmall fwd/bwd, LSGAN + 15*multi-TD + 7*FM, 2x AdamW), "
                        "bf16, batch 16/GPU, 100 unit frames -> 1600x8 EMG samples (BASELINE.json configs[1])",
            "batch_per_gpu": BATCH_PER_GPU, "global_batch": BATCH_PER_GPU * world, "unit_frames": FRAMES,
            "emg_samples": FRAMES * HOP, "parallelism": f"dp{world}",
            "l2": "per-step working set (weights 212 MB + activations) exceeds the 126 MB L2; inputs rotate over 4 batches"}


# ------------------------------------------------------------------------------------------------ CPU reference arm
class CpuArm:
    """The reference's CPU path on the host cores (all threads): reference modules from baseline/_ref when installed
    (kind "reference"), the oracle port otherwise.  Step 0 runs on `seed_of_step0` and doubles as the warm-up; its losses
    are what the GPU arm's parity gate compares against."""

    def __init__(self):
        import torch
        from baseline import ref_runner as R
        torch.set_num_threads(os.cpu_count() or 1)
        self.R, self.torch = R, torch
        self.tr = R.make_trainer("cpu", small=True)
        self.kind, self.cores = self.tr.kind, torch.get_num_threads()

    def first_step(self, batch):
        t0 = time.perf_counter()
        L = self.R.losses_to_float(self.tr.step(*batch))
        self.first_s = time.perf_counter() - t0
        return L

    def timed(self, steps: int, warmup_extra: int, budget_s: float, seed0: int = 100):
        from ste_gan_b200.synthetic import synthetic_batch
        batch = BATCH_PER_GPU
        if self.first_s * (steps + warmup_extra) > budget_s:      # bound the sample: fewer samples per step
            batch = max(1, int(batch * budget_s / (self.first_s * (steps + warmup_extra))))
        for i in range(warmup_extra):
            self.tr.step(*synthetic_batch(batch, FRAMES, seed=1 + i))
        times = []
        for i in range(steps):
            b = synthetic_batch(batch, FRAMES, seed=seed0 + i)
            t0 = time.perf_counter(); self.tr.step(*b); times.append(time.perf_counter() - t0)
        ms = 1e3 * sum(times) / len(times)
        return dict(value=batch / (ms / 1e3), ms_per_step=ms, batch=batch, cores=self.cores, kind=self.kind,
                    sample=f"{steps} timed steps of batch {batch} x {FRAMES} frames (fp32, torch CPU ops, {self.cores} threads, "
                           f"{'reference modules from baseline/_ref' if self.kind == 'reference' else 'oracle port'})")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from ste_gan_b200.synthetic import synthetic_batch
    arm = CpuArm()
    arm.first_step(synthetic_batch(BATCH_PER_GPU, FRAMES, seed=0))
    r = arm.timed(args.steps, max(0, args.warmup - 1), budget_s=200.0)
    sample = r["sample"] + (f"; a bounded sample (batch {r['batch']}) of the global batch {BATCH_PER_GPU * args.gpus} per step"
                            if args.gpus > 1 or r["batch"] != BATCH_PER_GPU else "")
    line = {"impl": "reference", "metric": "GAN train samples/s", "value": r["value"], "unit": "samples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args.gpus),
            "cpu_baseline": {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": r["kind"], "sample": sample},
            "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ helpers (GPU arm)
KERNEL_KEYS = ("conv_tc_kernel", "wgrad_tc_kernel", "conv_simt_kernel", "wgrad_simt_kernel", "c1_fwd_kernel", "c1_dgrad_kernel",
               "c1_wgrad_kernel", "wn_fold_rows_kernel", "wn_bwd_multi_kernel", "adamw_kernel", "l1_mean_multi_kernel",
               "period_first_kernel", "scale_first_kernel")


def cupti_by_kernel(fn, n_rep: int):
    """Busy time per kernel NAME over n_rep calls of fn() from a CUPTI activity trace (torch.profiler): the per-launch
    durations of the kernels AS SCHEDULED in the replayed graphs (concurrent streams share the chip).  Returns
    {name: (launches per call, busy us per call)}, span us per call - or None when CUPTI is unavailable."""
    import torch
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n_rep):
                fn()
            torch.cuda.synchronize()
        with tempfile.NamedTemporaryFile(suffix=".json", delete=False) as tf:
            path = tf.name
        prof.export_chrome_trace(path)
        with open(path) as f:
            ev = json.load(f)["traceEvents"]
        os.unlink(path)
    except Exception as exc:      # noqa: BLE001
        return None, f"CUPTI timeline unavailable: {exc!r}"
    ks = [e for e in ev if e.get("cat") == "kernel"]
    if not ks:
        return None, "CUPTI timeline empty"
    out = {}
    for e in ks:
        nm = e["name"]
        key = next((k for k in KERNEL_KEYS if k in nm), None)
        if key is None:
            ids = [w for w in re.findall(r"([A-Za-z_][A-Za-z_0-9]*)\s*[<(]", nm) if w not in ("void", "anonymous")]
            key = "other:" + (ids[0] if ids else nm)[:48]
        a = out.setdefault(key, [0, 0.0])
        a[0] += 1; a[1] += float(e["dur"])
    span = (max(e["ts"] + e["dur"] for e in ks) - min(e["ts"] for e in ks)) / n_rep
    return {k: (v[0] / n_rep, v[1] / n_rep) for k, v in out.items()}, span


def timed_region(fn_step, fn_tail, steps: int, repeats: int, barrier, max_over_ranks):
    """Exactly `steps` steps in all, split into `repeats` consecutive timed regions of (nearly) equal length, every one
    bracketed by barrier + synchronize on both sides and timed with CUDA events on the launching stream; returns
    (median ms per step, ms per step of every region)."""
    import torch
    per = []
    n_regions = min(repeats, steps)
    done = 0
    for r in range(n_regions):
        n = steps // n_regions + (r < steps % n_regions)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(done, done + n):
            fn_step(i)
        fn_tail()
        e1.record()
        barrier()
        per.append(max_over_ranks(e0.elapsed_time(e1)) / n)
        done += n
    return statistics.median(per), per


def dump_outputs(out_dir: str, tr, net_g, net_d, sample: int = 1 << 20) -> None:
    """What the timed train step has handed its caller after its last step, as float32 .npy files: the loss slots
    (losses.npy, in the order of trainer.LOSS_NAMES), the generated EMG batch (x_pred.npy, [B, T, C]) and the updated
    weights of both networks (g_params.npy, d_params.npy: `sample` elements of all parameters concatenated in
    registration order, at indices drawn with seed 0, the same in every run) - 9 MB in all."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"losses": tr.slots, "x_pred": tr.x_pred}
    for name, net in (("g_params", net_g), ("d_params", net_d)):
        flat = torch.cat([p.detach().reshape(-1) for p in net.parameters()])
        idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:sample].sort().values
        arrays[name] = flat[idx.to(flat.device)]
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


# ------------------------------------------------------------------------------------------------ GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from ste_gan_b200 import _lib, ops
    from ste_gan_b200.dist import init_from_env
    from ste_gan_b200.inference import UtteranceGenerator
    from ste_gan_b200.models.discriminator import Discriminator, DiscriminatorSmall
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    from ste_gan_b200.synthetic import synthetic_batch
    from ste_gan_b200.trainer import GanTrainer

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product path has no CPU fallback (use --impl reference for the CPU arm)")
    rank, world, local = init_from_env("nccl")
    if world != args.gpus:
        raise SystemExit(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; launch N>1 with torch.distributed.run")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    lib = _lib.load(build_if_missing=False)
    peaks = load_peaks()
    solo = rank == 0 and world == 1
    repeats = 1 if args.quick else args.repeats

    torch.manual_seed(0); g = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8).to(dev)
    torch.manual_seed(0); d = DiscriminatorSmall(8).to(dev)
    tr = GanTrainer(g, d, precision="bf16")
    tr.reducer.broadcast(tr.G.flat); tr.reducer.broadcast(tr.D.flat)

    nb = 4
    host = [synthetic_batch(BATCH_PER_GPU, FRAMES, seed=1000 * rank + i) for i in range(nb)]
    pinned = [tuple(t.pin_memory() for t in b) for b in host]
    devb = [tuple(t.to(dev) for t in b) for b in host]

    # capture (2 eager warm-up steps whose state changes are rolled back, then the capture pass); the launches recorded
    # while the graphs are captured are exactly the launches a replay runs
    c0 = lib.stg_launch_count()
    flop_log_all = []
    ops.flop_log = flop_log_all
    tr.capture(BATCH_PER_GPU, FRAMES, UNIT_DIM, HOP, CHANNELS)
    ops.flop_log = None
    launches_per_step = (lib.stg_launch_count() - c0) // 3
    flop_log = flop_log_all[2 * len(flop_log_all) // 3:]          # the capture pass (the third of three identical passes)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- CPU reference arm first (rank 0, N = 1): its step 0 is the parity gate of the GPU arm's step 0
    cpu, cpu_arm, gate = None, None, None
    if solo and not args.no_cpu_baseline:
        cpu_arm = CpuArm()
        ref_losses = cpu_arm.first_step(host[0])
        tr.step_graph(*devb[0]); tr.flush()
        mine = tr.losses()
        gate = {"against": f"CPU {cpu_arm.kind} arm, same seed-0 weights and batch, step 0", "tolerance": GATE_TOL, "losses": {}}
        for k in ("loss_d", "loss_g", "loss_adv", "loss_td", "loss_fm"):
            rel = abs(mine[k] - ref_losses[k]) / max(1.0, abs(ref_losses[k]))
            gate["losses"][k] = {"ours": round(mine[k], 5), "reference": round(ref_losses[k], 5), "rel": round(rel, 6)}
            if not rel <= GATE_TOL:
                raise SystemExit(f"bench.py: parity gate FAILED before timing: {k} ours {mine[k]} vs reference {ref_losses[k]}")
        gate["passed"] = True
        r = cpu_arm.timed(2, 0, budget_s=30.0)
        cpu = {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}

    for i in range(max(3, args.warmup)):
        tr.step_graph(*devb[i % nb])
    sampler = ClockSampler(local)
    # ---- timed region 1: device-resident inputs
    sampler.start()
    ms_step, ms_all = timed_region(lambda i: tr.step_graph(*devb[i % nb]), tr.flush, args.steps, repeats, barrier, max_over_ranks)
    # (the last step's deferred all-reduce + generator optimiser belong to the timed region: fn_tail = flush)
    clocks = sampler.stop()
    value = BATCH_PER_GPU * world / (ms_step / 1e3)
    final_losses = tr.losses()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, tr, g, d)

    # ---- timed region 2: end to end (pinned host inputs, loss read back every step)
    for i in range(2):
        tr.step_graph(*pinned[i % nb]); tr.losses()

    def e2e_step(i):
        tr.step_graph(*pinned[i % nb])
        tr.slots.tolist()
    ms_e2e, ms_e2e_all = timed_region(e2e_step, tr.flush, args.steps, repeats, barrier, max_over_ranks)
    h2d = sum(t.numel() * t.element_size() for t in pinned[0])
    e2e = {"value": BATCH_PER_GPU * world / (ms_e2e / 1e3), "unit": "samples/s", "ms_per_step": ms_e2e,
           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": tr.slots.numel() * 4,
           "ms_per_step_all_repeats": [round(x, 4) for x in ms_e2e_all]}

    # ---- generator inference (configs[3]): 30 s utterances, batch 1 per call, round-robin over ranks
    ug = UtteranceGenerator(g, "bf16", trainer=tr)
    su_i, sess_i, _ = synthetic_batch(1, INFER_FRAMES, seed=7 + rank)
    su_d, sess_d = su_i.to(dev), sess_i.to(dev)
    su_p, sess_p = su_i.pin_memory(), sess_i.pin_memory()
    for _ in range(3):
        ug.generate_graph(su_d, sess_d)
    n_utt = max(10, args.steps)
    ms_inf, _ = timed_region(lambda i: ug.generate_graph(su_d, sess_d), lambda: None, n_utt, repeats, barrier, max_over_ranks)
    host_out = torch.empty(1, INFER_FRAMES * HOP, CHANNELS).pin_memory()

    def inf_e2e(i):
        host_out.copy_(ug.generate_graph(su_p, sess_p), non_blocking=True)
        torch.cuda.current_stream().synchronize()
    ms_inf_e2e, _ = timed_region(inf_e2e, lambda: None, n_utt, repeats, barrier, max_over_ranks)
    # throughput mode: 4 utterances of equal length per call (same engine, one captured graph per (batch, frames))
    IB = 4
    su_b, sess_b, _ = synthetic_batch(IB, INFER_FRAMES, seed=70 + rank)
    su_b, sess_b = su_b.to(dev), sess_b.to(dev)
    for _ in range(3):
        ug.generate_graph(su_b, sess_b)
    ms_inf_b, _ = timed_region(lambda i: ug.generate_graph(su_b, sess_b), lambda: None, n_utt, repeats, barrier, max_over_ranks)
    inference = {"workload": "generator-only, 1500 unit frames -> 24000x8 EMG samples per utterance, batch 1, bf16 (configs[3]); "
                             "utterances sharded round-robin over ranks, no collective",
                 "metric": "generator inference utterances/s", "value": world / (ms_inf / 1e3), "unit": "utterances/s",
                 "utterances_per_s": world / (ms_inf / 1e3), "emg_samples_per_s": world * INFER_FRAMES * HOP / (ms_inf / 1e3),
                 "ms_per_utterance": ms_inf,
                 "e2e": {"value": world / (ms_inf_e2e / 1e3), "unit": "utterances/s", "h2d_bytes_per_step": su_p.numel() * 4 + 8,
                         "d2h_bytes_per_step": host_out.numel() * 4},
                 "e2e_utterances_per_s": world / (ms_inf_e2e / 1e3),
                 "roofline": {"bound": "tensor", "achieved": round(G_FWD_GFLOP_PER_FRAME * INFER_FRAMES / ms_inf, 2), "peak": peaks["tflops"],
                              "unit": "TFLOP/s", "frac": round(G_FWD_GFLOP_PER_FRAME * INFER_FRAMES / ms_inf / peaks["tflops"], 4),
                              "flops": "207.1 GFLOP per utterance (SURVEY.md 8d), whole forward pass / device time"},
                 "tensor_frac": round(G_FWD_GFLOP_PER_FRAME * INFER_FRAMES / ms_inf / peaks["tflops"], 4),
                 "batch4": {"utterances_per_s": world * IB / (ms_inf_b / 1e3), "ms_per_call": ms_inf_b,
                            "tensor_frac": round(G_FWD_GFLOP_PER_FRAME * INFER_FRAMES * IB / ms_inf_b / peaks["tflops"], 4)},
                 "cpu_baseline": None}
    if cpu_arm is not None:      # the reference's generate() on the host cores: 1 warm-up + 2 timed 30 s utterances
        cpu_arm.tr.load_generator_state({k: v.cpu() for k, v in g.state_dict().items()})   # the weights the GPU engine serves
        cpu_arm.tr.generate(su_i, sess_i)
        t0 = time.perf_counter()
        for _ in range(2):
            y_cpu = cpu_arm.tr.generate(su_i, sess_i)
        s_utt = (time.perf_counter() - t0) / 2
        y_gpu = ug.generate_graph(su_d, sess_d).float().cpu()
        rel = float((y_gpu - y_cpu).norm() / y_cpu.norm())
        if not rel <= GATE_TOL:
            raise SystemExit(f"bench.py: inference parity gate FAILED: rel-L2 {rel} of the 30 s utterance vs the CPU {cpu_arm.kind} arm")
        inference["cpu_baseline"] = {"value": 1.0 / s_utt, "unit": "utterances/s", "cores": cpu_arm.cores, "kind": cpu_arm.kind,
                                     "sample": "2 timed calls of generate() on one 1500-frame utterance (fp32)"}
        inference["parity_rel_l2_vs_cpu"] = round(rel, 6)

    # ---- configs[4]: discriminator stacks + TD / FM / LSGAN losses in isolation, fwd + bwd, batch sweep (N = 1 only)
    disc_losses = None
    if solo and not args.quick:
        disc_losses = disc_losses_sweep(torch, tr, dev, peaks, cpu_arm is not None, DiscriminatorSmall, Discriminator, GanTrainer,
                                        EMGGeneratorGanTTS, synthetic_batch, timed_region, barrier)

    def roofline_block():
        """Instrumentation runs AFTER every timed region of this library (CUPTI stays out of the measurements)."""
        # ---- roofline of the timed schedule: CUPTI timeline of replays of the SAME graphs + the FLOPs recorded at capture
        roofline = None
        timeline, span = cupti_by_kernel(lambda: tr.step_graph(*devb[0]), 3)
        tr.flush(); torch.cuda.synchronize()
        # "alone": every distinct conv / wgrad launch of the timed schedule (one eager step with the same batching records the
        # descriptors), replayed 10x back to back in its own CUDA graph - the kernel by itself on the chip, no launch gaps,
        # its operands L2-warm; time per step = sum over launches of (replay time of its shape)
        tr.step(*devb[0])
        ops.profile = []
        tr.step(*devb[1])
        torch.cuda.synchronize()
        prof, ops.profile = ops.profile, None
        if rank == 0:
            kname = {("tcgen05", "fwd"): "conv_tc_kernel", ("tcgen05", "dgrad"): "conv_tc_kernel", ("tcgen05", "wgrad"): "wgrad_tc_kernel",
                     ("simt", "fwd"): "conv_simt_kernel", ("simt", "dgrad"): "conv_simt_kernel", ("simt", "wgrad"): "wgrad_simt_kernel",
                     ("matvec", "fwd"): "c1_fwd_kernel", ("matvec", "dgrad"): "c1_dgrad_kernel", ("matvec", "wgrad"): "c1_wgrad_kernel"}
            sched = {}
            for p in flop_log:                       # what the timed graphs launch
                a = sched.setdefault(kname[(p["engine"], p["kind"])], dict(launches=0, flops=0.0, bytes=0.0))
                a["launches"] += 1; a["flops"] += p["flops"]; a["bytes"] += p["bytes"]
            alone, replay_us = {}, {}
            st = torch.cuda.Stream()
            for p in prof:
                key = (p["kind"], p["engine"], p["shape"])
                if key not in replay_us:
                    fn = getattr(lib, p["fn"])
                    with torch.cuda.stream(st):
                        gr = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(gr, stream=st):
                            for _ in range(10):
                                fn(ctypes.byref(p["desc"]), ctypes.c_void_p(st.cuda_stream))
                        gr.replay(); torch.cuda.synchronize()
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record(st); gr.replay(); e1.record(st); torch.cuda.synchronize()
                    replay_us[key] = e0.elapsed_time(e1) * 1e3 / 10
                a = alone.setdefault(kname[(p["engine"], p["kind"])], dict(launches=0, ms=0.0, flops=0.0))
                a["launches"] += 1; a["ms"] += replay_us[key] * 1e-3; a["flops"] += p["flops"]
            by_kernel = []
            for k, a in sched.items():
                row = {"kernel": k, "launches_per_step": a["launches"], "gflop_per_step": round(a["flops"] / 1e9, 2),
                       "algorithmic_mb_per_step": round(a["bytes"] / 1e6, 1)}
                if timeline and k in timeline:
                    n_tl, us = timeline[k]
                    row.update(timeline_launches_per_step=round(n_tl, 1), busy_us_per_step=round(us, 1),
                               tflops=round(a["flops"] / (us * 1e-6) / 1e12, 2))
                if k in alone:
                    row["alone_tflops"] = round(alone[k]["flops"] / (alone[k]["ms"] * 1e-3) / 1e12, 2)
                    row["alone_ms_per_step"] = round(alone[k]["ms"], 4)
                by_kernel.append(row)
            by_kernel.sort(key=lambda x: -x.get("busy_us_per_step", x.get("alone_ms_per_step", 0) * 1e3))
            traffic = None
            tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")   # written from the ncu --set full capture
            if os.path.exists(tp):
                with open(tp) as f:
                    traffic = json.load(f).get("conv_tc_kernel")
            top = next((r_ for r_ in by_kernel if r_["kernel"] == "conv_tc_kernel"), by_kernel[0])
            if "tflops" in top:
                achieved, timing = top["tflops"], ("CUPTI activity timeline of 3 replays of the timed CUDA graphs (torch.profiler, outside the timed "
                                                   "regions): busy time of every launch of the kernel as scheduled, concurrent streams included")
                avg_us = top["busy_us_per_step"] / top["launches_per_step"]
            else:
                achieved, timing = top.get("alone_tflops"), f"{span}; fell back to the stand-alone graph replay of every launch"
                avg_us = 1e3 * top.get("alone_ms_per_step", 0.0) / max(1, top["launches_per_step"])
            # HBM-bound kernels of the same timeline: algorithmic bytes / busy time vs the measured copy bandwidth
            hbm = []
            if timeline:
                v_g = sum(m.weight_v.numel() for m in tr.g_plan.wn); v_d = sum(m.weight_v.numel() for m in tr.d_plan.wn)
                pk = tr.g_plan._packs.numel() * 2 + tr.d_plan._packs.numel() * 2
                n_par = tr.G.numel + tr.D.numel
                fm_elems = sum(a.numel() for fm in tr._last_g_fmaps[0] for a in fm[:-1])
                alg = {"wn_fold_rows_kernel": ((v_g + v_d) * 4 + pk, "v fp32 read + bf16 pack written, G + D once per step"),
                       "wn_bwd_multi_kernel": ((tr.g_plan.arena.numel() + tr.d_plan.arena.numel() + 2 * (v_g + v_d)) * 4,
                                               "dw arena + v read, dv written (fp32), G + D"),
                       "adamw_kernel": (n_par * 28, "p, g, m, v read + p, m, v written (fp32), G + D"),
                       "l1_mean_multi_kernel": (fm_elems * 3 * 2, "27 fake + real feature maps read, sign gradient written (bf16)")}
                for k, (nbytes, what) in alg.items():
                    if k in timeline and timeline[k][1] > 0:
                        gbs = nbytes / (timeline[k][1] * 1e-6) / 1e9
                        hbm.append({"kernel": k, "launches_per_step": round(timeline[k][0], 1), "algorithmic_mb_per_step": round(nbytes / 1e6, 1),
                                    "busy_us_per_step": round(timeline[k][1], 1), "achieved_gbs": round(gbs, 1), "peak_gbs": peaks["hbm"],
                                    "frac": round(gbs / peaks["hbm"], 4), "bytes": what})
            roofline = {"bound": "tensor", "kernel": top["kernel"], "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s",
                        "frac": round(achieved / peaks["tflops"], 4) if achieved else None, "traffic": traffic,
                        "peak_source": peaks["source"], "timing": timing,
                        "launches_per_step": top["launches_per_step"], "avg_launch_us": round(avg_us, 2),
                        "algorithmic_gflop_per_launch": round(top["gflop_per_step"] / top["launches_per_step"], 3),
                        "algorithmic_bytes_per_launch": int(top["algorithmic_mb_per_step"] * 1e6 / top["launches_per_step"]),
                        "flops_accounting": "2*B*T_out*C_out*k*C_in/groups with the MODULE's groups (redundant MMAs of merged pack groups are not work)",
                        "alone": {"tflops": top.get("alone_tflops"), "frac": round(top["alone_tflops"] / peaks["tflops"], 4) if top.get("alone_tflops") else None,
                                  "timing": "every distinct launch of the timed schedule replayed 10x back to back in its own CUDA graph (kernel alone on the chip, L2-warm), summed over the step's launches"},
                        "timeline_span_us_per_step": round(span, 1) if isinstance(span, float) else None,
                        "step_tflops": round(STEP_GFLOP_PER_SAMPLE * BATCH_PER_GPU / ms_step, 2),
                        "step_frac": round(STEP_GFLOP_PER_SAMPLE * BATCH_PER_GPU / ms_step / peaks["tflops"], 4),
                        "by_kernel": by_kernel, "hbm": hbm,
                        "timeline_top": [{"kernel": k, "launches_per_step": round(v[0], 1), "busy_us_per_step": round(v[1], 1)}
                                         for k, v in sorted((timeline or {}).items(), key=lambda kv: -kv[1][1])[:16]]}
        return roofline

    roofline = roofline_block()

    # ---- the train step WITH the EMG-encoder perceptual losses (train.py:219-230; SURVEY.md 8f rank 1): random-init frozen
    # 768-d encoder (no checkpoint ships with the reference), same batch shape; + 35.0 GFLOP per sample (encoder forward +
    # input gradient: 4 ResBlocks 8.6 + 6 transformer layers 8.9 GFLOP forward)
    encoder_step = None
    if solo and not args.quick:
        from ste_gan_b200.models.emg_encoder import EMGEncoderTransformer
        torch.manual_seed(0); g2 = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8).to(dev)
        torch.manual_seed(0); d2 = DiscriminatorSmall(8).to(dev)
        torch.manual_seed(0); enc = EMGEncoderTransformer(8, 256, 48).eval().to(dev)
        tr2 = GanTrainer(g2, d2, precision="bf16", emg_encoder=enc)
        tr2.capture(BATCH_PER_GPU, FRAMES, UNIT_DIM, HOP, CHANNELS)
        ph = torch.randint(0, 48, (BATCH_PER_GPU, FRAMES), generator=torch.Generator().manual_seed(3)).to(dev)
        for i in range(3):
            tr2.step_graph(*devb[i % nb], phoneme_targets=ph)
        ms_enc, _ = timed_region(lambda i: tr2.step_graph(*devb[i % nb], phoneme_targets=ph), tr2.flush, 30, 3, barrier, max_over_ranks)
        L2 = tr2.losses()
        gf = STEP_GFLOP_PER_SAMPLE + 35.0
        encoder_step = {"workload": "configs[1] + speech-unit and phoneme losses through the frozen EMG encoder (768-d, 4 ResBlocks, 6 rel-pos "
                                    "transformer layers; random init), bf16, batch 16",
                        "ms_per_step": round(ms_enc, 4), "value": round(BATCH_PER_GPU / (ms_enc / 1e3), 1), "unit": "samples/s",
                        "roofline": {"bound": "tensor", "achieved": round(gf * BATCH_PER_GPU / ms_enc, 1), "peak": peaks["tflops"],
                                     "unit": "TFLOP/s", "frac": round(gf * BATCH_PER_GPU / ms_enc / peaks["tflops"], 4)},
                        "finite": all(v == v and abs(v) < 1e30 for v in L2.values()),
                        "loss_speech_unit": round(L2["loss_speech_unit"], 4), "loss_phoneme": round(L2["loss_phoneme"], 4)}
        del tr2, g2, d2, enc
        torch.cuda.empty_cache()

    # ---- the same reference step on THIS GPU through torch + cuDNN (BASELINE.md section 5): context, not the target
    context = None
    if solo and not args.quick and not args.no_cpu_baseline:
        context = {"torch_gpu": torch_gpu_context(torch, host, args.torch_compile)}

    if rank == 0:
        line = {"metric": "GAN train samples/s", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config_dict(world), "clocks": clocks,
                "timed_repeats": len(ms_all), "ms_per_step_all_repeats": [round(x, 4) for x in ms_all],
                "e2e": e2e, "gpu_launches": int(launches_per_step * args.steps), "launches_per_step": int(launches_per_step),
                "parity_gate": gate, "roofline": roofline, "cpu_baseline": cpu, "inference": inference, "disc_losses": disc_losses,
                "encoder_step": encoder_step,
                "context": context, "losses_last_step": {k: round(v, 5) for k, v in final_losses.items()}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def disc_losses_sweep(torch, tr_unused, dev, peaks, with_cpu, DiscriminatorSmall, Discriminator, GanTrainer, EMGGeneratorGanTTS,
                      synthetic_batch, timed_region, barrier):
    """BASELINE.json configs[4] (GanTrainer.disc_losses_step): per discriminator family and batch size, one CUDA graph of
    the whole isolated step, device-timed; the CPU baseline per family is measured once on a bounded batch."""
    out = {"workload": "D stacks + multi-TD + FM + LSGAN losses isolated, fwd + bwd incl. D AdamW and the gradient w.r.t. x_pred "
                       "(train.py:189-264 without the generator), bf16, 1600x8 EMG samples per item (configs[4])",
           "metric": "disc+losses samples/s", "unit": "samples/s", "points": []}
    cpu_by_family = {}
    for family, ctor in (("small", DiscriminatorSmall), ("full", Discriminator)):
        if with_cpu:
            from baseline import ref_runner as R
            cb = 4
            ct = R.make_trainer("cpu", small=family == "small")
            _, _, xr = synthetic_batch(cb, FRAMES, seed=5)
            xp = torch.tanh(torch.randn(cb, FRAMES * HOP, CHANNELS, generator=torch.Generator().manual_seed(6)))
            ct.disc_losses_step(xp, xr)
            t0 = time.perf_counter()
            for _ in range(2):
                ct.disc_losses_step(xp, xr)
            s = (time.perf_counter() - t0) / 2
            cpu_by_family[family] = {"value": cb / s, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": ct.kind,
                                     "sample": f"2 timed steps of batch {cb} (fp32); CPU samples/s does not grow with the batch"}
            del ct
        for B in DISC_BATCHES:
            torch.manual_seed(0); g = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8, channels=64).to(dev)   # (unused by this workload)
            torch.manual_seed(0); d = ctor(8).to(dev)
            tr = GanTrainer(g, d, precision="bf16")
            _, _, xr = synthetic_batch(B, FRAMES, seed=11)
            x_real = xr.to(dev)
            x_pred = torch.tanh(torch.randn(B, FRAMES * HOP, CHANNELS, generator=torch.Generator().manual_seed(12))).to(dev)
            side = torch.cuda.Stream(); side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    tr.disc_losses_step(x_pred, x_real)
            torch.cuda.current_stream().wait_stream(side); torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                dx = tr.disc_losses_step(x_pred, x_real)
            for _ in range(3):
                graph.replay()
            ms, _ = timed_region(lambda i: graph.replay(), lambda: None, 30, 3, barrier, lambda x: x)
            tf = DISC_GFLOP_PER_SAMPLE[family] * B / ms
            finite = bool(torch.isfinite(dx).all()) and bool(torch.isfinite(tr.slots).all())
            out["points"].append({"discriminator": family, "batch": B, "ms_per_step": round(ms, 4), "value": round(B / (ms / 1e3), 1),
                                  "roofline": {"bound": "tensor", "achieved": round(tf, 1), "peak": peaks["tflops"], "unit": "TFLOP/s",
                                               "frac": round(tf / peaks["tflops"], 4)},
                                  "cpu_baseline": cpu_by_family.get(family), "finite": finite})
            del graph, tr, g, d, dx
            torch.cuda.empty_cache()
    return out


def torch_gpu_context(torch, host, with_compile: bool):
    """The reference step (reference modules when installed, else the oracle port) on THIS GPU through the container's
    torch + cuDNN: fp32, bf16 autocast and the reference's own AMP mode (fp16 autocast + GradScaler, train.py:151,181);
    torch.compile (train.py:140-146) only with --torch-compile (its compile time does not fit the default run)."""
    from baseline import ref_runner as R
    out = {"what": "reference modules (baseline/_ref) or the oracle port, torch " + torch.__version__ + " + cuDNN " +
                   str(torch.backends.cudnn.version()) + ", eager, cudnn.benchmark, batch 16 x 100 frames; samples/s"}
    variants = [("eager_fp32", None, False), ("eager_bf16_autocast", torch.bfloat16, False), ("eager_fp16_amp_gradscaler", torch.float16, False)]
    if with_compile:
        variants.append(("compile_bf16_autocast", torch.bfloat16, True))
    for name, amp, comp in variants:
        try:
            t = R.make_trainer("cuda", small=True, amp=amp, compile_=comp)
            batches = [tuple(x.cuda() for x in b) for b in host]
            for i in range(4):
                t.step(*batches[i % len(batches)])
            s = R.time_steps(lambda: t.step(*batches[0]), 10, "cuda")
            out[name] = {"value": round(BATCH_PER_GPU / s, 1), "unit": "samples/s", "ms_per_step": round(1e3 * s, 3), "kind": t.kind}
            del t
            torch.cuda.empty_cache()
        except Exception as exc:      # noqa: BLE001 - context only: a failing library arm must not take the bench line down
            out[name] = {"unavailable": repr(exc)[:200]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=1,
                    help="timed regions the --steps steps are split into; the median of their ms per step is reported")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--torch-compile", action="store_true", help="also time the reference step under torch.compile on the GPU")
    ap.add_argument("--quick", action="store_true", help="train + inference lines only, one timed region")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed train step computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.repeats < 1:
        ap.error("--steps and --repeats must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU train step; --impl reference does not run it")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
