"""Serving benchmark of UtteranceGenerator: the cost of the length masks and serve() against serve_batched() on a
mixed-length request list.  Prints one JSON line.

    python tools/serve_bench.py [--n 512] [--reps 7] [--sweep]

  mask_overhead  generate_graph with and without lengths at bench.py's batch-4 inference shape (4 x 1500 frames, every
                 length = 1500), alternating the two in `reps` rounds of `calls` replays; ms per call of each
  mixed          seed 0, n utterances of 100..1500 frames (uniform; 2-30 s of 16 kHz EMG at 16 samples per frame), full-size
                 seed-0 generator, bf16: serve() and serve_batched() from a fresh engine (graph captures included), then
                 serve_batched() again once every bucket's graph is resident (max_graphs = number of buckets)
  parity         before any timing: serve_batched against serve on every 16th utterance (rel-L2 <= 1e-2, bf16)
  sweep          (--sweep) warm serve_batched for other batch sizes and bucket ladders

The GPU name and power limit are read in the same run: every number here is for that card.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import ste_gan_oracle as O   # noqa: E402
from ste_gan_b200 import inference       # noqa: E402
from ste_gan_b200.inference import UtteranceGenerator, bucket_frames   # noqa: E402
from ste_gan_b200.models.generator import EMGGeneratorGanTTS   # noqa: E402

HOP = 16


def gpu_info() -> dict:
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        pl, clk = [v.strip() for v in r.stdout.strip().split(",")]
        info.update(power_limit_w=float(pl), sm_max_mhz=float(clk))
    except Exception as e:   # noqa: BLE001 - the numbers are still valid, only unlabelled
        info.update(power_limit_w=None, note=f"nvidia-smi unavailable: {e}")
    return info


def counting(ug: UtteranceGenerator) -> UtteranceGenerator:
    """Count the graph captures of an engine (ug.n_captures)."""
    ug.n_captures = 0
    cap = ug.capture

    def wrapped(*a, **kw):
        ug.n_captures += 1
        return cap(*a, **kw)
    ug.capture = wrapped
    return ug


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def _paired(runs: dict, reps: int, calls: int) -> dict:
    """ms per call of the two runs in `reps` rounds; each round times A B B A (or B A A B, alternating), so an order or
    drift effect cancels in the per-round difference."""
    (ka, fa), (kb, fb) = runs.items()
    ms = {ka: [], kb: []}
    diff = []
    for r in range(reps):
        order = [ka, kb, kb, ka] if r % 2 == 0 else [kb, ka, ka, kb]
        t = {ka: 0.0, kb: 0.0}
        for k in order:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(calls):
                runs[k]()
            e1.record()
            e1.synchronize()
            t[k] += e0.elapsed_time(e1) / (2 * calls)
        for k in t:
            ms[k].append(round(t[k], 4))
        diff.append(round(t[kb] / t[ka] - 1.0, 4))
    med = {k: sorted(v)[len(v) // 2] for k, v in ms.items()}
    ds = sorted(diff)
    return {"ms_per_call": ms, "median_ms": med, f"{kb}_over_{ka}_per_round": diff, "median_diff": ds[len(ds) // 2],
            "diff_range": [ds[0], ds[-1]]}


def mask_overhead(g, reps: int, calls: int) -> dict:
    """generate_graph with / without lengths (what a caller pays: the masked call also copies the lengths into the graph's
    buffer), and the two captured graphs replayed bare (the kernels alone)."""
    ug = UtteranceGenerator(g, "bf16")
    su, sess, _ = O.synthetic_batch(4, 1500, seed=34)
    su, sess = su.cuda(), sess.cuda()
    lens = torch.full((4,), 1500, dtype=torch.int32, device="cuda")
    y0 = ug.generate_graph(su, sess).clone()
    y1 = ug.generate_graph(su, sess, lengths=lens).clone()
    same = bool(torch.equal(y0, y1))      # nothing masked: the masked graph computes the same bits
    calls_ = {"unmasked": lambda: ug.generate_graph(su, sess), "masked": lambda: ug.generate_graph(su, sess, lengths=lens)}
    g0, g1 = ug._graphs[(4, 1500)][0], ug._graphs[(4, 1500, True)][0]
    replays = {"unmasked": g0.replay, "masked": g1.replay}
    for f in list(calls_.values()) + list(replays.values()):
        for _ in range(3):
            f()
    return {"shape": "B=4, T=1500 frames (24000 x 8 EMG samples each), bf16, every length = T", "calls_per_timing": calls,
            "rounds": reps, "order": "ABBA / BAAB alternating", "generate_graph": _paired(calls_, reps, calls),
            "graph_replay_only": _paired(replays, reps, calls), "identical_outputs": same}


def run_serve(g, utts, kind: str, max_batch: int = 8, max_graphs: int = 8, warm: bool = False, per_octave=None,
              warm_reps: int = 5) -> dict:
    ug = counting(UtteranceGenerator(g, "bf16", max_graphs=max_graphs))
    po = inference.BUCKETS_PER_OCTAVE if per_octave is None else per_octave
    lens = [int(u[0].shape[0]) for u in utts]
    if warm:
        ug.serve_batched(utts, max_batch=max_batch, per_octave=po)
        ug.n_captures = 0
    torch.cuda.reset_peak_memory_stats()
    fn = (lambda: ug.serve(utts)) if kind == "serve" else (lambda: ug.serve_batched(utts, max_batch=max_batch, per_octave=po))
    runs = [timed(fn) for _ in range(warm_reps if warm else 1)]     # a warm pass is short: median of several
    secs, out = sorted(runs, key=lambda r: r[0])[len(runs) // 2]
    plan = inference.plan_batches(lens, max_batch, po)
    rows = sum(lens)
    computed = rows if kind == "serve" else sum(max_batch * T for T, _ in plan)
    res = {"seconds": round(secs, 3), "timed_passes": len(runs), "utterances_per_s": round(len(utts) / secs, 1),
           "emg_samples_per_s": round(rows * HOP / secs, 0), "padded_rows_fraction": round(1.0 - rows / computed, 4),
           "graphs_captured": ug.n_captures, "peak_allocated_gb": round(torch.cuda.max_memory_allocated() / 1e9, 2),
           "peak_reserved_gb": round(torch.cuda.max_memory_reserved() / 1e9, 2)}
    if kind != "serve":
        res.update(max_batch=max_batch, batches=len(plan), buckets=len({T for T, _ in plan}), max_graphs=max_graphs)
    del ug
    torch.cuda.empty_cache()
    return res, out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--calls", type=int, default=100)
    ap.add_argument("--sweep", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("serve_bench.py: needs a CUDA device")
    torch.manual_seed(0)
    g = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8).cuda()
    gen = torch.Generator().manual_seed(0)
    lens = torch.randint(100, 1501, (a.n,), generator=gen).tolist()
    utts = [(torch.randn(L, 256, generator=gen), torch.randint(0, 17, (), generator=gen)) for L in lens]
    n_buckets = len({bucket_frames(L) for L in lens})
    line = {"metric": "mixed-length serving utterances/s (serve_batched, warm)", "gpu": gpu_info(),
            "workload": f"{a.n} utterances, 100..1500 unit frames uniform (seed 0), full-size seed-0 generator, bf16"}

    # parity gate first: serve_batched vs serve on a sample
    sample = utts[::16]
    ref = UtteranceGenerator(g, "bf16", max_graphs=4).serve(sample)
    got = UtteranceGenerator(g, "bf16", max_graphs=4).serve_batched(sample)
    worst = max(O.rel_l2(got[i], ref[i]) for i in ref)
    line["parity"] = {"utterances": len(sample), "worst_rel_l2_vs_serve": worst, "tolerance": 1e-2, "ok": worst <= 1e-2}
    if not line["parity"]["ok"]:
        print(json.dumps(line), flush=True)
        raise SystemExit(f"serve_bench.py: parity gate FAILED (rel-L2 {worst})")

    line["mask_overhead"] = mask_overhead(g, a.reps, a.calls)
    print("mask overhead done", file=sys.stderr, flush=True)
    mixed = {}
    mixed["serve_cold"], _ = run_serve(g, utts, "serve")
    print("serve done", file=sys.stderr, flush=True)
    mixed["serve_batched_cold"], _ = run_serve(g, utts, "batched")
    mixed["serve_batched_warm"], _ = run_serve(g, utts, "batched", max_graphs=n_buckets, warm=True)
    line["mixed"] = mixed
    line["value"] = mixed["serve_batched_warm"]["utterances_per_s"]
    line["unit"] = "utterances/s"
    line["speedup_cold"] = round(mixed["serve_cold"]["seconds"] / mixed["serve_batched_cold"]["seconds"], 2)
    if a.sweep:
        sweep = []
        for mb, po in ((4, 4), (8, 4), (16, 4), (32, 4), (8, 2), (8, 8), (16, 8)):
            nb = len({bucket_frames(L, po) for L in lens})
            r, _ = run_serve(g, utts, "batched", max_batch=mb, max_graphs=nb, warm=True, per_octave=po)
            sweep.append(dict(r, buckets_per_octave=po))
            print(f"sweep {mb} {po} done", file=sys.stderr, flush=True)
        line["sweep_warm"] = sweep
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
