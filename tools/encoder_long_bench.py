"""Throughput of the frozen full-size EMG encoder (768-d, 6 layers, 8 heads of 96, random seed-0 init, bf16) from the train-step
lengths to 30 s utterances, and the band-tiled against the one-CTA-per-head attention kernels where both run.  Prints one JSON
line and writes it to --out.

    python tools/encoder_long_bench.py [--out profiles/r4_encoder_long.json] [--seconds 1.0]

  encoder     (B, EMG samples) in {(16, 1600), (16, 2048), (8, 4096), (1, 24000), (8, 24000)}: forward only (no saved context)
              and forward + input gradient of both perceptual losses (passes_encoder.encoder_losses), each captured in a CUDA
              graph and replayed warm, >= --seconds of timed replays per round, 3 rounds (median); which attention kernels ran
  profile     a separate torch.profiler run of the eager calls: the attention kernels' share of the device kernel time
  kernels     attention alone at B = 16, H = 8, d = 96, L = 100 / 128, bf16: the dense and the band kernels, forward and
              backward, CUDA events over repeated launches (the operands, < 10 MB, stay in L2 between launches)

The GPU name and power limit are read in the same run: every number here is for that card.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from ste_gan_b200 import ops                                   # noqa: E402
from ste_gan_b200 import passes_encoder as pe                  # noqa: E402
from ste_gan_b200.models.emg_encoder import EMGEncoderTransformer   # noqa: E402
from tools.serve_bench import gpu_info                         # noqa: E402

POINTS = [(16, 1600), (16, 2048), (8, 4096), (1, 24000), (8, 24000)]


def _events_ms(fn, n: int) -> float:
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def time_call(fn, seconds: float, rounds: int = 3) -> dict:
    """ms per call: warm-up, then `rounds` rounds of enough calls for >= `seconds` of timed work each; median round."""
    for _ in range(3):
        fn()
    est = _events_ms(fn, 3)
    n = max(10, math.ceil(seconds * 1e3 / max(est, 1e-3)))
    ms = sorted(_events_ms(fn, n) for _ in range(rounds))
    return {"ms_per_call": round(ms[rounds // 2], 4), "rounds_ms": [round(v, 4) for v in ms], "calls_per_round": n}


def graphed(fn):
    """fn captured in a CUDA graph (after two eager warm-up calls) -> the graph's replay."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g.replay


def attention_share(fn) -> dict:
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
    tot = attn = 0.0
    per_kernel = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if ev.key.startswith(("cudaLaunch", "cudaGraph", "cudaMemcpy", "cudaStream", "cudaEvent", "cudaFunc")):
            continue
        tot += t
        if "relattn" in ev.key:
            attn += t
            name = next(n for n in ev.key.replace("<", " ").replace("(", " ").replace("::", " ").split() if "relattn" in n)
            per_kernel[name] = per_kernel.get(name, 0.0) + t / 3
    return {"attention_share": round(attn / tot, 4) if tot else None, "attention_us_per_call": round(attn / 3, 1),
            "kernels_us_per_call": round(tot / 3, 1), "attention_us_per_call_by_kernel": {k: round(v, 1) for k, v in per_kernel.items()}}


def encoder_points(seconds: float) -> list:
    torch.manual_seed(0)
    enc = EMGEncoderTransformer(8, 256, 48).eval().cuda()
    plan = enc.plan(torch.bfloat16)
    d = 768 // 8
    out = []
    for B, T in POINTS:
        g = torch.Generator().manual_seed(T + B)
        L = T // 16
        x = torch.tanh(torch.randn(B, T, 8, generator=g)).cuda()
        ut, ph = torch.randn(B, L, 256, generator=g).cuda(), torch.randint(0, 48, (B, L), generator=g).cuda()
        slots = torch.zeros(2, device="cuda")
        fwd = lambda: pe.encoder_forward(plan, x, need_ctx=False)
        both = lambda: pe.encoder_losses(plan, x, ut, ph, slots)
        row = {"B": B, "emg_samples": T, "frames": L,
               "attention_forward_only": "dense" if ops.relattn_dense_supported(L, d, False) else "band",
               "attention_with_gradient": "dense" if ops.relattn_dense_supported(L, d, True) else "band"}
        for name, fn in (("forward", fwd), ("forward_and_input_gradient", both)):
            r = time_call(graphed(fn), seconds)
            r["utterances_per_s"] = round(B * 1e3 / r["ms_per_call"], 1)
            r.update(attention_share(fn))
            row[name] = r
            torch.cuda.synchronize()
        out.append(row)
        print(f"encoder B={B} T={T} done", file=sys.stderr, flush=True)
        torch.cuda.empty_cache()
    return out


def kernel_points(seconds: float) -> list:
    B, H, d, M = 16, 8, 96, 100
    out = []
    for L in (100, 128):
        g = torch.Generator().manual_seed(L)
        qkv = torch.randn(B, L, 3 * H * d, generator=g).cuda().to(torch.bfloat16)
        do = torch.randn(B, L, H * d, generator=g).cuda().to(torch.bfloat16)
        emb = (torch.randn(H, 2 * M - 1, d, generator=g) * d ** -0.5).cuda()
        o_d, p_d = ops.relattn_fwd(qkv, emb, H, M)
        o_b, p_b = ops.relattn_band_fwd(qkv, emb, H, M)
        dq_d = ops.relattn_bwd(qkv, emb, p_d, do, H, M)
        dq_b = ops.relattn_band_bwd(qkv, emb, p_b, do, H, M)
        rel = lambda a, b: float((a.float() - b.float()).norm() / b.float().norm())
        row = {"B": B, "H": H, "d": d, "L": L, "dtype": "bf16", "o_rel_diff": rel(o_b, o_d), "dqkv_rel_diff": rel(dq_b, dq_d)}
        for name, fn in (("dense_forward", lambda: ops.relattn_fwd(qkv, emb, H, M)),
                         ("band_forward", lambda: ops.relattn_band_fwd(qkv, emb, H, M)),
                         ("dense_backward", lambda: ops.relattn_bwd(qkv, emb, p_d, do, H, M)),
                         ("band_backward", lambda: ops.relattn_band_bwd(qkv, emb, p_b, do, H, M))):
            row[name] = time_call(fn, seconds)
        row["band_over_dense_forward"] = round(row["band_forward"]["ms_per_call"] / row["dense_forward"]["ms_per_call"], 3)
        row["band_over_dense_backward"] = round(row["band_backward"]["ms_per_call"] / row["dense_backward"]["ms_per_call"], 3)
        out.append(row)
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r4_encoder_long.json"))
    ap.add_argument("--seconds", type=float, default=1.0)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("encoder_long_bench.py: needs a CUDA device")
    line = {"metric": "frozen EMG encoder ms per call / utterances per s (full size, bf16, CUDA-graph replay, warm)",
            "gpu": gpu_info(), "encoder": encoder_points(a.seconds), "attention_kernels": kernel_points(a.seconds)}
    s = json.dumps(line)
    print(s, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
