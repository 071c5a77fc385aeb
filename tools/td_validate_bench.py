"""Time-domain validation benchmark: the per-utterance TD score kernel (stg_td_scores) alone, and validate_batched with and
without real_emg against the per-utterance pattern.  Prints one JSON line and writes it to --out.

    python tools/td_validate_bench.py [--n 512] [--rounds 3] [--reps 7] [--calls 200] [--out profiles/r6_td_validate_bench.json]

  td_kernel   ops.td_scores at 8 x 24000 x 8 and 16 x 1600 x 8 fp32 (every sample full length, the three default resolutions),
              one captured graph replayed `calls` times per timing, alternated with stg_td_loss_ex (the whole-batch forward of
              the train step's loss, for scale) in `reps` ABBA rounds; CUDA events, ms per call.  The inputs (12 MB at
              8 x 24000) stay in the 126 MB L2 between replays, so these are warm-L2 times.
  validation  seed 0, n utterances of 100..1500 frames (uniform), full-size seed-0 generator, full-size random-init encoder,
              random tanh real EMG, bf16.  Three forms of validate_batched: "encoder" (no real_emg), "encoder_td" (real_emg
              with an encoder), "td" (real_emg, no encoder).  Each round runs every form from cold (a fresh engine, graph
              captures included) and warm (every bucket's graph resident, median of 3 passes), the order of the forms
              rotating between rounds.
  per_utterance_td   the pattern without batching, once, cold: serve() (one graph per length, EMG to the host) followed by
                     MultiTimeDomainFeatureLoss on each utterance at batch 1.
  parity      before any timing: the "td" form against the per-utterance pattern on every 16th utterance.

The GPU name and power limit are read in the same run: every number here is for that card.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from serve_bench import _paired, gpu_info, timed   # noqa: E402
from validate_bench import _graph, full_size_encoder   # noqa: E402
from ste_gan_b200 import ops   # noqa: E402
from ste_gan_b200.inference import UtteranceGenerator, bucket_frames   # noqa: E402
from ste_gan_b200.losses.time_domain_loss import _RES, MultiTimeDomainFeatureLoss   # noqa: E402
from ste_gan_b200.models.generator import EMGGeneratorGanTTS   # noqa: E402

HOP = 16


def td_kernel(B: int, T: int, reps: int, calls: int) -> dict:
    g = torch.Generator().manual_seed(T)
    xr, xg = torch.randn(B, T, 8, generator=g).cuda(), torch.tanh(torch.randn(B, T, 8, generator=g)).cuda()
    lens = torch.full((B,), T // HOP, dtype=torch.int32, device="cuda")
    losses = torch.empty(len(_RES), device="cuda")
    g_scores, out = _graph(lambda: ops.td_scores(xr, xg, lens, HOP))
    g_loss, _ = _graph(lambda: ops.td_loss_ex(xr, xg, _RES, losses))
    g_scores.replay()
    torch.cuda.synchronize()
    res = _paired({"td_scores": g_scores.replay, "td_loss_ex": g_loss.replay}, reps, calls)
    ms = res["median_ms"]["td_scores"]
    return dict(shape=f"B={B}, T={T} rows, C=8, fp32, every sample {T} rows, resolutions {_RES}", calls_per_timing=calls,
                rounds=reps, launches=3, input_mb=round(2 * B * T * 8 * 4 / 1e6, 2),
                input_gb_per_s=round(2 * B * T * 8 * 4 / (ms * 1e-3) / 1e9, 1), finite=bool(torch.isfinite(out).all()), **res)


def per_utterance_td(g, utts, real) -> tuple:
    """serve() at each utterance's own length, then MultiTimeDomainFeatureLoss at batch 1."""
    ug = UtteranceGenerator(g, "bf16")
    loss = MultiTimeDomainFeatureLoss(8)

    def run():
        emg = ug.serve([u[:2] for u in utts])
        out = {}
        with torch.no_grad():
            for i, y in emg.items():
                _, parts = loss.time_domain_loss(real[i][None].cuda(), y[None].cuda())
                out[i] = [float(p) for p in parts]
        return out
    secs, out = timed(run)
    del ug
    torch.cuda.empty_cache()
    return {"seconds": round(secs, 3), "utterances_per_s": round(len(utts) / secs, 1)}, out


def validation_pass(g, enc, utts, real, form: str, warm: bool, n_buckets: int) -> tuple:
    ug = UtteranceGenerator(g, "bf16", max_graphs=2 * n_buckets if warm else 8, emg_encoder=enc if form != "td" else None)
    items = [u[:2] for u in utts] if form == "td" else utts
    kw = {} if form == "encoder" else {"real_emg": real}
    fn = lambda: ug.validate_batched(items, **kw)        # noqa: E731
    if warm:
        fn()
    runs = [timed(fn) for _ in range(3 if warm else 1)]
    secs, out = sorted(runs, key=lambda r: r[0])[len(runs) // 2]
    del ug
    torch.cuda.empty_cache()
    return secs, out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_td_validate_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("td_validate_bench.py: needs a CUDA device")
    line = {"metric": "utterances validated per second (validate_batched with real_emg, no encoder, warm)", "gpu": gpu_info()}
    line["td_kernel"] = [td_kernel(8, 24000, a.reps, max(1, a.calls // 4)), td_kernel(16, 1600, a.reps, a.calls)]
    print("kernel done", file=sys.stderr, flush=True)

    enc = full_size_encoder()
    torch.manual_seed(0)
    g = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8).cuda()
    gen = torch.Generator().manual_seed(0)
    lens = torch.randint(100, 1501, (a.n,), generator=gen).tolist()
    utts = [(torch.randn(L, 256, generator=gen), torch.randint(0, 17, (), generator=gen), torch.randn(L, 256, generator=gen),
             torch.randint(0, 48, (L,), generator=gen)) for L in lens]
    real = [torch.tanh(torch.randn(HOP * L, 8, generator=gen)) for L in lens]
    n_buckets = len({bucket_frames(L) for L in lens})
    line["workload"] = (f"{a.n} utterances, 100..1500 frames uniform (seed 0), full-size seed-0 generator + full-size encoder, "
                        "bf16, random targets and tanh real EMG")

    idx = list(range(0, a.n, 16))                        # parity first
    _, ref = per_utterance_td(g, [utts[i] for i in idx], [real[i] for i in idx])
    _, got = validation_pass(g, enc, [utts[i] for i in idx], [real[i] for i in idx], "td", False, n_buckets)
    worst = max(abs(v / m - 1) for j in ref for v, m in zip(got[j].td.values, ref[j]))
    line["parity"] = {"utterances": len(idx), "worst_rel_diff_vs_per_utterance": worst, "tolerance": 2e-2, "ok": worst <= 2e-2}

    forms = ["encoder", "encoder_td", "td"]
    secs = {f"{f}_{w}": [] for f in forms for w in ("cold", "warm")}
    for r in range(a.rounds):
        for f in forms[r % 3:] + forms[:r % 3]:
            for warm in (False, True):
                s, _ = validation_pass(g, enc, utts, real, f, warm, n_buckets)
                secs[f"{f}_{'warm' if warm else 'cold'}"].append(round(s, 3))
        print(f"round {r} done", file=sys.stderr, flush=True)
    v = {k: {"seconds": s, "median_s": statistics.median(s), "utterances_per_s": round(a.n / statistics.median(s), 1)}
         for k, s in secs.items()}
    v["per_utterance_td_cold"], _ = per_utterance_td(g, utts, real)
    line["validation"] = v
    line["td_share_warm"] = round(1 - v["encoder_warm"]["median_s"] / v["encoder_td_warm"]["median_s"], 4)
    line["value"] = v["td_warm"]["utterances_per_s"]
    line["unit"] = "utterances/s"
    line["speedup_cold_vs_per_utterance"] = round(v["per_utterance_td_cold"]["seconds"] / v["td_cold"]["median_s"], 2)
    s = json.dumps(line)
    print(s, flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
