"""Validation benchmark: the cost of the encoder's length masks, and scoring generated utterances with the frozen EMG encoder
one utterance at a time against UtteranceGenerator.validate_batched().  Prints one JSON line and writes it to --out.

    python tools/validate_bench.py [--n 512] [--reps 7] [--calls 20] [--out profiles/r5_validate_bench.json]

  encoder_mask_cost  full-size random-init encoder, bf16, forward only: captured graphs of encoder_forward without lengths and
                     with every length = T, at 16 x 1600 EMG samples (100 frames: the dense attention route) and 8 x 24000
                     (1500 frames: the band route), alternating the two in `reps` rounds of `calls` replays (ms per call);
                     the two graphs' outputs must be bit-identical
  validation         seed 0, n utterances of 100..1500 frames (uniform), full-size seed-0 generator + the encoder above, bf16:
                     per_utterance_loop  generate_graph at the utterance's own length (one graph per length, as serve()),
                                         then encoder_scores at that length, eager
                     validate_batched    from a fresh engine (graph captures included), then again with every bucket's graph
                                         resident (max_graphs = number of buckets); reserved_gb_per_resident_graph
                                         is the reserved memory the timed pass added per resident graph, so it is
                                         meaningful from cold only (warm: the graphs were resident before)
  parity            before any timing: validate_batched against the per-utterance loop on every 16th utterance

The GPU name and power limit are read in the same run: every number here is for that card.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from serve_bench import _paired, gpu_info, timed   # noqa: E402
from ste_gan_b200 import inference, ops, passes_encoder as pe   # noqa: E402
from ste_gan_b200.inference import EncoderScore, UtteranceGenerator, bucket_frames   # noqa: E402
from ste_gan_b200.models.emg_encoder import EMGEncoderTransformer   # noqa: E402
from ste_gan_b200.models.generator import EMGGeneratorGanTTS   # noqa: E402

HOP = 16


def full_size_encoder():
    """768-d, 6 layers, 8 heads of 96 (the train step's configuration), seed-0 random init with non-trivial BatchNorm statistics
    (no trained checkpoint ships with the reference)."""
    torch.manual_seed(0)
    enc = EMGEncoderTransformer(8, 256, 48).eval()
    g = torch.Generator().manual_seed(5)
    for mod in enc.modules():
        if isinstance(mod, torch.nn.BatchNorm1d):
            mod.running_mean.normal_(0, 0.3, generator=g); mod.running_var.uniform_(0.5, 1.5, generator=g)
            mod.weight.data.uniform_(0.5, 1.5, generator=g); mod.bias.data.normal_(0, 0.2, generator=g)
    return enc.cuda()


def _graph(fn):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fn()
    return g, out


def encoder_mask_cost(enc, B: int, T: int, reps: int, calls: int) -> dict:
    plan = enc.plan(torch.bfloat16)
    x = torch.tanh(torch.randn(B, T, 8, generator=torch.Generator().manual_seed(T))).cuda()
    lens = torch.full((B,), T // plan.frame_rows, dtype=torch.int32, device="cuda")
    g0, (u0, l0, _) = _graph(lambda: pe.encoder_forward(plan, x, need_ctx=False))
    g1, (u1, l1, _) = _graph(lambda: pe.encoder_forward(plan, x, need_ctx=False, lengths=lens))
    g0.replay(); g1.replay()
    torch.cuda.synchronize()
    same = bool(torch.equal(u0, u1) and torch.equal(l0, l1))
    res = _paired({"unmasked": g0.replay, "masked": g1.replay}, reps, calls)
    route = "dense" if ops.relattn_dense_supported(T // plan.frame_rows, 96, False) else "band"
    del g0, g1
    torch.cuda.empty_cache()
    return dict(shape=f"B={B}, T={T} EMG samples ({T // plan.frame_rows} frames), bf16, every length = T", attention=route,
                calls_per_timing=calls, rounds=reps, order="ABBA / BAAB alternating", identical_outputs=same, **res)


def counting(ug: UtteranceGenerator) -> UtteranceGenerator:
    """Count every graph capture of an engine (ug.n_captures): generator graphs and validation graphs."""
    ug.n_captures = 0
    cap, capv = ug.capture, ug._capture_validate

    def wrapped(*a, **kw):
        ug.n_captures += 1
        return cap(*a, **kw)

    def wrapped_v(*a, **kw):
        ug.n_captures += 1
        return capv(*a, **kw)
    ug.capture, ug._capture_validate = wrapped, wrapped_v
    return ug


def per_utterance_loop(ug: UtteranceGenerator, enc, utts) -> dict:
    """The pattern without batching: one generator graph per utterance length, the encoder and scores at that length."""
    plan = enc.plan(ug.dtype)
    out = {}
    for i, (su, sid, ut, ph) in enumerate(utts):
        n = su.shape[0]
        x = ug.generate_graph(su.unsqueeze(0), sid.reshape(1))
        sums, counts = pe.encoder_scores(plan, x, ut[None].cuda(), ph[None].cuda(),
                                         torch.full((1,), n, dtype=torch.int32, device="cuda"))
        s, c = sums.to("cpu").tolist()[0], counts.to("cpu").tolist()[0]
        out[i] = EncoderScore(s[0], s[1], *c)
    return out


def run(g, enc, utts, kind: str, max_graphs: int = 8, warm: bool = False, warm_reps: int = 3) -> tuple:
    ug = counting(UtteranceGenerator(g, "bf16", max_graphs=max_graphs, emg_encoder=enc))
    if warm:
        ug.validate_batched(utts)
        ug.n_captures = 0
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_reserved()
    fn = (lambda: per_utterance_loop(ug, enc, utts)) if kind == "loop" else (lambda: ug.validate_batched(utts))
    runs = [timed(fn) for _ in range(warm_reps if warm else 1)]
    secs, out = sorted(runs, key=lambda r: r[0])[len(runs) // 2]
    lens = [int(u[0].shape[0]) for u in utts]
    res = {"seconds": round(secs, 3), "timed_passes": len(runs), "utterances_per_s": round(len(utts) / secs, 1),
           "emg_samples_per_s": round(sum(lens) * HOP / secs, 0), "graphs_captured": ug.n_captures,
           "peak_reserved_gb": round(torch.cuda.max_memory_reserved() / 1e9, 2)}
    if kind != "loop":
        plan = inference.plan_batches(lens)
        n_graphs = sum(1 for k in ug._graphs if k[0] == "validate")
        res.update(batches=len(plan), buckets=len({T for T, _ in plan}), max_graphs=max_graphs, resident_graphs=n_graphs,
                   padded_rows_fraction=round(1.0 - sum(lens) / sum(8 * T for T, _ in plan), 4),
                   reserved_gb_per_resident_graph=round((torch.cuda.memory_reserved() - base) / 1e9 / max(1, n_graphs), 3))
    del ug
    torch.cuda.empty_cache()
    return res, out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_validate_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("validate_bench.py: needs a CUDA device")
    enc = full_size_encoder()
    line = {"metric": "generated utterances scored by the EMG encoder per second (validate_batched, warm)", "gpu": gpu_info()}
    line["encoder_mask_cost"] = [encoder_mask_cost(enc, 16, 1600, a.reps, a.calls),
                                 encoder_mask_cost(enc, 8, 24000, a.reps, max(1, a.calls // 4))]
    print("mask cost done", file=sys.stderr, flush=True)

    torch.manual_seed(0)
    g = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8).cuda()
    gen = torch.Generator().manual_seed(0)
    lens = torch.randint(100, 1501, (a.n,), generator=gen).tolist()
    utts = [(torch.randn(L, 256, generator=gen), torch.randint(0, 17, (), generator=gen), torch.randn(L, 256, generator=gen),
             torch.randint(0, 48, (L,), generator=gen)) for L in lens]
    n_buckets = len({bucket_frames(L) for L in lens})
    line["workload"] = (f"{a.n} utterances, 100..1500 frames uniform (seed 0), full-size seed-0 generator + full-size encoder, bf16, "
                        "random unit / phoneme targets")

    sample = utts[::16]                                  # parity first
    _, ref_out = run(g, enc, sample, "loop", max_graphs=4)
    _, got = run(g, enc, sample, "batched", max_graphs=4)
    worst = max(max(abs(got[i].speech_unit_loss / ref_out[i].speech_unit_loss - 1),
                    abs(got[i].phoneme_loss / ref_out[i].phoneme_loss - 1)) for i in ref_out)
    frames_ok = all(got[i].num_phones == ref_out[i].num_phones for i in ref_out)
    line["parity"] = {"utterances": len(sample), "worst_rel_loss_diff_vs_loop": worst, "tolerance": 2e-2,
                      "ok": worst <= 2e-2 and frames_ok}
    if not line["parity"]["ok"]:
        print(json.dumps(line), flush=True)
        raise SystemExit(f"validate_bench.py: parity gate FAILED ({worst})")

    v = {}
    v["per_utterance_loop_cold"], _ = run(g, enc, utts, "loop")
    print("loop done", file=sys.stderr, flush=True)
    v["validate_batched_cold"], _ = run(g, enc, utts, "batched")
    v["validate_batched_warm"], _ = run(g, enc, utts, "batched", max_graphs=n_buckets, warm=True)
    line["validation"] = v
    line["value"] = v["validate_batched_warm"]["utterances_per_s"]
    line["unit"] = "utterances/s"
    line["speedup_cold"] = round(v["per_utterance_loop_cold"]["seconds"] / v["validate_batched_cold"]["seconds"], 2)
    s = json.dumps(line)
    print(s, flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
