"""Generator-only inference (EMGGenerator.generate, models/generator.py:48-50; called at
ste_gan/train.py:394) as a serving loop: weights are folded once, each (batch, frames) shape
is captured as a CUDA graph, utterances are sharded round-robin over ranks with no collective.
serve_batched() pads utterances of similar length to a common bucket length and runs them as one
batch with per-sample length masks (stg_conv_masked), which leaves each utterance's result exact.
validate_batched() scores generated utterances with the frozen EMG encoder in the same padded batches.
"""
from __future__ import annotations

from collections import OrderedDict
from dataclasses import dataclass
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import torch

from . import passes, passes_encoder
from .dist import round_robin
from .models.emg_encoder import SILENCE_PHONEME_INDEX

Tensor = torch.Tensor

# Bucket ladder of serve_batched: MIN_BUCKET frames, then BUCKETS_PER_OCTAVE evenly spaced lengths per octave
# (16, 20, 24, 28, 32, 40, 48, 56, 64, 80, ...): an utterance is padded by less than 1 / BUCKETS_PER_OCTAVE of its length.
MIN_BUCKET = 16
BUCKETS_PER_OCTAVE = 4


def bucket_frames(n: int, per_octave: int = BUCKETS_PER_OCTAVE) -> int:
    """Smallest length of the bucket ladder that holds an utterance of n frames."""
    b = MIN_BUCKET
    while True:
        for j in range(per_octave):
            v = b + j * b // per_octave
            if v >= n:
                return v
        b *= 2


def plan_batches(lengths: Sequence[int], max_batch: int = 8,
                 per_octave: int = BUCKETS_PER_OCTAVE) -> List[Tuple[int, List[int]]]:
    """The batches serve_batched runs for utterances of these lengths (frames): [(bucket frames, utterance indices)],
    in ascending bucket order, each bucket's utterances in index order, at most max_batch per batch.  Pure host code
    of the lengths alone, so every rank computes the same plan; rank r of world w runs batches r, r + w, r + 2w, ..."""
    if max_batch < 1:
        raise ValueError("plan_batches: max_batch must be >= 1")
    by_bucket: Dict[int, List[int]] = {}
    for i, n in enumerate(lengths):
        by_bucket.setdefault(bucket_frames(int(n), per_octave), []).append(i)
    plan = []
    for T in sorted(by_bucket):
        idx = by_bucket[T]
        plan += [(T, idx[j:j + max_batch]) for j in range(0, len(idx), max_batch)]
    return plan


@dataclass
class EncoderScore:
    """EMGEncoderLoss (losses/emg_encoder_loss.py:19-84) of one generated utterance, or summed over several
    (aggregate_scores): the sums over frames and the phone counts, from which the frame-weighted means follow."""
    speech_unit_sum: float              # sum over frames of ||target - pred + 1e-6||_2
    phoneme_sum: float                  # sum over frames of the phoneme cross-entropy
    num_phones: int                     # frames
    num_correct_phones: int
    num_silence_phones: int
    num_correct_phones_no_silence: int

    @property
    def speech_unit_loss(self) -> float:
        """Mean speech-unit distance (NaN for zero frames, as the mean of nothing)."""
        return self.speech_unit_sum / self.num_phones if self.num_phones else float("nan")

    @property
    def phoneme_loss(self) -> float:
        """Mean phoneme cross-entropy (NaN for zero frames)."""
        return self.phoneme_sum / self.num_phones if self.num_phones else float("nan")


def aggregate_scores(scores: Iterable[EncoderScore]) -> EncoderScore:
    """Frame-weighted totals over a set of utterances: the sums and counts added up (in double precision), so the means of
    the result weight every frame equally.  Accepts the values of validate_batched dicts, also merged across ranks."""
    total = EncoderScore(0.0, 0.0, 0, 0, 0, 0)
    for sc in scores:
        total.speech_unit_sum += sc.speech_unit_sum
        total.phoneme_sum += sc.phoneme_sum
        total.num_phones += sc.num_phones
        total.num_correct_phones += sc.num_correct_phones
        total.num_silence_phones += sc.num_silence_phones
        total.num_correct_phones_no_silence += sc.num_correct_phones_no_silence
    return total


class UtteranceGenerator:
    """max_graphs bounds the per-shape CUDA-graph cache (least recently used shape is dropped): each captured (batch,
    frames) shape pins its activations, so serving arbitrary utterance lengths would otherwise grow without limit.
    The generator is purely convolutional with zero padding, so a zero-padded utterance is NOT identical near its end -
    unless the padding is masked: with `lengths`, every convolution writes 0 past each sample's own end, so every
    convolution reads exactly the zero padding the utterance gets on its own.  serve() runs one utterance per call
    at its own length; serve_batched() pads utterances to a few bucket lengths and batches them with length masks.
    Graphs are cached per (batch, frames) shape, masked graphs under (batch, frames, True): a masked graph reads the
    lengths from a device buffer refreshed before each replay, so one graph serves every length mix of its shape.
    emg_encoder (a frozen EMGEncoderTransformer on the same device): validate_batched() scores the generated EMG with it;
    its graphs are cached under ("validate", batch, frames) in the same LRU cache."""

    def __init__(self, net_g, precision: str = "bf16", max_graphs: int = 8, trainer=None, emg_encoder=None):
        self.net_g = net_g
        self.dtype = torch.bfloat16 if precision == "bf16" else torch.float32
        self.device = next(net_g.parameters()).device
        if self.device.type != "cuda":
            raise RuntimeError("UtteranceGenerator: move the generator to a CUDA device first (no CPU path)")
        self.trainer = trainer            # a GanTrainer that owns net_g: its deferred optimiser step is flushed first
        if trainer is not None:
            trainer.flush()
        self.folds = passes.fold_generator(net_g, self.dtype, want_dgrad=False)   # weights are frozen while serving
        self.max_graphs = max(1, int(max_graphs))
        self._graphs: "OrderedDict[tuple, tuple]" = OrderedDict()
        self._uses_mode = bool(getattr(net_g, "use_speaking_mode_embedding", False))
        self.emg_encoder = emg_encoder

    def refold(self) -> None:
        """Call after the generator's weights changed (drops every captured graph, the validation graphs included)."""
        if self.trainer is not None:
            self.trainer.flush()          # (pipelined step_graph defers the last generator AdamW)
        self.folds = passes.fold_generator(self.net_g, self.dtype, want_dgrad=False)
        self._graphs.clear()

    @torch.no_grad()
    def generate(self, speech_units: Tensor, session_ids: Tensor, speaking_mode_ids: Optional[Tensor] = None,
                 lengths: Optional[Tensor] = None) -> Tensor:
        """[B,T,D] units -> [B,rT,C] fp32 EMG (eager launches; r = 16 output rows per frame for speech units, 8 for
        MFCCs).  lengths ([B] ints, frames): sample b is an utterance of lengths[b] frames zero-padded to T; its rows
        [0, r*lengths[b]) are what it gives on its own and the rest are 0, whatever the padded units hold."""
        if lengths is not None:
            lengths = lengths.to(self.device, torch.int32)
        x, _ = passes.generator_forward(self.net_g, speech_units, session_ids, speaking_mode_ids, self.dtype, False,
                                        folds=self.folds, lengths=lengths)
        return x

    @torch.no_grad()
    def capture(self, batch: int, frames: int, unit_dim: int, masked: bool = False) -> None:
        key = (batch, frames, True) if masked else (batch, frames)
        while len(self._graphs) >= self.max_graphs:      # LRU bound
            self._graphs.popitem(last=False)
        su = torch.zeros(batch, frames, unit_dim, device=self.device)
        sess = torch.zeros(batch, device=self.device, dtype=torch.int64)
        mode = torch.zeros(batch, device=self.device, dtype=torch.int64) if self._uses_mode else None
        lens = torch.full((batch,), frames, device=self.device, dtype=torch.int32) if masked else None
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                self.generate(su, sess, mode, lens)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = self.generate(su, sess, mode, lens)
        self._graphs[key] = (g, su, sess, mode, lens, out)

    @torch.no_grad()
    def generate_graph(self, speech_units: Tensor, session_ids: Tensor, speaking_mode_ids: Optional[Tensor] = None,
                       lengths: Optional[Tensor] = None) -> Tensor:
        """Replay the captured graph for this shape (and masking, see generate); inputs may be pinned-host tensors.
        The returned tensor is the graph's static output buffer (overwritten by the next call of the same shape)."""
        B, T, D = speech_units.shape
        key = (B, T) if lengths is None else (B, T, True)
        if key not in self._graphs:
            self.capture(B, T, D, masked=lengths is not None)
        self._graphs.move_to_end(key)
        g, su, sess, mode, lens, out = self._graphs[key]
        su.copy_(speech_units, non_blocking=True)
        sess.copy_(session_ids, non_blocking=True)
        if mode is not None:
            if speaking_mode_ids is None:
                raise ValueError("generate_graph: this generator uses speaking-mode embeddings - pass speaking_mode_ids")
            mode.copy_(speaking_mode_ids, non_blocking=True)
        if lens is not None:
            lens.copy_(lengths, non_blocking=True)
        g.replay()
        return out

    def serve(self, utterances: List[Tuple[Tensor, Tensor]], rank: int = 0, world: int = 1) -> Dict[int, Tensor]:
        """Generate this rank's share (round-robin) of a list of (units [T,D], session_id) utterances;
        returns {utterance index: EMG [16T, C] on the host}."""
        out = {}
        for i in round_robin(rank, world, len(utterances)):
            su, sid = utterances[i]
            y = self.generate_graph(su.unsqueeze(0), sid.reshape(1))
            out[i] = y[0].to("cpu", non_blocking=False)
        return out

    def serve_batched(self, utterances: List[Tuple[Tensor, Tensor]], rank: int = 0, world: int = 1,
                      max_batch: int = 8, per_octave: int = BUCKETS_PER_OCTAVE) -> Dict[int, Tensor]:
        """serve() in padded batches: the same {utterance index: EMG [rT, C] on the host} for this rank's share.
        Utterances are padded to a bucket length (bucket_frames) and grouped into batches of up to max_batch
        (plan_batches, sharded round-robin by batch); a partial batch is filled with zero-length rows, so each bucket
        replays one masked graph shape, and each output is trimmed to its utterance's r * frames rows.  per_octave sets
        the bucket ladder (fewer buckets: fewer graphs, more padding)."""
        lengths = [int(su.shape[0]) for su, _ in utterances]
        plan = plan_batches(lengths, max_batch, per_octave)
        out = {}
        for T, idx in plan[rank::world]:
            D = utterances[idx[0]][0].shape[1]
            su = torch.zeros(max_batch, T, D)
            sess = torch.zeros(max_batch, dtype=torch.int64)
            lens = torch.zeros(max_batch, dtype=torch.int32)
            for j, i in enumerate(idx):
                su[j, :lengths[i]] = utterances[i][0]
                sess[j] = utterances[i][1].reshape(())
                lens[j] = lengths[i]
            y = self.generate_graph(su, sess, lengths=lens)
            r = y.shape[1] // T
            host = y[:len(idx)].to("cpu", non_blocking=False)     # one copy per batch
            for j, i in enumerate(idx):
                out[i] = host[j, :r * lengths[i]].clone()
        return out

    @torch.no_grad()
    def _score(self, su: Tensor, sess: Tensor, lens: Tensor, ut: Tensor, ph: Tensor) -> Tuple[Tensor, Tensor]:
        """Masked generate -> masked encode -> per-utterance scores, all on the device (see validate_batched)."""
        x, _ = passes.generator_forward(self.net_g, su, sess, None, self.dtype, False, folds=self.folds, lengths=lens)
        plan = self.emg_encoder.plan(self.dtype)
        if x.shape[1] != plan.frame_rows * su.shape[1]:
            raise ValueError(f"validate_batched: the generator gives {x.shape[1] // su.shape[1]} EMG rows per frame, the "
                             f"encoder takes {plan.frame_rows}")
        return passes_encoder.encoder_scores(plan, x, ut, ph, lens)

    @torch.no_grad()
    def _capture_validate(self, batch: int, frames: int, unit_dim: int, target_dim: int) -> None:
        while len(self._graphs) >= self.max_graphs:      # LRU bound, shared with the serving graphs
            self._graphs.popitem(last=False)
        dev = self.device
        su = torch.zeros(batch, frames, unit_dim, device=dev)
        sess = torch.zeros(batch, device=dev, dtype=torch.int64)
        lens = torch.full((batch,), frames, device=dev, dtype=torch.int32)
        ut = torch.zeros(batch, frames, target_dim, device=dev)
        ph = torch.zeros(batch, frames, device=dev, dtype=torch.int64)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                self._score(su, sess, lens, ut, ph)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            sums, counts = self._score(su, sess, lens, ut, ph)
        self._graphs[("validate", batch, frames)] = (g, su, sess, lens, ut, ph, sums, counts)

    def validate_batched(self, utterances: List[Tuple[Tensor, Tensor, Tensor, Tensor]], rank: int = 0, world: int = 1,
                         max_batch: int = 8, per_octave: int = BUCKETS_PER_OCTAVE) -> Dict[int, EncoderScore]:
        """Score generated utterances with the frozen EMG encoder: this rank's share of (generator input [n, D], session_id,
        unit_target [n, Du], phoneme_target [n]) items -> {utterance index: EncoderScore}, each equal to EMGEncoderLoss on
        that utterance's generated EMG alone.  Batches as serve_batched (plan_batches, round-robin by batch); each bucket
        replays one captured graph of masked generate -> masked encode -> scores, so the EMG never leaves the device and
        only the [max_batch] sums and counts come back per batch.  Merge the dicts of several ranks with aggregate_scores."""
        if self.emg_encoder is None:
            raise ValueError("validate_batched: construct UtteranceGenerator with emg_encoder=")
        if self._uses_mode:
            raise ValueError("validate_batched: speaking-mode generators are not supported (as in serve_batched)")
        lengths = [int(u[0].shape[0]) for u in utterances]
        plan = plan_batches(lengths, max_batch, per_octave)
        out = {}
        for T, idx in plan[rank::world]:
            D, Du = utterances[idx[0]][0].shape[1], utterances[idx[0]][2].shape[1]
            key = ("validate", max_batch, T)
            if key not in self._graphs:
                self._capture_validate(max_batch, T, D, Du)
            self._graphs.move_to_end(key)
            g, su_d, sess_d, lens_d, ut_d, ph_d, sums_d, counts_d = self._graphs[key]
            su = torch.zeros(max_batch, T, D)
            sess = torch.zeros(max_batch, dtype=torch.int64)
            lens = torch.zeros(max_batch, dtype=torch.int32)
            ut = torch.zeros(max_batch, T, Du)
            ph = torch.zeros(max_batch, T, dtype=torch.int64)
            for j, i in enumerate(idx):
                units, sid, u_t, p_t = utterances[i]
                n = lengths[i]
                if u_t.shape[0] != n or p_t.shape[0] != n:
                    raise ValueError(f"validate_batched: utterance {i} has {n} input frames but targets of "
                                     f"{u_t.shape[0]} / {p_t.shape[0]} frames")
                su[j, :n], sess[j], lens[j], ut[j, :n], ph[j, :n] = units, sid.reshape(()), n, u_t, p_t
            for dst, src in ((su_d, su), (sess_d, sess), (lens_d, lens), (ut_d, ut), (ph_d, ph)):
                dst.copy_(src, non_blocking=True)
            g.replay()
            sums, counts = sums_d.to("cpu").tolist(), counts_d.to("cpu").tolist()      # the only copies back per batch
            for j, i in enumerate(idx):
                out[i] = EncoderScore(sums[j][0], sums[j][1], *counts[j])
        return out
