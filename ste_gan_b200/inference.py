"""Generator-only inference (EMGGenerator.generate, models/generator.py:48-50; called at
ste_gan/train.py:394) as a serving loop: weights are folded once, each (batch, frames) shape
is captured as a CUDA graph, utterances are sharded round-robin over ranks with no collective.
serve_batched() pads utterances of similar length to a common bucket length and runs them as one
batch with per-sample length masks (stg_conv_masked), which leaves each utterance's result exact.
validate_batched() scores generated utterances in the same padded batches: with the frozen EMG encoder and / or, against
the utterances' real EMG, with the time-domain feature losses.
"""
from __future__ import annotations

import math
from collections import OrderedDict
from dataclasses import dataclass
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import torch

from . import ops, passes, passes_encoder
from .dist import round_robin
from .losses.time_domain_loss import _RES
from .models.emg_encoder import SILENCE_PHONEME_INDEX

Tensor = torch.Tensor

# Bucket ladder of serve_batched: MIN_BUCKET frames, then BUCKETS_PER_OCTAVE evenly spaced lengths per octave
# (16, 20, 24, 28, 32, 40, 48, 56, 64, 80, ...): an utterance is padded by less than 1 / BUCKETS_PER_OCTAVE of its length.
MIN_BUCKET = 16
BUCKETS_PER_OCTAVE = 4
# Fewest EMG rows the time-domain losses take: F.pad(..., 'reflect') raises unless the pad (avg_window // 2 = 4 for the
# average filter, win // 2 for the padded windows) is smaller than the signal.
TD_MIN_ROWS = max(9 // 2, max(w // 2 for w, _ in _RES)) + 1


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


@dataclass
class TdScore:
    """MultiTimeDomainFeatureLoss (losses/time_domain_loss.py:76-107) of one generated utterance against its real EMG, or
    the mean over several (aggregate_td): one value per resolution of MultiTimeDomainFeatureLoss, (20, 8), (51, 13),
    (80, 16), unweighted (the caller applies w_td)."""
    values: Tuple[float, ...]

    @property
    def loss(self) -> float:
        """The sum over the resolutions: MultiTimeDomainFeatureLoss's value."""
        return sum(self.values)


@dataclass
class ValidationScore:
    """One utterance's scores from validate_batched(real_emg=...): the time-domain losses against its real EMG, and the
    EMG-encoder score when the engine has an encoder (else None)."""
    td: TdScore
    encoder: Optional[EncoderScore]


def aggregate_td(scores: Iterable[TdScore]) -> TdScore:
    """The mean over utterances of each per-resolution value.  The reference validates at batch 1 (collate.py:87,149-151)
    and averages over batches, so every utterance weighs the same whatever its length - unlike aggregate_scores, which
    weights every frame equally.  The sums are exact (math.fsum), so the result does not depend on the order of the
    utterances: the dicts of several ranks merge into the value of one rank's dict."""
    vals = [sc.values for sc in scores]
    if not vals:
        return TdScore((float("nan"),) * len(_RES))
    return TdScore(tuple(math.fsum(v[i] for v in vals) / len(vals) for i in range(len(vals[0]))))


class UtteranceGenerator:
    """max_graphs bounds the per-shape CUDA-graph cache (least recently used shape is dropped): each captured (batch,
    frames) shape pins its activations, so serving arbitrary utterance lengths would otherwise grow without limit.
    The generator is purely convolutional with zero padding, so a zero-padded utterance is NOT identical near its end -
    unless the padding is masked: with `lengths`, every convolution writes 0 past each sample's own end, so every
    convolution reads exactly the zero padding the utterance gets on its own.  serve() runs one utterance per call
    at its own length; serve_batched() pads utterances to a few bucket lengths and batches them with length masks.
    Graphs are cached per (batch, frames) shape, masked graphs under (batch, frames, True): a masked graph reads the
    lengths from a device buffer refreshed before each replay, so one graph serves every length mix of its shape.
    emg_encoder (a frozen EMGEncoderTransformer on the same device): validate_batched() scores the generated EMG with it
    and / or, given the real EMG, with the time-domain losses; its graphs are cached under ("validate", batch, frames,
    encoder?, time-domain?) in the same LRU cache."""

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
            self.trainer.flush()          # (step_graph defers the last generator AdamW)
        self.folds = passes.fold_generator(self.net_g, self.dtype, want_dgrad=False)
        self._graphs.clear()

    @property
    def rows_per_frame(self) -> int:
        """EMG rows the generator gives per input frame: 16 for speech units, 8 for MFCCs."""
        return math.prod(int(b.upsample) for b in list(self.net_g.gblocks)[1:])

    def _mode_ids(self, speaking_mode_ids: Optional[Sequence[int]], n: int, who: str) -> Optional[List[int]]:
        """The speaking-mode ids of n utterances, checked on the host; None for a generator without the embedding."""
        if not self._uses_mode:
            return None
        if speaking_mode_ids is None:
            raise ValueError(f"{who}: this generator uses speaking-mode embeddings - pass speaking_mode_ids")
        ids = [int(m) for m in speaking_mode_ids]
        n_modes = self.net_g.speaking_mode_embeddings.num_embeddings
        if len(ids) != n:
            raise ValueError(f"{who}: {len(ids)} speaking_mode_ids for {n} utterances")
        if any(not 0 <= m < n_modes for m in ids):
            raise ValueError(f"{who}: speaking_mode_ids must lie in [0, {n_modes})")
        return ids

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
                      max_batch: int = 8, per_octave: int = BUCKETS_PER_OCTAVE,
                      speaking_mode_ids: Optional[Sequence[int]] = None) -> Dict[int, Tensor]:
        """serve() in padded batches: the same {utterance index: EMG [rT, C] on the host} for this rank's share.
        Utterances are padded to a bucket length (bucket_frames) and grouped into batches of up to max_batch
        (plan_batches, sharded round-robin by batch); a partial batch is filled with zero-length rows, so each bucket
        replays one masked graph shape, and each output is trimmed to its utterance's r * frames rows.  per_octave sets
        the bucket ladder (fewer buckets: fewer graphs, more padding).  speaking_mode_ids: one per utterance, required by a
        generator with speaking-mode embeddings and ignored by one without (filler rows take mode 0)."""
        modes = self._mode_ids(speaking_mode_ids, len(utterances), "serve_batched")
        lengths = [int(su.shape[0]) for su, _ in utterances]
        plan = plan_batches(lengths, max_batch, per_octave)
        out = {}
        for T, idx in plan[rank::world]:
            D = utterances[idx[0]][0].shape[1]
            su = torch.zeros(max_batch, T, D)
            sess = torch.zeros(max_batch, dtype=torch.int64)
            lens = torch.zeros(max_batch, dtype=torch.int32)
            mode = torch.zeros(max_batch, dtype=torch.int64) if modes is not None else None
            for j, i in enumerate(idx):
                su[j, :lengths[i]] = utterances[i][0]
                sess[j] = utterances[i][1].reshape(())
                lens[j] = lengths[i]
                if mode is not None:
                    mode[j] = modes[i]
            y = self.generate_graph(su, sess, mode, lengths=lens)
            r = y.shape[1] // T
            host = y[:len(idx)].to("cpu", non_blocking=False)     # one copy per batch
            for j, i in enumerate(idx):
                out[i] = host[j, :r * lengths[i]].clone()
        return out

    @torch.no_grad()
    def _score(self, su: Tensor, sess: Tensor, mode: Optional[Tensor], lens: Tensor, ut: Optional[Tensor],
               ph: Optional[Tensor], real: Optional[Tensor]):
        """Masked generate -> (masked encode -> encoder scores) and / or (time-domain scores against the real EMG), all on the
        device (see validate_batched).  Returns (sums, counts, td), None for what is not computed."""
        x, _ = passes.generator_forward(self.net_g, su, sess, mode, self.dtype, False, folds=self.folds, lengths=lens)
        sums = counts = td = None
        if ut is not None:
            plan = self.emg_encoder.plan(self.dtype)
            if x.shape[1] != plan.frame_rows * su.shape[1]:
                raise ValueError(f"validate_batched: the generator gives {x.shape[1] // su.shape[1]} EMG rows per frame, the "
                                 f"encoder takes {plan.frame_rows}")
            sums, counts = passes_encoder.encoder_scores(plan, x, ut, ph, lens)
        if real is not None:
            td = ops.td_scores(real, x, lens, x.shape[1] // su.shape[1])
        return sums, counts, td

    @torch.no_grad()
    def _capture_validate(self, batch: int, frames: int, unit_dim: int, target_dim: Optional[int] = None,
                          emg_channels: Optional[int] = None) -> None:
        """Capture the validation graph of one bucket: with the encoder's targets when target_dim is given, with a static
        real-EMG buffer [batch, r * frames, emg_channels] and the time-domain scores when emg_channels is given."""
        while len(self._graphs) >= self.max_graphs:      # LRU bound, shared with the serving graphs
            self._graphs.popitem(last=False)
        dev = self.device
        enc, td = target_dim is not None, emg_channels is not None
        ins = (torch.zeros(batch, frames, unit_dim, device=dev),                                   # units
               torch.zeros(batch, device=dev, dtype=torch.int64),                                  # session ids
               torch.zeros(batch, device=dev, dtype=torch.int64) if self._uses_mode else None,     # speaking modes
               torch.full((batch,), frames, device=dev, dtype=torch.int32),                        # lengths
               torch.zeros(batch, frames, target_dim, device=dev) if enc else None,                # unit targets
               torch.zeros(batch, frames, device=dev, dtype=torch.int64) if enc else None,         # phoneme targets
               torch.zeros(batch, self.rows_per_frame * frames, emg_channels, device=dev) if td else None)   # real EMG
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                self._score(*ins)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            outs = self._score(*ins)
        self._graphs[("validate", batch, frames, enc, td)] = (g, ins, outs)

    def validate_batched(self, utterances: List[Tuple[Tensor, ...]], rank: int = 0, world: int = 1, max_batch: int = 8,
                         per_octave: int = BUCKETS_PER_OCTAVE, real_emg: Optional[Sequence[Tensor]] = None,
                         speaking_mode_ids: Optional[Sequence[int]] = None) -> Dict[int, object]:
        """Score generated utterances: this rank's share of (generator input [n, D], session_id, unit_target [n, Du],
        phoneme_target [n]) items -> {utterance index: EncoderScore}, each equal to EMGEncoderLoss on that utterance's
        generated EMG alone.  Batches as serve_batched (plan_batches, round-robin by batch); each bucket replays one captured
        graph of masked generate -> masked encode -> scores, so the EMG never leaves the device and only the [max_batch]
        sums and counts come back per batch.  Merge the dicts of several ranks with aggregate_scores.

        real_emg: the real EMG [r * n, C] of each utterance (r = rows_per_frame), aligned with utterances.  Each value is
        then a ValidationScore: td holds MultiTimeDomainFeatureLoss(real, generated) of that utterance alone, per resolution
        (stg_td_scores in the same graph; only the [max_batch, 3] values come back), and encoder the EncoderScore above, or
        None for an engine without emg_encoder, whose items may then be (units, session_id) alone.  An utterance shorter
        than TD_MIN_ROWS EMG rows raises ValueError, as the reference's reflect padding does.  Merge with aggregate_td.
        speaking_mode_ids: one per utterance, required by a generator with speaking-mode embeddings, ignored otherwise.
        Every argument is checked before the first launch."""
        td, enc = real_emg is not None, self.emg_encoder is not None
        if not enc and not td:
            raise ValueError("validate_batched: construct UtteranceGenerator with emg_encoder=, or pass real_emg=")
        modes = self._mode_ids(speaking_mode_ids, len(utterances), "validate_batched")
        lengths = [int(u[0].shape[0]) for u in utterances]
        for i, u in enumerate(utterances if enc else ()):
            if len(u) < 4 or u[2].shape[0] != lengths[i] or u[3].shape[0] != lengths[i]:
                raise ValueError(f"validate_batched: utterance {i} has {lengths[i]} input frames but no unit / phoneme targets "
                                 f"of as many frames")
        r = self.rows_per_frame
        if td:
            if len(real_emg) != len(utterances):
                raise ValueError(f"validate_batched: {len(real_emg)} real_emg items for {len(utterances)} utterances")
            c_out = self.net_g.num_output_channels
            for i, x in enumerate(real_emg):
                if tuple(x.shape) != (r * lengths[i], c_out):
                    raise ValueError(f"validate_batched: real_emg[{i}] is {tuple(x.shape)}, the generator gives "
                                     f"{(r * lengths[i], c_out)} for utterance {i}")
                if r * lengths[i] < TD_MIN_ROWS:
                    raise ValueError(f"validate_batched: utterance {i} has {r * lengths[i]} EMG rows, the time-domain losses "
                                     f"need at least {TD_MIN_ROWS} (their reflect padding)")
        plan = plan_batches(lengths, max_batch, per_octave)
        out = {}
        for T, idx in plan[rank::world]:
            D = utterances[idx[0]][0].shape[1]
            Du = utterances[idx[0]][2].shape[1] if enc else None
            key = ("validate", max_batch, T, enc, td)
            if key not in self._graphs:
                self._capture_validate(max_batch, T, D, Du, self.net_g.num_output_channels if td else None)
            self._graphs.move_to_end(key)
            g, (su_d, sess_d, mode_d, lens_d, ut_d, ph_d, real_d), (sums_d, counts_d, td_d) = self._graphs[key]
            su = torch.zeros(max_batch, T, D)
            sess = torch.zeros(max_batch, dtype=torch.int64)
            lens = torch.zeros(max_batch, dtype=torch.int32)
            host = [(su_d, su), (sess_d, sess), (lens_d, lens)]
            if enc:
                ut = torch.zeros(max_batch, T, Du)
                ph = torch.zeros(max_batch, T, dtype=torch.int64)
                host += [(ut_d, ut), (ph_d, ph)]
            if mode_d is not None:
                mode = torch.zeros(max_batch, dtype=torch.int64)
                host.append((mode_d, mode))
            for j, i in enumerate(idx):
                n = lengths[i]
                su[j, :n], sess[j], lens[j] = utterances[i][0], utterances[i][1].reshape(()), n
                if enc:
                    ut[j, :n], ph[j, :n] = utterances[i][2], utterances[i][3]
                if mode_d is not None:
                    mode[j] = modes[i]
                if td:
                    real_d[j, :r * n].copy_(real_emg[i], non_blocking=True)    # rows past r * n are never read
            for dst, src in host:
                dst.copy_(src, non_blocking=True)
            g.replay()
            if enc:
                sums, counts = sums_d.to("cpu").tolist(), counts_d.to("cpu").tolist()     # the only copies back per batch
            if td:
                tds = td_d.to("cpu").tolist()
            for j, i in enumerate(idx):
                es = EncoderScore(sums[j][0], sums[j][1], *counts[j]) if enc else None
                out[i] = ValidationScore(TdScore(tuple(tds[j])), es) if td else es
        return out
