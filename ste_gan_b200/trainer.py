"""The GAN train step (ste_gan/train.py:165-268) as an explicit schedule over the fused passes,
with data-parallel gradient averaging and CUDA-graph replay.

One `GanTrainer.step()` = one iteration of the reference's inner loop without the encoder
losses (SURVEY.md 2 row 8 - no checkpoint exists for them):

    D phase   x_pred = G(units)                                   train.py:182
              D(x_pred.detach()), D(x_real) -> loss_D             train.py:190-196
              backward (both passes), all-reduce, AdamW on D      train.py:198-199
    G phase   D(x_pred), D(x_real) with the UPDATED D             train.py:206-207
              adv + 15*TD + 7*FM -> loss_G                        train.py:209-217,257-263
              backward through D (data-gradient only - the reference's D weight gradients of
              this phase are discarded by zero_grad, train.py:166) and G, all-reduce, AdamW on G

Parameters, gradients and AdamW moments of each network live in one flat fp32 buffer each
(`FlatParams`), so the optimiser is a single kernel and the data-parallel exchange is one
bucketed NCCL all-reduce over NVLink per phase.  Spectral-norm layers are re-folded on every
discriminator forward (4 power iterations per step, as in the reference); weight-norm folds
are reused while the weights are unchanged.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch
from . import ops, passes
from .dist import GradReducer

Tensor = torch.Tensor

W_TD_DEFAULT, W_FM_DEFAULT = 15.0, 7.0         # configs/ste_gan_base_gantts.yaml:33,37
LOSS_NAMES = ["loss_d", "loss_adv", "loss_fm", "loss_td_20_8", "loss_td_51_13", "loss_td_80_16", "loss_speech_unit", "loss_phoneme"]
W_SU_DEFAULT, W_PH_DEFAULT = 1.0, 1.0          # configs/ste_gan_base_gantts.yaml: loss_speech_unit_weight / loss_phoneme_weight


class FlatParams:
    """Re-homes a module's parameters (registration order) into one flat fp32 buffer with a
    matching flat gradient; `param.data` / `param.grad` become views."""

    def __init__(self, module: torch.nn.Module):
        self.params = [p for p in module.parameters()]
        dev = self.params[0].device
        if dev.type != "cuda":
            raise RuntimeError("FlatParams: move the module to a CUDA device first")
        # every parameter starts on a 16-byte boundary (the 1-element bias / weight_g of the logits convs would otherwise
        # misalign everything behind them and switch the fold kernels to 4-byte accesses); the gaps stay zero
        al = lambda k: (k + 3) // 4 * 4
        n = sum(al(p.numel()) for p in self.params)
        self.flat = torch.zeros(n, device=dev, dtype=torch.float32)
        self.grad = torch.zeros(n, device=dev, dtype=torch.float32)
        off = 0
        self.offsets: Dict[str, int] = {}        # parameter name -> offset into the flat buffers (registration order)
        names = [nm for nm, _ in module.named_parameters()]
        for nm, p in zip(names, self.params):
            k = p.numel()
            self.flat[off:off + k].copy_(p.data.reshape(-1))
            p.data = self.flat[off:off + k].view(p.shape)
            p.grad = self.grad[off:off + k].view(p.shape)
            self.offsets[nm] = off
            off += al(k)
        self.m = torch.zeros_like(self.flat)
        self.v = torch.zeros_like(self.flat)
        self.step = torch.zeros(1, device=dev, dtype=torch.int64)
        self.numel = n

    def zero_grad(self) -> None:
        self.grad.zero_()

    def adamw(self, lr, betas=(0.8, 0.99), eps: float = 1e-8, weight_decay: float = 1e-2,
              grad_scale: float = 1.0, enable: Optional[Tensor] = None, lo: int = 0, hi: Optional[int] = None,
              keep_step: bool = False) -> None:
        """torch.optim.AdamW(lr=2e-4, betas=(.8,.99)) - ste_gan/constants.py:57.  grad_scale = 1/world
        turns the all-reduced gradient SUM into the data-parallel mean inside the kernel.  [lo, hi): update only this
        slice of the flat buffers (one gradient bucket); every slice but the first of a step passes keep_step."""
        hi = self.numel if hi is None else hi
        ops.adamw(self.flat[lo:hi], self.grad[lo:hi], self.m[lo:hi], self.v[lo:hi], self.step, lr, betas[0], betas[1], eps,
                  weight_decay, grad_scale, enable, keep_step)


def generator_grad_buckets(offsets: Dict[str, int], numel: int, nblk: int) -> list:
    """Gradient buckets of the generator, back to front (= the order its backward completes them): GBlocks [k2, n) +
    last_conv | [k1, k2) | [0, k1) + gblocks.0 + embeddings, cut at the GBlock boundaries nearest to 1/3 and 2/3 of the
    parameters (base model: GB3..GB8 | GB2 | GB1, ~8 M parameters each).  `offsets`: parameter name -> offset into the flat
    buffer (registration order).  Each entry: (first GBlock, end GBlock, first conv, end conv of
    passes.generator_convs, flat-gradient slice)."""
    first = [offsets[next(nm for nm in offsets if nm.startswith(f"gblocks.{i + 1}."))] for i in range(nblk)]
    last = offsets[next(nm for nm in offsets if nm.startswith("last_conv."))]
    near = lambda frac, lo: min(range(lo, nblk), key=lambda i: abs(first[i] - frac * numel), default=nblk)
    k1 = near(1.0 / 3.0, 1)            # the GBlock boundary nearest to 1/3 ...
    k2 = near(2.0 / 3.0, k1)           # ... and to 2/3 of the parameters
    n_conv = 5 * nblk + 2
    cut = lambda i: first[i] if i < nblk else last
    return [(k2, nblk, 1 + 5 * k2, n_conv, (cut(k2), numel)),
            (k1, k2, 1 + 5 * k1, 1 + 5 * k2, (cut(k1), cut(k2))),
            (0, k1, 0, 1 + 5 * k1, (0, cut(k1)))]


class GanTrainer:
    def __init__(self, net_g, net_d, precision: str = "bf16", lr: float = 2e-4, w_td: float = W_TD_DEFAULT,
                 w_fm: float = W_FM_DEFAULT, loss_adversarial: bool = True, loss_multi_td: bool = True,
                 loss_feat_match: bool = True, group=None, grad_buckets: Optional[int] = None, data_parallel: bool = True,
                 emg_encoder=None, loss_speech_unit: Optional[bool] = None, loss_phoneme: Optional[bool] = None,
                 w_su: float = W_SU_DEFAULT, w_ph: float = W_PH_DEFAULT):
        """emg_encoder: a frozen ste_gan_b200.models.emg_encoder.EMGEncoderTransformer (eval mode) - switches on the two
        perceptual losses of the generator step (train.py:219-230: speech-unit distance and phoneme cross-entropy of the
        encoder's predictions on the GENERATED EMG; both default to on when an encoder is given, as in the YAML)."""
        self.net_g, self.net_d = net_g, net_d
        self.dtype = torch.bfloat16 if precision == "bf16" else torch.float32
        self.w_td, self.w_fm = w_td, w_fm
        self.use_adv, self.use_td, self.use_fm = loss_adversarial, loss_multi_td, loss_feat_match
        self.emg_encoder = emg_encoder
        self.use_su = (emg_encoder is not None) if loss_speech_unit is None else bool(loss_speech_unit)
        self.use_ph = (emg_encoder is not None) if loss_phoneme is None else bool(loss_phoneme)
        if (self.use_su or self.use_ph) and emg_encoder is None:
            raise ValueError("loss_speech_unit / loss_phoneme need an emg_encoder")
        self.w_su, self.w_ph = w_su, w_ph
        self._enc_plan = None
        if emg_encoder is not None:
            if emg_encoder.training:
                raise ValueError("the EMG encoder of the perceptual losses is frozen: call emg_encoder.eval() (emg_encoder_loss.py:61)")
            self._enc_plan = emg_encoder.plan(self.dtype)
        self._cur_su = self._cur_ph = None
        self.G, self.D = FlatParams(net_g), FlatParams(net_d)
        # packed operands, gradient arenas and multi-tensor fold tables at fixed addresses (after the re-homing above)
        self.g_plan = passes.FoldPlan(passes.generator_convs(net_g), self.dtype)
        self.d_plan = passes.FoldPlan(passes.discriminator_convs(net_d), self.dtype)
        self._d_folded = False                  # d_plan packs match the current D weights
        self.reducer = GradReducer(group, enabled=data_parallel)
        # data parallel with the own NCCL communicator: the all-reduces are stream-ordered launches issued INSIDE the phases
        # (and therefore inside the captured graph); without it (a group that is not CUDA + NCCL) the eager step() calls
        # torch.distributed between its phases, and capture() refuses
        self._inline = self.reducer.comm is not None
        dev = self.G.flat.device
        self.device = dev
        # The learning rate lives on the DEVICE (next to FlatParams.step): the AdamW kernels read it when they run, so
        # the reference's per-epoch ExponentialLR(.999) (train.py:98-104,470-472) and the lr restored from a checkpoint
        # take effect in captured CUDA graphs as well.  `trainer.lr = x` updates both copies.
        self.base_lr = float(lr)                  # ExponentialLR's `initial_lr` (checkpoint interchange)
        self._lr = float(lr)
        self.lr_dev = torch.full((1,), float(lr), device=dev, dtype=torch.float32)
        self.slots = torch.zeros(8, device=dev, dtype=torch.float32)
        self.d_folds: Optional[Dict[int, passes.Folded]] = None
        self._d_persist: Dict[int, passes.Folded] = {}
        self._static = None
        self.x_pred: Optional[Tensor] = None
        # the discriminator passes on x_pred and on x_real are independent: they run on two streams (forked from and
        # joined back into the current stream, also under graph capture), which fills the SMs that the many
        # sub-148-tile kernels of the small discriminator layers leave idle
        self._side = torch.cuda.Stream(device=dev)
        self._side2 = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]   # per pass: the heavy sub-discriminator
        self._wg = [torch.cuda.Stream(device=dev) for _ in range(7)]                  # weight-gradient side streams
        self._ps = [torch.cuda.Stream(device=dev) for _ in range(2)]                  # period stacks dealt over these + their branch's stream
        self._ss = [torch.cuda.Stream(device=dev)]                                    # the same for the batched scale stacks
        self._sn = [torch.cuda.Stream(device=dev) for _ in range(4)]                  # spectral-norm fold chains, one per layer
        self._aux = torch.cuda.Stream(device=dev)                                     # time-domain loss beside the D passes
        self._enc = torch.cuda.Stream(device=dev)                                     # EMG-encoder losses beside the D passes
        self._comm = torch.cuda.Stream(device=dev)                                    # gradient all-reduces (own NCCL communicator)
        self._pend = torch.zeros(1, device=dev, dtype=torch.int32)                    # device flag: a generator AdamW is pending (fused graph)
        self._fused = None                                                            # (step graph, flush graph) of capture()
        self._pending_host = False
        self._d_slices = self._disc_grad_slices()
        self.g_buckets = generator_grad_buckets(self.G.offsets, self.G.numel, len(list(net_g.gblocks)) - 1)
        # without a data-parallel group there is nothing to overlap: one bucket (one fold-backward launch)
        if (grad_buckets if grad_buckets is not None else (3 if self.reducer.enabled else 1)) == 1:
            nblk = len(list(net_g.gblocks)) - 1
            self.g_buckets = [(0, nblk, 0, 5 * nblk + 2, (0, self.G.numel))]

    @property
    def lr(self) -> float:
        return self._lr

    @lr.setter
    def lr(self, value: float) -> None:
        self.flush()                              # a deferred generator AdamW of the previous step keeps ITS learning rate
        self._lr = float(value)
        self.lr_dev.fill_(self._lr)               # stream-ordered; graphs replayed after this read the new value

    def scheduler_step(self, gamma: float = 0.999) -> float:
        """One ExponentialLR step (train.py:98-104: gamma .999, stepped once per epoch at train.py:470-472)."""
        self.lr = self._lr * gamma
        return self._lr

    def _disc_grad_slices(self):
        """Discriminator gradient as three exchange pieces in the order its backward completes them: period stacks | coarse
        scale stacks (both "early") | the full-rate scale stack ("late": spectral norm, half of the backward work).  Each:
        (range of weight-normed convs in d_plan's table, slice of the flat gradient).  None when the discriminator does not
        have that shape (no spectral-norm stack between the period stacks and the remaining scale stacks)."""
        subs = passes.disc_subnets(self.net_d)
        heavy, rest = passes._heavy_split(subs)
        if len(heavy) != 1 or any(i > heavy[0] for i in rest if subs[i][0] == "P") or any(i < heavy[0] for i in rest if subs[i][0] == "S"):
            return None
        wn = self.d_plan.wn
        def item_range(mods):
            ids = [k for k, m in enumerate(wn) if any(m is c for d_ in mods for c in list(d_.layers) + [d_.output])]
            return (ids[0], ids[-1] + 1) if ids and ids == list(range(ids[0], ids[-1] + 1)) else None
        def grad_range(prefixes):
            offs = [o for nm, o in self.D.offsets.items() if nm.startswith(tuple(prefixes))]
            nxt = [o for nm, o in self.D.offsets.items() if o > max(offs) and not nm.startswith(tuple(prefixes))]
            return min(offs), (min(nxt) if nxt else self.D.numel)
        p_mods = [subs[i][1] for i in rest if subs[i][0] == "P"]
        s_mods = [subs[i][1] for i in rest if subs[i][0] == "S"]
        h_mods = [subs[heavy[0]][1]]
        names = {id(m): nm for nm, m in self.net_d.named_modules()}
        pre = lambda mods: [names[id(m)] + "." for m in mods]
        out = dict(early=[], late=None)
        for mods in (p_mods, s_mods):
            if mods:
                ir = item_range(mods)
                if ir is None:
                    return None
                out["early"].append((ir, grad_range(pre(mods))))
        ir = item_range(h_mods)
        if ir is None:
            return None
        out["late"] = (ir, grad_range(pre(h_mods)))
        # the three slices must tile the flat gradient exactly
        cover = sorted([g for _, g in out["early"]] + [out["late"][1]])
        if cover[0][0] != 0 or cover[-1][1] != self.D.numel or any(a[1] != b[0] for a, b in zip(cover, cover[1:])):
            return None
        return out

    def _fold_d(self, refold: bool):
        return passes.fold_discriminator(self.net_d, self.dtype, training=True, plan=self.d_plan, refold=refold,
                                         sn_streams=self._sn)

    def _reduce(self, flat_slice: Tensor):
        """Data parallel: all-reduce (sum) a slice of a flat gradient on the communication stream, ordered after
        everything enqueued on the current stream so far; returns the event to wait for before the slice is consumed
        (None without a data-parallel group).  Stream-ordered only - no host wait - so it is the same under capture."""
        if not self.reducer.enabled or flat_slice.numel() == 0:
            return None
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        self._comm.wait_event(ev)
        self.reducer.all_reduce_on(flat_slice, self._comm)
        done = torch.cuda.Event()
        done.record(self._comm)
        return done

    @staticmethod
    def _wait_events(evs) -> None:
        for e in evs:
            if e is not None:
                torch.cuda.current_stream().wait_event(e)

    def _fork(self) -> None:
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        self._side.wait_event(ev)

    def _join(self) -> None:
        ev = torch.cuda.Event()
        ev.record(self._side)
        torch.cuda.current_stream().wait_event(ev)

    # ------------------------------------------------------------------ phases
    # The fake and the real pass of a discriminator forward share their weights except in the spectral-norm
    # sub-discriminator (the full-rate scale stack: its sigma advances between the two forwards).  That stack runs once per
    # pass and all the others run ONCE, forward and backward, on the concatenated batch [x_pred | x_real]: half the
    # launches, twice the rows per launch (their layers have too few tiles to fill the chip), one weight-gradient
    # contraction over both.
    def _split_subs(self):
        subs = passes.disc_subnets(self.net_d)
        heavy, rest = passes._heavy_split(subs)
        return subs, heavy, [i for i in rest if subs[i][0] == "P"], [i for i in rest if subs[i][0] == "S"]

    def _disc_forward(self, x: Tensor, folds, idx: list, spread=None):
        """Forward of the sub-discriminators `idx` (none: (None, None)), dealt over the `spread` streams."""
        if not idx:
            return None, None
        return passes.discriminator_forward(self.net_d, x, self.dtype, folds, subset=idx, spread=spread)

    def _per_pass(self, heavy: list, fake_h, real_h, batched):
        """Per-pass views of every sub-discriminator's feature maps: the batched stacks (`batched`: pairs of a forward over
        [x_pred | x_real] and its indices) split behind x_pred's rows, the spectral-norm stack from its two own passes
        (fake_h, real_h).  Returns (fake maps, real maps, per-sub contexts of the fake pass); views only, no launches."""
        nd, Bq = len(passes.disc_subnets(self.net_d)), self.x_pred.shape[0]
        res_f, res_r, sub_f = [None] * nd, [None] * nd, [None] * nd
        for (r_b, c_b), idx in batched:
            if idx:
                a, b, sa = passes.split_disc_batch(r_b, c_b, idx, Bq)
                for i in idx:
                    res_f[i], res_r[i], sub_f[i] = a[i], b[i], sa[i]
        (rh_f, ch_f), (rh_r, _) = fake_h, real_h
        for i in heavy:
            res_f[i], res_r[i], sub_f[i] = rh_f[i], rh_r[i], ch_f.subs[i]
        return res_f, res_r, sub_f

    def _g_forward(self, su: Tensor, sess: Tensor, mode: Optional[Tensor], x_pred: Optional[Tensor] = None) -> None:
        self.slots.zero_()
        self.G.zero_grad(); self.D.zero_grad()
        self._gctx = None
        self._cur_su = su
        if x_pred is not None:            # discriminator-only workload (disc_losses_step): the fake batch is an input
            self.x_pred = x_pred
            return
        self.x_pred, self._gctx = passes.generator_forward(self.net_g, su, sess, mode, self.dtype, True, folds=self.g_plan.fold(),
                                                           side=self._side2[1] if self.use_adv else None)

    def _d_update(self, fake_h, real_h, p_b, s_b) -> None:
        """loss_D of the two passes, its backward (weight gradients only) and the data-parallel exchange of the
        discriminator gradient."""
        dt = self.dtype
        subs, heavy, p_idx, s_idx = self._split_subs()
        ch_f, ch_r, cp, cs = fake_h[1], real_h[1], p_b[1], s_b[1]
        Bq, nd = self.x_pred.shape[0], len(subs)
        res_f, res_r, _ = self._per_pass(heavy, fake_h, real_h, ((p_b, p_idx), (s_b, s_idx)))
        self._last_d_fmaps = (res_f, res_r, ch_f)      # kept for the parity tests (references only)
        # loss_D = sum_i mse(fake_i, 0) + mse(real_i, 1) and its gradients, one launch      train.py:192-196
        # (batched stacks: the two gradients land in the two halves of one [2B, rows, 1] tensor)
        dcat = {i: torch.empty((2 * Bq,) + tuple(res_f[i][-1].shape[1:]), device=self.device, dtype=dt) for i in p_idx + s_idx}
        outs = [dcat[i][:Bq] if i in dcat else None for i in range(nd)] + [dcat[i][Bq:] if i in dcat else None for i in range(nd)]
        dl = ops.mse_const_multi([fm[-1] for fm in res_f] + [fm[-1] for fm in res_r], [0.0] * nd + [1.0] * nd, self.slots,
                                 [0] * (2 * nd), 1.0, dt, outs=outs)
        dl_f, dl_r = dl[:nd], dl[nd:]
        dl_b = [dcat.get(i) for i in range(nd)]
        # every pass / stack accumulates its packed weight gradients in the plan's arena; the weight-norm backward is
        # linear in them, so it runs once (spectral-norm layers un-fold per pass: their sigma differs)
        self.d_plan.zero()
        cur = torch.cuda.current_stream()
        # four backward branches, each with its own weight-gradient side stream
        self.d_plan.async_wgrads({st.cuda_stream: w for st, w in zip((cur, self._side, self._side2[0], self._side2[1], *self._ps, *self._ss), self._wg)})
        bwd = lambda ctx, dlog: passes.discriminator_backward(self.net_d, ctx, dlog, None, want_input_grad=False,
                                                              want_weight_grad=True, plan=self.d_plan,
                                                              spread=self._ps if ctx is cp else (self._ss if ctx is cs else None)) if ctx is not None else None
        only = lambda dlog, idx: [dlog[i] if i in idx else None for i in range(nd)]
        self._fork()
        with torch.cuda.stream(self._side):       # side: spectral-norm stack, fake | its side: spectral-norm stack, real
            passes.fork_join(self._side2[0], lambda: bwd(ch_r, only(dl_r, heavy)), lambda: bwd(ch_f, only(dl_f, heavy)))
        # current: P stacks, batched | its side: S stacks, batched
        passes.fork_join(self._side2[1], lambda: bwd(cs, only(dl_b, s_idx)), lambda: bwd(cp, only(dl_b, p_idx)))
        early = []
        if self._inline and heavy and self._d_slices is not None:
            # data parallel: the period stacks and the two coarse scale stacks are through (the spectral-norm stack, half
            # of the work, still runs on the side stream): make THEIR gradients final and exchange them now, so that only
            # the spectral-norm stack's share of the 47 MB is left exposed behind the backward pass
            self.d_plan.join_wgrads_of([cur, self._side2[1], *self._ps, *self._ss])
            for (i_lo, i_hi), (g_lo, g_hi) in self._d_slices["early"]:
                self.d_plan.backward_range(i_lo, i_hi, accumulate=False)
                early.append(self._reduce(self.D.grad[g_lo:g_hi]))
        self._join()
        self.d_plan.join_wgrads()
        if early:
            (i_lo, i_hi), (g_lo, g_hi) = self._d_slices["late"]
            self.d_plan.backward_range(i_lo, i_hi, accumulate=False)
            self._wait_events(early + [self._reduce(self.D.grad[g_lo:g_hi])])
            return
        self.d_plan.backward(accumulate=False)    # the only contribution since zero_grad: overwrite
        if self._inline:
            # data parallel, one piece right behind the backward: everything that follows (D AdamW, phase G) depends on it
            self._wait_events([self._reduce(self.D.grad)])

    def _phase_d(self, su: Tensor, sess: Tensor, mode: Optional[Tensor], x_real: Tensor, x_pred: Optional[Tensor] = None,
                 head=None) -> None:
        """Phase D.  The discriminator folds and the real pass of the spectral-norm stack need neither the generator nor
        x_pred: they run on the side stream while the current stream runs `head`, the generator fold + forward and - once
        the fake pass's folds are there - the fake pass.  `head` (captured step): the pending generator update of the
        previous step."""
        head = head or (lambda: None)
        if not self.use_adv:
            head()
            self._g_forward(su, sess, mode, x_pred)
            return
        _, heavy, p_idx, s_idx = self._split_subs()
        cur = torch.cuda.current_stream()
        self._fork()
        with torch.cuda.stream(self._side):
            # folds of the fake pass (f1) and of the real pass (f2): the spectral-norm power iterations of the two
            # forwards happen in that order (train.py:190-191)
            refold_d = not self._d_folded
            self._d_folded = True
            f1 = self._fold_d(refold_d)
            ev_f1 = torch.cuda.Event()
            ev_f1.record(self._side)
            f2 = self._fold_d(False)
            real_h = self._disc_forward(x_real, f2, heavy)
        head()
        self._g_forward(su, sess, mode, x_pred)
        cur.wait_event(ev_f1)
        x_cat = torch.cat([self.x_pred, x_real], 0)
        # current: fake pass of the spectral-norm stack | side2[1]: S stacks batched | side2[0]: P stacks batched
        (s_b, p_b), fake_h = passes.fork_join(
            self._side2[1], lambda: passes.fork_join(self._side2[0], lambda: self._disc_forward(x_cat, f1, p_idx, self._ps),
                                                     lambda: self._disc_forward(x_cat, f1, s_idx, self._ss))[::-1],
            lambda: self._disc_forward(self.x_pred, f1, heavy))
        self._join()
        self._d_update(fake_h, real_h, p_b, s_b)

    def _phase_g_head(self, x_real: Tensor, update_d: bool = True) -> None:
        """Phase G up to and including the generator backward of the first (rearmost) gradient bucket."""
        dx_pred = self._g_losses(x_real, update_d)
        # generator backward, bucket by bucket (G.grad was zeroed in phase D and this is its only writer: overwrite)
        self._last_gctx = self._gctx                       # kept for the parity tests (references only)
        self._gb = passes.GenBackward(self.net_g, self._gctx, dx_pred, plan=self.g_plan, side=self._side2[1], res_side=self._side2[0],
                                      overwrite_grads=True)
        self._g_bucket(0)

    def _g_losses(self, x_real: Tensor, update_d: bool = True) -> Tensor:
        """Phase G in front of the generator: D optimiser step, the two discriminator passes with the updated weights,
        adv + 15 TD + 7 FM (train.py:206-217,257-263) and their gradient w.r.t. x_pred (returned, fp32 [B,T,C])."""
        dt = self.dtype
        x_pred = self.x_pred
        dx_pred = torch.zeros_like(x_pred)
        td_ev = None
        enc_ev, dx_enc = None, None
        if self.use_su or self.use_ph:
            # EMG-encoder perceptual losses (train.py:219-230): frozen encoder forward on x_pred, speech-unit distance to the
            # step's own input units and phoneme cross-entropy, gradient w.r.t. x_pred.  Independent of the discriminator:
            # on its own stream beside the discriminator passes.
            from . import passes_encoder as pe
            if self._cur_ph is None:
                raise ValueError("the phoneme loss needs phoneme_targets ([B, frames] int64) in step() / step_graph()")
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            self._enc.wait_event(ev)
            with torch.cuda.stream(self._enc):
                dx_enc, self._enc_units, self._enc_logits = pe.encoder_losses(
                    self._enc_plan, x_pred, self._cur_su, self._cur_ph, self.slots[6:8], self.w_su, self.w_ph, True,
                    self.use_su, self.use_ph)
                enc_ev = torch.cuda.Event()
                enc_ev.record(torch.cuda.current_stream())
        if self.use_td and self.use_adv:
            # the time-domain loss needs only x_real / x_pred: it runs on its own stream beside the discriminator passes
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            self._aux.wait_event(ev)
            with torch.cuda.stream(self._aux):
                ops.td_loss(x_real, x_pred, self.slots[3:6], [self.w_td] * 3, dx_pred)   # train.py:215-216
                td_ev = torch.cuda.Event()
                td_ev.record(self._aux)
        if self.use_adv:
            if update_d:
                self.D.adamw(self.lr_dev, grad_scale=self.reducer.grad_scale)   # train.py:199
            refold_d = update_d or not self._d_folded
            self._d_folded = True
            # the split of phase D: the spectral-norm stack once per pass (fake on the side stream, real after the second
            # power iteration), all the others once on [x_pred | x_real]
            _, heavy, p_idx, s_idx = self._split_subs()
            f3 = self._fold_d(refold_d)
            x_cat = torch.cat([x_pred, x_real], 0)
            self._fork()
            with torch.cuda.stream(self._side):       # side: fake pass of the spectral-norm stack | its side: S stacks, batched
                s_b, fake_h = passes.fork_join(self._side2[0], lambda: self._disc_forward(x_cat, f3, s_idx, self._ss),
                                               lambda: self._disc_forward(x_pred, f3, heavy))
            f4 = self._fold_d(False)                  # current: second power iteration, then real pass of that stack | P stacks, batched
            real_h, p_b = passes.fork_join(self._side2[1], lambda: self._disc_forward(x_real, f4, heavy),
                                           lambda: self._disc_forward(x_cat, f3, p_idx, self._ps))
            self._join()
            res_f, res_r, sub_f = self._per_pass(heavy, fake_h, real_h, ((p_b, p_idx), (s_b, s_idx)))
            assert all(r is not None for r in res_f)
            ctx_f = passes.DiscCtx(B=x_pred.shape[0], T=x_pred.shape[1], C=x_pred.shape[2], dtype=dt, folds=f3, subs=sub_f)
            ctx_f.keep = (fake_h[1], p_b[1], s_b[1], x_cat)
            self.d_folds = f4
            self._last_g_fmaps = (res_f, res_r)             # kept for the parity tests (references only)
            nd = len(res_f)
            dlog = ops.mse_const_multi([fm[-1] for fm in res_f], [1.0] * nd, self.slots, [1] * nd, 1.0, dt)   # train.py:210-211
            if self.use_fm:                                                 # train.py:259-262, one launch for all 27 maps
                pairs = [(a, b) for fm_f, fm_r in zip(res_f, res_r) for a, b in zip(fm_f[:-1], fm_r[:-1])]
                grads = ops.l1_mean_multi(pairs, self.slots[2:3], self.w_fm)
                dfm, i = [], 0
                for fm_f in res_f:
                    dfm.append(grads[i:i + len(fm_f) - 1]); i += len(fm_f) - 1
            else:
                dfm = [[None] * (len(fm_f) - 1) for fm_f in res_f]
            dx_d = passes.discriminator_backward(self.net_d, ctx_f, dlog, dfm, want_input_grad=True, want_weight_grad=False,
                                                 side=self._side2[0], spread=self._ps)
            if td_ev is not None:
                torch.cuda.current_stream().wait_event(td_ev)
            ops.axpy_f32(dx_pred, dx_d, 1.0)
        if self.use_td and td_ev is None:
            ops.td_loss(x_real, x_pred, self.slots[3:6], [self.w_td] * 3, dx_pred)   # train.py:215-216
        if dx_enc is not None:
            torch.cuda.current_stream().wait_event(enc_ev)
            ops.axpy_f32(dx_pred, dx_enc, 1.0)
        return dx_pred

    def _g_bucket(self, i: int) -> None:
        """Backward of the GBlocks of generator-gradient bucket i (after it, self.G.grad[slice i] is final)."""
        lo, hi, c_lo, c_hi, _ = self.g_buckets[i]
        gb = self._gb
        gb.blocks(lo, hi)
        if i == len(self.g_buckets) - 1:
            gb.finish()
        gb.bucket(c_lo, c_hi, last=i == len(self.g_buckets) - 1)
        if i == len(self.g_buckets) - 1:
            self._gb = self._gctx = None

    def _phase_g(self, x_real: Tensor, update_d: bool = True, reduce: bool = False) -> list:
        """Phase G; with reduce=True the all-reduce of each generator-gradient bucket is issued as soon as the bucket is
        final (it then overlaps the backward of the buckets in front of it).  Returns the pending all-reduce handles
        (own communicator: events)."""
        handles = []
        self._phase_g_head(x_real, update_d)
        for i in range(len(self.g_buckets)):
            if i > 0:
                self._g_bucket(i)
            if reduce:
                handles += self._reduce_g_bucket(i)
        return handles

    def _reduce_g_bucket(self, i: int) -> list:
        lo, hi = self.g_buckets[i][4]
        if self._inline:
            return [self._reduce(self.G.grad[lo:hi])]
        return self.reducer.all_reduce_async(self.G.grad[lo:hi]) if hi > lo else []

    def _wait_handles(self, handles) -> None:
        if self._inline:
            self._wait_events(handles)
        else:
            self.reducer.wait(handles)

    def _phase_opt_g(self) -> None:
        self.G.adamw(self.lr_dev, grad_scale=self.reducer.grad_scale)       # train.py:267

    def _opt_g_head(self) -> None:
        """Fused graph: the part of the generator update that the PREVIOUS replay left pending - exchange of the LAST
        gradient bucket (deferred so that it, too, runs beside work that does not depend on the generator), then AdamW of
        that bucket's slice under the device flag `_pend` (a no-op on the first replay and after flush(), which runs the
        same launches on its own).  The other buckets were updated inside the previous replay, each right behind its
        all-reduce (_fused_step), so what is left here is short enough to hide behind the discriminator folds."""
        n = len(self.g_buckets)
        lo, hi = self.g_buckets[n - 1][4]
        if self._inline:
            self._wait_events(self._reduce_g_bucket(n - 1))
        self.G.adamw(self.lr_dev, grad_scale=self.reducer.grad_scale, enable=self._pend, lo=lo, hi=hi, keep_step=n > 1)

    def _fused_step(self, s: dict) -> None:
        """The whole train step as ONE capturable sequence (no host-side seam): pending generator update of the previous
        step beside the discriminator folds / real pass -> phase D -> phase G.  Every generator-gradient bucket but the
        last is exchanged AND applied (AdamW on its slice of the flat buffers) on the communication stream while the
        buckets in front of it are still in their backward pass - the backward reads the packed operands, not the fp32
        master weights, so updating them early is safe; the last bucket is left pending (_opt_g_head)."""
        self._phase_d(s["su"], s["sess"], s["mode"], s["x_real"], head=self._opt_g_head)
        self._phase_g_head(s["x_real"])
        n, evs = len(self.g_buckets), []
        for i in range(n - 1):
            if i > 0:
                self._g_bucket(i)
            lo, hi = self.g_buckets[i][4]
            ev = self._reduce(self.G.grad[lo:hi])
            if ev is None:                      # no data-parallel group: the slice is final now, fork the side stream here
                ev = torch.cuda.Event()
                ev.record(torch.cuda.current_stream())
                self._comm.wait_event(ev)
            with torch.cuda.stream(self._comm):
                self.G.adamw(self.lr_dev, grad_scale=self.reducer.grad_scale, lo=lo, hi=hi, keep_step=i > 0)
                done = torch.cuda.Event()
                done.record(self._comm)
            evs.append(done)
        if n > 1:
            self._g_bucket(n - 1)
        self._wait_events(evs)
        self._pend.fill_(1)

    # ------------------------------------------------------------------ public API
    def step(self, speech_units: Tensor, session_ids: Tensor, x_real: Tensor,
             speaking_mode_ids: Optional[Tensor] = None, phoneme_targets: Optional[Tensor] = None) -> Tensor:
        """One train step on device tensors (eager launches).  Returns the loss-slot tensor (device, fp32[8]):
        see LOSS_NAMES; no host synchronisation happens here."""
        self.flush()
        su = speech_units.contiguous().float()
        xr = x_real.contiguous().float()
        self._cur_ph = phoneme_targets
        self._phase_d(su, session_ids, speaking_mode_ids, xr)
        if not self._inline:
            self.reducer.all_reduce(self.D.grad)
        self._wait_handles(self._phase_g(xr, reduce=True))
        self._phase_opt_g()
        return self.slots

    def disc_losses_step(self, x_pred: Tensor, x_real: Tensor) -> Tensor:
        """BASELINE.json configs[4]: the discriminator stacks + multi-TD + feature-matching + LSGAN losses of one train
        step in isolation, forward and backward - everything of train.py:189-264 except the generator: phase D on the
        given fake batch (two passes, loss_D, weight gradients, D AdamW), then phase G's two passes with the updated
        weights, the three losses and their gradient w.r.t. x_pred, which is returned (fp32 [B,T,C]).  Eager launches;
        capturable into one CUDA graph (no collective: single-process workload)."""
        self._phase_d(None, None, None, x_real, x_pred=x_pred)
        return self._g_losses(x_real, update_d=True)

    def capture(self, batch: int, frames: int, unit_dim: int = 256, hop: int = 16, channels: int = 8) -> None:
        """Capture the whole step (_fused_step) as ONE CUDA graph over static input buffers, plus the graph that flush()
        replays.  With the own NCCL communicator the gradient all-reduces are graph nodes too, so a replay has no
        host-side seam; data parallelism over any other process group is refused (train with step() there).  The
        generator update of step k is left pending on the device (flag `_pend`) and runs at the head of replay k+1,
        beside that step's discriminator folds and real pass, which depend on neither the generator nor its gradient;
        flush() applies a pending update on its own (the eager step(), checkpointing, `lr` changes and the inference
        engine call it).

        Two eager warm-up steps run first (allocator / lazy-initialisation warm-up, on all-zero inputs); the trainer's
        state - parameters, AdamW moments and step counters, spectral-norm u / v, loss slots - is snapshotted before and
        restored after them, so capture() leaves the training state exactly as it found it (resume-then-capture is
        safe, and `steps` in the next checkpoint still counts real steps only)."""
        if self.reducer.enabled and not self._inline:
            raise RuntimeError("GanTrainer.capture: data-parallel graph capture needs the own NCCL communicator, i.e. a "
                               "process group with the nccl backend on CUDA devices; train with step() over this group")
        dev = self.device
        self.flush()
        self._fused = None
        self._static = dict(
            su=torch.zeros(batch, frames, unit_dim, device=dev), sess=torch.zeros(batch, device=dev, dtype=torch.int64),
            x_real=torch.zeros(batch, frames * hop, channels, device=dev),
            mode=torch.zeros(batch, device=dev, dtype=torch.int64) if self.net_g.use_speaking_mode_embedding else None,
            ph=torch.zeros(batch, frames, device=dev, dtype=torch.int64) if (self.use_su or self.use_ph) else None)
        s = self._static
        self._cur_ph = s["ph"]
        snap = self._snapshot_state()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                self.step(s["su"], s["sess"], s["x_real"], s["mode"], s["ph"])
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self._restore_state(snap)
        torch.cuda.synchronize()
        gkw = dict(pool=torch.cuda.graph_pool_handle())
        if self.reducer.enabled:      # the process group's watchdog thread may touch the CUDA API while we capture
            gkw["capture_error_mode"] = "thread_local"
        # Data parallel: the persistent conv / wgrad kernels take one CTA per SM with (nearly) the whole register file,
        # so a concurrent NCCL kernel only finds room on SMs that a launch leaves idle - measured at N = 8, the
        # all-reduces then cost their full stand-alone time (0.67 ms for the 141 MB of a step) however they are
        # overlapped.  STG_NCCL_SMS=R keeps R SMs free of them for the communicator inside this graph.
        # Measured at N = 2 (bench.py, ms per step): R = 0: 4.32, 8: 4.70 (with 8 NCCL channels), 16: 4.25, 24: 4.31; capping
        # NCCL's channel count to R always lost.  Default 16.
        import os
        from . import _lib
        reserve = int(os.environ.get("STG_NCCL_SMS", "16")) if self.reducer.enabled else 0
        n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        step_g, flush_g = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        self._pend.zero_()
        if reserve > 0:
            _lib.load().stg_set_sm_limit(n_sm - reserve)
        try:
            with torch.cuda.graph(step_g, **gkw):
                self._fused_step(s)
        finally:
            if reserve > 0:
                _lib.load().stg_set_sm_limit(0)
        with torch.cuda.graph(flush_g, **gkw):
            self._opt_g_head()
        self._pend.zero_()
        self._fused, self._pending_host = (step_g, flush_g), False

    def _sn_buffers(self) -> list:
        return [b for c in passes.discriminator_convs(self.net_d) if c.norm != "weight_norm" for b in (c.weight_u, c.weight_v)]

    def _snapshot_state(self) -> dict:
        return dict(flat=[(fp, fp.flat.clone(), fp.m.clone(), fp.v.clone(), fp.step.clone()) for fp in (self.G, self.D)],
                    sn=[(b, b.clone()) for b in self._sn_buffers()], slots=self.slots.clone())

    def _restore_state(self, snap: dict) -> None:
        for fp, flat, m, v, step in snap["flat"]:
            fp.flat.copy_(flat); fp.m.copy_(m); fp.v.copy_(v); fp.step.copy_(step)
            fp.grad.zero_()
        for b, val in snap["sn"]:
            b.copy_(val)
        self.slots.copy_(snap["slots"])
        self._pend.zero_()
        self._pending_host = False
        self.refold()

    def refold(self) -> None:
        """Re-pack the weight-normed discriminator convs from the current weights, eagerly.  Inside the captured step the
        discriminator packs are refreshed right after ITS optimiser step (phase G) and phase D of the next step reuses
        them, so anything that changes the weights from outside - a checkpoint load, the state restore of capture() -
        must re-pack here.  (The generator re-packs at the start of every step.)"""
        self.d_plan.fold()
        self._d_folded = True

    def flush(self) -> None:
        """Complete the generator update that the last step_graph() left pending: exchange of the last gradient bucket
        (data parallel) and its AdamW, under the device flag `_pend`, which it clears."""
        if self._pending_host:
            self._pending_host = False
            self._fused[1].replay()

    def step_graph(self, speech_units: Tensor, session_ids: Tensor, x_real: Tensor,
                   speaking_mode_ids: Optional[Tensor] = None, phoneme_targets: Optional[Tensor] = None) -> Tensor:
        """Replay the captured step; inputs may be pinned-host or device tensors (copied into the static buffers).
        The generator update of this step stays pending until the next replay or flush()."""
        s = self._static
        s["su"].copy_(speech_units, non_blocking=True)
        s["sess"].copy_(session_ids, non_blocking=True)
        s["x_real"].copy_(x_real, non_blocking=True)
        if s["mode"] is not None:
            if speaking_mode_ids is None:
                raise ValueError("step_graph: this generator uses speaking-mode embeddings - pass speaking_mode_ids")
            s["mode"].copy_(speaking_mode_ids, non_blocking=True)
        if s["ph"] is not None:
            if phoneme_targets is None:
                raise ValueError("step_graph: the EMG-encoder losses are on - pass phoneme_targets")
            s["ph"].copy_(phoneme_targets, non_blocking=True)
        self._fused[0].replay()
        self._pending_host = True
        return self.slots

    def save_checkpoint(self, directory, steps: int, epoch: int, final: bool = False) -> None:
        """The reference's netG-/netD-/checkpoint-{steps:08d}.pt triple (train.py:421-436), optimiser state in
        torch.optim.AdamW format - see checkpoint.py."""
        from . import checkpoint
        checkpoint.save_checkpoint(self, directory, steps, epoch, final)

    def load_latest_checkpoint(self, directory):
        """Resume from the newest triple in `directory` (utils/common.py:23-61), written by either loop.
        Returns (start_epoch, steps)."""
        from . import checkpoint
        return checkpoint.load_latest_checkpoint(self, directory)

    def losses(self) -> Dict[str, float]:
        """Host read of the loss slots (synchronises)."""
        v = self.slots.tolist()
        out = dict(zip(LOSS_NAMES, v[:8]))
        out["loss_td"] = v[3] + v[4] + v[5]
        out["loss_g"] = v[1] + self.w_td * out["loss_td"] + self.w_fm * v[2] + \
            (self.w_su * v[6] if self.use_su else 0.0) + (self.w_ph * v[7] if self.use_ph else 0.0)
        return out
