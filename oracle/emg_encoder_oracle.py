"""CPU ORACLE (test infrastructure only) for the next hot-path row, SURVEY.md section 8f rank 1: the frozen EMG encoder's
forward and the two perceptual losses the generator step takes through it.  Product code must not import this module.

Every function restates the reference algorithm with explicit tensor formulas and cites the file:line it follows
(paths under /root/reference):

  emg_encoder_forward   ste_gan/models/emg_encoder.py:71-88   (EMGEncoderTransformer.forward, eval mode)
  res_block             ste_gan/layers/conv.py:106-132         (ResBlock with BatchNorm in eval mode)
  encoder_layer         ste_gan/layers/transformer.py:45-60    (post-norm TransformerEncoderLayer)
  attention             ste_gan/layers/transformer.py:87-113   (per-head projections, relative positional logits)
  relative_logits       ste_gan/layers/transformer.py:163-306  (LearnedRelativePositionalEmbedding, unmasked, per head)
  encoder_losses        ste_gan/losses/emg_encoder_loss.py:63-84

Pinned by tests/golden/emg_encoder_tiny.pt (oracle/make_golden.py; the reference pins torch 2.0.1 - under this
container's torch 2.11 `nn.TransformerEncoder.forward` no longer accepts the reference's custom layer, so the fixture
generator applies `encoder.transformer.layers` one after the other, which is what the 2.0.1 container does for a stack
without masks and without a final norm).  The CUDA implementation (ste_gan_b200/passes_encoder.py, csrc/encoder.cu) is
checked against this oracle and the fixture by tests/test_encoder_gpu.py.
"""
from __future__ import annotations

from typing import Dict, Tuple

import torch
import torch.nn.functional as F

Tensor = torch.Tensor
StateDict = Dict[str, Tensor]
BN_EPS, LN_EPS = 1e-5, 1e-5
MAX_REL = 100          # relative_positional_distance (emg_encoder.py:64)

# tests/golden/emg_encoder_tiny.pt holds the reference's outputs only: the weights and inputs they were computed from are
# drawn from seeds by the two functions below, for the reference module (oracle/make_golden.py) and for the tests alike
TINY_ENCODER = dict(model_size=32, num_extra_res_blocks=3, num_transformer_layers=2)
TINY_CASE_SHAPES = ((2, 400, 8), (1, 1776, 8))          # 25 frames; 111 frames (> 100: out-of-range relative positions)


def tiny_encoder_state(encoder_cls) -> StateDict:
    """Weights of the fixture encoder, as halves: the seed-0 initialisation of encoder_cls(8, 256, 48, **TINY_ENCODER) (the
    reference's EMGEncoderTransformer, or the drop-in, which initialises bit-identically), then non-trivial BatchNorm
    statistics (a trained checkpoint has them), everything rounded to the fp16 grid."""
    torch.manual_seed(0)
    enc = encoder_cls(8, 256, 48, **TINY_ENCODER)
    with torch.no_grad():
        for mod in enc.modules():
            if isinstance(mod, torch.nn.BatchNorm1d):
                mod.running_mean.normal_(0, 0.3); mod.running_var.uniform_(0.5, 1.5)
                mod.weight.uniform_(0.5, 1.5); mod.bias.normal_(0, 0.2)
    return {k: (v.half() if v.is_floating_point() else v.clone()) for k, v in enc.state_dict().items()}


def tiny_case_inputs(i: int) -> Tuple[Tensor, Tensor, Tensor]:
    """Fixture case i: EMG input [B, T, 8] in (-1, 1), speech-unit targets [B, T/16, 256], phoneme labels [B, T/16]."""
    B, T, C = TINY_CASE_SHAPES[i]
    g = torch.Generator().manual_seed(20 + i)
    x = torch.tanh(torch.randn(B, T, C, generator=g))
    return x, torch.randn(B, T // 16, 256, generator=g), torch.randint(0, 48, (B, T // 16), generator=g)


def _bn_eval(sd: StateDict, p: str, x: Tensor) -> Tensor:
    """BatchNorm1d in eval mode on [B,C,T] (conv.py:112,114,118)."""
    scale = sd[p + ".weight"] / torch.sqrt(sd[p + ".running_var"] + BN_EPS)
    return (x - sd[p + ".running_mean"][None, :, None]) * scale[None, :, None] + sd[p + ".bias"][None, :, None]


def _relu(x: Tensor, mask) -> Tensor:
    """ReLU; with `mask` (bool, same shape) the BACKWARD uses its sign pattern (ste_gan_oracle._ActWithMask: parity tests
    feed the implementation-under-test's own pattern so that both differentiate the same piecewise-linear branch)."""
    if mask is None:
        return F.relu(x)
    from oracle.ste_gan_oracle import _act
    return _act(x, 0.0, mask)


def res_block(sd: StateDict, p: str, x: Tensor, stride: int, masks=None) -> Tensor:
    """conv.py:122-132: relu(bn2(conv2(relu(bn1(conv1 x)))) + res), res = res_norm(1x1 strided conv x) or x."""
    m = masks if masks is not None else (None, None)
    y = _relu(_bn_eval(sd, p + ".bn1", F.conv1d(x, sd[p + ".conv1.weight"], sd[p + ".conv1.bias"], stride=stride, padding=1)), m[0])
    y = _bn_eval(sd, p + ".bn2", F.conv1d(y, sd[p + ".conv2.weight"], sd[p + ".conv2.bias"], padding=1))
    if p + ".residual_path.weight" in sd:
        res = _bn_eval(sd, p + ".res_norm", F.conv1d(x, sd[p + ".residual_path.weight"], sd[p + ".residual_path.bias"], stride=stride))
    else:
        res = x
    return _relu(y + res, m[1])


def relative_logits(q: Tensor, emb: Tensor) -> Tensor:
    """Positional logits of an unmasked, per-head learned relative embedding (transformer.py:163-306).
    q: [B,H,L,d]; emb: [H, 2*MAX_REL-1, d] (the parameter's trailing singleton removed).
    logits[b,h,i,j] = q[b,h,i] . emb[h, (j - i) + MAX_REL - 1] for |j - i| < MAX_REL.  Beyond that distance the
    reference pads the table with zero embeddings and subtracts 1e8 from those logits (:262-268); its pad / view
    re-indexing (:287-300) is the standard relative -> absolute skew and equals this direct gather."""
    B, H, L, d = q.shape
    idx = torch.arange(L)[None, :] - torch.arange(L)[:, None]                 # j - i
    ok = idx.abs() < MAX_REL
    table = torch.einsum("bhid,hmd->bhim", q, emb)                             # all relative positions
    gathered = torch.gather(table, 3, (idx.clamp(-(MAX_REL - 1), MAX_REL - 1) + MAX_REL - 1)[None, None].expand(B, H, L, L))
    return torch.where(ok[None, None], gathered, torch.full_like(gathered, -1e8))


def attention(sd: StateDict, p: str, x: Tensor) -> Tensor:
    """transformer.py:87-113 on x [B,L,D] (batch-first here; the reference is time-first)."""
    w_q, w_k, w_v, w_o = (sd[p + n] for n in (".w_q", ".w_k", ".w_v", ".w_o"))    # [H,D,d] x3, [H,d,D]
    q = torch.einsum("blf,hfa->bhla", x, w_q)
    k = torch.einsum("blf,hfa->bhla", x, w_k)
    v = torch.einsum("blf,hfa->bhla", x, w_v)
    logits = torch.einsum("bhqa,bhka->bhqk", q, k) / (w_q.shape[2] ** 0.5)
    logits = logits + relative_logits(q, sd[p + ".relative_positional.embeddings"][..., 0])
    probs = torch.softmax(logits, dim=-1)
    return torch.einsum("bhta,haf->btf", torch.einsum("bhqk,bhka->bhqa", probs, v), w_o)


def encoder_layer(sd: StateDict, p: str, x: Tensor, mask=None) -> Tensor:
    """transformer.py:54-60 (dropout is the identity in eval mode)."""
    D = x.shape[-1]
    x = F.layer_norm(x + attention(sd, p + ".self_attn", x), (D,), sd[p + ".norm1.weight"], sd[p + ".norm1.bias"], LN_EPS)
    ff = F.linear(_relu(F.linear(x, sd[p + ".linear1.weight"], sd[p + ".linear1.bias"]), mask), sd[p + ".linear2.weight"], sd[p + ".linear2.bias"])
    return F.layer_norm(x + ff, (D,), sd[p + ".norm2.weight"], sd[p + ".norm2.bias"], LN_EPS)


def emg_encoder_forward(sd: StateDict, emg: Tensor, masks=None) -> Tuple[Tensor, Tensor]:
    """emg_encoder.py:71-88 in eval mode: emg [B,T,C] -> (speech-unit prediction [B,T/16,256], phoneme logits [B,T/16,P]).
    masks (parity tests): dict(blocks=[(inner ReLU [B,C,T], output ReLU [B,C,T]) per ResBlock], layers=[FFN ReLU [B,L,F]])."""
    x = emg.transpose(1, 2)
    i = 0
    while f"conv_blocks.{i}.conv1.weight" in sd:
        x = res_block(sd, f"conv_blocks.{i}", x, stride=2, masks=masks["blocks"][i] if masks else None)   # every block: stride 2 (:50-53)
        i += 1
    x = F.linear(x.transpose(1, 2), sd["w_raw_in.weight"], sd["w_raw_in.bias"])
    i = 0
    while f"transformer.layers.{i}.linear1.weight" in sd:
        x = encoder_layer(sd, f"transformer.layers.{i}", x, masks["layers"][i] if masks else None)
        i += 1
    return F.linear(x, sd["w_out.weight"], sd["w_out.bias"]), F.linear(x, sd["w_aux.weight"], sd["w_aux.bias"])


def encoder_losses(unit_pred: Tensor, phoneme_logits: Tensor, unit_target: Tensor, phoneme_target: Tensor) -> Tuple[Tensor, Tensor]:
    """emg_encoder_loss.py:63-84: mean pairwise L2 distance over (b t) rows - F.pairwise_distance adds eps = 1e-6 to the
    difference before the norm - and cross-entropy over the phoneme classes."""
    diff = unit_target.reshape(-1, unit_target.shape[-1]) - unit_pred.reshape(-1, unit_pred.shape[-1]) + 1e-6
    unit_loss = diff.pow(2).sum(-1).sqrt().mean()
    logp = torch.log_softmax(phoneme_logits, dim=-1)
    ce = -logp.gather(-1, phoneme_target[..., None]).mean()
    return unit_loss, ce
