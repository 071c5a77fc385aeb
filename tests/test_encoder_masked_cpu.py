"""CPU: the argument checks of the length-masked encoder entry points (they run before any CUDA call), the host-side checks of
the masked encoder forward, and the arithmetic of aggregate_scores."""
import ctypes as C
import math
from types import SimpleNamespace

import pytest
import torch

EINVAL, EUNSUPPORTED = -1, -3


def _buf():
    return C.cast((C.c_float * 16)(), C.c_void_p)


def _attn(lib, band, **kw):
    a = dict(qkv=_buf(), dtype=0, emb=_buf(), B=2, L=100, H=8, d=96, M=100, o=_buf(), probs=_buf(), lengths=_buf())
    a.update(kw)
    fn = lib.stg_relattn_band_fwd_masked if band else lib.stg_relattn_fwd_masked
    return fn(a["qkv"], a["dtype"], a["emb"], a["B"], a["L"], a["H"], a["d"], a["M"], 0.1, a["o"], a["probs"], a["lengths"], None)


BAD = [dict(lengths=None), dict(qkv=None), dict(emb=None), dict(o=None), dict(probs=None), dict(d=6), dict(d=0), dict(L=0),
       dict(M=0), dict(B=0), dict(H=0), dict(dtype=2)]
BAD_IDS = ["no_lengths", "no_qkv", "no_emb", "no_o", "no_probs", "d6", "d0", "L0", "M0", "B0", "H0", "dtype2"]


@pytest.mark.parametrize("bad", BAD, ids=BAD_IDS)
@pytest.mark.parametrize("band", [False, True], ids=["dense", "band"])
def test_masked_attention_rejects_bad_arguments(band, bad):
    """(The pointers are dummies: the call must return before it touches the device.)"""
    from ste_gan_b200 import _lib
    assert _attn(_lib.load(), band, **bad) == EINVAL


def test_masked_attention_keeps_the_bounds_of_the_unmasked_calls():
    from ste_gan_b200 import _lib
    lib = _lib.load()
    assert _attn(lib, False, L=207) == EUNSUPPORTED                 # the dense kernel's shared-memory limit at d = 96
    assert _attn(lib, True, d=132) == EUNSUPPORTED and _attn(lib, True, M=257) == EUNSUPPORTED


def _scores(lib, **kw):
    a = dict(pred=_buf(), tgt=_buf(), logits=_buf(), ph=_buf(), lengths=_buf(), B=2, T=10, Du=256, P=48, sil=47, sums=_buf(),
             counts=_buf())
    a.update(kw)
    return lib.stg_encoder_scores(a["pred"], a["tgt"], a["logits"], a["ph"], a["lengths"], a["B"], a["T"], a["Du"], a["P"],
                                  a["sil"], a["sums"], a["counts"], None)


@pytest.mark.parametrize("bad", [dict(pred=None), dict(tgt=None), dict(logits=None), dict(ph=None), dict(lengths=None),
                                 dict(sums=None), dict(counts=None), dict(B=0), dict(T=0), dict(Du=0), dict(P=0), dict(P=-1)],
                         ids=["no_pred", "no_tgt", "no_logits", "no_ph", "no_lengths", "no_sums", "no_counts", "B0", "T0",
                              "Du0", "P0", "Pneg"])
def test_encoder_scores_rejects_bad_arguments(bad):
    from ste_gan_b200 import _lib
    assert _scores(_lib.load(), **bad) == EINVAL


def _fake_plan():
    return SimpleNamespace(dtype=torch.float32, frame_rows=16)


def test_masked_encoder_forward_is_forward_only():
    from ste_gan_b200 import passes_encoder as pe
    lens = torch.tensor([10, 4], dtype=torch.int32)
    with pytest.raises(ValueError, match="forward-only"):
        pe.encoder_forward(_fake_plan(), torch.zeros(2, 160, 8), need_ctx=True, lengths=lens)


@pytest.mark.parametrize("T", [161, 168, 8])
def test_masked_encoder_forward_rejects_partial_frames(T):
    from ste_gan_b200 import passes_encoder as pe
    with pytest.raises(ValueError, match="multiple of 16"):
        pe.encoder_forward(_fake_plan(), torch.zeros(2, T, 8), need_ctx=False, lengths=torch.tensor([1, 0], dtype=torch.int32))


def test_aggregate_scores_weights_every_frame():
    from ste_gan_b200.inference import EncoderScore, aggregate_scores
    a = EncoderScore(speech_unit_sum=30.0, phoneme_sum=3.0, num_phones=10, num_correct_phones=4, num_silence_phones=2,
                     num_correct_phones_no_silence=3)
    b = EncoderScore(5.0, 9.0, 1, 1, 0, 1)
    empty = EncoderScore(0.0, 0.0, 0, 0, 0, 0)                     # a zero-length utterance
    assert (a.speech_unit_loss, a.phoneme_loss) == (3.0, 0.3)
    assert math.isnan(empty.speech_unit_loss) and math.isnan(empty.phoneme_loss)
    # two ranks' dicts merge by their values
    rank0, rank1 = {0: a, 2: empty}, {1: b}
    t = aggregate_scores(list(rank0.values()) + list(rank1.values()))
    assert t == EncoderScore(35.0, 12.0, 11, 5, 2, 4)
    assert t.speech_unit_loss == 35.0 / 11 and t.phoneme_loss == 12.0 / 11      # frame-weighted, not the mean of the means
    assert aggregate_scores([]) == empty
    assert aggregate_scores([t]) == t
