"""CPU: the argument checks of stg_td_scores (they run before any CUDA call), the host-side checks of validate_batched and
serve_batched that run before any launch, and the arithmetic of aggregate_td."""
import ctypes as C
import math
from collections import OrderedDict

import pytest
import torch

EINVAL, EUNSUPPORTED = -1, -3


def _buf():
    return C.cast((C.c_float * 16)(), C.c_void_p)


def _td_scores(lib, **kw):
    a = dict(xr=_buf(), xg=_buf(), B=2, T=160, C=8, units=_buf(), rate=16, n_res=3, wins=(20, 51, 80), shifts=(8, 13, 16),
             pad=1, avg=9, out=_buf(), scratch=_buf())
    a.update(kw)
    wins = None if a["wins"] is None else (C.c_int * 3)(*a["wins"])
    shifts = None if a["shifts"] is None else (C.c_int * 3)(*a["shifts"])
    return lib.stg_td_scores(a["xr"], a["xg"], a["B"], a["T"], a["C"], a["units"], a["rate"], a["n_res"], wins, shifts,
                             a["pad"], a["avg"], a["out"], a["scratch"], None)


def test_td_scores_is_exported_with_its_signature():
    from ste_gan_b200 import _lib
    assert "stg_td_scores" in _lib.EXPORTS and len(_lib._SIGS["stg_td_scores"]) == 15
    assert _lib.load().stg_td_scores.argtypes[6] is C.c_int32


BAD = {"no_real": dict(xr=None), "no_gen": dict(xg=None), "no_units": dict(units=None), "no_wins": dict(wins=None),
       "no_shifts": dict(shifts=None), "no_out": dict(out=None), "no_scratch": dict(scratch=None), "B0": dict(B=0),
       "T0": dict(T=0), "C0": dict(C=0), "n_res0": dict(n_res=0), "n_res9": dict(n_res=9), "avg_even": dict(avg=8),
       "avg0": dict(avg=0), "avg_neg": dict(avg=-3), "rate0": dict(rate=0), "rate_neg": dict(rate=-16),
       "T_not_multiple": dict(T=161), "win0": dict(wins=(20, 0, 80)), "shift0": dict(shifts=(8, 13, 0))}


@pytest.mark.parametrize("bad", list(BAD.values()), ids=list(BAD))
def test_td_scores_rejects_bad_arguments(bad):
    """(The pointers are dummies: the call must return before it touches the device.)"""
    from ste_gan_b200 import _lib
    assert _td_scores(_lib.load(), **bad) == EINVAL


def test_td_scores_batch_bound():
    from ste_gan_b200 import _lib
    assert _td_scores(_lib.load(), B=65536) == EUNSUPPORTED


# ---------------------------------------------------------------------------------------------
# validate_batched / serve_batched: checks before any launch
# ---------------------------------------------------------------------------------------------
def _engine(feature="SPEECH_UNITS", modes=False, encoder=None):
    """An UtteranceGenerator over a CPU generator whose every launch path raises: a check that passes reaches a launch."""
    from ste_gan_b200.inference import UtteranceGenerator
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    torch.manual_seed(0)
    ug = object.__new__(UtteranceGenerator)
    ug.net_g = EMGGeneratorGanTTS(feature, 256 if feature == "SPEECH_UNITS" else 25, 17, 8, use_speaking_mode_embedding=modes,
                                  channels=32)
    ug.emg_encoder, ug._uses_mode, ug._graphs, ug.max_graphs = encoder, modes, OrderedDict(), 8

    def launch(*a, **kw):
        raise RuntimeError("launched")
    ug.capture = ug._capture_validate = ug.generate_graph = launch
    return ug


def _utts(lengths, D=256):
    return [(torch.zeros(n, D), torch.tensor(1)) for n in lengths]


def _real(lengths, r=16):
    return [torch.zeros(r * n, 8) for n in lengths]


def test_rows_per_frame():
    assert _engine().rows_per_frame == 16 and _engine("MFCCS").rows_per_frame == 8


def test_validate_batched_checks_real_emg_before_any_launch():
    from ste_gan_b200.inference import TD_MIN_ROWS
    ug = _engine()
    lens = [3, 10, 40]
    with pytest.raises(RuntimeError, match="launched"):             # valid arguments reach the first capture
        ug.validate_batched(_utts(lens), real_emg=_real(lens))
    bad_rows = _real(lens); bad_rows[1] = torch.zeros(16 * 10 + 1, 8)
    with pytest.raises(ValueError, match=r"real_emg\[1\]"):
        ug.validate_batched(_utts(lens), real_emg=bad_rows)
    bad_channels = _real(lens); bad_channels[2] = torch.zeros(16 * 40, 7)
    with pytest.raises(ValueError, match=r"real_emg\[2\]"):
        ug.validate_batched(_utts(lens), real_emg=bad_channels)
    with pytest.raises(ValueError, match="2 real_emg items for 3 utterances"):
        ug.validate_batched(_utts(lens), real_emg=_real(lens)[:2])
    assert TD_MIN_ROWS == 41                                        # win 80: reflect pad 40 < rows
    for short in ([2, 10], [0, 10]):                                # 32 and 0 EMG rows
        with pytest.raises(ValueError, match="at least 41"):
            ug.validate_batched(_utts(short), real_emg=_real(short))
    mfcc = _engine("MFCCS")
    with pytest.raises(ValueError, match="at least 41"):            # 40 rows at 8 rows per frame
        mfcc.validate_batched(_utts([5], 25), real_emg=_real([5], 8))
    with pytest.raises(RuntimeError, match="launched"):
        mfcc.validate_batched(_utts([6], 25), real_emg=_real([6], 8))


def test_validate_batched_needs_an_encoder_or_real_emg():
    ug = _engine()
    with pytest.raises(ValueError, match="emg_encoder"):
        ug.validate_batched(_utts([10]))


def test_validate_batched_with_an_encoder_needs_targets():
    ug = _engine(encoder=object())
    with pytest.raises(ValueError, match="unit / phoneme targets"):
        ug.validate_batched(_utts([10]), real_emg=_real([10]))


@pytest.mark.parametrize("call", ["serve_batched", "validate_batched"])
def test_speaking_mode_ids_are_checked_before_any_launch(call):
    ug = _engine(modes=True)
    lens = [10, 12]
    run = lambda **kw: getattr(ug, call)(_utts(lens), **({"real_emg": _real(lens)} if call == "validate_batched" else {}),
                                         **kw)                      # noqa: E731
    with pytest.raises(ValueError, match="speaking_mode_ids"):
        run()
    with pytest.raises(ValueError, match="1 speaking_mode_ids for 2 utterances"):
        run(speaking_mode_ids=[0])
    with pytest.raises(ValueError, match=r"\[0, 3\)"):
        run(speaking_mode_ids=[0, 3])
    with pytest.raises(RuntimeError, match="launched"):
        run(speaking_mode_ids=[2, 1])
    plain = _engine()                                               # a generator without the embedding ignores the ids
    with pytest.raises(RuntimeError, match="launched"):
        getattr(plain, call)(_utts(lens), **({"real_emg": _real(lens)} if call == "validate_batched" else {}),
                             speaking_mode_ids=[7])


def test_aggregate_td_is_the_mean_over_utterances():
    from ste_gan_b200.inference import TdScore, aggregate_td
    a, b, c = TdScore((0.1, 0.2, 0.3)), TdScore((1.0, 2.0, 4.0)), TdScore((1e-9, 3.0, 1e7))
    assert a.loss == pytest.approx(0.6)
    rank0, rank1 = {0: a, 2: c}, {1: b}
    union = {**rank0, **rank1}
    t = aggregate_td(list(rank0.values()) + list(rank1.values()))
    assert t == aggregate_td(union.values()) == aggregate_td([c, b, a])          # exact sums: the order does not matter
    assert t.values == tuple(math.fsum(v) / 3 for v in zip(a.values, b.values, c.values))
    assert t.loss == pytest.approx(sum(sc.loss for sc in union.values()) / 3)    # unweighted by length
    assert aggregate_td([a]) == a
    assert all(math.isnan(v) for v in aggregate_td([]).values)
