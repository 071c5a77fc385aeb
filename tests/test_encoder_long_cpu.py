"""CPU: which sequence lengths the one-CTA-per-head attention kernels take (the rule encoder_forward routes on), and the argument
checks of the band-tiled attention entry points (which run before any CUDA call)."""
import ctypes as C

import pytest

EINVAL, EUNSUPPORTED = -1, -3


# (d, longest forward L, longest backward L) of stg_relattn_fwd / stg_relattn_bwd
DENSE_LIMITS = [(96, 206, 133), (16, 548, 512), (4, 720, 888)]


@pytest.mark.parametrize("d,fwd,bwd", DENSE_LIMITS, ids=["d96", "d16", "d4"])
def test_dense_attention_limits(d, fwd, bwd):
    from ste_gan_b200 import _lib, ops
    lib = _lib.load()
    assert lib.stg_relattn_dense_supported(fwd, d, 0) == 1 and lib.stg_relattn_dense_supported(fwd + 1, d, 0) == 0
    both = min(fwd, bwd)                      # with need_bwd both kernels must take L
    assert lib.stg_relattn_dense_supported(both, d, 1) == 1 and lib.stg_relattn_dense_supported(both + 1, d, 1) == 0
    assert ops.relattn_dense_supported(1, d, True) and not ops.relattn_dense_supported(1500, d, False)


def test_dense_attention_limits_reject_bad_shapes():
    from ste_gan_b200 import _lib
    lib = _lib.load()
    for L, d in [(0, 96), (-5, 96), (100, 6), (100, 0), (1 << 30, 96), (2 ** 31 - 1, 4), (100, 1 << 29), (1, 2 ** 31 - 4)]:
        assert lib.stg_relattn_dense_supported(L, d, 0) == 0 and lib.stg_relattn_dense_supported(L, d, 1) == 0


def _buf():
    return C.cast((C.c_float * 16)(), C.c_void_p)


def _fwd(lib, **kw):
    a = dict(qkv=_buf(), dtype=0, emb=_buf(), B=1, L=300, H=8, d=96, M=100, o=_buf(), probs=_buf())
    a.update(kw)
    return lib.stg_relattn_band_fwd(a["qkv"], a["dtype"], a["emb"], a["B"], a["L"], a["H"], a["d"], a["M"], 0.1, a["o"], a["probs"],
                                    None)


def _bwd(lib, **kw):
    a = dict(qkv=_buf(), dtype=0, emb=_buf(), probs=_buf(), dout=_buf(), B=1, L=300, H=8, d=96, M=100, dqkv=_buf(), scratch=_buf())
    a.update(kw)
    return lib.stg_relattn_band_bwd(a["qkv"], a["dtype"], a["emb"], a["probs"], a["dout"], a["B"], a["L"], a["H"], a["d"], a["M"],
                                    0.1, a["dqkv"], a["scratch"], None)


BAD = [dict(qkv=None), dict(emb=None), dict(d=6), dict(d=0), dict(L=0), dict(L=-1), dict(M=0), dict(B=0), dict(H=0), dict(dtype=2),
       dict(dtype=-1)]
BAD_IDS = ["no_qkv", "no_emb", "d6", "d0", "L0", "Lneg", "M0", "B0", "H0", "dtype2", "dtype_neg"]


@pytest.mark.parametrize("bad", BAD + [dict(o=None), dict(probs=None)], ids=BAD_IDS + ["no_o", "no_probs"])
def test_band_fwd_rejects_bad_arguments(bad):
    """(The pointers are dummies: the call must return before it touches the device.)"""
    from ste_gan_b200 import _lib
    assert _fwd(_lib.load(), **bad) == EINVAL


@pytest.mark.parametrize("bad", BAD + [dict(probs=None), dict(dout=None), dict(dqkv=None), dict(scratch=None)],
                         ids=BAD_IDS + ["no_probs", "no_dout", "no_dqkv", "no_scratch"])
def test_band_bwd_rejects_bad_arguments(bad):
    from ste_gan_b200 import _lib
    assert _bwd(_lib.load(), **bad) == EINVAL


@pytest.mark.parametrize("big", [dict(d=132), dict(M=257), dict(B=65536), dict(H=65536)], ids=["d132", "M257", "B", "H"])
def test_band_rejects_shapes_past_its_bounds(big):
    from ste_gan_b200 import _lib
    lib = _lib.load()
    assert _fwd(lib, **big) == EUNSUPPORTED and _bwd(lib, **big) == EUNSUPPORTED
