"""CPU: the host side of padded-batch serving - the bucket ladder and batching plan of serve_batched, and the argument
checks of stg_conv_masked (which run before any CUDA call)."""
import ctypes as C
import random

import pytest


def test_bucket_ladder():
    from ste_gan_b200.inference import BUCKETS_PER_OCTAVE, MIN_BUCKET, bucket_frames
    assert [bucket_frames(n) for n in (0, 1, 16, 17, 20, 21, 28, 29, 32, 33)] == [16, 16, 16, 20, 20, 24, 28, 32, 32, 40]
    assert bucket_frames(1500) == 1536 and bucket_frames(1536) == 1536 and bucket_frames(1537) == 1792
    prev = 0
    for n in range(1, 5000):
        b = bucket_frames(n)
        assert b >= n and b >= MIN_BUCKET
        assert b >= prev                                             # monotone: a longer utterance never gets a shorter bucket
        prev = b
        if n > MIN_BUCKET:
            assert (b - n) * BUCKETS_PER_OCTAVE < n                  # padding < 1 / BUCKETS_PER_OCTAVE of the length
    # about 4 buckets per octave over the 2-30 s utterances (100..1500 frames)
    assert len({bucket_frames(n) for n in range(100, 1501)}) == 16
    assert [bucket_frames(n, 2) for n in (17, 25, 33, 49)] == [24, 32, 48, 64]      # a coarser ladder: 2 per octave


def test_plan_batches_buckets_partial_batches_and_order():
    from ste_gan_b200.inference import bucket_frames, plan_batches
    lengths = [5, 100, 17, 1500, 16, 16, 16, 1, 112, 113]
    plan = plan_batches(lengths, max_batch=2)
    assert plan == [(16, [0, 4]), (16, [5, 6]), (16, [7]), (20, [2]), (112, [1, 8]), (128, [9]), (1536, [3])]
    for T, idx in plan:
        assert 1 <= len(idx) <= 2 and all(bucket_frames(lengths[i]) == T for i in idx)
    assert plan_batches([]) == []
    with pytest.raises(ValueError):
        plan_batches([3], max_batch=0)


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_plan_shards_cover_every_index_once_and_are_deterministic(world):
    from ste_gan_b200.inference import plan_batches
    rng = random.Random(0)
    lengths = [rng.randint(1, 1500) for _ in range(300)]
    plan = plan_batches(lengths, max_batch=8)
    assert plan == plan_batches(list(lengths), max_batch=8)          # every rank computes the same plan
    seen = []
    for rank in range(world):
        for _, idx in plan[rank::world]:                             # serve_batched's round-robin over batches
            seen += idx
    assert sorted(seen) == list(range(len(lengths)))
    assert all(len(idx) <= 8 for _, idx in plan)
    assert [T for T, _ in plan] == sorted(T for T, _ in plan)        # ascending buckets: one graph capture per bucket


def _desc(**kw):
    from ste_gan_b200 import _lib
    base = dict(dtype=1, engine=0, n_samples=2, phases=1, t_src=64, t_dst=64, c_src=64, c_dst=64, groups=1, k=3, dilation=1,
                stride=1, pad=1, src=16, w=16, y_raw=16)
    base.update(kw)
    return _lib.StgConv(**base)


@pytest.mark.parametrize("bad", [dict(transposed=1, w_fwd_pack=1), dict(transposed=1), dict(pair_sum=1), dict(phases=2),
                                 dict(phases=4, t_src=16, t_dst=16), dict(src=0)],
                         ids=["transposed_fwd_pack", "transposed", "pair_sum", "phases2", "phases4", "no_src"])
def test_conv_masked_rejects_unsupported_calls(bad):
    """Only the forward, single-phase, non-pair-summed contraction takes a length mask.  (The pointers are dummies:
    the call must return before it touches the device.)"""
    from ste_gan_b200 import _lib
    lib = _lib.load()
    lens = (C.c_int32 * 2)(3, 4)
    assert lib.stg_conv_masked(C.byref(_desc(**bad)), C.cast(lens, C.c_void_p), 1, None) == -1


@pytest.mark.parametrize("valid_units,rows_per_unit", [(False, 1), (True, 0), (True, -2)],
                         ids=["null_lengths", "zero_rate", "negative_rate"])
def test_conv_masked_rejects_bad_mask_arguments(valid_units, rows_per_unit):
    from ste_gan_b200 import _lib
    lib = _lib.load()
    lens = (C.c_int32 * 2)(3, 4)
    ptr = C.cast(lens, C.c_void_p) if valid_units else None
    for engine in (0, 1, 2):
        assert lib.stg_conv_masked(C.byref(_desc(engine=engine)), ptr, rows_per_unit, None) == -1
