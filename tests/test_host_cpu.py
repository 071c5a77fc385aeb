"""CPU: host-side logic - C-ABI exports, drop-in module surface, data-parallel plumbing (gloo, world 2)."""
import os
import re
import sys
import types

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def test_library_exports_every_declared_symbol():
    from ste_gan_b200 import _lib
    lib = _lib.load()
    hdr = open(os.path.join(ROOT, "include", "stegan_b200.h")).read()
    declared = set(re.findall(r"\b(stg_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/stegan_b200.h but not exported"
    assert declared == set(_lib.EXPORTS)
    assert lib.stg_version() >= 100 and lib.stg_strerror(-3).decode().startswith("shape")


def test_ctypes_struct_layout_matches_header():
    import ctypes as C
    from ste_gan_b200 import _lib
    assert C.sizeof(_lib.StgConv) == 21 * 4 + 4 + 8 * 8        # 21 ints, padding to 8, 8 pointers
    assert C.sizeof(_lib.StgWgrad) == 13 * 4 + 4 + 4 * 8      # 13 ints, padding to 8, 4 pointers


def test_init_matches_golden_checksums():
    """Same seed -> bit-identical parameters / buffers / key order as the reference modules."""
    from ste_gan_b200.models.discriminator import Discriminator, DiscriminatorSmall
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    init = torch.load(os.path.join(GOLD, "init_checksums.pt"))
    ctors = {"generator": lambda: EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8), "disc_small": lambda: DiscriminatorSmall(8),
             "disc_full": lambda: Discriminator(8), "generator_mfcc": lambda: EMGGeneratorGanTTS("MFCCS", 25, 17, 8)}
    for name, ctor in ctors.items():
        torch.manual_seed(0)
        mod = ctor()
        sd = mod.state_dict()
        assert list(sd.keys()) == list(init[name].keys()), name
        for k, ref in init[name].items():
            assert list(sd[k].shape) == ref["shape"], (name, k)
            assert torch.equal(sd[k].double().flatten()[ref["idx"]].float(), ref["samples"]), (name, k)
        if name in init["param_order"]:
            assert [n for n, _ in mod.named_parameters()] == init["param_order"][name]


def test_module_surface():
    from ste_gan_b200.losses.time_domain_loss import MultiTimeDomainFeatureLoss
    from ste_gan_b200.models.discriminator import DiscriminatorSmall, init_emg_discriminators
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS, init_emg_generator
    class AttrDict(dict):          # stands in for omegaconf.DictConfig: attribute access + `in`
        __getattr__ = dict.__getitem__
    cfg = AttrDict(model=AttrDict(speech_feature_type="SPEECH_UNITS", type="EMGGeneratorGanTTS", discriminator_small=True),
                   data=AttrDict(num_emg_channels=8, num_emg_sessions=17))
    g = init_emg_generator(cfg)
    assert isinstance(g, EMGGeneratorGanTTS) and g.input_size == 320 and g.num_output_channels == 8
    assert g.speech_feature_type == "SPEECH_UNITS" and g.use_session_embeddings and not g.use_speaking_mode_embedding
    assert sum(p.numel() for p in g.parameters()) == 23546832          # SURVEY.md 2 row 1
    d = init_emg_discriminators(cfg)
    assert isinstance(d, DiscriminatorSmall) and sum(p.numel() for p in d.parameters()) == 11856336
    assert d.discriminator_names == [f"DiscriminatorP-{p}" for p in (2, 3, 5, 7, 11)] + [f"DiscriminatorS-{i}" for i in range(3)]
    assert len(MultiTimeDomainFeatureLoss(8).time_domain_losses) == 3
    su = torch.randn(1, 8, 256)
    with pytest.raises(RuntimeError):            # no CPU fallback
        g(su, torch.zeros(1, dtype=torch.long), torch.zeros(1, dtype=torch.long))


def test_shard_helpers():
    from ste_gan_b200.dist import GradReducer, round_robin, shard_range
    assert [shard_range(r, 3, 10) for r in range(3)] == [(0, 4), (4, 7), (7, 10)]
    assert sorted(sum((round_robin(r, 4, 10) for r in range(4)), [])) == list(range(10))
    red = GradReducer(bucket_mb=1.0)
    assert not red.enabled and red.grad_scale == 1.0
    b = red.buckets(700000)
    assert b[0] == (700000 - 262144, 700000) and b[-1][0] == 0 and sum(h - l for l, h in b) == 700000


def _dp_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    from ste_gan_b200.dist import GradReducer, init_from_env, shard_range
    r, w, _ = init_from_env("gloo")
    red = GradReducer(bucket_mb=0.001)
    g = torch.full((1000,), float(r + 1))
    red.all_reduce(g)
    flat = torch.arange(8.0) * (r + 1)
    red.broadcast(flat, src=0)
    # the bucket-by-bucket exchange of the generator gradient: slices reduced asynchronously, back to front, waited on
    # together (trainer._reduce_g_bucket / _wait_handles)
    g2 = torch.full((900,), float(r + 1))
    handles = []
    for lo_, hi_ in ((600, 900), (300, 600), (0, 300)):
        handles += red.all_reduce_async(g2[lo_:hi_])
    red.wait(handles)
    ok = red.enabled and bool((g == 3.0).all()) and red.grad_scale == 0.5 and bool((flat == torch.arange(8.0)).all()) \
        and bool((g2 == 3.0).all()) and len(handles) >= 3
    lo, hi = shard_range(r, w, 32)
    out[rank] = (ok, lo, hi)
    dist.destroy_process_group()


def test_data_parallel_gloo_world2():
    """The N>1 exchange step on CPU: bucketed all-reduce (sum) + 1/world scale + initial broadcast."""
    port = 29500 + os.getpid() % 1000
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_dp_worker, args=(2, port, out), nprocs=2, join=True)
    assert out[0] == (True, 0, 16) and out[1] == (True, 16, 32)


def test_capture_refuses_data_parallel_without_own_communicator():
    """Over a group that is not CUDA + NCCL (no own communicator) the gradient exchange cannot be captured: capture()
    says so before it runs anything (here: on a trainer with nothing but its reducer set)."""
    from ste_gan_b200.trainer import GanTrainer
    tr = object.__new__(GanTrainer)
    tr.reducer, tr._inline = types.SimpleNamespace(enabled=True, comm=None), False
    with pytest.raises(RuntimeError, match="own NCCL communicator"):
        tr.capture(2, 64)


def test_precision_context():
    import ste_gan_b200
    assert ste_gan_b200.get_precision() == "fp32"
    with ste_gan_b200.precision("bf16"):
        assert ste_gan_b200.get_precision() == "bf16"
    assert ste_gan_b200.get_precision() == "fp32"
    with pytest.raises(ValueError):
        ste_gan_b200.set_precision("fp8")


def test_generator_gradient_buckets():
    """The three data-parallel gradient buckets of the base generator: contiguous, back to front, ~1/3 of the
    parameters each, cut at GBlock boundaries (trainer.generator_grad_buckets; flat offsets 16-byte aligned as in
    FlatParams)."""
    from ste_gan_b200.models.generator import EMGGeneratorGanTTS
    from ste_gan_b200.trainer import generator_grad_buckets
    torch.manual_seed(0)
    g = EMGGeneratorGanTTS("SPEECH_UNITS", 256, 17, 8)
    offsets, off = {}, 0
    for nm, p in g.named_parameters():
        offsets[nm] = off
        off += (p.numel() + 3) // 4 * 4
    nblk = len(list(g.gblocks)) - 1
    b = generator_grad_buckets(offsets, off, nblk)
    assert len(b) == 3 and nblk == 8
    # GBlocks: [2, 8) | [1, 2) | [0, 1)   convs of passes.generator_convs: gblocks.0 = 0, GBlock i = 1 + 5 i .. , last_conv = 41
    assert [(x[0], x[1]) for x in b] == [(2, 8), (1, 2), (0, 1)]
    assert [(x[2], x[3]) for x in b] == [(11, 42), (6, 11), (0, 6)]
    # flat slices: back to front, contiguous, covering everything, roughly balanced
    assert b[0][4][1] == off and b[2][4][0] == 0 and b[0][4][0] == b[1][4][1] and b[1][4][0] == b[2][4][1]
    assert b[0][4][0] == offsets["gblocks.3.conv1.2.bias"] or b[0][4][0] == min(v for k, v in offsets.items() if k.startswith("gblocks.3."))
    sizes = [x[4][1] - x[4][0] for x in b]
    assert all(0.25 * off < s < 0.42 * off for s in sizes), sizes


def test_conv_row_classes_cover_every_row_once():
    """Host-only check of the tcgen05 convolution's row classes (stg_debug_row_classes): for every T the classes tile
    rows [0, T) of a sample exactly once (tail tiles over-cover only past T or past the last sample, where the TMA unit
    zero-fills loads and clips stores), never need more tiles than plain 128-row tiling, and reach the ideal count
    ceil(B*T/128) up to the tail granularity."""
    import ctypes as C
    from ste_gan_b200 import _lib
    lib = _lib.load()
    out = (C.c_int * 12)()
    for T in list(range(1, 700)) + [800, 1600, 1601, 24000]:
        n = lib.stg_debug_row_classes(T, out)
        assert 1 <= n <= 4, (T, n)
        cls = [(out[3 * c], out[3 * c + 1], out[3 * c + 2]) for c in range(n)]
        covered = 0
        for seg, h0, tps in cls:
            assert seg in (8, 16, 32, 64, 128) and h0 == covered, (T, cls)      # contiguous, in order
            covered += seg * (tps if tps > 0 else 1)
            assert (tps > 0) == (seg == 128), (T, cls)
        assert T <= covered < T + 8 or (covered >= T and n == 4), (T, cls)        # over-cover < 8 rows unless the last slot rounds up
        # (with few samples the classes can need MORE tiles than plain 128-row tiling - conv_tc then keeps the classic
        # tiles; at the bench batch they never do)
        tiles16 = sum(16 * tps if tps > 0 else -(-16 // (128 // seg)) for seg, h0, tps in cls)
        assert tiles16 <= 16 * -(-T // 128) + 2, (T, tiles16)
    # the shapes of the bench configuration (B = 16)
    for T, want in ((100, 13), (200, 25), (400, 50), (800, 100), (1600, 200)):
        n = lib.stg_debug_row_classes(T, out)
        tiles = sum(16 * out[3 * c + 2] if out[3 * c + 2] > 0 else -(-16 // (128 // out[3 * c])) for c in range(n))
        assert tiles == want, (T, tiles)


def _conv_plan(**kw):
    import ctypes as C
    import torch
    from ste_gan_b200 import _lib, ops
    names = ("bn", "staged", "taps_per_stage", "stages", "smem", "occ2", "row_classes", "tiles", "grid", "compact_k", "k_chunks",
             "tmem_cols", "in_ring", "out_ring", "residues")
    ptrs = {k: 8 for k in ("src", "w")}
    ptrs.update({k: 8 for k in kw.pop("ptrs", ("y_raw",))})
    d = ops.StgConv(dtype=ops.code_of(torch.bfloat16), engine=ops.ENGINE_AUTO, **ptrs, **kw)
    out = (C.c_int * 15)()
    rc = _lib.load().stg_debug_conv_plan(C.byref(d), out)
    return rc, dict(zip(names, out))


def test_conv_plans_of_every_bench_layer_class():
    """Host-only check of the tcgen05 convolution planner (stg_debug_conv_plan) on every layer class of the benchmarked
    configurations (SURVEY.md 8 a7 / a8 / a9 / a11, B = 16 and the batched 32): the plan fits the hardware (227 KB of shared
    memory, 512 TMEM columns, <= 2 x 148 CTAs), pipelines (>= 2 stages, >= 3 with a tap window), tiles the channels exactly,
    uses compact per-group MMAs for groups narrower than a 64-channel chunk, and shares an SM between two CTAs exactly for
    the two classes it was measured to pay for (DESIGN.md 3.1)."""
    from ste_gan_b200 import ops
    G = [(768, 768, 3, d, 100) for d in (1, 3, 9, 27)] + [(768, 768, 1, 1, 100), (768, 384, 3, 1, 200), (384, 384, 3, 9, 400),
         (384, 384, 3, 27, 800), (384, 192, 3, 1, 1600), (192, 192, 3, 3, 1600), (192, 192, 1, 1, 1600), (320, 768, 1, 1, 100)]
    cases = []
    for ci, co, k, dil, T in G:                                           # generator: forward (residual, raw + act) and data-gradient
        geo = dict(n_samples=16, phases=1, t_src=T, t_dst=T, groups=1, k=k, dilation=dil, stride=1, pad=dil * (k - 1) // 2)
        cases.append(("g fwd", dict(geo, c_src=ci, c_dst=co, act=ops.ACT_RELU, ptrs=("y_raw", "y_act", "add_post", "bias"))))
        cases.append(("g dgrad", dict(geo, c_src=co, c_dst=ci, transposed=1, w_fwd_pack=1, mask_mode=ops.ACT_RELU, ptrs=("y_raw", "mask"))))
    S = [(128, 256, 37, 2, 4, 1600), (256, 512, 37, 2, 16, 800), (512, 1024, 5, 1, 1, 400),                 # DiscriminatorSmallerS
         (128, 128, 41, 2, 4, 1600), (128, 256, 41, 2, 16, 800), (256, 512, 41, 4, 16, 400), (512, 1024, 41, 4, 16, 100),
         (1024, 1024, 41, 1, 16, 25), (1024, 1024, 5, 1, 1, 25)]                                              # DiscriminatorS (full)
    for ci, co, k, st, g, T in S:
        for B in (16, 32):
            To = (T + 2 * (k // 2) - (k - 1) - 1) // st + 1
            pg = ops.tc_pack_groups(ci, co, g)
            geo = dict(n_samples=B, phases=1, k=k, dilation=1, stride=st, pad=k // 2, groups=pg)
            cases.append(("s fwd", dict(geo, t_src=T, t_dst=To, c_src=ci, c_dst=co, act=ops.ACT_LEAKY, ptrs=("y_act", "bias"))))
            cases.append(("s dgrad", dict(geo, t_src=To, t_dst=T, c_src=co, c_dst=ci, transposed=1, w_fwd_pack=int(g == 1),
                                          mask_mode=ops.ACT_LEAKY, ptrs=("y_raw", "mask"))))
    for p_, H in ((2, 803), (3, 536), (5, 323), (7, 231), (11, 148)):     # DiscriminatorSmallerP: 32 -> 256 -> 512, (3,1) stride 3
        for ci, co in ((32, 256), (256, 512)):
            Ho = (H + 4 - 2 - 1) // 3 + 1
            geo = dict(n_samples=32, phases=p_, k=3, dilation=1, stride=3, pad=2, groups=1)
            cases.append(("p fwd", dict(geo, t_src=H, t_dst=Ho, c_src=ci, c_dst=co, act=ops.ACT_LEAKY, ptrs=("y_act", "bias"))))
            cases.append(("p dgrad", dict(geo, t_src=Ho, t_dst=H, c_src=co, c_dst=ci, transposed=1, w_fwd_pack=1,
                                          mask_mode=ops.ACT_LEAKY, ptrs=("y_raw", "mask"))))
            H = Ho
    n_occ2 = 0
    for what, kw in cases:
        rc, pl = _conv_plan(**dict(kw))
        tag = (what, {k: v for k, v in kw.items() if k != "ptrs"}, pl)
        assert rc == 0, tag
        cd_g = kw["c_dst"] // kw["groups"]
        assert pl["smem"] <= 227 * 1024 and pl["stages"] >= 2 and pl["taps_per_stage"] >= 1, tag
        assert pl["taps_per_stage"] == 1 or pl["stages"] >= 3, tag
        assert pl["bn"] % 16 == 0 and 16 <= pl["bn"] <= 256, tag
        assert pl["compact_k"] or cd_g % pl["bn"] == 0 or pl["bn"] >= cd_g, tag
        assert 1 <= pl["grid"] <= pl["tiles"] and pl["grid"] <= (2 if pl["occ2"] else 1) * 148, tag
        cs_g = kw["c_src"] // kw["groups"]
        assert (pl["compact_k"] == cs_g) == (kw["groups"] > 1 and cs_g < 64), tag
        if pl["occ2"]:
            n_occ2 += 1
            assert pl["staged"] and pl["smem"] <= 113 * 1024 and pl["bn"] <= 128 and pl["tmem_cols"] == 256 and pl["out_ring"] == 2, tag
            assert (pl["compact_k"] and kw.get("transposed")) or (kw["groups"] > 1 and not pl["compact_k"] and pl["bn"] <= 64), tag
        else:
            assert pl["tmem_cols"] == 512 and pl["out_ring"] == 3, tag
        if what.startswith("g "):
            assert not pl["occ2"], tag                                      # dense layers: one CTA per SM (measured)
        if pl["staged"] and what.endswith("dgrad"):
            assert pl["in_ring"] in (2, 4, 8), tag
    assert n_occ2 >= 8      # the compact-group data-gradients and the 1024-channel grouped layers of the full discriminator


def test_checkpoint_interchange_with_torch_adamw(tmp_path):
    """SURVEY.md 8f rank 3 (host side, CPU): the fused trainer's flat AdamW moments <-> the state_dict of the reference's
    torch.optim.AdamW (ste_gan/utils/common.py:23-61, train.py:421-436) - both directions, file naming and the choice of
    the latest checkpoint, the `_orig_mod.` key fix."""
    from ste_gan_b200 import checkpoint as ck
    from ste_gan_b200.models.discriminator import DiscriminatorSmall
    torch.manual_seed(0)
    net = DiscriminatorSmall(8)                       # has 1-element parameters: exercises the 16-byte aligned layout
    params = list(net.parameters())
    opt = torch.optim.AdamW(params, lr=2e-4, betas=(0.8, 0.99))
    for it in range(3):
        for p in params:
            p.grad = torch.randn_like(p) * 0.01
        opt.step()
    ref_sd = opt.state_dict()
    shapes = [(nm, p.shape) for nm, p in net.named_parameters()]
    offsets, off = {}, 0
    for nm, p in net.named_parameters():              # FlatParams' layout
        offsets[nm] = off
        off += (p.numel() + 3) // 4 * 4
    m, v = torch.full((off,), 7.0), torch.full((off,), 7.0)
    step = ck.adamw_state_to_flat(ref_sd, shapes, offsets, m, v)
    assert step == 3
    for i, (nm, shp) in enumerate(shapes):
        n = int(torch.Size(shp).numel())
        assert torch.equal(m[offsets[nm]:offsets[nm] + n].view(shp), ref_sd["state"][i]["exp_avg"])
        assert torch.equal(v[offsets[nm]:offsets[nm] + n].view(shp), ref_sd["state"][i]["exp_avg_sq"])
    assert float(m.sum()) == pytest.approx(float(sum(s["exp_avg"].double().sum() for s in ref_sd["state"].values())), rel=1e-5)  # gaps are zero
    back = ck.flat_to_adamw_state(shapes, offsets, m, v, step, dict(lr=2e-4 * 0.999 ** 2, initial_lr=2e-4))
    opt2 = torch.optim.AdamW(params, lr=1.0)          # a fresh reference optimiser accepts the converted state ...
    opt2.load_state_dict(back)
    # ... and the reference's resume path can re-create its scheduler on it (train.py:98-104:
    # ExponentialLR(opt, gamma=.999, last_epoch=start_epoch) raises KeyError without `initial_lr` in the param groups)
    sched = torch.optim.lr_scheduler.ExponentialLR(opt2, gamma=0.999, last_epoch=2)
    assert sched.base_lrs == [2e-4] and opt2.param_groups[0]["lr"] == pytest.approx(2e-4 * 0.999 ** 2)
    opt2.param_groups[0]["lr"] = 2e-4
    sd2 = opt2.state_dict()
    assert sd2["param_groups"][0]["lr"] == 2e-4 and sd2["param_groups"][0]["betas"] == (0.8, 0.99)
    for i in range(len(shapes)):
        assert float(sd2["state"][i]["step"]) == 3.0
        assert torch.equal(sd2["state"][i]["exp_avg"], ref_sd["state"][i]["exp_avg"])
        assert torch.equal(sd2["state"][i]["exp_avg_sq"], ref_sd["state"][i]["exp_avg_sq"])
    # ... and continues exactly like the original one
    w0 = [p.detach().clone() for p in params]
    grads = [torch.randn_like(p) * 0.01 for p in params]
    for p, g_ in zip(params, grads):
        p.grad = g_.clone()
    opt.step()
    w_ref = [p.detach().clone() for p in params]
    with torch.no_grad():
        for p, w in zip(params, w0):
            p.copy_(w)
    opt2.step()
    assert all(torch.equal(a, b.detach()) for a, b in zip(w_ref, params))
    # file naming / latest selection / key fix
    for n in (100, 2500, 30):
        torch.save({}, tmp_path / f"checkpoint-{n:08d}.pt")
    torch.save({}, tmp_path / "checkpoint-final.pt")
    assert ck.latest_step(tmp_path) == "00002500" and ck.latest_step(tmp_path / "nope") is None
    fixed = ck.fix_state_dict({"_orig_mod.gblocks.0.bias": 1, "last_conv.1.bias": 2})
    assert list(fixed) == ["gblocks.0.bias", "last_conv.1.bias"]
    with pytest.raises(ValueError):
        ck.adamw_state_to_flat(ref_sd, shapes[:-1], offsets, m, v)


def test_synthetic_batch_matches_oracle_generator():
    """bench.py's GPU arm draws its inputs from ste_gan_b200.synthetic (it must not import oracle/); the tests draw theirs
    from the oracle: the two generators are the same sequence."""
    from oracle import ste_gan_oracle as O
    from ste_gan_b200.synthetic import synthetic_batch
    for kw in (dict(batch=3, frames=7, seed=5), dict(batch=2, frames=4, seed=9, unit_dim=25, hop=8)):
        for a, b in zip(synthetic_batch(**kw), O.synthetic_batch(**kw)):
            assert torch.equal(a, b)


def test_nccl_library_binding_loads():
    """ste_gan_b200/nccl.py binds the NCCL library PyTorch ships (no GPU needed for the version query)."""
    from ste_gan_b200 import nccl
    assert nccl.version() >= 21800
    for sym in ("ncclGetUniqueId", "ncclCommInitRank", "ncclAllReduce", "ncclCommDestroy"):
        assert hasattr(nccl.load_library(), sym)
