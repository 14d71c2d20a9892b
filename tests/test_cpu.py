"""CPU suite (`-m "not gpu"`): the oracle against the committed golden vectors, the host logic (tiling, sharding,
parameter layout, schedules), the C-ABI surface (library loads and exports every symbol include/b2u.h declares — no
compute calls without a GPU) and the data-parallel host logic on a world_size-2 gloo group."""
import hashlib
import json
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


# ------------------------------------------------------------------------------------------------ windows (bit-exact)
def test_windows_oracle_and_product_match_golden():
    from oracle import windows as ow
    from unet_b200 import tiling
    gold = json.load(open(os.path.join(GOLD, "windows.json")))
    for g in gold:
        args = (g["height"], g["width"], g["patch"], g["overlap"])
        for impl in (ow.compute_windows, tiling.compute_windows):
            ws = impl(*args)
            assert len(ws) == g["count"]
            assert [list(w) for w in ws[:3]] == g["first"] and [list(w) for w in ws[-3:]] == g["last"]
            assert hashlib.sha256(json.dumps([list(w) for w in ws]).encode()).hexdigest() == g["sha256"]
        assert tiling.axis_offsets(g["width"], g["patch"], g["overlap"])[0] == g["xs"]
        assert tiling.axis_offsets(g["height"], g["patch"], g["overlap"])[0] == g["ys"]


def test_windows_survey_facts():
    """SURVEY.md 8(a) row A8: config 3 has 90 offsets per axis [0,224,...,19712,19744] -> 8100 tiles, x-outer order."""
    from unet_b200.tiling import axis_offsets, compute_windows
    xs, win = axis_offsets(20000, 256, 0.125)
    assert win == 256 and len(xs) == 90 and xs[:3] == [0, 224, 448] and xs[-2:] == [19712, 19744]
    ws = compute_windows(20000, 20000, 256, 0.125)
    assert len(ws) == 8100 and ws[0] == (0, 0, 256, 256) and ws[1] == (0, 224, 256, 256) and ws[90] == (224, 0, 256, 256)
    with pytest.raises(ValueError):
        compute_windows(100, 100, 64, 1.5)
    # raster smaller than the patch: a single window clipped to the raster
    assert compute_windows(64, 64, 256, 0.2) == [(0, 0, 64, 64)]


def test_coverage_counts_and_colour_classes():
    from unet_b200.tiling import colour_classes, compute_windows, shard_windows_by_columns
    for (h, w, p, ov) in [(2000, 2000, 256, 0.125), (257, 511, 256, 0.5), (300, 300, 256, 0.75), (700, 500, 128, 0.2)]:
        ws = compute_windows(h, w, p, ov)
        cov = np.zeros((h, w), np.int32)
        for (x, y, ww, hh) in ws:
            cov[y:y + hh, x:x + ww] += 1
        assert cov.min() >= 1
        if ov <= 0.125:
            assert set(np.unique(cov)) <= {1, 2, 4}          # predict.py:287: "1, 2, or 4 tiles"
        classes = colour_classes(ws)
        assert sorted(i for c in classes for i in c) == list(range(len(ws)))
        for c in classes:                                      # tiles of one class never overlap
            m = np.zeros((h, w), np.int8)
            for i in c:
                x, y, ww, hh = ws[i]
                assert m[y:y + hh, x:x + ww].max() == 0
                m[y:y + hh, x:x + ww] = 1
        # owner-computes sharding: strips partition the columns, and every tile touching a strip is assigned to it
        for world in (2, 3, 8):
            xs = []
            for r in range(world):
                idx, xb, xe = shard_windows_by_columns(ws, w, r, world)
                xs.append((xb, xe))
                need = [i for i, (x, y, ww, hh) in enumerate(ws) if x < xe and x + ww > xb]
                assert idx == need
            assert xs[0][0] == 0 and xs[-1][1] == w and all(xs[i][1] == xs[i + 1][0] for i in range(world - 1))


@pytest.mark.parametrize("world", range(1, 9))
def test_column_owned_gives_every_tile_one_owner(world):
    """tiling.column_owned over the strips of shard_windows_by_columns (the merge of save_predictions): every tile of
    randomly placed mosaics is owned by exactly one rank, which counts it in a validation_vision assessment."""
    from unet_b200.tiling import column_owned, shard_windows_by_columns
    rng = np.random.default_rng(world)
    P = 16
    for _ in range(5):
        n = int(rng.integers(1, 60))
        place = [(int(rng.integers(0, 200)), int(rng.integers(0, 50)), P, P) for _ in range(n)]
        x_len = max(x for x, *_ in place) + P
        owners = [[] for _ in range(n)]
        for r in range(world):
            mine, xb, xe = shard_windows_by_columns(place, x_len, r, world)
            for i, o in zip(mine, column_owned(place, mine, xb, xe)):
                if o:
                    owners[i].append(r)
        assert all(len(o) == 1 for o in owners)


# ------------------------------------------------------------------------------------------------ stitch oracle
def test_stitch_oracle_matches_golden():
    from oracle import stitch
    g = np.load(os.path.join(GOLD, "stitch.npz"))
    h, w, p, c = g["shape"]
    ws = [tuple(int(v) for v in r) for r in g["windows"]]
    probs = [stitch.softmax_probs(l) for l in g["logits"]]
    merged = stitch.merge_pixel_windows(probs, ws, int(h), int(w))
    assert np.array_equal(merged.astype(np.uint8), g["merged"])
    gts = [[float(x), float(ww), 1.0, -float(y), float(hh), -1.0] for (x, y, ww, hh) in ws]
    m8, _ = stitch.merge_tiles(probs, gts, large_file=True)
    assert np.array_equal(m8.astype(np.uint8), g["merged_large_file"])
    # placement arithmetic of predict.py:294-297 through real geotransforms (0.2 m pixels, UTM-like origin)
    from unet_b200.tiling import placement_from_geotransform
    gt = (382000.0, 0.2, 0.0, 5812000.0, 0.0, -0.2)
    gts2 = [[gt[0] + x * gt[1], ww, gt[1], gt[3] + y * gt[5], hh, gt[5]] for (x, y, ww, hh) in ws]
    merged2, origin = stitch.merge_tiles(probs, gts2)
    assert np.array_equal(merged2, merged) and origin[0] == gt[0] and origin[2] == gt[3]
    for (x, y, ww, hh), q in zip(ws, gts2):
        assert placement_from_geotransform(q[0], q[1], q[2], q[3], q[4], q[5], gt[0], gt[3]) == (x, y, x + ww, y + hh)


# ------------------------------------------------------------------------------------------------ model oracle
def test_oracle_model_matches_golden_and_survey_counts():
    from oracle.unet_oracle import count_conv_flops, make_oracle, weighted_ce
    g = np.load(os.path.join(GOLD, "model_xresnet18_32.npz"))
    torch.set_num_threads(4)
    m = make_oracle("xresnet18", 3, 2, seed=0).train()
    p = dict(m.named_parameters())
    assert np.allclose(p["layers.0.0.0.weight"].detach().flatten()[:8].numpy(), g["weight_probe"][0], atol=1e-7)
    x = torch.from_numpy(g["x_u8"]).float() / 255.0
    y = torch.from_numpy(g["y"]).long()
    m.eval()                      # eval first (fresh running statistics), exactly as the generator does
    with torch.no_grad():
        assert np.allclose(m(x).numpy(), g["logits_eval"], rtol=1e-4, atol=1e-4)
    m.train()
    logits = m(x)
    loss = weighted_ce(logits, y, torch.full((2,), 0.5))
    loss.backward()
    assert np.allclose(logits.detach().numpy(), g["logits_train"], rtol=1e-4, atol=1e-4)
    assert abs(loss.item() - g["loss"][0]) <= 1e-5
    for k in g.files:
        if k.startswith("grad::"):
            assert np.allclose(p[k[6:]].grad.numpy(), g[k], rtol=1e-3, atol=1e-6), k
    # SURVEY.md 8(a): parameter totals and forward conv FLOPs of the restated topology
    m34 = make_oracle("xresnet34", 4, 2)
    assert sum(q.numel() for q in m34.parameters()) == 41244274 and len(list(m34.parameters())) == 160
    assert count_conv_flops(m34, 256) == 63922241536


def test_bf16_emulation_tracks_oracle():
    from oracle.bf16_emulation import emulated_forward
    from oracle.unet_oracle import make_oracle
    m = make_oracle("xresnet18", 3, 2).train()
    x = torch.rand(2, 3, 32, 32, generator=torch.Generator().manual_seed(0))
    a, b = m(x), emulated_forward(m, x, True)
    assert ((a - b).abs().max() / a.abs().max()).item() < 5e-2
    b.sum().backward()
    assert all(q.grad is not None for q in m.parameters())


@pytest.mark.parametrize("self_attention", [False, True])
def test_teacher_forced_emulation(self_attention):
    """Why the model-level gradient test teacher-forces the emulation (oracle/bf16_emulation.py `taps=`): a free-running
    bf16 emulation is chaotic - perturbing the values in front of every rounding by 1e-6 relative (an accumulation-order
    sized difference) moves deep-layer gradients by tens of percent - whereas with the forward activations pinned to
    the perturbed run's own values every gradient agrees to a few percent, and a zeroed or sign-flipped tensor is
    caught by the shared checker."""
    import copy
    from oracle.bf16_emulation import emulated_forward
    from oracle.unet_oracle import make_oracle, weighted_ce
    from parity_util import gradient_mismatches
    from unet_b200.synth import aerial_like_tiles
    o = make_oracle("xresnet18", 3, 2, self_attention=self_attention).train()
    x_u8, y = aerial_like_tiles(4, 3, 64, 64, 2)
    x, y, w = x_u8.float() / 255, y.long(), torch.full((2,), 0.5)

    def run(**kw):
        m = copy.deepcopy(o)
        weighted_ce(emulated_forward(m, x, True, **kw), y, w).backward()
        return {n: q.grad.clone() for n, q in m.named_parameters()}

    torch.manual_seed(1)
    rec = {}
    g_plan = run(noise=1e-6, record=rec)          # stands in for the CUDA plan: same graph, other accumulation order
    g_free, g_tf = run(), run(taps=rec)
    assert len(gradient_mismatches(g_plan, g_free, 5e-2, 0.99)) > 20      # free running: no power on the deep layers
    assert not gradient_mismatches(g_plan, g_tf, 5e-2, 0.999)             # teacher forced: everything agrees
    broken = dict(g_plan)
    name = "layers.0.7.1.convpath.1.0.weight"
    broken[name] = torch.zeros_like(g_plan[name])
    assert [b[0] for b in gradient_mismatches(broken, g_tf, 5e-2, 0.999)] == [name]
    broken[name] = -g_plan[name]
    assert [b[0] for b in gradient_mismatches(broken, g_tf, 5e-2, 0.999)] == [name]


# ------------------------------------------------------------------------------------------------ layout / host logic
@pytest.mark.parametrize("arch,n_in,n_out,size,params,mflops", [
    ("xresnet34", 4, 2, 256, 41244274, 63922.241536), ("xresnet18", 3, 2, 128, 31132240, 14652.801024),
    ("xresnet50", 4, 8, 512, 339101776, 2515290.554368)])
def test_param_layout_matches_oracle_names(arch, n_in, n_out, size, params, mflops):
    from oracle.unet_oracle import make_oracle, param_groups
    from unet_b200.layout import ParamLayout, build_spec, conv_flops
    spec = build_spec(arch, n_in, n_out)
    L = ParamLayout(spec)
    m = make_oracle(arch, n_in, n_out)
    assert [(e.name, e.shape) for e in L.entries] == [(n, tuple(p.shape)) for n, p in m.named_parameters()]
    assert L.n_params() == params
    assert abs(conv_flops(spec, size) / 1e6 - mflops) < 1e-3
    groups = param_groups(m)
    for e in L.entries:
        assert e.name in groups[e.group]
        assert e.offset % 4 == 0
        assert e.decay == (len(e.shape) == 4)
    buf = {k for k, _ in m.named_buffers() if not k.endswith("num_batches_tracked")}
    assert {pfx + s for pfx, _ in L.buffers for s in (".running_mean", ".running_var")} == buf


def test_shuffle_row_permutation():
    from unet_b200.layout import shuffle_row_of_co
    roc = shuffle_row_of_co(16)
    assert sorted(roc) == list(range(16))
    x = torch.arange(16.0).view(1, 16, 1, 1)
    ps = torch.nn.functional.pixel_shuffle(x, 2)[0]                  # [4, 2, 2]
    for co in range(16):
        r = roc[co]
        ij, c = divmod(r, 4)
        assert ps[c, ij // 2, ij % 2].item() == co                    # row (i,j,c) holds torch channel 4c+2i+j


def test_one_cycle_and_shard_range():
    from oracle.unet_oracle import one_cycle_lr
    from unet_b200.engine import one_cycle, shard_range
    for pct in (0.0, 0.1, 0.25, 0.5, 0.99, 1.0):
        assert one_cycle(pct, 1e-3) == pytest.approx(one_cycle_lr(pct, 1e-3))
    assert one_cycle(0.0, 1e-3)[0] == pytest.approx(1e-3 / 25) and one_cycle(0.25, 1e-3)[0] == pytest.approx(1e-3)
    for n, world in ((8100, 8), (10, 3), (5, 8)):
        parts = [shard_range(n, r, world) for r in range(world)]
        assert parts[0][0] == 0 and parts[-1][1] == n
        assert all(parts[i][1] == parts[i + 1][0] for i in range(world - 1))
        assert max(b - a for a, b in parts) - min(b - a for a, b in parts) <= 1


def test_synthetic_data_is_deterministic():
    from unet_b200.synth import aerial_like_tiles, uniform_tiles
    a, b = uniform_tiles(2, 4, 32, 32, 2), uniform_tiles(2, 4, 32, 32, 2)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and a[0].dtype == torch.uint8
    x, y = aerial_like_tiles(2, 4, 32, 32, 3)
    assert x.shape == (2, 4, 32, 32) and int(y.max()) <= 2


# ------------------------------------------------------------------------------------------------ C-ABI surface
def test_c_abi_exports_every_declared_symbol():
    import ctypes
    from unet_b200 import _lib
    header = open(os.path.join(ROOT, "include", "b2u.h")).read()
    declared = set(re.findall(r"\b(b2u_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 35
    lib = _lib.load()
    missing = [n for n in sorted(declared) if not hasattr(lib, n)]
    assert not missing, missing
    assert lib.b2u_version() >= 1
    # struct layouts mirrored in ctypes must match the C side (sizes are part of the ABI)
    lib.b2u_abi_sizeof.restype = ctypes.c_int
    mirrors = [_lib.View, _lib.ConvDesc, _lib.ConvInfo, _lib.WgradDesc, _lib.WgradInfo, _lib.WStageItem, _lib.BNFin]
    for which, cls in enumerate(mirrors):
        assert ctypes.sizeof(cls) == lib.b2u_abi_sizeof(which), cls.__name__
    assert ctypes.sizeof(_lib.View) == 48 and ctypes.sizeof(_lib.WStageItem) == 88


def test_product_never_imports_the_oracle():
    """the oracle is test infrastructure: unet_b200/ must not import it (bench.py may, in its CPU-baseline legs only)"""
    pkg = os.path.join(ROOT, "unet_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), fn


def test_network_requires_cuda():
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from unet_b200 import _lib
    from unet_b200.network import UNetB200
    with pytest.raises(_lib.B2UError):
        UNetB200("xresnet18", 3, 2, (64, 64), 1)


# ------------------------------------------------------------------------------------------------ gloo, world_size 2
def _ddp_worker(rank, world, port, data_dir, out):
    """The host side of the data-parallel step on a gloo group: the product's batch dealing (`reference_api._tile_batches`
    with rank / world) and the product's segment + bucket schedule of the gradient all-reduce (`engine.plan_segments`,
    `engine.bucket_ranges`) driving real collectives."""
    import torch.distributed as dist
    from pathlib import Path
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from unet_b200.engine import bucket_ranges, plan_segments
    from unet_b200.reference_api import _tile_batches
    files = sorted((Path(data_dir) / "trai" / "img_tiles").glob("*.tif"))
    gen = _tile_batches(files, 2, 2, False, shuffle_seed=3, drop_last=True, rank=rank, world=world)
    seen = []
    for epoch in range(2):
        ids = []
        for x, y, n in gen():
            assert n == 2 and x.shape == (2, 1, 4, 4) and y.dtype == torch.uint8
            ids += [int(v) for v in x[:, 0, 0, 0]]          # every tile carries its id in its pixels
        seen.append(ids)
    everyone = [None] * world
    dist.all_gather_object(everyone, (gen.n_batches, seen))
    # gradient exchange: rank r contributes r + 1 everywhere; segments x buckets must touch every element exactly once
    total, n_ops = 1003, 40
    marks = [(10, 700), (22, 420), (31, 90)]
    flat = torch.full((total,), float(rank + 1))
    ranges = []
    for b, e, lo, hi in plan_segments(marks, total, n_ops, min_seg_elems=200):
        for a, z in bucket_ranges(lo, hi, 97):
            dist.all_reduce(flat[a:z], op=dist.ReduceOp.SUM)
            ranges.append((a, z))
    if rank == 0:
        torch.save({"everyone": everyone, "flat": flat, "ranges": ranges}, out)
    dist.destroy_process_group()


def test_data_parallel_host_logic_gloo(tmp_path):
    import torch.multiprocessing as mp
    from unet_b200.geotiff import GeoInfo, write_geotiff
    for sub in ("img_tiles", "mask_tiles"):
        (tmp_path / "trai" / sub).mkdir(parents=True)
    for i in range(11):
        write_geotiff(tmp_path / "trai" / "img_tiles" / f"t{i:02d}.tif", np.full((1, 4, 4), i, dtype=np.uint8), GeoInfo())
        write_geotiff(tmp_path / "trai" / "mask_tiles" / f"t{i:02d}.tif", np.full((4, 4), i % 2, dtype=np.uint8), GeoInfo())
    out = str(tmp_path / "g.pt")
    port = 29500 + (os.getpid() % 500)
    mp.spawn(_ddp_worker, args=(2, port, str(tmp_path), out), nprocs=2, join=True)
    got = torch.load(out, weights_only=False)
    (nb0, seen0), (nb1, seen1) = got["everyone"]
    assert nb0 == nb1 == 2                      # 11 tiles, batch 2, 2 ranks: 5 global batches -> 2 per rank, equal step counts
    for ep in range(2):
        a, b = seen0[ep], seen1[ep]
        assert len(a) == len(b) == 4 and not set(a) & set(b)       # disjoint shares of the same shuffled order
        order = list(range(11))
        np.random.default_rng(3 + ep).shuffle(order)
        assert a == order[0:2] + order[4:6] and b == order[2:4] + order[6:8]   # global batches dealt round-robin
    assert seen0[0] != seen0[1]                                     # reshuffled every epoch
    assert torch.equal(got["flat"], torch.full((1003,), 3.0))       # every gradient element reduced exactly once
    cover = sorted(got["ranges"])
    assert cover[0][0] == 0 and cover[-1][1] == 1003 and all(cover[i][1] == cover[i + 1][0] for i in range(len(cover) - 1))


def test_allreduce_segments_tile_ops_and_gradients():
    """engine.plan_segments: the per-segment all-reduce ranges of the data-parallel step cover the flat gradient buffer
    exactly once, in backward order, and small stages are merged."""
    from unet_b200.engine import plan_segments
    total, n_ops = 41_000_000, 300
    # (op index, offset) in backward order: decoder+post-BN done, then encoder stages 7, 6, 5, 4
    marks = [(120, 21_300_000), (160, 8_200_000), (220, 1_400_000), (260, 260_000), (285, 30_000)]
    segs = plan_segments(marks, total, n_ops, 24 * (1 << 20) // 4)
    assert segs == [(0, 120, 21_300_000, total), (120, 160, 8_200_000, 21_300_000), (160, 220, 1_400_000, 8_200_000),
                    (220, 300, 0, 1_400_000)]
    assert segs[0][0] == 0 and segs[-1][1] == n_ops and all(a[1] == b[0] and a[2] == b[3] for a, b in zip(segs, segs[1:]))
    assert plan_segments(marks, total, n_ops, 10 ** 9) == [(0, n_ops, 0, total)]          # everything merged: one graph
    assert plan_segments([], total, n_ops, 1) == [(0, n_ops, 0, total)]


def _gather_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from unet_b200.predict_engine import gather_mask_strips
    from unet_b200.tiling import compute_windows, shard_windows_by_columns
    Y, X = 37, 101                                   # odd width: strips of 51 and 50 columns
    full = (torch.arange(Y * X, dtype=torch.int64).reshape(Y, X) % 251).to(torch.uint8)
    wins = compute_windows(Y, X, 32, 0.25)
    idx, xb, xe = shard_windows_by_columns(wins, X, rank, world)
    got = gather_mask_strips(full[:, xb:xe].contiguous(), X, rank, world)
    # the 2-D ownership grid (here forced to 1 x 2: one column, two row cells) gathers the same way
    from unet_b200.predict_engine import gather_mask_cells
    from unet_b200.tiling import shard_windows_2d
    _, (cxb, cxe, cyb, cye) = shard_windows_2d(wins, X, Y, rank, world, (1, 2))
    got2 = gather_mask_cells(full[cyb:cye, cxb:cxe].contiguous(), Y, X, (1, 2), rank, world)
    if rank == 0:
        torch.save((got, got2), out)
    else:
        assert got is None and got2 is None
    dist.destroy_process_group()


def test_prediction_strip_gather_gloo(tmp_path):
    """world_size 2: the column strips the ranks own (SURVEY.md 8(e)) reassemble to the full mask on rank 0; every tile is
    run by at least one rank and boundary tile columns by both."""
    import torch.multiprocessing as mp
    from unet_b200.tiling import compute_windows, shard_windows_by_columns
    out = str(tmp_path / "m.pt")
    port = 29500 + ((os.getpid() + 7) % 500)
    mp.spawn(_gather_worker, args=(2, port, out), nprocs=2, join=True)
    Y, X = 37, 101
    full = (torch.arange(Y * X, dtype=torch.int64).reshape(Y, X) % 251).to(torch.uint8)
    g1, g2 = torch.load(out)
    assert torch.equal(g1, full) and torch.equal(g2, full)
    wins = compute_windows(Y, X, 32, 0.25)
    i0, b0, e0 = shard_windows_by_columns(wins, X, 0, 2)
    i1, b1, e1 = shard_windows_by_columns(wins, X, 1, 2)
    assert (b0, e0, b1, e1) == (0, 51, 51, 101) and set(i0) | set(i1) == set(range(len(wins))) and set(i0) & set(i1)


def test_ownership_grid_covers_every_pixel_with_all_its_tiles():
    """tiling.shard_windows_2d: every output pixel belongs to exactly one cell, and the cell's rank runs EVERY tile covering
    that pixel (so sums / counts / argmax are local); the grid chosen for BASELINE configs[2] at 8 ranks is 4 x 2 with
    1104 tiles on the fullest rank (column strips: 1170)."""
    from unet_b200.tiling import compute_windows, shard_grid, shard_windows_2d, shard_windows_by_columns
    Y, X, P = 150, 230, 64
    wins = compute_windows(Y, X, P, 0.25)
    for world, grid in ((4, (2, 2)), (6, (3, 2)), (3, (1, 3))):
        owner = np.full((Y, X), -1)
        for r in range(world):
            idx, (xb, xe, yb, ye) = shard_windows_2d(wins, X, Y, r, world, grid)
            assert (owner[yb:ye, xb:xe] == -1).all()
            owner[yb:ye, xb:xe] = r
            need = {i for i, (x, y, w, h) in enumerate(wins) if x < xe and x + w > xb and y < ye and y + h > yb}
            assert set(idx) == need
        assert (owner >= 0).all()
    big = compute_windows(20000, 20000, 256, 0.125)
    assert shard_grid(big, 20000, 20000, 8) == (4, 2) and shard_grid(big, 20000, 20000, 2) == (2, 1)
    assert max(len(shard_windows_2d(big, 20000, 20000, r, 8, (4, 2))[0]) for r in range(8)) == 1104
    assert max(len(shard_windows_by_columns(big, 20000, r, 8)[0]) for r in range(8)) == 1170


def test_ctypes_signatures_match_the_header():
    """every prototype of include/b2u.h has a ctypes binding with the same number of parameters (a miscounted argtypes
    list would shift every argument after it), and 64-bit parameters of the header are bound as 64-bit."""
    import ctypes
    from unet_b200 import _lib
    lib = _lib.load()
    header = re.sub(r"/\*.*?\*/", " ", open(os.path.join(ROOT, "include", "b2u.h")).read(), flags=re.S)
    protos = re.findall(r"\n(?:int|void|const char\*|size_t)\s+(b2u_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", header)
    assert len(protos) >= 45
    checked = 0
    for name, args in protos:
        params = [a.strip() for a in args.split(",") if a.strip() and a.strip() != "void"]
        fn = getattr(lib, name)
        if fn.argtypes is None:
            continue
        assert len(fn.argtypes) == len(params), (name, len(fn.argtypes), params)
        for ct, decl in zip(fn.argtypes, params):
            if re.match(r"(u?int64_t|size_t)\s", decl):
                assert ctypes.sizeof(ct) == 8, (name, decl)
            elif "*" in decl:
                assert ctypes.sizeof(ct) == ctypes.sizeof(ctypes.c_void_p), (name, decl)
            elif re.match(r"(double)\s", decl):
                assert ct is ctypes.c_double, (name, decl)
        checked += 1
    assert checked >= 40


def test_every_kernel_waits_for_its_predecessor():
    """Programmatic dependent launch: every kernel is launched with programmatic stream serialization (launch_k), so every
    __global__ function must execute griddepcontrol.wait (pdl_enter) before it touches global memory - a kernel that
    does not would race with the tail of its predecessor."""
    csrc = os.path.join(ROOT, "unet_b200", "csrc")
    kernels = 0
    for fn in sorted(os.listdir(csrc)):
        if not fn.endswith(".cu"):
            continue
        src = open(os.path.join(csrc, fn)).read()
        assert "<<<" not in re.sub(r"//.*", "", src), f"{fn}: raw <<< >>> launch bypasses launch_k / the PDL attribute"
        for m in re.finditer(r"__global__\s+void[^{;]*?\b(\w+)\s*\([^{;]*?\)\s*\{", src, flags=re.S):
            # body up to the matching closing brace
            depth, i = 1, m.end()
            while depth and i < len(src):
                depth += {"{": 1, "}": -1}.get(src[i], 0)
                i += 1
            assert "pdl_enter()" in src[m.end():i], f"{fn}: kernel {m.group(1)} never calls pdl_enter()"
            kernels += 1
    assert kernels >= 35


def test_augmentation_is_a_dihedral_transform_of_image_and_mask_together(tmp_path):
    """reference_api.augmented (transforms=True): ceil(B * n_transform_imgs) tiles of every batch get one of the eight flips /
    90-degree rotations, image and mask with the SAME transform, raw integer values untouched (utils.py:196-295 applies its
    pipeline to image and mask together); share 0 changes nothing, a share outside [0, 1] raises as utils.py:236 does."""
    from unet_b200.geotiff import GeoInfo, write_geotiff
    from unet_b200.reference_api import _tile_batches, augmented
    for sub in ("img_tiles", "mask_tiles"):
        (tmp_path / "trai" / sub).mkdir(parents=True)
    rng = np.random.default_rng(0)
    for i in range(8):
        img = rng.integers(0, 256, size=(3, 8, 8), dtype=np.uint8)
        write_geotiff(tmp_path / "trai" / "img_tiles" / f"t{i}.tif", img, GeoInfo())
        write_geotiff(tmp_path / "trai" / "mask_tiles" / f"t{i}.tif", (img[0] > 127).astype(np.uint8), GeoInfo())
    files = sorted((tmp_path / "trai" / "img_tiles").glob("*.tif"))
    plain = list(_tile_batches(files, 4, 2, False, None, False)())
    aug = augmented(_tile_batches(files, 4, 2, False, None, False), 0.5, seed=1)
    assert aug.n_batches == 2
    changed = 0
    for (x0, y0, n0), (x1, y1, n1) in zip(plain, aug()):
        assert n0 == n1 and x1.dtype == torch.uint8
        for i in range(4):
            ok = False
            for op in range(8):
                xi, yi = (x0[i].flip(-1), y0[i].flip(-1)) if op & 4 else (x0[i], y0[i])
                xi, yi = torch.rot90(xi, op & 3, (-2, -1)), torch.rot90(yi, op & 3, (-2, -1))
                ok = ok or (torch.equal(xi, x1[i]) and torch.equal(yi, y1[i]))
            assert ok                                                  # a dihedral transform, mask moved with the image
            assert torch.equal((x1[i][0] > 127).to(torch.uint8), y1[i])    # pixel values untouched, mask still matches
            changed += int(not torch.equal(x0[i], x1[i]))
    assert 1 <= changed <= 4                                           # 2 of 4 tiles per batch were selected (identity allowed)
    same = list(augmented(_tile_batches(files, 4, 2, False, None, False), 0.0)())
    assert all(torch.equal(a[0], b[0]) for a, b in zip(plain, same))
    with pytest.raises(ValueError):
        augmented(_tile_batches(files, 4, 2, False, None, False), 1.5)


def test_gradient_checker_flags_what_it_should():
    """tests/parity_util.gradient_mismatches on synthetic tensors: rounding-sized noise passes; a zeroed, a sign-flipped and a
    5 %-scaled tensor, one corrupted element of a large tensor and a rotated direction are each flagged - and only them."""
    from parity_util import gradient_mismatches
    g = torch.Generator().manual_seed(0)
    ref = {f"t{i}": torch.randn(64, 32, 3, 3, generator=g) for i in range(6)}
    ref["bn"] = torch.randn(64, generator=g)
    noisy = {k: v * (1 + 2.0 ** -8 * torch.randn(v.shape, generator=g)) for k, v in ref.items()}      # ~1 bf16 ulp per element
    check = lambda gr: [b[0] for b in gradient_mismatches(gr, ref, 3e-2, 0.999, 0.1)]
    assert check(noisy) == []
    for name, mutate in (("t0", torch.zeros_like), ("t1", lambda t: -t), ("t2", lambda t: 1.05 * t),
                         ("bn", lambda t: t.roll(1))):
        broken = dict(noisy)
        broken[name] = mutate(noisy[name])
        assert check(broken) == [name], name
    broken = dict(noisy)
    broken["t3"] = noisy["t3"].clone()
    broken["t3"].view(-1)[7] += 0.5 * ref["t3"].abs().max()             # one wrong element: invisible to the L2 norm alone
    assert check(broken) == ["t3"]
    # a tensor that is one cancelling sum passes up to 4 x its measured floor, and not beyond
    ref1, got1 = {"gamma": torch.tensor([1.0])}, {"gamma": torch.tensor([1.2])}
    assert gradient_mismatches(got1, ref1, 3e-2, 0.999, 0.1, floors={"gamma": 0.06}) == []
    assert [b[0] for b in gradient_mismatches(got1, ref1, 3e-2, 0.999, 0.1, floors={"gamma": 0.04})] == ["gamma"]


def test_im2col_stem_identity():
    """The identity behind the im2col stem of the training plan (network.py `stem_im2col`, csrc/glue.cu `im2col_kernel`):
    with lanes ordered c * 9 + ky * 3 + kx (torch `unfold`), the 3x3 stride-2 convolution equals a 1x1 product with the
    weight tensor [Cout][Cin][3][3] READ AS rows of Cin*9 - no re-layout of the master weight - and the gradient of that
    1x1 weight, reshaped, is the convolution's weight gradient."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 4, 18, 22, generator=g)
    w = torch.randn(32, 4, 3, 3, generator=g, requires_grad=True)
    y = F.conv2d(x, w, stride=2, padding=1)
    cols = F.unfold(x, 3, padding=1, stride=2)                      # [N, 36, Ho*Wo]
    w2 = w.detach().reshape(32, 36).clone().requires_grad_(True)
    y2 = (w2 @ cols).view(2, 32, y.shape[2], y.shape[3])
    assert torch.allclose(y, y2, atol=1e-5)
    dy = torch.randn(y.shape, generator=g)
    y.backward(dy)
    y2.backward(dy)
    assert torch.allclose(w.grad.reshape(32, 36), w2.grad, atol=1e-4)


@pytest.mark.parametrize("arch,tv_name", [("xresnet18", "resnet18"), ("xresnet34", "resnet34"), ("xresnet50", "resnet50")])
def test_oracle_residual_stages_equal_torchvision(arch, tv_name):
    """An independent pin of the oracle's encoder (the reference's fastai xresnet cannot be imported): every residual stage
    of the restated body computes exactly what torchvision's ResNet stage computes with the same weights - block order
    conv -> BN -> ReLU, no conv bias next to BN, stride on the 3x3 of a bottleneck, residual add before the last ReLU -
    once torchvision's strided 1x1 shortcut is replaced by the ResNet-D shortcut xresnet uses (AvgPool2d(2, ceil_mode) ->
    1x1 conv -> BN, fastai layers.ResBlock pool_first).  And the parameter totals differ from torchvision's body by the
    stem alone (three 3x3 convolutions + BN vs one 7x7 + BN): SURVEY.md 8(c) sanity check (i)."""
    import torchvision
    from oracle.unet_oracle import xresnet_body
    torch.manual_seed(0)
    body = xresnet_body(arch, 4)
    tv = getattr(torchvision.models, tv_name)(weights=None)
    count = lambda mods: sum(p.numel() for m in mods for p in m.parameters())
    ours_stages, tv_stages = list(body.children())[4:], [tv.layer1, tv.layer2, tv.layer3, tv.layer4]
    assert count(ours_stages) == count(tv_stages)
    stem_ours, stem_tv = count(list(body.children())[:3]), count([tv.conv1, tv.bn1])
    assert count(body.children()) - count([tv.conv1, tv.bn1] + tv_stages) == stem_ours - stem_tv
    x = torch.randn(2, 64, 20, 20)
    for so, st in zip(ours_stages, tv_stages):
        for bo, bt in zip(so, st):
            for m in bo.modules():                      # non-trivial BatchNorm everywhere (BatchZero gamma would hide the path)
                if isinstance(m, torch.nn.BatchNorm2d):
                    m.weight.data.uniform_(0.5, 1.5); m.bias.data.normal_(0, 0.1)
                    m.running_mean.normal_(0, 0.1); m.running_var.uniform_(0.5, 1.5)
            convs = [l[0] for l in bo.convpath]
            bns = [l[1] for l in bo.convpath]
            for i, (c, b) in enumerate(zip(convs, bns), start=1):
                assert c.bias is None
                getattr(bt, f"conv{i}").load_state_dict(c.state_dict())
                getattr(bt, f"bn{i}").load_state_dict(b.state_dict())
                assert getattr(bt, f"conv{i}").stride == c.stride and getattr(bt, f"conv{i}").kernel_size == c.kernel_size
            bt.downsample = bo.idpath if len(bo.idpath) else None      # ResNet-D shortcut (identity when empty)
        for mode in (True, False):
            so.train(mode); st.train(mode)
            with torch.no_grad():
                yo, yt = so(x), st(x)
            assert yo.shape == yt.shape and torch.allclose(yo, yt, atol=1e-5, rtol=1e-5), (arch, mode)
        so.eval()
        with torch.no_grad():
            x = so(x)


def test_oracle_adam_and_dice_equal_independent_implementations():
    """Two more independent pins of the oracle: fastai's Adam with decoupled weight decay as restated in
    oracle.fastai_adam_step (train.py:218 `opt_func=Adam`; eps 1e-5, wd 0.01) is torch.optim.AdamW step for step, and
    oracle.dice_multi (train.py:196 `DiceMulti`) is scikit-learn's macro F1 when every class occurs."""
    from sklearn.metrics import f1_score
    from oracle.unet_oracle import dice_multi, fastai_adam_step
    g = torch.Generator().manual_seed(0)
    p0 = torch.randn(257, generator=g)
    p, m, v = p0.clone(), torch.zeros(257), torch.zeros(257)
    q = torch.nn.Parameter(p0.clone())
    opt = torch.optim.AdamW([q], lr=3e-3, betas=(0.9, 0.99), eps=1e-5, weight_decay=0.01)
    for step in range(1, 8):
        grad = torch.randn(257, generator=g)
        fastai_adam_step(p, grad, m, v, step, lr=3e-3, mom=0.9, sqr_mom=0.99, eps=1e-5, wd=0.01)
        q.grad = grad.clone()
        opt.step()
        assert torch.allclose(p, q.detach(), atol=1e-6, rtol=1e-5), step
    pred = torch.randint(0, 4, (3, 50, 50), generator=g)
    tgt = torch.randint(0, 4, (3, 50, 50), generator=g)
    ref = f1_score(tgt.flatten().numpy(), pred.flatten().numpy(), average="macro")
    assert abs(dice_multi(pred, tgt, 4) - ref) < 1e-12


def test_oracle_merge_equals_fold_on_a_regular_grid():
    """Independent cross-check of the oracle's overlap merge (predict.py:284-326 restated in oracle/stitch.py): where the
    sliding windows form a regular grid, summing overlapping tiles is torch.nn.functional.fold (col2im) and the count is
    the fold of ones - the averaged probabilities and the argmax mask must agree exactly."""
    import torch.nn.functional as F
    from oracle.stitch import merge_pixel_windows, merge_tiles
    from oracle.windows import compute_windows
    P, ov, C = 32, 0.25, 3
    stride = P - int(P * ov)
    H, W = P + 4 * stride, P + 6 * stride                          # (H - P) % stride == 0: no border-snapped window
    wins = compute_windows(H, W, P, ov)
    ys, xs = sorted({w[1] for w in wins}), sorted({w[0] for w in wins})
    assert ys == list(range(0, H - P + 1, stride)) and xs == list(range(0, W - P + 1, stride))
    rng = np.random.default_rng(0)
    preds = [rng.random((C, P, P), dtype=np.float32) for _ in wins]
    mask = merge_pixel_windows(preds, wins, H, W)
    avg, _ = merge_tiles(preds, [[float(x), float(w), 1.0, -float(y), float(h), -1.0] for (x, y, w, h) in wins], all_classes=True)
    order = {(w[1], w[0]): i for i, w in enumerate(wins)}           # fold walks blocks row-major (y outer, x inner)
    cols = torch.stack([torch.from_numpy(preds[order[(y, x)]]).reshape(-1) for y in ys for x in xs], dim=1)[None]
    num = F.fold(cols, (H, W), kernel_size=P, stride=stride)[0]
    cnt = F.fold(torch.ones_like(cols), (H, W), kernel_size=P, stride=stride)[0]
    ref = (num / cnt).numpy()
    assert np.allclose(avg, ref, atol=1e-6)
    assert (mask == ref.argmax(0)).mean() > 0.9999                  # (ties between float sums in another order aside)
