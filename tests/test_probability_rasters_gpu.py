"""Class probability rasters on the B200: `b2u_stitch_finalize_probs` against the numpy restatement, and
`predict_geotiff(all_classes= / specific_class=)` against `save_predictions(merge=True)` over the raster's windows
written as tiles and against the reference merge fed each window's `learn.predict` probabilities."""
import numpy as np
import pytest
import torch

from oracle.stitch import merge_tiles
from test_probability_rasters_cpu import finalize_probs_ref
from unet_b200 import _lib, ops
from unet_b200.geotiff import GeoInfo, read_geotiff, write_geotiff
from unet_b200.reference_api import predict_geotiff, save_predictions, unet_learner_MS
from unet_b200.synth import aerial_like_tiles
from unet_b200.tiling import compute_windows

pytestmark = pytest.mark.gpu

GEO = GeoInfo((383000.0, 0.2, 0.0, 5819000.0, 0.0, -0.2), (1, 1, 0, 3, 1024, 0, 1, 1, 1025, 0, 1, 1, 3072, 0, 1, 25833),
              georeferenced=True)
P = 64


def _accumulators(rng, C, Y, X, large_file):
    """accumulators as the stitch leaves them: counts 0..16, sums of int8-quantised (x31) or fp32 probabilities"""
    cnt = rng.integers(0, 17, size=(Y, X)).astype(np.uint8)
    if large_file:
        acc = (rng.integers(0, 32, size=(C, Y, X)) * cnt / 2).round().astype(np.float32)   # up to 496: wraps
        acc[:, cnt > 0] = np.minimum(acc[:, cnt > 0], 31 * cnt[cnt > 0])
    else:
        acc = (rng.random((C, Y, X)) * cnt).astype(np.float32)
    acc[:, cnt == 0] = 0
    return acc, cnt


def _finalize(acc_d, cnt_d, c0, nc, x0, w, mode, pitch):
    C, Y, X = acc_d.shape
    dt = torch.int8 if mode else torch.float32
    out = torch.full((Y, pitch), 77, dtype=dt, device="cuda")
    _lib.check(_lib.load().b2u_stitch_finalize_probs(acc_d.data_ptr(), cnt_d.data_ptr(), C, Y, X, c0, nc, x0, w, mode,
                                                     out.data_ptr(), pitch, ops.stream_ptr()), "b2u_stitch_finalize_probs")
    return out.cpu().numpy()


@pytest.mark.parametrize("large_file", [False, True])
@pytest.mark.parametrize("C", [1, 2, 5, 32])
def test_kernel_matches_the_restatement(C, large_file):
    rng = np.random.default_rng(C * 2 + large_file)
    Y, X = 37, 2600                                          # rows of several chunks of the kernel
    acc, cnt = _accumulators(rng, C, Y, X, large_file)
    if large_file:
        assert (acc > 127).any()
    acc_d, cnt_d = torch.from_numpy(acc).cuda(), torch.from_numpy(cnt).cuda()
    cases = [(0, C, 0, X), (0, C, 1, 2599), (0, C, 3, 2597), (C // 2, 1, 3, 1031), (0, 1, 1025, 7)]
    if C > 2:
        cases += [(1, C - 2, 5, 2301), (C - 1, 1, 0, X)]
    for c0, nc, x0, w in cases:
        ref = finalize_probs_ref(acc, cnt, c0, nc, x0, w, large_file).reshape(Y, w * nc)
        # tight rows, an unaligned pitch, and 16-byte aligned rows whose chunks end in a partial 16-byte group
        for pitch in (w * nc, w * nc + 13, (w * nc + 15) // 16 * 16 + 16):
            got = _finalize(acc_d, cnt_d, c0, nc, x0, w, int(large_file), pitch)
            assert np.array_equal(got[:, :w * nc], ref), (c0, nc, x0, w, pitch)
            assert (got[:, w * nc:] == 77).all()                 # nothing written beyond w * nc in a row


def test_kernel_rejects_bad_arguments():
    lib = _lib.load()
    acc = torch.zeros((3, 8, 10), device="cuda")
    cnt = torch.zeros((8, 10), dtype=torch.uint8, device="cuda")
    out = torch.zeros(8 * 64, device="cuda")
    good = dict(acc=acc.data_ptr(), cnt=cnt.data_ptr(), C=3, Y=8, X=10, c0=0, nc=3, x0=0, w=10, mode=0,
                out=out.data_ptr(), pitch=30)

    def call(**kw):
        a = dict(good, **kw)
        return lib.b2u_stitch_finalize_probs(a["acc"], a["cnt"], a["C"], a["Y"], a["X"], a["c0"], a["nc"], a["x0"],
                                             a["w"], a["mode"], a["out"], a["pitch"], ops.stream_ptr())

    assert call() == 0
    for bad in (dict(acc=None), dict(cnt=None), dict(out=None), dict(C=0), dict(c0=-1), dict(c0=1), dict(nc=0),
                dict(C=40, nc=33), dict(x0=-1), dict(x0=1), dict(w=0), dict(pitch=29), dict(mode=2), dict(Y=0)):
        assert call(**bad) != 0, bad
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------- predict_geotiff
def _learner(C, seed=1):
    learn = unet_learner_MS(4, C, arch="xresnet18", size=(P, P), batch_size=8)
    learn.net.init_parameters(seed=seed, randomize_bn=True)
    learn._version += 1
    return learn


def _raster(d, dtype, seed=11, H=150, W=200):
    x, _ = aerial_like_tiles(1, 4, H, W, 2, seed=seed)
    img = x[0].numpy()
    if dtype == np.uint16:
        img = (img.astype(np.int32) * 200 + 17).astype(np.uint16)
    write_geotiff(d / "r.tif", img, GEO)
    return d / "r.tif", img


def _tile_route(learn, img, d, ov):
    """the raster's windows written as GeoTIFF tiles, and each window's `learn.predict` probabilities"""
    tdir = d / "aoi" / "tiles"
    tdir.mkdir(parents=True)
    probs, gts = [], []
    for i, (wx, wy, ww, wh) in enumerate(compute_windows(img.shape[1], img.shape[2], P, ov)):
        tile = np.ascontiguousarray(img[:, wy:wy + wh, wx:wx + ww])
        g = GEO.window(wx, wy)
        write_geotiff(tdir / f"img_{i:03d}.tif", tile, GeoInfo(g.geotransform, g.geokeys, georeferenced=True))
        probs.append(learn.predict(torch.from_numpy(tile))[2].numpy())
        gts.append([g.geotransform[0], P, g.geotransform[1], g.geotransform[3], P, g.geotransform[5]])
    return tdir, probs, gts


@pytest.mark.parametrize("C,dtype,ov", [(3, np.uint8, 0.25), (5, np.uint16, 0.25), (3, np.uint16, 0.6),
                                        (5, np.uint8, 0.6), (3, np.uint8, 0.75), (5, np.uint16, 0.75)])
def test_predict_geotiff_matches_the_tile_route(tmp_path, C, dtype, ov):
    learn = _learner(C)
    rpath, img = _raster(tmp_path, dtype)
    H, W = img.shape[1:]
    tdir, probs, gts = _tile_route(learn, img, tmp_path, ov)
    flags = [dict(all_classes=True), dict(specific_class=0), dict(specific_class=C - 1),
             dict(all_classes=True, specific_class=1)]
    for i, f in enumerate(flags):
        for large_file in (False, True):
            for class_zero in ((False, True) if i == 0 else (False,)):
                tag = f"{i}_{int(large_file)}_{int(class_zero)}"
                tiles_out = save_predictions(learn, str(tdir), False, merge=True, large_file=large_file,
                                             class_zero=class_zero, AOI=tag, **f)
                ref_t, geo_t = read_geotiff(tiles_out)
                got, geo = read_geotiff(predict_geotiff(learn, rpath, tmp_path / f"p{tag}.tif", patch_overlap=ov,
                                                        large_file=large_file, class_zero=class_zero, **f))
                bands = C if f.get("all_classes") else 1
                assert got.shape == ref_t.shape == (bands, H, W), tag
                assert got.dtype == ref_t.dtype == (np.int8 if large_file else np.float32), tag
                assert geo.geotransform == geo_t.geotransform == GEO.geotransform and geo.geokeys == GEO.geokeys
                assert geo.nodata is None and geo_t.nodata is None
                ref_o, _ = merge_tiles(probs, gts, large_file=large_file, all_classes=bool(f.get("all_classes")),
                                       specific_class=f.get("specific_class"))
                ref_o = ref_o.reshape(got.shape)
                if class_zero:
                    ref_o = np.where(ref_o == 0, 0, ref_o - 1).astype(ref_o.dtype)
                if large_file:
                    assert np.array_equal(got, ref_t), tag
                    assert np.array_equal(got, ref_o), tag
                else:
                    assert np.abs(got - ref_t).max() <= 1e-6, tag
                    assert np.abs(got - ref_o).max() <= 1e-5, tag


def test_strips_and_ranks_give_the_one_shot_raster(tmp_path):
    learn = _learner(3)
    rpath, _ = _raster(tmp_path, np.uint8, seed=4)
    for large_file in (False, True):
        for f in (dict(all_classes=True), dict(specific_class=2)):
            kw = dict(patch_overlap=0.6, large_file=large_file, **f)
            whole = read_geotiff(predict_geotiff(learn, rpath, tmp_path / "w.tif", **kw))[0]
            outs = [read_geotiff(predict_geotiff(learn, rpath, tmp_path / f"s{n}.tif", max_strip_columns=n, **kw))[0]
                    for n in (45, 70)]
            parts = [predict_geotiff(learn, rpath, tmp_path / "r.tif", rank=r, world=2, **kw) for r in range(2)]
            assert [p.name for p in parts] == ["r.part0.tif", "r.part1.tif"]
            arrs = [read_geotiff(p) for p in parts]
            assert arrs[1][1].geotransform == GEO.window(arrs[0][0].shape[2], 0).geotransform
            outs.append(np.concatenate([a for a, _ in arrs], axis=2))
            for o in outs:
                assert o.shape == whole.shape and o.dtype == whole.dtype
                if large_file:
                    assert np.array_equal(o, whole)
                else:
                    assert np.abs(o - whole).max() <= 1e-6


def test_mask_path_reports_the_argmax(tmp_path):
    learn = _learner(3)
    rpath, img = _raster(tmp_path, np.uint8, seed=6)
    mdir = tmp_path / "masks"
    mdir.mkdir()
    truth = (img[0] // 86).astype(np.uint8)                    # labels 0..2
    write_geotiff(mdir / "m.tif", truth, GEO)
    out = tmp_path / "o.tif"
    reports = [mdir / "o_assessment.json", mdir / "o_assessment_confusion.csv"]
    for f in (dict(all_classes=True, large_file=True), dict(specific_class=1)):
        # the argmax call with the same `large_file` (which changes the argmax: int8 floor division)
        predict_geotiff(learn, rpath, out, patch_overlap=0.25, mask_path=mdir / "m.tif",
                        large_file=f.get("large_file", False))
        argmax_reports = [p.read_bytes() for p in reports]
        for p in reports:
            p.unlink()
        predict_geotiff(learn, rpath, out, patch_overlap=0.25, mask_path=mdir / "m.tif", **f)
        assert [p.read_bytes() for p in reports] == argmax_reports
        plain = predict_geotiff(learn, rpath, tmp_path / "plain.tif", patch_overlap=0.25, **f)
        assert out.read_bytes() == plain.read_bytes()


def test_bad_specific_class_and_regression(tmp_path):
    learn = _learner(3)
    rpath, _ = _raster(tmp_path, np.uint8)
    for k in (3, -1):
        with pytest.raises(ValueError):
            predict_geotiff(learn, rpath, tmp_path / f"bad{k}.tif", specific_class=k)
        assert not (tmp_path / f"bad{k}.tif").exists()
    reg = unet_learner_MS(4, 1, "xresnet18", (P, P), 4, regression=True)
    reg.net.init_parameters(seed=5, randomize_bn=True)
    reg._version += 1
    plain = predict_geotiff(reg, rpath, tmp_path / "reg.tif")
    probs = predict_geotiff(reg, rpath, tmp_path / "reg_all.tif", all_classes=True)
    assert probs.read_bytes() == plain.read_bytes()
