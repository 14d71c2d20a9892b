"""Regression rasters on the B200: `b2u_regression_assess` against float64 numpy, `predict_geotiff` of a regression
model against the tile route and the numpy merge, and the regression `validation_vision` / `mask_path` reports against
scikit-learn over the files they write."""
import csv
import json
import math
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch
from sklearn.metrics import mean_absolute_error, mean_squared_error, r2_score

from unet_b200 import _lib, ops
from unet_b200.assessment import REG_K, MOMENT_FIELDS, RegressionAssessment, RegressionCounter, merge_moments
from unet_b200.geotiff import GeoInfo, read_geotiff, write_geotiff
from unet_b200.reference_api import Learner, predict_geotiff, save_predictions, unet_learner_MS
from unet_b200.synth import aerial_like_tiles
from unet_b200.tiling import compute_windows

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GEO = GeoInfo(geotransform=(383000.0, 0.2, 0.0, 5819000.0, 0.0, -0.2),
              geokeys=(1, 1, 0, 3, 1024, 0, 1, 1, 1025, 0, 1, 1, 3072, 0, 1, 25833), georeferenced=True)
PND, TND = -9999.0, -1.0


def moments(p, t) -> np.ndarray:
    """the record of b2u_regression_assess computed two-pass in float64"""
    p, t = np.asarray(p, np.float64).ravel(), np.asarray(t, np.float64).ravel()
    if p.size == 0:
        return np.zeros(REG_K)
    mt, mp = t.mean(), p.mean()
    dt, dp, e = t - mt, p - mp, p - t
    return np.array([p.size, mt, mp, dt @ dt, dp @ dp, dt @ dp, np.abs(e).sum(), e.sum(), e @ e, t.min(), t.max(),
                     p.min(), p.max(), e.min(), e.max()])


def _valid(p, t, pnd=PND, tnd=TND):
    return np.isfinite(p) & np.isfinite(t) & (p != pnd) & (t != tnd)


def _close(got, ref, rel=1e-12):
    assert got[0] == ref[0]
    if ref[0] == 0:
        return
    scale = np.abs(ref).copy()
    scale[7] = max(scale[7], ref[6])
    scale[5] = max(scale[5], math.sqrt(ref[3] * ref[4]))
    assert np.all(np.abs(got - ref) <= rel * scale), list(zip(MOMENT_FIELDS, (got - ref) / np.maximum(scale, 1e-300)))
    assert np.array_equal(got[9:], ref[9:])


# (T, H, W, column offset of pred, column offset of truth, row pitch): odd widths, rows at the same and at different
# 16-byte offsets, unaligned starts, images further apart than H rows, rows long enough for the four-chunk loop
LAYOUTS = [(1, 37, 53, 0, 0, None), (3, 29, 301, 1, 1, 333), (3, 17, 130, 2, 3, 150), (64, 16, 40, 0, 0, None),
           (64, 9, 67, 3, 1, 75), (1, 9, 5000, 3, 3, 5011)]


def _maps(rng, T, H, W, op, ot, pitch, offset=0.0, spread=1.0):
    pitch = pitch or W
    t = (offset + spread * rng.standard_normal((T, H + 2, pitch + 8))).astype(np.float32)
    p = (t + 0.3 * spread * rng.standard_normal(t.shape)).astype(np.float32)
    for a, nd in ((p, PND), (t, TND)):
        for v in (np.nan, np.inf, -np.inf, nd):
            a[rng.random(a.shape) < 0.01] = v
    pv, tv = p[:, :H, op:op + W], t[:, :H, ot:ot + W]
    pd, td = torch.from_numpy(p).cuda(), torch.from_numpy(t).cuda()
    return pv, tv, pd[:, :H, op:op + W], td[:, :H, ot:ot + W]


def _launch(pv, tv, totals, tiles, skipped, scratch, n_scratch, ticket):
    T, H, W = pv.shape
    _lib.check(_lib.load().b2u_regression_assess(pv.data_ptr(), pv.stride(1), pv.stride(0), tv.data_ptr(), tv.stride(1),
                                                 tv.stride(0), T, H, W, PND, TND, totals.data_ptr(),
                                                 None if tiles is None else tiles.data_ptr(), skipped.data_ptr(),
                                                 scratch.data_ptr(), n_scratch, ticket.data_ptr(), ops.stream_ptr()),
               "b2u_regression_assess")


@pytest.mark.parametrize("layout", LAYOUTS, ids=lambda l: "x".join(map(str, l[:3])) + f"_o{l[3]}{l[4]}")
def test_kernel_matches_numpy(layout):
    T, H, W, op, ot, pitch = layout
    rng = np.random.default_rng(T * 1000 + W)
    p_np, t_np, pv, tv = _maps(rng, T, H, W, op, ot, pitch)
    assert pv.stride(0) > pv.stride(1) * H                  # images further apart than their rows
    totals = torch.zeros(REG_K, dtype=torch.float64, device="cuda")
    tiles = torch.zeros((T, REG_K), dtype=torch.float64, device="cuda")
    skipped = torch.zeros(1, dtype=torch.int64, device="cuda")
    n_scratch = 1184 + T
    scratch = torch.empty(n_scratch * REG_K, dtype=torch.float64, device="cuda")
    ticket = torch.zeros(1, dtype=torch.int32, device="cuda")
    _launch(pv, tv, totals, tiles, skipped, scratch, n_scratch, ticket)
    first, first_tiles, first_skip = totals.cpu().numpy().copy(), tiles.cpu().numpy().copy(), int(skipped.item())
    ok = _valid(p_np, t_np)
    _close(first, moments(p_np[ok], t_np[ok]))
    assert first_skip == int((~ok).sum()) > 0
    for i in range(T):
        _close(first_tiles[i], moments(p_np[i][ok[i]], t_np[i][ok[i]]))
    assert int(ticket.item()) == 0
    # a second call accumulates: the record of the sample taken twice
    _launch(pv, tv, totals, tiles, skipped, scratch, n_scratch, ticket)
    _close(totals.cpu().numpy(), merge_moments(first, first))
    assert int(skipped.item()) == 2 * first_skip
    for i in range(T):
        _close(tiles.cpu().numpy()[i], merge_moments(first_tiles[i], first_tiles[i]))
    # fewer scratch records: fewer blocks, the same statistics
    totals.zero_()
    _launch(pv, tv, totals, None, skipped, scratch, T, ticket)
    _close(totals.cpu().numpy(), first)


@pytest.mark.parametrize("T", [1, 3, 64])
def test_offset_data_r2_and_bit_identical_reruns(T):
    rng = np.random.default_rng(T)
    p_np, t_np, pv, tv = _maps(rng, T, 300 // T + 20, 517, 1, 1, 530, offset=1000.0, spread=0.01)
    ok = _valid(p_np, t_np)
    bufs = []
    for _ in range(2):
        c = RegressionCounter("cuda", tile_slots=T, pred_nodata=PND, truth_nodata=TND)
        c.count(pv, tv, per_tile=True)
        bufs.append(c.buf.cpu())
    assert torch.equal(bufs[0].view(torch.int64), bufs[1].view(torch.int64))
    totals, skipped, recs = c.read()
    p_ok, t_ok = p_np[ok].astype(np.float64), t_np[ok].astype(np.float64)
    a = RegressionAssessment.from_moments(totals, skipped)
    assert a.n == p_ok.size and skipped == int((~ok).sum())
    assert abs(a.r2 - r2_score(t_ok, p_ok)) <= 1e-9
    assert a.rmse == pytest.approx(math.sqrt(mean_squared_error(t_ok, p_ok)), rel=1e-9)
    assert a.truth_std == pytest.approx(t_ok.std(), rel=1e-9)
    assert recs.shape == (1, T, REG_K)
    _close(totals, moments(p_ok, t_ok), rel=1e-10)


def test_kernel_rejects_bad_arguments():
    lib = _lib.load()
    a = torch.zeros((4, 8), dtype=torch.float32, device="cuda")
    r = torch.zeros(4 * REG_K + 16, dtype=torch.float64, device="cuda")
    tk = torch.zeros(1, dtype=torch.int32, device="cuda")
    # totals, skipped, then scratch records
    p, d, st = a.data_ptr(), r.data_ptr(), ops.stream_ptr()
    good = dict(pred=p, pp=8, ps=32, truth=p, tp=8, ts=32, T=1, H=4, W=8, totals=d, skipped=d + 8 * REG_K,
                scratch=d + 8 * (REG_K + 1), ns=1, ticket=tk.data_ptr())

    def call(**kw):
        g = {**good, **kw}
        return lib.b2u_regression_assess(g["pred"], g["pp"], g["ps"], g["truth"], g["tp"], g["ts"], g["T"], g["H"], g["W"],
                                         PND, TND, g["totals"], None, g["skipped"], g["scratch"], g["ns"], g["ticket"], st)
    _lib.check(call())
    for bad in (dict(pred=None), dict(truth=None), dict(totals=None), dict(skipped=None), dict(scratch=None),
                dict(ticket=None), dict(T=0), dict(T=70000), dict(H=0), dict(W=0), dict(pp=7), dict(tp=7),
                dict(T=2, ps=24, ns=2), dict(T=2, ts=24, ns=2), dict(T=2, ns=1), dict(pred=p + 2)):
        with pytest.raises(_lib.B2UError):
            _lib.check(call(**bad), "b2u_regression_assess")
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------------------------------- predict_geotiff
P, B = 64, 4


def _learner(batch=B) -> Learner:
    learn = unet_learner_MS(4, 1, "xresnet18", (P, P), batch, regression=True)
    learn.net.init_parameters(seed=5, randomize_bn=True)
    learn._version += 1
    return learn


def _raster(d, H=150, W=200):
    x, _ = aerial_like_tiles(1, 4, H, W, 2, seed=12)
    img = x[0].numpy().copy()
    img[:, 10:20, 30:60] = 0                                  # image no-data
    msk = ((img[3].astype(np.float32) - img[0]) / 64.0 + 1.0).astype(np.float32)
    msk[100:110, 5:40] = -1.0                                 # mask no-data
    msk[40:44, 150:170] = 0.0                                 # a real value, counted
    write_geotiff(d / "r.tif", img, GEO, nodata=0)
    write_geotiff(d / "m.tif", msk, GEO, nodata=-1)
    return d / "r.tif", d / "m.tif"


def test_predict_geotiff_regression_matches_tile_route(tmp_path):
    from oracle.stitch import merge_tiles
    learn = _learner(8)
    raster, _ = _raster(tmp_path)
    img = read_geotiff(raster)[0]
    H, W, ov = img.shape[1], img.shape[2], 0.25
    tdir = tmp_path / "aoi" / "tiles"
    tdir.mkdir(parents=True)
    vals, gts = [], []
    for i, (wx, wy, ww, wh) in enumerate(compute_windows(H, W, P, ov)):
        g = GEO.window(wx, wy)
        write_geotiff(tdir / f"img_{i:03d}.tif", img[:, wy:wy + wh, wx:wx + ww], GeoInfo(g.geotransform, g.geokeys,
                                                                                           georeferenced=True))
        vals.append(learn.predict(torch.from_numpy(img[:, wy:wy + wh, wx:wx + ww].copy()))[1].numpy())
        gts.append([g.geotransform[0], P, g.geotransform[1], g.geotransform[3], P, g.geotransform[5]])
    merged = save_predictions(learn, str(tdir), True, merge=True, AOI="aoi")
    ref_tiles, ref_geo = read_geotiff(merged)
    ref_np, _ = merge_tiles(vals, gts, regression=True)
    out = predict_geotiff(learn, raster, tmp_path / "p.tif", patch_overlap=ov, large_file=True)   # no effect
    got, geo = read_geotiff(out)
    assert got.dtype == np.float32 and got.shape == (1, H, W) and geo.nodata == -9999
    assert geo.geotransform == ref_geo.geotransform == GEO.geotransform
    # the same batched network outputs as the tile route; `learn.predict` runs each tile on its own
    assert np.allclose(got[0], ref_tiles[0], rtol=1e-5, atol=1e-5) and np.allclose(got[0], ref_np, rtol=1e-5, atol=1e-5)
    assert not (got == -9999).any()                          # the windows cover the raster
    scale = np.abs(got).max()
    narrow, _ = read_geotiff(predict_geotiff(learn, raster, tmp_path / "n.tif", patch_overlap=ov, max_strip_columns=45))
    assert np.abs(narrow - got).max() <= 1e-6 * scale
    parts = [predict_geotiff(learn, raster, tmp_path / "w.tif", patch_overlap=ov, rank=r, world=2) for r in range(2)]
    assert [p.name for p in parts] == ["w.part0.tif", "w.part1.tif"]
    arrs = [read_geotiff(p) for p in parts]
    assert all(a.dtype == np.float32 and g.nodata == -9999 for a, g in arrs)
    assert arrs[1][1].geotransform == GEO.window(arrs[0][0].shape[2], 0).geotransform
    assert np.abs(np.concatenate([a for a, _ in arrs], axis=2) - got).max() <= 1e-6 * scale


def test_predict_geotiff_regression_mask_assessment(tmp_path):
    learn = _learner()
    raster, mask = _raster(tmp_path)
    out = predict_geotiff(learn, raster, tmp_path / "p.tif", mask_path=mask)
    plain = predict_geotiff(learn, raster, tmp_path / "q.tif")
    assert read_geotiff(out)[0].tobytes() == read_geotiff(plain)[0].tobytes()      # mask_path changes no output
    doc = json.loads((tmp_path / "p_assessment.json").read_text())
    pred = read_geotiff(out)[0][0].astype(np.float64)
    img = read_geotiff(raster)[0]
    truth = read_geotiff(mask)[0][0].astype(np.float64)
    bad = (img == 0).any(axis=0) | (truth == -1)
    assert bad[100:110, 5:40].all() and bad[10:20, 30:60].all() and not bad[40:44, 150:170].any()
    p, t = pred[~bad], truth[~bad]
    assert doc["n"] == p.size and doc["skipped"] == int(bad.sum())
    assert doc["mae"] == pytest.approx(mean_absolute_error(t, p), rel=1e-9)
    assert doc["rmse"] == pytest.approx(math.sqrt(mean_squared_error(t, p)), rel=1e-9)
    assert doc["r2"] == pytest.approx(r2_score(t, p), rel=1e-9, abs=1e-9)
    assert doc["bias"] == pytest.approx((p - t).mean(), rel=1e-9, abs=1e-12)
    assert doc["prediction"] == str(out) and doc["mask"] == str(mask)
    # two ranks: the merged moments of their reports give the one-rank report.  A rank stitches its strip's tiles in
    # its own colour-class order, so its fp32 means may differ from the one-rank raster in the last bit: the merge is
    # held to 1e-12 against the values the ranks wrote, and to rounding against the one-rank report.
    parts = [predict_geotiff(learn, raster, tmp_path / "w.tif", rank=r, world=2, mask_path=mask) for r in range(2)]
    docs = [json.loads((tmp_path / f"w.part{r}_assessment.json").read_text()) for r in range(2)]
    m = merge_moments(*[np.array([d["moments"][k] for k in MOMENT_FIELDS]) for d in docs])
    a = RegressionAssessment.from_moments(m, sum(d["skipped"] for d in docs))
    assert a.n == doc["n"] and a.skipped == doc["skipped"]
    pw = np.concatenate([read_geotiff(q)[0][0] for q in parts], axis=1).astype(np.float64)[~bad]
    assert np.abs(pw - p).max() <= 1e-6 * np.abs(p).max()
    ref = RegressionAssessment.from_moments(moments(pw, t))
    for k in ("mae", "mse", "rmse", "bias", "r2", "pearson_r", "truth_mean", "pred_mean", "truth_std", "pred_std"):
        assert getattr(a, k) == pytest.approx(getattr(ref, k), rel=1e-12, abs=1e-12), k
        assert getattr(a, k) == pytest.approx(doc[k], rel=1e-6, abs=1e-9), k
    # streamed strips count the same pixels
    predict_geotiff(learn, raster, tmp_path / "s.tif", mask_path=mask, max_strip_columns=45)
    ds = json.loads((tmp_path / "s_assessment.json").read_text())
    assert ds["n"] == doc["n"] and ds["skipped"] == doc["skipped"] and ds["rmse"] == pytest.approx(doc["rmse"], rel=1e-6)
    # a mask on another grid
    write_geotiff(tmp_path / "small.tif", truth[:, :160].astype(np.float32), GEO)
    with pytest.raises(ValueError):
        predict_geotiff(learn, raster, tmp_path / "o.tif", mask_path=tmp_path / "small.tif")


# -------------------------------------------------------------------------------------------------- save_predictions
def _tiles(root, n=10, suffix=".tif"):
    """n overlapping tiles on a 5-column grid with float32 mask tiles (some declaring no-data pixels): n % B != 0 pads
    the last batch"""
    x, _ = aerial_like_tiles(n, 4, P, P, 2, seed=11)
    for sub in ("img_tiles", "mask_tiles"):
        (root / sub).mkdir(parents=True)
    gts = {}
    for i in range(n):
        g = GEO.window((i % 5) * 48, (i // 5) * 48)
        name = f"t{i:02d}{suffix}"
        y = ((x[i, 3].float() - x[i, 0].float()) / 64.0 + 1.0).numpy()
        if i % 3 == 0:
            y[5:9, 10:30] = -1.0
        if suffix == ".tif":
            write_geotiff(root / "img_tiles" / name, x[i].numpy(), g)
            write_geotiff(root / "mask_tiles" / name, y, g, nodata=-1 if i % 3 == 0 else None)
        else:
            np.save(root / "img_tiles" / name, x[i].numpy())
            np.save(root / "mask_tiles" / name, y)
        gts[name] = g.geotransform
    return root / "img_tiles", gts


def _read_csv(path):
    with open(path, newline="") as f:
        return list(csv.reader(f))


def test_save_predictions_regression_validation_vision(tmp_path):
    learn = _learner()
    tiles, _ = _tiles(tmp_path)
    outs = save_predictions(learn, tiles, regression=True, validation_vision=True)
    out_dir = tmp_path / "predicted_tiles_model"
    doc = json.loads((out_dir / "model_validation.json").read_text())
    names = sorted(p.name for p in outs)
    assert len(names) == 10 and len(names) % B != 0
    pred = np.stack([read_geotiff(out_dir / nm)[0][0] for nm in names]).astype(np.float64)
    mtiles = [read_geotiff(tiles.parent / "mask_tiles" / nm) for nm in names]
    truth = np.stack([a[0] for a, _ in mtiles]).astype(np.float64)
    skip = np.stack([(a[0] == g.nodata) if g.nodata is not None else np.zeros(a[0].shape, bool) for a, g in mtiles])
    p, t = pred[~skip], truth[~skip]
    assert doc["n"] == p.size and doc["skipped"] == int(skip.sum()) > 0 and doc["tiles"] == 10
    assert doc["mae"] == pytest.approx(mean_absolute_error(t, p), rel=1e-9)
    assert doc["mse"] == pytest.approx(mean_squared_error(t, p), rel=1e-9)
    assert doc["r2"] == pytest.approx(r2_score(t, p), rel=1e-9, abs=1e-9)
    rows = _read_csv(out_dir / "model_validation_tile_metrics.csv")
    assert rows[0] == ["tile", "n", "mae", "rmse", "bias", "truth_mean", "pred_mean"]
    assert [r[0] for r in rows[1:]] == names
    for r, pi, ti, si in zip(rows[1:], pred, truth, skip):
        pk, tk = pi[~si], ti[~si]
        assert int(r[1]) == pk.size
        ref = [np.abs(pk - tk).mean(), math.sqrt(((pk - tk) ** 2).mean()), (pk - tk).mean(), tk.mean(), pk.mean()]
        assert [float(v) for v in r[2:]] == pytest.approx(ref, rel=1e-9, abs=1e-12)
    # the outputs do not depend on validation_vision
    before = {o.name: o.read_bytes() for o in outs}
    assert {o.name: o.read_bytes() for o in save_predictions(learn, tiles, regression=True)} == before
    # the merge counts each tile's raw prediction once: the same report
    merged = save_predictions(learn, tiles, regression=True, merge=True, validation_vision=True)
    mdoc = json.loads((tmp_path / "model_validation.json").read_text())
    assert mdoc["n"] == doc["n"] and mdoc["skipped"] == doc["skipped"] and mdoc["tiles"] == doc["tiles"]
    for k in ("mae", "mse", "rmse", "bias", "r2", "pearson_r", "truth_mean", "pred_mean"):
        assert mdoc[k] == pytest.approx(doc[k], rel=1e-12, abs=1e-12), k
    assert [r[:2] for r in _read_csv(tmp_path / "model_validation_tile_metrics.csv")] == [r[:2] for r in rows]
    mb = merged.read_bytes()
    merged.unlink()
    assert save_predictions(learn, tiles, regression=True, merge=True).read_bytes() == mb


def test_save_predictions_regression_npy_tiles_and_missing_mask(tmp_path):
    learn = _learner()
    tiles, gts = _tiles(tmp_path, n=6, suffix=".npy")
    save_predictions(learn, tiles, regression=True, validation_vision=True)
    doc = json.loads((tmp_path / "predicted_tiles_model" / "model_validation.json").read_text())
    assert doc["n"] == 6 * P * P and doc["skipped"] == 0           # .npy masks declare no no-data value
    (tmp_path / "mask_tiles" / "t04.npy").unlink()
    shutil.rmtree(tmp_path / "predicted_tiles_model")
    for merge in (False, True):
        with pytest.raises(FileNotFoundError):
            save_predictions(learn, tiles, regression=True, merge=merge, validation_vision=True, geotransforms=gts)
        assert not (tmp_path / "predicted_tiles_model").exists()
        assert not list(tmp_path.glob("*prediction*")) and not list(tmp_path.glob("*validation*"))


# ------------------------------------------------------------------------------------------------------ two GPUs
WORKER = """
import sys
sys.path.insert(0, {root!r})
from unet_b200.engine import init_distributed
from unet_b200.reference_api import save_predictions
init_distributed()
save_predictions({model!r}, {tiles!r}, regression=True, merge={merge}, validation_vision=True)
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
@pytest.mark.parametrize("merge", [False, True])
def test_regression_validation_on_two_gpus_matches_one(tmp_path, merge):
    learn = _learner()
    learn.export(tmp_path / "m.pkl")
    one, _ = _tiles(tmp_path / "one")
    two = tmp_path / "two" / "img_tiles"
    shutil.copytree(tmp_path / "one", tmp_path / "two")
    save_predictions(str(tmp_path / "m.pkl"), one, regression=True, merge=merge, validation_vision=True)
    script = tmp_path / "worker.py"
    script.write_text(WORKER.format(root=ROOT, model=str(tmp_path / "m.pkl"), tiles=str(two), merge=merge))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29743", str(script)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    sub = "" if merge else "predicted_tiles_m"
    a = json.loads((tmp_path / "one" / sub / "m_validation.json").read_text())
    b = json.loads((tmp_path / "two" / sub / "m_validation.json").read_text())
    assert a["n"] == b["n"] and a["skipped"] == b["skipped"] and a["tiles"] == b["tiles"] == 10
    for k in ("mae", "mse", "rmse", "bias", "r2", "pearson_r", "truth_mean", "pred_mean", "truth_std", "pred_std"):
        assert b[k] == pytest.approx(a[k], rel=1e-12, abs=1e-12), k
    ra = _read_csv(tmp_path / "one" / sub / "m_validation_tile_metrics.csv")
    rb = _read_csv(tmp_path / "two" / sub / "m_validation_tile_metrics.csv")
    assert [r[:2] for r in ra] == [r[:2] for r in rb]
