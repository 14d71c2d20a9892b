"""Accuracy assessment on the B200: `b2u_confusion_counts` against numpy, `save_predictions(validation_vision=True)`
and `predict_geotiff(mask_path=)` against scikit-learn over the files they write."""
import json
import os
import shutil
import subprocess
import sys
import warnings

import numpy as np
import pytest
import torch
from sklearn.metrics import accuracy_score, cohen_kappa_score, confusion_matrix, precision_recall_fscore_support

from unet_b200 import _lib, ops
from unet_b200.create_tiles import mask_tile_values, prepare_raster
from unet_b200.geotiff import GeoInfo, read_geotiff, write_geotiff
from unet_b200.reference_api import Learner, predict_geotiff, save_predictions, unet_learner_MS
from unet_b200.synth import aerial_like_tiles

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GEO = GeoInfo(geotransform=(383000.0, 0.2, 0.0, 5819000.0, 0.0, -0.2),
              geokeys=(1, 1, 0, 3, 1024, 0, 1, 1, 1025, 0, 1, 1, 3072, 0, 1, 25833), georeferenced=True)


def _numpy_counts(pred, truth, C):
    valid = (pred < C) & (truth < C)
    joint = np.bincount(truth[valid].astype(np.int64) * C + pred[valid], minlength=C * C).reshape(C, C)
    hist = np.stack([np.stack([np.bincount(t[v], minlength=C), np.bincount(p[v], minlength=C)])
                     for p, t, v in zip(pred, truth, valid)])
    return joint, int((~valid).sum()), hist


# (T, H, W, column offset of pred, column offset of truth, row pitch): widths that are not multiples of 16, rows at the
# same and at different 16-byte offsets, and rows long enough for the four-chunk loop
LAYOUTS = [(5, 37, 53, 0, 0, None), (3, 64, 64, 0, 0, None), (1, 29, 301, 5, 5, 333), (2, 17, 130, 7, 3, 150),
           (1, 9, 5000, 3, 3, 5011)]


@pytest.mark.parametrize("layout", LAYOUTS, ids=lambda l: "x".join(map(str, l[:3])) + f"_o{l[3]}{l[4]}")
@pytest.mark.parametrize("C", [1, 2, 3, 8, 9, 31, 32])
def test_confusion_counts_match_numpy(C, layout):
    T, H, W, op, ot, pitch = layout
    rng = np.random.default_rng(C * 100 + W)
    pitch = pitch or W

    def plane():
        a = rng.integers(0, C, size=(T, H, pitch + 8), dtype=np.uint8)
        # land-cover-like runs of one class, and values >= C that must be skipped
        a[:, :, : (pitch + 8) // 2] = rng.integers(0, C)
        bad = rng.random(a.shape) < 0.03
        a[bad] = rng.integers(C, 256, size=int(bad.sum()))
        return a

    pbuf, tbuf = plane(), plane()
    pred_np, truth_np = pbuf[:, :, op:op + W], tbuf[:, :, ot:ot + W]
    pd, td = torch.from_numpy(pbuf).cuda(), torch.from_numpy(tbuf).cuda()
    pv, tv = pd[:, :, op:op + W], td[:, :, ot:ot + W]
    joint = torch.zeros(C * C, dtype=torch.int64, device="cuda")
    hist = torch.zeros(T * 2 * C, dtype=torch.int32, device="cuda")
    skipped = torch.zeros(1, dtype=torch.int64, device="cuda")
    lib = _lib.load()
    for _ in range(2):
        _lib.check(lib.b2u_confusion_counts(pv.data_ptr(), pv.stride(1), pv.stride(0), tv.data_ptr(), tv.stride(1),
                                            tv.stride(0), T, H, W, C, joint.data_ptr(), hist.data_ptr(),
                                            skipped.data_ptr(), ops.stream_ptr()), "b2u_confusion_counts")
        if _ == 0:
            j1, s1, h1 = joint.cpu().numpy().copy(), int(skipped.item()), hist.cpu().numpy().copy()
    ref_j, ref_s, ref_h = _numpy_counts(pred_np, truth_np, C)
    assert np.array_equal(j1.reshape(C, C), ref_j)
    assert s1 == ref_s and (ref_s > 0 or C == 32)
    assert np.array_equal(h1.reshape(T, 2, C), ref_h)
    # a second launch accumulates: exactly twice the counts
    assert np.array_equal(joint.cpu().numpy(), 2 * j1)
    assert int(skipped.item()) == 2 * s1
    assert np.array_equal(hist.cpu().numpy(), 2 * h1)


def test_confusion_counts_rejects_bad_arguments():
    lib = _lib.load()
    a = torch.zeros((4, 4), dtype=torch.uint8, device="cuda")
    j = torch.zeros(33 * 33, dtype=torch.int64, device="cuda")
    for C, pitch in ((0, 4), (33, 4), (2, 3)):
        with pytest.raises(_lib.B2UError):
            _lib.check(lib.b2u_confusion_counts(a.data_ptr(), pitch, 16, a.data_ptr(), 4, 16, 1, 4, 4, C, j.data_ptr(),
                                                None, j.data_ptr(), ops.stream_ptr()))


# ------------------------------------------------------------------------------------------------ save_predictions
N_CLASSES, P, B = 3, 64, 4


def _learner() -> Learner:
    learn = unet_learner_MS(4, N_CLASSES, "xresnet18", (P, P), B)
    learn.net.init_parameters(seed=3, randomize_bn=True)      # varied predictions over all classes
    learn._version += 1
    return learn


def _tiles(root, n=10, suffix=".tif"):
    """n overlapping tiles on a 5-column grid (stride 48 px) with their mask tiles: n % B != 0 pads the last batch"""
    x, y = aerial_like_tiles(n, 4, P, P, N_CLASSES, seed=11)
    for sub in ("img_tiles", "mask_tiles"):
        (root / sub).mkdir(parents=True)
    gts = {}
    for i in range(n):
        g = GEO.window((i % 5) * 48, (i // 5) * 48)
        name = f"t{i:02d}{suffix}"
        if suffix == ".tif":
            write_geotiff(root / "img_tiles" / name, x[i].numpy(), g)
            write_geotiff(root / "mask_tiles" / name, y[i].numpy(), g)
        else:
            np.save(root / "img_tiles" / name, x[i].numpy())
            np.save(root / "mask_tiles" / name, y[i].numpy())
        gts[name] = g.geotransform
    return root / "img_tiles", gts


def _sk_report(pred, truth):
    labels = list(range(N_CLASSES))
    cm = confusion_matrix(truth.ravel(), pred.ravel(), labels=labels)
    p, r, f, s = precision_recall_fscore_support(truth.ravel(), pred.ravel(), labels=labels, zero_division=0)
    return cm, accuracy_score(truth.ravel(), pred.ravel()), p, r, f, s, cohen_kappa_score(truth.ravel(), pred.ravel())


def _check_report(doc, pred, truth):
    cm, acc, p, r, f, s, k = _sk_report(pred, truth)
    assert doc["confusion"] == cm.tolist() and doc["skipped_pixels"] == 0 and doc["pixels"] == truth.size
    assert doc["accuracy"] == pytest.approx(acc) and doc["kappa"] == pytest.approx(k)
    for c in range(N_CLASSES):
        pc = doc["per_class"][str(c)]
        assert (pc["precision"], pc["recall"], pc["f1"], pc["support"]) == pytest.approx((p[c], r[c], f[c], s[c]))


@pytest.mark.parametrize("suffix", [".tif", ".npy"])
def test_save_predictions_validation_vision(tmp_path, suffix):
    learn = _learner()
    tiles, gts = _tiles(tmp_path, suffix=suffix)
    gkw = {} if suffix == ".tif" else {"geotransforms": gts}
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        outs = save_predictions(learn, tiles, validation_vision=True, **gkw)
    out_dir = tmp_path / "predicted_tiles_model"
    doc = json.loads((out_dir / "model_validation.json").read_text())
    names = sorted(p.name for p in outs)
    load = (lambda p: read_geotiff(p)[0][0]) if suffix == ".tif" else np.load
    pred = np.stack([load(out_dir / nm) for nm in names])
    truth = np.stack([load(tiles.parent / "mask_tiles" / nm) for nm in names])
    assert len(pred) % B != 0
    _check_report(doc, pred, truth)
    majority = lambda a: np.argmax(np.bincount(a.ravel(), minlength=N_CLASSES))
    tm = np.zeros((N_CLASSES, N_CLASSES), np.int64)
    for pt, tt in zip(pred, truth):
        tm[majority(tt), majority(pt)] += 1
    assert doc["tile_confusion"] == tm.tolist() and doc["tiles"] == len(pred)
    assert (out_dir / "model_validation_confusion.csv").exists()
    assert (out_dir / "model_validation_tile_confusion.csv").exists()
    before = {p.name: p.read_bytes() for p in outs}
    # validation_vision=False writes the same predictions
    outs2 = save_predictions(learn, tiles, validation_vision=False, **gkw)
    assert {p.name: p.read_bytes() for p in outs2} == before
    # the merge counts each tile's argmax once: the same report
    merged = save_predictions(learn, tiles, merge=True, validation_vision=True, **gkw)
    assert json.loads((tmp_path / "model_validation.json").read_text()) == doc
    merged_bytes = merged.read_bytes()
    merged.unlink()
    assert save_predictions(learn, tiles, merge=True, **gkw).read_bytes() == merged_bytes


def test_save_predictions_checks_masks_before_predicting(tmp_path):
    learn = _learner()
    tiles, _ = _tiles(tmp_path)
    (tmp_path / "mask_tiles" / "t07.tif").unlink()
    with pytest.raises(FileNotFoundError):
        save_predictions(learn, tiles, validation_vision=True)
    assert not (tmp_path / "predicted_tiles_model").exists()
    write_geotiff(tmp_path / "mask_tiles" / "t07.tif", np.full((P, P), N_CLASSES, np.uint8), GEO)
    with pytest.raises(ValueError):
        save_predictions(learn, tiles, validation_vision=True)


# --------------------------------------------------------------------------------------------------- predict_geotiff
def _raster(d, H=150, W=170):
    x, y = aerial_like_tiles(1, 4, H, W, 2, seed=21)
    img, msk = x[0].numpy().copy(), y[0].numpy().copy()
    img[:, 10:20, 30:60] = 0                                  # image no-data
    msk[100:110, 5:40] = 255                                  # mask no-data
    write_geotiff(d / "r.tif", img, GEO, nodata=0)
    write_geotiff(d / "m.tif", msk, GEO, nodata=255)
    return d / "r.tif", d / "m.tif"


def test_predict_geotiff_mask_assessment(tmp_path):
    learn = _learner()
    raster, mask = _raster(tmp_path)
    plain = predict_geotiff(learn, raster, tmp_path / "plain.tif")
    ids = read_geotiff(plain)[0][0]                           # model class ids (no class_zero un-shift)
    for class_zero in (False, True):
        out = predict_geotiff(learn, raster, tmp_path / f"p{int(class_zero)}.tif", class_zero=class_zero, mask_path=mask)
        doc = json.loads((tmp_path / f"p{int(class_zero)}_assessment.json").read_text())
        labels = mask_tile_values(prepare_raster(raster, mask, P, 0.125, 0.9, class_zero).mask[0])
        _check_report(doc, ids, labels)
        ref = predict_geotiff(learn, raster, tmp_path / "ref.tif", class_zero=class_zero)
        assert out.read_bytes() == ref.read_bytes()           # the written mask does not depend on mask_path
        narrow = predict_geotiff(learn, raster, tmp_path / "n.tif", class_zero=class_zero, mask_path=mask,
                                 max_strip_columns=45)
        assert json.loads((tmp_path / "n_assessment.json").read_text())["confusion"] == doc["confusion"]
        assert narrow.read_bytes() == out.read_bytes()
        parts = [predict_geotiff(learn, raster, tmp_path / "w.tif", class_zero=class_zero, rank=r, world=2,
                                 mask_path=mask) for r in range(2)]
        assert [p.name for p in parts] == ["w.part0.tif", "w.part1.tif"]
        cms = [np.array(json.loads((tmp_path / f"w.part{r}_assessment.json").read_text())["confusion"]) for r in range(2)]
        assert (cms[0] + cms[1]).tolist() == doc["confusion"]


def test_predict_geotiff_mask_errors(tmp_path):
    learn = _learner()
    raster, mask = _raster(tmp_path)
    x, _ = aerial_like_tiles(1, 1, 150, 160, 2, seed=1)
    write_geotiff(tmp_path / "small.tif", x[0].numpy()[0] % 2, GEO)
    with pytest.raises(ValueError):
        predict_geotiff(learn, raster, tmp_path / "o.tif", mask_path=tmp_path / "small.tif")
    bad = read_geotiff(mask)[0].copy()
    bad[0, 0, :] = N_CLASSES
    write_geotiff(tmp_path / "bad.tif", bad, GEO, nodata=255)
    with pytest.raises(ValueError):
        predict_geotiff(learn, raster, tmp_path / "o.tif", mask_path=tmp_path / "bad.tif")


# ------------------------------------------------------------------------------------------------------ two GPUs
WORKER = """
import sys
sys.path.insert(0, {root!r})
from unet_b200.engine import init_distributed
from unet_b200.reference_api import save_predictions
init_distributed()
save_predictions({model!r}, {tiles!r}, merge={merge}, validation_vision=True)
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
@pytest.mark.parametrize("merge", [False, True])
def test_validation_vision_on_two_gpus_matches_one(tmp_path, merge):
    learn = _learner()
    learn.export(tmp_path / "m.pkl")
    one, _ = _tiles(tmp_path / "one")
    two = tmp_path / "two" / "img_tiles"
    shutil.copytree(tmp_path / "one", tmp_path / "two")
    save_predictions(str(tmp_path / "m.pkl"), one, merge=merge, validation_vision=True)
    script = tmp_path / "worker.py"
    script.write_text(WORKER.format(root=ROOT, model=str(tmp_path / "m.pkl"), tiles=str(two), merge=merge))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29741", str(script)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    sub = "" if merge else "predicted_tiles_m"
    a = json.loads((tmp_path / "one" / sub / "m_validation.json").read_text())
    b = json.loads((tmp_path / "two" / sub / "m_validation.json").read_text())
    assert a == b and a["tiles"] == 10
