"""The accuracy report of `validation_vision` / `predict_geotiff(mask_path=)` without a GPU: the metrics of
`unet_b200.assessment` against scikit-learn, the report files, the per-tile majority rule, the label conversion shared
with `prepare_raster`, the merge-mode tile ownership and the mask-tile lookup."""
import json
import math
import warnings

import numpy as np
import pytest
from sklearn.metrics import (accuracy_score, cohen_kappa_score, confusion_matrix, jaccard_score,
                             precision_recall_fscore_support)

from unet_b200.assessment import Assessment, read_matrix, tile_majority_matrix, write_report
from unet_b200.create_tiles import mask_labels, mask_tile_values, prepare_raster
from unet_b200.geotiff import GeoInfo, write_geotiff


def _pixels(cm):
    """(truth, pred) pixel lists of a confusion matrix"""
    t, p = np.nonzero(cm)
    n = cm[t, p]
    return np.repeat(t, n), np.repeat(p, n)


def _cases():
    rng = np.random.default_rng(0)
    out = []
    for C in (1, 2, 3, 5, 8):
        for _ in range(4):
            cm = rng.integers(0, 50, size=(C, C))
            cm[rng.random((C, C)) < 0.3] = 0
            cm[0, 0] += cm.sum() == 0                # scikit-learn needs one sample
            out.append(cm)
    absent = rng.integers(1, 30, size=(4, 4))
    absent[2, :] = 0                     # class 2 never in the truth
    absent[:, 1] = 0                     # class 1 never predicted
    out.append(absent)
    out.append(np.diag([0, 7, 0]))       # perfect on one class, others absent: expected agreement 1 -> kappa NaN
    out.append(np.array([[0, 9], [0, 0]]))
    return out


@pytest.mark.parametrize("cm", _cases(), ids=lambda c: f"C{len(c)}")
def test_metrics_equal_scikit_learn(cm):
    C = len(cm)
    yt, yp = _pixels(cm)
    labels = list(range(C))
    assert np.array_equal(confusion_matrix(yt, yp, labels=labels), cm)
    a = Assessment.from_confusion(cm)
    assert a.accuracy == pytest.approx(accuracy_score(yt, yp))
    p, r, f, s = precision_recall_fscore_support(yt, yp, labels=labels, zero_division=0)
    np.testing.assert_allclose(a.precision, p, rtol=1e-12)
    np.testing.assert_allclose(a.recall, r, rtol=1e-12)
    np.testing.assert_allclose(a.f1, f, rtol=1e-12, atol=1e-15)
    assert np.array_equal(a.support, s)
    np.testing.assert_allclose(a.iou, jaccard_score(yt, yp, labels=labels, average=None, zero_division=0), rtol=1e-12)
    avg = a.averages()
    for name, sk in (("macro avg", "macro"), ("weighted avg", "weighted")):
        p, r, f, _ = precision_recall_fscore_support(yt, yp, labels=labels, average=sk, zero_division=0)
        assert avg[name]["precision"] == pytest.approx(p) and avg[name]["recall"] == pytest.approx(r)
        assert avg[name]["f1"] == pytest.approx(f)
    assert a.mean_iou == pytest.approx(jaccard_score(yt, yp, labels=labels, average="macro", zero_division=0))
    with warnings.catch_warnings(), np.errstate(all="ignore"):
        warnings.simplefilter("ignore")
        k = cohen_kappa_score(yt, yp, labels=labels)
    assert (math.isnan(k) and math.isnan(a.kappa)) or a.kappa == pytest.approx(k)


def test_kappa_is_nan_when_expected_agreement_is_one():
    assert math.isnan(Assessment.from_confusion(np.diag([0, 7, 0])).kappa)
    assert math.isnan(Assessment.from_confusion(np.zeros((3, 3), np.int64)).accuracy)


def test_report_files_round_trip(tmp_path):
    cm = np.array([[5, 1, 0], [2, 7, 0], [0, 0, 0]])
    hist = np.array([[[9, 1, 0], [3, 7, 0]], [[0, 4, 4], [0, 8, 0]], [[6, 0, 0], [6, 0, 0]]], dtype=np.uint32)
    paths = write_report(tmp_path, "r", cm, skipped=3, tile_hist=hist, class_zero=True, extra={"k": 1})
    assert [p.name for p in paths] == ["r.json", "r_confusion.csv", "r_tile_confusion.csv"]
    doc = json.loads(paths[0].read_text())
    assert doc["confusion"] == cm.tolist() and doc["pixels"] == 15 and doc["skipped_pixels"] == 3
    assert doc["class_zero"] is True and doc["tiles"] == 3 and doc["k"] == 1
    assert doc["per_class"]["2"] == {"precision": 0.0, "recall": 0.0, "f1": 0.0, "iou": 0.0, "support": 0}
    assert np.array_equal(read_matrix(paths[1]), cm)
    tm = read_matrix(paths[2])
    assert np.array_equal(tm, np.array(doc["tile_confusion"]))
    assert tm[0, 1] == 1 and tm[1, 1] == 1 and tm[0, 0] == 1
    # NaN kappa is written as null; no tile file without tiles
    paths = write_report(tmp_path, "one", np.diag([4, 0]))
    assert len(paths) == 2 and json.loads(paths[0].read_text())["kappa"] is None
    assert not (tmp_path / "one_tile_confusion.csv").exists()


def test_tile_majority_takes_the_lowest_class_on_ties():
    hist = np.array([[[3, 3, 1], [0, 2, 2]],          # truth tie 0/1 -> 0, prediction tie 1/2 -> 1
                     [[0, 5, 5], [4, 4, 4]]], dtype=np.uint32)   # truth tie 1/2 -> 1, prediction three-way -> 0
    m = tile_majority_matrix(hist, 3)
    for h in hist:
        t = np.argmax(np.bincount(np.repeat(np.arange(3), h[0]), minlength=3))
        p = np.argmax(np.bincount(np.repeat(np.arange(3), h[1]), minlength=3))
        assert m[t, p] >= 1
    assert m[0, 1] == 1 and m[1, 0] == 1 and m.sum() == 2


GEO = GeoInfo(geotransform=(383000.0, 0.2, 0.0, 5819000.0, 0.0, -0.2), georeferenced=True)


@pytest.mark.parametrize("class_zero", [False, True])
def test_mask_labels_reproduce_prepare_raster_on_windows(tmp_path, class_zero):
    rng = np.random.default_rng(3)
    img = rng.integers(1, 255, size=(3, 70, 90)).astype(np.uint8)
    img[:, 5:9, 10:20] = 0                      # image no-data (0) in every band
    msk = rng.integers(0, 3, size=(1, 70, 90)).astype(np.uint8)
    msk[0, 40:50, 60:70] = 255                  # mask no-data
    write_geotiff(tmp_path / "r.tif", img, GEO, nodata=0)
    write_geotiff(tmp_path / "m.tif", msk, GEO, nodata=255)
    full = prepare_raster(tmp_path / "r.tif", tmp_path / "m.tif", 32, 0.25, 0.9, class_zero).mask
    ref = mask_tile_values(full[0])
    for x0, w in ((0, 90), (0, 33), (17, 40), (57, 33)):
        lab, bad = mask_labels(img[:, :, x0:x0 + w], 0, msk[:, :, x0:x0 + w], 255, class_zero)
        assert np.array_equal(mask_tile_values(lab[0]), ref[:, x0:x0 + w]), (x0, w)
    assert ref[45, 65] == 0 and ref[6, 12] == 0


@pytest.mark.parametrize("world", range(1, 9))
def test_merge_tiles_have_exactly_one_owner(world):
    from unet_b200.reference_api import _merge_strip
    rng = np.random.default_rng(world)
    P = 16
    for _ in range(5):
        n = int(rng.integers(1, 60))
        place = [(int(rng.integers(0, 200)), int(rng.integers(0, 50)), P, P) for _ in range(n)]
        x_len = max(x for x, *_ in place) + P
        owners = [[] for _ in range(n)]
        for r in range(world):
            xb, xe, mine, own = _merge_strip(place, P, x_len, r, world)
            for i, o in zip(mine, own):
                if o:
                    owners[i].append(r)
        assert all(len(o) == 1 for o in owners)


def test_missing_mask_tile_raises(tmp_path):
    from unet_b200.reference_api import _mask_path
    (tmp_path / "img_tiles").mkdir()
    (tmp_path / "mask_tiles").mkdir()
    t = tmp_path / "img_tiles" / "a.tif"
    t.touch()
    with pytest.raises(FileNotFoundError):
        _mask_path(t)
    (tmp_path / "mask_tiles" / "a.tif").touch()
    assert _mask_path(t) == tmp_path / "mask_tiles" / "a.tif"
    with pytest.raises(FileNotFoundError):       # a tile outside an img_tiles folder has no mask tile
        _mask_path(tmp_path / "a.tif")
