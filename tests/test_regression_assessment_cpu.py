"""Regression assessment on the host: the report from moment records against scikit-learn / scipy, the pairwise merge
of moments against whole-sample statistics, and the report files."""
import csv
import itertools
import json
import math
import warnings

import numpy as np
import pytest
from scipy.stats import pearsonr
from sklearn.metrics import mean_absolute_error, mean_squared_error, r2_score

from unet_b200.assessment import (MOMENT_FIELDS, REG_K, TILE_METRICS_HEADER, RegressionAssessment, merge_all,
                                  merge_moments, write_regression_report)


def moments(p, t) -> np.ndarray:
    """the record of b2u_regression_assess computed two-pass in float64"""
    p, t = np.asarray(p, np.float64).ravel(), np.asarray(t, np.float64).ravel()
    if p.size == 0:
        return np.zeros(REG_K)
    mt, mp = t.mean(), p.mean()
    dt, dp, e = t - mt, p - mp, p - t
    return np.array([p.size, mt, mp, dt @ dt, dp @ dp, dt @ dp, np.abs(e).sum(), e.sum(), e @ e, t.min(), t.max(),
                     p.min(), p.max(), e.min(), e.max()])


def _check_against_sklearn(a: RegressionAssessment, p, t, rel=1e-12):
    assert a.n == p.size
    assert a.mae == pytest.approx(mean_absolute_error(t, p), rel=rel)
    assert a.mse == pytest.approx(mean_squared_error(t, p), rel=rel)
    assert a.rmse == pytest.approx(math.sqrt(mean_squared_error(t, p)), rel=rel)
    assert a.r2 == pytest.approx(r2_score(t, p), rel=rel, abs=rel)
    assert a.bias == pytest.approx(np.mean(p - t), rel=1e-9, abs=1e-12)
    assert a.max_abs_error == np.abs(p - t).max()
    assert (a.truth_mean, a.truth_std, a.truth_min, a.truth_max) == pytest.approx((t.mean(), t.std(), t.min(), t.max()),
                                                                                  rel=rel)
    assert (a.pred_mean, a.pred_std, a.pred_min, a.pred_max) == pytest.approx((p.mean(), p.std(), p.min(), p.max()),
                                                                              rel=rel)


@pytest.mark.parametrize("seed", range(4))
def test_report_matches_sklearn_and_scipy(seed):
    rng = np.random.default_rng(seed)
    t = rng.normal(5.0, 2.0, 5000)
    p = 0.8 * t + rng.normal(0.3, 1.0, t.size)
    a = RegressionAssessment.from_moments(moments(p, t), skipped=7)
    _check_against_sklearn(a, p, t)
    assert a.skipped == 7
    assert a.pearson_r == pytest.approx(pearsonr(t, p).statistic, rel=1e-12)


def test_constant_truth_single_pixel_and_empty():
    t = np.full(100, 3.5)
    perfect = RegressionAssessment.from_moments(moments(t, t))
    assert perfect.r2 == r2_score(t, t) == 1.0 and perfect.mse == 0.0
    p = t + np.linspace(-1, 1, t.size)
    off = RegressionAssessment.from_moments(moments(p, t))
    assert off.r2 == r2_score(t, p) == 0.0
    assert math.isnan(off.pearson_r) and math.isnan(perfect.pearson_r)            # a variance is 0
    _check_against_sklearn(off, p, t)
    one = RegressionAssessment.from_moments(moments([2.0], [1.5]))
    assert (one.n, one.mae, one.mse, one.bias, one.max_abs_error) == (1, 0.5, 0.25, 0.5, 0.5)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")                   # scikit-learn warns that R² is undefined for one sample
        assert math.isnan(r2_score([1.5], [2.0])) and math.isnan(one.r2)
    assert math.isnan(one.pearson_r)
    empty = RegressionAssessment.from_moments(np.zeros(REG_K), skipped=3)
    assert empty.n == 0 and empty.skipped == 3
    assert all(math.isnan(v) for k, v in empty.as_dict().items() if k not in ("n", "skipped"))


def _assert_records_close(got, ref, rel=1e-12):
    assert got[0] == ref[0]
    scale = np.abs(ref).copy()
    scale[7] = max(scale[7], ref[6])                      # sum e may cancel: measure it against sum |e|
    scale[5] = max(scale[5], math.sqrt(ref[3] * ref[4]))  # the co-moment against the variances
    assert np.all(np.abs(got - ref) <= rel * scale), (got - ref) / np.maximum(scale, 1e-300)
    assert np.array_equal(got[9:], ref[9:])               # extremes are exact


@pytest.mark.parametrize("offset", [0.0, 1000.0])
def test_merged_splits_equal_whole_sample(offset):
    rng = np.random.default_rng(3)
    t = offset + rng.normal(0.0, 0.01 if offset else 1.0, 20000)
    p = t + rng.normal(0.0, 0.002 if offset else 0.5, t.size)
    whole = moments(p, t)
    for trial in range(6):
        cuts = np.sort(rng.choice(np.arange(1, t.size), size=rng.integers(1, 40), replace=False))
        parts = [moments(pp, tt) for pp, tt in zip(np.split(p, cuts), np.split(t, cuts))]
        orders = [parts, parts[::-1], [parts[i] for i in rng.permutation(len(parts))]]
        for order in orders:
            _assert_records_close(merge_all(order), whole)
        # a balanced tree gives the same statistics
        level = parts + [np.zeros(REG_K)]                 # an empty record changes nothing
        while len(level) > 1:
            level = [merge_moments(level[i], level[i + 1]) if i + 1 < len(level) else level[i]
                     for i in range(0, len(level), 2)]
        _assert_records_close(level[0], whole)
    if offset:
        # raw sums of t and t² lose the variance of offset data to cancellation
        naive = (t @ t) - t.sum() ** 2 / t.size
        assert abs(naive - whole[3]) > 1e-9 * whole[3]
    a = RegressionAssessment.from_moments(merge_all(parts))
    _check_against_sklearn(a, p, t, rel=1e-9)


def test_report_files(tmp_path):
    rng = np.random.default_rng(5)
    tiles = [(rng.normal(10, 2, 64), rng.normal(10, 2, 64)) for _ in range(3)]
    recs = [moments(p, t) for p, t in tiles] + [np.zeros(REG_K)]
    names = ["a.tif", "b.tif", "c.tif", "empty.tif"]
    total = merge_all(recs)
    paths = write_regression_report(tmp_path, "v", total, 11, recs, names, extra={"raster": "r.tif"})
    assert [p.name for p in paths] == ["v.json", "v_tile_metrics.csv"]
    doc = json.loads(paths[0].read_text())
    assert set(doc) == {"n", "skipped", "mae", "mse", "rmse", "bias", "max_abs_error", "r2", "pearson_r", "truth_mean",
                        "truth_std", "truth_min", "truth_max", "pred_mean", "pred_std", "pred_min", "pred_max",
                        "moments", "tiles", "raster"}
    assert doc["n"] == 192 and doc["skipped"] == 11 and doc["tiles"] == 4 and doc["raster"] == "r.tif"
    assert list(doc["moments"]) == list(MOMENT_FIELDS)
    assert np.array_equal(np.array([doc["moments"][k] for k in MOMENT_FIELDS]), total)     # round trip, exact
    p_all, t_all = np.concatenate([p for p, _ in tiles]), np.concatenate([t for _, t in tiles])
    assert doc["rmse"] == pytest.approx(math.sqrt(mean_squared_error(t_all, p_all)), rel=1e-12)
    with open(paths[1], newline="") as f:
        rows = list(csv.reader(f))
    assert rows[0] == TILE_METRICS_HEADER == ["tile", "n", "mae", "rmse", "bias", "truth_mean", "pred_mean"]
    assert [r[0] for r in rows[1:]] == names
    for r, (p, t) in zip(rows[1:], tiles):
        assert int(r[1]) == p.size
        got = [float(v) for v in r[2:]]
        ref = [np.abs(p - t).mean(), math.sqrt(((p - t) ** 2).mean()), (p - t).mean(), t.mean(), p.mean()]
        assert got == pytest.approx(ref, rel=1e-12, abs=1e-12)
    assert rows[4][1] == "0" and all(math.isnan(float(v)) for v in rows[4][2:])
    # no tiles: no CSV, and an empty assessment still writes
    paths = write_regression_report(tmp_path, "e", np.zeros(REG_K))
    assert [p.name for p in paths] == ["e.json"]
    doc = json.loads(paths[0].read_text())
    assert doc["n"] == 0 and doc["rmse"] is None and "tiles" not in doc


def test_merge_is_symmetric_in_content():
    rng = np.random.default_rng(9)
    a = moments(rng.normal(size=50), rng.normal(size=50))
    b = moments(rng.normal(size=70), rng.normal(size=70))
    ab, ba = merge_moments(a, b), merge_moments(b, a)
    _assert_records_close(ab, ba)
    assert np.array_equal(merge_moments(a, np.zeros(REG_K)), a) and np.array_equal(merge_moments(np.zeros(REG_K), a), a)
    for x, y in itertools.permutations([a, b]):
        assert merge_moments(x, y)[0] == 120
