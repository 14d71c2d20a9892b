"""Accuracy assessment of predicted class maps: the confusion matrix and classification report of the reference's
`validation_vision` (predict.py:56-143 `plot_valid_predict`: a per-tile majority-class confusion matrix and a scikit-learn
classification report), counted on the device by `b2u_confusion_counts` and reported once from the integer counts.

`ConfusionCounter` owns the device counts of one assessment; `Assessment` is the report computed from a pixel confusion
matrix with scikit-learn's conventions (`zero_division=0` per class, Cohen's kappa NaN when the expected agreement is 1);
`write_report` writes `<name>.json`, `<name>_confusion.csv` and, when tiles were counted, `<name>_tile_confusion.csv`.
Rows of every matrix are truth, columns prediction (`sklearn.metrics.confusion_matrix`); class ids are the model's.

The regression variant has its counterparts: `RegressionCounter` accumulates the error moments of fp32 prediction maps
against fp32 truth on the device (`b2u_regression_assess`), `RegressionAssessment` is the report computed from them
(MAE, RMSE, bias, R² and Pearson r with scikit-learn's / scipy's conventions), and `write_regression_report` writes
`<name>.json` with the raw moments and, when tiles were counted, `<name>_tile_metrics.csv`.
"""
from __future__ import annotations

import csv
import json
import math
from dataclasses import dataclass
from pathlib import Path
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _lib, ops


class ConfusionCounter:
    """Device counts of one assessment, in one int64 buffer so that they come back with one copy and sum with one
    all-reduce: the joint matrix [C*C] (uint64), the skipped-pixel count, then `tile_slots` per-image histograms
    uint32 [2][C] (truth, prediction).  Under `torch.distributed` rank r fills slots [r * tile_slots, (r+1) * tile_slots):
    the ranks' slot ranges are disjoint, so the integer sum of the buffers holds every rank's tiles."""

    def __init__(self, n_classes: int, device, tile_slots: int = 0, rank: int = 0, world: int = 1):
        if not 1 <= n_classes <= 32:
            raise ValueError(f"the assessment counts 1 to 32 classes, not {n_classes}")
        self.C, self.lib = int(n_classes), _lib.load()
        self.tile_slots, self.world = int(tile_slots), int(world)
        self.hist_words = (self.world * self.tile_slots * 2 * self.C + 1) // 2
        self.buf = torch.zeros(self.C * self.C + 1 + self.hist_words, dtype=torch.int64, device=device)
        self.tiles = 0
        self._slot0 = rank * self.tile_slots

    def count(self, pred: torch.Tensor, truth: torch.Tensor, per_tile: bool = False) -> None:
        """pred / truth: uint8 [T, H, W] or [H, W] device views (any pitch and column offset; images of a [T, H, W]
        view one stride apart).  `per_tile`: also record the class histograms of the T images in the next tile slots."""
        if pred.dim() == 2:
            pred, truth = pred[None], truth[None]
        if pred.shape != truth.shape or pred.dtype != torch.uint8 or truth.dtype != torch.uint8:
            raise ValueError(f"pred {tuple(pred.shape)} {pred.dtype} / truth {tuple(truth.shape)} {truth.dtype}: "
                             "two uint8 maps of one shape")
        T, H, W = pred.shape
        if pred.stride(2) != 1 or truth.stride(2) != 1:
            raise ValueError("the class maps need unit column stride")
        hist = None
        if per_tile:
            if self.tiles + T > self.tile_slots:
                raise ValueError(f"{self.tiles + T} tiles counted, {self.tile_slots} slots")
            off = self.C * self.C + 1
            hist = self.buf.data_ptr() + 8 * off + 4 * 2 * self.C * (self._slot0 + self.tiles)
            self.tiles += T
        _lib.check(self.lib.b2u_confusion_counts(pred.data_ptr(), pred.stride(1), pred.stride(0), truth.data_ptr(),
                                                 truth.stride(1), truth.stride(0), T, H, W, self.C,
                                                 self.buf.data_ptr(), hist, self.buf.data_ptr() + 8 * self.C * self.C,
                                                 ops.stream_ptr()), "b2u_confusion_counts")

    def read(self, all_reduce: bool = False):
        """(pixel matrix int64 [C, C], skipped pixels, tile histograms uint32 [n, 2, C] of the counted tiles).  With
        `all_reduce` the buffers of all ranks are summed first (one integer all-reduce)."""
        buf = self.buf
        if all_reduce:
            import torch.distributed as dist
            buf = buf.clone()
            dist.all_reduce(buf)
        h = buf.cpu().numpy()
        C = self.C
        hist = h[C * C + 1:].view(np.uint32)[:self.world * self.tile_slots * 2 * C].reshape(-1, 2, C)
        # unused slots (a rank with fewer tiles than slots) hold no pixel
        hist = hist[hist[:, 0].sum(axis=1) > 0]
        return h[:C * C].reshape(C, C).copy(), int(h[C * C]), hist


def tile_majority_matrix(hist: np.ndarray, n_classes: int) -> np.ndarray:
    """The per-tile matrix of `plot_valid_predict`: majority class of each tile's truth (rows) against the majority class of
    its prediction (columns); a tie takes the lowest class, as np.argmax(np.bincount(...)) does."""
    m = np.zeros((n_classes, n_classes), dtype=np.int64)
    if len(hist):
        np.add.at(m, (hist[:, 0].argmax(axis=1), hist[:, 1].argmax(axis=1)), 1)
    return m


def _div(a, b):
    """a / b elementwise, 0 where b == 0 (scikit-learn's zero_division=0)"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.divide(a, b, out=np.zeros(np.broadcast(a, b).shape), where=b != 0)


@dataclass
class Assessment:
    """The report of a pixel confusion matrix `confusion` [C, C] (rows truth, columns prediction)."""
    confusion: np.ndarray
    accuracy: float
    precision: np.ndarray
    recall: np.ndarray
    f1: np.ndarray
    iou: np.ndarray
    support: np.ndarray
    kappa: float

    @classmethod
    def from_confusion(cls, confusion) -> "Assessment":
        cm = np.asarray(confusion, dtype=np.int64)
        n = int(cm.sum())
        tp = np.diag(cm).astype(np.float64)
        rows, cols = cm.sum(axis=1), cm.sum(axis=0)
        recall, precision = _div(tp, rows), _div(tp, cols)
        f1 = _div(2 * tp, rows + cols)
        iou = _div(tp, rows + cols - tp)
        # sklearn.metrics.cohen_kappa_score: 1 - sum(off-diagonal observed) / sum(off-diagonal expected)
        kappa = float("nan")
        if n:
            expected = np.outer(rows, cols).astype(np.float64) / n
            off = 1.0 - np.eye(len(cm))
            den = float((off * expected).sum())
            if den != 0:
                kappa = 1.0 - float((off * cm).sum()) / den
        return cls(cm, float(tp.sum() / n) if n else float("nan"), precision, recall, f1, iou, rows, kappa)

    def averages(self) -> Dict[str, Dict[str, float]]:
        """macro and support-weighted averages of precision, recall and F1 (classification_report's rows)"""
        w = self.support.astype(np.float64)
        avg = lambda v: float(v.mean())
        wavg = lambda v: float((v * w).sum() / w.sum()) if w.sum() else 0.0
        return {"macro avg": {"precision": avg(self.precision), "recall": avg(self.recall), "f1": avg(self.f1)},
                "weighted avg": {"precision": wavg(self.precision), "recall": wavg(self.recall), "f1": wavg(self.f1)}}

    @property
    def mean_iou(self) -> float:
        return float(self.iou.mean())

    def as_dict(self) -> dict:
        per_class = {str(c): {"precision": float(self.precision[c]), "recall": float(self.recall[c]),
                              "f1": float(self.f1[c]), "iou": float(self.iou[c]), "support": int(self.support[c])}
                     for c in range(len(self.confusion))}
        return {"accuracy": self.accuracy, "per_class": per_class, **self.averages(), "mean_iou": self.mean_iou,
                "kappa": self.kappa}


def _json_safe(v):
    """NaN -> None (JSON null); numpy containers -> lists"""
    if isinstance(v, dict):
        return {k: _json_safe(x) for k, x in v.items()}
    if isinstance(v, (list, tuple)):
        return [_json_safe(x) for x in v]
    if isinstance(v, np.ndarray):
        return _json_safe(v.tolist())
    if isinstance(v, float) and math.isnan(v):
        return None
    return v


def _write_matrix(path: Path, m: np.ndarray) -> None:
    with open(path, "w", newline="") as f:
        wr = csv.writer(f)
        wr.writerow(["truth\\prediction"] + list(range(len(m))))
        for c, row in enumerate(m):
            wr.writerow([c] + [int(v) for v in row])


def read_matrix(path) -> np.ndarray:
    """a matrix written by `write_report` (`<name>_confusion.csv`, `<name>_tile_confusion.csv`)"""
    with open(path, newline="") as f:
        rows = list(csv.reader(f))
    return np.array([[int(v) for v in r[1:]] for r in rows[1:]], dtype=np.int64).reshape(len(rows) - 1, -1)


def write_report(out_dir, name: str, confusion: np.ndarray, skipped: int = 0, tile_hist: Optional[np.ndarray] = None,
                 class_zero: bool = False, extra: Optional[dict] = None) -> List[Path]:
    """`<name>.json` (matrices, metrics, pixel and tile counts, class_zero), `<name>_confusion.csv` and, when tiles were
    counted (`tile_hist` [n, 2, C]), `<name>_tile_confusion.csv`.  Returns the paths written."""
    out_dir = Path(out_dir)
    a = Assessment.from_confusion(confusion)
    C = len(a.confusion)
    doc = {"classes": list(range(C)), "class_zero": bool(class_zero), "pixels": int(a.confusion.sum()),
           "skipped_pixels": int(skipped), "confusion": a.confusion, **a.as_dict()}
    paths = [out_dir / f"{name}.json", out_dir / f"{name}_confusion.csv"]
    _write_matrix(paths[1], a.confusion)
    if tile_hist is not None:
        tm = tile_majority_matrix(tile_hist, C)
        doc.update(tiles=int(tm.sum()), tile_confusion=tm)
        paths.append(out_dir / f"{name}_tile_confusion.csv")
        _write_matrix(paths[2], tm)
    doc.update(extra or {})
    with open(paths[0], "w") as f:
        json.dump(_json_safe(doc), f, indent=1, allow_nan=False)
    return paths


# ----------------------------------------------------------------------------------------------------------- regression
# The moment record of b2u_regression_assess (b2u.h), 15 float64: n, means, centred second moments and co-moment of
# truth t and prediction p, sums of |e|, e and e² for e = p - t, and the extremes of t, p and e.
MOMENT_FIELDS = ("n", "mean_t", "mean_p", "m2_t", "m2_p", "c_tp", "sum_abs_e", "sum_e", "sum_sq_e",
                 "min_t", "max_t", "min_p", "max_p", "min_e", "max_e")
REG_K = len(MOMENT_FIELDS)


def merge_moments(a, b) -> np.ndarray:
    """The record of the union of two samples from theirs: Chan et al.'s pairwise update of (n, means, M2, co-moment),
    the same update the device applies; an empty record (n == 0) leaves the other unchanged."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    if b[0] == 0:
        return a.copy()
    if a[0] == 0:
        return b.copy()
    n = a[0] + b[0]
    f = b[0] / n
    w = a[0] * f
    dt, dp = b[1] - a[1], b[2] - a[2]
    return np.array([n, a[1] + dt * f, a[2] + dp * f, a[3] + b[3] + dt * dt * w, a[4] + b[4] + dp * dp * w,
                     a[5] + b[5] + dt * dp * w, a[6] + b[6], a[7] + b[7], a[8] + b[8],
                     min(a[9], b[9]), max(a[10], b[10]), min(a[11], b[11]), max(a[12], b[12]),
                     min(a[13], b[13]), max(a[14], b[14])])


def merge_all(records) -> np.ndarray:
    """`merge_moments` over a sequence of records, left to right"""
    out = np.zeros(REG_K)
    for r in records:
        out = merge_moments(out, r)
    return out


class RegressionCounter:
    """Device moments of one regression assessment in one float64 buffer: the totals [REG_K], the skipped-pixel count
    (uint64 bits), then `tile_slots` per-image records [REG_K] of this rank.  Under `torch.distributed` the ranks
    all-gather their buffers and the records are merged on the host in rank order (`merge_moments`): deterministic, and
    no floating-point all-reduce.  `pred_nodata` / `truth_nodata`: values skipped in the maps (NaN: none)."""

    def __init__(self, device, tile_slots: int = 0, rank: int = 0, world: int = 1, pred_nodata: float = float("nan"),
                 truth_nodata: float = float("nan")):
        self.lib = _lib.load()
        self.tile_slots, self.world = int(tile_slots), int(world)
        self.pred_nodata, self.truth_nodata = float(pred_nodata), float(truth_nodata)
        self.buf = torch.zeros(REG_K + 1 + self.tile_slots * REG_K, dtype=torch.float64, device=device)
        self.tiles = 0
        # block records of one launch; more than the ~8 blocks per SM the launch would use are never needed
        self.scratch_records = 8 * torch.cuda.get_device_properties(device).multi_processor_count
        self.scratch = torch.empty(self.scratch_records * REG_K, dtype=torch.float64, device=device)
        self.ticket = torch.zeros(1, dtype=torch.int32, device=device)

    def count(self, pred: torch.Tensor, truth: torch.Tensor, per_tile: bool = False) -> None:
        """pred / truth: float32 [T, H, W] or [H, W] device views (any pitch and column offset; images of a [T, H, W]
        view one stride apart).  `per_tile`: also record the moments of the T images in the next tile slots."""
        if pred.dim() == 2:
            pred, truth = pred[None], truth[None]
        if pred.shape != truth.shape or pred.dtype != torch.float32 or truth.dtype != torch.float32:
            raise ValueError(f"pred {tuple(pred.shape)} {pred.dtype} / truth {tuple(truth.shape)} {truth.dtype}: "
                             "two float32 maps of one shape")
        T, H, W = pred.shape
        if pred.stride(2) != 1 or truth.stride(2) != 1:
            raise ValueError("the maps need unit column stride")
        tile = None
        if per_tile:
            if self.tiles + T > self.tile_slots:
                raise ValueError(f"{self.tiles + T} tiles counted, {self.tile_slots} slots")
            tile = self.buf.data_ptr() + 8 * (REG_K + 1 + REG_K * self.tiles)
            self.tiles += T
        if T > self.scratch_records:
            self.scratch_records = T
            self.scratch = torch.empty(T * REG_K, dtype=torch.float64, device=self.buf.device)
        _lib.check(self.lib.b2u_regression_assess(pred.data_ptr(), pred.stride(1), pred.stride(0), truth.data_ptr(),
                                                  truth.stride(1), truth.stride(0), T, H, W, self.pred_nodata,
                                                  self.truth_nodata, self.buf.data_ptr(), tile,
                                                  self.buf.data_ptr() + 8 * REG_K, self.scratch.data_ptr(),
                                                  self.scratch_records, self.ticket.data_ptr(), ops.stream_ptr()),
                   "b2u_regression_assess")

    def read(self, all_reduce: bool = False):
        """(totals float64 [REG_K], skipped pixels, tile records float64 [world, tile_slots, REG_K]).  With `all_reduce`
        the buffers of all ranks are all-gathered and merged in rank order; rank r's tiles are row r."""
        bufs = [self.buf]
        if all_reduce:
            import torch.distributed as dist
            bufs = [torch.empty_like(self.buf) for _ in range(self.world)]
            dist.all_gather(bufs, self.buf)
        hs = [b.cpu().numpy() for b in bufs]
        totals = merge_all(h[:REG_K] for h in hs)
        skipped = sum(int(h[REG_K:REG_K + 1].view(np.int64)[0]) for h in hs)
        tiles = np.stack([h[REG_K + 1:].reshape(self.tile_slots, REG_K) for h in hs])
        return totals, skipped, tiles


@dataclass
class RegressionAssessment:
    """The report of a moment record: scikit-learn's `mean_absolute_error`, `mean_squared_error` and `r2_score` (1 -
    SSE/SST; with constant truth 1.0 when SSE = 0, else 0.0; NaN for one pixel), scipy's Pearson r (NaN when either
    variance is 0), the
    bias mean(p - t), the largest |p - t|, and the mean, population std, min and max of truth and prediction.  With
    n = 0 every metric is NaN."""
    n: int
    skipped: int
    mae: float
    mse: float
    rmse: float
    bias: float
    max_abs_error: float
    r2: float
    pearson_r: float
    truth_mean: float
    truth_std: float
    truth_min: float
    truth_max: float
    pred_mean: float
    pred_std: float
    pred_min: float
    pred_max: float

    @classmethod
    def from_moments(cls, m, skipped: int = 0) -> "RegressionAssessment":
        m = np.asarray(m, np.float64)
        n = int(m[0])
        if n == 0:
            nan = float("nan")
            return cls(0, int(skipped), *([nan] * 15))
        mse = float(m[8] / n)
        sst, sse = float(m[3]), float(m[8])
        # r2_score: undefined (NaN) below two samples
        r2 = float("nan") if n < 2 else (1.0 if sse == 0 else 0.0) if sst == 0 else 1.0 - sse / sst
        r = float("nan")
        if m[3] > 0 and m[4] > 0:
            r = float(np.clip(m[5] / math.sqrt(m[3] * m[4]), -1.0, 1.0))
        return cls(n, int(skipped), float(m[6] / n), mse, math.sqrt(mse), float(m[7] / n),
                   float(max(abs(m[13]), abs(m[14]))), r2, r, float(m[1]), math.sqrt(m[3] / n), float(m[9]),
                   float(m[10]), float(m[2]), math.sqrt(m[4] / n), float(m[11]), float(m[12]))

    def as_dict(self) -> dict:
        return dict(self.__dict__)


TILE_METRICS_HEADER = ["tile", "n", "mae", "rmse", "bias", "truth_mean", "pred_mean"]


def write_regression_report(out_dir, name: str, moments, skipped: int = 0, tile_moments=None,
                            tile_names: Optional[Sequence[str]] = None, extra: Optional[dict] = None) -> List[Path]:
    """`<name>.json` (the metrics of `RegressionAssessment`, the raw moment record so that reports of separate ranks or
    runs can be merged with `merge_moments`, and the tile count) and, when tiles were counted (`tile_moments` [n, REG_K]
    with their `tile_names`), `<name>_tile_metrics.csv`: one row per tile with its name, n, MAE, RMSE, bias, truth mean
    and prediction mean.  Returns the paths written."""
    out_dir = Path(out_dir)
    a = RegressionAssessment.from_moments(moments, skipped)
    doc = {**a.as_dict(), "moments": dict(zip(MOMENT_FIELDS, map(float, np.asarray(moments, np.float64))))}
    paths = [out_dir / f"{name}.json"]
    if tile_moments is not None:
        doc["tiles"] = len(tile_moments)
        paths.append(out_dir / f"{name}_tile_metrics.csv")
        with open(paths[1], "w", newline="") as f:
            wr = csv.writer(f)
            wr.writerow(TILE_METRICS_HEADER)
            for tn, tm in zip(tile_names, tile_moments):
                t = RegressionAssessment.from_moments(tm)
                wr.writerow([tn, t.n] + [repr(v) for v in (t.mae, t.rmse, t.bias, t.truth_mean, t.pred_mean)])
    doc.update(extra or {})
    with open(paths[0], "w") as f:
        json.dump(_json_safe(doc), f, indent=1, allow_nan=False)
    return paths
