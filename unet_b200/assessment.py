"""Accuracy assessment of predicted class maps: the confusion matrix and classification report of the reference's
`validation_vision` (predict.py:56-143 `plot_valid_predict`: a per-tile majority-class confusion matrix and a scikit-learn
classification report), counted on the device by `b2u_confusion_counts` and reported once from the integer counts.

`ConfusionCounter` owns the device counts of one assessment; `Assessment` is the report computed from a pixel confusion
matrix with scikit-learn's conventions (`zero_division=0` per class, Cohen's kappa NaN when the expected agreement is 1);
`write_report` writes `<name>.json`, `<name>_confusion.csv` and, when tiles were counted, `<name>_tile_confusion.csv`.
Rows of every matrix are truth, columns prediction (`sklearn.metrics.confusion_matrix`); class ids are the model's.
"""
from __future__ import annotations

import csv
import json
import math
from dataclasses import dataclass
from pathlib import Path
from typing import Dict, List, Optional

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
