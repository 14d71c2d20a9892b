"""The training loss a user picks with `loss_func` (params_and_main.py extra parameter -> train_func -> unet_learner_MS):
fastai's CrossEntropyLossFlat(axis=1) (the default), FocalLossFlat(axis=1, gamma=...) or DiceLoss(axis=1, ...).

`LossSpec` is the choice as plain values: it travels into the plan (`UNetB200(loss_spec=...)`), into an exported
checkpoint and into `<description>.json`.  `parse_loss_func` reads it from what a user can hand over: a string in fastai
call syntax (what a params.json carries; parsed with `ast`, literal keyword values only, nothing is evaluated) or an
object whose class is one of the three.  `launch_loss` issues the kernels of the focal and Dice losses for both the
training step and validation.  Every loss keeps softmax as its activation and argmax as its decodes.
"""
from __future__ import annotations

import ast
import warnings
from dataclasses import asdict, dataclass
from typing import Any, Dict, Optional

NAMES = {"CrossEntropyLossFlat": "ce", "FocalLossFlat": "focal", "DiceLoss": "dice"}
# the keywords each call accepts (fastai 2.5.1 defaults in LossSpec); `axis` must be 1 (the class axis of [N,C,H,W])
_KEYWORDS = {"ce": ("axis",), "focal": ("axis", "gamma", "reduction"),
             "dice": ("axis", "smooth", "reduction", "square_in_union")}
_DEFAULT_REDUCTION = {"ce": "mean", "focal": "mean", "dice": "sum"}


@dataclass(frozen=True)
class LossSpec:
    """name 'ce' | 'focal' | 'dice'; gamma (focal), smooth / square_in_union (dice); reduction 'mean' | 'sum'."""
    name: str = "ce"
    gamma: float = 2.0
    smooth: float = 1e-6
    reduction: str = "mean"
    square_in_union: bool = False

    def __post_init__(self):
        if self.name not in _KEYWORDS:
            raise ValueError(f"loss {self.name!r} not understood; choose from {sorted(_KEYWORDS)}")
        if self.reduction not in ("mean", "sum"):
            raise ValueError(f"reduction must be 'mean' or 'sum', got {self.reduction!r}")
        if self.name == "ce" and self.reduction != "mean":
            raise ValueError("CrossEntropyLossFlat is built with reduction 'mean' only")
        if not (float(self.gamma) >= 0.0):
            raise ValueError(f"gamma must be >= 0, got {self.gamma!r}")
        if not (float(self.smooth) > 0.0):
            raise ValueError(f"smooth must be > 0, got {self.smooth!r}")

    def as_dict(self) -> Dict[str, Any]:
        return asdict(self)

    @classmethod
    def from_dict(cls, d: Optional[Dict[str, Any]]) -> "LossSpec":
        """what `as_dict` wrote; None (a checkpoint written before the loss was recorded) is cross-entropy"""
        return cls() if d is None else cls(**d)


def _make(name: str, kw: Dict[str, Any]) -> LossSpec:
    unknown = sorted(set(kw) - set(_KEYWORDS[name]))
    if unknown:
        raise ValueError(f"{name} loss: unsupported keyword(s) {unknown}; accepted: {list(_KEYWORDS[name])}")
    axis = kw.pop("axis", 1)
    if axis != 1:
        raise ValueError(f"loss axis must be 1 (the class axis of the [N,C,H,W] logits), got {axis!r}")
    for k, typ in (("gamma", (int, float)), ("smooth", (int, float)), ("square_in_union", (bool,)),
                   ("reduction", (str,))):
        if k in kw and (not isinstance(kw[k], typ) or (typ != (bool,) and isinstance(kw[k], bool))):
            raise ValueError(f"{name} loss: {k}={kw[k]!r} has the wrong type")
    kw.setdefault("reduction", _DEFAULT_REDUCTION[name])
    for k in ("gamma", "smooth"):
        if k in kw:
            kw[k] = float(kw[k])
    return LossSpec(name=name, **kw)


def _parse_string(s: str) -> LossSpec:
    try:
        node = ast.parse(s.strip(), mode="eval").body
    except SyntaxError as e:
        raise ValueError(f"loss_func {s!r} is not a call such as 'FocalLossFlat(axis=1, gamma=2)'") from e
    if isinstance(node, ast.Name):                      # a bare class name: its defaults
        node = ast.Call(func=node, args=[], keywords=[])
    if not isinstance(node, ast.Call) or not isinstance(node.func, ast.Name):
        raise ValueError(f"loss_func {s!r} is not a call such as 'FocalLossFlat(axis=1, gamma=2)'")
    if node.func.id not in NAMES:
        raise ValueError(f"loss_func {node.func.id!r} is not supported; choose from {sorted(NAMES)}")
    if node.args:
        raise ValueError(f"loss_func {s!r}: pass keyword arguments only (e.g. gamma=2)")
    kw: Dict[str, Any] = {}
    for k in node.keywords:
        if k.arg is None:
            raise ValueError(f"loss_func {s!r}: **kwargs are not accepted")
        try:
            kw[k.arg] = ast.literal_eval(k.value)
        except (ValueError, TypeError, SyntaxError) as e:
            raise ValueError(f"loss_func {s!r}: {k.arg} must be a literal value") from e
    return _make(NAMES[node.func.id], kw)


def parse_loss_func(loss_func) -> Optional[LossSpec]:
    """None -> cross-entropy; a LossSpec as is; a string in fastai call syntax; an object of class CrossEntropyLossFlat,
    FocalLossFlat or DiceLoss (its settings read off its attributes).  Returns None for any other object (the caller
    warns and trains with cross-entropy).  Raises ValueError for a bad string, axis or keyword."""
    if loss_func is None:
        return LossSpec()
    if isinstance(loss_func, LossSpec):
        return loss_func
    if isinstance(loss_func, str):
        return _parse_string(loss_func)
    name = NAMES.get(type(loss_func).__name__)
    if name is None:
        return None
    kw: Dict[str, Any] = {"axis": getattr(loss_func, "axis", 1)}
    if name == "focal":
        kw["gamma"] = getattr(loss_func, "gamma", 2.0)
        kw["reduction"] = getattr(loss_func, "reduce", getattr(loss_func, "reduction", "mean"))   # fastai keeps it in .reduce
    elif name == "dice":
        for k, d in (("smooth", 1e-6), ("reduction", "sum"), ("square_in_union", False)):
            kw[k] = getattr(loss_func, k, d)
    return _make(name, kw)


def dice_blocks_per_sample(N: int, HW: int) -> int:
    """blocks per sample of the Dice kernels: about 592 blocks (4 per SM) in all, at least 2048 pixels per block"""
    return max(1, min(-(-592 // N), -(-HW // 2048)))


def launch_loss(lib, spec: LossSpec, logits, labels, N: int, HW: int, C: int, weight: Optional[int], dlogits: Optional[int],
                ldg: int, loss_part, rows: int, dice_part, dice_bps: int, loss, grad_scale: float, stream: int) -> None:
    """focal or Dice loss (+ dlogits unless None) of the first N samples into the device scalar `loss`.
    loss_part: >= rows floats (focal) / >= N floats (dice); dice_part: >= N * dice_bps * 3 * C floats."""
    from ._lib import check
    ld = logits.shape[-1]
    mean = int(spec.reduction == "mean")
    if spec.name == "focal":
        P = N * HW
        check(lib.b2u_focal_fwd_bwd(logits.data_ptr(), ld, labels.data_ptr(), P, C, weight, spec.gamma, mean, dlogits,
                                    ldg, loss_part.data_ptr(), rows, grad_scale, stream), "b2u_focal_fwd_bwd")
        check(lib.b2u_mse_finalize(loss_part.data_ptr(), rows, P if mean else 1, loss.data_ptr(), stream),
              "b2u_mse_finalize")
    elif spec.name == "dice":
        sq = int(spec.square_in_union)
        check(lib.b2u_dice_stats(logits.data_ptr(), ld, labels.data_ptr(), N, HW, C, sq, dice_part.data_ptr(), dice_bps,
                                 stream), "b2u_dice_stats")
        check(lib.b2u_dice_bwd(logits.data_ptr(), ld, labels.data_ptr(), N, HW, C, sq, dice_part.data_ptr(), dice_bps,
                               spec.smooth, mean, dlogits, ldg, loss_part.data_ptr(), grad_scale, stream), "b2u_dice_bwd")
        check(lib.b2u_mse_finalize(loss_part.data_ptr(), N, N * C if mean else 1, loss.data_ptr(), stream),
              "b2u_mse_finalize")
    else:
        raise ValueError(f"launch_loss handles the focal and Dice losses, not {spec.name!r}")


def warn_dice_weights(spec: LossSpec, class_weights) -> None:
    """DiceLoss has no class weights (fastai: not a BaseLoss, no .func.weight)"""
    if spec.name == "dice" and class_weights is not None and len(set(float(w) for w in class_weights)) > 1:
        warnings.warn("DiceLoss has no class weights: CLASS_WEIGHTS other than 'even' are ignored")
