"""Plain-torch references of the optional training losses (test infrastructure, next to oracle/unet_oracle.py's
`weighted_ce`): fastai 2.5.1's FocalLossFlat and DiceLoss, restated from memory of the upstream source [fastai-mem].

Pinned where an independent implementation exists (tests/test_losses_cpu.py): `focal_loss_flat` at gamma 0 equals
torch's weighted cross-entropy summed over pixels / P, `dice_loss` on one-hot probabilities equals 1 - scikit-learn's
per-class F1, and both gradients equal the closed forms the kernels implement (autograd + gradcheck in float64)."""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn.functional as F


def focal_loss_flat(logits: torch.Tensor, target: torch.Tensor, weight: Optional[torch.Tensor] = None,
                    gamma: float = 2.0, reduction: str = "mean") -> torch.Tensor:
    """FocalLossFlat(axis=1, gamma, weight): the CrossEntropyLossFlat pixel losses with reduction 'none'
    (l = w[y] * nll, so pt = exp(-l) = p_y^w[y] with weights), f = (1 - pt)^gamma * l, plain mean over all pixels or sum."""
    c = logits.shape[1]
    ce = F.cross_entropy(logits.permute(0, 2, 3, 1).reshape(-1, c), target.reshape(-1).long(), weight=weight,
                         reduction="none")
    f = (-torch.expm1(-ce)) ** gamma * ce
    return f.mean() if reduction == "mean" else f.sum()


def dice_loss(logits: torch.Tensor, target: torch.Tensor, smooth: float = 1e-6, reduction: str = "sum",
              square_in_union: bool = False) -> torch.Tensor:
    """DiceLoss(axis=1, smooth, reduction, square_in_union): p = softmax over the classes, t = one-hot target; per
    sample and class I = sum p t, U = sum (p + t) (or p^2 + t); loss = 1 - (2I + smooth) / (U + smooth), summed
    (fastai's default) or averaged over all (sample, class)."""
    c = logits.shape[1]
    p = logits.softmax(1)
    t = F.one_hot(target.long(), c).permute(0, 3, 1, 2).to(p.dtype)
    inter = (p * t).sum((2, 3))
    union = ((p * p if square_in_union else p) + t).sum((2, 3))
    loss = 1 - (2.0 * inter + smooth) / (union + smooth)
    return loss.mean() if reduction == "mean" else loss.sum()
