"""The `loss_func` choice on the CPU: the oracle's FocalLossFlat / DiceLoss pinned where independent code exists
(torch's cross-entropy, scikit-learn's F1, autograd's gradcheck of the hand-derived gradients the kernels implement),
the parser of the fastai call strings and objects, and the params_and_main pass-through."""
import warnings

import numpy as np
import pytest
import torch
import torch.nn.functional as F


def _case(N=2, C=3, H=5, W=4, seed=0, dtype=torch.float64):
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(N, C, H, W, generator=g, dtype=dtype) * 2
    y = torch.randint(0, C, (N, H, W), generator=g)
    return z, y


def focal_grad(z, y, w, gamma, reduction):
    """the kernel's formula: dz = s * f'(l) * w[y] * (p - onehot), f'(l) = (1-pt)^g * (1 + g pt l / (1-pt))"""
    C = z.shape[1]
    p = z.softmax(1)
    t = F.one_hot(y, C).permute(0, 3, 1, 2).to(z.dtype)
    wy = w[y][:, None]
    l = wy * -(z.log_softmax(1) * t).sum(1, keepdim=True)
    omp = -torch.expm1(-l)
    second = torch.where(omp > 0, gamma * torch.exp(-l) * l / omp.clamp_min(1e-300), torch.zeros_like(l))
    s = 1.0 / y.numel() if reduction == "mean" else 1.0
    return s * omp ** gamma * (1 + second) * wy * (p - t)


def dice_grad(z, y, smooth, reduction, square):
    """the kernel's formula: g = -r [2 t (U+s) - (2I+s) u'] / (U+s)^2, dz_j = p_j (g_j - sum_c p_c g_c)"""
    N, C = z.shape[:2]
    p = z.softmax(1)
    t = F.one_hot(y, C).permute(0, 3, 1, 2).to(z.dtype)
    inter = (p * t).sum((2, 3), keepdim=True)
    union = ((p * p if square else p) + t).sum((2, 3), keepdim=True)
    r = 1.0 / (N * C) if reduction == "mean" else 1.0
    du = 2 * p if square else torch.ones_like(p)
    g = -r * (2 * t * (union + smooth) - (2 * inter + smooth) * du) / (union + smooth) ** 2
    return p * (g - (p * g).sum(1, keepdim=True))


def test_focal_gamma0_is_weighted_ce_sum_over_pixels():
    from loss_oracle import focal_loss_flat
    z, y = _case(C=4)
    w = torch.tensor([0.1, 0.4, 0.3, 0.2], dtype=torch.float64)
    ref = F.cross_entropy(z, y, weight=w, reduction="sum") / y.numel()
    assert torch.allclose(focal_loss_flat(z, y, w, gamma=0.0), ref, rtol=1e-12, atol=0)
    assert torch.allclose(focal_loss_flat(z, y, w, gamma=0.0, reduction="sum"), ref * y.numel(), rtol=1e-12, atol=0)
    # the focal term down-weights confident pixels: gamma > 0 lowers every pixel's loss
    assert focal_loss_flat(z, y, w, gamma=2.0) < ref


def test_dice_on_one_hot_probabilities_is_one_minus_f1():
    from sklearn.metrics import f1_score
    from loss_oracle import dice_loss
    N, C = 3, 4
    g = torch.Generator().manual_seed(1)
    pred = torch.randint(0, C, (N, 16, 16), generator=g)
    y = torch.randint(0, C, (N, 16, 16), generator=g)
    pred[1][pred[1] == 3] = 0          # class 3 absent from prediction and target of sample 1: d = smooth / smooth = 1
    y[1][y[1] == 3] = 1
    z = F.one_hot(pred, C).permute(0, 3, 1, 2).double() * 200.0       # softmax saturates to the one-hot prediction
    per = torch.stack([1 - (2 * ((z.softmax(1)[n] * F.one_hot(y[n], C).permute(2, 0, 1)).sum((1, 2))) + 1e-6) /
                       ((z.softmax(1)[n] + F.one_hot(y[n], C).permute(2, 0, 1)).sum((1, 2)) + 1e-6) for n in range(N)])
    f1 = torch.tensor(np.stack([f1_score(y[n].flatten().numpy(), pred[n].flatten().numpy(), labels=list(range(C)),
                                         average=None, zero_division=1) for n in range(N)]), dtype=torch.float64)
    assert torch.allclose(per, 1 - f1, atol=1e-6)
    assert abs(float(dice_loss(z, y)) - float((1 - f1).sum())) <= 1e-5
    assert abs(float(dice_loss(z, y, reduction="mean")) - float((1 - f1).mean())) <= 1e-6
    assert per[1, 3] == 0.0


@pytest.mark.parametrize("gamma", [0.0, 0.5, 2.0, 5.0])
@pytest.mark.parametrize("reduction", ["mean", "sum"])
def test_focal_gradcheck_and_closed_form(gamma, reduction):
    from loss_oracle import focal_loss_flat
    z, y = _case(C=3, seed=2)
    w = torch.tensor([0.2, 0.5, 0.3], dtype=torch.float64)
    zz = z.clone().requires_grad_(True)
    assert torch.autograd.gradcheck(lambda a: focal_loss_flat(a, y, w, gamma, reduction), (zz,))
    focal_loss_flat(zz, y, w, gamma, reduction).backward()
    assert torch.allclose(zz.grad, focal_grad(z, y, w, gamma, reduction), rtol=1e-10, atol=1e-14)


def test_focal_closed_form_is_finite_on_saturated_pixels():
    z = torch.zeros(1, 2, 2, 2, dtype=torch.float64)
    z[:, 0] = 800.0                                   # p_0 == 1 exactly: l = 0 on the pixels labelled 0
    y = torch.tensor([[[0, 0], [0, 1]]])
    w = torch.ones(2, dtype=torch.float64)
    for gamma in (0.0, 0.3, 0.5, 2.0):
        g = focal_grad(z, y, w, gamma, "mean")
        assert torch.isfinite(g).all(), gamma
        assert (g[0, :, 0, 0] == 0).all()


@pytest.mark.parametrize("square", [False, True])
@pytest.mark.parametrize("reduction", ["sum", "mean"])
def test_dice_gradcheck_and_closed_form(square, reduction):
    from loss_oracle import dice_loss
    z, y = _case(C=3, seed=3)
    y[0][y[0] == 2] = 0                               # a class absent from sample 0
    zz = z.clone().requires_grad_(True)
    assert torch.autograd.gradcheck(lambda a: dice_loss(a, y, 1e-6, reduction, square), (zz,))
    dice_loss(zz, y, 1e-6, reduction, square).backward()
    assert torch.allclose(zz.grad, dice_grad(z, y, 1e-6, reduction, square), rtol=1e-10, atol=1e-14)


# ------------------------------------------------------------------------------------------------ loss_func parser
def test_parser_accepts_every_form():
    from unet_b200.losses import LossSpec, parse_loss_func
    assert parse_loss_func(None) == LossSpec()
    assert parse_loss_func("CrossEntropyLossFlat(axis=1)") == LossSpec()
    assert parse_loss_func("CrossEntropyLossFlat") == LossSpec()
    assert parse_loss_func("FocalLossFlat(axis=1, gamma=3)") == LossSpec("focal", gamma=3.0)
    assert parse_loss_func(" FocalLossFlat() ") == LossSpec("focal", gamma=2.0, reduction="mean")
    assert parse_loss_func("FocalLossFlat(gamma=0.5, reduction='sum')") == LossSpec("focal", gamma=0.5, reduction="sum")
    assert parse_loss_func("DiceLoss()") == LossSpec("dice", reduction="sum", smooth=1e-6)
    assert parse_loss_func("DiceLoss(axis=1, smooth=1e-3, reduction='mean', square_in_union=True)") == \
        LossSpec("dice", smooth=1e-3, reduction="mean", square_in_union=True)
    spec = LossSpec("dice", square_in_union=True)
    assert parse_loss_func(spec) is spec
    assert LossSpec.from_dict(spec.as_dict()) == spec and LossSpec.from_dict(None) == LossSpec()

    # objects of the fastai classes: settings read off their attributes (FocalLossFlat keeps the reduction in .reduce)
    class FocalLossFlat:
        def __init__(self):
            self.axis, self.gamma, self.reduce = 1, 4, "sum"

    class DiceLoss:
        def __init__(self):
            self.axis, self.smooth, self.reduction, self.square_in_union = 1, 0.5, "mean", True

    class CrossEntropyLossFlat:
        axis = 1

    assert parse_loss_func(FocalLossFlat()) == LossSpec("focal", gamma=4.0, reduction="sum")
    assert parse_loss_func(DiceLoss()) == LossSpec("dice", smooth=0.5, reduction="mean", square_in_union=True)
    assert parse_loss_func(CrossEntropyLossFlat()) == LossSpec()
    assert parse_loss_func(torch.nn.L1Loss()) is None          # not recognised: the caller warns and keeps CE


@pytest.mark.parametrize("bad", [
    "FocalLossFlat(axis=-1)", "DiceLoss(axis=2)", "LabelSmoothingCrossEntropyFlat()", "BCEWithLogitsLossFlat(axis=1)",
    "FocalLossFlat(gamma=2, weight=None)", "DiceLoss(gamma=2)", "CrossEntropyLossFlat(axis=1, reduction='sum')",
    "FocalLossFlat(gamma=__import__('os'))", "FocalLossFlat(gamma=2+x)", "FocalLossFlat(2)", "FocalLossFlat(**{})",
    "losses.FocalLossFlat()", "FocalLossFlat(gamma=-1)", "FocalLossFlat(gamma='2')", "FocalLossFlat(gamma=True)",
    "DiceLoss(reduction='none')", "DiceLoss(smooth=0)", "DiceLoss(square_in_union=1)", "FocalLossFlat(", "",
    "[FocalLossFlat()]"])
def test_parser_rejects(bad):
    from unet_b200.losses import parse_loss_func
    with pytest.raises(ValueError):
        parse_loss_func(bad)


def test_parser_rejects_a_bad_axis_on_an_object():
    from unet_b200.losses import parse_loss_func

    class FocalLossFlat:
        axis, gamma, reduce = -1, 2.0, "mean"
    with pytest.raises(ValueError):
        parse_loss_func(FocalLossFlat())


def test_dice_ignores_class_weights_with_a_warning():
    from unet_b200.losses import LossSpec, warn_dice_weights
    with pytest.warns(UserWarning, match="no class weights"):
        warn_dice_weights(LossSpec("dice"), [0.2, 0.8])
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        warn_dice_weights(LossSpec("dice"), [0.5, 0.5])          # "even"
        warn_dice_weights(LossSpec("dice"), None)
        warn_dice_weights(LossSpec("focal"), [0.2, 0.8])


def test_blocks_per_sample():
    from unet_b200.losses import dice_blocks_per_sample
    assert dice_blocks_per_sample(64, 256 * 256) == 10          # the training shape: 640 blocks of 6 554 pixels
    assert dice_blocks_per_sample(1, 64 * 64) == 2
    assert dice_blocks_per_sample(1000, 32 * 32) == 1


# ------------------------------------------------------------------------------------------------ params_and_main
@pytest.mark.parametrize("extra,want", [(True, "DiceLoss(square_in_union=True)"), (False, None)])
def test_params_and_main_passes_loss_func_to_train_func(monkeypatch, extra, want):
    import unet_b200.reference_api as ra
    from unet_b200 import params_and_main
    seen = {}

    def fake_train_func(*args, **kwargs):
        seen["loss_func"] = args[13]
        return "learner"
    monkeypatch.setattr(ra, "train_func", fake_train_func)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        out = params_and_main.main({"Create_tiles": False, "Train": True, "enable_extra_parameters": extra,
                                    "loss_func": "DiceLoss(square_in_union=True)"})
    assert out["learner"] == "learner" and seen["loss_func"] == want
