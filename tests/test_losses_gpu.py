"""FocalLossFlat and DiceLoss on the B200: the kernels against a float64 torch evaluation of the oracle, the plan's
loss_and_grad against autograd and the teacher-forced emulation, and the `loss_func` choice through the reference API.

Bounds: loss <= 1e-5 relative, dlogits <= 1e-2 of the tensor maximum (bf16 storage; the CE kernel's bound), zeros in the
padding lanes beyond C, bit-identical results on a second call."""
import copy
import json

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from parity_util import gradient_mismatches, plan_taps, rel

GRAD_TOL, GRAD_COS, GRAD_TOL_MAX = 3e-2, 0.999, 1e-1      # as tests/test_network_gpu.py
ACT_TOL = 2 * 2.0 ** -8


def _oracle_loss(spec, w):
    from loss_oracle import dice_loss, focal_loss_flat
    if spec.name == "focal":
        return lambda z, y: focal_loss_flat(z, y, w, spec.gamma, spec.reduction)
    return lambda z, y: dice_loss(z, y, spec.smooth, spec.reduction, spec.square_in_union)


def _run_kernels(spec, z_nhwc, y, C, ldg, weight, grad_scale, with_grad=True):
    """z_nhwc: fp32 [N,H,W,ld] on the device; returns (loss scalar, dlogits [N,H,W,ldg] bf16 or None)"""
    from unet_b200 import _lib, ops
    from unet_b200.losses import dice_blocks_per_sample, launch_loss
    lib = _lib.load()
    N, H, W, _ = z_nhwc.shape
    dev = z_nhwc.device
    rows = 592
    bps = dice_blocks_per_sample(N, H * W)
    part = torch.full((max(rows, N),), float("nan"), device=dev)
    dpart = torch.full((N * bps * 3 * C,), float("nan"), device=dev)
    loss = torch.zeros(1, device=dev)
    dl = torch.full((N, H, W, ldg), 7.0, dtype=torch.bfloat16, device=dev) if with_grad else None
    launch_loss(lib, spec, z_nhwc, y, N, H * W, C, None if weight is None else weight.data_ptr(),
                None if dl is None else dl.data_ptr(), ldg, part, rows, dpart, bps, loss, grad_scale, ops.stream_ptr())
    torch.cuda.synchronize()
    return loss.clone(), dl


def _check_kernels(spec, N, H, W, C, ld, ldg, weighted, saturate=False, absent=False, seed=0):
    dev = "cuda"
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(N, H, W, ld, generator=g) * 3
    if saturate:                    # the top class leads by >= 400: softmax is exactly one-hot in fp32
        z[..., :C] += 400.0 * torch.nn.functional.one_hot(z[..., :C].argmax(-1), C)
    y = torch.randint(0, C, (N, H, W), generator=g, dtype=torch.uint8)
    if absent:
        y[0][y[0] == 1] = 0         # class 1 absent from sample 0
    if saturate:                    # most pixels correct and saturated (l == 0 exactly)
        keep = torch.rand(N, H, W, generator=g) < 0.9
        y = torch.where(keep, z[..., :C].argmax(-1).to(torch.uint8), y)
    w = (torch.rand(C, generator=g) + 0.2) if weighted else torch.full((C,), 1.0 / C)
    zd, yd, wd = z.to(dev), y.to(dev), w.to(dev)
    gs = 2.0
    loss, dl = _run_kernels(spec, zd, yd, C, ldg, wd, gs)
    z64 = z[..., :C].double().permute(0, 3, 1, 2).contiguous().requires_grad_(True)
    ref = _oracle_loss(spec, w.double())(z64, y.long())
    (gs * ref).backward()
    assert abs(loss.item() - ref.item()) <= 1e-5 * abs(ref.item()) + 1e-7, (loss.item(), ref.item())
    got = dl[..., :C].float().cpu().permute(0, 3, 1, 2)
    assert torch.isfinite(dl.float()).all()
    # autograd of (1 - pt)^gamma at l == 0 exactly (saturated correct pixels, gamma < 1) is 0 * inf = NaN in float64;
    # the gradient's limit there is 0, which is what the kernel writes (tests/test_losses_cpu.py pins the closed form)
    want = torch.nan_to_num(z64.grad, nan=0.0) if saturate else z64.grad
    assert rel(got, want) <= 1e-2, rel(got, want)
    assert (dl[..., C:] == 0).all()
    loss2, dl2 = _run_kernels(spec, zd, yd, C, ldg, wd, gs)
    assert torch.equal(loss, loss2) and torch.equal(dl, dl2)
    # loss only (validation): the same loss, no gradient written
    loss3, _ = _run_kernels(spec, zd, yd, C, ldg, wd, gs, with_grad=False)
    assert torch.equal(loss, loss3)


@pytest.mark.parametrize("C", [2, 3, 8, 32])
@pytest.mark.parametrize("gamma", [0.0, 0.5, 2.0, 5.0])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("reduction", ["mean", "sum"])
def test_focal_kernel(C, gamma, weighted, reduction):
    from unet_b200.losses import LossSpec
    spec = LossSpec("focal", gamma=gamma, reduction=reduction)
    ld, ldg = C + 3, ((C + 7) // 8) * 8 + 8
    _check_kernels(spec, 2, 24, 20, C, ld, ldg, weighted, seed=C)
    if gamma < 1.0:
        _check_kernels(spec, 2, 24, 20, C, ld, ldg, weighted, saturate=True, seed=C + 1)


@pytest.mark.parametrize("C", [2, 3, 8, 32])
@pytest.mark.parametrize("square", [False, True])
@pytest.mark.parametrize("reduction", ["sum", "mean"])
def test_dice_kernel(C, square, reduction):
    from unet_b200.losses import LossSpec
    spec = LossSpec("dice", reduction=reduction, square_in_union=square)
    ld, ldg = C + 3, ((C + 7) // 8) * 8 + 8
    _check_kernels(spec, 3, 40, 36, C, ld, ldg, False, absent=True, seed=10 + C)


@pytest.mark.parametrize("spec_kw", [dict(name="focal", gamma=2.0), dict(name="dice", reduction="sum")])
def test_losses_at_the_training_shape(spec_kw):
    """64 x 256^2 x 2: many blocks per sample (Dice) and the 592-block focal grid"""
    from unet_b200.losses import LossSpec
    _check_kernels(LossSpec(**spec_kw), 64, 256, 256, 2, 2, 8, False, seed=5)


# ------------------------------------------------------------------------------------------------ the plan
def _teacher_forced(oracle, net, x, yl, loss_fn, logits):
    """tests/test_network_gpu.py::teacher_forced_check with the chosen loss in place of weighted_ce"""
    from oracle.bf16_emulation import emulated_forward
    o_tf = copy.deepcopy(oracle)
    o_tf.zero_grad()
    taps, free, mism = plan_taps(net), {}, {}
    l_tf = emulated_forward(o_tf, x, True, taps=taps, record=free, mismatch=mism)
    loss_fn(l_tf, yl).backward()
    assert rel(logits, l_tf) <= 1e-4, rel(logits, l_tf)
    assert len(mism) >= len(free) - 1
    off = {k: e for k, e in mism.items() if e > ACT_TOL}
    assert not off, sorted(off.items(), key=lambda kv: -kv[1])[:5]
    ref = {n: p.grad for n, p in o_tf.named_parameters()}
    grads = net.named_grads()
    check = lambda g: gradient_mismatches(g, ref, GRAD_TOL, GRAD_COS, GRAD_TOL_MAX, {})
    bad = check(grads)
    assert not bad, sorted(bad, key=lambda b: -b[1])[:10]
    victim = [n for n in ref if n.endswith("convpath.1.0.weight") and n.startswith("layers.0.7.")][-1]
    for mutate in (torch.zeros_like, lambda g: -g, lambda g: 1.05 * g):
        broken = dict(grads)
        broken[victim] = mutate(grads[victim])
        assert [b[0] for b in check(broken)] == [victim]


@pytest.mark.parametrize("spec_kw", [dict(name="focal", gamma=2.0), dict(name="dice", reduction="sum"),
                                     dict(name="dice", reduction="mean", square_in_union=True)])
def test_plan_loss_and_grad(spec_kw):
    from oracle.unet_oracle import make_oracle
    from unet_b200.losses import LossSpec
    from unet_b200.network import UNetB200
    from unet_b200.synth import aerial_like_tiles
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    arch, n_in, n_out, size, batch = "xresnet34", 4, 2, 128, 4
    spec = LossSpec(**spec_kw)
    oracle = make_oracle(arch, n_in, n_out, seed=0).cuda().train()
    o_init = copy.deepcopy(oracle)
    net = UNetB200(arch, n_in, n_out, (size, size), batch, training=True, loss_spec=spec)
    net.load_state_dict(oracle.state_dict())
    x_u8, y = aerial_like_tiles(batch, n_in, size, size, n_out)
    x_u8, y = x_u8.cuda(), y.cuda()
    x, yl = x_u8.float() / 255.0, y.long()
    w = torch.full((n_out,), 1.0 / n_out, device="cuda")
    loss_fn = _oracle_loss(spec, w)
    net.set_input(x_u8)
    net.set_labels(y)
    net.forward()
    loss = net.loss_and_grad()
    net.backward()
    torch.cuda.synchronize()
    logits = net.logits_nchw()
    # the loss and dlogits on the plan's own logits
    z64 = logits.double().requires_grad_(True)
    ref = _oracle_loss(spec, w.double())(z64, yl)
    ref.backward()
    assert abs(loss.item() - ref.item()) <= 1e-5 * abs(ref.item()), (loss.item(), ref.item())
    dl = net.dlogits[..., :n_out].float().permute(0, 3, 1, 2)
    assert rel(dl, z64.grad) <= 1e-2 and (net.dlogits[..., n_out:] == 0).all()
    # every parameter gradient against the teacher-forced bf16 emulation under the same loss
    _teacher_forced(o_init, net, x, yl, loss_fn, logits)
    g1 = net.grads.clone()
    net.forward()
    net.loss_and_grad()
    net.backward()
    torch.cuda.synchronize()
    assert torch.equal(g1, net.grads)


# ------------------------------------------------------------------------------------------------ the reference API
def _tiles(tmp_path, n_train=16, n_valid=4, seed=5):
    from unet_b200.geotiff import GeoInfo, write_geotiff
    from unet_b200.synth import aerial_like_tiles
    x, y = aerial_like_tiles(n_train + n_valid, 4, 64, 64, 2, seed=seed)
    for scene, sl in (("trai", slice(0, n_train)), ("vali", slice(n_train, n_train + n_valid))):
        for sub in ("img_tiles", "mask_tiles"):
            (tmp_path / "data" / scene / sub).mkdir(parents=True)
        for i in range(sl.start, sl.stop):
            write_geotiff(tmp_path / "data" / scene / "img_tiles" / f"t{i}.tif", x[i].numpy(), GeoInfo())
            write_geotiff(tmp_path / "data" / scene / "mask_tiles" / f"t{i}.tif", y[i].numpy(), GeoInfo())
    return x, y


@pytest.mark.parametrize("loss_func,want", [("FocalLossFlat(axis=1, gamma=2)", dict(name="focal", gamma=2.0)),
                                            ("DiceLoss()", dict(name="dice", reduction="sum"))])
def test_train_func_with_loss_func(tmp_path, loss_func, want):
    from unet_b200.losses import LossSpec
    from unet_b200.reference_api import load_learner, train_func
    x, y = _tiles(tmp_path)
    learn = train_func(tmp_path / "data", None, tmp_path / "models", "run", 8, False, False, "even", "xresnet18", 4, 2e-3,
                       10, None, loss_func, "dice_multi", False, "vali", ["background", "forest"])
    spec = LossSpec(**want)
    assert learn.loss_spec == spec and learn.net.loss_spec == spec
    h = learn.history
    assert len(h) == 4 and all(np.isfinite(r["train_loss"]) and np.isfinite(r["valid_loss"]) for r in h)
    d = tmp_path / "models" / "run"
    assert json.load(open(d / "run.json"))["loss_func"] == spec.as_dict()
    again = load_learner(d / "run.pkl")
    assert again.loss_spec == spec
    assert torch.equal(again.predict(x[0])[1], learn.predict(x[0])[1])

    # valid_loss in the chosen loss, AvgLoss over the real samples of a padded last batch
    pad = lambda t: torch.cat([t[8:], t[8:9].expand(3, *t.shape[1:])], 0)
    xs, ys = x[:13], y[:13]
    batches = [(xs[:8], ys[:8], 8), (pad(xs), pad(ys), 5)]
    got = again.validate(batches)
    net = again._eval_net()
    loss_fn = _oracle_loss(spec, torch.full((2,), 0.5, dtype=torch.float64, device="cuda"))
    tot = 0.0
    for xb, yb, n in batches:
        net.set_input(xb.cuda().contiguous())
        net.forward()
        lg = net.logits_nchw()[:n].double()
        tot += loss_fn(lg, yb[:n].cuda().long()).item() * n
    want_loss = tot / 13
    assert abs(got["valid_loss"] - want_loss) <= 1e-5 * abs(want_loss), (got["valid_loss"], want_loss)

    # the captured training step lowers the chosen loss on the learnable synthetic task (training-mode loss of repeated
    # steps on the same batches at a fixed learning rate: no BatchNorm running statistics involved)
    learn.trainer.set_adam_hyper(2e-3, 0.9)
    first = [learn.trainer.step(x[i:i + 8], y[i:i + 8]).item() for i in (0, 8)]
    for _ in range(10):
        last = [learn.trainer.step(x[i:i + 8], y[i:i + 8]).item() for i in (0, 8)]
    assert np.isfinite(last).all() and sum(last) < sum(first), (first, last)


def test_loss_choice_round_trips_and_old_checkpoints_load_as_ce(tmp_path):
    from unet_b200.losses import LossSpec
    from unet_b200.reference_api import load_learner, unet_learner_MS
    learn = unet_learner_MS(4, 3, arch="xresnet18", size=(64, 64), batch_size=2,
                            loss_func="DiceLoss(smooth=0.01, reduction='mean', square_in_union=True)")
    spec = LossSpec("dice", smooth=0.01, reduction="mean", square_in_union=True)
    assert learn.loss_spec == spec
    learn.export(tmp_path / "m.pkl")
    ck = torch.load(tmp_path / "m.pkl", map_location="cpu", weights_only=True)
    assert ck["loss_func"] == spec.as_dict()
    assert load_learner(tmp_path / "m.pkl").loss_spec == spec
    del ck["loss_func"]                                  # a checkpoint written before the loss was recorded
    torch.save(ck, tmp_path / "old.pkl")
    assert load_learner(tmp_path / "old.pkl").loss_spec == LossSpec()
    with pytest.warns(UserWarning, match="not supported"):
        assert unet_learner_MS(4, 2, arch="xresnet18", size=(64, 64), batch_size=2,
                               loss_func=torch.nn.L1Loss()).loss_spec == LossSpec()
    with pytest.warns(UserWarning, match="no class weights"):
        unet_learner_MS(4, 2, arch="xresnet18", size=(64, 64), batch_size=2, class_weights=[0.3, 0.7],
                        loss_func="DiceLoss()")


@pytest.mark.parametrize("loss_func", ["FocalLossFlat(gamma=2)", "DiceLoss()"])
def test_regression_accepts_only_mse(loss_func):
    from unet_b200.losses import parse_loss_func
    from unet_b200.network import UNetB200
    from unet_b200.reference_api import unet_learner_MS
    with pytest.raises(ValueError):
        unet_learner_MS(4, 1, arch="xresnet18", size=(64, 64), batch_size=2, regression=True, loss_func=loss_func)
    with pytest.raises(ValueError):
        UNetB200("xresnet18", 4, 1, (64, 64), 2, regression=True, loss_spec=parse_loss_func(loss_func))
