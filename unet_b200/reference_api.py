"""Host-side mirror of the reference's Python seams for the hot path (same names, argument meaning and error behaviour),
running on the B200 plan instead of fastai.

    reference                                               here
    --------------------------------------------------------------------------------------------------------------
    train.unet_learner_MS(dls, arch, ...)  train.py:98      unet_learner_MS(n_in, n_classes, arch, size, batch_size, ...)
    learn.fit_one_cycle(epochs, lr_max=slice(lr/ef, lr))    Learner.fit_one_cycle(epochs, lr_max, train_batches, valid_batches)
                                           train.py:246-250
    learn.predict(tile) -> (dec, argmax, probs)             Learner.predict(tile_u8)
                                           predict.py:193
    learn.export(path) / load_learner(path) train.py:373    Learner.export(path) / load_learner(path)   (state_dict with fastai keys)
    predict.save_predictions(...)          predict.py:146   save_predictions(...) over GeoTIFF (or .npy) tiles
    train.train_func(...)                  train.py:287     train_func(...) over data_path/{trai,vali}/{img,mask}_tiles/*.tif
    create_tiles_unet.compute_windows      :30              unet_b200.tiling.compute_windows

Data enters as uint8 tiles `[B, n_in, H, W]` (the reference reads GeoTIFF bands as int32 -> float32 and fastai divides by
255, data.py:24 + IntToFloatTensor; both happen inside the cast kernel) and class-id masks `[B, H, W]`.
Tiles on disk are GeoTIFFs (`unet_b200/geotiff.py`, a numpy restatement of the rasterio/GDAL calls of the path) or `.npy`
arrays; `train_func` / `save_predictions` keep the reference's positional signatures, `predict_geotiff` is the tile-free
whole-raster variant.
"""
from __future__ import annotations

import csv
import math
import os
import time
import warnings
from pathlib import Path
from typing import Callable, Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib, ops
from .assessment import ConfusionCounter, RegressionCounter, write_regression_report, write_report
from .engine import Trainer, one_cycle
from .network import UNetB200, input_divisors
from .predict_engine import StitchPlan, TiledPredictor, finalize_probs, gather_mask_strips
from .losses import LossSpec, dice_blocks_per_sample, launch_loss, parse_loss_func, warn_dice_weights
from .geotiff import GeoInfo, geotiff_info, open_mask, open_tile, read_geotiff, write_geotiff
from .tiling import column_owned, compute_windows, placement_from_geotransform, shard_windows_by_columns, split_range

ARCHITECTURES = ("xresnet18", "xresnet34", "xresnet50", "xresnet101")   # params_and_main.py:12,99


def _arch_name(arch) -> str:
    name = arch if isinstance(arch, str) else getattr(arch, "__name__", str(arch))
    if name not in ARCHITECTURES:
        # the reference only works with xresnet bodies: body[0][0] must be a ConvLayer (train.py:130)
        raise TypeError(f"architecture {name!r} is not an xresnet body; choose from {ARCHITECTURES}")
    return name


class Learner:
    """What `unet_learner_MS` returns: model + loss + optimizer + schedule, on one GPU (or one rank of a DP job:
    under `torch.distributed` the trainer all-reduces the gradients, see engine.Trainer)."""

    def __init__(self, arch: str, n_in: int, n_classes: int, size: Tuple[int, int], batch_size: int,
                 class_weights: Optional[Sequence[float]] = None, opt_func: str = "adam", lr: float = 1e-3,
                 wd: float = 0.01, encoder_factor: float = 10.0, moms: Sequence[float] = (0.95, 0.85, 0.95),
                 self_attention: bool = False, regression: bool = False, input_dtype: torch.dtype = torch.uint8,
                 sixteen_bit: bool = False, loss_spec: Optional[LossSpec] = None):
        self.arch, self.n_in, self.n_classes, self.size, self.bs = arch, n_in, n_classes, tuple(size), batch_size
        self.class_weights = list(class_weights) if class_weights is not None else None
        self.self_attention, self.regression = bool(self_attention), bool(regression)
        # A0 input contract: raw band values of `input_dtype`; a dataset whose values exceed 8 bits ('int16' in the
        # reference, utils.py:72-89) is divided by 255 twice, the regression variant once less (network.input_divisors)
        self.input_dtype, self.sixteen_bit = input_dtype, bool(sixteen_bit)
        self.input_div = input_divisors(self.sixteen_bit, self.regression)
        self.n_out = 1 if self.regression else n_classes                    # train.py:137-140
        self.loss_spec = loss_spec or LossSpec()
        self.net = UNetB200(arch, n_in, self.n_out, self.size, batch_size, training=True,
                            class_weights=None if self.regression else self.class_weights,
                            self_attention=self.self_attention, input_div=self.input_div, regression=self.regression,
                            loss_spec=self.loss_spec)
        # fastai's own start: BatchNorm gamma 1 / beta 1e-3, gamma 0 on the last BatchNorm of every ResBlock (BatchZero),
        # decoder biases N(0, 0.01) (network.init_parameters)
        self.net.init_parameters(seed=0, randomize_bn=False)
        self.trainer = Trainer(self.net, optimizer=opt_func, lr=lr, wd=wd, encoder_factor=encoder_factor,
                               input_dtype=input_dtype)
        self.lr, self.moms = lr, tuple(moms)
        self._eval: Optional[UNetB200] = None
        self._version, self._eval_version = 0, -1       # the eval plan is re-staged only when the weights changed
        self._val: Optional[dict] = None
        self.history: List[Dict[str, float]] = []

    # ---- training ------------------------------------------------------------------------------------------------
    @property
    def metric_names(self) -> List[str]:
        return ["_rmse", "r2_score"] if self.regression else ["dice_multi"]      # train.py:190,194 (fastai metric names)

    def fit_one_cycle(self, epochs: int, lr_max: Optional[float] = None,
                      train_batches: Optional[Callable[[], Iterable]] = None,
                      valid_batches: Optional[Callable[[], Iterable]] = None, history_csv: Optional[str] = None,
                      monitor: Optional[str] = None, best_path: Optional[str] = None) -> List[Dict[str, float]]:
        """fastai fit_one_cycle: cosine warm-up over the first 25 % from lr/25, anneal to lr/1e5, momentum 0.95->0.85->0.95;
        CSVLogger columns epoch,train_loss,valid_loss,<metrics>,time (history.csv:1) with train_loss = fastai's
        AvgSmoothLoss (debiased exponential average, beta 0.98, running across epochs); SaveModelCallback keeps the best
        epoch by `monitor` and reloads it after the fit (train.py:198-209).  Batches are (x, y) or (x, y, n_real)."""
        assert train_batches is not None, "train_batches: callable returning an iterable of (x_raw, y) batches"
        if os.environ.get("B2U_DIAG_SKIP_ALLREDUCE") is not None:
            raise RuntimeError("B2U_DIAG_SKIP_ALLREDUCE is a bench diagnostic (un-reduced gradients): unset it to train")
        lr_max = self.lr if lr_max is None else lr_max
        monitor = monitor or ("r2_score" if self.regression else "dice_multi")      # train.py:198-201
        n_per_epoch = getattr(train_batches, "n_batches", None)
        if n_per_epoch is None:
            n_per_epoch = sum(1 for _ in train_batches())
        total, step = max(1, epochs * n_per_epoch), 0
        best = None
        rank0 = _rank() == 0
        losses = torch.zeros(max(1, n_per_epoch), dtype=torch.float32, device=self.net.device)
        smooth, count = 0.0, 0
        for ep in range(epochs):
            t0 = time.time()
            n = 0
            it = iter(train_batches())
            cur = next(it, None)
            while cur is not None:
                nxt = next(it, None)
                x, y = cur[0], cur[1]
                lr, mom = one_cycle(step / total, lr_max, moms=self.moms)
                if self.trainer.optimizer == "adam":
                    self.trainer.set_adam_hyper(lr, mom)
                else:
                    self.trainer.lr = lr
                # the next batch's H2D copy runs behind this step; the loss stays on the device (no host sync per step).
                # Device batches are not prefetched: the side copy stream would not wait for the kernel producing them.
                loss = self.trainer.step(x, y, prefetch=None if nxt is None or nxt[0].is_cuda else (nxt[0], nxt[1]))
                if n < losses.numel():
                    losses[n:n + 1].copy_(loss, non_blocking=True)
                n += 1
                step += 1
                cur = nxt
            self._version += 1
            for v in losses[:min(n, losses.numel())].cpu().tolist():     # fastai AvgSmoothLoss: lerp + debias
                count += 1
                smooth = 0.98 * smooth + 0.02 * v
            row = {"epoch": ep, "train_loss": smooth / (1 - 0.98 ** count) if count else float("nan")}
            if valid_batches is not None:
                row.update(self.validate(valid_batches()))
            row["time"] = time.time() - t0
            self.history.append(row)
            score = row.get(monitor)
            if best_path and score is not None and not math.isnan(score) and \
                    (best is None or (score < best if "loss" in monitor else score > best)):
                best = score
                if rank0:
                    torch.save(self.state_dict(), best_path)
        if best_path and best is not None:
            _barrier()
            if os.path.exists(best_path):
                # fastai SaveModelCallback(monitor, fname='best-model') reloads the best epoch after fit (train.py:209)
                self.load_state_dict(torch.load(best_path, map_location="cpu", weights_only=True))
        if history_csv and rank0:
            cols = ["valid_loss"] + self.metric_names
            with open(history_csv, "w", newline="") as f:
                wr = csv.writer(f)
                wr.writerow(["epoch", "train_loss"] + cols + ["time"])
                for r in self.history:
                    m, s_ = divmod(int(r["time"]), 60)
                    wr.writerow([r["epoch"], r["train_loss"]] + [r.get(c, "") for c in cols] + [f"{m:02d}:{s_:02d}"])
        return self.history

    def _eval_net(self) -> UNetB200:
        """the eval plan (running BatchNorm statistics folded into the convolutions); its weights are re-staged only when
        the training plan's parameters changed since the last call"""
        if self._eval is None:
            self._eval = UNetB200(self.arch, self.n_in, self.n_out, self.size, self.bs, training=False,
                                  class_weights=None if self.regression else self.class_weights,
                                  self_attention=self.self_attention, input_div=self.input_div,
                                  regression=self.regression)
        if self._eval_version != self._version:
            self._eval.load_state_dict(self.net.state_dict())
            self._eval_version = self._version
        return self._eval

    def _val_buffers(self, net: UNetB200) -> dict:
        if self._val is None:
            dev, rows = net.device, 592
            f = lambda n, dt=torch.float32: torch.zeros(n, dtype=dt, device=dev)
            bps = dice_blocks_per_sample(net.N, net.H * net.W) if self.loss_spec.name == "dice" else 0
            self._val = dict(rows=rows, wsum=f(rows), part=f(max(rows, net.N)), loss=f(1), losses=f(4096),
                             dice_bps=bps, dice_part=f(max(1, net.N * bps * 3 * self.n_out)),
                             labels=torch.zeros((net.N, net.H, net.W), device=dev,
                                                dtype=torch.float32 if self.regression else torch.uint8),
                             counts=f(3 * max(1, self.n_classes), torch.int64), sums=f(4, torch.float64),
                             partial=f(3 * rows, torch.float64), ticket=f(1, torch.int32))
        return self._val

    def validate(self, batches: Iterable) -> Dict[str, float]:
        """One pass over the validation batches on the eval plan, reduced on the device: valid_loss as fastai's AvgLoss
        (per-batch loss weighted by the number of REAL samples: a padded last batch does not count its padding; the loss
        is the one the model trains with, and a Dice loss sums its statistics over the real samples only) and
        DiceMulti (macro Dice over the classes present; regression: rmse and R2Score).  One device-to-host read at the end."""
        net = self._eval_net()
        lib, v = net.lib, self._val_buffers(net)
        s = ops.stream_ptr()
        ld, HW = net.logits.shape[-1], net.H * net.W
        v["counts"].zero_()
        v["sums"].zero_()
        ns: List[int] = []
        for batch in batches:
            x, y = batch[0], batch[1]
            n = int(batch[2]) if len(batch) > 2 else int(x.shape[0])
            if len(ns) >= v["losses"].numel():
                raise ValueError("more than 4096 validation batches")
            net.set_input(x.to(net.device, non_blocking=True).contiguous())
            v["labels"].copy_(y.to(v["labels"].dtype), non_blocking=True)
            net.forward()
            P_ = n * HW
            if self.regression:
                _lib.check(lib.b2u_mse_fwd_bwd(net.logits.data_ptr(), ld, v["labels"].data_ptr(), P_, None, 0,
                                               v["part"].data_ptr(), v["rows"], 1.0, s), "b2u_mse_fwd_bwd")
                _lib.check(lib.b2u_mse_finalize(v["part"].data_ptr(), v["rows"], P_, v["loss"].data_ptr(), s),
                           "b2u_mse_finalize")
                _lib.check(lib.b2u_regression_sums(net.logits.data_ptr(), ld, v["labels"].data_ptr(), P_,
                                                   v["partial"].data_ptr(), v["rows"], v["sums"].data_ptr(),
                                                   v["ticket"].data_ptr(), s), "b2u_regression_sums")
            elif self.loss_spec.name != "ce":
                # the loss the model trains with (FocalLossFlat / DiceLoss), over the n real samples
                launch_loss(lib, self.loss_spec, net.logits, v["labels"], n, HW, net.n_out, net.class_weights.data_ptr(),
                            None, 0, v["part"], v["rows"], v["dice_part"], v["dice_bps"], v["loss"], 1.0, s)
                _lib.check(lib.b2u_dice_counts(net.logits.data_ptr(), ld, v["labels"].data_ptr(), P_, net.n_out,
                                               v["counts"].data_ptr(), s), "b2u_dice_counts")
            else:
                w = net.class_weights.data_ptr()
                _lib.check(lib.b2u_ce_weight_sum(v["labels"].data_ptr(), P_, w, net.n_out, v["wsum"].data_ptr(),
                                                 v["rows"], s), "b2u_ce_weight_sum")
                _lib.check(lib.b2u_ce_fwd_bwd(net.logits.data_ptr(), ld, v["labels"].data_ptr(), P_, net.n_out, w,
                                              v["wsum"].data_ptr(), v["rows"], None, 0, v["part"].data_ptr(), v["rows"],
                                              1.0, s), "b2u_ce_fwd_bwd")
                _lib.check(lib.b2u_ce_finalize(v["part"].data_ptr(), v["rows"], v["wsum"].data_ptr(), v["rows"],
                                               v["loss"].data_ptr(), s), "b2u_ce_finalize")
                _lib.check(lib.b2u_dice_counts(net.logits.data_ptr(), ld, v["labels"].data_ptr(), P_, net.n_out,
                                               v["counts"].data_ptr(), s), "b2u_dice_counts")
            v["losses"][len(ns):len(ns) + 1].copy_(v["loss"], non_blocking=True)
            ns.append(n)
        if not ns:
            return {"valid_loss": float("nan"), **{m: float("nan") for m in self.metric_names}}
        losses = v["losses"][:len(ns)].cpu().double().numpy()
        out = {"valid_loss": float((losses * np.array(ns)).sum() / sum(ns))}
        if self.regression:
            sse, st, stt, cnt = v["sums"].cpu().tolist()
            ss_tot = stt - st * st / cnt
            out["_rmse"] = math.sqrt(sse / cnt)
            out["r2_score"] = 1.0 - sse / ss_tot if ss_tot > 0 else float("nan")
        else:
            c = v["counts"].cpu().double().numpy().reshape(3, -1)
            den = c[1] + c[2]
            dice = [2 * c[0][k] / den[k] for k in range(c.shape[1]) if den[k] > 0]
            out["dice_multi"] = float(np.mean(dice)) if dice else float("nan")
        return out

    # ---- inference -------------------------------------------------------------------------------------------------
    def predict(self, tile):
        """fastai `Learner.predict` (predict.py:193): (decoded mask, argmax [H,W], probabilities [C,H,W]) as CPU tensors;
        the regression variant returns (prediction [1,H,W], prediction [1,H,W]) as `Learner_adjust.predict` does
        (train.py:87-95)."""
        t = torch.as_tensor(tile)
        if t.dim() != 3 or t.shape[0] != self.n_in:
            raise ValueError(f"expected a [{self.n_in}, H, W] tile, got {tuple(t.shape)}")
        net = self._eval_net()
        pred = TiledPredictor(net)
        if self.regression:
            out = pred.predict_tiles_raw(t[None].to(net.device).contiguous())[0].cpu()
            return out, out
        probs, amax = pred.predict_tiles(t[None].to(net.device).contiguous())
        return amax[0].cpu(), amax[0].cpu(), probs[0].cpu()

    # ---- persistence -------------------------------------------------------------------------------------------------
    def state_dict(self) -> Dict[str, torch.Tensor]:
        return self.net.state_dict()

    def load_state_dict(self, sd: Dict[str, torch.Tensor]) -> None:
        self.net.load_state_dict(sd)
        self._version += 1

    def export(self, path) -> None:
        """`learn.export` (train.py:373): a plain torch checkpoint with fastai state_dict keys + the constructor args
        (a pickled fastai Learner cannot be produced without fastai).  Tensors, strings, numbers and lists only, so
        that it loads with `weights_only=True`."""
        Path(path).parent.mkdir(parents=True, exist_ok=True)
        torch.save({"arch": self.arch, "n_in": self.n_in, "n_classes": self.n_classes, "size": list(self.size),
                    "batch_size": self.bs, "class_weights": self.class_weights, "self_attention": self.self_attention,
                    "regression": self.regression, "sixteen_bit": self.sixteen_bit,
                    "input_dtype": str(self.input_dtype).replace("torch.", ""), "loss_func": self.loss_spec.as_dict(),
                    "state_dict": {k: v.cpu() for k, v in self.state_dict().items()}}, path)


def _rank() -> int:
    import torch.distributed as dist
    return dist.get_rank() if dist.is_available() and dist.is_initialized() else 0


def _world() -> int:
    import torch.distributed as dist
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def _barrier() -> None:
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        dist.barrier()


def unet_learner_MS(n_in: int, n_classes: int, arch="xresnet34", size: Tuple[int, int] = (256, 256),
                    batch_size: int = 4, pretrained=None, loss_func=None, class_weights=None, opt_func: str = "adam",
                    lr: float = 1e-3, wd: float = 0.01, encoder_factor: float = 10.0, moms=(0.95, 0.85, 0.95),
                    regression: bool = False, self_attention: bool = False, input_dtype: torch.dtype = torch.uint8,
                    sixteen_bit: bool = False) -> Learner:
    """train.py:98-160.  `n_in` / `size` replace what the reference probes from `dls.train_ds` (:124-125) and
    `n_classes` replaces `len(dls.vocab)` (:140); `pretrained` may be a state_dict with fastai keys.  `regression`:
    n_out = 1 (:137-138), MSELossFlat (:189-192), rmse / R2Score metrics (:190).  `input_dtype` / `sixteen_bit`: the
    element type of the raw tiles and whether the dataset is the reference's 'int16' kind (utils.py:72-89).
    `loss_func`: None (CrossEntropyLossFlat(axis=1) with `class_weights`), a string in fastai call syntax such as
    "FocalLossFlat(axis=1, gamma=3)" or "DiceLoss(square_in_union=True)", or a CrossEntropyLossFlat / FocalLossFlat /
    DiceLoss object (see `losses.parse_loss_func`).  FocalLossFlat takes `class_weights` as its weight; DiceLoss has
    none.  The regression variant trains with MSELossFlat only."""
    spec = parse_loss_func(loss_func)
    if spec is None:
        warnings.warn(f"loss_func {type(loss_func).__name__} is not supported: the plan trains with "
                      "CrossEntropyLossFlat(axis=1) with class weights (MSELossFlat(axis=1) for regression)")
        spec = LossSpec()
    if not regression:
        warn_dice_weights(spec, class_weights)
    learn = Learner(_arch_name(arch), n_in, n_classes, size, batch_size, class_weights, opt_func, lr, wd,
                    encoder_factor, moms, self_attention=self_attention, regression=regression,
                    input_dtype=input_dtype, sixteen_bit=sixteen_bit, loss_spec=spec)
    if isinstance(pretrained, dict):
        learn.load_state_dict(pretrained)
    return learn


_DTYPES = {"uint8": torch.uint8, "uint16": torch.uint16, "int16": torch.int16, "float32": torch.float32}


def load_learner(path, batch_size: Optional[int] = None) -> Learner:
    """predict.py:161 / train.py:225 — loads what `Learner.export` wrote (tensors and plain containers only:
    `weights_only=True`, nothing in the file is executed)."""
    if not os.path.exists(path):
        raise FileNotFoundError(path)
    ck = torch.load(path, map_location="cpu", weights_only=True)
    learn = Learner(ck["arch"], ck["n_in"], ck["n_classes"], tuple(ck["size"]), batch_size or ck["batch_size"],
                    ck.get("class_weights"), self_attention=ck.get("self_attention", False),
                    regression=ck.get("regression", False), sixteen_bit=ck.get("sixteen_bit", False),
                    input_dtype=_DTYPES[ck.get("input_dtype", "uint8")],
                    loss_spec=LossSpec.from_dict(ck.get("loss_func")))
    learn.load_state_dict(ck["state_dict"])
    return learn


_NP_OK = (np.uint8, np.uint16, np.int16)


def _load_tile(path: Path):
    """(raw [n_in,H,W] tile of uint8 / uint16 / int16, GeoInfo or None).  `.tif` tiles carry their own georeferencing
    (predict.py:206-215); the reference reads any integer dtype as int32 -> float32 (data.py:24)."""
    if path.suffix.lower() in (".tif", ".tiff"):
        arr, geo = read_geotiff(path)
    else:
        arr, geo = np.load(path), None
    if arr.dtype not in _NP_OK:
        raise ValueError(f"{path}: {arr.dtype} tiles are not supported (uint8, uint16 or int16 band values)")
    return arr, geo


def _store(path: Path, arr: np.ndarray, geo: Optional[GeoInfo], nodata, class_zero: bool) -> Path:
    """`store_tif` (predict.py:19-52) for `.tif` tiles; `.npy` otherwise (same class_zero un-shift)."""
    if geo is not None:
        write_geotiff(path, arr, geo, nodata=nodata, class_zero=class_zero)
        return path
    if class_zero and arr.dtype.kind in "ui":
        arr = np.where(arr == 0, 0 if nodata is None else nodata, arr - 1).astype(arr.dtype)
    path = path.with_suffix(".npy")
    np.save(path, arr)
    return path


def _gather_strips(strip: torch.Tensor, width: int, rank: int, world: int) -> Optional[torch.Tensor]:
    """[Y, w] or [Y, w, bands] column strips of every rank -> the full-width array on rank 0
    (predict_engine.gather_mask_strips)."""
    if strip.dim() == 2:
        return gather_mask_strips(strip, width, rank, world)
    parts = [gather_mask_strips(strip[:, :, k].contiguous(), width, rank, world) for k in range(strip.shape[2])]
    return None if parts[0] is None else torch.stack(parts, 2)


def save_predictions(predict_model, predict_path, regression: bool = False, merge: bool = False,
                     all_classes: bool = False, specific_class: Optional[int] = None, large_file: bool = False,
                     AOI=None, year=None, validation_vision: bool = False, class_zero: bool = False,
                     geotransforms: Optional[Dict[str, Sequence[float]]] = None):
    """predict.py:146-355 over the tiles in `predict_path`: GeoTIFF tiles (`*.tif`, `[n_in,H,W]` uint8 / uint16 / int16 -
    georeferencing is read from every tile as the reference does) or `.npy` tiles (then `geotransforms[name] = (ulx, xres,
    xskew, uly, yskew, yres)` must be given for `merge`).  Without `merge` one prediction per tile goes to
    `../predicted_tiles_<model>/` (argmax Byte, `specific_class` or `all_classes` probabilities Float32 - or int8 x31
    with `large_file`, predict.py:226-254; `regression`: the raw prediction, Float32); with `merge` the tiles are placed
    by their geotransform with the same python `round()` arithmetic as predict.py:294-297, overlap-averaged and
    arg-maxed on the device, and ONE `<AOI>_<year>_<model>_prediction.tif` is written next to the tile folder
    (`all_classes` / `specific_class` write the averaged probabilities instead; `large_file` uses the int8 x31 /
    floor-division merge; `regression` the mean prediction with nodata -9999, predict.py:307-316).
    Under `torch.distributed` the tiles are sharded over the ranks: per-tile outputs round-robin, the merge as
    owner-computes column strips of the mosaic gathered on rank 0 (no other collective).  Returns the output path(s).
    `validation_vision`: every tile's prediction is compared on the device with its mask tile (`_mask_path`), and rank 0
    writes `<AOI>_<year>_<model>_validation*` next to the outputs: the confusion report (`assessment.write_report`), or
    for `regression` the error statistics against the float32 mask values, the mask tile's no-data skipped
    (`assessment.write_regression_report`)."""
    learn = predict_model if isinstance(predict_model, Learner) else load_learner(predict_model)
    if bool(regression) != learn.regression:
        raise ValueError(f"regression={regression} but the model was trained with regression={learn.regression}")
    assess = bool(validation_vision)
    path = Path(predict_path)
    model_name = "model" if isinstance(predict_model, Learner) else os.path.basename(str(predict_model)).split(".")[0]
    tiles = sorted(path.glob("*.tif")) or sorted(path.glob("*.npy"))
    if not tiles:
        raise FileNotFoundError(f"no .tif / .npy tiles in {path}")
    masks = {t: _mask_path(t) for t in tiles} if assess else {}
    rank, world = _rank(), _world()
    out_dir = path.parent if merge else path.parent / ("predicted_tiles_" + model_name)
    if rank == 0:
        out_dir.mkdir(parents=True, exist_ok=True)
    _barrier()
    net = learn._eval_net()
    pred = TiledPredictor(net)
    B, P = net.N, net.H
    dev, lib = net.device, net.lib

    def batches(sel_tiles, counted=None):
        """(b0, tiles, georeferencing, staged tiles [B, n_in, P, P], staged labels [B, P, P], n_labels): with `counted`
        (one flag per tile of `sel_tiles`) the labels of the flagged tiles of the batch fill the first n_labels slots"""
        stage = ystage = None
        for b0 in range(0, len(sel_tiles), B):
            chunk = sel_tiles[b0:b0 + B]
            loaded = [_load_tile(t) for t in chunk]
            arr = np.stack([a for a, _ in loaded])
            if tuple(arr.shape[1:]) != (net.n_in, P, P):
                raise ValueError(f"tiles must be [{net.n_in},{P},{P}], got {tuple(arr.shape[1:])}")
            ys = [] if counted is None else [_load_labels(masks[t], net.n_out, P, regression)
                                             for t, k in zip(chunk, counted[b0:b0 + B]) if k]
            if stage is None or stage.dtype != torch.from_numpy(arr[:0]).dtype:
                stage = torch.empty((B,) + arr.shape[1:], dtype=torch.from_numpy(arr[:0]).dtype).pin_memory()
            if counted is not None and ystage is None:
                ystage = torch.empty((B, P, P), dtype=ydtype).pin_memory()
            torch.cuda.current_stream().synchronize()      # the previous batch's H2D copies have left the staging buffers
            stage[:len(chunk)] = torch.from_numpy(arr)
            if len(chunk) < B:
                stage[len(chunk):] = stage[:1]
            if ys:
                ystage[:len(ys)] = torch.from_numpy(np.stack(ys))
            yield b0, chunk, [g for _, g in loaded], stage, ystage, len(ys)

    ydtype = torch.float32 if regression else torch.uint8
    if assess:
        y_dev = torch.empty((B, P, P), dtype=ydtype, device=dev)

    if merge:
        # ---- pass 1 over the headers: extent of the mosaic (predict.py:257-276)
        geos: List[Optional[GeoInfo]] = []
        gts = []
        for t in tiles:
            if t.suffix.lower() in (".tif", ".tiff"):
                nb, h, w, _, g = geotiff_info(t)
                geos.append(g)
                gt = g.geotransform
            else:
                if geotransforms is None:
                    raise ValueError("merge=True over .npy tiles needs the tiles' geotransforms")
                geos.append(None)
                gt, h, w = geotransforms[t.name], P, P
            gts.append([gt[0], w, gt[1], gt[3], h, gt[5]])
        gts = np.array(gts, dtype=np.float64)
        if geos[0] is not None and any(not geos[0].same_projection(g) for g in geos[1:]):
            warnings.warn("Geoprojection is not the same for all prediction tiles.")          # predict.py:211-212
        if len(set(gts[:, 1])) != 1 or len(set(gts[:, 4])) != 1:
            warnings.warn("Not all tiles have the same resolution.")                           # predict.py:272-273
        ulx_full, uly_full = gts[:, 0].min(), gts[:, 3].max()
        xmax_r, ymin_r = int(np.argmax(gts[:, 0])), int(np.argmin(gts[:, 3]))
        x_len = round((gts[:, 0].max() + gts[xmax_r, 1] * gts[xmax_r, 2] - ulx_full) / gts[0, 2])
        y_len = round((gts[:, 3].min() + gts[ymin_r, 4] * gts[ymin_r, 5] - uly_full) / gts[0, 5])
        wins = [(x0, y0, P, P) for x0, y0, _, _ in
                (placement_from_geotransform(g[0], P, g[2], g[3], P, g[5], ulx_full, uly_full) for g in gts)]
        # owner-computes column strip of this rank (the whole mosaic on one GPU): every tile that intersects it; the
        # rank owning a tile's left edge assesses it
        mine, xb, xe = shard_windows_by_columns(wins, x_len, rank, world)
        own = column_owned(wins, mine, xb, xe)
        if assess:
            # the tiles each rank owns, in its batch order
            owned = []
            for r in range(world):
                mine_r, xb_r, xe_r = shard_windows_by_columns(wins, x_len, r, world)
                owned.append([tiles[i].name for i, o in zip(mine_r, column_owned(wins, mine_r, xb_r, xe_r)) if o])
            n_own = max(len(o) for o in owned)
            if regression:
                counter = RegressionCounter(dev, n_own, rank, world)
            else:
                counter = ConfusionCounter(net.n_out, dev, n_own, rank, world)
                amax_dev = torch.empty((B, P, P), dtype=torch.uint8, device=dev)
        plan = StitchPlan(net, wins, [mine[b0:b0 + B] for b0 in range(0, len(mine), B)], (0, y_len, xb, xe),
                          2 if regression else 1 if large_file else 0)
        s_ = ops.stream_ptr()
        for b, (b0, chunk, _, x, ys, ny) in enumerate(batches([tiles[i] for i in mine], own if assess else None)):
            plan.load(b)
            net.set_input(x.to(dev, non_blocking=True))
            net.forward()
            plan.accumulate(s_)
            if ny and regression:
                # the per-tile raw prediction (what predict_tiles_raw returns) of each tile this rank owns
                vals = net.logits_nchw()[:, 0]
                y_dev[:ny].copy_(ys[:ny], non_blocking=True)
                k = 0
                for i0, i1 in _runs(own[b0:b0 + len(chunk)]):
                    counter.count(vals[i0:i1], y_dev[k:k + i1 - i0], per_tile=True)
                    k += i1 - i0
            elif ny:
                # the per-tile argmax (what predict_tiles returns) of the tiles this rank owns, packed in batch order
                k, ld = 0, net.logits.shape[-1]
                for i0, i1 in _runs(own[b0:b0 + len(chunk)]):
                    _lib.check(lib.b2u_softmax_nchw(net.logits.data_ptr() + 4 * i0 * P * P * ld, ld, net.n_out, i1 - i0,
                                                    P, P, None, amax_dev.data_ptr() + k * P * P, s_), "b2u_softmax_nchw")
                    k += i1 - i0
                y_dev[:ny].copy_(ys[:ny], non_blocking=True)
                counter.count(amax_dev[:ny], y_dev[:ny], per_tile=True)
        if assess and regression:
            _write_regression_validation(counter, owned, world, rank, out_dir, AOI, year, model_name)
        elif assess:
            _write_validation(counter, world, rank, out_dir, AOI, year, model_name, class_zero)
        nodata = None
        if regression:
            strip, nodata = plan.mean(-9999, s_)[0], -9999                                   # predict.py:313-316
        elif all_classes or specific_class is not None:
            # [y_len, xe - xb, bands], float32 or with `large_file` the int8 merge (predict.py:318-326)
            c0, nc = (0, net.n_out) if all_classes else (range(net.n_out)[specific_class], 1)     # python indexing
            strip = finalize_probs(plan.acc, plan.cnt, c0, nc, 0, plan.SX, large_file, s_)
        else:
            strip = plan.mask(s_)
        full = _gather_strips(strip, x_len, rank, world) if world > 1 else strip
        if rank != 0:
            return None
        out = full.cpu().numpy()
        if out.ndim == 3:
            # [bands, Y, X] (one band: [Y, X]) as a view: write_geotiff stores it without a transposing copy
            out = np.moveaxis(out, 2, 0) if all_classes else out[:, :, 0]
        name = "_".join([p_ for p_ in (AOI, year, model_name, "prediction") if p_])
        geo = None
        if geos[0] is not None:
            g0 = geos[0]
            geo = GeoInfo((float(ulx_full), float(gts[0, 2]), 0.0, float(uly_full), 0.0, float(gts[0, 5])), g0.geokeys,
                          g0.geodoubles, g0.geoascii, None, True)                                # predict.py:350-352
        return _store(out_dir / (name + ".tif"), out, geo, nodata, class_zero)

    outs = []
    sel = tiles[rank::world]
    if assess and regression:
        counter = RegressionCounter(dev, -(-len(tiles) // world), rank, world)
    elif assess:
        counter = ConfusionCounter(net.n_out, dev, -(-len(tiles) // world), rank, world)
    for b0, chunk, geos, x, ys, ny in batches(sel, [True] * len(sel) if assess else None):
        xd = x.to(dev, non_blocking=True)
        if regression:
            vals = pred.predict_tiles_raw(xd)
            if assess:                                          # the real tiles of a padded last batch
                y_dev[:ny].copy_(ys[:ny], non_blocking=True)
                counter.count(vals[:ny, 0], y_dev[:ny], per_tile=True)
            vals = vals.cpu().numpy()
        else:
            probs, amax = pred.predict_tiles(xd)
            if assess:                                          # the real tiles of a padded last batch
                y_dev[:ny].copy_(ys[:ny], non_blocking=True)
                counter.count(amax[:ny], y_dev[:ny], per_tile=True)
            probs, amax = probs.cpu().numpy(), amax.cpu().numpy()
        for i, t in enumerate(chunk):
            if regression:
                arr = vals[i]                                           # predict.py:226-227: stored as is (Float32)
            elif all_classes:
                arr = probs[i]
            elif specific_class is None:
                arr = amax[i]                                           # decoded argmax (predict.py:232)
            else:
                arr = probs[i][specific_class]
            if large_file and not regression and (all_classes or specific_class):   # predict.py:245-249 (sic: class 0 is falsy there)
                arr = np.around(arr * ((128 / 4) - 1)).astype(np.int8)
            outs.append(_store(out_dir / t.name, arr, geos[i], None, class_zero))
    if assess and regression:
        _write_regression_validation(counter, [[t.name for t in tiles[r::world]] for r in range(world)], world, rank,
                                     out_dir, AOI, year, model_name)
    elif assess:
        _write_validation(counter, world, rank, out_dir, AOI, year, model_name, class_zero)
    return outs


def _mask_path(tile: Path) -> Path:
    """`open_mask`'s rule (utils.py:51-55): the mask tile of an image tile is the file of the same name with `img_tiles`
    replaced by `mask_tiles` in its path (a `.npy` tile has a `.npy` mask)"""
    m = Path(str(tile).replace("img_tiles", "mask_tiles"))
    if m == tile:
        raise FileNotFoundError(f"{tile}: validation_vision needs the tiles in an img_tiles folder with a mask_tiles sibling")
    if not m.exists():
        raise FileNotFoundError(f"mask tile {m} of {tile} is missing")
    return m


def _load_labels(path: Path, n_classes: int, P: int, regression: bool = False) -> np.ndarray:
    """band 1 of a mask tile as uint8 class ids below `n_classes` (the labels training reads, `_label_values`); for the
    regression variant the float32 targets, NaN (skipped by the assessment) where the tile declares its no-data value"""
    nodata = None
    if path.suffix.lower() in (".tif", ".tiff"):
        y, geo = read_geotiff(path)
        nodata = geo.nodata
    else:
        y = np.load(path)
    y = y[0] if y.ndim == 3 else y
    if y.shape != (P, P):
        raise ValueError(f"{path}: mask tile of shape {y.shape}, expected ({P}, {P})")
    if not regression:
        return _label_values(y, n_classes, False, path)
    t = _label_values(y, n_classes, True, path)
    if nodata is not None:
        t[y == nodata] = np.nan
    return t


def _runs(flags: Sequence[bool]) -> List[Tuple[int, int]]:
    """[i0, i1) ranges of consecutive True flags"""
    out, i0 = [], None
    for i, f in enumerate(list(flags) + [False]):
        if f and i0 is None:
            i0 = i
        elif not f and i0 is not None:
            out.append((i0, i))
            i0 = None
    return out


def _write_validation(counter: ConfusionCounter, world: int, rank: int, out_dir: Path, AOI, year, model_name: str,
                      class_zero: bool) -> None:
    """the counts of all ranks summed; rank 0 writes `<AOI>_<year>_<model>_validation{.json,_confusion.csv,
    _tile_confusion.csv}`"""
    cm, skipped, hist = counter.read(all_reduce=world > 1)
    if rank == 0:
        name = "_".join([str(p_) for p_ in (AOI, year, model_name, "validation") if p_])
        write_report(out_dir, name, cm, skipped, hist, class_zero)


def _write_regression_validation(counter: RegressionCounter, names: Sequence[Sequence[str]], world: int, rank: int,
                                 out_dir: Path, AOI, year, model_name: str) -> None:
    """the moments of all ranks merged in rank order (`names[r]`: the tiles rank r counted, in its slot order); rank 0
    writes `<AOI>_<year>_<model>_validation{.json,_tile_metrics.csv}` with the tile rows sorted by name"""
    totals, skipped, recs = counter.read(all_reduce=world > 1)
    if rank == 0:
        rows = sorted(((n, recs[r][j]) for r in range(world) for j, n in enumerate(names[r])), key=lambda e: e[0])
        name = "_".join([str(p_) for p_ in (AOI, year, model_name, "validation") if p_])
        write_regression_report(out_dir, name, totals, skipped, [m for _, m in rows], [n for n, _ in rows])


def predict_geotiff(predict_model, raster_path, out_path=None, patch_overlap: float = 0.125, large_file: bool = False,
                    class_zero: bool = False, rank: int = 0, world: int = 1, max_strip_columns: Optional[int] = None,
                    mask_path=None, all_classes: bool = False, specific_class: Optional[int] = None):
    """Tile-free variant of the predict path: what `split_raster` (create_tiles_unet.py:252-431) + `save_predictions(merge=
    True)` produce together - the stitched argmax mask of a whole multi-band GeoTIFF (uint8 / uint16 / int16 bands) -
    without writing tiles to disk: the raster is windowed on the device with `compute_windows` offsets, predicted and
    stitched in HBM.
    `max_strip_columns`: rasters that should not sit in host / device memory at once are streamed as vertical strips of
    at most that many output columns - each strip reads only the file window of the tile columns it needs
    (`read_geotiff(window=)`), is predicted as an owner-computes strip and lands in its columns of the mask, so the
    result is bit-identical to the one-shot prediction.  With `world > 1` every rank writes the column strip it owns
    (`<out>.part<rank>.tif`, georeferenced to its origin).
    `mask_path`: a reference mask on the raster's grid.  Each strip's stitched mask is then compared, on the device, with
    the labels `prepare_raster` makes of the mask (class_zero shift, no-data of image or mask -> 0; a label >= the number
    of classes raises ValueError) over the columns the strip owns, and the accuracy report of the rank's columns goes next
    to the mask as `<out stem>_assessment{.json,_confusion.csv}` (`assessment.write_report`).  The written mask and the
    return value do not change.
    A regression model (`enable_regression`) writes what `save_predictions(regression=True, merge=True)` writes: the
    overlap mean of its output as a Float32 GeoTIFF with nodata -9999 (`large_file` has no effect).  With `mask_path`
    its error statistics against the mask values (the same window read, grid check and class_zero shift) go to
    `<out stem>_assessment.json` (`assessment.write_regression_report`); pixels that are no-data in the image or the
    mask are skipped and counted, not zeroed.
    `all_classes` / `specific_class=k`: the averaged class probabilities instead of the mask, as `save_predictions(merge=
    True)` writes them over the tiles of the same raster with the same flags - all `n_out` bands, or band k alone
    (`all_classes` wins if both are given); Float32, or with `large_file` the reference's int8 x31 merge; no nodata tag;
    `class_zero` applied by `write_geotiff` as for the mask.  Each strip's accumulators are finalized on the device
    straight into the file's pixel-interleaved sample order.  With `mask_path` the assessment still counts the stitched
    argmax of the same prediction pass.  The output is held in host memory until it is written: Y * X * bands * 4 bytes
    for Float32 (1 byte per sample for int8), plus the strips `write_geotiff` builds while writing.  A `specific_class`
    outside [0, n_out) raises ValueError before anything is predicted.  A regression model ignores both flags, as
    `save_predictions` does."""
    from .create_tiles import check_same_grid, mask_labels, mask_tile_values
    learn = predict_model if isinstance(predict_model, Learner) else load_learner(predict_model)
    regression = learn.regression
    net = learn._eval_net()
    probs = not regression and (all_classes or specific_class is not None)
    if probs and not all_classes and not 0 <= specific_class < net.n_out:
        raise ValueError(f"specific_class={specific_class} outside the model's {net.n_out} classes")
    bands, Y, X, dt, geo = geotiff_info(raster_path)
    if dt not in _NP_OK:
        raise ValueError(f"{raster_path}: {dt} rasters are not supported (uint8, uint16 or int16 band values)")
    if bands != net.n_in:
        raise ValueError(f"raster has {bands} bands, the model expects {net.n_in}")
    P = net.H
    pred = TiledPredictor(net)
    windows = compute_windows(Y, X, P, patch_overlap)
    _, xb, xe = shard_windows_by_columns(windows, X, rank, world)
    n_strips = 1 if not max_strip_columns else max(1, -(-(xe - xb) // int(max_strip_columns)))
    if probs:
        c0, nc = (0, net.n_out) if all_classes else (specific_class, 1)
        mask = np.empty((Y, xe - xb, nc), dtype=np.int8 if large_file else np.float32)
    else:
        mask = np.empty((Y, xe - xb), dtype=np.float32 if regression else np.uint8)
    counter = None
    if mask_path is not None:
        _, mY, mX, _, mgeo = geotiff_info(mask_path)
        check_same_grid(geo, mgeo, (Y, X), (mY, mX))
        counter = RegressionCounter(net.device, pred_nodata=-9999) if regression else ConfusionCounter(net.n_out, net.device)
    for k in range(n_strips):
        # strip k of this rank's columns: the balanced partition of [xb, xe), then the tile columns intersecting it
        sb, se = (xb + v for v in split_range(xe - xb, n_strips, k))
        idx = [i for i, (x, y, w, h) in enumerate(windows) if x < se and x + w > sb]
        xs0 = min(windows[i][0] for i in idx)
        xs1 = max(windows[i][0] + windows[i][2] for i in idx)
        strip, _ = read_geotiff(raster_path, window=(xs0, 0, xs1 - xs0, Y))
        dev_s = torch.from_numpy(np.ascontiguousarray(strip)).pin_memory().to(net.device, non_blocking=True)
        # the strip holds exactly the tile columns of [sb, se): a one-rank prediction of it reproduces those tiles
        m, _, _, acc, cnt = pred.predict_raster(dev_s, patch_overlap, 0, 1, return_probs=True, large_file=large_file)
        if counter is not None:
            # the truth of the same window, laid out like `m` so that both rows sit at the same 16-byte offset
            truth, _ = read_geotiff(mask_path, window=(xs0, 0, xs1 - xs0, Y))
            truth, bad = mask_labels(strip, geo.nodata, truth, mgeo.nodata, class_zero)
            truth = _label_values(mask_tile_values(truth[0]), net.n_out, regression, mask_path)
            if regression:
                truth[bad] = np.nan                 # 0 is a real value of a continuous target: skip, do not zero
            truth_d = torch.from_numpy(np.ascontiguousarray(truth)).pin_memory().to(net.device, non_blocking=True)
            counter.count(m[:, sb - xs0:se - xs0], truth_d[:, sb - xs0:se - xs0])
        if probs:
            mask[:, sb - xb:se - xb] = finalize_probs(acc, cnt, c0, nc, sb - xs0, se - sb, large_file,
                                                      ops.stream_ptr()).cpu().numpy()
        else:
            mask[:, sb - xb:se - xb] = m[:, sb - xs0:se - xs0].cpu().numpy()
    out_path = Path(out_path) if out_path is not None else Path(raster_path).with_name(Path(raster_path).stem + "_prediction.tif")
    if world > 1:
        out_path = out_path.with_suffix(f".part{rank}.tif")
    # [Y, X, bands] as the [bands, Y, X] view whose transpose write_geotiff stores without a copy
    write_geotiff(out_path, np.moveaxis(mask, 2, 0) if probs else mask, geo.window(xb, 0),
                  nodata=-9999 if regression else None, class_zero=class_zero)
    if counter is not None:
        extra = {"raster": str(raster_path), "mask": str(mask_path), "prediction": str(out_path), "columns": [xb, xe]}
        if regression:
            totals, skipped, _ = counter.read()
            write_regression_report(Path(mask_path).parent, out_path.stem + "_assessment", totals, skipped, extra=extra)
        else:
            cm, skipped, _ = counter.read()
            write_report(Path(mask_path).parent, out_path.stem + "_assessment", cm, skipped, None, class_zero, extra=extra)
    return out_path


# ---------------------------------------------------------------------------------------------------- training entry
def get_datatype(files: Sequence[Path]) -> str:
    """utils.py:72-89: the dataset kind is read off the FIRST training tile - 'int8' when its largest value (ignoring
    nodata pixels of band 1) is below 257, else 'int16' - and decides whether the batch transform divides by 255."""
    arr, geo = read_geotiff(files[0])
    return _dataset_kind(arr, getattr(geo, "nodata", None))


def _dataset_kind(tile: np.ndarray, nodata) -> str:
    """`get_datatype` on the values of a `[bands, H, W]` tile"""
    keep = np.ones(tile.shape[1:], dtype=bool) if nodata is None else tile[0] != nodata
    vals = tile[:, keep]
    return "int8" if (vals.size == 0 or vals.max() < 257) else "int16"


class _BatchDeal:
    """The batch sequence of one epoch over `n_items` samples (data.py:100-105 DataLoader semantics): a shuffle seeded
    with `shuffle_seed + epoch` (None: file order), `drop_last`, and with `drop_last=False` a last partial batch padded
    by repeating its first sample (`n_real` tells how many samples count).  Data parallel: the global batch sequence is
    dealt round-robin, rank r takes batches r, r + world, ... and every rank sees the same number of batches (the
    gradient all-reduce needs equal step counts)."""

    def __init__(self, n_items: int, batch_size: int, shuffle_seed: Optional[int], drop_last: bool, rank: int = 0,
                 world: int = 1):
        self.n_items, self.batch_size, self.shuffle_seed, self.rank, self.world = n_items, batch_size, shuffle_seed, rank, world
        n_global = n_items // batch_size if drop_last else -(-n_items // batch_size)
        self.n_batches = n_global // world if world > 1 else n_global

    def __call__(self, epoch: int) -> List[Tuple[List[int], int]]:
        """[(sample indices of the batch, n_real)] of this rank in `epoch`"""
        order = list(range(self.n_items))
        if self.shuffle_seed is not None:
            np.random.default_rng(self.shuffle_seed + epoch).shuffle(order)      # the same order on every rank
        out = []
        for k in range(self.n_batches):
            b0 = (k * self.world + self.rank) * self.batch_size
            idx = order[b0:b0 + self.batch_size]
            n_real = len(idx)
            if n_real < self.batch_size:
                idx = idx + [idx[0]] * (self.batch_size - n_real)
            out.append((idx, n_real))
        return out


def _tile_batches(files: Sequence[Path], batch_size: int, n_classes: int, class_zero: bool, shuffle_seed: Optional[int],
                  drop_last: bool, regression: bool = False, rank: int = 0, world: int = 1):
    """Batches of (raw tiles [B,n_in,H,W], labels [B,H,W], n_real) from `img_tiles/*.tif` + `mask_tiles/*.tif`
    (data.py:100-105, utils.py:40-55) in the order `_BatchDeal` deals them: labels are uint8 class ids, or the float32
    mask band for the regression variant (RegressionBlock)."""
    deal = _BatchDeal(len(files), batch_size, shuffle_seed, drop_last, rank, world)

    def gen():
        epoch = gen.epoch
        if shuffle_seed is not None:
            gen.epoch += 1
        for idx, n_real in deal(epoch):
            xs, ys = [], []
            for i in idx:
                x = open_tile(files[i])
                if x.dtype not in _NP_OK:
                    raise ValueError(f"{files[i]}: {x.dtype} tiles are not supported (uint8, uint16 or int16 band values)")
                xs.append(x)
                ys.append(_label_values(open_mask(files[i]), n_classes, regression, files[i]))
            yield torch.from_numpy(np.stack(xs)), torch.from_numpy(np.stack(ys)), n_real
    gen.epoch = 0
    gen.n_batches = deal.n_batches   # known without touching the files (fit_one_cycle sizes its schedule with it)
    return gen


def _label_values(y: np.ndarray, n_classes: int, regression: bool, where) -> np.ndarray:
    """mask tile values -> training labels: float32 targets (regression) or uint8 class ids below `n_classes`"""
    if regression:
        return y.astype(np.float32)
    if y.max() >= n_classes:
        raise ValueError(f"{where}: mask label {int(y.max())} >= number of classes {n_classes}")
    return y.astype(np.uint8)


def _class_weights(CLASS_WEIGHTS, n_classes: int, regression: bool, train_masks: Iterable[np.ndarray]) -> List[float]:
    """train.py:330-339: the loss weights.  `train_masks` (the mask tiles of the first 1200 training samples, read only
    for "weighted") feed utils.py:105-117 get_class_weights: total / count per class.  The reference takes the counts
    from `unique()`, which silently drops absent classes; here an absent class keeps its slot (count clamped to 1).  The
    weighted-mean CE is invariant to the common scale."""
    if regression:
        return [1.0]                                                               # train.py:330-331
    if isinstance(CLASS_WEIGHTS, str):
        if CLASS_WEIGHTS == "even":
            return [1.0 / n_classes] * n_classes                                   # train.py:338-339
        if CLASS_WEIGHTS == "weighted":
            counts = np.zeros(n_classes, dtype=np.float64)
            for m in train_masks:
                counts += np.bincount(m.ravel(), minlength=n_classes)[:n_classes]
            # plain floats: the exported checkpoint must load with weights_only=True (no numpy scalars)
            return [float(v) for v in counts.sum() / np.maximum(counts, 1.0)]
        raise ValueError(f"CLASS_WEIGHTS {CLASS_WEIGHTS!r} not understood")
    return list(CLASS_WEIGHTS)


def train_func(data_path, existing_model, model_Path, description, BATCH_SIZE, visualize_data_example=False,
               enable_regression=False, CLASS_WEIGHTS="even", ARCHITECTURE="xresnet34", EPOCHS=1, LEARNING_RATE=1e-3,
               ENCODER_FACTOR=10, LR_FINDER=None, loss_func=None, monitor=None, self_attention=False,
               VALID_SCENES=("vali",), CODES=("background", "class1"), transforms=False, split_idx=None,
               export_model_summary=False, aug_pipe=None, n_transform_imgs=0, info=False, class_zero=False):
    """`train_func` (train.py:287-375) with the reference's positional signature, on the B200 plan.  Expects
    `data_path/{trai,vali}/{img_tiles,mask_tiles}/*.tif` (utils.py:25-36, data.py:102-105); trains with fastai's recipe
    (Adam, wd 0.01, discriminative lrs `slice(lr/ENCODER_FACTOR, lr)`, one-cycle) and writes
    `<model_Path>/<description>/<description>.pkl`, `.json` and `_history.csv` (train.py:314-320, 234, 255).
    `enable_regression`: n_out 1, MSELossFlat, rmse / R2Score, monitor r2_score (train.py:189-201).  `loss_func` picks
    the classification loss as `unet_learner_MS` describes; it is recorded in `<description>.json`.  8- and 16-bit tiles
    follow the reference's input contract (`get_datatype`).  `transforms=True` applies the geometric part of the reference's
    augmentation (flips / 90-degree rotations of image and mask together, on the device-bound batch) to the share
    `n_transform_imgs` of every batch; albumentations pipeline objects (`aug_pipe`), the LR finder, plots and the model
    summary are outside the built path and are skipped with a warning.
    Data parallel: launched under `torch.distributed.run` (params_and_main `N_GPUS`), every rank trains on its share of
    the batches, gradients are all-reduced by the trainer, and only rank 0 writes files.  Returns the trained Learner."""
    from .engine import init_distributed
    rank, _, world = init_distributed() if int(os.environ.get("WORLD_SIZE", "1")) > 1 else (0, 0, 1)
    if LR_FINDER:
        warnings.warn("LR_FINDER is outside the built path; training proceeds with LEARNING_RATE")
    if aug_pipe:
        warnings.warn("albumentations pipeline objects are outside the built path; `transforms` applies flips / rot90 only")
    data_path = Path(data_path)
    valid_scenes = [VALID_SCENES] if isinstance(VALID_SCENES, str) else list(VALID_SCENES)
    train_files, valid_files = [], []
    if not data_path.exists():
        raise FileNotFoundError(data_path)                                         # train.py:54
    for scene in sorted(p for p in data_path.iterdir() if p.is_dir()):
        files = sorted((scene / "img_tiles").glob("*.tif"))
        (valid_files if scene.name in valid_scenes else train_files).extend(files)
    if not train_files:
        raise FileNotFoundError(f"no training tiles under {data_path}/*/img_tiles")
    nb, h, w, np_dt, _ = geotiff_info(train_files[0])                              # train.py:124-125 probes the first item
    if np_dt not in _NP_OK:
        raise ValueError(f"{train_files[0]}: {np_dt} tiles are not supported (uint8, uint16 or int16 band values)")
    n_classes = len(CODES)
    regression = bool(enable_regression)
    tb = _tile_batches(train_files, BATCH_SIZE, n_classes, class_zero, shuffle_seed=0,
                       drop_last=len(train_files) >= BATCH_SIZE * world, regression=regression, rank=rank, world=world)
    if transforms:
        tb = augmented(tb, float(n_transform_imgs), seed=0 if split_idx is None else int(split_idx))
    # every rank validates the whole validation set (identical metrics on every rank: no collective, same best epoch)
    vb = _tile_batches(valid_files, BATCH_SIZE, n_classes, class_zero, None, False, regression=regression) if valid_files else None
    return _train_and_export(
        tb, vb, len(train_files), len(valid_files), rank, world, nb, (h, w), np_dt,
        sixteen_bit=get_datatype(train_files) == "int16",                                                    # train.py:298
        class_weights=_class_weights(CLASS_WEIGHTS, n_classes, regression, (open_mask(f) for f in train_files[:1200])),
        model_Path=model_Path, description=description, BATCH_SIZE=BATCH_SIZE, existing_model=existing_model,
        enable_regression=regression, ARCHITECTURE=ARCHITECTURE, EPOCHS=EPOCHS, LEARNING_RATE=LEARNING_RATE,
        ENCODER_FACTOR=ENCODER_FACTOR, loss_func=loss_func, monitor=monitor, self_attention=self_attention, CODES=CODES,
        class_zero=class_zero)


def _train_and_export(tb, vb, n_train: int, n_valid: int, rank: int, world: int, nb: int, tile_hw: Tuple[int, int], np_dt,
                      sixteen_bit: bool, class_weights: List[float], *, model_Path, description, BATCH_SIZE,
                      existing_model, enable_regression, ARCHITECTURE, EPOCHS, LEARNING_RATE, ENCODER_FACTOR, loss_func,
                      monitor, self_attention, CODES, class_zero, extra_json: Optional[dict] = None):
    """train.py:287-375 after the data is found: learner, monitor rules, fit, export and the description JSON, over the
    training / validation batch sources `tb` / `vb` (callables as `fit_one_cycle` takes them; `vb` may be None)."""
    import json
    codes = list(CODES)
    n_classes = len(codes)
    regression = bool(enable_regression)
    cw = class_weights
    h, w = tile_hw
    learn = unet_learner_MS(nb, n_classes, ARCHITECTURE, (h, w), BATCH_SIZE, class_weights=cw, lr=LEARNING_RATE,
                            encoder_factor=ENCODER_FACTOR, self_attention=self_attention, regression=regression,
                            input_dtype=torch.from_numpy(np.zeros(0, dtype=np_dt)).dtype, sixteen_bit=sixteen_bit,
                            loss_func=loss_func)
    if existing_model:
        if not os.path.exists(existing_model):
            raise FileNotFoundError(existing_model)
        learn.load_state_dict(torch.load(existing_model, map_location="cpu", weights_only=True)["state_dict"])
    out_dir = Path(model_Path) / description
    if rank == 0:
        out_dir.mkdir(parents=True, exist_ok=True)
    if monitor not in (None, "train_loss", "valid_loss", "r2_score", "dice_multi"):
        raise ValueError("Monitor must be one of ['train_loss', 'valid_loss', 'r2_score', 'dice_multi']")    # train.py:207-208
    mon = monitor or ("r2_score" if regression else "dice_multi")                                             # train.py:198-201
    if vb is None and mon != "train_loss":
        mon = "train_loss"
    _barrier()
    learn.fit_one_cycle(EPOCHS, LEARNING_RATE, tb, vb, history_csv=str(out_dir / f"{description}_history.csv"),
                        monitor=mon, best_path=str(out_dir / "best-model.pth"))
    if rank == 0:
        learn.export(out_dir / f"{description}.pkl")
        with open(out_dir / f"{description}.json", "w") as f:
            json.dump({"description": description, "architecture": learn.arch, "bands": nb, "tile": [h, w], "codes": codes,
                       "class_weights": cw, "batch_size": BATCH_SIZE, "epochs": EPOCHS, "learning_rate": LEARNING_RATE,
                       "encoder_factor": ENCODER_FACTOR, "train_tiles": n_train, "valid_tiles": n_valid,
                       "class_zero": bool(class_zero), "enable_regression": regression, "datatype": "int16" if sixteen_bit else "int8",
                       "n_gpus": world, "loss_func": learn.loss_spec.as_dict(), **(extra_json or {}),
                       "history": learn.history}, f, indent=1)
    _barrier()
    return learn


def train_geotiff(pairs, patch_size: int = 400, patch_overlap: float = 0.20, split: Optional[Sequence[float]] = None,
                  max_empty: float = 0.9, class_zero: bool = False, seed: int = 0, *, model_Path, description,
                  BATCH_SIZE, existing_model=None, enable_regression=False, CLASS_WEIGHTS="even",
                  ARCHITECTURE="xresnet34", EPOCHS=1, LEARNING_RATE=1e-3, ENCODER_FACTOR=10, loss_func=None,
                  monitor=None, self_attention=False, VALID_SCENES=("vali",), CODES=("background", "class1"),
                  transforms=False, split_idx=None, n_transform_imgs=0):
    """Tile-free variant of the training path: what `split_raster(raster, mask, base_dir, patch_size, patch_overlap,
    split, max_empty, class_zero, seed)` for every pair into one `base_dir`, then `train_func(base_dir, ...)` with the
    same training arguments produce - the same weights, history, metrics and exported model - without writing a tile.
    `pairs` is one (raster, mask) pair of GeoTIFF paths or a list of them.  The prepared rasters and labels are uploaded
    once; every batch is cut out of them on the device by `b2u_crop_train_batch`, with the dihedral augmentation of
    `transforms` in the same pass, so no host work on pixels remains per step.  The windows are listed, split and
    ordered exactly as `train_func` would find the tile files (`_raster_windows`).  Rasters must fit in host memory and
    in HBM.  Data parallel under `torch.distributed.run`: every rank uploads the rasters and takes its share of the
    batches; only rank 0 writes.  Returns the trained Learner."""
    from .engine import init_distributed
    share = _aug_share(n_transform_imgs) if transforms else None
    regression = bool(enable_regression)
    n_classes = len(CODES)
    images, labels, train, valid = _raster_windows(pairs, patch_size, patch_overlap, split, max_empty, class_zero, seed,
                                                   VALID_SCENES)
    crop = lambda a, e: a[..., e[2][1]:e[2][1] + patch_size, e[2][0]:e[2][0] + patch_size]
    for e in train + valid:
        _label_values(crop(labels[e[1]], e), n_classes, regression, e[0])       # _tile_batches' check, before training
    rank, _, world = init_distributed() if int(os.environ.get("WORLD_SIZE", "1")) > 1 else (0, 0, 1)
    nb, np_dt = images[0].shape[0], images[0].dtype
    # one device raster for all pairs: pair k occupies rows [yoff[k], yoff[k] + Y_k) and its own columns
    yoff = np.cumsum([0] + [a.shape[1] for a in images])
    Y, X = int(yoff[-1]), max(a.shape[2] for a in images)
    dev = torch.device("cuda", torch.cuda.current_device())
    bits = lambda a: torch.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a)     # uint16 moved as its bits
    pad = any(a.shape[2] != X for a in images)
    alloc = torch.zeros if pad else torch.empty
    img_d = alloc((nb, Y, X), dtype=bits(np.zeros(0, np_dt)).dtype, device=dev)
    lab_d = alloc((Y, X), dtype=torch.float32 if regression else torch.uint8, device=dev)
    for k, (a, lab) in enumerate(zip(images, labels)):
        img_d[:, yoff[k]:yoff[k + 1], :a.shape[2]].copy_(bits(a))
        lab_d[yoff[k]:yoff[k + 1], :a.shape[2]].copy_(torch.from_numpy(lab.astype(np.float32 if regression else np.uint8)))
    yx = lambda es: np.array([(yoff[e[1]] + e[2][1], e[2][0]) for e in es], dtype=np.int32).reshape(-1, 2)
    x_dtype = torch.from_numpy(np.zeros(0, dtype=np_dt)).dtype
    tb = _raster_batches(img_d, lab_d, x_dtype, yx(train), patch_size, BATCH_SIZE,
                         _BatchDeal(len(train), BATCH_SIZE, 0, len(train) >= BATCH_SIZE * world, rank, world),
                         share, 0 if split_idx is None else int(split_idx))
    # every rank validates the whole validation set, as train_func does
    vb = _raster_batches(img_d, lab_d, x_dtype, yx(valid), patch_size, BATCH_SIZE,
                         _BatchDeal(len(valid), BATCH_SIZE, None, False), None, 0) if valid else None
    return _train_and_export(
        tb, vb, len(train), len(valid), rank, world, nb, (patch_size, patch_size), np_dt,
        sixteen_bit=_dataset_kind(crop(images[train[0][1]], train[0]), None) == "int16",
        class_weights=_class_weights(CLASS_WEIGHTS, n_classes, regression, (crop(labels[e[1]], e) for e in train[:1200])),
        model_Path=model_Path, description=description, BATCH_SIZE=BATCH_SIZE, existing_model=existing_model,
        enable_regression=regression, ARCHITECTURE=ARCHITECTURE, EPOCHS=EPOCHS, LEARNING_RATE=LEARNING_RATE,
        ENCODER_FACTOR=ENCODER_FACTOR, loss_func=loss_func, monitor=monitor, self_attention=self_attention, CODES=CODES,
        class_zero=class_zero,
        extra_json={"rasters": [str(r) for r, _ in _as_pairs(pairs)], "masks": [str(m) for _, m in _as_pairs(pairs)],
                    "patch_size": patch_size, "patch_overlap": patch_overlap,
                    "split": None if split is None else list(split), "max_empty": max_empty, "split_seed": seed})


def _as_pairs(pairs) -> List[Tuple]:
    """one (raster, mask) pair or a list of them -> a list of pairs"""
    if isinstance(pairs, (tuple, list)) and len(pairs) == 2 and all(isinstance(q, (str, os.PathLike)) for q in pairs):
        pairs = [pairs]
    return [tuple(q) for q in pairs]


def _raster_windows(pairs, patch_size: int, patch_overlap: float, split, max_empty: float, class_zero: bool, seed: int,
                    VALID_SCENES):
    """The tiles `split_raster` would write for every pair into one directory, in the order `train_func` would read
    them: scenes in sorted order, names sorted inside a scene, every scene not in VALID_SCENES training (`test` of a
    three-way split included).  Returns (prepared images, mask-tile values per pair, training entries, validation
    entries); an entry is (tile name, pair index, window (x, y, w, h))."""
    from .create_tiles import mask_tile_values, prepare_raster, split_names
    pairs = _as_pairs(pairs)
    if not pairs or any(len(q) != 2 or q[1] is None for q in pairs):
        raise ValueError("train_geotiff needs one or more (raster, mask) pairs")
    stems = [os.path.splitext(os.path.basename(str(r)))[0] for r, _ in pairs]
    if len(set(stems)) != len(stems):
        raise ValueError(f"raster names {stems} collide: split_raster would write their tiles over each other")
    valid_scenes = [VALID_SCENES] if isinstance(VALID_SCENES, str) else list(VALID_SCENES)
    images, labels, scenes = [], [], {}
    for k, (raster, mask) in enumerate(pairs):
        prep = prepare_raster(raster, mask, patch_size, patch_overlap, max_empty, class_zero)
        if prep.image.dtype not in _NP_OK:
            raise ValueError(f"{raster}: {prep.image.dtype} rasters are not supported (uint8, uint16 or int16 band values)")
        wins = dict(prep.tiles)
        for scene, names in split_names(list(wins), split, seed).items():
            scenes.setdefault(scene, []).extend((name, k, wins[name]) for name in names)
        images.append(prep.image)
        labels.append(mask_tile_values(prep.mask[0]))
    if len({(a.shape[0], a.dtype) for a in images}) != 1:
        raise ValueError("the rasters differ in band count or sample type")
    train, valid = [], []
    for scene in sorted(scenes):
        (valid if scene in valid_scenes else train).extend(sorted(scenes[scene], key=lambda e: e[0]))
    if not train:
        raise ValueError("no training windows: none was kept, or all of them went to validation scenes")
    return images, labels, train, valid


def _epoch_table(deal: _BatchDeal, epoch: int, yx: np.ndarray, share: Optional[float], aug_seed: int):
    """The crop table of one epoch, int32 [n_batches, (y0, x0, op), B], and the n_real of every batch: the windows of
    `deal(epoch)` and, when `share` is not None, the dihedral ops `augmented` would draw for them, in its order."""
    batches = deal(epoch)
    B = deal.batch_size
    table = np.zeros((max(1, len(batches)), 3, B), dtype=np.int32)
    rng = np.random.default_rng(aug_seed + epoch) if share is not None else None
    for k, (idx, _) in enumerate(batches):
        table[k, :2] = yx[idx].T
        for i, op in (_aug_ops(rng, B, share) if rng is not None else ()):
            table[k, 2, i] = op
    return table, [n for _, n in batches]


_RASTER_DT = {torch.uint8: _lib.DT_U8, torch.uint16: _lib.DT_U16, torch.int16: _lib.DT_I16}


def _raster_batches(img_d: torch.Tensor, lab_d: torch.Tensor, x_dtype: torch.dtype, yx: np.ndarray, P: int, B: int,
                    deal: _BatchDeal, share: Optional[float], aug_seed: int):
    """Device batches of (raw tiles [B,C,P,P], labels [B,P,P], n_real) cut out of the device raster `img_d` [C,Y,X] and
    labels `lab_d` [Y,X] at the window origins `yx` [N, (y0, x0)]: the batches `_tile_batches` (wrapped in `augmented`
    when `share` is not None) yields over the same windows.  An epoch's `_epoch_table` goes to the device in one copy
    and each batch's crop reads its slice of it: no per-step host-to-device copy, no per-step synchronisation.  Batches
    are cut into a ring of two buffers: `fit_one_cycle` takes batch k+1 before it enqueues step k, and stream order
    keeps the buffer of step k intact until the step's input copy has run."""
    lib, dev = _lib.load(), img_d.device
    C, Y, X = img_d.shape
    ring = [(torch.empty((B, C, P, P), dtype=x_dtype, device=dev), torch.empty((B, P, P), dtype=lab_d.dtype, device=dev))
            for _ in range(2)]
    r_dt = _RASTER_DT[x_dtype]
    l_dt = _lib.DT_F32 if lab_d.dtype == torch.float32 else _lib.DT_U8

    def gen():
        epoch = gen.epoch
        gen.epoch += 1
        table, n_real = _epoch_table(deal, epoch, yx, share, aug_seed)
        tab = torch.from_numpy(table).to(dev)
        s = ops.stream_ptr()
        for k, n in enumerate(n_real):
            xb, yb = ring[k % 2]
            t0 = tab.data_ptr() + k * 3 * B * 4
            _lib.check(lib.b2u_crop_train_batch(img_d.data_ptr(), r_dt, C, Y, X, lab_d.data_ptr(), l_dt, t0, t0 + 4 * B,
                                                t0 + 8 * B, B, P, xb.data_ptr(), yb.data_ptr(), s), "b2u_crop_train_batch")
            yield xb, yb, n
    gen.epoch = 0
    gen.n_batches = deal.n_batches
    return gen


def augmented(batches: Callable[[], Iterable], share: float, seed: int = 0):
    """The geometric core of the reference's augmentation (utils.py:196-295 SegmentationAlbumentationsTransform applied to
    `ceil(B * n_transform_imgs)` images of every batch, image and mask together; the reference's default pipelines are
    flips and 90-degree rotations): each selected sample gets one of the eight dihedral transforms (`_aug_ops`).  Pure
    index permutations of the raw integer tiles - no resampling, no value change - executed on the batch before it is
    copied to the device; square tiles only (a 90-degree rotation must keep the shape)."""
    share = _aug_share(share)

    def gen():
        rng = np.random.default_rng(seed + gen.epoch)
        gen.epoch += 1
        for x, y, n in batches():
            if x.shape[-1] == x.shape[-2]:
                ops = _aug_ops(rng, x.shape[0], share)
                if ops:
                    # uint16 tiles are permuted as their int16 bits: torch has no CPU flip / rot90 for uint16
                    dt = x.dtype
                    x, y = (x.view(torch.int16) if dt == torch.uint16 else x).clone(), y.clone()
                    for i, op in ops:
                        xi, yi = x[i], y[i]
                        if op & 4:
                            xi, yi = xi.flip(-1), yi.flip(-1)
                        xi, yi = torch.rot90(xi, op & 3, (-2, -1)), torch.rot90(yi, op & 3, (-2, -1))
                        x[i], y[i] = xi, yi
                    x = x.view(dt)
            yield x, y, n
    gen.epoch = 0
    gen.n_batches = getattr(batches, "n_batches", None)
    return gen


def _aug_share(share) -> float:
    share = float(share)
    if not (0.0 <= share <= 1.0):
        raise ValueError(f"The n_transform_imgs parameter ({share}) must be between 1 and 0.")      # utils.py:236
    return share


def _aug_ops(rng: np.random.Generator, B: int, share: float) -> List[Tuple[int, int]]:
    """The random draws of one augmented batch, in the order they are made: `ceil(B * share)` distinct samples, then one
    dihedral op in [0, 8) for each - bit 2 flips the last axis, then op & 3 quarter turns of torch.rot90(., k, (-2, -1))."""
    k_aug = math.ceil(B * share)
    if not k_aug:
        return []
    return [(int(i), int(rng.integers(0, 8))) for i in rng.choice(B, size=k_aug, replace=False)]
