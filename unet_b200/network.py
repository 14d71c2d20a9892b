"""The xresnet-DynamicUnet as a static plan of libb2u.so launches (forward, backward, loss, optimizer).

This is the B200-native replacement for `learn.model` + `loss.backward()` + `opt.step()` of the reference
(train.py:141-154 model construction, train.py:246-250 fit loop -> fastai Learner._do_one_batch) and for the per-tile
forward of `learn.predict` (predict.py:193).  torch is used for device memory, streams and NCCL only; every FLOP and
every byte moved on the hot path is issued by a kernel in unet_b200/csrc.

Data layout: activations NHWC bf16 with channel pitch padc(C); parameters/gradients fp32 in ONE flat buffer each, in
fastai's state_dict order and torch shapes (so reference weights load and the optimizer / NCCL all-reduce see a
single contiguous range); bf16 GEMM copies of the weights are re-staged from the fp32 masters once per step by one
batched kernel.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import sys
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib, ops
from .losses import LossSpec, dice_blocks_per_sample, launch_loss
from .layout import ConvSpec, NetSpec, ParamLayout, build_spec, conv_flops, shuffle_row_of_co
from .ops import ConvPlan, WgradPlan, padc, view_nhwc

import os

BN_EPS = 1e-5
SIDE_STREAM_WGRAD = os.environ.get("B2U_NO_SIDE_STREAM") is None   # A/B switches for profiling
FUSED_FINAL_SHUFFLE = os.environ.get("B2U_NO_FUSED_SHUFFLE") is None
FUSED_HEAD = os.environ.get("B2U_NO_FUSED_HEAD") is None
STEM_IM2COL = os.environ.get("B2U_NO_STEM_IM2COL") is None      # A/B switch for profiling
BN_MOMENTUM = 0.1
STATS_ROWS = 592  # block partial rows of the standalone reductions (4 per SM)


_RAW_DTYPES = {torch.float32: _lib.DT_F32, torch.uint8: _lib.DT_U8, torch.uint16: _lib.DT_U16, torch.int16: _lib.DT_I16}


def input_contract(dtype: torch.dtype, input_div: Tuple[float, float]) -> Tuple[int, float, float]:
    """(b2u dtype code, div, div2) of the reference's input contract (SURVEY 8(a) row A0): every GeoTIFF dtype is read
    as int32 -> float32 (data.py:24); a dataset whose values exceed 8 bits ('int16', utils.py:72-89) is divided by 255
    inside the reference's batch transform (utils.py:248-249, 288-289) and fastai's IntToFloatTensor divides by 255
    once more (MaskBlock, data.py:100); the regression variant has no IntToFloatTensor (RegressionBlock, data.py:98).
    `input_div` is the plan's (div, div2) for RAW integer tiles; fp32 input is taken as already scaled."""
    if dtype not in _RAW_DTYPES:
        raise TypeError(f"tiles must be float32, uint8, uint16 or int16, got {dtype}")
    if dtype == torch.float32:
        return _lib.DT_F32, 1.0, 1.0
    return _RAW_DTYPES[dtype], float(input_div[0]), float(input_div[1])


def input_divisors(sixteen_bit: bool, regression: bool = False) -> Tuple[float, float]:
    """the (div, div2) pair of a dataset: 8-bit classification 255 / 1, 16-bit classification 255 / 255, regression
    1 / 1 (8-bit) or 255 / 1 (16-bit: only the batch transform's division remains)"""
    if regression:
        return (255.0, 1.0) if sixteen_bit else (1.0, 1.0)
    return (255.0, 255.0) if sixteen_bit else (255.0, 1.0)


class Act:
    """An NHWC bf16 activation and (lazily) its gradient."""

    def __init__(self, N: int, H: int, W: int, Cc: int, dev, name: str = "", zero: bool = False):
        self.N, self.H, self.W, self.C, self.ld = N, H, W, Cc, padc(Cc)
        alloc = torch.zeros if (zero or self.ld != Cc) else torch.empty
        self.t = alloc((N, H, W, self.ld), dtype=torch.bfloat16, device=dev)
        self.name = name
        self.grad: Optional[torch.Tensor] = None
        self.grad_written = False
        self.pre_relu_grad = False  # decoder tensors: the producer of the gradient applies the (t > 0) ReLU mask

    @property
    def pixels(self) -> int:
        return self.N * self.H * self.W

    def ensure_grad(self) -> torch.Tensor:
        if self.grad is None:
            self.grad = torch.zeros_like(self.t)
        return self.grad


class BNState:
    def __init__(self, net: "UNetB200", prefix: str, Cc: int):
        dev = net.device
        self.C = Cc
        self.gamma = net.param(prefix + ".weight")
        self.beta = net.param(prefix + ".bias")
        self.dgamma = net.grad(prefix + ".weight")
        self.dbeta = net.grad(prefix + ".bias")
        self.running_mean = net.buffers[prefix + ".running_mean"]
        self.running_var = net.buffers[prefix + ".running_var"]
        f = lambda: torch.zeros(ops.pad32(Cc), dtype=torch.float32, device=dev)  # conv epilogue reads whole 32-float groups
        self.mean, self.invstd, self.scale, self.shift = f(), f(), f(), f()
        self.mean_g, self.mean_gx = f(), f()


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


class UNetB200:
    """Static launch plan for one (arch, n_in, n_out, H, W, batch) configuration."""

    def __init__(self, arch: str = "xresnet34", n_in: int = 4, n_out: int = 2, size: Tuple[int, int] = (256, 256),
                 batch: int = 8, training: bool = True, device: Optional[torch.device] = None,
                 class_weights: Optional[Sequence[float]] = None, self_attention: bool = False,
                 input_div: Tuple[float, float] = (255.0, 1.0), regression: bool = False,
                 loss_spec: Optional[LossSpec] = None):
        if not torch.cuda.is_available():
            raise _lib.B2UError("UNetB200 needs a CUDA device (sm_100a); there is no CPU path")
        self.lib = _lib.load()
        _lib.check(self.lib.b2u_device_check(), "b2u_device_check")
        self.device = device or torch.device("cuda", torch.cuda.current_device())
        self.self_attention = bool(self_attention)
        self.input_div = (float(input_div[0]), float(input_div[1]))
        self.regression = bool(regression)
        if self.regression and n_out != 1:
            raise ValueError("the regression variant has n_out = 1 (train.py:137-138)")
        # the training loss (losses.LossSpec): cross-entropy by default, MSE for regression, focal or Dice on request
        self.loss_spec = loss_spec or LossSpec()
        if self.regression and self.loss_spec.name != "ce":
            raise ValueError(f"the regression variant trains with MSELossFlat only, not the {self.loss_spec.name} loss")
        self.spec: NetSpec = build_spec(arch, n_in, n_out, self.self_attention)
        self.layout = ParamLayout(self.spec)
        self.N, (self.H, self.W) = batch, size
        if self.H < 32 or self.W < 32:
            raise ValueError("tile height/width must be at least 32 (five stride-2 stages)")
        # any size works: odd extents halve upwards in the encoder, and where the upsampled size exceeds an odd skip by one
        # the decoder crops (== fastai's F.interpolate(up_out, skip.shape[-2:], mode='nearest'), unet.py UnetBlock.forward;
        # the reference's default 400-px tiles reach 25 -> 13 -> 26 vs 25)
        self.training = training
        self.n_in, self.n_out = n_in, n_out
        dev = self.device
        self.params = torch.zeros(self.layout.total, dtype=torch.float32, device=dev)
        self.grads = torch.zeros(self.layout.total, dtype=torch.float32, device=dev) if training else None
        self.buffers: Dict[str, torch.Tensor] = {}
        for prefix, c in self.layout.buffers:
            self.buffers[prefix + ".running_mean"] = torch.zeros(c, dtype=torch.float32, device=dev)
            self.buffers[prefix + ".running_var"] = torch.ones(c, dtype=torch.float32, device=dev)
        for prefix, co, ci in self.layout.sn_buffers:      # spectral norm power-iteration vectors (unit norm)
            g = torch.Generator(device=dev).manual_seed(len(self.buffers))
            for key, nvec in ((".weight_u", co), (".weight_v", ci)):
                t = torch.randn(nvec, generator=g, device=dev)
                self.buffers[prefix + key] = t / t.norm().clamp_min(1e-12)
        cw = [1.0 / n_out] * n_out if class_weights is None else list(class_weights)  # "even" weights, train.py:338-339
        self.class_weights = torch.tensor(cw, dtype=torch.float32, device=dev)
        self.flops_fwd_per_tile = conv_flops(self.spec, self.H) if self.H == self.W else None

        self._keep: List[object] = []
        self.acts: List[Act] = []
        self.op_tags: List[Tuple[str, str, int]] = []   # (phase, builder function, source line) per op, for profiling
        self.named_acts: Dict[str, Act] = {}
        self.fwd_ops: List[Callable[[int], None]] = []
        self.bwd_ops: List[Callable[[int], None]] = []
        self.fwd_meta: List[Tuple[str, int]] = []      # (kernel kind, algorithmic bytes) per op, "" for the GEMMs
        self.bwd_meta: List[Tuple[str, int]] = []
        self.bwd_side: List[bool] = []   # weight-gradient launches: independent of the dgrad chain -> second stream
        self._side_stream: Optional[torch.cuda.Stream] = None
        self._bwd_builders: List[Callable[[], None]] = []
        self._wstage: List[_lib.WStageItem] = []
        self._wstage_sa: List[_lib.WStageItem] = []   # spectral-normed weights: re-staged inside every forward (1/sigma)
        self._sn_sigma: Dict[str, torch.Tensor] = {}
        self._wgrad_specs: List[dict] = []
        self.launches_fwd = 0
        self.launches_bwd = 0
        self._w: Dict[str, Dict[str, torch.Tensor]] = {}
        self._bn: Dict[str, BNState] = {}
        self._scratch = torch.zeros(1 << 20, dtype=torch.float32, device=dev)  # finalize scratch (4 MB)
        self._build()

    # ------------------------------------------------------------------------------------------------ parameters
    def param(self, name: str) -> torch.Tensor:
        e = self.layout.by_name[name]
        return self.params[e.offset:e.offset + e.numel].view(e.shape)

    def grad(self, name: str) -> Optional[torch.Tensor]:
        if self.grads is None:
            return None
        e = self.layout.by_name[name]
        return self.grads[e.offset:e.offset + e.numel].view(e.shape)

    def load_state_dict(self, sd: Dict[str, torch.Tensor]) -> None:
        """Accepts a fastai/oracle state_dict (keys `layers.N....`). Missing keys raise."""
        with torch.no_grad():
            for e in self.layout.entries:
                self.param(e.name).copy_(sd[e.name].to(self.device, torch.float32))
            for k, b in self.buffers.items():
                b.copy_(sd[k].to(self.device, torch.float32))
        self.weights_changed()

    def init_parameters(self, seed: int = 0, randomize_bn: bool = True) -> None:
        """Random initialisation on the device (no checkpoint is reachable offline).

        randomize_bn=False is fastai's own start (what `unet_learner_MS` hands to `fit_one_cycle`, train.py:128-144):
        encoder convs kaiming-normal (xresnet init_cnn), the replaced first conv with torch's default Conv2d init
        (train.py:130-135); BatchNorm gamma 1, beta 1e-3, and gamma 0 on the last BatchNorm of every ResBlock convpath
        (NormType.BatchZero: each block starts as the identity); decoder ConvLayers kaiming-uniform with bias
        N(0, 0.01) (ConvLayer / init_linear defaults), PixelShuffle convs ICNR (every 4 consecutive output channels
        share one kernel), middle conv and final ResBlock kaiming-normal with bias 0 (DynamicUnet's apply_init), head
        and the spectral-normed attention convs torch's default conv init, attention gamma 0.
        randomize_bn=True (benchmarks and parity tests) draws kaiming-normal convs and moves every BatchNorm affine
        parameter and running statistic away from its default - with gamma = 0 the conv paths are switched off and
        throughput / parity measurements would be vacuous (SURVEY.md 7)."""
        g = torch.Generator(device=self.device).manual_seed(seed)
        dev = self.device
        zero_bn = set()
        if not randomize_bn:
            for st in self.spec.stages:
                for b in st:
                    zero_bn.add(b.convpath[-1].bn_prefix + ".weight")
        fastai = not randomize_bn
        first = self.spec.stem[0].wname
        zero_bias = {cs.bname for cs in list(self.spec.middle) + list(self.spec.final_res)}
        shuf = {cs.wname for cs in [u.shuf for u in self.spec.unet] + [self.spec.final_shuf]}
        default_init = {first, self.spec.head.wname}
        kaiming_normal_w = {cs.wname for cs in list(self.spec.middle) + list(self.spec.final_res)}
        with torch.no_grad():
            for e in self.layout.entries:
                p = self.param(e.name)
                if len(e.shape) == 4:
                    fan_in = e.shape[1] * e.shape[2] * e.shape[3]
                    decoder = e.group == 2
                    if fastai and e.name in default_init:       # nn.Conv2d default: kaiming_uniform(a=sqrt(5))
                        b = 1.0 / fan_in ** 0.5
                        p.copy_((torch.rand(e.shape, generator=g, device=dev) * 2 - 1) * b)
                    elif fastai and e.name in shuf:             # icnr_init: one kaiming-normal kernel per 4 outputs
                        k = torch.randn((e.shape[0] // 4,) + tuple(e.shape[1:]), generator=g, device=dev) * (2.0 / fan_in) ** 0.5
                        p.copy_(k.repeat_interleave(4, dim=0))
                    elif fastai and decoder and e.name not in kaiming_normal_w:   # ReLU ConvLayer: kaiming_uniform
                        b = (6.0 / fan_in) ** 0.5
                        p.copy_((torch.rand(e.shape, generator=g, device=dev) * 2 - 1) * b)
                    else:
                        p.copy_(torch.randn(e.shape, generator=g, device=dev) * (2.0 / fan_in) ** 0.5)
                elif len(e.shape) == 3:              # spectral-normed Conv1d weight_orig of SelfAttention
                    if fastai:
                        b = 1.0 / e.shape[1] ** 0.5
                        p.copy_((torch.rand(e.shape, generator=g, device=dev) * 2 - 1) * b)
                    else:
                        p.copy_(torch.randn(e.shape, generator=g, device=dev) * (2.0 / e.shape[1]) ** 0.5)
                elif e.name.endswith(".gamma"):      # fastai: 0 (the block starts as the identity)
                    p.fill_(0.5 if randomize_bn else 0.0)
                elif e.name.endswith(".0.bias"):
                    if fastai and e.name not in zero_bias:
                        p.copy_(torch.randn(e.shape, generator=g, device=dev) * 0.01)
                    else:
                        p.zero_()
                elif e.name.endswith(".weight"):   # BN gamma
                    if randomize_bn:
                        p.copy_(torch.rand(e.shape, generator=g, device=dev) + 0.5)
                    else:
                        p.fill_(0.0 if e.name in zero_bn else 1.0)
                else:                              # BN beta
                    if randomize_bn:
                        p.copy_(torch.randn(e.shape, generator=g, device=dev) * 0.1)
                    else:
                        p.fill_(1e-3)
            for k, b in self.buffers.items():
                if k.endswith(("weight_u", "weight_v")):
                    continue
                if k.endswith("running_mean"):
                    b.copy_(torch.randn(b.shape, generator=g, device=dev) * 0.1 if randomize_bn else torch.zeros_like(b))
                else:
                    b.copy_(torch.rand(b.shape, generator=g, device=dev) + 0.5 if randomize_bn else torch.ones_like(b))
        self.weights_changed()

    def state_dict(self) -> Dict[str, torch.Tensor]:
        out = {e.name: self.param(e.name).detach().clone() for e in self.layout.entries}
        for k, b in self.buffers.items():
            out[k] = b.detach().clone()
            if k.endswith("running_var"):
                out[k.replace("running_var", "num_batches_tracked")] = torch.tensor(0, dtype=torch.long)
        return out

    def weights_changed(self) -> None:
        """Re-stage bf16 GEMM weights (and, in eval mode, the folded BN affines) from the fp32 masters."""
        s = ops.stream_ptr()
        self._stage_weights(s)
        if not self.training:
            for bn in self._bn.values():
                _lib.check(self.lib.b2u_bn_eval_affine(bn.C, _p(bn.gamma), _p(bn.beta), _p(bn.running_mean),
                                                       _p(bn.running_var), BN_EPS, _p(bn.scale), _p(bn.shift), s),
                           "b2u_bn_eval_affine")

    # ------------------------------------------------------------------------------------------------ build helpers
    def _act(self, H: int, W: int, Cc: int, name: str = "", zero: bool = False) -> Act:
        a = Act(self.N, H, W, Cc, self.device, name, zero)
        # every activation stays referenced for the life of the plan: the launch plans hold raw device pointers, so a
        # garbage-collected tensor would hand its memory to a later allocation while kernels still address it
        self.acts.append(a)
        if name:
            self.named_acts[name] = a
        return a

    def _bn_state(self, prefix: str, Cc: int) -> BNState:
        st = BNState(self, prefix, Cc)
        self._bn[prefix] = st
        return st

    def _weights(self, cs: ConvSpec, need_dgrad: bool, master_cin: Optional[int] = None) -> Dict[str, torch.Tensor]:
        """bf16 GEMM copies of one conv's weights + staging item for the batched cast kernel.  master_cin: row length of
        the fp32 master when the GEMM sees zero pad lanes behind it (the im2col stem: 36 of 48 lanes)."""
        dev = self.device
        kk = cs.ks * cs.ks
        wf = torch.zeros((cs.nf, kk, padc(cs.ni)), dtype=torch.bfloat16, device=dev)
        wd = torch.zeros((cs.ni, kk, padc(cs.nf)), dtype=torch.bfloat16, device=dev) if need_dgrad else None
        w = {"wf": wf, "wd": wd, "bias_rows": None, "row_of_co": None, "row_perm": None}
        if cs.shuffle:
            roc = shuffle_row_of_co(cs.nf)
            w["row_of_co"] = torch.tensor(roc, dtype=torch.int32, device=dev)
            perm = [0] * cs.nf
            for co, r in enumerate(roc):
                perm[r] = co
            w["row_perm"] = torch.tensor(perm, dtype=torch.int32, device=dev)
        if not cs.bn:
            w["bias_rows"] = torch.zeros(ops.pad32(cs.nf), dtype=torch.float32, device=dev)
        it = _lib.WStageItem()
        it.w = self.param(cs.wname).data_ptr()
        it.bias = self.param(cs.bname).data_ptr() if cs.bname else None
        it.row_of_co = _p(w["row_of_co"])
        it.wf, it.wd, it.bias_rows = wf.data_ptr(), _p(wd), _p(w["bias_rows"])
        it.Cout, it.Cin, it.kk, it.wf_cinp, it.wd_coutp = cs.nf, master_cin or cs.ni, kk, padc(cs.ni), padc(cs.nf)
        it.scale = 0.25 if cs.pool else 1.0
        if cs.sn:
            sig = torch.ones(2, dtype=torch.float32, device=dev)      # {sigma, 1/sigma}, written by b2u_spectral_norm
            self._sn_sigma[cs.name] = sig
            it.dscale = sig[1:].data_ptr()
            self._wstage_sa.append(it)
        else:
            self._wstage.append(it)
        self._w[cs.name] = w
        return w

    def _pack_wstage(self, items):
        n = len(items)
        arr = (_lib.WStageItem * n)()
        blocks = 0
        for i, it in enumerate(items):
            it.block_start = blocks
            blocks += ((it.Cout + 31) // 32) * ((it.Cin + 31) // 32)   # one block per 32x32 channel tile
            arr[i] = it
        raw = bytes(arr)
        host = torch.frombuffer(bytearray(raw), dtype=torch.uint8)
        return host.to(self.device), n, blocks

    def _finish_wstage(self) -> None:
        self._wstage_dev, self._wstage_n, self._wstage_blocks = self._pack_wstage(self._wstage)
        if self._wstage_sa:
            self._wstage_sa_dev, self._wstage_sa_n, self._wstage_sa_blocks = self._pack_wstage(self._wstage_sa)

    def _stage_weights(self, s: int) -> None:
        _lib.check(self.lib.b2u_stage_weights(self._wstage_dev.data_ptr(), self._wstage_n, self._wstage_blocks, s),
                   "b2u_stage_weights")

    @staticmethod
    def _views_taps(cs: ConvSpec, x: Act):
        """A-operand views and tap table for fprop / wgrad of conv `cs` reading activation x."""
        if cs.pool:
            views = [view_nhwc(x.t, x.C, parity=(py, px)) for py in range(2) for px in range(2)]
            return views, ops.taps_avgpool_1x1()
        if cs.stride == 2:
            assert cs.ks == 3
            views = [view_nhwc(x.t, x.C, parity=(py, px)) for py in range(2) for px in range(2)]
            return views, ops.taps_conv3_s2()
        return [view_nhwc(x.t, x.C)], ops.taps_conv(cs.ks)

    def _fwd(self, fn: Callable[[int], None], n: int = 1, kind: str = "", nbytes: int = 0) -> None:
        """kind / nbytes: kernel name and ALGORITHMIC bytes (inputs read once + outputs written once) of a memory-bound
        op - what bench.py's `roofline_mem` divides by the measured time."""
        self.fwd_ops.append(fn)
        self.op_tags.append(("fwd", sys._getframe(1).f_code.co_name, sys._getframe(1).f_lineno))
        self.fwd_meta.append((kind, int(nbytes)))
        self.launches_fwd += n

    def _bwd(self, fn: Callable[[int], None], n: int = 1, side: bool = False, kind: str = "", nbytes: int = 0) -> None:
        self.bwd_ops.append(fn)
        self.bwd_side.append(side)
        self.op_tags.append(("bwd", sys._getframe(1).f_code.co_name, sys._getframe(1).f_lineno))
        self.bwd_meta.append((kind, int(nbytes)))
        self.launches_bwd += n

    def _conv_fwd(self, cs: ConvSpec, x: Act, y: Act, *, out_C: Optional[int] = None, scale=None, shift=None,
                  relu=False, res: Optional[Act] = None, stats=False, out_f32: Optional[torch.Tensor] = None,
                  fin: Optional[dict] = None, head: Optional[dict] = None):
        w = self._w[cs.name]
        views, taps = self._views_taps(cs, x)
        plan = ConvPlan(views, view_nhwc(y.t, out_C or cs.nf), w["wf"], cs.ni, taps, scale=scale, shift=shift,
                        res=view_nhwc(res.t, cs.nf) if res is not None else None, relu=relu, stats=stats,
                        out_f32=out_f32, fin=fin, head=head)
        self._keep.append(plan)
        if cs is self._cs0_col:
            plan.alg_cin = self.spec.stem[0].ni * 9      # 36 real lanes of the 48 the GEMM sees (ConvPlan.flops)
        # convolutions over a handful of input or output channels are HBM-bound: input once + output once
        stem = cs.ni <= 8 or cs is self._cs0_col        # (the im2col form of the stem: 36 lanes in, 32 channels out - still HBM-bound)
        small = stem or cs.nf <= 8
        nb = x.pixels * x.ld * 2 + (y.pixels * 4 * out_f32.shape[-1] if out_f32 is not None else y.pixels * y.ld * 2)
        self._fwd(plan.run, kind=("conv_gemm(stem)" if stem else "conv_gemm(head)") if small else "", nbytes=nb if small else 0)
        return plan

    def _bn_finalize_op(self, bn: BNState, partial: torch.Tensor, count: float, train_stats: bool = True):
        rows, _, ld = partial.shape
        lib, sc = self.lib, self._scratch

        def run(s, bn=bn, partial=partial, rows=rows, ld=ld, count=count):
            _lib.check(lib.b2u_bn_finalize(partial.data_ptr(), rows, ld, bn.C, float(count), _p(bn.gamma), _p(bn.beta),
                                           BN_EPS, BN_MOMENTUM, _p(bn.running_mean), _p(bn.running_var), _p(bn.mean),
                                           _p(bn.invstd), _p(bn.scale), _p(bn.shift), sc.data_ptr(), sc.numel(), s),
                       "b2u_bn_finalize")
        return run, (2 if rows > 128 else 1) + (1 if rows > 128 * 128 else 0)

    def _bn_apply_op(self, x: torch.Tensor, ldx: int, bn: BNState, y: torch.Tensor, ldy: int, pixels: int, relu: bool,
                     r: Optional[torch.Tensor] = None, ldr: int = 0, rbn: Optional[BNState] = None):
        lib = self.lib

        def run(s):
            _lib.check(lib.b2u_bn_apply(x.data_ptr(), ldx, _p(bn.scale), _p(bn.shift), _p(r), ldr,
                                        _p(rbn.scale) if rbn else None, _p(rbn.shift) if rbn else None, int(relu),
                                        y.data_ptr(), ldy, pixels, bn.C, s), "b2u_bn_apply")
        return run

    def _stats_op(self, x: torch.Tensor, ldx: int, pixels: int, Cc: int):
        rows = max(1, min(STATS_ROWS, pixels // 64))
        partial = torch.zeros((rows, 2, padc(Cc)), dtype=torch.float32, device=self.device)
        lib = self.lib

        def run(s):
            _lib.check(lib.b2u_bn_stats(x.data_ptr(), ldx, pixels, Cc, partial.data_ptr(), rows, padc(Cc), s),
                       "b2u_bn_stats")
        return run, partial

    def _self_attention(self, sa, c2: Act, h: int, w_: int):
        """fastai layers.SelfAttention on the output of UnetBlock.conv2 (after its ReLU): spectral-normed 1x1 query / key /
        value convolutions, beta = softmax(q_i . k_j over i), o_j = sum_i beta_ij v_i, out = gamma * o + x.  The
        convolutions AND the batched attention products (two forward, four backward; 2 n^2 (C/8 + C) FLOP per image and
        direction = 1.4 % of the forward FLOPs at 256-px tiles) run on the implicit-GEMM kernel - the products as 1x1
        convolutions with per-image weights - the rest is csrc/attention.cu.  Returns (output Act, backward builder)."""
        lib, dev, N, train = self.lib, self.device, self.N, self.training
        n, Cc = h * w_, sa.c
        convs = sa.convs()
        gamma = self.param(sa.gamma)
        for cs in convs:
            W, sig = self.param(cs.wname), self._sn_sigma[cs.name]
            u, v = self.buffers[cs.name + ".0.weight_u"], self.buffers[cs.name + ".0.weight_v"]
            self._fwd(lambda s, W=W, u=u, v=v, sig=sig, cs=cs: _lib.check(
                lib.b2u_spectral_norm(W.data_ptr(), cs.nf, cs.ni, u.data_ptr(), v.data_ptr(), int(train), sig.data_ptr(), s),
                "b2u_spectral_norm"))
        self._fwd(lambda s: _lib.check(lib.b2u_stage_weights(self._wstage_sa_dev.data_ptr(), self._wstage_sa_n,
                                                             self._wstage_sa_blocks, s), "b2u_stage_weights"))
        Q = self._act(h, w_, sa.query.nf, sa.name + ".q")
        K = self._act(h, w_, sa.key.nf, sa.name + ".k")
        V = self._act(h, w_, sa.value.nf, sa.name + ".v")
        for cs, y in zip(convs, (Q, K, V)):
            self._conv_fwd(cs, c2, y)
        ldn = padc(n)
        zt = lambda *shape: torch.zeros(shape, dtype=torch.bfloat16, device=dev)
        S = zt(N, h, w_, ldn)             # logits q_i . k_j ([image][i][j]); reused for d(beta) and dS in the backward pass
        # softmax over i (a named activation: the parity tests pin it), and its transpose ([image][j][i])
        beta, betaT = self._act(h, w_, n, sa.name + ".beta", zero=True).t, zt(N, h, w_, ldn)
        VT = zt(N, Cc, ldn)               # value^T: channels x positions (the contraction index of `o` innermost)
        O = self._act(h, w_, Cc, sa.name + ".o")
        out = self._act(h, w_, Cc, sa.name + ".out")
        self._keep += [S, beta, betaT, VT]

        def bmm(a_t: torch.Tensor, a_c: int, w_t: torch.Tensor, rows: int, out_t: torch.Tensor) -> ConvPlan:
            """out[img, p, r] = sum_c a[img, p, c] * w[img, r, c]: torch.bmm(A, W^T) as a 1x1 'convolution' whose weights
            change with the image (b2u_conv_desc.w_batch_rows)"""
            plan = ConvPlan([view_nhwc(a_t, a_c)], view_nhwc(out_t, rows), w_t.view(N * rows, 1, w_t.shape[-1]), a_c,
                            ops.taps_conv(1), w_batch_rows=rows)
            self._keep.append(plan)
            return plan

        p_s = bmm(Q.t, sa.query.nf, K.t, n, S)                  # S[i][j] = q_i . k_j          (bmm(f^T, g))
        p_o = bmm(betaT, n, VT, Cc, O.t)                        # o_j = sum_i beta_ij v_i      (bmm(h, beta))
        self._fwd(p_s.run)
        self._fwd(lambda s: _lib.check(lib.b2u_softmax_dim1(S.data_ptr(), beta.data_ptr(), betaT.data_ptr(), N, n, ldn, s),
                                       "b2u_softmax_dim1"))
        self._fwd(lambda s: _lib.check(lib.b2u_transpose_bnc(V.t.data_ptr(), V.ld, VT.data_ptr(), ldn, N, n, Cc, s),
                                       "b2u_transpose_bnc"))
        self._fwd(p_o.run)
        self._fwd(lambda s: _lib.check(lib.b2u_attn_out(O.t.data_ptr(), c2.t.data_ptr(), gamma.data_ptr(), out.t.data_ptr(),
                                                        out.t.numel(), s), "b2u_attn_out"))
        if not train:
            return out, None

        def build_bwd():
            assert out.grad is not None and out.grad_written, sa.name
            dOut = out.grad
            dO = torch.zeros_like(O.t)
            dQ, dK, dV = torch.zeros_like(Q.t), torch.zeros_like(K.t), torch.zeros_like(V.t)
            dOT, KT, QT = zt(N, Cc, ldn), zt(N, sa.key.nf, ldn), zt(N, sa.query.nf, ldn)
            scratch = torch.zeros(1025, dtype=torch.float32, device=dev)
            self._keep += [dO, dQ, dK, dV, dOT, KT, QT, scratch]
            dgamma = self.grad(sa.gamma)
            tr = lambda x, ldx, y, cc: (lambda s: _lib.check(lib.b2u_transpose_bnc(x.data_ptr(), ldx, y.data_ptr(), ldn, N, n, cc, s),
                                                            "b2u_transpose_bnc"))
            p_dv = bmm(beta, n, dOT, Cc, dV)                     # dV_i = sum_j beta_ij dO_j
            p_db = bmm(V.t, Cc, dO, n, S)                        # d(beta)_ij = v_i . dO_j   (into S)
            p_dq = bmm(S, n, KT, sa.query.nf, dQ)                # dQ_i = sum_j dS_ij k_j
            p_dk = bmm(betaT, n, QT, sa.key.nf, dK)              # dK_j = sum_i dS_ij q_i    (dS^T lives in betaT's buffer)
            self._bwd(lambda s: _lib.check(lib.b2u_attn_out_bwd(dOut.data_ptr(), O.t.data_ptr(), gamma.data_ptr(),
                                                                dO.data_ptr(), dgamma.data_ptr(), scratch.data_ptr(),
                                                                dO.numel(), s), "b2u_attn_out_bwd"))
            self._bwd(tr(dO, O.ld, dOT, Cc))
            self._bwd(p_dv.run)
            self._bwd(p_db.run)
            self._bwd(lambda s: _lib.check(lib.b2u_softmax_dim1_bwd(beta.data_ptr(), S.data_ptr(), S.data_ptr(),
                                                                    betaT.data_ptr(), N, n, ldn, s),
                                           "b2u_softmax_dim1_bwd"))                  # dS in place, dS^T over beta^T
            self._bwd(tr(K.t, K.ld, KT, sa.key.nf))
            self._bwd(tr(Q.t, Q.ld, QT, sa.query.nf))
            self._bwd(p_dq.run)
            self._bwd(p_dk.run)
            for cs, d in zip(convs, (dQ, dK, dV)):
                self._wgrad(cs, d, c2)
                # gradient through W / sigma(W), after the split-K reduce of this weight (same stream as the wgrad)
                W, dW, sig = self.param(cs.wname), self.grad(cs.wname), self._sn_sigma[cs.name]
                u, v = self.buffers[cs.name + ".0.weight_u"], self.buffers[cs.name + ".0.weight_v"]
                self._bwd(lambda s, W=W, dW=dW, u=u, v=v, sig=sig, cs=cs: _lib.check(
                    lib.b2u_spectral_norm_bwd(dW.data_ptr(), W.data_ptr(), cs.nf, cs.ni, u.data_ptr(), v.data_ptr(),
                                              sig.data_ptr(), s), "b2u_spectral_norm_bwd"), side=True)
            # c2.grad = (dOut + Wq^T dQ + Wk^T dK + Wv^T dV) * (c2 > 0): a pre-ReLU gradient, as conv2's backward expects
            self._dgrad(convs[0], dQ, c2, res=dOut)
            self._dgrad(convs[1], dK, c2)
            self._dgrad(convs[2], dV, c2, zmask=True)
        return out, build_bwd

    # ---- backward helpers ---------------------------------------------------------------------------------------
    def _bn_bwd(self, bn: BNState, dz: torch.Tensor, lddz: int, x: torch.Tensor, ldx: int, y: Optional[torch.Tensor],
                ldy: int, relu: bool, dx: torch.Tensor, lddx: int, pixels: int, accumulate: bool):
        """reduce -> finalize -> apply in one launch (grid barrier inside); dgamma/dbeta land in the flat gradient
        buffer."""
        rows = max(1, min(STATS_ROWS, pixels * ((bn.C + 7) // 8) // int(os.environ.get("B2U_BN_BWD_ITEMS", "1024"))))   # >= ~4 (pixel, 8-channel) items per thread
        partial = torch.zeros((rows, 2, padc(bn.C)), dtype=torch.float32, device=self.device)
        lib = self.lib
        ld = padc(bn.C)
        if not hasattr(self, "_bn_sync"):
            self._bn_sync = torch.zeros(2, dtype=torch.int32, device=self.device)
        sync = self._bn_sync

        def run(s):
            _lib.check(lib.b2u_bn_bwd_fused(dz.data_ptr(), lddz, x.data_ptr(), ldx, _p(y), ldy, _p(bn.scale),
                                            _p(bn.shift), _p(bn.mean), _p(bn.invstd), _p(bn.gamma), int(relu),
                                            int(accumulate), dx.data_ptr(), lddx, pixels, bn.C, partial.data_ptr(),
                                            rows, ld, float(pixels), _p(bn.dgamma), _p(bn.dbeta), _p(bn.mean_g),
                                            _p(bn.mean_gx), sync.data_ptr(), s), "b2u_bn_bwd_fused")
        self._keep.append(partial)
        # algorithmic bytes: dz, x (and the block output that carries the ReLU mask) read once, dx written once
        self._bwd(run, 1, kind="bn_bwd_fused", nbytes=pixels * 2 * (lddz + ldx + (ldy if y is not None else 0) + lddx))

    def _wgrad(self, cs: ConvSpec, dy: torch.Tensor, x: Act):
        """dW (and db) of conv `cs` from dy (bf16 NHWC tensor [N,Ho,Wo,padc(nf)]) and its input activation x."""
        w = self._w[cs.name]
        views, taps = self._views_taps(cs, x)
        kidx = [0] * len(taps) if cs.pool else [t[3] for t in taps]
        spec = dict(cs=cs, dy_view=view_nhwc(dy, cs.nf), views=views, taps=taps, kidx=kidx,
                    dw=self.grad(cs.wname), db=self.grad(cs.bname) if cs.bname else None, row_perm=w["row_perm"],
                    alpha=0.25 if cs.pool else 1.0, keep=(dy, x))
        # (im2col stem: the views expose 48 lanes, the master weight - and its gradient - has n_in*9 = 36 columns)
        spec["cin"] = self.spec.stem[0].ni * 9 if cs is self._cs0_col else cs.ni
        info = WgradPlan.query(spec["dy_view"], views, taps, cs.nf, spec["cin"], spec["db"] is not None)
        spec["bytes"] = info.partial_bytes
        self._wgrad_specs.append(spec)
        slot = len(self._wgrad_specs) - 1

        def run(s, slot=slot):
            self._wgrad_plans[slot].run(s)
        self._bwd(run, 2, side=True)

    def _dgrad(self, cs: ConvSpec, dy: torch.Tensor, x: Act, *, zmask: bool = False, res: Optional[torch.Tensor] = None,
               res_mask: Optional[torch.Tensor] = None, out_C: Optional[int] = None):
        """dX of conv `cs` (accumulating if x.grad already holds a contribution)."""
        w = self._w[cs.name]
        dx = x.ensure_grad()
        Cx = out_C or cs.ni
        acc = x.grad_written
        assert not (acc and res is not None), "dgrad: accumulate + extra residual not supported"
        wd = w["wd"][:Cx] if Cx != cs.ni else w["wd"]
        a = [view_nhwc(dy, cs.nf)]

        def mk(out_view, taps, par):
            r = out_view if acc else (view_nhwc(res, Cx, parity=par) if res is not None else None)
            rm = view_nhwc(res_mask, Cx, parity=par) if (res_mask is not None and not acc) else None
            zm = view_nhwc(x.t, Cx, parity=par) if zmask else None
            plan = ConvPlan(a, out_view, wd, cs.nf, taps, res=r, res_mask=rm, zmask=zm)
            self._keep.append(plan)
            self._bwd(plan.run)

        if cs.pool:
            for py in range(2):
                for px in range(2):
                    mk(view_nhwc(dx, Cx, parity=(py, px)), [(0, 0, 0, 0)], (py, px))
        elif cs.stride == 2:
            for py in range(2):
                for px in range(2):
                    mk(view_nhwc(dx, Cx, parity=(py, px)), ops.taps_dgrad_s2(py, px), (py, px))
        else:
            mk(view_nhwc(dx, Cx), ops.taps_conv(cs.ks), None)
        x.grad_written = True

    # ------------------------------------------------------------------------------------------------ the network
    def _build(self) -> None:
        spec, N, H, W, dev, lib = self.spec, self.N, self.H, self.W, self.device, self.lib
        train = self.training
        # weights for every conv (first stem conv never needs a dgrad copy: the image has no gradient)
        # im2col stem: the first convolution (3x3, stride 2, n_in bands) runs as a 1x1 convolution over the n_in*9 im2col
        # lanes written by b2u_im2col (zero padded to whole 32-byte sectors) - its weight [nf][n_in][3][3] read as rows of
        # n_in*9 IS the 1x1 weight, and so is its gradient
        cs0 = spec.stem[0]
        # (training only: the win is the weight gradient - 0.167 -> 0.04 ms, the 8-byte pixels of the 4-band image are one
        # TMA request each; for the inference forward the extra im2col pass costs more than the 1x1 form saves)
        self.stem_im2col = STEM_IM2COL and train and cs0.ks == 3 and cs0.stride == 2 and cs0.ni * 9 <= 64 and not cs0.pool
        self._cs0_col = dataclasses.replace(cs0, ni=(cs0.ni * 9 + 15) // 16 * 16, ks=1, stride=1) if self.stem_im2col else None
        for i, cs in enumerate(spec.convs()):
            if i == 0 and self.stem_im2col:
                assert cs is cs0
                self._weights(self._cs0_col, need_dgrad=False, master_cin=cs0.ni * 9)
            else:
                self._weights(cs, need_dgrad=train and i != 0)
        self._finish_wstage()

        # ---- input
        self.x_in = self._act(H, W, spec.n_in, "input", zero=True)
        # fp32 logits [N, H, W, ld]: ld = n_out for up to 8 classes (8 bytes per pixel at C = 2; a pitch of 8 floats made the
        # head store - and the loss / stitch kernels read - 4 x the useful bytes in partial sectors)
        self.logits = torch.zeros((N, H, W, spec.n_out if spec.n_out <= 8 else padc(spec.n_out)), dtype=torch.float32,
                                  device=dev)
        bwd_layers: List[Callable[[], None]] = []

        # ---- encoder ConvLayer = conv -> BN -> [ReLU]
        def conv_bn(cs: ConvSpec, x: Act, h: int, w_: int, apply: bool) -> Tuple[Act, Optional[Act], BNState]:
            bn = self._bn_state(cs.bn_prefix, cs.nf)
            if train:
                R = self._act(h, w_, cs.nf, cs.name + ".raw")
                # the conv kernel's last CTA finalizes the batch statistics (mean/invstd/scale/shift, running stats)
                plan = self._conv_fwd(cs, x, R, stats=True, fin=dict(
                    count=N * h * w_, gamma=bn.gamma, beta=bn.beta, eps=BN_EPS, momentum=BN_MOMENTUM,
                    running_mean=bn.running_mean, running_var=bn.running_var, mean=bn.mean, invstd=bn.invstd,
                    scale=bn.scale, shift=bn.shift))
                if not plan.fused_finalize:   # Cout > 512 (xresnet50/101): per-tile partial rows, separate finalize
                    fin, nl = self._bn_finalize_op(bn, plan.stats, N * h * w_)
                    self._fwd(fin, nl)
                Z = None
                if apply:
                    Z = self._act(h, w_, cs.nf, cs.name + ".out")
                    self._fwd(self._bn_apply_op(R.t, R.ld, bn, Z.t, Z.ld, R.pixels, cs.act), kind="bn_apply",
                              nbytes=R.pixels * (R.ld + Z.ld) * 2)
                return R, Z, bn
            Z = self._act(h, w_, cs.nf, cs.name + ".out")
            if apply:
                self._conv_fwd(cs, x, Z, scale=bn.scale, shift=bn.shift, relu=cs.act)
            return Z, Z, bn  # (eval: when apply is False the caller fuses scale/shift itself)

        def conv_bn_bwd(cs: ConvSpec, x: Act, R: Act, Z: Act, bn: BNState, need_dx: bool):
            def build():
                dR = torch.zeros_like(R.t)
                self._keep.append(dR)
                self._bn_bwd(bn, Z.grad, Z.ld, R.t, R.ld, None, 0, cs.act, dR, R.ld, R.pixels, False)
                self._wgrad(cs, dR, x)
                if need_dx:
                    self._dgrad(cs, dR, x)
            return build

        x = self.x_in
        up2 = lambda v, st=2: (v + st - 1) // st
        h, w_ = up2(H), up2(W)
        feats: Dict[int, Act] = {}
        for i, cs in enumerate(spec.stem):
            if i == 0 and self.stem_im2col:
                xc = self._act(h, w_, self._cs0_col.ni, "input.im2col", zero=True)
                self._fwd(lambda s, a=x, b=xc, c0=cs: _lib.check(
                    lib.b2u_im2col(a.t.data_ptr(), a.ld, c0.ni, N, a.H, a.W, c0.ks, c0.stride, c0.ks // 2, b.t.data_ptr(), b.ld, s),
                    "b2u_im2col"), kind="im2col", nbytes=x.pixels * x.ld * 2 + xc.pixels * xc.ld * 2)
                cs, x = self._cs0_col, xc
            R, Z, bn = conv_bn(cs, x, h, w_, apply=True)
            if train:
                bwd_layers.append(conv_bn_bwd(cs, x, R, Z, bn, need_dx=i != 0))
            x = Z
        feats[2] = x
        # ---- maxpool
        mp_in = x
        h, w_ = up2(h), up2(w_)
        mp = self._act(h, w_, mp_in.C, "maxpool")
        idx = torch.zeros((N, h, w_, mp.ld), dtype=torch.uint8, device=dev) if train else None
        self._fwd(lambda s, a=mp_in, b=mp, idx=idx: _lib.check(
            lib.b2u_maxpool_fwd(a.t.data_ptr(), b.t.data_ptr(), _p(idx), N, a.H, a.W, a.C, a.ld, s), "b2u_maxpool_fwd"),
            kind="maxpool_fwd", nbytes=mp_in.pixels * mp_in.ld * 2 + mp.pixels * mp.ld * (3 if train else 2))
        if train:
            def mp_bwd():
                g = mp_in.ensure_grad()
                acc = int(mp_in.grad_written)
                self._bwd(lambda s: _lib.check(lib.b2u_maxpool_bwd(mp.grad.data_ptr(), idx.data_ptr(), g.data_ptr(), acc,
                                                                   N, mp_in.H, mp_in.W, mp_in.C, mp_in.ld, s),
                                               "b2u_maxpool_bwd"), kind="maxpool_bwd",
                          nbytes=mp.pixels * mp.ld * 3 + mp_in.pixels * mp_in.ld * (4 if acc else 2))
                mp_in.grad_written = True
            bwd_layers.append(mp_bwd)
        x = mp

        # ---- residual stages
        for si, blocks in enumerate(spec.stages):
            for blk in blocks:
                xin = x
                ho, wo = up2(h, blk.stride), up2(w_, blk.stride)
                cur, ch, cw = xin, h, w_
                recs = []
                for j, cs in enumerate(blk.convpath):
                    ch, cw = up2(ch, cs.stride), up2(cw, cs.stride)
                    last = j == len(blk.convpath) - 1
                    R, Z, bn = conv_bn(cs, cur, ch, cw, apply=not last)
                    recs.append((cs, cur, R, Z, bn))
                    cur = Z if not last else R
                idrec = None
                xid, xpad = xin, None
                if blk.idconv is not None:
                    if blk.idconv.pool and (h % 2 or w_ % 2):
                        # AvgPool2d(2, ceil_mode=True) on an odd extent: replicate the last row / column first, then the
                        # plain 2x2 mean (folded into the 1x1 conv taps) equals torch's clipped-window average
                        xpad = self._act(h + h % 2, w_ + w_ % 2, xin.C, blk.name + ".idpad")
                        self._fwd(lambda s, a=xin, b=xpad: _lib.check(
                            lib.b2u_pad_even_fwd(a.t.data_ptr(), b.t.data_ptr(), a.ld, N, a.H, a.W, s), "b2u_pad_even_fwd"))
                        xid = xpad
                    Rid, _, bnid = conv_bn(blk.idconv, xid, ho, wo, apply=False)
                    idrec = (blk.idconv, Rid, bnid)
                out = self._act(ho, wo, blk.nf, blk.name + ".out")
                csl, xl, Rl, _, bnl = recs[-1]
                if train:
                    if idrec is not None:
                        self._fwd(self._bn_apply_op(Rl.t, Rl.ld, bnl, out.t, out.ld, out.pixels, True, idrec[1].t,
                                                    idrec[1].ld, idrec[2]), kind="bn_apply", nbytes=out.pixels * out.ld * 6)
                    else:
                        self._fwd(self._bn_apply_op(Rl.t, Rl.ld, bnl, out.t, out.ld, out.pixels, True, xin.t, xin.ld),
                                  kind="bn_apply", nbytes=out.pixels * out.ld * 6)
                else:
                    # eval: BN folded into the conv epilogues; the block tail is one fused launch
                    if idrec is not None:
                        self._conv_fwd(idrec[0], xid, idrec[1], scale=idrec[2].scale, shift=idrec[2].shift)
                        self._conv_fwd(csl, xl, out, scale=bnl.scale, shift=bnl.shift, relu=True, res=idrec[1])
                    else:
                        self._conv_fwd(csl, xl, out, scale=bnl.scale, shift=bnl.shift, relu=True, res=xin)

                if train:
                    def blk_bwd(blk=blk, xin=xin, out=out, recs=recs, idrec=idrec, xid=xid, xpad=xpad):
                        dOut = out.grad
                        assert dOut is not None and out.grad_written, blk.name
                        # tail: BN of the last convpath conv, masked by the block output
                        csl, xl, Rl, _, bnl = recs[-1]
                        dRl = torch.zeros_like(Rl.t)
                        self._keep.append(dRl)
                        self._bn_bwd(bnl, dOut, out.ld, Rl.t, Rl.ld, out.t, out.ld, False, dRl, Rl.ld, Rl.pixels, False)
                        if idrec is not None:
                            csi, Rid, bnid = idrec
                            dRid = torch.zeros_like(Rid.t)
                            self._keep.append(dRid)
                            self._bn_bwd(bnid, dOut, out.ld, Rid.t, Rid.ld, out.t, out.ld, False, dRid, Rid.ld,
                                         Rid.pixels, False)
                            self._wgrad(csi, dRid, xid)
                            self._dgrad(csi, dRid, xid)
                            if xpad is not None:
                                g = xin.ensure_grad()
                                acc = int(xin.grad_written)
                                self._bwd(lambda s: _lib.check(lib.b2u_pad_even_bwd(
                                    xpad.grad.data_ptr(), g.data_ptr(), acc, xin.ld, N, xin.H, xin.W, s), "b2u_pad_even_bwd"))
                                xin.grad_written = True
                        dcur = dRl
                        for j in range(len(recs) - 1, -1, -1):
                            cs, xj, Rj, Zj, bnj = recs[j]
                            self._wgrad(cs, dcur, xj)
                            if j == 0:
                                if idrec is None:
                                    assert not xin.grad_written
                                    self._dgrad(cs, dcur, xj, res=dOut, res_mask=out.t)  # identity path: + dOut*(out>0)
                                else:
                                    self._dgrad(cs, dcur, xj)
                            else:
                                self._dgrad(cs, dcur, xj)
                                csp, xp, Rp, Zp, bnp = recs[j - 1]
                                dRp = torch.zeros_like(Rp.t)
                                self._keep.append(dRp)
                                self._bn_bwd(bnp, Zp.grad, Zp.ld, Rp.t, Rp.ld, None, 0, True, dRp, Rp.ld, Rp.pixels, False)
                                dcur = dRp
                    if blk is blocks[0]:
                        # backward reaches this block LAST within its stage: once it has run, every gradient of the
                        # stage's parameters is final (all-reduce mark, see engine.Trainer)
                        blk_bwd.ar_mark = blk.convpath[0].wname
                    bwd_layers.append(blk_bwd)
                x, h, w_ = out, ho, wo
            feats[4 + si] = x

        # ---- layers.1/2: BatchNorm + ReLU on the encoder output
        E = x
        bnE = self._bn_state(spec.post_bn, E.C)
        ZE = self._act(h, w_, E.C, "enc.bnrelu")
        if train:
            st, partial = self._stats_op(E.t, E.ld, E.pixels, E.C)
            self._fwd(st)
            fin, nl = self._bn_finalize_op(bnE, partial, E.pixels)
            self._fwd(fin, nl)
        self._fwd(self._bn_apply_op(E.t, E.ld, bnE, ZE.t, ZE.ld, E.pixels, True))
        if train:
            def post_bwd():
                dE = E.ensure_grad()
                self._bn_bwd(bnE, ZE.grad, ZE.ld, E.t, E.ld, None, 0, True, dE, E.ld, E.pixels, E.grad_written)
                E.grad_written = True
            post_bwd.is_encoder_boundary = True
            bwd_layers.append(post_bwd)

        # ---- decoder conv (+bias, ReLU fused): gradient buffers hold PRE-activation gradients
        def conv_bias(cs: ConvSpec, xa: Act, hh: int, ww: int, res: Optional[Act] = None, relu: bool = True,
                      head: Optional[dict] = None) -> Act:
            y = self._act(hh, ww, cs.nf, cs.name + ".out")
            y.pre_relu_grad = relu
            self._conv_fwd(cs, xa, y, shift=self._w[cs.name]["bias_rows"], relu=relu, res=res, head=head)
            return y

        def conv_bias_bwd(cs: ConvSpec, xa: Act, y: Act, **dg):
            def build():
                assert y.grad is not None and y.grad_written, cs.name
                self._wgrad(cs, y.grad, xa)
                self._dgrad(cs, y.grad, xa, zmask=xa.pre_relu_grad, **dg)
            return build

        x = ZE
        for cs in spec.middle:
            y = conv_bias(cs, x, h, w_)
            if train:
                bwd_layers.append(conv_bias_bwd(cs, x, y))
            x = y

        # ---- UnetBlocks
        for ub in spec.unet:
            U, S = x, feats[ub.skip_child]
            P = conv_bias(ub.shuf, U, h, w_)
            bnS = self._bn_state(ub.bn_prefix, S.C)
            if train:
                st, partial = self._stats_op(S.t, S.ld, S.pixels, S.C)
                self._fwd(st)
                fin, nl = self._bn_finalize_op(bnS, partial, S.pixels)
                self._fwd(fin, nl)
            assert S.H in (2 * h, 2 * h - 1) and S.W in (2 * w_, 2 * w_ - 1), "skip / upsample size mismatch"
            h, w_ = S.H, S.W       # an odd skip crops the last row / column of the upsampled tensor (nearest interpolate)
            cat = self._act(h, w_, ub.cu + S.C, ub.name + ".cat")
            cat.pre_relu_grad = True
            self._fwd(lambda s, P=P, S=S, cat=cat, bnS=bnS, cu=ub.cu: _lib.check(
                lib.b2u_shuffle_cat_fwd_crop(P.t.data_ptr(), P.ld, cu, 1, S.t.data_ptr(), S.ld, S.C, _p(bnS.scale),
                                             _p(bnS.shift), 1, cat.t.data_ptr(), cat.ld, N, P.H, P.W, cat.H, cat.W, s),
                "b2u_shuffle_cat_fwd"), kind="shuffle_cat_fwd",
                nbytes=(P.pixels * P.ld + S.pixels * S.ld + cat.pixels * cat.ld) * 2)
            c1 = conv_bias(ub.conv1, cat, h, w_)
            c2 = conv_bias(ub.conv2, c1, h, w_)
            sa_bwd = None
            x_out = c2
            if ub.sa is not None:
                x_out, sa_bwd = self._self_attention(ub.sa, c2, h, w_)
            if train:
                def ub_bwd(ub=ub, U=U, S=S, P=P, cat=cat, c1=c1, c2=c2, bnS=bnS, sa_bwd=sa_bwd):
                    if sa_bwd is not None:
                        sa_bwd()
                    conv_bias_bwd(ub.conv2, c1, c2)()
                    conv_bias_bwd(ub.conv1, cat, c1)()
                    dP = P.ensure_grad()
                    dcat = cat.grad
                    self._bwd(lambda s: _lib.check(lib.b2u_shuffle_bwd_crop(dcat.data_ptr(), cat.ld, P.t.data_ptr(),
                                                                            dP.data_ptr(), P.ld, ub.cu, 1, N, P.H, P.W,
                                                                            cat.H, cat.W, s), "b2u_shuffle_bwd"),
                              kind="shuffle_bwd", nbytes=(cat.pixels * ub.cu + 2 * P.pixels * P.ld) * 2)
                    P.grad_written = True
                    dS = S.ensure_grad()
                    self._bn_bwd(bnS, dcat[..., ub.cu:], cat.ld, S.t, S.ld, None, 0, False, dS, S.ld, S.pixels,
                                 S.grad_written)
                    S.grad_written = True
                    conv_bias_bwd(ub.shuf, U, P)()
                bwd_layers.append(ub_bwd)
            x = x_out

        # ---- final PixelShuffle_ICNR (no blur) + MergeLayer(dense) + ResBlock(no norm) + head
        U = x
        fs = spec.final_shuf
        cu = fs.nf // 4
        xin = self.x_in
        # no blur in this stage, so PixelShuffle is a pure permutation: the 1x1 convolution stores its four (i,j) phases
        # straight into the four stride-2 parity planes of the concat tensor (one launch, four N tiles, four output
        # maps) - no pre-shuffle tensor, no shuffle pass.  Needs cu (= one N tile) to be a multiple of 16 and <= 256.
        # (the TMA store covers whole 64-lane chunks: they must stay inside the pixel's pitch, or a parity plane would
        # write into its neighbour's lanes)
        fused_shuffle = (FUSED_FINAL_SHUFFLE and cu % 16 == 0 and cu <= 256 and (2 * h, 2 * w_) == (H, W) and
                         (cu + 63) // 64 * 64 <= padc(cu + spec.n_in))
        P8 = None if fused_shuffle else conv_bias(fs, U, h, w_)
        hs, ws = h, w_
        assert H in (2 * h, 2 * h - 1) and W in (2 * w_, 2 * w_ - 1)
        h, w_ = H, W               # ResizeToOrig: an odd tile crops the last row / column (nearest interpolate)
        cat = self._act(h, w_, cu + spec.n_in, "layers.10.cat", zero=True)
        if fused_shuffle:
            wfs = self._w[fs.name]
            outs = [view_nhwc(cat.t, cu, parity=(i, j)) for i in range(2) for j in range(2)]
            geom = view_nhwc(cat.t, cu, parity=(0, 0))
            geom.C = fs.nf                      # GEMM space: (N, hs, ws) pixels x 4*cu output channels
            plan = ConvPlan([view_nhwc(U.t, U.C)], geom, wfs["wf"], fs.ni, ops.taps_conv(1), shift=wfs["bias_rows"],
                            relu=True, outs=outs)
            self._keep.append(plan)
            self._fwd(plan.run)
            # MergeLayer(dense=True): the image bands go behind the shuffled channels (the conv zeroed lanes >= cu)
            lanes = min(xin.ld, cat.ld - cu)
            self._fwd(lambda s: _lib.check(
                lib.b2u_copy_lanes(xin.t.data_ptr(), xin.ld, 0, cat.t.data_ptr(), cat.ld, cu, lanes, cat.pixels, s),
                "b2u_copy_lanes"), kind="copy_lanes", nbytes=cat.pixels * lanes * 4)
        else:
            self._fwd(lambda s: _lib.check(
                lib.b2u_shuffle_cat_fwd_crop(P8.t.data_ptr(), P8.ld, cu, 0, xin.t.data_ptr(), xin.ld, xin.C, None, None, 0,
                                             cat.t.data_ptr(), cat.ld, N, P8.H, P8.W, cat.H, cat.W, s),
                "b2u_shuffle_cat_fwd"))
        ra, rb = spec.final_res
        A1 = conv_bias(ra, cat, h, w_)
        hd = spec.head
        # Inference: layers.12 (the 1x1 head) rides in the epilogue of the last ResBlock convolution when that is a single
        # N tile (<= 256 channels) and there are <= 8 outputs - the logits come out of the pass that would have produced
        # A2, and A2 (the largest activation of the network, read by nothing else) is never written: 10.5k -> 11.4k
        # tiles/s on the 20000^2 raster.  Training keeps the separate head launch: A2 must be stored for the backward pass
        # anyway and the fused epilogue measured the same step time (19.85 ms both ways).
        self.fused_head = FUSED_HEAD and not train and rb.nf <= 256 and hd.nf <= 8
        head = dict(w=self._w[hd.name]["wf"], b=self._w[hd.name]["bias_rows"], out=self.logits,
                    only=True) if self.fused_head else None
        A2 = conv_bias(rb, A1, h, w_, res=cat, relu=True, head=head)  # relu(convpath(x) + x)
        if not self.fused_head:
            hv = self._act(h, w_, hd.nf, "head.geom")  # geometry carrier only; the head stores fp32 logits
            self._conv_fwd(hd, A2, hv, shift=self._w[hd.name]["bias_rows"], out_f32=self.logits)
        self.out_act = A2

        if train:
            # loss buffers
            P_ = N * H * W
            # class ids (uint8) - or the continuous target of the regression variant (RegressionBlock, data.py:98)
            self.labels = torch.zeros((N, H, W), dtype=torch.float32 if self.regression else torch.uint8, device=dev)
            self.dlogits = torch.zeros((N, H, W, padc(spec.n_out)), dtype=torch.bfloat16, device=dev)
            self.loss = torch.zeros(1, dtype=torch.float32, device=dev)
            self._ce_rows = 592
            self._wsum_part = torch.zeros(self._ce_rows, dtype=torch.float32, device=dev)
            self._loss_part = torch.zeros(max(self._ce_rows, N), dtype=torch.float32, device=dev)   # Dice: one per sample
            # DiceLoss: per-block statistics of every (sample, class), folded by its backward kernel
            self._dice_bps = dice_blocks_per_sample(N, H * W) if self.loss_spec.name == "dice" else 0
            self._dice_part = torch.zeros(N * self._dice_bps * 3 * spec.n_out, dtype=torch.float32, device=dev) \
                if self._dice_bps else None

            def tail_bwd():
                dL = self.dlogits
                self._wgrad(hd, dL, A2)
                if hd.nf <= 8:
                    # GEMM K = number of classes: a tensor-core tile would be almost all padding -> streaming kernel
                    dA2 = A2.ensure_grad()
                    wd = self._w[hd.name]["wd"]
                    self._bwd(lambda s: _lib.check(lib.b2u_pointwise_smallk(
                        dL.data_ptr(), dL.shape[-1], hd.nf, wd.data_ptr(), wd.shape[-1], A2.t.data_ptr(), A2.ld,
                        dA2.data_ptr(), A2.ld, A2.pixels, A2.C, s), "b2u_pointwise_smallk"), kind="pointwise_smallk",
                        nbytes=A2.pixels * (dL.shape[-1] + 2 * A2.ld) * 2)
                else:
                    self._dgrad(hd, dL, A2, zmask=True)
                A2.grad_written = True
                self._wgrad(rb, A2.grad, A1)
                self._dgrad(rb, A2.grad, A1, zmask=True)
                self._wgrad(ra, A1.grad, cat)
                # only the shuffled channels need a gradient (the image does not): restrict dgrad to [0, cu)
                self._dgrad(ra, A1.grad, cat, res=A2.grad, out_C=cu)
                if fused_shuffle:
                    dP8 = torch.zeros((N, hs, ws, padc(fs.nf)), dtype=torch.bfloat16, device=dev)
                    self._keep.append(dP8)
                    # the ReLU mask of the shuffle conv is read from cat itself (cat[..., :cu] = relu(conv) shuffled)
                    self._bwd(lambda s: _lib.check(lib.b2u_shuffle_bwd_from_cat(
                        cat.grad.data_ptr(), cat.t.data_ptr(), cat.ld, dP8.data_ptr(), dP8.shape[-1], cu, N, hs, ws, s),
                        "b2u_shuffle_bwd_from_cat"), kind="shuffle_bwd(final)",
                        nbytes=(2 * cat.pixels * cu + N * hs * ws * dP8.shape[-1]) * 2)
                    self._wgrad(fs, dP8, U)
                    self._dgrad(fs, dP8, U, zmask=U.pre_relu_grad)
                else:
                    dP8 = P8.ensure_grad()
                    self._bwd(lambda s: _lib.check(lib.b2u_shuffle_bwd_crop(cat.grad.data_ptr(), cat.ld, P8.t.data_ptr(),
                                                                            dP8.data_ptr(), P8.ld, cu, 0, N, P8.H, P8.W,
                                                                            cat.H, cat.W, s), "b2u_shuffle_bwd"))
                    P8.grad_written = True
                    conv_bias_bwd(fs, U, P8)()
            bwd_layers.append(tail_bwd)

            # build backward in true reverse order (gradient accumulation flags depend on it)
            # all-reduce marks (op index, parameter offset): after op index k every gradient at offsets >= off is final.
            # The flat layout is in forward order and backward runs in reverse, so the marks fall out of the build order:
            # after the decoder + post-encoder BN (off = layers.1), after encoder stage 7, 6, 5, 4 (off = first conv).
            self.bwd_marks: List[Tuple[int, int]] = []
            for b in reversed(bwd_layers):
                b()
                if getattr(b, "is_encoder_boundary", False):
                    self.bwd_marks.append((len(self.bwd_ops), self.layout.by_name[self.spec.post_bn + ".weight"].offset))
                if getattr(b, "ar_mark", None):
                    self.bwd_marks.append((len(self.bwd_ops), self.layout.by_name[b.ar_mark].offset))
            ws_bytes = max(sp["bytes"] for sp in self._wgrad_specs)
            self._wgrad_ws = torch.zeros((ws_bytes + 3) // 4, dtype=torch.float32, device=dev)
            self._wgrad_plans = []
            for sp in self._wgrad_specs:
                cs = sp["cs"]
                self._wgrad_plans.append(WgradPlan(sp["dy_view"], sp["views"], sp["taps"], cs.nf, sp["cin"], cs.ks * cs.ks,
                                                   sp["kidx"], sp["dw"].reshape(-1), sp["db"], sp["row_perm"],
                                                   sp["alpha"], self._wgrad_ws))
        self.feats = feats

    # ------------------------------------------------------------------------------------------------ execution
    def set_input(self, x: torch.Tensor, stream: Optional[int] = None) -> None:
        """x: [N, n_in, H, W] on the device — fp32 already scaled (the reference's x = raw/255, data.py:24 +
        IntToFloatTensor) or raw uint8 / uint16 / int16 band values, divided in the kernel as `input_contract` says."""
        assert x.is_cuda and x.is_contiguous() and tuple(x.shape) == (self.N, self.n_in, self.H, self.W), x.shape
        dt, div, div2 = input_contract(x.dtype, self.input_div)
        s = stream if stream is not None else ops.stream_ptr()
        _lib.check(self.lib.b2u_nchw_to_nhwc(x.data_ptr(), dt, div, div2, self.x_in.t.data_ptr(), self.N,
                                             self.n_in, self.H, self.W, self.x_in.ld, 0, self.x_in.ld, s),
                   "b2u_nchw_to_nhwc")

    def set_labels(self, y: torch.Tensor) -> None:
        assert self.training and tuple(y.shape) == (self.N, self.H, self.W)
        self.labels.copy_(y if y.dtype == self.labels.dtype else y.to(self.labels.dtype), non_blocking=True)

    def forward(self, stream: Optional[int] = None) -> torch.Tensor:
        """Runs the forward plan; returns the fp32 NHWC logits buffer [N,H,W,ld] (first n_out lanes valid)."""
        s = stream if stream is not None else ops.stream_ptr()
        for op in self.fwd_ops:
            op(s)
        return self.logits

    def loss_and_grad(self, stream: Optional[int] = None, grad_scale: float = 1.0) -> torch.Tensor:
        s = stream if stream is not None else ops.stream_ptr()
        lib, P_ = self.lib, self.N * self.H * self.W
        ld = self.logits.shape[-1]
        if self.regression:
            # MSELossFlat(axis=1) (train.py:189-192): mean squared error over the flattened batch
            _lib.check(lib.b2u_mse_fwd_bwd(self.logits.data_ptr(), ld, self.labels.data_ptr(), P_, self.dlogits.data_ptr(),
                                           self.dlogits.shape[-1], self._loss_part.data_ptr(), self._ce_rows, grad_scale,
                                           s), "b2u_mse_fwd_bwd")
            _lib.check(lib.b2u_mse_finalize(self._loss_part.data_ptr(), self._ce_rows, P_, self.loss.data_ptr(), s),
                       "b2u_mse_finalize")
            return self.loss
        if self.loss_spec.name != "ce":
            # FocalLossFlat / DiceLoss (losses.py): one fused pass, or Dice statistics + backward
            launch_loss(lib, self.loss_spec, self.logits, self.labels, self.N, self.H * self.W, self.n_out,
                        _p(self.class_weights), self.dlogits.data_ptr(), self.dlogits.shape[-1], self._loss_part,
                        self._ce_rows, self._dice_part, self._dice_bps, self.loss, grad_scale, s)
            return self.loss
        _lib.check(lib.b2u_ce_weight_sum(self.labels.data_ptr(), P_, _p(self.class_weights), self.n_out,
                                         self._wsum_part.data_ptr(), self._ce_rows, s), "b2u_ce_weight_sum")
        _lib.check(lib.b2u_ce_fwd_bwd(self.logits.data_ptr(), ld, self.labels.data_ptr(), P_, self.n_out,
                                      _p(self.class_weights), self._wsum_part.data_ptr(), self._ce_rows,
                                      self.dlogits.data_ptr(), self.dlogits.shape[-1], self._loss_part.data_ptr(),
                                      self._ce_rows, grad_scale, s), "b2u_ce_fwd_bwd")
        _lib.check(lib.b2u_ce_finalize(self._loss_part.data_ptr(), self._ce_rows, self._wsum_part.data_ptr(),
                                       self._ce_rows, self.loss.data_ptr(), s), "b2u_ce_finalize")
        return self.loss

    def backward(self, stream: Optional[int] = None, begin: int = 0, end: Optional[int] = None) -> None:
        """Runs the backward plan (ops [begin, end): the engine splits it at `bwd_split` to overlap the gradient
        all-reduce of the decoder with the encoder's backward).  The critical path is the chain of activation gradients (BN backward -> dgrad -> ...);
        the weight gradients (wgrad GEMM + split-K reduce) hang off it as leaves, so they are issued on a second stream:
        each one waits for the ops recorded before it and the streams join before the optimizer.  The small encoder
        layers are latency-bound single-wave launches - the two streams fill each other's ramp-up and tail bubbles.
        (Works the same under CUDA-graph capture: the fork/join become graph edges.)"""
        main = torch.cuda.current_stream()
        s = stream if stream is not None else main.cuda_stream
        two = (SIDE_STREAM_WGRAD and ops.PROFILE is None and s == main.cuda_stream)
        end = len(self.bwd_ops) if end is None else end
        if not two:
            for op in self.bwd_ops[begin:end]:
                op(s)
            return
        if self._side_stream is None:
            # (both streams at the default priority: raising either one measured slower - 21.6 / 24.0 vs 20.4 ms/step)
            self._side_stream = torch.cuda.Stream(device=self.device)
        side = self._side_stream
        ss = side.cuda_stream
        pending = False   # main-stream work issued since the last fork: the next side op must wait for it
        first = True
        for op, is_side in zip(self.bwd_ops[begin:end], self.bwd_side[begin:end]):
            if is_side:
                if pending or first:
                    ev = torch.cuda.Event()
                    ev.record(main)
                    side.wait_event(ev)
                    pending, first = False, False
                op(ss)
            else:
                op(s)
                pending = True
        main.wait_stream(side)

    def sgd_step(self, lr: float, stream: Optional[int] = None) -> None:
        s = stream if stream is not None else ops.stream_ptr()
        _lib.check(self.lib.b2u_sgd_step(self.params.data_ptr(), self.grads.data_ptr(), self.layout.total, lr, 1.0, s),
                   "b2u_sgd_step")
        self._stage_weights(s)

    def logits_nchw(self) -> torch.Tensor:
        out = torch.empty((self.N, self.n_out, self.H, self.W), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.b2u_nhwc_to_nchw_f32(self.logits.data_ptr(), 1, self.logits.shape[-1], out.data_ptr(),
                                                 self.N, self.n_out, self.H, self.W, ops.stream_ptr()),
                   "b2u_nhwc_to_nchw_f32")
        return out

    def named_grads(self) -> Dict[str, torch.Tensor]:
        return {e.name: self.grad(e.name) for e in self.layout.entries}

    @property
    def launches_per_train_step(self) -> int:
        # forward + loss (CE and Dice 3, focal 2) + backward + optimizer (1) + weight staging (1)
        return self.launches_fwd + (2 if self.loss_spec.name == "focal" else 3) + self.launches_bwd + 2
