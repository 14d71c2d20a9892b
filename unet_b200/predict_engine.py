"""Tiled prediction of a large raster on the GPU: crop -> forward (BN folded) -> softmax -> overlap accumulate ->
normalise + argmax, sharded over GPUs by output column strips.

Replaces the reference's `save_predictions` hot loops (predict.py:191-254 per-tile `learn.predict`, predict.py:284-337
numpy merge): the reference keeps every tile's probabilities in a host list and merges with numpy slicing; here tiles
never leave HBM between the network and the stitch.
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import torch

from . import _lib, ops
from .network import UNetB200, input_contract
from .tiling import colour_classes, compute_windows, shard_windows_2d, shard_windows_by_columns, split_range


def gather_mask_strips(strip: torch.Tensor, width: int, rank: int, world: int, dst: int = 0) -> Optional[torch.Tensor]:
    """The only collective of the prediction path (SURVEY.md 8(e)): the uint8 column strips every rank owns are gathered
    on rank `dst` into the full `[Y, width]` mask (NCCL over NVLink on GPUs, gloo on CPU).  Strips are the balanced
    column partition of `shard_windows_by_columns`; they are padded to the widest strip for the all_gather."""
    import torch.distributed as dist
    if world == 1:
        return strip
    Y = strip.shape[0]
    widest = split_range(width, world, 0)[1]          # the first part is the widest
    # all_gather of column-major strips: [widest, Y] rows are contiguous columns of the mask
    buf = torch.zeros((widest, Y), dtype=strip.dtype, device=strip.device)
    buf[:strip.shape[1]] = strip.t()
    parts = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(parts, buf)
    if rank != dst:
        return None
    cols = []
    for r in range(world):
        xb, xe = split_range(width, world, r)
        cols.append(parts[r][:xe - xb])
    return torch.cat(cols, 0).t().contiguous()


def gather_mask_cells(cell: torch.Tensor, height: int, width: int, grid: Tuple[int, int], rank: int, world: int,
                      dst: int = 0) -> Optional[torch.Tensor]:
    """the 2-D counterpart of `gather_mask_strips`: the uint8 cells of a gx x gy ownership grid (`tiling.shard_windows_2d`)
    are all-gathered (padded to the largest cell) and assembled into the full [height, width] mask on rank `dst`"""
    import torch.distributed as dist
    if world == 1:
        return cell
    gx, gy = grid
    hmax, wmax = split_range(height, gy, 0)[1], split_range(width, gx, 0)[1]     # the first parts are the largest
    buf = torch.zeros((hmax, wmax), dtype=cell.dtype, device=cell.device)
    buf[:cell.shape[0], :cell.shape[1]] = cell
    parts = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(parts, buf)
    if rank != dst:
        return None
    full = torch.empty((height, width), dtype=cell.dtype, device=cell.device)
    for r in range(world):
        xb, xe = split_range(width, gx, r % gx)
        yb, ye = split_range(height, gy, r // gx)
        full[yb:ye, xb:xe] = parts[r][:ye - yb, :xe - xb]
    return full


def finalize_probs(acc: torch.Tensor, cnt: torch.Tensor, c0: int, nc: int, x0: int, w: int, large_file: bool,
                   stream: int) -> torch.Tensor:
    """the averaged probabilities of classes [c0, c0 + nc) over columns [x0, x0 + w) of stitch accumulators (`acc` fp32
    [C, SY, SX] and `cnt` uint8 [SY, SX] of a `StitchPlan` in mode 0, or mode 1 with `large_file`), as the device tensor
    [SY, w, nc] the bands of a striped GeoTIFF are stored in: float32 acc / cnt, or with `large_file` the reference's
    int8 merge (sums wrapped to int8, floor-divided by the count); 0 where no tile was placed"""
    C, SY, SX = acc.shape
    out = torch.empty((SY, w, nc), dtype=torch.int8 if large_file else torch.float32, device=acc.device)
    _lib.check(_lib.load().b2u_stitch_finalize_probs(acc.data_ptr(), cnt.data_ptr(), C, SY, SX, c0, nc, x0, w,
                                                     int(large_file), out.data_ptr(), w * nc, stream),
               "b2u_stitch_finalize_probs")
    return out


class StitchPlan:
    """The overlap stitching of one job's predicted tiles into the output rectangle `region` = (yb, ye, xb, xe) of the
    raster: per batch of tiles the network has just run, one `b2u_stitch_accumulate` launch per colour class adds the
    tiles into `acc` (fp32 [n_out, ye-yb, xe-xb]) and `cnt` (uint8 [ye-yb, xe-xb]); `mask` / `mean` finalize them.
    mode 0: softmax probabilities, 1: the reference's int8 `large_file` merge (x31, floor division), 2: the raw
    network output (regression).  `origins[i][:2]` is the (x, y) of tile i of the raster; `batches[b]` lists the tiles
    of batch b in batch order (at most net.N).
    Per-batch metadata block (int32): y0[B] x0[B], then one (count, sel[B]) slot per colour class, as many slots as the
    batch with the most classes needs (tiles overlapping beyond their direct neighbours need more than 2 x 2).  The
    blocks of the whole job go to the device in ONE copy: a small pageable host-to-device copy per batch would block
    the host behind the previous batch's kernels every time (measured on the 20000 x 20000 raster: 10.08k -> 10.46k
    tiles/s); `load` refills the current block device-to-device in front of the batch."""

    def __init__(self, net: UNetB200, origins: Sequence[Sequence[int]], batches: Sequence[Sequence[int]],
                 region: Tuple[int, int, int, int], mode: int):
        B, P = net.N, net.H
        self.net, self.mode = net, mode
        self.yb, ye, self.xb, xe = region
        self.SY, self.SX = ye - self.yb, xe - self.xb
        classes = [colour_classes([(origins[i][0], origins[i][1], P, P) for i in idx]) for idx in batches]
        self.n_classes = max((len(c) for c in classes), default=0)
        blk = 2 * B + self.n_classes * (1 + B)
        host = torch.zeros((max(1, len(batches)), blk), dtype=torch.int32)
        for row, idx, cls_b in zip(host, batches, classes):
            pad = list(idx) + [idx[0]] * (B - len(idx))      # padded tiles are never selected for stitching
            row[:B] = torch.tensor([origins[i][1] for i in pad], dtype=torch.int32)
            row[B:2 * B] = torch.tensor([origins[i][0] for i in pad], dtype=torch.int32)
            for k, cls in enumerate(cls_b):
                o = 2 * B + k * (1 + B)
                row[o] = len(cls)
                row[o + 1:o + 1 + len(cls)] = torch.tensor(cls, dtype=torch.int32)
        self.meta = host.to(net.device)
        self.cur = torch.zeros(blk, dtype=torch.int32, device=net.device)
        self.acc = torch.zeros((net.n_out, self.SY, self.SX), dtype=torch.float32, device=net.device)
        self.cnt = torch.zeros((self.SY, self.SX), dtype=torch.uint8, device=net.device)

    def load(self, b: int) -> Tuple[int, int]:
        """makes batch b's block current (a device copy on the current stream, which the plan's launches must use too);
        returns the device pointers of its tile rows y0[B] and x0[B]"""
        self.cur.copy_(self.meta[b], non_blocking=True)
        cb = self.cur.data_ptr()
        return cb, cb + 4 * self.net.N

    def accumulate(self, stream: int) -> None:
        """adds the current batch's tiles, as the network left them in its logits, into the accumulators"""
        net, B, P = self.net, self.net.N, self.net.H
        cb = self.cur.data_ptr()
        for k in range(self.n_classes):
            o = cb + 4 * (2 * B + k * (1 + B))
            _lib.check(net.lib.b2u_stitch_accumulate(net.logits.data_ptr(), net.logits.shape[-1], net.n_out, B, P, P, cb,
                                                     cb + 4 * B, o + 4, o, B, self.mode, self.acc.data_ptr(),
                                                     self.cnt.data_ptr(), self.SY, self.SX, self.yb, self.xb, stream),
                       "b2u_stitch_accumulate")

    def mask(self, stream: int) -> torch.Tensor:
        """the stitched argmax, uint8 [SY, SX] (unplaced pixels 0)"""
        out = torch.empty((self.SY, self.SX), dtype=torch.uint8, device=self.acc.device)
        _lib.check(self.net.lib.b2u_stitch_finalize(self.acc.data_ptr(), self.cnt.data_ptr(), self.net.n_out, self.SY,
                                                    self.SX, int(self.mode == 1), out.data_ptr(), stream),
                   "b2u_stitch_finalize")
        return out

    def mean(self, nodata: float, stream: int) -> torch.Tensor:
        """the overlap average, fp32 [n_out, SY, SX], `nodata` where no tile was placed"""
        out = torch.empty_like(self.acc)
        _lib.check(self.net.lib.b2u_stitch_finalize_mean(self.acc.data_ptr(), self.cnt.data_ptr(), self.net.n_out,
                                                         self.SY, self.SX, float(nodata), out.data_ptr(), stream),
                   "b2u_stitch_finalize_mean")
        return out


class TiledPredictor:
    def __init__(self, net: UNetB200):
        assert not net.training, "prediction uses the eval plan (running BN statistics folded into the convolutions)"
        self.net, self.lib, self.dev = net, net.lib, net.device
        self.B, self.P = net.N, net.H
        assert net.H == net.W

    def predict_raster(self, raster: torch.Tensor, patch_overlap: float, rank: int = 0, world: int = 1,
                       return_probs: bool = False, large_file: bool = False, grid: Optional[Tuple[int, int]] = None):
        """raster: uint8 / uint16 / int16 [C, Y, X] on the device (raw band values, scaled by the plan's input contract).
        Returns (mask uint8 [Y, x_end-x_begin], x_begin, x_end) for the
        column strip this rank owns (the whole raster when world == 1).  A regression net (`net.regression`) returns the
        overlap mean of its output in place of the mask: fp32, -9999 where no tile was placed (predict.py:307-316).
        With `grid=(gx, gy)` the rank owns cell (rank % gx, rank // gx) of a gx x gy grid instead
        (`tiling.shard_windows_2d`; fewer duplicated tiles at 8 ranks) and the return value is (mask [y_end-y_begin, x_end-x_begin], (x_begin, x_end, y_begin, y_end)).  `large_file`: the
        reference's int8 merge (predict.py:217-219, 318-323).  `return_probs` also returns the accumulators.
        One batch = crop -> forward -> one accumulate per colour class, every launch reading the batch's tile origins /
        class lists from the `StitchPlan`'s device block, refilled (device-to-device) in front of it - no host round trip,
        no per-batch host-to-device copy.  (Replaying the batch as a captured CUDA graph was measured and dropped: with
        programmatic dependent launch the eager launches already overlap, 5.86 vs 6.07 ms per batch of 64 tiles.)"""
        net, lib, P, B = self.net, self.lib, self.P, self.B
        assert raster.is_cuda and raster.dim() == 3 and raster.is_contiguous()
        r_dt, r_div, r_div2 = input_contract(raster.dtype, net.input_div)
        Cc, Y, X = raster.shape
        assert Cc == net.n_in and Y >= P and X >= P, "raster smaller than one tile is not supported"
        windows = compute_windows(Y, X, P, patch_overlap)
        if grid is None:
            idx, xb, xe = shard_windows_by_columns(windows, X, rank, world)
            yb, ye = 0, Y
        else:
            idx, (xb, xe, yb, ye) = shard_windows_2d(windows, X, Y, rank, world, grid)
        self.tiles_run = len(idx)
        batches = [idx[b0:b0 + B] for b0 in range(0, len(idx), B)]
        plan = StitchPlan(net, windows, batches, (yb, ye, xb, xe), 2 if net.regression else 1 if large_file else 0)
        self._keep = plan           # its device blocks are read by launches still in flight when this returns
        s = ops.stream_ptr()
        for b in range(len(batches)):
            y0, x0 = plan.load(b)
            _lib.check(lib.b2u_crop_tiles(raster.data_ptr(), r_dt, r_div, r_div2, Cc, Y, X, y0, x0, B, P,
                                          net.x_in.t.data_ptr(), net.x_in.ld, s), "b2u_crop_tiles")
            net.forward(s)
            plan.accumulate(s)
        mask = plan.mean(-9999, s)[0] if net.regression else plan.mask(s)
        self.last_stitch_profile = {"batches": len(batches), "tiles_run": len(idx),
                                    "launches_per_batch": 1 + net.launches_fwd + plan.n_classes + 1}
        if grid is not None:
            return (mask, (xb, xe, yb, ye), plan.acc, plan.cnt) if return_probs else (mask, (xb, xe, yb, ye))
        if return_probs:
            return mask, xb, xe, plan.acc, plan.cnt
        return mask, xb, xe

    def _forward_tiles(self, tiles: torch.Tensor) -> int:
        T = tiles.shape[0]
        assert T <= self.B
        x = tiles
        if T < self.B:
            x = torch.cat([tiles, tiles[:1].expand(self.B - T, -1, -1, -1)], 0).contiguous()
        self.net.set_input(x)
        self.net.forward()
        return T

    def predict_tiles_raw(self, tiles: torch.Tensor) -> torch.Tensor:
        """the regression variant's `Learner_adjust.predict` (train.py:87-95): the network output itself, [T,1,H,W] fp32"""
        T = self._forward_tiles(tiles)
        return self.net.logits_nchw()[:T]

    def predict_tiles(self, tiles_u8: torch.Tensor):
        """what `learn.predict` returns per tile (predict.py:193-203): softmax probabilities [T,C,H,W] fp32 and the
        argmax [T,H,W] uint8, for a batch of uint8 tiles [T<=B, C, P, P] on the device."""
        net, lib = self.net, self.lib
        T = tiles_u8.shape[0]
        assert T <= self.B
        x = tiles_u8
        if T < self.B:
            x = torch.cat([tiles_u8, tiles_u8[:1].expand(self.B - T, -1, -1, -1)], 0).contiguous()
        net.set_input(x)
        net.forward()
        probs = torch.empty((self.B, net.n_out, self.P, self.P), dtype=torch.float32, device=self.dev)
        amax = torch.empty((self.B, self.P, self.P), dtype=torch.uint8, device=self.dev)
        _lib.check(lib.b2u_softmax_nchw(net.logits.data_ptr(), net.logits.shape[-1], net.n_out, self.B, self.P, self.P,
                                        probs.data_ptr(), amax.data_ptr(), ops.stream_ptr()), "b2u_softmax_nchw")
        return probs[:T], amax[:T]
