#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native U-Net hot path.

Workload (BASELINE.json configs[1]): xresnet34-DynamicUnet, 4-band 256x256 tiles, 2 classes, bf16 data-parallel
training, batch 64 per GPU; one "step" = H2D of a tile batch -> forward -> weighted CE -> backward -> (N>1: NCCL
gradient all-reduce) -> SGD update -> bf16 weight re-staging.  Metric: train tiles/s (whole job) and the fraction of
the measured bf16 tensor-core peak reached by the implicit-GEMM kernel.

    python bench.py --gpus N --steps K --warmup W           (N>1: launched by torch.distributed.run, one rank per GPU)
    python bench.py --impl reference ...                    (the reference's CPU path = fp32 torch oracle, host cores)
    python bench.py --dump-outputs DIR ...                  (also writes what the last timed step computed, DIR/*.npy)

Prints ONE JSON line on rank 0 (schema in the task contract; extra keys: roofline, cpu_baseline, e2e, gpu_launches,
clocks, kernels).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ARCH, N_IN, N_OUT, SIZE = "xresnet34", 4, 2, 256
METRIC = "train tiles/sec (256x256x4-band xresnet34-DynamicUnet, bf16, batch 64/GPU)"
UNIT = "tiles/s"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "tf_burst": p["bf16_tflops"], "tf_sustained": p["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (recipe's clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float = 0.0, t1: float = float("inf")):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if ts < t0 or ts > t1 + 0.15:   # only samples taken DURING the timed region
                continue
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            try:
                pw.append(float(parts[2]))
            except ValueError:
                pass
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        pw.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w": pw[len(pw) // 2] if pw else None}


def cpu_oracle_step_time(batch: int, steps: int, warmup: int):
    """The reference's CPU path: fp32 torch restatement (oracle/), fwd + weighted CE + bwd + SGD, all host threads."""
    from oracle.unet_oracle import make_oracle, sgd_step, weighted_ce
    from unet_b200.synth import uniform_tiles
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    m = make_oracle(ARCH, N_IN, N_OUT).train()
    x, y = uniform_tiles(batch, N_IN, SIZE, SIZE, N_OUT)
    x = x.float() / 255.0
    y = y.long()
    w = torch.full((N_OUT,), 1.0 / N_OUT)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        for p in m.parameters():
            p.grad = None
        loss = weighted_ce(m(x), y, w)
        loss.backward()
        sgd_step(m.parameters(), 1e-3)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return sum(times) / len(times), cores, float(loss.detach())


def run_reference(args, rank: int, out):
    """--impl reference: the reference's own CPU implementation of the path (oracle port) on the host cores."""
    if rank != 0:
        return
    # bounded sample of the batch-64 workload: probe with batch 2, then size the sample for <= ~150 s in total
    t_probe, cores, _ = cpu_oracle_step_time(2, 1, 1)
    per_tile = t_probe / 2
    budget = 150.0
    total_steps = args.steps + args.warmup
    sample = int(max(1, min(64, budget / max(per_tile * total_steps, 1e-9))))
    t_step, cores, _ = cpu_oracle_step_time(sample, args.steps, args.warmup)
    tiles_s = sample / t_step
    line = {
        "impl": "reference", "metric": METRIC, "value": tiles_s, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t_step * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "xresnet34-DynamicUnet 4-band 256x256 train step (fwd+CE+bwd+SGD), CPU fp32",
                   "tile": SIZE, "bands": N_IN, "classes": N_OUT, "batch_per_step": sample},
        "cpu_baseline": {"value": tiles_s, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{sample} tiles per step of the batch-64 workload, {args.steps} timed steps"},
        "e2e": {"value": tiles_s, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), file=out, flush=True)


def _guard_stdout():
    """The driver parses ONE JSON line from stdout; libraries (NCCL prints its version banner there) must not share
    it.  fd 1 is pointed at stderr for the whole run and the saved descriptor is used for the result line only."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(saved, "w")


def load_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture (newest profiles/rNN_traffic.json;
    ncu cannot run inside the timed bench, so this one field is read from the evidence file of the same code)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(path):
            with open(path) as f:
                d = json.load(f)
            d["file"] = "profiles/" + name
            return d
    return None


def load_secondary_bar():
    """stock torch + cuDNN (bf16 autocast, channels_last) on the same B200, same network / batch: tools/torch_baseline.py,
    recorded in profiles/ (the oracle module may not run inside this file outside the cpu_baseline leg)."""
    path = os.path.join(ROOT, "profiles", "r02_torch_cudnn_baseline.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return None


def profile_step(net, trainer, x, y):
    """One eager training step with a CUDA-event pair around EVERY op (real order, warm caches).  Returns
    [(kind, algorithmic bytes, ms)] of the memory-bound ops (network.py registers kind / bytes per op)."""
    from unet_b200 import ops
    st = torch.cuda.current_stream()
    s = ops.stream_ptr()
    trainer.x_static.copy_(x)
    net.labels.copy_(y)
    evs = []

    def timed(fn, meta):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        fn()
        b.record(st)
        evs.append((meta, a, b))

    timed(lambda: net.set_input(trainer.x_static, s), ("nchw_to_nhwc", net.N * net.H * net.W * (net.n_in + net.x_in.ld * 2)))
    for op, meta in zip(net.fwd_ops, net.fwd_meta):
        timed(lambda op=op: op(s), meta)
    P_ = net.N * net.H * net.W
    timed(lambda: net.loss_and_grad(s), ("ce_weight_sum+ce_fwd_bwd+ce_finalize",
                                         P_ * (net.logits.shape[-1] * 4 + 2 + net.dlogits.shape[-1] * 2)))
    for op, meta in zip(net.bwd_ops, net.bwd_meta):
        timed(lambda op=op: op(s), meta)
    timed(lambda: net.sgd_step(1e-3, s), ("sgd+stage_weights", net.layout.total * 12 + net.layout.total * 4))
    torch.cuda.synchronize()
    return [(m[0], m[1], a.elapsed_time(b)) for m, a, b in evs if m[0]]


def predict_section(dev, rank, world, side, batch, max_over_ranks, barrier, peaks):
    """The other half of BASELINE's metric: tiled prediction (256x256 tiles, 32-px overlap, overlap-average + argmax) of
    a synthetic 4-band raster, tiles sharded over the ranks by output column strips.  `value`: raster resident in HBM;
    `e2e`: the raster strip comes from pinned host memory and the uint8 mask strip is read back, inside the timed region."""
    from unet_b200.network import UNetB200
    from unet_b200.predict_engine import TiledPredictor, gather_mask_cells
    from unet_b200.tiling import compute_windows, shard_grid, shard_windows_2d
    net = UNetB200(ARCH, N_IN, N_OUT, (SIZE, SIZE), batch, training=False, device=dev)
    net.init_parameters(seed=0)
    pred = TiledPredictor(net)
    g = torch.Generator(device=dev).manual_seed(1234)
    raster = torch.randint(0, 256, (N_IN, side, side), dtype=torch.uint8, device=dev, generator=g)
    windows = compute_windows(side, side, SIZE, 0.125)
    n_tiles = len(windows)
    grid = shard_grid(windows, side, side, world)          # ownership grid of the output: strips up to 4 ranks, 4 x 2 at 8
    pred.predict_raster(raster[:, :1024, :1024].contiguous(), 0.125)   # warm-up
    pred.predict_raster(raster, 0.125, rank, world, grid=grid)         # second warm-up at full size (allocator, caches)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    mask, rect = pred.predict_raster(raster, 0.125, rank, world, grid=grid)
    full = gather_mask_cells(mask, side, side, grid, rank, world)       # the path's only collective (NCCL all-gather)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    stitch = pred.last_stitch_profile
    tiles_max = int(max_over_ranks(float(stitch["tiles_run"])))
    # e2e: this rank's part of the raster (the tiles it runs) from pinned host memory, its mask cell back to the host
    idx, (xb, xe, yb, ye) = shard_windows_2d(windows, side, side, rank, world, grid)
    xs0, xs1 = min(windows[i][0] for i in idx), max(windows[i][0] + windows[i][2] for i in idx)
    ys0, ys1 = min(windows[i][1] for i in idx), max(windows[i][1] + windows[i][3] for i in idx)
    host = raster[:, ys0:ys1, xs0:xs1].contiguous().cpu().pin_memory()
    host_mask = torch.empty((ye - yb, xe - xb), dtype=torch.uint8).pin_memory()
    barrier()
    t0 = time.perf_counter()
    part = host.to(dev, non_blocking=True)
    # the part holds exactly this rank's tiles: a 1-rank prediction of it, cropped to the owned cell
    m2, _, _ = pred.predict_raster(part, 0.125, 0, 1)
    m2 = m2[yb - ys0:ye - ys0, xb - xs0:xe - xs0]
    host_mask.copy_(m2, non_blocking=True)
    torch.cuda.synchronize()
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    same = bool(torch.equal(m2, mask))
    flops = n_tiles * net.flops_fwd_per_tile
    return {"metric": "predict tiles/sec (256x256x4-band xresnet34-DynamicUnet, bf16, tiled predict + stitch + argmax)",
            "workload": f"BASELINE configs[2]: {side}x{side} 4-band raster, 256-px tiles, 32-px overlap: {n_tiles} tiles, "
                        f"owner-computes {grid[0]} x {grid[1]} grid of output cells over {world} GPU(s) (tiles on a cell border run "
                        f"on both sides: {tiles_max} tiles on the fullest rank), final uint8 mask all-gather inside the timed region",
            "value": n_tiles / (ms * 1e-3), "unit": UNIT, "seconds": ms * 1e-3, "tiles": n_tiles,
            "tiles_run_max_rank": tiles_max, "ownership_grid": list(grid), "fwd_gflop_per_tile": net.flops_fwd_per_tile / 1e9,
            "algorithmic_tflops_per_gpu": flops / (ms * 1e-3) / 1e12 / world,
            "tensor_core_frac_of_burst_peak": flops / (ms * 1e-3) / 1e12 / world / peaks["tf_burst"],
            "stitch_kernels": stitch,
            "e2e": {"value": n_tiles / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes": host.numel() * world,
                    "d2h_bytes": host_mask.numel() * world, "part_mask_equals_sharded_mask": same}}


DUMP_SAMPLE = 1 << 20        # elements kept of each parameter-sized vector (4 MB as float32)
DUMP_LOGITS_MAX = 8 << 20    # logits kept whole up to 32 MB (batch 64 x 2 x 256 x 256), sampled beyond


def _seeded_sample(t: torch.Tensor, k: int, seed: int) -> torch.Tensor:
    """t flattened, or k of its elements at indices drawn from a fixed seed: the same indices on every run and build"""
    flat = t.reshape(-1)
    if flat.numel() <= k:
        return flat
    idx = torch.randint(0, flat.numel(), (k,), generator=torch.Generator().manual_seed(seed))
    return flat[idx.to(flat.device)]


def dump_outputs(path: str, net) -> None:
    """What a caller of the timed training step holds after its last step, as float32 .npy files (about 40 MB in all):
    the loss the step returns, the logits of its forward pass, and a fixed sample of the parameters after its update
    and of its gradients.  Parameters and gradients are taken in the oracle's parameter order, not the plan's flat
    layout, so that two builds of the project can be compared output for output."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    logits = net.logits_nchw()
    names = [e.name for e in net.layout.entries]
    params = torch.cat([net.param(n).reshape(-1) for n in names])
    grads = torch.cat([net.grad(n).reshape(-1) for n in names])
    arrays = {"loss": net.loss,
              "logits": logits if logits.numel() <= DUMP_LOGITS_MAX else _seeded_sample(logits, DUMP_LOGITS_MAX, 1),
              "params_sample": _seeded_sample(params, DUMP_SAMPLE, 2),
              "grads_sample": _seeded_sample(grads, DUMP_SAMPLE, 3)}
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())


def plan_bytes(plan) -> int:
    """algorithmic bytes of one implicit-GEMM launch: activations in (every view once), weights, residual / mask
    operands, output - all bf16 at their unpadded channel counts (fp32 for the head's logits)"""
    d = plan.desc
    px_out = d.out.N * d.out.H * d.out.W
    b = 0
    for i in range(d.num_a):
        b += d.a[i].N * d.a[i].H * d.a[i].W * d.w_cin * 2
    b += d.w_rows * d.num_taps * d.w_cin * 2
    for v in (d.res, d.res_mask, d.zmask):
        if v.ptr:
            b += px_out * d.out.C * 2
    b += px_out * d.out.C * (4 if d.out_f32 else 2)
    return b


def extra_configs(dev, rank, world, args, peaks, max_over_ranks, barrier):
    """BASELINE configs[3] and configs[4] as sub-records of the one JSON line (every rank runs its own replica of the
    per-GPU workload; values are whole-job aggregates): xresnet50-DynamicUnet 4-band 512x512, 8 classes, bf16 training
    with batch statistics (fwd + CE + bwd + SGD, CUDA graph), and xresnet18-DynamicUnet 3-band 128x128 inference at
    batch 512 per GPU (eval plan, BN folded) - the memory-bound kernel stress."""
    from unet_b200.engine import Trainer
    from unet_b200.network import UNetB200
    from unet_b200.synth import uniform_tiles
    out = {}
    # ---- configs[3]: R50 / 512 / 8 classes, training
    try:
        B = args.r50_batch
        net = UNetB200("xresnet50", 4, 8, (512, 512), B, training=True, device=dev)
        net.init_parameters(seed=0)
        tr = Trainer(net, optimizer="sgd", lr=1e-3, use_graph=True)
        x, y = uniform_tiles(B, 4, 512, 512, 8, seed=99 + rank)
        x, y = x.to(dev), y.to(dev)
        for _ in range(3):
            tr.step(x, y)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        steps = 5
        e0.record()
        for _ in range(steps):
            tr.step(x, y)
        e1.record()
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1)) / steps
        tf = 3 * net.flops_fwd_per_tile * B / (ms * 1e-3) / 1e12
        out["config4_xresnet50_512_train"] = {
            "workload": "BASELINE configs[3]: xresnet50-DynamicUnet 4-band 512x512, 8 classes, train-mode BN, bf16, "
                        f"batch {B}/GPU, fwd+CE+bwd+SGD (CUDA graph)", "value": B * world / (ms * 1e-3), "unit": UNIT,
            "ms_per_step": ms, "steps": steps, "warmup": 3, "batch_per_gpu": B,
            "train_gflop_per_tile": 3 * net.flops_fwd_per_tile / 1e9, "algorithmic_tflops_per_gpu": tf,
            "tensor_core_frac_of_burst_peak": tf / peaks["tf_burst"], "final_loss": float(net.loss.item()),
            "gpu_launches_per_step": net.launches_per_train_step}
        del tr, net, x, y
    except Exception as ex:   # e.g. out of memory on a smaller part: reported, never hidden
        out["config4_xresnet50_512_train"] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
    torch.cuda.empty_cache()
    # ---- the reference's DEFAULT model (params_and_main.py:83 self_attention=True): BASELINE configs[1] with fastai's
    # SelfAttention block on UnetBlock #1 (1 024 positions at 256-px tiles), training, same batch
    try:
        B = args.batch
        net = UNetB200(ARCH, N_IN, N_OUT, (SIZE, SIZE), B, training=True, self_attention=True, device=dev)
        net.init_parameters(seed=0)
        tr = Trainer(net, optimizer="sgd", lr=1e-3, use_graph=True)
        x, y = uniform_tiles(B, N_IN, SIZE, SIZE, N_OUT, seed=199 + rank)
        x, y = x.to(dev), y.to(dev)
        for _ in range(3):
            tr.step(x, y)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        steps = 10
        e0.record()
        for _ in range(steps):
            tr.step(x, y)
        e1.record()
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1)) / steps
        out["config2_self_attention_train"] = {
            "workload": f"BASELINE configs[1] with self_attention=True (the reference's default): {ARCH}-DynamicUnet "
                        f"{N_IN}-band {SIZE}x{SIZE}, bf16, batch {B}/GPU, fwd+CE+bwd+SGD (CUDA graph); attention products "
                        "on the implicit-GEMM kernel", "value": B * world / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
            "steps": steps, "warmup": 3, "batch_per_gpu": B, "final_loss": float(net.loss.item()),
            "gpu_launches_per_step": net.launches_per_train_step}
        del tr, net, x, y
    except Exception as ex:
        out["config2_self_attention_train"] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
    torch.cuda.empty_cache()
    # ---- configs[4]: R18 / 128 / 3-band, batch 512 inference
    try:
        B = 512
        net = UNetB200("xresnet18", 3, 2, (128, 128), B, training=False, device=dev)
        net.init_parameters(seed=0)
        x, _ = uniform_tiles(B, 3, 128, 128, 2, seed=7 + rank)
        x = x.to(dev)
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            net.set_input(x)
            net.forward()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=side):
            net.set_input(x)
            net.forward()
        for _ in range(3):
            g.replay()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        iters = 20
        e0.record()
        for _ in range(iters):
            g.replay()
        e1.record()
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1)) / iters
        tf = net.flops_fwd_per_tile * B / (ms * 1e-3) / 1e12
        act_bytes = sum(a.t.numel() * 2 for a in net.acts)          # every stored activation written once (+ read once)
        out["config5_xresnet18_128_infer"] = {
            "workload": "BASELINE configs[4]: xresnet18-DynamicUnet 3-band 128x128, batch 512/GPU, inference "
                        "(eval plan, BN folded into the conv epilogues, uint8 tiles in, fp32 logits out, CUDA graph)",
            "value": B * world / (ms * 1e-3), "unit": UNIT, "ms_per_batch": ms, "iters": iters, "warmup": 3,
            "fwd_gflop_per_tile": net.flops_fwd_per_tile / 1e9, "algorithmic_tflops_per_gpu": tf,
            "tensor_core_frac_of_burst_peak": tf / peaks["tf_burst"],
            "activation_bytes_written_per_batch": act_bytes,
            "activation_write_plus_read_gbs": 2 * act_bytes / (ms * 1e-3) / 1e9,
            "hbm_frac_of_measured_peak": 2 * act_bytes / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
            "gpu_launches_per_batch": net.launches_fwd + 1}
        del g, net, x
    except Exception as ex:
        out["config5_xresnet18_128_infer"] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
    torch.cuda.empty_cache()
    return out


def main():
    out = _guard_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b2u", choices=["b2u", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="tiles per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-predict", action="store_true")
    ap.add_argument("--predict-side", type=int, default=20000, help="side of the synthetic raster of the predict section "
                    "(BASELINE configs[2]: 20000)")
    ap.add_argument("--no-extra", action="store_true", help="skip the BASELINE configs[3] / configs[4] sub-records")
    ap.add_argument("--r50-batch", type=int, default=16, help="tiles per GPU per step of the xresnet50 / 512-px line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the loss, logits and a fixed "
                    "sample of the parameters and gradients of the last timed training step (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b2u":
        ap.error("--dump-outputs writes the outputs of the CUDA training step (--impl b2u)")
    args.warmup = max(args.warmup, 3) if args.impl == "b2u" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, out)
        return

    import torch.distributed as dist
    from unet_b200 import ops
    from unet_b200.engine import Trainer, init_distributed
    from unet_b200.network import UNetB200
    from unet_b200.synth import uniform_tiles

    rank, local, world = init_distributed()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    dev = torch.device("cuda", local)
    peaks = load_peaks()
    B = args.batch
    net = UNetB200(ARCH, N_IN, N_OUT, (SIZE, SIZE), B, training=True, device=dev)
    net.init_parameters(seed=0)
    trainer = Trainer(net, optimizer="sgd", lr=1e-3, use_graph=True)

    # synthetic tiles: a pool of distinct batches in pinned host memory (e2e) and resident in HBM (kernel-only value)
    n_pool = 4
    host_x, host_y, dev_x, dev_y = [], [], [], []
    for i in range(n_pool):
        x, y = uniform_tiles(B, N_IN, SIZE, SIZE, N_OUT, seed=1234 + 17 * i + 1000 * rank, label_seed=4321 + i + 1000 * rank)
        host_x.append(x.pin_memory())
        host_y.append(y.pin_memory())
        dev_x.append(x.to(dev))
        dev_y.append(y.to(dev))
    h2d_bytes = host_x[0].numel() + host_y[0].numel()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v: float) -> float:
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    vis = [v for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip().isdigit()]
    sampler = ClockSampler(int(vis[local]) if local < len(vis) else local)    # nvidia-smi counts physical GPUs
    if rank == 0:
        sampler.start()   # started early (nvidia-smi needs ~1 s to produce its first sample); filtered by time below
    # ---- warm-up (includes graph capture)
    for i in range(args.warmup):
        trainer.step(dev_x[i % n_pool], dev_y[i % n_pool])
    barrier()

    # ---- kernel-only value: inputs resident in HBM, CUDA events on the launching stream, max over ranks
    st = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    e0.record(st)
    sync_each = os.environ.get("B2U_BENCH_SYNC_EACH_STEP") is not None     # A/B switch: host waits for every step
    for i in range(args.steps):
        trainer.step(dev_x[i % n_pool], dev_y[i % n_pool])
        if sync_each:
            st.synchronize()
    e1.record(st)
    barrier()
    t_wall1 = time.time()
    dev_ms = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    loss_val = float(net.loss.item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, net)     # before the e2e steps below overwrite the plan's buffers

    # ---- e2e: public API with HOST buffers, H2D of the tiles and D2H of the loss every step inside the timed region
    # (every step copies its own batch from pinned host memory; the copy of batch i+1 is enqueued on a copy stream
    # behind the kernels of step i - `prefetch=` of the public Trainer.step - and the loss of every step is read back)
    nxt = lambda i: (host_x[(i + 1) % n_pool], host_y[(i + 1) % n_pool])
    for i in range(2):
        float(trainer.step(host_x[i % n_pool], host_y[i % n_pool], prefetch=nxt(i)).item())
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        loss = trainer.step(host_x[(i + 2) % n_pool], host_y[(i + 2) % n_pool], prefetch=nxt(i + 2))
        _ = float(loss.item())
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)

    tiles = B * world * args.steps
    value = tiles / (dev_ms * 1e-3)
    e2e_value = tiles / (e2e_ms * 1e-3)

    # ---- roofline of the dominant kernel (implicit-GEMM conv: fprop + dgrad launches), measured live with CUDA events
    kernels = {}
    roofline = None
    roofline_mem = None
    if not args.no_profile:
        ops.PROFILE = []
        trainer.use_graph = False
        for i in range(2):
            trainer.step(dev_x[i % n_pool], dev_y[i % n_pool])
        torch.cuda.synchronize()
        prof, ops.PROFILE = ops.PROFILE, None
        trainer.use_graph = True
        half = len(prof) // 2
        prof = prof[half:]  # second instrumented step only
        for kind in ("conv", "wgrad"):
            rows = [(p.flops, a.elapsed_time(b)) for k, p, a, b in prof if k == kind]
            fl, ms = sum(r[0] for r in rows), sum(r[1] for r in rows)
            kernels[kind] = {"launches": len(rows), "ms": ms, "tflops": fl / (ms * 1e-3) / 1e12 if ms > 0 else None,
                             "share_of_step": ms / (dev_ms / args.steps)}
        c = kernels["conv"]
        tr_ncu = load_traffic()
        conv_plans = [p for k, p, a, b in prof if k == "conv"]
        # algorithmic bytes of a conv launch: every operand once (input views, weights, residual / masks) + the output
        alg_bytes = sum(plan_bytes(p) for p in conv_plans) / max(1, len(conv_plans))
        roofline = {"bound": "tensor", "kernel": "conv_gemm_kernel (fprop+dgrad launches)",
                    "achieved": c["tflops"], "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                    "frac": c["tflops"] / peaks["tf_sustained"],
                    "frac_burst": c["tflops"] / peaks["tf_burst"], "peak_burst": peaks["tf_burst"],
                    "traffic": tr_ncu["conv_gemm_kernel"]["dram_bytes_per_launch"] if tr_ncu else None,
                    "traffic_source": (tr_ncu.get("file", "") + ": " + tr_ncu["source"]) if tr_ncu else None,
                    "algorithmic_flops_per_launch": sum(p.flops for p in conv_plans) / max(1, c["launches"]),
                    "algorithmic_bytes_per_launch": alg_bytes,
                    "avg_launch_ms": c["ms"] / max(1, c["launches"]), "launches_per_step": c["launches"],
                    "peak_source": peaks["source"] + ", sustained figure (kernel timed inside a long step); frac_burst uses the burst figure BASELINE.md's 50 % target is defined on"}
        kernels["wgrad"]["frac_burst"] = kernels["wgrad"]["tflops"] / peaks["tf_burst"]
        # HBM roofline of the memory-bound kernels: algorithmic bytes (inputs once + outputs once) / event time, per kind
        agg = {}
        trainer.use_graph = False
        for kind, nbytes, ms in profile_step(net, trainer, dev_x[0], dev_y[0]):
            a = agg.setdefault(kind, [0, 0, 0.0])
            a[0] += 1; a[1] += nbytes; a[2] += ms
        trainer.use_graph = True
        roofline_mem = [{"kernel": k, "launches": a[0], "algorithmic_bytes": a[1], "ms": a[2],
                         "achieved_gbs": a[1] / (a[2] * 1e-3) / 1e9, "peak_gbs": peaks["hbm_gbs"],
                         "frac": a[1] / (a[2] * 1e-3) / 1e9 / peaks["hbm_gbs"]}
                        for k, a in sorted(agg.items(), key=lambda t: -t[1][2]) if a[2] > 0]

    # ---- whole-step tensor-core fraction from algorithmic FLOPs (fwd + dgrad + wgrad = 3x fwd conv FLOPs, SURVEY 8(d))
    launches_per_step = net.launches_per_train_step
    train_flops_per_tile = 3 * net.flops_fwd_per_tile
    step_tflops = value * train_flops_per_tile / 1e12 / world

    # free the training plan before the other workloads (each builds its own static plan)
    del trainer, net
    torch.cuda.empty_cache()
    predict = None
    if not args.no_predict:
        predict = predict_section(dev, rank, world, args.predict_side, B, max_over_ranks, barrier, peaks)
        torch.cuda.empty_cache()
    extra = None
    if not args.no_extra:
        extra = extra_configs(dev, rank, world, args, peaks, max_over_ranks, barrier)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        t_step, cores, _ = cpu_oracle_step_time(8, 5, 1)
        cpu_baseline = {"value": 8 / t_step, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": "BASELINE config 1: batch 8, fwd+CE+bwd+SGD, fp32 torch oracle, 5 timed steps after 1 warm-up"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "BASELINE configs[1]: xresnet34-DynamicUnet 4-band 256x256, 2 classes, bf16 DP training",
                       "arch": ARCH, "tile": SIZE, "bands": N_IN, "classes": N_OUT, "batch_per_gpu": B,
                       "global_batch": B * world, "optimizer": "sgd", "parallelism": f"dp{world}",
                       "l2": "per-step working set (activations+gradients, several GB) far exceeds the 126 MB L2; no flush needed",
                       "cuda_graph": True},
            "roofline": roofline, "roofline_mem": roofline_mem, "cpu_baseline": cpu_baseline,
            "secondary_bar": load_secondary_bar(),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                    "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": launches_per_step * args.steps + args.steps,
            "clocks": clocks, "kernels": kernels,
            "tensor_core_frac_step": {"algorithmic_tflops_per_gpu": step_tflops,
                                      "of_burst_peak": step_tflops / peaks["tf_burst"],
                                      "of_sustained_peak": step_tflops / peaks["tf_sustained"],
                                      "train_gflop_per_tile": train_flops_per_tile / 1e9},
            "final_loss": loss_val, "predict": predict, "extra": extra,
        }
        print(json.dumps(line), file=out, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
