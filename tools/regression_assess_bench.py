"""Cost of the regression assessment: `b2u_regression_assess` alone, and `predict_geotiff` of a regression model with
and without `mask_path`.

In one process it reports:
- the kernel alone on two workloads: one prediction batch (64 tiles of 256 x 256 fp32 pairs, T = 64, per-tile records
  on) and a 20000 x 20000 fp32 pair (T = 1, 3.2 GB).  Truth is 1000 + a smooth field, the prediction the truth plus
  noise, 1 % of the truth pixels NaN.  CUDA events around each of `--reps` launches, with a 256 MB buffer overwritten
  before each launch so that the maps are read from HBM, not from the 126 MB L2.  The bytes read (8 per pixel) over the
  median time, against the project's HBM denominator (6 548 GB/s, bench.py); the totals of two launches are compared
  bit for bit;
- `predict_geotiff` on a synthetic `--side`^2 4-band uint8 GeoTIFF with a regression model (xresnet34, 256 x 256 tiles,
  overlap 0.125, batch 64), with and without `mask_path` (a Float32 mask), alternated over `--rounds` rounds after one
  warm-up call of each: wall time per call including the file reads and the Float32 raster write;
- the GPU name and power limit.

    python tools/regression_assess_bench.py [--side 20000 --rounds 3 --reps 50 --out report.txt]
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

HBM_GBS = 6548.0


def value_maps(T: int, H: int, W: int, seed: int, dev):
    """(prediction, truth) float32 [T, H, W]: truth 1000 + a smooth field with 1 % NaN, prediction = truth + noise"""
    g = torch.Generator(device=dev).manual_seed(seed)
    low = torch.randn((T, 1, -(-H // 16), -(-W // 16)), generator=g, device=dev)
    truth = torch.nn.functional.interpolate(low, scale_factor=16, mode="nearest")[:, 0, :H, :W] + 1000.0
    pred = truth + 0.1 * torch.randn((T, H, W), generator=g, device=dev)
    truth = torch.where(torch.rand((T, H, W), generator=g, device=dev) < 0.01, float("nan"), truth)
    return pred.contiguous(), truth.contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--side", type=int, default=20000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("regression_assess_bench needs a CUDA device")
    from unet_b200.assessment import RegressionCounter
    from unet_b200.geotiff import GeoInfo, write_geotiff
    from unet_b200.reference_api import predict_geotiff, unet_learner_MS

    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    gpu = q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else "nvidia-smi unavailable"
    say(f"gpu: {gpu} (torch: {torch.cuda.get_device_name()})")
    dev = torch.device("cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    say(f"b2u_regression_assess alone (L2 flushed by a 256 MB write before each launch, {args.reps} launches, median):")
    for name, (T, H, W) in (("batch 64 x 256^2", (64, 256, 256)), (f"pair {args.side}^2", (1, args.side, args.side))):
        pred, truth = value_maps(T, H, W, T, dev)
        counter = RegressionCounter(dev, tile_slots=T if T > 1 else 0)
        per_tile = T > 1

        def launch():
            counter.tiles = 0
            counter.count(pred, truth, per_tile=per_tile)
        for _ in range(5):
            launch()
        recs = []
        for _ in range(2):
            counter.buf.zero_()
            launch()
            recs.append(counter.buf.cpu())
        same = torch.equal(recs[0], recs[1])
        ms = []
        for i in range(args.reps):
            flush.fill_(i & 255)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            launch()
            e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        med = statistics.median(ms)
        nbytes = 8 * T * H * W
        say(f"  {name:18s}: {med * 1e3:9.1f} us (min {min(ms) * 1e3:.1f}); {nbytes / 1e6:7.1f} MB read -> "
            f"{nbytes / med / 1e6:6.0f} GB/s = {nbytes / med / 1e6 / HBM_GBS * 100:5.1f} % of {HBM_GBS:.0f} GB/s; "
            f"two launches bit-identical: {same}")
        del pred, truth, counter
        torch.cuda.empty_cache()
    del flush
    torch.cuda.empty_cache()

    tmp = tempfile.mkdtemp(prefix="regression_assess_bench_")
    try:
        side = args.side
        rng = np.random.default_rng(0)
        img = rng.integers(1, 256, size=(4, side, side), dtype=np.uint8)
        msk = (img[3].astype(np.float32) - img[0]) / 64.0 + 1.0
        geo = GeoInfo(geotransform=(383000.0, 0.2, 0.0, 5819000.0, 0.0, -0.2), georeferenced=True)
        raster, mask = os.path.join(tmp, "scene.tif"), os.path.join(tmp, "scene_mask.tif")
        write_geotiff(raster, img, geo)
        write_geotiff(mask, msk, geo)
        del img, msk
        learn = unet_learner_MS(4, 1, "xresnet34", (256, 256), 64, regression=True)
        say(f"predict_geotiff, regression model, {side} x {side} 4-band uint8 GeoTIFF, xresnet34, 256^2 tiles, overlap "
            f"0.125, batch 64; wall time per call (file reads, prediction, Float32 raster write), {args.rounds} "
            f"alternated rounds after one warm-up call of each:")
        times = {"without mask_path": [], "with mask_path": []}
        outs = {}
        for r in range(args.rounds + 1):
            for key in times:
                kw = {"mask_path": mask} if key == "with mask_path" else {}
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = predict_geotiff(learn, raster, os.path.join(tmp, key.replace(" ", "_") + ".tif"), 0.125, **kw)
                torch.cuda.synchronize()
                if r:
                    times[key].append(time.perf_counter() - t0)
                outs[key] = out
        for key, ts in times.items():
            say(f"  {key:18s}: median {statistics.median(ts):.3f} s  (" + " ".join(f"{t:.3f}" for t in ts) + ")")
        same = open(outs["without mask_path"], "rb").read() == open(outs["with mask_path"], "rb").read()
        with open(os.path.join(tmp, "with_mask_path_assessment.json")) as f:
            rep = json.load(f)
        say(f"  written rasters identical: {same}; assessment of the untrained model: {rep['n']} pixels, "
            f"{rep['skipped']} skipped, RMSE {rep['rmse']:.4g}")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
