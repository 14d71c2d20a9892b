"""Cost of class probability rasters: `b2u_stitch_finalize_probs` alone, and `predict_geotiff` with `all_classes` /
`specific_class` against the argmax mask.

In one process it reports:
- the kernel alone on a `--side`^2 strip (fp32 accumulators of C = 2, 8 and 32 classes, uint8 counts 1..4): all
  classes as Float32, one class as Float32 and all classes as int8 (`large_file`).  CUDA events around each of `--reps`
  launches, with a 256 MB buffer overwritten before each launch so that the accumulators are read from HBM, not from
  the 126 MB L2.  Bytes from shapes (nc planes and the counts read, nc values per pixel written) over the median time,
  against the project's HBM denominator (6 548 GB/s, bench.py);
- `predict_geotiff` on a synthetic `--side`^2 4-band uint8 GeoTIFF (xresnet34, 2 classes, 256 x 256 tiles, overlap
  0.125, batch 64): the argmax mask, `all_classes`, `all_classes` + `large_file` and `specific_class=1`, alternated over
  `--rounds` rounds after one warm-up call of each: wall time per call including the file reads and the raster write;
- the GPU name and power limit.

    python tools/probability_bench.py [--side 20000 --rounds 2 --reps 20 --out report.txt]
"""
import argparse
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--side", type=int, default=20000)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("probability_bench needs a CUDA device")
    from unet_b200 import ops
    from unet_b200.geotiff import GeoInfo, write_geotiff
    from unet_b200.predict_engine import finalize_probs
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
    side = args.side
    s = ops.stream_ptr()

    say(f"b2u_stitch_finalize_probs alone on a {side}^2 strip (L2 flushed by a 256 MB write before each launch, "
        f"{args.reps} launches, median):")
    cnt = torch.randint(1, 5, (side, side), dtype=torch.uint8, device=dev)
    for C in (2, 8, 32):
        acc = torch.rand((C, side, side), device=dev).mul_(cnt)
        for name, c0, nc, large_file in (("all classes fp32", 0, C, False), ("one class fp32", C // 2, 1, False),
                                         ("all classes int8", 0, C, True)):
            for _ in range(2):              # warm-up; the output block stays in the caching allocator afterwards
                finalize_probs(acc, cnt, c0, nc, 0, side, large_file, s)
            ms = []
            for i in range(args.reps):
                flush.fill_(i & 255)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                finalize_probs(acc, cnt, c0, nc, 0, side, large_file, s)
                e1.record()
                e1.synchronize()
                ms.append(e0.elapsed_time(e1))
            med = statistics.median(ms)
            px = side * side
            nbytes = px * (4 * nc + 1) + px * nc * (1 if large_file else 4)
            say(f"  C={C:2d} {name:17s}: {med * 1e3:9.1f} us (min {min(ms) * 1e3:.1f}); {nbytes / 1e9:6.2f} GB -> "
                f"{nbytes / med / 1e6:6.0f} GB/s = {nbytes / med / 1e6 / HBM_GBS * 100:5.1f} % of {HBM_GBS:.0f} GB/s")
        del acc
        torch.cuda.empty_cache()
    del flush, cnt
    torch.cuda.empty_cache()

    tmp = tempfile.mkdtemp(prefix="probability_bench_")
    try:
        rng = np.random.default_rng(0)
        img = rng.integers(1, 256, size=(4, side, side), dtype=np.uint8)
        geo = GeoInfo(geotransform=(383000.0, 0.2, 0.0, 5819000.0, 0.0, -0.2), georeferenced=True)
        raster = os.path.join(tmp, "scene.tif")
        write_geotiff(raster, img, geo)
        del img
        learn = unet_learner_MS(4, 2, "xresnet34", (256, 256), 64)
        say(f"predict_geotiff, {side} x {side} 4-band uint8 GeoTIFF, xresnet34, 2 classes, 256^2 tiles, overlap 0.125, "
            f"batch 64; wall time per call (file reads, prediction, raster write), {args.rounds} alternated rounds "
            f"after one warm-up call of each:")
        modes = {"argmax": {}, "all_classes": dict(all_classes=True),
                 "all_classes+large_file": dict(all_classes=True, large_file=True),
                 "specific_class=1": dict(specific_class=1)}
        times = {k: [] for k in modes}
        sizes = {}
        for r in range(args.rounds + 1):
            for key, kw in modes.items():
                path = os.path.join(tmp, "out.tif")
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                predict_geotiff(learn, raster, path, 0.125, **kw)
                torch.cuda.synchronize()
                if r:
                    times[key].append(time.perf_counter() - t0)
                sizes[key] = os.path.getsize(path)
                os.remove(path)
        for key, ts in times.items():
            say(f"  {key:23s}: median {statistics.median(ts):.3f} s  (" + " ".join(f"{t:.3f}" for t in ts) +
                f"); file {sizes[key] / 1e9:.2f} GB")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
