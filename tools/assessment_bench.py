"""Cost of the accuracy assessment: `b2u_confusion_counts` alone, and `predict_geotiff` with and without `mask_path`.

In one process it reports:
- the kernel alone for C = 2, 3, 4, 5, 8 and 32 classes (4 is the largest C counted in registers, 5 the smallest counted
  in shared memory) on two workloads: one prediction batch (64 tiles of 256 x 256, T = 64) and a 20000 x 20000 strip
  pair (T = 1, 0.8 GB).  The maps are land-cover-like: 16 x 16-pixel blocks of one class, and the prediction differs
  from the truth on 10 % of the pixels.  CUDA events around each of `--reps` launches, with a 256 MB buffer overwritten
  before each launch so that the maps are read from HBM, not from the 126 MB L2.  The bytes read (both maps once) over
  the median time, against the project's HBM denominator (6 548 GB/s, bench.py);
- `predict_geotiff` on a synthetic `--side`^2 4-band uint8 GeoTIFF (xresnet34, 256 x 256 tiles, overlap 0.125, batch
  64, 2 classes), with and without `mask_path`, alternated over `--rounds` rounds after one warm-up call of each: wall
  time per call including the file reads and the mask write;
- the GPU name and power limit.

    python tools/assessment_bench.py [--side 20000 --rounds 3 --reps 100 --out report.txt]
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
CLASSES = (2, 3, 4, 5, 8, 32)


def class_maps(T: int, H: int, W: int, C: int, seed: int, dev):
    """(prediction, truth) uint8 [T, H, W]: 16 x 16 blocks of one class, the prediction wrong on 10 % of the pixels"""
    g = torch.Generator(device=dev).manual_seed(seed)
    low = torch.randint(0, C, (T, -(-H // 16), -(-W // 16)), generator=g, device=dev, dtype=torch.uint8)
    truth = low.repeat_interleave(16, 1).repeat_interleave(16, 2)[:, :H, :W].contiguous()
    noise = torch.randint(0, C, (T, H, W), generator=g, device=dev, dtype=torch.uint8)
    wrong = torch.rand((T, H, W), generator=g, device=dev) < 0.1
    return torch.where(wrong, noise, truth).contiguous(), truth


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--side", type=int, default=20000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("assessment_bench needs a CUDA device")
    from unet_b200 import _lib, ops
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
    lib, dev = _lib.load(), torch.device("cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    st = ops.stream_ptr()
    joint = torch.zeros(32 * 32 + 1, dtype=torch.int64, device=dev)
    hist = torch.zeros(64 * 2 * 32, dtype=torch.int32, device=dev)

    say(f"b2u_confusion_counts alone (L2 flushed by a 256 MB write before each launch, {args.reps} launches, median):")
    for name, (T, H, W) in (("batch 64 x 256^2", (64, 256, 256)), (f"strip {args.side}^2", (1, args.side, args.side))):
        for C in CLASSES:
            pred, truth = class_maps(T, H, W, C, C, dev)
            hp = hist.data_ptr() if T > 1 else None

            def launch():
                _lib.check(lib.b2u_confusion_counts(pred.data_ptr(), W, H * W, truth.data_ptr(), W, H * W, T, H, W, C,
                                                    joint.data_ptr(), hp, joint.data_ptr() + 8 * 1024, st),
                           "b2u_confusion_counts")
            for _ in range(5):
                launch()
            joint.zero_()
            launch()
            ok = torch.equal(joint[:C * C].cpu(), torch.bincount((truth.long() * C + pred.long()).flatten(),
                                                                 minlength=C * C).cpu())
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
            nbytes = 2 * T * H * W
            say(f"  {name:18s} C={C:2d}: {med * 1e3:8.1f} us (min {min(ms) * 1e3:.1f}); {nbytes / 1e6:7.1f} MB read -> "
                f"{nbytes / med / 1e6:6.0f} GB/s = {nbytes / med / 1e6 / HBM_GBS * 100:5.1f} % of {HBM_GBS:.0f} GB/s; "
                f"counts equal torch.bincount: {ok}")
            del pred, truth
    del flush
    torch.cuda.empty_cache()

    tmp = tempfile.mkdtemp(prefix="assessment_bench_")
    try:
        side = args.side
        rng = np.random.default_rng(0)
        img = rng.integers(1, 256, size=(4, side, side), dtype=np.uint8)
        msk = (img[3] > img[0]).astype(np.uint8)
        geo = GeoInfo(geotransform=(383000.0, 0.2, 0.0, 5819000.0, 0.0, -0.2), georeferenced=True)
        raster, mask = os.path.join(tmp, "scene.tif"), os.path.join(tmp, "scene_mask.tif")
        write_geotiff(raster, img, geo)
        write_geotiff(mask, msk, geo)
        del img, msk
        learn = unet_learner_MS(4, 2, "xresnet34", (256, 256), 64)
        say(f"predict_geotiff, {side} x {side} 4-band uint8 GeoTIFF, xresnet34, 256^2 tiles, overlap 0.125, batch 64, "
            f"2 classes; wall time per call (file reads, prediction, mask write), {args.rounds} alternated rounds after "
            f"one warm-up call of each:")
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
        say(f"  written masks identical: {same}; assessment of the untrained model: {rep['pixels']} pixels, "
            f"accuracy {rep['accuracy']:.4f}")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
