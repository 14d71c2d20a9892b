"""Training input from a whole raster: `split_raster` + `train_func` (tile files decoded on the host for every step)
against `train_geotiff` (tiles cut on the device by `b2u_crop_train_batch`), at the benchmark's training configuration:
xresnet34, 256 x 256 tiles, batch 64, 4-band uint8, 2 classes, `transforms=True` at share 1.0.

The data is a seeded synthetic raster and mask (`--side`, default 8192), cut with overlap 0.2 and split 100 % into
training so that an epoch holds training steps only.  In one process it reports:
- the wall time of `split_raster`, which the tile-free path does not need;
- steady-state training tiles/s of both paths and of the same learner on one fixed device batch (the synthetic-input
  rate): the median over the epochs after the first (the first one captures the CUDA graph), from the epoch times in
  the history;
- whether both paths trained to the same weights;
- `b2u_crop_train_batch` alone: CUDA events around each of `--reps` launches over random windows and ops, with a
  256 MB buffer overwritten before each launch so that the raster is read from HBM, not from the 126 MB L2.  The bytes
  it must move (every image and label byte of the batch read once and written once) over its median time, against the
  project's HBM denominator (6 548 GB/s, bench.py);
- the GPU name and power limit.

    python tools/raster_train_bench.py [--side 8192 --epochs 5 --reps 200 --out report.txt]
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
ARCH, C, P, B, OVERLAP = "xresnet34", 4, 256, 64, 0.2


def synthetic_scene(side: int, seed: int = 0):
    """4-band uint8 raster with no zero pixels (every window is kept) and a 2-class mask that depends on the bands"""
    rng = np.random.default_rng(seed)
    img = rng.integers(1, 256, size=(C, side, side), dtype=np.uint8)
    msk = (img[3].astype(np.int16) > img[0]).astype(np.uint8)
    return img, msk


def steady_tiles_per_s(history, steps: int) -> float:
    times = [r["time"] for r in history[1:]]
    return steps * B / statistics.median(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--side", type=int, default=8192)
    ap.add_argument("--epochs", type=int, default=5)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("raster_train_bench needs a CUDA device")
    from unet_b200 import _lib, ops
    from unet_b200.create_tiles import split_raster
    from unet_b200.geotiff import GeoInfo, write_geotiff
    from unet_b200.reference_api import train_func, train_geotiff, unet_learner_MS

    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    gpu = q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else "nvidia-smi unavailable"
    say(f"gpu: {gpu} (torch: {torch.cuda.get_device_name()})")
    say(f"config: {ARCH}, {C}-band uint8 raster {args.side} x {args.side}, P {P}, overlap {OVERLAP}, batch {B}, "
        f"transforms=True share 1.0, {args.epochs} epochs (steady state: median of epochs 2..{args.epochs})")
    tmp = tempfile.mkdtemp(prefix="raster_train_bench_")
    try:
        img, msk = synthetic_scene(args.side)
        geo = GeoInfo(geotransform=(383000.0, 0.2, 0.0, 5819000.0, 0.0, -0.2), georeferenced=True)
        raster, mask = os.path.join(tmp, "scene.tif"), os.path.join(tmp, "scene_mask.tif")
        write_geotiff(raster, img, geo)
        write_geotiff(mask, msk, geo)
        base = os.path.join(tmp, "tiles")
        t0 = time.perf_counter()
        written = split_raster(raster, mask, base, P, OVERLAP, [1.0, 0.0], 0.9, False, 0)
        t_split = time.perf_counter() - t0
        n = len(written)
        steps = n // B
        say(f"split_raster: {n} tiles written in {t_split:.2f} s (image + mask GeoTIFFs, uncompressed)")

        common = dict(ARCHITECTURE=ARCH, EPOCHS=args.epochs, LEARNING_RATE=1e-3, CODES=("background", "class1"),
                      transforms=True, n_transform_imgs=1.0)
        a = train_func(base, None, os.path.join(tmp, "m"), "files", B, False, False, "even", ARCH, args.epochs, 1e-3, 10,
                       None, None, None, False, "vali", common["CODES"], True, None, False, None, 1.0)
        b = train_geotiff((raster, mask), P, OVERLAP, [1.0, 0.0], 0.9, False, 0, model_Path=os.path.join(tmp, "m"),
                          description="raster", BATCH_SIZE=B, **common)
        sa, sb = a.state_dict(), b.state_dict()
        same = all(torch.equal(sa[k], sb[k]) for k in sa)
        s = unet_learner_MS(C, 2, ARCH, (P, P), B)
        xd = torch.from_numpy(img[:, :P, :P].copy()).expand(B, C, P, P).contiguous().cuda()
        yd = torch.from_numpy(msk[:P, :P].copy()).expand(B, P, P).contiguous().cuda()
        fixed = lambda: [(xd, yd, B)] * steps
        fixed.n_batches = steps
        s.fit_one_cycle(args.epochs, 1e-3, fixed)
        r_files, r_raster, r_fixed = (steady_tiles_per_s(h, steps) for h in (a.history, b.history, s.history))
        say(f"training, {steps} steps of {B} tiles per epoch:")
        say(f"  split_raster + train_func : {r_files:8.1f} tiles/s   epochs [s]: "
            + " ".join(f"{r['time']:.3f}" for r in a.history))
        say(f"  train_geotiff             : {r_raster:8.1f} tiles/s   epochs [s]: "
            + " ".join(f"{r['time']:.3f}" for r in b.history))
        say(f"  one fixed device batch    : {r_fixed:8.1f} tiles/s   epochs [s]: "
            + " ".join(f"{r['time']:.3f}" for r in s.history))
        say(f"  train_geotiff / fixed batch: {r_raster / r_fixed:.3f};  train_geotiff / files: {r_raster / r_files:.2f}x")
        say(f"  same weights after training (torch.equal on every state_dict tensor): {same}")
        del a, b, s

        lib = _lib.load()
        dev = torch.device("cuda")
        r_d = torch.from_numpy(img).to(dev)
        l_d = torch.from_numpy(msk).to(dev)
        rng = np.random.default_rng(1)
        side = args.side
        tabs = torch.from_numpy(np.stack([
            np.stack([rng.integers(0, side - P + 1, B), rng.integers(0, side - P + 1, B), rng.integers(0, 8, B)])
            for _ in range(args.reps)]).astype(np.int32)).to(dev)
        xb = torch.empty((B, C, P, P), dtype=torch.uint8, device=dev)
        yb = torch.empty((B, P, P), dtype=torch.uint8, device=dev)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        st = ops.stream_ptr()

        def launch(i):
            t = tabs[i]
            _lib.check(lib.b2u_crop_train_batch(r_d.data_ptr(), _lib.DT_U8, C, side, side, l_d.data_ptr(), _lib.DT_U8,
                                                t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), B, P, xb.data_ptr(),
                                                yb.data_ptr(), st), "b2u_crop_train_batch")
        for i in range(10):
            launch(i)
        ms = []
        for i in range(args.reps):
            flush.fill_(i & 255)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            launch(i)
            e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        med = statistics.median(ms)
        nbytes = 2 * B * (C + 1) * P * P
        say(f"b2u_crop_train_batch ({B} x {C + 1} planes of {P}^2 uint8, random windows and ops, L2 flushed by a 256 MB "
            f"write before each launch, {args.reps} launches):")
        say(f"  median {med * 1e3:.1f} us (min {min(ms) * 1e3:.1f}, p90 {sorted(ms)[int(0.9 * len(ms))] * 1e3:.1f}); "
            f"{nbytes / 1e6:.1f} MB moved -> {nbytes / med / 1e6:.0f} GB/s = {nbytes / med / 1e6 / HBM_GBS * 100:.1f} % "
            f"of {HBM_GBS:.0f} GB/s; {med / (1000 * B / r_raster) * 100:.2f} % of a train_geotiff step")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
