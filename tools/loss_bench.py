"""Step time and loss-kernel time of the three training losses (CrossEntropyLossFlat, FocalLossFlat gamma 2, DiceLoss) at
the benchmark's training configuration: xresnet34, 256 x 256 tiles, batch 64, 2 classes, SGD, one CUDA graph per step.

One trainer per loss lives in the same process.  Their captured steps are replayed in alternation (`--replays` back to
back per trainer and round, `--rounds` rounds, CUDA events around each run of replays) and the median ms/step per loss
is reported, so the three see the same clocks and the same neighbours.  Separately, each plan's `loss_and_grad` alone is
timed with CUDA events over `--reps` launches, with a 256 MB buffer overwritten before each one so that logits and labels
come from HBM, not from the 126 MB L2.  Algorithmic bytes are computed from the shapes below and divided by the
project's HBM denominator (6 548 GB/s, bench.py).  Prints the GPU name and power limit of the run.

    python tools/loss_bench.py [--rounds 5 --replays 50 --reps 200]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

HBM_GBS = 6548.0
ARCH, N_IN, N_OUT, SIZE, B = "xresnet34", 4, 2, 256, 64
LOSSES = [("ce", "CrossEntropyLossFlat(axis=1)"), ("focal", "FocalLossFlat(axis=1, gamma=2)"), ("dice", "DiceLoss()")]


def loss_bytes(name: str, P: int, ld: int, ldg: int) -> int:
    """bytes the loss launches must move: fp32 logits [P][ld], uint8 labels [P], bf16 dlogits [P][ldg] written once"""
    logits, labels, dl = P * ld * 4, P, P * ldg * 2
    if name == "ce":
        return logits + 2 * labels + dl           # weight sum reads the labels, the fused pass reads them again
    if name == "focal":
        return logits + labels + dl
    return 2 * (logits + labels) + dl             # Dice: statistics pass + backward pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--replays", type=int, default=50)
    ap.add_argument("--reps", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("loss_bench needs a CUDA device")
    from unet_b200.engine import Trainer
    from unet_b200.losses import parse_loss_func
    from unet_b200.network import UNetB200
    from unet_b200.synth import uniform_tiles
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    gpu = q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else "nvidia-smi unavailable"
    print(f"gpu: {gpu} (torch: {torch.cuda.get_device_name()})")
    x, y = uniform_tiles(B, N_IN, SIZE, SIZE, N_OUT, seed=1234, label_seed=4321)
    x, y = x.cuda(), y.cuda()
    runs = {}
    for name, call in LOSSES:
        net = UNetB200(ARCH, N_IN, N_OUT, (SIZE, SIZE), B, training=True, loss_spec=parse_loss_func(call))
        net.init_parameters(seed=0)
        tr = Trainer(net, optimizer="sgd", lr=1e-3, use_graph=True)
        tr.step(x, y)                               # captures the graph
        torch.cuda.synchronize()
        runs[name] = (net, tr)
        print(f"{name}: built, {torch.cuda.memory_allocated() / 2**30:.1f} GiB allocated in all")
    for _, tr in runs.values():                     # warm-up of every graph
        for _ in range(10):
            tr.graph.replay()
    torch.cuda.synchronize()
    step_ms = {n: [] for n in runs}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(args.rounds):
        order = list(runs) if r % 2 == 0 else list(reversed(list(runs)))
        for name in order:
            tr = runs[name][1]
            e0.record()
            for _ in range(args.replays):
                tr.graph.replay()
            e1.record()
            e1.synchronize()
            step_ms[name].append(e0.elapsed_time(e1) / args.replays)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    loss_ms = {}
    for name, (net, _) in runs.items():
        for _ in range(5):
            net.loss_and_grad()
        tot = 0.0
        for _ in range(args.reps):
            flush.fill_(1)
            e0.record()
            net.loss_and_grad()
            e1.record()
            e1.synchronize()
            tot += e0.elapsed_time(e1)
        loss_ms[name] = tot / args.reps
    P = B * SIZE * SIZE
    ld, ldg = runs["ce"][0].logits.shape[-1], runs["ce"][0].dlogits.shape[-1]
    out = {"gpu": gpu, "config": f"{ARCH}/{SIZE}/batch {B}/{N_OUT} classes, sgd, CUDA graph", "rounds": args.rounds,
           "replays_per_round": args.replays, "loss_reps": args.reps, "losses": {}}
    print(f"\n{'loss':6s} {'median ms/step':>14s} {'min':>7s} {'max':>7s} {'loss ms':>8s} {'alg. MB':>8s} {'GB/s':>7s} "
          f"{'frac':>5s}")
    for name, call in LOSSES:
        s = step_ms[name]
        nb = loss_bytes(name, P, ld, ldg)
        gbs = nb / (loss_ms[name] * 1e-3) / 1e9
        row = {"call": call, "step_ms_median": statistics.median(s), "step_ms_all": [round(v, 4) for v in s],
               "loss_ms": loss_ms[name], "loss_alg_bytes": nb, "loss_GBps": gbs, "loss_frac_hbm": gbs / HBM_GBS,
               "launches_per_step": runs[name][0].launches_per_train_step}
        out["losses"][name] = row
        print(f"{name:6s} {row['step_ms_median']:14.3f} {min(s):7.3f} {max(s):7.3f} {loss_ms[name]:8.4f} {nb / 1e6:8.1f} "
              f"{gbs:7.0f} {gbs / HBM_GBS:5.2f}")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
