"""What one collab round of IterDenoise costs: the bench headline workload (eight seeded 12 MP frames, bench.ARCH / PIPE_FRAME /
P0, bench weights) through iter_denoise_batch at max_iter = 0, 1, 2, 3, alternated in one process, timed with CUDA events.

    python tools/rounds_bench.py [--steps 5] [--warmup 2] [--out bench_out/rounds]

Writes <out>/rounds_bench.json: ms per step and launches per step for every max_iter, ms per extra round (least-squares slope over
max_iter and the step-to-step differences), the rounds the frames completed, and the card (name, power limit, max SM clock) read with
nvidia-smi in the same run.  A batch runs max_iter + 1 rounds on the device whatever the estimates say (images that stopped are
carried by selection), so the cost per round does not depend on the data."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
import yond_public_b200 as Y  # noqa: E402
from yond_public_b200 import synth  # noqa: E402


def card():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
        return dict(zip(q.split(","), [c.strip() for c in out.split(",")]))
    except Exception as e:  # the numbers are still written, with the reason the card is unknown
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--max-iters", default="0,1,2,3")
    ap.add_argument("--out", default="bench_out/rounds")
    args = ap.parse_args()
    if args.steps < 5:
        ap.error("--steps must be at least 5")
    iters = [int(v) for v in args.max_iters.split(",")]
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    sd = synth.bench_state_dict(bench.ARCH, seed=0)
    frames = torch.from_numpy(bench.synth_frames(bench.N_FRAMES, seed=2024).reshape(bench.N_FRAMES, 1, bench.FRAME_H, bench.FRAME_W)).to(dev)
    net = Y.build_net(bench.ARCH, dev)
    Y.archs.load_weights(net, sd, by_name=False)
    net.eval()
    drvs = {n: Y.YOND_SIDD(bench.ARCH, dict(bench.PIPE_FRAME, max_iter=n), net=net, device=dev) for n in iters}
    rounds = {}
    for n in iters:  # warm up every shape
        for _ in range(args.warmup):
            rounds[n] = drvs[n].iter_denoise_batch(frames, dict(bench.P0))["rounds"].tolist()
    torch.cuda.synchronize()
    ms = {n: [] for n in iters}
    launches = {n: [] for n in iters}
    for _ in range(args.steps):  # alternated: step s of every max_iter before step s + 1 of any
        for n in iters:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = Y._lib.launch_count()
            e0.record()
            res = drvs[n].iter_denoise_batch(frames, dict(bench.P0))  # ends in the read-back of the numbers
            e1.record()
            e1.synchronize()
            launches[n].append(Y._lib.launch_count() - l0)
            ms[n].append(e0.elapsed_time(e1))
            rounds[n] = res["rounds"].tolist()
            del res
    med = {n: float(np.median(ms[n])) for n in iters}
    slope = float(np.polyfit(iters, [med[n] for n in iters], 1)[0]) if len(iters) > 1 else None
    steps = {f"{a}->{b}": med[b] - med[a] for a, b in zip(iters, iters[1:])}
    line = {
        "workload": f"{bench.N_FRAMES} x {bench.FRAME_W}x{bench.FRAME_H} seeded frames (bench.synth_frames, seed 2024), bench.ARCH, "
                    "bench.PIPE_FRAME with max_iter varied, bench.P0, synth.bench_state_dict(seed=0); iter_denoise_batch, inputs resident",
        "timing": "CUDA events around one iter_denoise_batch call (its final read-back included); median of the timed steps; "
                  "max_iter values alternated step by step in one process",
        "steps": args.steps, "warmup": args.warmup, "card": card(),
        "ms_per_step": {str(n): med[n] for n in iters}, "ms_per_step_all": {str(n): ms[n] for n in iters},
        "launches_per_step": {str(n): int(np.median(launches[n])) for n in iters},
        "ms_per_extra_round": {"slope": slope, "steps": steps},
        "launches_per_extra_round": {f"{a}->{b}": int(np.median(launches[b]) - np.median(launches[a])) for a, b in zip(iters, iters[1:])},
        "rounds_completed": {str(n): rounds[n] for n in iters},
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "rounds_bench.json"), "w") as f:
        json.dump(line, f, indent=1)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
