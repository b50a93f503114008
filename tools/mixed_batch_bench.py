"""What a batch of images with different exposure parameters costs: the bench headline frames (eight seeded 12 MP frames, bench.ARCH /
PIPE_FRAME, bench weights) through iter_denoise_batch four ways, alternated step by step in one process and timed with CUDA events:

    uniform  one call, p = bench.P0 for every frame
    mixed    one call, eight distinct (bl, wp, ratio) given per image, scale = (wp - bl) / ratio
    split    the same eight as one call per distinct p (what a caller had to do without per-image parameters)
    split_uniform  one call per frame with p = bench.P0: against `split`, what the parameter values alone change (the VST front end's
             bias lookup takes a data-dependent branch per pixel), apart from how the batch is formed

    python tools/mixed_batch_bench.py [--steps 5] [--warmup 2] [--out bench_out/mixed_batch]

Writes <out>/mixed_batch_bench.json: ms per step and library launches per step for each way, and the card (name, power limit, max SM
clock) read with nvidia-smi in the same run.  The frames are the same float32 data in all four ways: only the parameters differ.  They
change the numbers (gain, sigma, VST range) and, with them, the per-pixel branch of the bias lookup, but not the launches."""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
import yond_public_b200 as Y  # noqa: E402
from rounds_bench import card  # noqa: E402
from yond_public_b200 import synth  # noqa: E402

# ELD / LRID-style exposures and two cameras' levels: (black, white, ratio)
EXPOSURES = [(64, 1023, 1), (512, 16383, 1), (512, 16383, 10), (512, 16383, 100), (600, 16383, 200), (480, 16383, 50),
             (256, 4095, 4), (240, 4095, 16)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="bench_out/mixed_batch")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    sd = synth.bench_state_dict(bench.ARCH, seed=0)
    n = bench.N_FRAMES
    assert n == len(EXPOSURES)
    frames = torch.from_numpy(bench.synth_frames(n, seed=2024).reshape(n, 1, bench.FRAME_H, bench.FRAME_W)).to(dev)
    drv = Y.YOND_SIDD(bench.ARCH, bench.PIPE_FRAME, state_dict=sd, device=dev)
    bl, wp, ratio = (np.array(v) for v in zip(*EXPOSURES))
    p_mixed = dict(bench.P0, wp=wp, bl=bl, ratio=ratio, scale=(wp - bl) / ratio)
    p_each = [dict(bench.P0, wp=int(wp[i]), bl=int(bl[i]), ratio=int(ratio[i]), scale=float((wp[i] - bl[i]) / ratio[i])) for i in range(n)]
    ways = {
        "uniform": lambda: [drv.iter_denoise_batch(frames, dict(bench.P0))],
        "mixed": lambda: [drv.iter_denoise_batch(frames, dict(p_mixed))],
        "split": lambda: [drv.iter_denoise_batch(frames[i:i + 1], dict(p_each[i])) for i in range(n)],
        "split_uniform": lambda: [drv.iter_denoise_batch(frames[i:i + 1], dict(bench.P0)) for i in range(n)],
    }
    rounds = {}
    for name, run in ways.items():  # warm up every shape
        for _ in range(args.warmup):
            rounds[name] = np.concatenate([r["rounds"] for r in run()]).tolist()
    torch.cuda.synchronize()
    ms = {k: [] for k in ways}
    launches = {k: [] for k in ways}
    for _ in range(args.steps):  # alternated: step s of every way before step s + 1 of any
        for name, run in ways.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = Y._lib.launch_count()
            e0.record()
            res = run()  # every call ends in the read-back of its numbers
            e1.record()
            e1.synchronize()
            launches[name].append(Y._lib.launch_count() - l0)
            ms[name].append(e0.elapsed_time(e1))
            rounds[name] = np.concatenate([r["rounds"] for r in res]).tolist()
            del res
    line = {
        "workload": f"{n} x {bench.FRAME_W}x{bench.FRAME_H} seeded frames (bench.synth_frames, seed 2024), bench.ARCH, bench.PIPE_FRAME, "
                    f"synth.bench_state_dict(seed=0); iter_denoise_batch, inputs resident; (black, white, ratio) of the mixed / split "
                    f"ways: {EXPOSURES}",
        "timing": "CUDA events around the calls of one step (each ends in the read-back of its numbers); median of the timed steps; "
                  "the ways alternated step by step in one process",
        "steps": args.steps, "warmup": args.warmup, "card": card(),
        "ms_per_step": {k: float(np.median(v)) for k, v in ms.items()}, "ms_per_step_all": ms,
        "launches_per_step": {k: int(np.median(v)) for k, v in launches.items()},
        "rounds_completed": rounds,
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "mixed_batch_bench.json"), "w") as f:
        json.dump(line, f, indent=1)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
