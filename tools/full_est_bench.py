"""What batching round 1 on the full-resolution frames (lr_full) saves: the SIDD evaluation shape, 40 images of 32 (256, 256) blocks, each
with its full noisy frame (five phone sensor sizes of 12-16 MP, as the SIDD full frames come from five phone models), bench.ARCH /
bench.PIPE (the shipped SIDD pipeline: est_type 'simple+full', max_iter 1), bench weights, timed two ways alternated in one process:

    per_image  the drop-in IterDenoise({'lr': blocks, 'lr_full': frame}) once per image (the only way before the batched lr_full path)
    batch      one iter_denoise_batch(blocks, p, lr_full=[...]) call for all 40 images

    python tools/full_est_bench.py [--steps 3] [--warmup 1] [--out bench_out/full_est]

Inputs are seeded and resident on the device.  Each size's full frame is synthesised once (synth.clean_smooth / synth.noisy with its own
seeded (K, sigma)) and shared by the images of that size; an image's blocks are 32 seeded crops of its frame.  Writes
<out>/full_est_bench.json: ms per step (CUDA events; each way ends in the read-back of its numbers), MP/s of denoised block pixels,
library launches per step, and the card (name, power limit, max SM clock) read with nvidia-smi in the same run."""
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

# (H, W) of the full frames: five phone sensors of 12.0 - 15.9 MP
FULL_SIZES = [(3000, 4000), (3024, 4032), (3044, 4048), (3120, 4208), (2988, 5328)]
N_IMG, N_BLK, BLK = 40, 32, 256


def workload(dev, seed=2025):
    rng = np.random.default_rng(seed)
    frames = []
    for H, W in FULL_SIZES:
        K, S = synth.sample_noise_params(rng)
        frames.append(torch.from_numpy(synth.noisy(rng, synth.clean_smooth(rng, H, W), K, S).astype(np.float32)).to(dev))
    full, blocks = [], torch.empty((N_IMG, N_BLK, BLK, BLK), device=dev)
    for i in range(N_IMG):
        f = frames[i % len(frames)]
        H, W = f.shape
        ys = 2 * rng.integers(0, (H - BLK) // 2, N_BLK)
        xs = 2 * rng.integers(0, (W - BLK) // 2, N_BLK)
        for b in range(N_BLK):
            blocks[i, b] = f[ys[b]:ys[b] + BLK, xs[b]:xs[b] + BLK]
        full.append(f)
    return blocks, full


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default="bench_out/full_est")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    blocks, full = workload(dev)
    drv = Y.YOND_SIDD(bench.ARCH, bench.PIPE, state_dict=synth.bench_state_dict(bench.ARCH, seed=0), device=dev)

    def per_image():
        return [drv.IterDenoise({"lr": blocks[i], "lr_full": full[i]}, {"p": dict(bench.P0), "img_id": i}) for i in range(N_IMG)]

    def batch():
        return drv.iter_denoise_batch(blocks, dict(bench.P0), lr_full=full)

    ways = {"per_image": per_image, "batch": batch}
    for _ in range(args.warmup):
        for run in ways.values():
            run()
    torch.cuda.synchronize()
    ms = {k: [] for k in ways}
    launches = {k: [] for k in ways}
    out = {}
    for _ in range(args.steps):  # alternated: step s of every way before step s + 1 of any
        for name, run in ways.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = Y._lib.launch_count()
            e0.record()
            out[name] = run()
            e1.record()
            e1.synchronize()
            launches[name].append(Y._lib.launch_count() - l0)
            ms[name].append(e0.elapsed_time(e1))
    # the two ways compute the same thing: the batch's rounds and its final frames against the per-image calls
    res, singles = out["batch"], out["per_image"]
    same_rounds = all(int(res["rounds"][i]) == len(s["raw_dns"]) for i, s in enumerate(singles))
    max_abs = max(float((res["raw_dns"][len(s["raw_dns"]) - 1][i] - s["raw_dns"][-1]).abs().max()) for i, s in enumerate(singles))
    mp_blocks = N_IMG * N_BLK * BLK * BLK / 1e6
    med = {k: float(np.median(v)) for k, v in ms.items()}
    line = {
        "workload": f"{N_IMG} SIDD-shaped images of {N_BLK} ({BLK}, {BLK}) blocks ({mp_blocks:.1f} MP), each with its full frame, sizes "
                    f"{FULL_SIZES} in turn ({sum(full[i].numel() for i in range(N_IMG)) / 1e6:.0f} MP estimated in round 1); "
                    "bench.ARCH, bench.PIPE, synth.bench_state_dict(seed=0), inputs resident",
        "timing": "CUDA events around the calls of one step, each way ending in the read-back of its numbers; median of the timed steps; "
                  "the two ways alternated step by step in one process",
        "steps": args.steps, "warmup": args.warmup, "card": card(),
        "ms_per_step": med, "ms_per_step_all": ms,
        "block_mp_per_s": {k: mp_blocks / (v / 1e3) for k, v in med.items()},
        "launches_per_step": {k: int(np.median(v)) for k, v in launches.items()},
        "speedup_batch_over_per_image": med["per_image"] / med["batch"],
        "rounds_equal": same_rounds, "final_max_abs_diff": max_abs,
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "full_est_bench.json"), "w") as f:
        json.dump(line, f, indent=1)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
