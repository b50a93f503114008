"""What one call for frames of different sizes saves: an ELD-style evaluation batch, uint16 sensor mosaics from four cameras (two frames
each, 2848x4256, 3476x5208, 3670x5496 and 5520x8288, 192 MP in all) with per-image black level, white level and ratio, through
bench.PIPE_FRAME (full_dn, max_iter 1) with bench weights, timed three ways alternated in one process:

    per_image  iter_denoise_batch(frame[None, None], p_i, raw=...) once per frame
    per_size   one iter_denoise_batch per sensor size, on frames stacked per size beforehand (the stacking is not timed)
    frames     one iter_denoise_frames(frames, p, raw=...) call for all eight

    python tools/frames_bench.py [--steps 3] [--warmup 1] [--out bench_out/frames]

Inputs are seeded and resident on the device.  Writes <out>/frames_bench.json: ms per step (CUDA events; each way ends in the read-back
of its numbers), MP/s, library launches per step, the largest difference of the final frames between the ways, and the card (name,
power limit, max SM clock) read with nvidia-smi in the same run."""
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

SIZES = [(2848, 4256), (3476, 5208), (3670, 5496), (5520, 8288)]
PER_SIZE = 2
# (black, white, ratio) per camera: 14-bit sensors at several black levels and low-light gains, one 12-bit sensor
CAMERAS = [(512, 16383, 100.0), (400, 15520, 50.0), (256, 4095, 8.0), (1024, 16383, 200.0)]


def workload(dev, seed=2026):
    """Seeded uint16 mosaics (Poisson-Gaussian around a smooth scene), frame order interleaved across the cameras, and their
    (black, white, ratio)."""
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    frames, bls, wps, ratios = [], [], [], []
    for j in range(PER_SIZE):
        for (H, W), (bl, wp, ratio) in zip(SIZES, CAMERAS):
            yy = torch.linspace(0, 1, H, device=dev)[:, None]
            xx = torch.linspace(0, 1, W, device=dev)[None, :]
            clean = 0.45 + 0.35 * torch.sin(6.0 * xx + 4.0 * yy + j) * torch.cos(3.0 * yy - 2.0 * xx)
            K = 2.0 + j  # DN per electron at the sensor
            dn = clean * (wp - bl) / ratio
            raw = torch.poisson(dn / K, generator=gen) * K + 3.0 * torch.randn(dn.shape, device=dev, generator=gen) + bl
            frames.append(raw.clamp(0, wp).round().to(torch.int32).to(torch.uint16).view(torch.int16).contiguous())
            bls.append(bl)
            wps.append(wp)
            ratios.append(ratio)
    return frames, np.array(bls), np.array(wps), np.array(ratios)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default="bench_out/frames")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    frames, bls, wps, ratios = workload(dev)
    n = len(frames)
    scale = (wps - bls) / ratios
    p = dict(bench.P0, wp=wps, bl=bls, scale=scale)
    raw = (bls, wps, ratios)
    drv = Y.YOND_SIDD(bench.ARCH, bench.PIPE_FRAME, state_dict=synth.bench_state_dict(bench.ARCH, seed=0), device=dev)
    by_size = {}
    for i, f in enumerate(frames):
        by_size.setdefault(tuple(f.shape), []).append(i)
    stacked = {s: torch.stack([frames[i] for i in idx])[:, None] for s, idx in by_size.items()}

    def pick(v, idx):
        return v[idx]

    def per_image():
        return [drv.iter_denoise_batch(frames[i][None, None], dict(bench.P0, wp=wps[i], bl=bls[i], scale=scale[i]),
                                       raw=(bls[i], wps[i], ratios[i])) for i in range(n)]

    def per_size():
        return {s: drv.iter_denoise_batch(stacked[s], dict(bench.P0, wp=pick(wps, idx), bl=pick(bls, idx), scale=pick(scale, idx)),
                                          raw=tuple(pick(v, idx) for v in raw)) for s, idx in by_size.items()}

    def frames_call():
        return drv.iter_denoise_frames(frames, dict(p), raw=raw)

    ways = {"per_image": per_image, "per_size": per_size, "frames": frames_call}
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
    # the final frames of every image, three ways
    final = {"per_image": [r["raw_dns"][-1][0] for r in out["per_image"]], "frames": out["frames"]["raw_dns"][-1]}
    final["per_size"] = [None] * n
    for s, idx in by_size.items():
        for j, i in enumerate(idx):
            final["per_size"][i] = out["per_size"][s]["raw_dns"][-1][j]
    diff = {f"{a}_vs_per_image": max(float((x - y).abs().max()) for x, y in zip(final[a], final["per_image"])) for a in ("per_size", "frames")}
    rounds_equal = all(int(out["frames"]["rounds"][i]) == int(out["per_image"][i]["rounds"][0]) for i in range(n))
    mp = sum(f.numel() for f in frames) / 1e6
    med = {k: float(np.median(v)) for k, v in ms.items()}
    line = {
        "workload": f"{n} uint16 sensor mosaics, sizes {SIZES} x {PER_SIZE} interleaved ({mp:.0f} MP), per-image (black, white, ratio) "
                    f"{CAMERAS}; bench.ARCH, bench.PIPE_FRAME (full_dn, max_iter 1), synth.bench_state_dict(seed=0), inputs resident",
        "timing": "CUDA events around the calls of one step, each way ending in the read-back of its numbers; median of the timed steps; "
                  "the three ways alternated step by step in one process",
        "steps": args.steps, "warmup": args.warmup, "card": card(),
        "ms_per_step": med, "ms_per_step_all": ms,
        "mp_per_s": {k: mp / (v / 1e3) for k, v in med.items()},
        "launches_per_step": {k: int(np.median(v)) for k, v in launches.items()},
        "final_max_abs_diff": diff, "rounds_equal": rounds_equal,
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "frames_bench.json"), "w") as f:
        json.dump(line, f, indent=1)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
