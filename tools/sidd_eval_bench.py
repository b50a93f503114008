"""What scoring a SIDD evaluation as one batch saves: 40 SIDD-shaped images (32 blocks of 256 x 256 side by side, 256 x 8192), the clean
mosaics and two rounds of synthetic outputs, five phone models (one CFA phase and colour matrix each) with per-image white-balance
jitter, timed two ways alternated in one process:

    per_image  sidd_eval_image([round 1, round 2], clean, meta) once per image (the per-image loop of multiprocess_plot)
    batch      one sidd_eval_batch(rounds, clean, metas) call for all 40

    python tools/sidd_eval_bench.py [--steps 5] [--warmup 1] [--out bench_out/sidd_eval]

Inputs are seeded and resident on the device.  Each step is timed with the host clock up to a device synchronise; both ways end in the
read-back of their numbers.  The same run checks that the two ways give the same tables (PSNR within 1e-12 relative, SSIM within 1e-12
absolute) and the same pictures byte for byte.  Writes <out>/sidd_eval_bench.json with the median ms per step, library launches per
step, the largest differences, and the card (name, power limit, max SM clock) read with nvidia-smi in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import yond_public_b200 as Y  # noqa: E402
from rounds_bench import card  # noqa: E402

NIMG, NBLK, HB = 40, 32, 256
# five phone models: the CFA phase of each, and a colour matrix near a typical camera's
PATTERNS = [[[1, 2], [2, 3]], [[2, 1], [3, 2]], [[2, 3], [1, 2]], [[3, 2], [2, 1]], [[1, 2], [2, 3]]]
CST = np.array([[0.8, 0.25, -0.05], [-0.3, 1.1, 0.2], [0.02, -0.2, 0.9]])


def workload(dev, seed=2026):
    """Seeded clean mosaics (NIMG, HB, NBLK*HB) in [0.02, 0.98], two rounds of outputs (noisy, then closer to clean, clipped to
    [0, 1]), and one metadata dict per image: its phone's CFA phase and colour matrix, its own white balance."""
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    W = NBLK * HB
    yy = torch.linspace(0, 1, HB, device=dev)[None, :, None]
    xx = torch.linspace(0, 1, W, device=dev)[None, None, :]
    ph = torch.rand((NIMG, 1, 1), device=dev, generator=gen) * 6.28
    clean = 0.45 + 0.3 * torch.sin(40.0 * xx + 5.0 * yy + ph) * torch.cos(7.0 * yy - 3.0 * xx + ph)
    clean = clean + 0.05 * torch.rand((NIMG, HB, W), device=dev, generator=gen)
    clean = clean.clamp(0.02, 0.98).contiguous()
    noise = torch.randn((NIMG, HB, W), device=dev, generator=gen)
    rounds = [(clean + s * noise).clamp(0, 1).contiguous() for s in (0.02, 0.008)]
    rng = np.random.default_rng(seed)
    phones = [(PATTERNS[k], CST + rng.normal(0, 0.03, (3, 3)), np.array([rng.uniform(1.6, 2.4), 1.0, rng.uniform(1.4, 2.1)]))
              for k in range(5)]
    metas = []
    for i in range(NIMG):
        pat, cst, wb = phones[i % 5]
        metas.append({"bayer_2by2": pat, "cst2": cst, "wb": (wb * [rng.uniform(0.95, 1.05), 1.0, rng.uniform(0.95, 1.05)])[None]})
    return clean, rounds, metas


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default="bench_out/sidd_eval")
    args = ap.parse_args()
    if args.steps < 3:
        ap.error("--steps must be at least 3")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    clean, rounds, metas = workload(dev)

    def per_image():
        return [Y.sidd_eval_image([r[i] for r in rounds], clean[i], metas[i], nblk=NBLK) for i in range(NIMG)]

    def batch():
        return Y.sidd_eval_batch(rounds, clean, metas, nblk=NBLK)

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
            l0 = Y._lib.launch_count()
            t0 = time.perf_counter()
            out[name] = run()
            torch.cuda.synchronize()
            ms[name].append((time.perf_counter() - t0) * 1e3)
            launches[name].append(Y._lib.launch_count() - l0)
    # the same numbers and pictures both ways
    b, ref = out["batch"], out["per_image"]
    diff = {"psnr_rel": 0.0, "ssim_abs": 0.0, "psnr_rgb_rel": 0.0, "ssim_rgb_abs": 0.0}
    pictures_equal = all(torch.equal(b["img_hr"][i], ref[i]["img_hr"]) for i in range(NIMG))
    for i in range(NIMG):
        for r in range(len(rounds)):
            for key, rel in (("psnr", True), ("ssim", False), ("psnr_rgb", True), ("ssim_rgb", False)):
                want = ref[i][key][r]
                d = abs(b[key][r, i] - want) / (abs(want) if rel else 1.0)
                k = f"{key}_{'rel' if rel else 'abs'}"
                diff[k] = max(diff[k], float(d))
            pictures_equal = pictures_equal and torch.equal(b["img_dn"][r, i], ref[i]["img_dn"][r])
    same = pictures_equal and bool(b["rendered"].all()) and diff["psnr_rel"] <= 1e-12 and diff["psnr_rgb_rel"] <= 1e-12 \
        and diff["ssim_abs"] <= 1e-12 and diff["ssim_rgb_abs"] <= 1e-12
    med = {k: float(np.median(v)) for k, v in ms.items()}
    line = {
        "workload": f"{NIMG} SIDD-shaped images ({NBLK} blocks of {HB} x {HB}), clean mosaics + 2 rounds of outputs, 5 phone models "
                    "(CFA phase, colour matrix) with per-image wb jitter, inputs resident",
        "timing": "host clock to a device synchronise per step, both ways ending in the read-back of their numbers; median of the timed "
                  "steps, the two ways alternated step by step in one process",
        "steps": args.steps, "warmup": args.warmup, "card": card(),
        "ms_per_step": med, "ms_per_step_all": ms, "speedup": med["per_image"] / med["batch"],
        "launches_per_step": {k: int(np.median(v)) for k, v in launches.items()},
        "max_diff": diff, "pictures_equal": pictures_equal, "same": same,
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "sidd_eval_bench.json"), "w") as f:
        json.dump(line, f, indent=1)
    print(json.dumps(line))
    if not same:
        sys.exit("sidd_eval_batch and the per-image loop disagree")


if __name__ == "__main__":
    main()
