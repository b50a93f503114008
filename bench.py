#!/usr/bin/env python
"""bench.py — end-to-end YOND blind raw denoising throughput on B200 (BASELINE.json metric: raw MP/s).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host cores (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/<name>.npy

Headline workload (north_star target, BASELINE.json configs[4]/[2]): synthetic 12 MP Bayer frames (4032x3024, 10-bit:
wp 1023, bl 64, Poisson-Gaussian noise), 8 frames per GPU per step, image-parallel across the GPUs; GuidedResUnet
(GRU_5to50_norm_mix arch block), the reference's full-frame pipeline (runfiles/YOND/{ANY,DND,ELD,LRID}_simple+full_pre_grumix.yml:
full_est, full_dn, bias_corr 'pre', iter, max_iter 1): per frame self-calibration estimate -> bias LUT -> VST -> network ->
inverse VST -> collab estimate -> second round.  Both rounds execute for every frame (`round2_denoise_images`).
A step = one pass over the GPU's 8 frames (97.5 MP).  `value`: inputs resident in HBM.  `e2e`: the same step from pinned
HOST buffers to pinned host buffers, H2D + D2H inside the timed region.
Secondary keys: `secondary` (BASELINE configs[1]: 1280 SIDD-shaped 256x256 blocks, the reference's shipped SIDD pipeline),
`e2e_dropin` (per-image `IterDenoise(np arrays)` through the reference's own call signature), `frame_sharded` (ONE 12 MP /
24 MP frame with the network stage band-sharded across the ranks: configs[2] / [3]), `roofline_hbm` (every HBM-bound kernel
timed live with CUDA events against its algorithmic bytes).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ARCH = {"name": "GuidedResUnet", "guided": True, "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1, "res": True, "norm": True}
PIPE = {"data_type": "SIDD", "full_est": True, "est_type": "simple+full", "k": 29, "full_dn": False, "vst_type": "exact",
        "bias_corr": "pre", "iter": "iter", "max_iter": 1, "clip": False}
PIPE_FRAME = dict(PIPE, data_type="ANY", full_dn=True)
P0 = {"wp": 1023, "bl": 64, "ratio": 1, "gain": 1, "sigma": 0, "scale": 959.0}
P_C4 = {"wp": 16383, "bl": 512, "ratio": 100, "gain": 1, "sigma": 0, "scale": (16383 - 512) / 100}
N_IMAGES, N_BLOCKS, BLK = 40, 32, 256
FRAME_H, FRAME_W, N_FRAMES = 3024, 4032, 8
METRIC = "raw_MP_per_s_end_to_end_YOND_denoise"
WORKLOAD = ("configs[4]/[2]: synthetic 12 MP Bayer frames (4032x3024, 10-bit), 8 per GPU per step, image-parallel; GuidedResUnet "
            "(GRU_5to50_norm_mix), full-frame pipeline *_simple+full_pre_grumix (full_est, full_dn, bias_corr pre, iter): "
            "self estimate + VST denoise + collab estimate + second VST denoise per frame; weights = mild smoother + 0.25 x the "
            "reference's random init (no checkpoint offline; passes the reference's round-2 guard so both rounds run)")
WORKLOAD_C2 = ("configs[1]: 1280 synthetic 256x256 Bayer blocks (40 images x 32), GuidedResUnet, SIDD_simple+full_pre_grumix "
               "pipeline (per-image estimate on the mosaic, 32 block-wise VST denoises, SIDD_256 collab estimate, second round)")
E2E_GROUP_FRAMES = int(os.environ.get("YOND_E2E_GROUP_FRAMES", "8"))
E2E_GROUP_IMAGES = int(os.environ.get("YOND_E2E_GROUP", "8"))


def synth_images(n_images, seed=2024):
    """(n_images, 32, 256, 256) float32 noisy blocks + the (K, sigma) drawn per image (yond_datasets.py:664-682,720)."""
    from yond_public_b200 import synth
    rng = np.random.default_rng(seed)
    out = np.empty((n_images, N_BLOCKS, BLK, BLK), np.float32)
    params = []
    for i in range(n_images):
        # K >= 0.6 DN/e-: keeps most blind estimates of sigma/K inside the BiasLUT (< 10 e-); the ones that leave it take
        # the numeric fallback table, which is generated on the device
        K, S = synth.sample_noise_params(rng, logk_min=-0.5)
        params.append((K, S))
        for b in range(N_BLOCKS):
            out[i, b] = synth.noisy(rng, synth.clean_smooth(rng, BLK, BLK), K, S, clip=True)
    return out, params


def synth_frame(rng, H, W, p):
    """One noisy frame in the dataset's normalisation.  10-bit (P0): clipped, K / sigma drawn like the reference's synthesis.
    14-bit low light (P_C4): (raw - bl) * ratio / (wp - bl), unclipped (yond_datasets.py:1053-1056), Sony-like K = 2.2, sigma = 3.1 DN."""
    from yond_public_b200 import synth
    clean = synth.clean_smooth(rng, H, W)
    if p["ratio"] == 1:
        K, S = synth.sample_noise_params(rng, logk_min=-0.5)
        return synth.noisy(rng, clean, K, S, scale=float(p["wp"] - p["bl"]), clip=True)
    return synth.noisy(rng, clean, 2.2 * p["ratio"], 3.1 * p["ratio"], scale=float(p["wp"] - p["bl"]), clip=False)


def synth_frames(n, seed, H=FRAME_H, W=FRAME_W):
    rng = np.random.default_rng(seed)
    return np.stack([synth_frame(rng, H, W, P0) for _ in range(n)])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,timestamp")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.idx, self.t0 = [], None, gpu_index, 0.0

    def mark(self):  # the timed region starts here; nvidia-smi itself was started earlier so that its start-up cost is not inside
        self.t0 = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    @staticmethod
    def _when(stamp, fallback):
        """nvidia-smi's own sample time ('YYYY/MM/DD HH:MM:SS.mmm', local time): its stdout is a pipe and arrives in bursts, so the
        time a line is READ says little about when it was sampled."""
        try:
            import datetime
            return datetime.datetime.strptime(stamp, "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except Exception:
            return fallback

    def _read(self):
        for line in self.proc.stdout:
            cols = [c.strip() for c in line.split(",")]
            self.rows.append(cols + [self._when(cols[-1], time.time())])

    def stop(self, span=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t_end = time.time()  # samples after this instant saw an idle GPU: not part of the timed region
        if span is not None:  # host clock around the timed device work itself (under torchrun the first all-reduce of the timing
            self.t0, t_end = span  # takes several hundred ms during which the GPU idles at its maximum clock)
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        self.t.join(timeout=2)  # the reader drains what nvidia-smi had buffered
        inside = [r for r in self.rows if self.t0 <= r[-1] <= t_end]
        scope = "timed region" if inside else "warm-up + timed region (no sample fell inside by nvidia-smi's clock)"
        self.rows = inside if inside else self.rows
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "scope": scope}


DUMP_SAMPLE = 1 << 22   # values kept of an output larger than this: a fixed seeded set of positions, the same for every output
DUMP_LIMIT = 64 << 20   # bytes written by --dump-outputs in all


def dump_outputs(out_dir, arrays):
    """Writes {name: array or tensor} as out_dir/<name>.npy in float32 / float64, so that the outputs of two builds can be compared
    file by file.  An output of more than DUMP_SAMPLE values is written as a 1-D array of its values at DUMP_SAMPLE seeded flat
    positions (sorted, duplicates dropped); the positions depend on the output's size only."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, a in arrays.items():
        a = a if torch.is_tensor(a) else torch.from_numpy(np.asarray(a))
        if a.numel() > DUMP_SAMPLE:
            pos = np.unique(np.random.default_rng(0).integers(0, a.numel(), DUMP_SAMPLE))
            a = a.reshape(-1)[torch.from_numpy(pos).to(a.device)]
        a = a.cpu().numpy()
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        total += a.nbytes
        if total > DUMP_LIMIT:
            raise ValueError(f"--dump-outputs would write more than {DUMP_LIMIT >> 20} MB")
        np.save(os.path.join(out_dir, name + ".npy"), a)


def last_step_outputs(res):
    """The arrays IterDenoise hands its caller: the denoised frames of the first and the final round, (beta1, beta2) of every
    round, and how many rounds each frame completed."""
    out = {"raw_dns_round1": res["raw_dns"][0], "raw_dns_final": res["raw_dns"][-1], "rounds": res["rounds"]}
    out.update({f"regs_round{i + 1}": np.asarray(r, np.float64) for i, r in enumerate(res["regs"])})
    return out


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# ---------------------------------------------------------------------------------------------------------
# CPU legs: the ONLY places bench.py touches oracle/ (the reference is Python and cannot travel to the GPU box: the
# oracle port is the reference algorithm, pinned against goldens generated by the reference itself)
CPU_SAMPLE = (1512, 2016)  # a quarter-area crop of a 12 MP frame per step: bounds the CPU arm to a few minutes


def cpu_reference_step(frame, sd, lut):
    from oracle import yond_oracle as O
    return O.IterDenoise(ARCH, sd, frame, dict(P0), PIPE_FRAME, biaslut=lut, sidd_256=False)


def cpu_threads():
    """All host cores, also under torchrun (which exports OMP_NUM_THREADS=1)."""
    import torch
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        pass
    torch.set_num_threads(n)
    return torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    cores = cpu_threads()
    from oracle import yond_oracle as O
    from yond_public_b200 import synth
    lut = O.BiasLUT(os.path.join(ROOT, "yond_public_b200", "data", "bias_lut_2d_f32.npz"))
    sd = synth.bench_state_dict(ARCH, seed=0)
    frames = synth_frames(2, seed=2024, H=CPU_SAMPLE[0], W=CPU_SAMPLE[1])
    rounds = []
    for w in range(args.warmup):
        cpu_reference_step(frames[w % 2], sd, lut)
    t0 = time.perf_counter()
    for s in range(args.steps):
        res = cpu_reference_step(frames[s % 2], sd, lut)
        rounds.append(len(res["raw_dns"]))
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_step_outputs(dict(res, rounds=np.array([rounds[-1]]))))
    mp = args.steps * CPU_SAMPLE[0] * CPU_SAMPLE[1] / 1e6
    val = mp / dt
    try:
        import cv2
        cvt = cv2.getNumThreads()
    except Exception:
        cvt = None
    sample = (f"one {CPU_SAMPLE[1]}x{CPU_SAMPLE[0]} frame (quarter-area crop of the 12 MP frame, {CPU_SAMPLE[0] * CPU_SAMPLE[1] / 1e6:.2f} MP) per step, "
              f"{args.steps} steps; oracle port of YOND_SIDD.IterDenoise (full_dn, two rounds), fp32, {cores} torch threads")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "MP/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": sample, "round2_denoise_images": int(sum(r == 2 for r in rounds)), "steps_run": len(rounds)},
            "cpu_baseline": {"value": val, "unit": "MP/s", "cores": cores, "kind": "port", "sample": sample,
                             "os_cpu_count": os.cpu_count(), "cv2_threads": cvt},
            "e2e": {"value": val, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
# algorithmic bytes per Bayer pixel of the HBM-bound stages (SURVEY 8d) are stated where the stages are launched
# (YondProfScope in csrc/): the live profiler returns bytes and milliseconds per stage
def hbm_table(prof, peak_gbs):
    rows = []
    for name, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"]):
        if v["ms"] <= 0 or v["bytes"] <= 0:
            continue
        gbs = v["bytes"] / (v["ms"] / 1e3) / 1e9
        rows.append({"kernel": name, "launch_groups": int(v["scopes"]), "algorithmic_bytes": float(v["bytes"]), "ms": float(v["ms"]),
                     "achieved_gbs": gbs, "frac": gbs / peak_gbs})
    return rows


def run_b200(args):
    import torch
    import torch.distributed as dist

    import yond_public_b200 as Y
    from yond_public_b200 import parallel, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # one process per GPU: run on (and first-touch the pinned staging buffers from) the CPUs of the GPU's own NUMA node
    numa_node = parallel.bind_to_gpu_numa_node(local) if os.environ.get("YOND_NUMA_BIND", "1") != "0" else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks, peak_src = measured_peaks()
    sd = synth.bench_state_dict(ARCH, seed=0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    pending = []  # outstanding gathers: (work handle, tensor kept alive)

    def drain():
        while pending:
            pending.pop(0)[0].wait()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_host0 = time.time()
        e0.record()
        for _ in range(steps):
            fn()
        drain()
        e1.record()
        e1.synchronize()
        last["timed_span"] = (t_host0, time.time())  # host clock around the device work of this region (clock samples are cut to it)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def make_gather(shape):
        buf = [torch.empty(shape, dtype=torch.float32, device=dev) for _ in range(world)] if (world > 1 and rank == 0) else None

        def gather_async(final):
            # the final gather of step i runs on NCCL's stream while step i+1 computes; at most two are in flight and all of
            # them are waited for before the timed region ends (`drain`)
            pending.append((dist.gather(final, buf, dst=0, async_op=True), final))
            if len(pending) > 2:
                pending.pop(0)[0].wait()
        return gather_async

    # =========================================== headline: 12 MP frames, image-parallel (weak scaling: 8 frames per rank)
    frames_np = synth_frames(N_FRAMES, seed=2024 + rank)
    host_in = torch.from_numpy(frames_np.reshape(N_FRAMES, 1, FRAME_H, FRAME_W)).pin_memory()
    host_out = torch.empty((N_FRAMES, FRAME_H, FRAME_W), dtype=torch.float32).pin_memory()
    dev_in = host_in.to(dev)
    drv = Y.YOND_SIDD(ARCH, PIPE_FRAME, state_dict=sd, device=dev)
    net = drv.net
    gather_frames = make_gather((N_FRAMES, FRAME_H, FRAME_W))
    last = {}

    def step_frames():  # one host thread, one stream: every stage once for all 8 frames; one small read-back at the end
        res = drv.iter_denoise_batch(dev_in, dict(P0))
        last["rounds"] = res["rounds"]
        if args.dump_outputs:  # only then are a step's outputs kept alive into the next step
            last["res"] = res
        if world > 1:
            gather_frames(res["raw_dns"][-1])

    host_outs = [host_out, torch.empty_like(host_out).pin_memory()]
    jobs = []  # batches in flight: the next batch is submitted before the previous one is collected (a streaming caller)

    def collect(limit):
        while len(jobs) > limit:
            last["rounds_e2e"] = jobs.pop(0).result()["rounds"]

    def step_frames_e2e():
        last["seq"] = last.get("seq", 0) + 1
        jobs.append(drv.iter_denoise_host(host_in, host_outs[last["seq"] % 2], dict(P0), group=E2E_GROUP_FRAMES, wait=False))
        collect(1)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step_frames()
    drain()
    sampler.mark()
    net.set_profile(True)  # the timed region itself is profiled: CUDA events around every conv launch / every HBM stage
    net.read_profile(reset=True)
    Y._lib.prof_enable(True)
    Y._lib.prof_read(reset=True)
    l0 = Y._lib.launch_count()
    ms = timed(step_frames, args.steps)
    launches = Y._lib.launch_count() - l0
    clocks = sampler.stop(last.get("timed_span")) if rank == 0 else None
    prof = net.read_profile(reset=True)
    hbm_prof = Y._lib.prof_read(reset=True)
    net.set_profile(False)
    Y._lib.prof_enable(False)
    last_res = last.pop("res", None)
    if last_res is not None and rank == 0:
        dump_outputs(args.dump_outputs, last_step_outputs(last_res))
    del last_res
    for _ in range(args.warmup):  # the end-to-end leg warms up like the device-resident one (pinned buffers, staging ring, streams)
        step_frames_e2e()
    collect(0)

    def e2e_steps():  # K batches streamed back to back; every result is collected inside the timed region
        for _ in range(args.steps):
            step_frames_e2e()
        collect(0)
    ms_e2e = timed(e2e_steps, 1)
    mp_step = N_FRAMES * FRAME_H * FRAME_W / 1e6
    value = world * mp_step * args.steps / (ms / 1e3)
    e2e = world * mp_step * args.steps / (ms_e2e / 1e3)

    # the same end-to-end step from uint16 sensor mosaics (SURVEY 8(f)-1): the frames quantised to the 10-bit sensor range, H2D of
    # 2 B/px, dataset normalisation applied on load by the estimator and the VST front end
    raw16 = np.clip(np.rint(frames_np * 959.0 + 64.0), 0, 1023).astype(np.uint16)
    host_in16 = torch.from_numpy(raw16.view(np.int16).reshape(N_FRAMES, 1, FRAME_H, FRAME_W)).pin_memory()

    def step_frames_e2e16():
        last["seq"] = last.get("seq", 0) + 1
        jobs.append(drv.iter_denoise_host(host_in16, host_outs[last["seq"] % 2], dict(P0), group=E2E_GROUP_FRAMES, wait=False, raw=(64, 1023, 1)))
        collect(1)

    def e2e16_steps():
        for _ in range(args.steps):
            step_frames_e2e16()
        collect(0)
    for _ in range(max(1, min(args.warmup, 2))):
        step_frames_e2e16()
    collect(0)
    ms_e2e16 = timed(e2e16_steps, 1)
    e2e16 = world * mp_step * args.steps / (ms_e2e16 / 1e3)

    # drop-in call: per-frame IterDenoise(np arrays) -> np arrays through the reference's signature (pageable NumPy in / out)
    def dropin(drv_, arrays, p):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for a in arrays:
            out = drv_.IterDenoise({"lr": a, "name": "bench"}, {"p": dict(p), "img_id": 0})
            assert isinstance(out["raw_dns"][-1], np.ndarray)
        torch.cuda.synchronize()
        return time.perf_counter() - t0
    dropin(drv, [frames_np[0]], P0)
    dt_drop = dropin(drv, list(frames_np[:4]), P0)
    dropin_frames = 4 * FRAME_H * FRAME_W / 1e6 / dt_drop

    # =========================================== one frame across the ranks (configs[2] / [3]): network stage band-sharded
    frame_sharded = {}
    for name, (H, W), p in (("C3_12MP_10bit", (FRAME_H, FRAME_W), P0), ("C4_24MP_14bit_ratio100_noclip", (4000, 6000), P_C4)):
        rng = np.random.default_rng(99)  # the same frame on every rank
        fr = torch.from_numpy(synth_frame(rng, H, W, p)).to(dev)
        drv.engine.max_value = 1.0 if p["ratio"] == 1 else 4.0
        step = lambda: parallel.denoise_frame_sharded(drv, fr, dict(p))  # noqa: E731
        for _ in range(2):
            step()
        ms_f = timed(step, args.steps) / args.steps
        res = step()
        _, rnds, _ = drv.read_summary(res)
        frame_sharded[name] = {"ms_per_frame": ms_f, "MP_per_s": H * W / 1e6 / (ms_f / 1e3), "ranks": world, "rounds": int(rnds[0]),
                               "scaling": "strong (one frame, N ranks)"}
        del fr
    drv.engine.max_value = 1.0
    del dev_in
    torch.cuda.empty_cache()

    # =========================================== secondary: configs[1], 1280 SIDD-shaped blocks
    imgs_np, _ = synth_images(N_IMAGES, seed=2024 + rank)
    host_in2 = torch.from_numpy(imgs_np).pin_memory()
    host_out2 = torch.empty((N_IMAGES, BLK, N_BLOCKS * BLK), dtype=torch.float32).pin_memory()
    dev_in2 = host_in2.to(dev)
    drv2 = Y.YOND_SIDD(ARCH, PIPE, state_dict=sd, device=dev)
    gather_blocks = make_gather((N_IMAGES, BLK, N_BLOCKS * BLK))

    def step_blocks():
        res = drv2.iter_denoise_batch(dev_in2, dict(P0))
        last["rounds2"] = res["rounds"]
        if world > 1:
            gather_blocks(res["raw_dns"][-1])

    host_outs2 = [host_out2, torch.empty_like(host_out2).pin_memory()]

    def step_blocks_e2e():
        last["seq"] = last.get("seq", 0) + 1
        jobs.append(drv2.iter_denoise_host(host_in2, host_outs2[last["seq"] % 2], dict(P0), group=E2E_GROUP_IMAGES, wait=False))
        collect(1)

    for _ in range(args.warmup):
        step_blocks()
    drain()
    ms2 = timed(step_blocks, args.steps)
    for _ in range(min(args.warmup, 2)):
        step_blocks_e2e()
    collect(0)

    def e2e_steps2():
        for _ in range(args.steps):
            step_blocks_e2e()
        collect(0)
    ms2_e2e_runs = [timed(e2e_steps2, 1) for _ in range(2)]  # secondary number only: two timed regions, both reported, the faster one quoted
    ms2_e2e = min(ms2_e2e_runs)                              # (one region in six box-runs came out 2x slow with everything else normal)
    mp2 = N_IMAGES * N_BLOCKS * BLK * BLK / 1e6
    dropin(drv2, [imgs_np[0]], P0)
    dt_drop2 = dropin(drv2, list(imgs_np[:8]), P0)
    secondary = {"workload": WORKLOAD_C2, "value": world * mp2 * args.steps / (ms2 / 1e3), "unit": "MP/s", "ms_per_step": ms2 / args.steps,
                 "e2e": {"value": world * mp2 * args.steps / (ms2_e2e / 1e3), "unit": "MP/s", "ms_per_step": ms2_e2e / args.steps,
                         "h2d_bytes_per_step": int(host_in2.numel() * 4), "d2h_bytes_per_step": int(host_out2.numel() * 4),
                         "ms_per_step_runs": [m / args.steps for m in ms2_e2e_runs]},
                 "e2e_dropin": {"value": 8 * N_BLOCKS * BLK * BLK / 1e6 / dt_drop2, "unit": "MP/s (one rank)",
                                "api": "YOND_SIDD.IterDenoise({'lr': np (32,256,256)}, {'p': p}) -> np, one image per call, 8 calls"},
                 "round2_denoise_images": int((last["rounds2"] == 2).sum()), "images_per_gpu": N_IMAGES}

    # =========================================== roofline + CPU baseline
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
    peak_hbm = float(peaks.get("hbm_gbs", 6650.0))
    ach_tf = prof["conv_flops"] / (prof["conv_ms"] / 1e3) / 1e12 if prof["conv_ms"] > 0 else 0.0
    traffic, traffic_note = None, None
    for name in ("r02_conv_traffic_frames.json", "r01_conv_traffic.json"):
        try:  # ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum over the conv launches of one forward
            with open(os.path.join(ROOT, "profiles", name)) as f:
                tj = json.load(f)
            traffic = tj["dram_bytes_per_launch"]
            traffic_note = f"profiles/{name}: mean DRAM bytes per conv_tc_kernel launch (ncu, cold cache): {tj.get('note', 'one network forward')}"
            break
        except Exception:
            pass
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = cpu_threads()
        from oracle import yond_oracle as O  # the CPU-baseline leg is the only place the GPU arm touches oracle/
        lut = O.BiasLUT(drv.biaslut.bias_lut)
        crop = frames_np[0][:CPU_SAMPLE[0], :CPU_SAMPLE[1]]
        t0 = time.perf_counter()
        reps = 0
        while reps < 2 or (time.perf_counter() - t0 < 10 and reps < 6):
            cpu_reference_step(np.ascontiguousarray(crop), sd, lut)
            reps += 1
        dt = time.perf_counter() - t0
        cpu_base = {"value": reps * CPU_SAMPLE[0] * CPU_SAMPLE[1] / 1e6 / dt, "unit": "MP/s", "cores": cores, "kind": "port",
                    "sample": f"{reps} x one {CPU_SAMPLE[1]}x{CPU_SAMPLE[0]} crop of a bench frame through the oracle port of IterDenoise (full_dn, two rounds), fp32, {dt:.1f} s",
                    "os_cpu_count": os.cpu_count()}

    if rank == 0:
        steps = args.steps
        line = {
            "metric": METRIC, "value": value, "unit": "MP/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "round2_denoise_images": int((last["rounds"] == 2).sum()), "frames_per_gpu": N_FRAMES,
                       "frame": [FRAME_H, FRAME_W], "whole_frame_forward": "each frame is forwarded whole after reflect-padding to x32 (the reference's semantics; 180 GB of HBM hold it); halo tiling is used where a frame is sharded (frame_sharded) and is parity-tested against the whole-frame forward",
                       "l2_policy": "inputs (390 MB per step) and activations exceed the 126 MB L2; no explicit flush",
                       "device_lanes": "one host thread, one stream, no host synchronisation between pack and the final inverse VST",
                       "parallelism": f"image-parallel x{world}, NCCL gather of the denoised frames to rank 0 every step (asynchronous: overlaps the next step, drained inside the timed region)" if world > 1 else "single GPU"},
            "e2e": {"value": e2e, "unit": "MP/s", "h2d_bytes_per_step": int(host_in.numel() * 4), "d2h_bytes_per_step": int(host_out.numel() * 4),
                    "ms_per_step": ms_e2e / steps,
                    "api": f"YOND_SIDD.iter_denoise_host(wait=False): pinned host buffers in/out, groups of {E2E_GROUP_FRAMES} frames; H2D of group g+1 and D2H of group g-1 on their own streams while group g computes; one host thread; the K steps are streamed (step k+1 is submitted before step k's numbers are collected, every step's result is collected inside the timed region)"},
            "e2e_dropin": {"value": dropin_frames, "unit": "MP/s (one rank)",
                           "api": "YOND_SIDD.IterDenoise({'lr': np (3024,4032)}, {'p': p}) -> np arrays, one frame per call, 4 calls (pageable NumPy in and out, like the reference's eval loop)"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_tf / peak_tf if peak_tf else None,
                         "traffic": traffic, "traffic_note": traffic_note,
                         "kernel": "conv_tc_kernel (tcgen05 implicit-GEMM conv stack)",
                         "flops_per_launch": prof["conv_flops"] / max(prof["launches"], 1),
                         "ms_per_launch": prof["conv_ms"] / max(prof["launches"], 1),
                         "share_of_step": (prof["conv_ms"] / steps) / (ms / steps),
                         "measured_in": "the timed region (CUDA events around every conv launch on the launching stream)",
                         "peak_source": peak_src + " bf16_tflops_sustained",
                         "conv_ms_per_step": prof["conv_ms"] / steps, "conv_launches": prof["launches"],
                         "algorithmic_flops_per_step": prof["conv_flops"] / steps},
            "roofline_hbm": {"peak_gbs": peak_hbm, "peak_source": peak_src + " hbm_gbs", "bound": "hbm",
                             "measured_in": "the timed region (CUDA events around every stage on the launching stream); bytes = algorithmic bytes per Bayer pixel (SURVEY 8d) x pixels",
                             "kernels": hbm_table(hbm_prof, peak_hbm)},
            "numa_node": numa_node,
            "e2e_raw16": {"value": e2e16, "unit": "MP/s", "ms_per_step": ms_e2e16 / steps, "h2d_bytes_per_step": int(host_in16.numel() * 2),
                          "d2h_bytes_per_step": int(host_out.numel() * 4),
                          "api": "the e2e call on uint16 sensor mosaics: iter_denoise_host(..., raw=(black, white, ratio)); the estimator and the "
                                 "VST front end normalise on load, the float32 input frame never exists"},
            "frame_sharded": frame_sharded,
            "secondary": secondary,
            "cpu_baseline": cpu_base,
        }
        if world == 1:  # BASELINE configs[4], second half: isolated HBM-kernel sweep (device-resident, ~5 s; tools/hbm_sweep.py)
            try:
                sys.path.insert(0, os.path.join(ROOT, "tools"))
                import hbm_sweep
                line["kernel_sweep"] = {"what": "pack / unpack / uint16 ingest / estimator (maps + fit) / fused VST front / fused inverse back / sRGB render / block metrics, isolated, "
                                                "1 ... 256 MP of Bayer pixels; frac = algorithmic bytes / time / hbm peak",
                                        "rows": hbm_sweep.sweep(peak_gbs=peak_hbm)}
            except Exception as e:  # the sweep is an extra: never lose the bench line over it
                line["kernel_sweep"] = {"error": repr(e)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step of the headline workload (rank 0) "
                    "as DIR/<name>.npy; the inputs are the same in every run")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
