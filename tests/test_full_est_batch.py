"""Round 1 of IterDenoise on the full-resolution frames (lr_full) for a whole batch: NlfEstimator.estimate_frames (the self estimate of
frames of different sizes in one pass), iter_denoise_dev / iter_denoise_batch(lr_full=...) and the drop-in IterDenoise with 'lr_full'.
The batch must equal one estimate / one call per image, and the oracle."""
import os
import re

import numpy as np
import pytest
import torch

from oracle import yond_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARCH = {"name": "GuidedResUnet", "guided": True, "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1, "res": True, "norm": True}
PIPE = {"full_est": True, "est_type": "simple+full", "k": 29, "full_dn": False, "vst_type": "exact", "bias_corr": "pre",
        "iter": "iter", "max_iter": 1}
P = {"wp": 1023, "bl": 64, "ratio": 1, "gain": 1, "sigma": 0, "scale": 959.0}
NQ = 20  # percentiles 5, 10, ..., 100 (step 5)
NEW_SYMBOLS = ("yond_nlf_maps_frames", "yond_nlf_fit_ragged_work_bytes", "yond_nlf_fit_ragged", "yond_seg_max")


# ------------------------------------------------------------------ CPU
def test_new_symbols_in_header_and_binding():
    from yond_public_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "yond_b200.h")).read()
    declared = set(re.findall(r"\b(yond_[a-z0-9_]+)\s*\(", hdr))
    for name in NEW_SYMBOLS:
        assert name in declared and name in _lib.SIGNATURES, name
    assert "typedef struct yond_frame_geom" in hdr
    from yond_public_b200.nlf import FRAME_GEOM
    assert FRAME_GEOM.itemsize == 24 and FRAME_GEOM.names == ("base", "H", "W", "off")


def _cpu_frame(H, W, dtype=torch.float32):
    return torch.zeros((H, W), dtype=dtype)


@pytest.mark.parametrize("frames,nimg,match", [
    ([_cpu_frame(64, 96)] * 2, 3, "3 frame"),                        # wrong number of frames
    (torch.zeros((2, 64, 96)), 3, "3 frame"),
    ([], None, "at least one"),
    ([_cpu_frame(64, 95)], 1, "even"),                                # odd W
    ([_cpu_frame(63, 96)], 1, "even"),                                # odd H
    ([_cpu_frame(28, 96), _cpu_frame(64, 96)], 2, "filter radius"),  # packed 14 rows: not larger than the radius 14
    ([_cpu_frame(96, 28)], 1, "filter radius"),
    ([_cpu_frame(64, 96, torch.float64)], 1, "float32"),
    ([_cpu_frame(96, 64).t()], 1, "contiguous"),
    ([_cpu_frame(64, 96)], 1, "CUDA"),
    ([np.zeros((64, 96), np.float32)], 1, "2-D"),
    (torch.zeros(64), 1, "tensor"),
])
def test_check_frames_rejects_malformed(frames, nimg, match):
    from yond_public_b200.nlf import check_frames
    with pytest.raises(ValueError, match=match):
        check_frames(frames, nimg, 29)


def test_lr_full_with_raw_rejected_before_any_launch():
    from yond_public_b200.pipeline import YOND_SIDD
    drv = object.__new__(YOND_SIDD)  # no network, no device: the check comes first
    drv.pipe = dict(PIPE)
    x = torch.zeros((1, 1, 64, 96), dtype=torch.int16)
    with pytest.raises(ValueError, match="raw"):
        drv.iter_denoise_dev(x, dict(P), lr_full=[_cpu_frame(64, 96)], raw=(64, 1023, 1))


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def Y():
    import yond_public_b200 as Y
    return Y


def _frame(rng, H, W, K=4.0, S=6.0, saturate=False):
    x = O.synth_noisy(rng, O.synth_clean_smooth(rng, H, W), K, S)
    if saturate:  # a saturated region: lap == 0 over a large area, the dense third-level select of the order statistics
        x[: H // 2, : W // 3] = 1.0
    return x


def _defined(detail):
    """The entries of estimate_*(details=True) rows the fit writes: th, index, percent, redo flag, ths[:NQ], npeaks[:NQ]."""
    return torch.cat([detail[..., :4 + NQ], detail[..., 4 + 24:4 + 24 + NQ]], -1)


def _maps_alone(Y, f, k=29):
    """var, mean, lap of yond_nlf_maps_bayer (mode 0) on one frame, flat."""
    from yond_public_b200._lib import check, ptr, stream_ptr
    lib = Y._lib.load()
    H, W = f.shape
    var, mean, lap = (torch.empty(H * W, device="cuda") for _ in range(3))
    work = torch.empty(int(lib.yond_nlf_work_bytes(1, H // 2, W // 2, 4)), device="cuda", dtype=torch.uint8)
    check(lib.yond_nlf_maps_bayer(ptr(f), 0, None, 0, ptr(var), ptr(mean), ptr(lap), 1, 1, H, W, 0, k, 0, None, ptr(work), stream_ptr()))
    return var, mean, lap


# three sizes; the second is much smaller than the others (the CTAs past its extent return at once), the third has a clipped region
SIZES = [(384, 1024, False), (128, 288, False), (512, 704, True)]


@pytest.fixture(scope="module")
def frames():
    rng = np.random.default_rng(31)
    return [_frame(rng, H, W, 3.0 + 2 * i, 5.0 + 4 * i, sat) for i, (H, W, sat) in enumerate(SIZES)]


@pytest.mark.gpu
def test_ragged_estimate_equals_per_frame_estimates(Y, frames):
    est = Y.nlf.NlfEstimator()
    fr = [torch.from_numpy(f).cuda() for f in frames]
    var, mean, lap, off, _ = est.maps_frames(fr)
    maps = [m.clone() for m in (var, mean, lap)]
    regs, detail = est.estimate_frames(fr, details=True)
    assert regs.shape == (3, 2) and regs.dtype == torch.float64 and regs.is_cuda
    for i, f in enumerate(fr):
        alone = _maps_alone(Y, f)
        for name, a, b in zip(("var", "mean", "lap"), maps, alone):
            assert torch.equal(a[int(off[i]):int(off[i + 1])], b), (i, name)
        r1, d1 = est.estimate_dev(f[None, None], details=True)
        # th, index, percent, redo flag, ths, npeaks: the same bits
        assert torch.equal(_defined(detail[i]), _defined(d1[0])), i
        # (beta1, beta2) come from float64 atomics: equal up to the order of the additions
        np.testing.assert_allclose(regs[i].cpu().numpy(), r1[0].cpu().numpy(), rtol=1e-10)
    assert float(detail[2, 4]) == 0.0  # the saturated frame's 5th percentile of lap sits in the flat region


@pytest.mark.gpu
def test_ragged_estimate_matches_oracle(Y, frames):
    regs = Y.nlf.NlfEstimator().estimate_frames([torch.from_numpy(f).cuda() for f in frames]).cpu().numpy()
    for i, f in enumerate(frames):
        ref = np.asarray(O.SimpleNLF(f, k=29, setting={"mode": "self"}), np.float64)
        np.testing.assert_allclose(regs[i], ref, rtol=1e-4, err_msg=str(i))


@pytest.mark.gpu
def test_same_size_frames_equal_stacked_estimate(Y):
    rng = np.random.default_rng(7)
    x = torch.from_numpy(np.stack([_frame(rng, 256, 512, 2.0 + i, 4.0 + 3 * i) for i in range(3)])).cuda()
    est = Y.nlf.NlfEstimator()
    r_dev, d_dev = est.estimate_dev(x[:, None], details=True)
    maps_dev = est._scr["maps3"][:3 * x.numel() * 4].view(torch.float32).clone()
    r_fr, d_fr = est.estimate_frames(x, details=True)
    maps_fr = est._scr["maps3"][:3 * x.numel() * 4].view(torch.float32)
    assert torch.equal(maps_dev, maps_fr)
    assert torch.equal(_defined(d_dev), _defined(d_fr))
    np.testing.assert_allclose(r_fr.cpu().numpy(), r_dev.cpu().numpy(), rtol=1e-10)
    r_list = est.estimate_frames(list(x.unbind(0)))  # a list of the same frames
    np.testing.assert_allclose(r_list.cpu().numpy(), r_dev.cpu().numpy(), rtol=1e-10)


def _sidd_image(rng, n, K, S):
    return np.stack([O.synth_noisy(rng, O.synth_clean_smooth(rng, n, n), K, S) for _ in range(32)])


def _batch(rng, full_sizes, n=64):
    """nimg SIDD-shaped images of 32 (n, n) blocks and a full frame of its own size for each, same noise per image."""
    ks = [(3.0, 5.0), (8.0, 20.0), (5.0, 9.0), (4.0, 7.0)]
    blocks, full = [], []
    for i, (H, W) in enumerate(full_sizes):
        K, S = ks[i % len(ks)]
        blocks.append(_sidd_image(rng, n, K, S))
        full.append(_frame(rng, H, W, K, S))
    return np.stack(blocks), full


@pytest.mark.gpu
@pytest.mark.parametrize("use_lut", [False, True])
def test_batch_lr_full_equals_per_image_iterdenoise(Y, use_lut):
    rng = np.random.default_rng(17)
    imgs, full = _batch(rng, [(256, 512), (192, 384), (320, 448)])
    drv = Y.YOND_SIDD(ARCH, PIPE, state_dict=O.smoother_state_dict(ARCH), biaslut="default" if use_lut else None)
    x = torch.from_numpy(imgs).cuda()
    fr = [torch.from_numpy(f).cuda() for f in full]
    res = drv.iter_denoise_batch(x, dict(P), lr_full=fr)
    assert len(res["raw_dns"]) == 2
    for i in range(3):
        one = drv.IterDenoise({"lr": x[i], "lr_full": fr[i]}, {"p": dict(P), "img_id": i})
        assert int(res["rounds"][i]) == len(one["raw_dns"]), i
        for r in range(len(one["raw_dns"])):
            assert torch.equal(res["raw_dns"][r][i], one["raw_dns"][r]), (i, r)
            np.testing.assert_allclose(res["regs"][r][i], np.asarray(one["regs"][r], np.float64), rtol=1e-10)
    # one (nimg, H, W) tensor when the frames share a size
    same = torch.stack([fr[0]] * 3)
    a = drv.iter_denoise_batch(x, dict(P), lr_full=same)
    b = drv.iter_denoise_batch(x, dict(P), lr_full=[fr[0]] * 3)
    assert torch.equal(a["raw_dns"][-1], b["raw_dns"][-1])
    with pytest.raises(ValueError, match="3 frame"):
        drv.iter_denoise_batch(x, dict(P), lr_full=fr[:2])
    with pytest.raises(ValueError, match="even"):
        drv.iter_denoise_batch(x, dict(P), lr_full=[fr[0], fr[1][:, :-1].contiguous(), fr[2]])


def _psnr(a, b):
    return 10 * np.log10(1.0 / np.mean((np.asarray(a, np.float64) - np.asarray(b, np.float64)) ** 2))


@pytest.mark.gpu
def test_batch_lr_full_matches_oracle(Y, lut_table):
    rng = np.random.default_rng(23)
    n = 64
    cleans, imgs, full = [], [], []
    for K, S, (H, W) in ((4.0, 6.0, (256, 384)), (9.0, 15.0, (192, 512))):
        c = np.stack([O.synth_clean_smooth(rng, n, n) for _ in range(32)])
        cleans.append(np.concatenate(list(c), axis=-1))
        imgs.append(np.stack([O.synth_noisy(rng, b, K, S) for b in c]))
        full.append(_frame(rng, H, W, K, S))
    sd = O.smoother_state_dict(ARCH)
    drv = Y.YOND_SIDD(ARCH, PIPE, state_dict=sd)
    res = drv.iter_denoise_batch(torch.from_numpy(np.stack(imgs)).cuda(), dict(P), lr_full=[torch.from_numpy(f).cuda() for f in full])
    for i in range(2):
        ref = O.IterDenoise(ARCH, sd, imgs[i], dict(P), PIPE, biaslut=O.BiasLUT(lut_table), lr_full=full[i])
        assert int(res["rounds"][i]) == len(ref["raw_dns"]), i
        # the round-1 estimate on the full frame; a collab round's estimate also reflects the network's bf16 output, so the later
        # rounds are held to the frame bars, as in the other oracle tests
        np.testing.assert_allclose(res["regs"][0][i], np.asarray(ref["regs"][0], np.float64), rtol=1e-4, err_msg=str(i))
        for r in range(len(ref["raw_dns"])):
            got = res["raw_dns"][r][i].cpu().numpy()
            assert float(np.abs(got - ref["raw_dns"][r]).max()) < 2e-3, (i, r)
            assert abs(_psnr(got, cleans[i]) - _psnr(ref["raw_dns"][r], cleans[i])) < 0.02, (i, r)


@pytest.mark.gpu
def test_batch_lr_full_per_image_exposure(Y):
    """Per-image p['wp'] / p['bl'] / p['scale'] with lr_full, without a LUT (each image gets a fallback table up to its own bound)."""
    rng = np.random.default_rng(29)
    imgs, full = _batch(rng, [(192, 320), (256, 448)])
    wps, bls = np.array([1023, 4095]), np.array([64, 256])
    drv = Y.YOND_SIDD(ARCH, PIPE, state_dict=O.smoother_state_dict(ARCH), biaslut=None)
    x = torch.from_numpy(imgs).cuda()
    fr = [torch.from_numpy(f).cuda() for f in full]
    res = drv.iter_denoise_batch(x, dict(P, wp=wps, bl=bls, scale=(wps - bls).astype(np.float64)), lr_full=fr)
    for i in range(2):
        one = drv.iter_denoise_batch(x[i:i + 1], dict(P, wp=int(wps[i]), bl=int(bls[i]), scale=float(wps[i] - bls[i])), lr_full=fr[i:i + 1])
        assert int(res["rounds"][i]) == int(one["rounds"][0])
        for r in range(len(res["raw_dns"])):
            assert torch.equal(res["raw_dns"][r][i], one["raw_dns"][r][0]), (i, r)
            np.testing.assert_allclose(res["regs"][r][i], one["regs"][r][0], rtol=1e-10, equal_nan=True)


@pytest.mark.gpu
def test_lr_full_launch_count_independent_of_sizes(Y):
    rng = np.random.default_rng(37)
    imgs, full = _batch(rng, [(256, 384), (192, 512), (256, 384), (320, 320)])
    x = torch.from_numpy(imgs).cuda()
    mixed = [torch.from_numpy(f).cuda() for f in full]
    uniform = [mixed[0]] * 4
    drv = Y.YOND_SIDD(ARCH, PIPE, state_dict=O.smoother_state_dict(ARCH))

    def launches(fr):
        drv.iter_denoise_dev(x, dict(P), lr_full=fr)  # warm-up: one-time attributes and buffers
        torch.cuda.synchronize()
        n0 = Y._lib.launch_count()
        drv.iter_denoise_dev(x, dict(P), lr_full=fr)
        torch.cuda.synchronize()
        return Y._lib.launch_count() - n0
    assert launches(mixed) == launches(uniform) > 0
