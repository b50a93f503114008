"""Full frames of different sizes through every round of the batched pipeline: YOND_SIDD.iter_denoise_frames(_dev), the ragged collab maps,
the ragged self maps of uint16 mosaics with per-frame normalisation and seg_max, and the table form of the VST front end.  Every image must
get what a call on its frame alone gives."""
import os
import re

import numpy as np
import pytest
import torch

from oracle import yond_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARCH = {"name": "GuidedResUnet", "guided": True, "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1, "res": True, "norm": True}
PIPE = {"full_est": True, "est_type": "simple+full", "k": 29, "full_dn": True, "vst_type": "exact", "bias_corr": "pre",
        "iter": "iter", "max_iter": 2}
P = {"wp": 1023, "bl": 64, "ratio": 1, "gain": 1, "sigma": 0, "scale": 959.0}
NEW_SYMBOLS = ("yond_nlf_maps_frames_max", "yond_nlf_maps_frames_raw16", "yond_nlf_maps_frames_collab_cached", "yond_vst_fwd_frames")


# ------------------------------------------------------------------ CPU
def test_new_symbols_in_header_and_binding():
    from yond_public_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "yond_b200.h")).read()
    declared = set(re.findall(r"\b(yond_[a-z0-9_]+)\s*\(", hdr))
    for name in NEW_SYMBOLS:
        assert name in declared and name in _lib.SIGNATURES, name


def _drv(**pipe):
    from yond_public_b200.pipeline import YOND_SIDD
    drv = object.__new__(YOND_SIDD)  # no network, no device: every check comes before the first launch
    drv.pipe = dict(PIPE, **pipe)
    return drv


def _cpu(H, W, dtype=torch.float32):
    return torch.zeros((H, W), dtype=dtype)


def _misaligned(H, W, dtype, shift):
    return torch.zeros(H * W + shift, dtype=dtype)[shift:].view(H, W)


@pytest.mark.parametrize("frames,p,raw,pipe,match", [
    ([_cpu(64, 95), _cpu(64, 96)], P, None, {}, "even"),                                           # malformed frame
    ([_cpu(28, 96), _cpu(64, 96)], P, None, {}, "filter radius"),
    ([_cpu(64, 96, torch.float64)], P, None, {}, "float32"),
    ([_cpu(96, 64).t()], P, None, {}, "contiguous"),
    ([_cpu(64, 96)], P, None, {}, "CUDA"),
    ([], P, None, {}, "at least one"),
    (torch.zeros((2, 64, 96)), P, None, {}, "list"),
    ([_cpu(64, 96), _cpu(64, 96, torch.uint16)], P, (64, 1023, 1), {}, "mixes"),                  # a mix of dtypes
    ([_cpu(64, 96, torch.int16), _cpu(64, 96)], P, None, {}, "mixes"),
    ([_cpu(64, 96, torch.uint16)], P, None, {}, "raw="),                                           # uint16 without raw=
    ([_cpu(64, 96, torch.int16)], P, None, {}, "raw="),
    ([_cpu(64, 96)], P, (64, 1023, 1), {}, "raw="),                                                # float32 with raw=
    ([_misaligned(64, 96, torch.float32, 1)], P, None, {}, "aligned"),                             # 4 bytes off: float2 loads
    ([_misaligned(64, 96, torch.uint16, 1)], P, (64, 1023, 1), {}, "aligned"),                     # 2 bytes off: 32-bit loads
    ([_cpu(64, 96)], P, None, {"sidd_256": True}, "sidd_256"),
    ([_cpu(64, 96)], P, None, {"full_est": False}, "full_est"),
    ([_cpu(64, 96)], P, None, {"est_type": "full"}, "est_type"),
    ([_cpu(64, 96)], P, None, {"max_iter": -1}, "max_iter"),
    ([_cpu(64, 96)] * 2, dict(P, wp=[1023, 1023, 1023]), None, {}, "2 values"),                    # batch_exposure
    ([_cpu(64, 96)] * 2, dict(P, wp=[1023, 60]), None, {}, "exceed"),
    ([_cpu(64, 96)] * 2, dict(P, scale=0.0), None, {}, "positive"),
    ([_cpu(64, 96, torch.uint16)] * 2, P, (64, 1023, [1, 0]), {}, "ratio"),
    ([_cpu(64, 96, torch.uint16)] * 2, P, (64, [1023, 10], 1), {}, "white"),
    ([_cpu(64, 96, torch.uint16)] * 2, P, (64, 1023), {}, "black, white, ratio"),
])
def test_frames_call_rejected_before_any_launch(frames, p, raw, pipe, match):
    with pytest.raises(ValueError, match=match):
        _drv(**pipe).iter_denoise_frames_dev(frames, dict(p), raw=raw)


def test_too_many_frames_rejected():
    f = _cpu(64, 96)
    with pytest.raises(ValueError, match="65535"):
        _drv().iter_denoise_frames([f] * 65536, dict(P))


def test_check_frames_alignment_and_dtypes():
    from yond_public_b200.nlf import check_frames
    with pytest.raises(ValueError, match="aligned"):
        check_frames([_misaligned(64, 96, torch.float32, 1)], 1, 29)
    with pytest.raises(ValueError, match="CUDA"):  # 8-byte aligned: the next check is reached
        check_frames([_misaligned(64, 96, torch.float32, 2)], 1, 29)
    with pytest.raises(ValueError, match="CUDA"):
        check_frames([_misaligned(64, 96, torch.uint16, 2)], 1, 29, raw=True)
    with pytest.raises(ValueError, match="raw="):
        check_frames([_cpu(64, 96, torch.uint16)], 1, 29)


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def Y():
    import yond_public_b200 as Y
    return Y


def _frame(rng, H, W, K=4.0, S=6.0):
    return O.synth_noisy(rng, O.synth_clean_smooth(rng, H, W), K, S)


# wider than 264 Bayer columns: the box filters take the wide layout, as on the uniform path; three padded sizes
A, B, C = (192, 320), (160, 384), (224, 288)
NOISE = [(3.0, 5.0), (8.0, 20.0), (5.0, 9.0), (4.0, 7.0), (2.0, 4.0)]


def _frames(seed, sizes):
    rng = np.random.default_rng(seed)
    return [torch.from_numpy(_frame(rng, H, W, *NOISE[i % len(NOISE)])).cuda() for i, (H, W) in enumerate(sizes)]


def _uint16(rng, sizes, bls, wps, ratios):
    out = []
    for (H, W), bl, wp, ratio in zip(sizes, bls, wps, ratios):
        dn = O.synth_clean_smooth(rng, H, W) * (wp - bl) / ratio
        raw = np.clip(rng.poisson(np.maximum(dn, 0) / 2.0) * 2.0 + rng.normal(0, 3.0, dn.shape) + bl, 0, wp).astype(np.uint16)
        out.append(torch.from_numpy(raw.view(np.int16)).cuda())
    return out


def _raw_records(Y, bls, wps, ratios):
    from yond_public_b200.pipeline import batch_exposure
    _, _, rec = batch_exposure({"wp": 1, "bl": 0}, len(bls), (bls, wps, ratios))
    return torch.from_numpy(rec.view(np.uint8).copy()).cuda()


@pytest.mark.gpu
def test_ragged_collab_maps_equal_per_frame(Y):
    est = Y.nlf.NlfEstimator()
    lr = _frames(41, [A, B, C])
    y = [torch.from_numpy(np.clip(f.cpu().numpy() * 0.9 + 0.01, 0, 1).astype(np.float32)).cuda() for f in lr]
    table = Y.nlf.FrameTable(lr)
    lr_var = torch.empty(table.n_el, device="cuda")
    est.maps_frames(table, 29, var_map=lr_var)
    flat = torch.cat([f.reshape(-1) for f in y])
    got = [m.clone() for m in est.collab_maps_frames(flat, table, lr_var, 29)]
    for i, (f, g) in enumerate(zip(lr, y)):
        H, W = f.shape
        lv = torch.empty(H * W, device="cuda")
        est.estimate_dev(f[None, None], var_map=lv)  # the cached var map of iter_denoise_dev on this frame alone
        ref = est.collab_maps_cached(g[None], lv, 1, 29)
        sl = slice(int(table.off[i]), int(table.off[i + 1]))
        for name, a, b in zip(("var", "mean", "lap"), got, ref):
            assert torch.equal(a[sl], b), (i, name)


@pytest.mark.gpu
def test_ragged_seg_max_equals_estimate_dev(Y):
    est = Y.nlf.NlfEstimator()
    fr = _frames(43, [A, C, B])
    fr[1][:8, :8] = 1.7  # a frame maximum above 1
    seg = torch.empty(3, device="cuda")
    est.estimate_frames(fr, 29, seg_max=seg)
    for i, f in enumerate(fr):
        one = torch.empty(1, device="cuda")
        est.estimate_dev(f[None, None], seg_max=one)
        assert torch.equal(seg[i:i + 1], one), i


@pytest.mark.gpu
def test_ragged_raw16_maps_equal_float_maps(Y):
    rng = np.random.default_rng(47)
    sizes, bls, wps, ratios = [A, B, C], [64, 512, 256], [1023, 16383, 4095], [1.0, 100.0, 8.0]
    t16 = _uint16(rng, sizes, bls, wps, ratios)
    est = Y.nlf.NlfEstimator()
    seg16, seg32 = torch.empty(3, device="cuda"), torch.empty(3, device="cuda")
    m16 = [m.clone() for m in est.maps_frames(t16, 29, seg_max=seg16, raw=_raw_records(Y, bls, wps, ratios))[:3]]
    f32 = [Y.normalize_raw(t, bl, wp, r) for t, bl, wp, r in zip(t16, bls, wps, ratios)]
    m32 = est.maps_frames(f32, 29, seg_max=seg32)[:3]
    for name, a, b in zip(("var", "mean", "lap"), m16, m32):
        assert torch.equal(a, b), name
    assert torch.equal(seg16, seg32)


@pytest.mark.gpu
def test_table_vst_front_end_equals_stacked(Y):
    from yond_public_b200._lib import check, ptr, stream_ptr
    from yond_public_b200.pipeline import RAW_REC
    drv = Y.YOND_SIDD(ARCH, PIPE, state_dict=O.smoother_state_dict(ARCH))
    eng, lib = drv.engine, drv.engine.lib
    eng.max_value = 4.0
    rng = np.random.default_rng(53)
    n, (H, W) = 3, A
    bls, wps, ratios = [64, 512, 256], [1023, 16383, 4095], [1.0, 100.0, 8.0]
    t16 = _uint16(rng, [A] * n, bls, wps, ratios)
    f32 = [Y.normalize_raw(t, bl, wp, r) for t, bl, wp, r in zip(t16, bls, wps, ratios)]
    regs = torch.tensor([[3e-3, 2e-5], [9e-3, 4e-4], [5e-3, 8e-5]], device="cuda", dtype=torch.float64)
    seg_max = torch.stack([f.amax() for f in f32]).float()
    ch = eng.chain_params(regs, seg_max, n, 1, 959.0, 959.0, 959.0, 1, "pre", "exact")
    nrm = _raw_records(Y, bls, wps, ratios)
    pl, pr, pt, pb = Y.isp.get_p2d((1, 4, H // 2, W // 2), base=32)
    hp, wp = H // 2 + pt + pb, W // 2 + pl + pr
    st = stream_ptr()
    for src, raw in ((f32, None), (t16, nrm)):
        table = Y.nlf.FrameTable(src[::-1])  # the records need not follow the memory order of the frames
        stacked = torch.stack(src[::-1])
        z0, z1 = (torch.empty((n, hp, wp, 4), device="cuda") for _ in range(2))
        u0, u1 = torch.empty(n, device="cuda"), torch.empty(n, device="cuda")
        args = (n, H, W, pl, pr, pt, pb, ptr(ch["params"]), ptr(ch["rows"]), ptr(ch["xnodes"]), ch["stride"], st)
        rec = None if raw is None else torch.from_numpy(np.ascontiguousarray(raw.cpu().numpy().view(RAW_REC)[::-1]).view(np.uint8)).cuda()
        check(lib.yond_vst_fwd_frames(ptr(table.records), ptr(rec), ptr(z1), ptr(u1), *args))
        if raw is None:
            check(lib.yond_vst_fwd(ptr(stacked), ptr(z0), ptr(u0), *args))
        else:
            check(lib.yond_vst_fwd_raw16(ptr(stacked), None, ptr(z0), ptr(u0), *args, ptr(rec), 1))
        assert torch.equal(z0, z1) and torch.equal(u0, u1), raw is None


def _alone(drv, f, p, raw=None):
    return drv.iter_denoise_batch(f[None, None], dict(p), raw=raw)


def _assert_same_as_alone(res, alone, i):
    assert int(res["rounds"][i]) == int(alone["rounds"][0]), i
    assert len(res["raw_dns"]) == len(alone["raw_dns"])
    for r in range(len(res["raw_dns"])):
        assert torch.equal(res["raw_dns"][r][i], alone["raw_dns"][r][0]), (i, r)
        # the masked sums of the fit are added in an order fixed by the frame's size: the same bits alone and in a batch
        np.testing.assert_array_equal(res["regs"][r][i], alone["regs"][r][0], err_msg=f"{i} {r}")


@pytest.mark.gpu
@pytest.mark.parametrize("full_dn", [True, False])
@pytest.mark.parametrize("use_lut", [False, True])
def test_interleaved_sizes_equal_per_frame_calls(Y, full_dn, use_lut):
    fr = _frames(59, [A, B, C, A, B])  # interleaved: the device order groups them by padded size
    drv = Y.YOND_SIDD(ARCH, dict(PIPE, full_dn=full_dn), state_dict=O.smoother_state_dict(ARCH),
                      biaslut="default" if use_lut else None)
    res = drv.iter_denoise_frames(fr, dict(P))
    assert len(res["raw_dns"]) == 3 and all(len(d) == 5 for d in res["raw_dns"])
    assert [tuple(d.shape) for d in res["raw_dns"][0]] == [tuple(f.shape) for f in fr]
    assert sorted(res["dev"]["order"].tolist()) == list(range(5))
    for i, f in enumerate(fr):
        _assert_same_as_alone(res, _alone(drv, f, P), i)


@pytest.mark.gpu
def test_mixed_cameras_uint16(Y):
    rng = np.random.default_rng(61)
    sizes, bls, wps, ratios = [B, A, B], [512, 64, 256], [16383, 1023, 4095], [100.0, 1.0, 8.0]
    t16 = _uint16(rng, sizes, bls, wps, ratios)
    drv = Y.YOND_SIDD(ARCH, PIPE, state_dict=O.smoother_state_dict(ARCH))
    drv.engine.max_value = 4.0
    p = dict(P, wp=wps, bl=bls, scale=[(w - b) / r for w, b, r in zip(wps, bls, ratios)])
    a = drv.iter_denoise_frames(t16, dict(p), raw=(bls, wps, ratios))
    b = drv.iter_denoise_frames([Y.normalize_raw(t, bl, wp, r) for t, bl, wp, r in zip(t16, bls, wps, ratios)], dict(p))
    assert np.array_equal(a["rounds"], b["rounds"])
    for r in range(len(a["raw_dns"])):
        for i in range(3):
            assert torch.equal(a["raw_dns"][r][i], b["raw_dns"][r][i]), (i, r)
        np.testing.assert_array_equal(a["regs"][r], b["regs"][r])
    for i in range(3):
        pi = dict(P, wp=wps[i], bl=bls[i], scale=(wps[i] - bls[i]) / ratios[i])
        _assert_same_as_alone(a, _alone(drv, t16[i], pi, raw=(bls[i], wps[i], ratios[i])), i)


@pytest.mark.gpu
def test_forced_stop(Y, monkeypatch):
    fr = _frames(67, [C, A, B])  # device order A, B, C: device rows 0, 1, 2 are caller frames 1, 2, 0
    drv = Y.YOND_SIDD(ARCH, PIPE, state_dict=O.smoother_state_dict(ARCH))
    base = drv.iter_denoise_frames(fr, dict(P))
    assert base["rounds"].tolist() == [3, 3, 3]  # unforced, every image completes both collab rounds
    est = Y.nlf._estimator()
    orig = type(est).estimate_collab_frames.__get__(est)
    calls = {"n": 0}

    def wrapped(*a, **k):  # device row 2 (caller frame 0) fails the beta1 guard in round 2
        regs = orig(*a, **k)
        if calls["n"] == 0:
            regs[2, 0] = -1e-3
        calls["n"] += 1
        return regs
    monkeypatch.setattr(est, "estimate_collab_frames", wrapped)
    res = drv.iter_denoise_frames(fr, dict(P))
    assert res["dev"]["order"].tolist() == [1, 2, 0]
    assert res["rounds"].tolist() == [1, 3, 3]
    for r in (1, 2):
        assert torch.equal(res["raw_dns"][r][0], res["raw_dns"][0][0]), r
        assert np.isnan(res["regs"][r][0]).all()
    for i in (1, 2):  # the other images continue, with the bits of the unforced run (the fit is deterministic)
        for r in range(3):
            assert torch.equal(res["raw_dns"][r][i], base["raw_dns"][r][i]), (i, r)
            np.testing.assert_array_equal(res["regs"][r][i], base["regs"][r][i])


@pytest.mark.gpu
def test_uniform_list_equals_stacked_batch(Y):
    fr = _frames(71, [A] * 3)
    drv = Y.YOND_SIDD(ARCH, PIPE, state_dict=O.smoother_state_dict(ARCH))
    a = drv.iter_denoise_frames(fr, dict(P))
    b = drv.iter_denoise_batch(torch.stack(fr)[:, None], dict(P))
    assert np.array_equal(a["rounds"], b["rounds"])
    for r in range(3):
        assert torch.equal(torch.stack(a["raw_dns"][r]), b["raw_dns"][r]), r
        np.testing.assert_array_equal(a["regs"][r], b["regs"][r])


def _psnr(a, b):
    return 10 * np.log10(1.0 / np.mean((np.asarray(a, np.float64) - np.asarray(b, np.float64)) ** 2))


@pytest.mark.gpu
def test_frames_match_oracle(Y, lut_table):
    rng = np.random.default_rng(73)
    pipe = dict(PIPE, max_iter=1)
    cleans, noisy = [], []
    for (H, W), (K, S) in zip((A, C), ((4.0, 6.0), (9.0, 15.0))):
        cleans.append(O.synth_clean_smooth(rng, H, W))
        noisy.append(O.synth_noisy(rng, cleans[-1], K, S))
    sd = O.smoother_state_dict(ARCH)
    drv = Y.YOND_SIDD(ARCH, pipe, state_dict=sd)
    res = drv.iter_denoise_frames([torch.from_numpy(f).cuda() for f in noisy], dict(P))
    for i in range(2):
        ref = O.IterDenoise(ARCH, sd, noisy[i], dict(P), pipe, biaslut=O.BiasLUT(lut_table), sidd_256=False)
        assert int(res["rounds"][i]) == len(ref["raw_dns"]), i
        np.testing.assert_allclose(res["regs"][0][i], np.asarray(ref["regs"][0], np.float64), rtol=1e-4, err_msg=str(i))
        for r in range(len(ref["raw_dns"])):
            got = res["raw_dns"][r][i].cpu().numpy()
            assert float(np.abs(got - ref["raw_dns"][r]).max()) < 2e-3, (i, r)
            assert abs(_psnr(got, cleans[i]) - _psnr(ref["raw_dns"][r], cleans[i])) < 0.02, (i, r)


@pytest.mark.gpu
def test_launch_count_depends_on_sizes_only(Y):
    fa, fb = _frames(79, [A, B])
    drv = Y.YOND_SIDD(ARCH, PIPE, state_dict=O.smoother_state_dict(ARCH))

    def launches(fr):
        drv.iter_denoise_frames_dev(fr, dict(P))  # warm-up: one-time attributes and buffers
        torch.cuda.synchronize()
        n0 = Y._lib.launch_count()
        drv.iter_denoise_frames_dev(fr, dict(P))
        torch.cuda.synchronize()
        return Y._lib.launch_count() - n0
    assert launches([fa, fb, fa, fb, fa, fb]) == launches([fa, fb]) > 0
    assert launches([fa] * 4) == launches([fa]) > 0
