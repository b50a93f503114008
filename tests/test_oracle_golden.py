"""CPU: the oracle (oracle/yond_oracle.py) replays the golden vectors produced by the UNMODIFIED reference
(tests/golden/make_golden.py).  This is what pins the oracle; the GPU tests then compare CUDA to the oracle."""
import zlib

import numpy as np
import pytest
import torch

from oracle import yond_oracle as O

ARCHS = {
    "unet": {"name": "UNetSeeInDark", "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1, "res": True, "norm": True},
    "gru": {"name": "GuidedResUnet", "guided": True, "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1,
            "res": True, "norm": True},
    "snr": {"name": "SNRnet", "guided": True, "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1,
            "res": True, "norm": True},
    "res2": {"name": "ResUnet2", "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1, "res": True, "norm": True},
    "selfres": {"name": "SelfResUNet", "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1, "res": True, "norm": True},
    "gself": {"name": "GuidedSelfUnet", "guided": True, "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1, "res": False, "norm": True},
}
PIPE = {"k": 29, "full_dn": False, "vst_type": "exact", "bias_corr": "pre", "iter": "iter", "max_iter": 1}


def crc(a):
    return np.uint32(zlib.crc32(np.ascontiguousarray(a).tobytes()))


def test_pack_bit_exact(golden):
    g = golden("pack")
    assert np.array_equal(O.bayer2rggb(g["bayer"]), g["rggb"])
    assert np.array_equal(O.rggb2bayer(g["rggb"]), g["back"])
    assert np.array_equal(g["back"], g["bayer"])


def test_vst_and_inverse(golden):
    g = golden("vst")
    K, s = np.float64(g["K"]), np.float64(g["sigma"])
    z = O.VST(g["x"], s, gain=K)
    assert z.dtype == np.float64  # NumPy-2 promotion: the reference runs this stage in float64
    np.testing.assert_array_equal(z, g["z"])
    np.testing.assert_array_equal(O.inverse_VST(z, s, gain=K, exact=False), g["inv_alg"])
    np.testing.assert_allclose(O.inverse_VST(np.concatenate([z, [0.0, -1.0]]), s, gain=K, exact=True), g["inv_exact"],
                               rtol=1e-15, atol=0)
    assert O.VST(0, s, gain=K) == g["lower"] and O.VST(959.0, s, gain=K) == g["upper"]


def test_biaslut(golden, lut_table):
    g = golden("biaslut")
    assert crc(lut_table) == g["lut_crc"], "stand-in LUT differs from the one the goldens were made with"
    lut = O.BiasLUT(lut_table)
    np.testing.assert_array_equal(lut.x_lut, g["x_lut"])
    np.testing.assert_array_equal(lut.sg_lut, g["sg_lut"])
    for i, (K, s) in enumerate(g["cases"]):
        out = lut.get_lut(g["x"], K=np.float64(K), sigGs=np.float64(s))
        np.testing.assert_array_equal(out, g[f"bias{i}"])
        row = lut.sigma_row(np.float64(K), np.float64(s))
        assert row.shape == (1921,)


def test_fallback_bias_table(golden):
    g = golden("getbias")
    f = O.get_bias(np.float32(700.0), np.float64(6.0), np.float64(4.0))
    np.testing.assert_array_equal(f.x, g["nodes"])
    np.testing.assert_allclose(f(g["x"]), g["bias"], rtol=0, atol=1e-12)
    f2 = O.get_bias(np.float32(40.0), np.float64(0.9), np.float64(0.4))
    np.testing.assert_array_equal(f2.x, g["nodes2"])
    np.testing.assert_allclose(f2(g["x2"]), g["bias2"], rtol=0, atol=1e-12)


def test_stdfilt_and_blur(golden):
    g = golden("stdfilt")
    np.testing.assert_array_equal(O.stdfilt(g["img"], 29), g["std29"])
    np.testing.assert_array_equal(O.stdfilt(g["img"], 5), g["std5"])
    np.testing.assert_array_equal(O.blur(g["img"], 19), g["blur19"])
    # the NumPy restatement of cv2.blur (used when cv2 is missing, and as the spec for the CUDA kernel)
    np.testing.assert_allclose(O.box_blur_np(g["img"], 19), g["blur19"], rtol=0, atol=6e-8)
    np.testing.assert_allclose(O.box_blur_np(g["img"], 29), O.blur(g["img"], 29), rtol=0, atol=6e-8)


def test_estimators(golden):
    g = golden("nlf")
    r2 = np.random.default_rng(int(g["seed"]))
    clean = O.synth_clean(r2, 256, 384)
    noisy = O.synth_noisy(r2, clean, 6.0, 9.0)
    rggb = O.bayer2rggb(noisy)
    var, mean, lap = O.self_maps(rggb, 29)
    assert crc(lap) == g["lap_crc"]
    np.testing.assert_array_equal(mean[::16, ::16], g["mean_sub"])
    np.testing.assert_array_equal(var[::16, ::16], g["var_sub"])
    th, pct, _ = O.get_threshold_score3(lap, mean, step=5)
    assert th == g["th"] and pct == g["pct"]
    np.testing.assert_allclose(O.SimpleNLF(noisy, k=29, setting={"mode": "self"}), g["reg_self"], rtol=1e-12)
    blocks_c = np.stack([O.synth_clean(r2, 64, 64) for _ in range(32)])
    blocks_n = np.stack([O.synth_noisy(r2, b, 6.0, 9.0) for b in blocks_c])
    blocks_d = np.stack([np.clip(b + 0.004 * r2.standard_normal(b.shape), 0, 1).astype(np.float32) for b in blocks_c])
    mos_n, mos_d = np.concatenate(list(blocks_n), -1), np.concatenate(list(blocks_d), -1)
    np.testing.assert_allclose(O.SimpleNLF(mos_n, mos_d, 29, {"mode": "collab", "SIDD_256": True}), g["reg_collab"],
                               rtol=1e-12)
    np.testing.assert_allclose(O.SimpleNLF(mos_n, mos_d, 29, {"mode": "collab"}), g["reg_collab_plain"], rtol=1e-12)


def test_get_p2d(golden):
    g = golden("p2d")
    for s, p in zip(g["shapes"], g["p2d"]):
        assert O.get_p2d(tuple(int(v) for v in s), base=32) == tuple(int(v) for v in p)


@pytest.mark.parametrize("key", ["unet", "gru", "snr", "res2", "selfres", "gself"])
def test_networks(golden, key):
    g = golden(f"net_{key}")
    arch = ARCHS[key]
    sd = O.init_state_dict(arch, seed=5)
    assert [str(k) for k in g["keys"]] == list(sd.keys())
    assert [str(s) for s in g["shapes"]] == [str(tuple(v.shape)) for v in sd.values()]
    assert np.array_equal(np.array([crc(v.numpy()) for v in sd.values()], np.uint32), g["sd_crc"])
    assert int(g["nparams"]) == {"unet": 7760484, "gru": 11173668, "snr": 11176612, "res2": 11173668, "selfres": 512036, "gself": 529540}[key]
    x = torch.from_numpy(g["x"])
    with torch.no_grad():
        y = O.net_forward(arch, sd, x, torch.tensor(0.043) if "guided" in arch else None)
    np.testing.assert_allclose(y.numpy(), g["y"], rtol=0, atol=2e-6)
    # bf16 emulation of the CUDA path's stores must stay well inside the 2e-3 budget on random-init weights
    with torch.no_grad():
        yb = O.net_forward(arch, sd, x, torch.tensor(0.043) if "guided" in arch else None, bf16=True)
    assert float((yb - y).abs().max()) < 5e-4


def test_vst_denoiser(golden, lut_table):
    g = golden("vst_denoiser")
    p = {"wp": 1023, "bl": 64, "ratio": 1, "scale": 959.0, "gain": np.float64(g["gain"]), "sigma": np.float64(g["sigma"])}
    lut = O.BiasLUT(lut_table)
    for key, out, kw in (("gru", "out_gru", dict(biaslut=lut)), ("snr", "out_snr", dict(biaslut=lut)),
                         ("unet", "out_unet", dict(biaslut=None)),
                         ("unet", "out_unet_nobias", dict(biaslut=None, bias_corr=None))):
        sd = O.init_state_dict(ARCHS[key], seed=5)
        bc = kw.pop("bias_corr", "pre")
        res = O.VST_Denoiser(ARCHS[key], sd, g["noisy"], p, bias_corr=bc, **kw)
        np.testing.assert_allclose(res, g[out], rtol=0, atol=3e-6, err_msg=out)
    sd = O.init_state_dict(ARCHS["unet"], seed=5)
    np.testing.assert_allclose(O.Simple_Denoiser(ARCHS["unet"], sd, g["noisy"]), g["out_simple"], rtol=0, atol=3e-6)


def _blocks(seed, K, S):
    r4 = np.random.default_rng(seed)
    return np.stack([O.synth_noisy(r4, O.synth_clean(r4, 256, 256), K, S) for _ in range(32)])


@pytest.mark.parametrize("key", ["gru", "unet"])
def test_iterdenoise_random_init(golden, lut_table, key):
    g = golden(f"iter_{key}")
    blocks = _blocks(int(g["seed"]), float(g["K"]), float(g["sigma"]))
    assert crc(blocks) == g["blocks_crc"], "synthetic input generator drifted"
    sd = O.init_state_dict(ARCHS[key], seed=5)
    p = {"wp": 1023, "bl": 64, "ratio": 1, "gain": 1, "sigma": 0, "scale": 959.0}
    res = O.IterDenoise(ARCHS[key], sd, blocks, p, PIPE, biaslut=O.BiasLUT(lut_table) if key == "gru" else None)
    assert len(res["raw_dns"]) == int(g["nrounds"]) == 1  # random weights: round 2 aborts on beta1 < 0 (:445-447)
    np.testing.assert_allclose(np.array(res["regs"][0]), g["regs"][0], rtol=1e-10)
    np.testing.assert_allclose(res["raw_dns"][0][::8, ::8], g["dn0_sub"], rtol=0, atol=3e-6)


@pytest.mark.parametrize("key", ["gru", "unet"])
def test_iterdenoise_two_rounds(golden, lut_table, key):
    g = golden(f"iter2_{key}")
    blocks = _blocks(int(g["seed"]), float(g["K"]), float(g["sigma"]))
    sd = O.smoother_state_dict(ARCHS[key])
    p = {"wp": 1023, "bl": 64, "ratio": 1, "gain": 1, "sigma": 0, "scale": 959.0}
    res = O.IterDenoise(ARCHS[key], sd, blocks, p, PIPE, biaslut=O.BiasLUT(lut_table))
    assert len(res["raw_dns"]) == 2
    np.testing.assert_allclose(np.array([np.asarray(r) for r in res["regs"]]), g["regs"], rtol=1e-9)
    np.testing.assert_allclose(res["raw_dns"][0][::8, ::8], g["dn0_sub"], rtol=0, atol=3e-6)
    np.testing.assert_allclose(res["raw_dns"][1][::8, ::8], g["dn1_sub"], rtol=0, atol=3e-6)


def test_pack_raw_bayer_golden(golden):
    """SURVEY 8(f)-1: the oracle's pack_raw_bayer == the reference's (data_process/process.py:40-64), bit for bit, on four CFA
    patterns, 10/12/14-bit ranges, per-channel black levels, clip on and off."""
    g = golden("pack_raw")
    for i in range(int(g["n"])):
        out = O.pack_raw_bayer(g[f"img{i}"], g[f"pattern{i}"], g[f"black{i}"].tolist(), wp=int(g[f"wp{i}"]), clip=bool(g[f"clip{i}"]))
        assert out.dtype == np.float32
        assert np.array_equal(out, g[f"out{i}"]), i


def test_rot_bayer_golden(golden):
    """The oracle's rot_bayer == the reference's (utils/sidd_utils.py:198-213) for every CFA pattern, forward and reverse."""
    g = golden("pack_raw")
    for pi in range(4):
        for rev in (0, 1):
            assert np.array_equal(O.rot_bayer(g["rot_in"], g[f"rot_pat{pi}"].tolist(), rev=bool(rev)), g[f"rot_out{pi}_{rev}"])
            assert np.array_equal(O.rot_bayer(g["rot_in"][0], g[f"rot_pat{pi}"].tolist(), rev=bool(rev)), g[f"rot2d_out{pi}_{rev}"])


# ---- BASELINE configs[3]: 14-bit frame, noclip, low-light gain, whole-frame denoise (full_dn), two rounds ----
ARCH_GRU = ARCHS["gru"]
PIPE_C4 = {"k": 29, "full_dn": True, "vst_type": "exact", "bias_corr": "pre", "iter": "iter", "max_iter": 1}


def c4_frame(ratio, H, W):
    """The frame make_golden_c4.py fed to the reference, regenerated from its seed."""
    rng = np.random.default_rng(4000 + ratio)
    clean = O.synth_clean_smooth(rng, H, W)
    return O.synth_noisy(rng, clean, 2.2 * ratio, 3.1 * ratio, scale=16383.0 - 512.0, clip=False)


def c4_weights(name):
    sm = O.smoother_state_dict(ARCH_GRU)
    if name == "smooth":
        return sm
    rnd = O.init_state_dict(ARCH_GRU, seed=0)
    return {k: sm[k] + 0.25 * rnd[k] for k in rnd}


@pytest.mark.parametrize("ratio,wname", [(1, "smooth"), (100, "smooth"), (100, "mix")])
def test_iterdenoise_c4_frame(golden, lut_table, ratio, wname):
    g = golden("c4_frame")
    H, W = int(g["H"]), int(g["W"])
    noisy = c4_frame(ratio, H, W)
    p = {"wp": 16383, "bl": 512, "ratio": ratio, "gain": 1, "sigma": 0, "scale": (16383 - 512) / ratio}
    res = O.IterDenoise(ARCH_GRU, c4_weights(wname), noisy, p, PIPE_C4, biaslut=O.BiasLUT(lut_table))
    tag = f"r{ratio}_{wname}"
    assert len(res["raw_dns"]) == int(g[f"{tag}_nrounds"]) == 2
    np.testing.assert_allclose(np.array([np.asarray(r, np.float64) for r in res["regs"]]), g[f"{tag}_regs"], rtol=1e-6)
    for i, dn in enumerate(res["raw_dns"]):
        assert float(np.abs(dn[::4, ::8] - g[f"{tag}_dn{i}_sub"]).max()) < 3e-6


# ---- SURVEY 8(f)-3: metrics of the SIDD driver ----
def test_metrics_golden(golden):
    """The oracle's ssim / calculate_ssim == the reference's on the same images (generated by make_golden_metrics.py)."""
    g = golden("metrics")
    nblk = int(g["nblk"])
    dn_ = np.array(np.split(g["dn"], nblk, axis=-1))
    hr_ = np.array(np.split(g["clean"], nblk, axis=-1))
    got = np.array([O.calculate_ssim(d * 255, h * 255) for d, h in zip(dn_, hr_)])
    np.testing.assert_allclose(got, g["ssim_blocks"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(O.calculate_ssim(g["rgb"], g["rgb2"]), g["ssim_rgb"], rtol=0, atol=1e-12)
    np.testing.assert_allclose([O.compare_psnr(d, h, data_range=1) for d, h in zip(dn_, hr_)], g["psnr_blocks"], rtol=1e-12)
    p, s = O.sidd_image_metrics(g["dn"], g["clean"], nblk)
    np.testing.assert_allclose([p, s], [g["psnr_blocks"].mean(), g["ssim_blocks"].mean()], rtol=1e-12)
    assert O.sidd_image_metrics(np.zeros_like(g["dn"]), g["clean"], nblk) == (-1, -1)


# ---- SURVEY 8(f)-3: sRGB render of the SIDD driver ----
RENDER_PATTERNS = [[[1, 2], [2, 3]], [[2, 1], [3, 2]], [[2, 3], [1, 2]], [[3, 2], [2, 1]]]


def test_render_golden(golden):
    """The oracle's process_sidd_image == the reference's (utils/sidd_utils.py:156-180, with this image's cv2 behind its demosaic),
    byte for byte, for every CFA phase incl. flat (all-ties), saturated and out-of-range areas (make_golden_render.py)."""
    g = golden("render")
    for i, pat in enumerate(RENDER_PATTERNS):
        assert np.array_equal(g[f"pat{i}"], np.array(pat))
        got = O.process_sidd_image(g[f"img{i}"], pat, g[f"wb{i}"], g[f"cst{i}"])
        assert got.dtype == np.uint8 and got.shape == g[f"srgb{i}"].shape
        assert np.array_equal(got, g[f"srgb{i}"]), f"pattern {pat}"
    for j in range(2):
        assert np.array_equal(O.demosaic_ea_u16(g[f"bayer{j}"]), g[f"ea{j}"])
    # the sRGB numbers of multiprocess_plot on the rendered pictures: the reference's calculate_ssim on uint8 (H,W,3) inputs
    np.testing.assert_allclose(O.calculate_ssim(g["srgb0"], g["srgb_clean0"]), g["ssim_u8"], rtol=0, atol=1e-12)
    _, ss = O.sidd_rgb_metrics(g["srgb0"], g["srgb_clean0"], nblk=2)
    np.testing.assert_allclose(ss, g["ssim_u8_blocks"].mean(), rtol=0, atol=1e-12)


def test_demosaic_restatement_matches_cv2(golden):
    """The edge-aware demosaic restatement against OpenCV (the third-party routine behind demosaic_CV2), bit for bit, on seeded
    mosaics: full 14-bit range, tiny ranges (gradient ties everywhere), constant images, the smallest legal size.  Checked against
    the CRC-32 of cv2's outputs (make_golden_demosaic.py), and against cv2 itself where it is installed."""
    g = golden("demosaic_cv2")
    rng = np.random.default_rng(int(g["seed"]))
    mosaics = [rng.integers(0, hi, size=(h, w), dtype=np.uint16) for (h, w, hi) in g["cases"].tolist()]
    h, w, v = g["flat"].tolist()
    mosaics.append(np.full((h, w), v, np.uint16))
    assert len(mosaics) == len(g["crc"])
    try:
        import cv2
    except ImportError:
        cv2 = None
    for b, want in zip(mosaics, g["crc"]):
        got = O.demosaic_ea_u16(b)
        assert crc(got) == want, b.shape
        if cv2 is not None:
            assert np.array_equal(got, cv2.cvtColor(b, cv2.COLOR_BayerBG2RGB_EA)), b.shape


def test_rgb_metrics_oracle():
    """compare_psnr on uint8 pictures promotes to float64 (scikit-image's rule for integer inputs); known answer."""
    a = np.zeros((16, 32, 3), np.uint8)
    b = np.full((16, 32, 3), 5, np.uint8)
    np.testing.assert_allclose(O.compare_psnr_u8(a, b), 10 * np.log10(255.0 ** 2 / 25.0), rtol=1e-15)
    c = np.full((16, 32, 3), 15, np.uint8)
    p, s = O.sidd_rgb_metrics(np.concatenate([a, b], 1), np.concatenate([b, c], 1), nblk=2)
    np.testing.assert_allclose(p, 0.5 * (10 * np.log10(255.0 ** 2 / 25.0) + 10 * np.log10(255.0 ** 2 / 100.0)), rtol=1e-15)
    assert 0 < s < 1
