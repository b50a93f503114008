"""Per-image exposure parameters in one batch: p['wp'] / p['bl'] / p['scale'] and raw = (black, white, ratio[, clip]) given per image
to the batched pipeline (iter_denoise_dev / _batch / _host).  A mixed batch must equal one call per image, and an array of equal
values must give the same bits as the scalar call."""
import numpy as np
import pytest
import torch

from oracle import yond_oracle as O

ARCH = {"name": "GuidedResUnet", "guided": True, "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1, "res": True, "norm": True}
PIPE = {"full_est": True, "est_type": "simple+full", "k": 29, "full_dn": False, "vst_type": "exact", "bias_corr": "pre",
        "iter": "iter", "max_iter": 2}
P = {"wp": 1023, "bl": 64, "ratio": 1, "gain": 1, "sigma": 0, "scale": 959.0}
TOL_ABS = 2e-3
TOL_EST = 1e-4


def _sidd_image(rng, n=64, K=4.0, S=6.0):
    return np.stack([O.synth_noisy(rng, O.synth_clean_smooth(rng, n, n), K, S) for _ in range(32)])


def _raw14(rng, shape, bls, wp, ratios):
    """uint16 (nimg, 1, H, W) mosaics synthesised like test_uint16_equals_float_max_iter_2, with each image's black level and ratio."""
    out = []
    for bl, ratio in zip(bls, ratios):
        dn = O.synth_clean_smooth(rng, *shape) * (wp - bl) / ratio
        out.append(np.clip(rng.poisson(np.maximum(dn, 0) / 2.0) * 2.0 + rng.normal(0, 3.0, dn.shape) + bl, 0, wp).astype(np.uint16))
    return np.stack(out)[:, None]


# ------------------------------------------------------------------ host-side resolution (CPU)
def test_batch_exposure_broadcasts_scalars():
    from yond_public_b200.pipeline import batch_exposure
    se, sc, rec = batch_exposure(dict(P), 3)
    assert se.tolist() == [959.0] * 3 and sc.tolist() == [959.0] * 3 and rec is None
    se, sc, rec = batch_exposure({"wp": 16383, "bl": [512, 600], "scale": np.array([158.71, 15783.0])}, 2, raw=(512, 16383, [100, 1]))
    assert se.tolist() == [15871.0, 15783.0] and sc.tolist() == [158.71, 15783.0]
    assert rec["black"].tolist() == [512.0, 512.0] and rec["white"].tolist() == [16383.0] * 2
    assert rec["ratio"].tolist() == [100.0, 1.0] and rec["clip"].tolist() == [0, 0]
    se, sc, _ = batch_exposure({"wp": (1023, 4095), "bl": (64, 256)}, 2)  # scale defaults to wp - bl
    assert se.tolist() == sc.tolist() == [959.0, 3839.0]
    _, _, rec = batch_exposure(dict(P), 2, raw=(64, 1023, 1, [True, False]))
    assert rec["clip"].tolist() == [1, 0]


@pytest.mark.parametrize("p,raw", [
    (dict(P, wp=[1023, 1023]), None),                       # wrong length
    (dict(P, scale=np.full((3, 1), 959.0)), None),          # not 1-D
    (dict(P, bl=[64, 64, 1023]), None),                     # wp <= bl
    (dict(P, wp=[1023, 60, 1023]), None),
    (dict(P, scale=[959.0, 0.0, 959.0]), None),             # scale <= 0
    (dict(P, scale=-1.0), None),
    (dict(P, wp=[1023, np.nan, 1023]), None),               # non-finite
    (dict(P, scale=np.inf), None),
    (dict(P), (64, 1023, [1, 0, 1])),                       # ratio <= 0
    (dict(P), (64, 1023, -2.0)),
    (dict(P), ([64, 64], 1023, 1)),                         # wrong length in raw
    (dict(P), (64, [1023, 64, 1023], 1)),                   # white <= black
    (dict(P), (np.nan, 1023, 1)),                           # non-finite in raw
    (dict(P), (64, 1023)),                                  # not (black, white, ratio[, clip])
])
def test_batch_exposure_rejects_malformed(p, raw):
    from yond_public_b200.pipeline import batch_exposure
    with pytest.raises(ValueError):
        batch_exposure(p, 3, raw)


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def Y():
    import yond_public_b200 as Y
    return Y


def _record_chains(monkeypatch, drv):
    """Keeps a copy of the params bytes and t of every chain the pipeline fills."""
    seen = []
    orig = drv.engine.chain_params

    def wrapped(*a, **k):
        ch = orig(*a, **k)
        seen.append((ch["params"].clone(), ch["t"].clone()))
        return ch
    monkeypatch.setattr(drv.engine, "chain_params", wrapped)
    return seen


def _dev_equal(a, b, ca, cb):
    assert len(a["dns"]) == len(b["dns"]) and len(ca) == len(cb) == len(a["dns"])
    for r in range(len(a["dns"])):
        assert torch.equal(a["dns"][r], b["dns"][r]), r
        assert torch.equal(a["live"][r], b["live"][r]), r
        # the fit's masked sums add float64 values with atomics, so two runs of the same call differ in the last bits of (beta1, beta2);
        # the intercept beta2 of a collab round can lose a few digits to cancellation (observed: 4.5e-12 relative on sigma)
        np.testing.assert_allclose(a["regs4"][r].cpu().numpy(), b["regs4"][r].cpu().numpy(), rtol=1e-10)
        assert torch.equal(ca[r][0], cb[r][0]) and torch.equal(ca[r][1], cb[r][1]), r


@pytest.mark.gpu
def test_uniform_arrays_bit_identical_to_scalars(Y, monkeypatch):
    rng = np.random.default_rng(4)
    sd = O.smoother_state_dict(ARCH)
    # SIDD blocks, two collab rounds, with the LUT
    x = torch.from_numpy(np.stack([_sidd_image(rng, 64, 4.0, 6.0 + 3 * i) for i in range(3)])).cuda()
    drv = Y.YOND_SIDD(ARCH, PIPE, state_dict=sd)
    seen = _record_chains(monkeypatch, drv)
    a = drv.iter_denoise_dev(x, dict(P))
    ca = list(seen)
    seen.clear()
    b = drv.iter_denoise_dev(x, dict(P, wp=[1023] * 3, bl=np.full(3, 64), scale=(959.0,) * 3))
    _dev_equal(a, b, ca, list(seen))
    # 14-bit full frames, full_dn, uint16 input, no LUT
    bl, wp, ratio = 512, 16383, 100
    t16 = torch.from_numpy(_raw14(rng, (192, 256), [bl] * 2, wp, [ratio] * 2).view(np.int16)).cuda()
    drv = Y.YOND_SIDD(ARCH, dict(PIPE, full_dn=True), state_dict=sd, biaslut=None)
    drv.engine.max_value = 4.0
    seen = _record_chains(monkeypatch, drv)
    p = {"wp": wp, "bl": bl, "ratio": ratio, "gain": 1, "sigma": 0, "scale": (wp - bl) / ratio}
    a = drv.iter_denoise_dev(t16, dict(p), raw=(bl, wp, ratio))
    ca = list(seen)
    seen.clear()
    pa = dict(p, wp=[wp] * 2, bl=[bl] * 2, scale=[(wp - bl) / ratio] * 2)
    b = drv.iter_denoise_dev(t16, pa, raw=([bl] * 2, np.array([wp] * 2), [ratio] * 2))
    _dev_equal(a, b, ca, list(seen))


def _equal_per_image(res, singles, tol_regs=1e-9):
    for i, one in enumerate(singles):
        assert int(res["rounds"][i]) == int(one["rounds"][0]), i
        for r in range(len(res["raw_dns"])):
            np.testing.assert_allclose(res["regs"][r][i], one["regs"][r][0], rtol=tol_regs, equal_nan=True)
            assert float((res["raw_dns"][r][i] - one["raw_dns"][r][0]).abs().max()) <= 1e-6, (i, r)


@pytest.mark.gpu
def test_mixed_ratio_batch_equals_per_image_calls(Y):
    """Four 14-bit frames at x1 / x10 / x100 / x200 with different black levels in one call, as float32 frames and as uint16 mosaics."""
    rng = np.random.default_rng(6)
    wp, bls, ratios = 16383, np.array([512, 512, 600, 480]), np.array([1, 10, 100, 200])
    scales = (wp - bls) / ratios
    raw = _raw14(rng, (192, 256), bls, wp, ratios)
    t16 = torch.from_numpy(raw.view(np.int16)).cuda()
    xf = torch.cat([Y.normalize_raw(t16[i:i + 1], int(bls[i]), wp, int(ratios[i])) for i in range(4)])
    drv = Y.YOND_SIDD(ARCH, dict(PIPE, full_dn=True), state_dict=O.smoother_state_dict(ARCH))
    drv.engine.max_value = 4.0
    assert float(xf.max()) < drv.engine.max_value
    p = {"wp": wp, "bl": bls, "ratio": ratios, "gain": 1, "sigma": 0, "scale": scales}
    mixed_f = drv.iter_denoise_batch(xf, dict(p))
    mixed_u = drv.iter_denoise_batch(t16, dict(p), raw=(bls, wp, ratios))
    singles = [drv.iter_denoise_batch(xf[i:i + 1], {"wp": wp, "bl": int(bls[i]), "ratio": int(ratios[i]), "gain": 1, "sigma": 0,
                                                    "scale": float(scales[i])}) for i in range(4)]
    assert len(mixed_f["raw_dns"]) == 3
    _equal_per_image(mixed_f, singles)
    _equal_per_image(mixed_u, singles)
    assert mixed_u["rounds"].tolist() == mixed_f["rounds"].tolist()
    for r in range(3):
        assert torch.equal(mixed_u["raw_dns"][r], mixed_f["raw_dns"][r]), r
        np.testing.assert_allclose(mixed_u["regs"][r], mixed_f["regs"][r], rtol=1e-10, equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("use_lut", [False, True])
def test_mixed_sidd_images_equal_per_image_calls(Y, use_lut):
    """32-block images with the SIDD_256 collab estimate and white / black levels 1023 / 64 and 4095 / 256 in one batch: without a
    LUT every image gets a fallback table of its own bound."""
    rng = np.random.default_rng(9)
    imgs = np.stack([_sidd_image(rng, 64, K, S) for K, S in ((3.0, 5.0), (8.0, 20.0), (5.0, 9.0))])
    wps, bls = np.array([1023, 4095, 1023]), np.array([64, 256, 64])
    drv = Y.YOND_SIDD(ARCH, PIPE, state_dict=O.smoother_state_dict(ARCH), biaslut="default" if use_lut else None)
    x = torch.from_numpy(imgs).cuda()
    res = drv.iter_denoise_batch(x, dict(P, wp=wps, bl=bls, scale=(wps - bls).astype(np.float64)))
    singles = [drv.iter_denoise_batch(x[i:i + 1], dict(P, wp=int(wps[i]), bl=int(bls[i]), scale=float(wps[i] - bls[i]))) for i in range(3)]
    _equal_per_image(res, singles)


@pytest.mark.gpu
def test_chain_params_per_image_scales_equal_make_params(Y):
    """yond_vst_params_fill with per-image (scale_est, scale, bound_scale) == the host make_params of each image on its own for given
    regs: bitwise for LUT rows, table values to 1e-7."""
    net = Y.build_net(ARCH)
    rec_dt = np.dtype([("gain", "<f4"), ("sigma", "<f4"), ("scale", "<f4"), ("lower", "<f4"), ("upper", "<f4"), ("lut_row", "<i4"),
                       ("table_n", "<i4"), ("exact", "<i4")])
    regs = np.array([[5e-3, 4e-5], [2.1e-3, -3e-6], [8e-4, 9e-5]], np.float64)  # third: sigma/K = 12.4 -> fallback
    scale_est = np.array([959.0, 3839.0, 15871.0])
    scale = scale_est / np.array([1.0, 10.0, 100.0])
    seg_max = torch.tensor([0.93, 1.0, 0.4], device="cuda")
    for biaslut in (Y.BiasLUT(), None):
        eng = Y.YondEngine(net, ARCH, biaslut)
        ch = eng.chain_params(torch.from_numpy(regs).cuda(), seg_max, 3, 2, scale_est, scale, scale_est, 1, "pre", "exact")
        a = ch["params"].cpu().numpy().view(rec_dt)
        r4 = ch["regs4"].cpu().numpy()
        for i in range(3):
            g, s = regs[i, 0] * scale_est[i], np.sqrt(max(regs[i, 1], 0)) * scale_est[i]
            fmax = lambda: np.repeat(seg_max[i:i + 1].cpu().numpy() * np.float32(scale_est[i]), 2)
            params, rows, xnodes, _, t = eng.make_params([g, g], [s, s], scale[i], "pre", "exact", fmax, "cuda")
            b = params.cpu().numpy().view(rec_dt)
            for f in ("gain", "sigma", "scale", "lower", "upper", "table_n", "exact"):
                assert np.array_equal(a[f][2 * i:2 * i + 2], b[f]), (i, f)
            assert np.array_equal(ch["t"].cpu().numpy()[2 * i:2 * i + 2], t.cpu().numpy())
            assert r4[i, 2] == g and r4[i, 3] == s
            for fr in range(2):
                n = int(b["table_n"][fr]) or 1921
                ra = ch["rows"][a["lut_row"][2 * i + fr], :n].cpu().numpy()
                rb = rows[b["lut_row"][fr], :n].cpu().numpy()
                np.testing.assert_allclose(ra, rb, rtol=0, atol=0 if b["table_n"][fr] == 0 else 1e-7)
                assert np.array_equal(ch["xnodes"][a["lut_row"][2 * i + fr], :n].cpu().numpy(), xnodes[b["lut_row"][fr], :n].cpu().numpy())
        if biaslut is None:  # rows sized for the largest bound of the batch
            assert ch["stride"] >= int(eng.lib.yond_bias_table_nodes(float(np.float32(eng.max_value) * np.float32(scale_est.max()))))


@pytest.mark.gpu
def test_vst_denoise_per_frame_scale(Y):
    """The caller-given (K, sigma) surface with one scale per frame equals one call per frame."""
    rng = np.random.default_rng(5)
    x = torch.from_numpy(np.stack([O.synth_noisy(rng, O.synth_clean_smooth(rng, 96, 128), 4.0, 6.0) for _ in range(3)])).cuda()
    eng = Y.YondEngine(Y.build_net(ARCH), ARCH, None)
    eng.net.load_state_dict(O.smoother_state_dict(ARCH))
    gains, sigmas, scales = [4.1, 30.0, 2.2], [6.2, 80.0, 1.5], [959.0, 3839.0, 158.71]
    out = eng.vst_denoise(x, gains, sigmas, scales)
    for i in range(3):
        one = eng.vst_denoise(x[i:i + 1], gains[i], sigmas[i], scales[i])
        assert float((out[i] - one[0]).abs().max()) <= 1e-6, i


@pytest.mark.gpu
def test_host_path_per_image_p_equals_batched(Y):
    rng = np.random.default_rng(13)
    imgs = np.stack([_sidd_image(rng, 64, 4.0, 6.0 + i) for i in range(6)])
    wps = np.array([1023, 4095, 1023, 16383, 4095, 1023])
    bls = np.array([64, 256, 64, 512, 240, 70])
    p = dict(P, wp=wps, bl=bls, scale=list((wps - bls) / np.array([1, 4, 1, 16, 4, 1])))
    drv = Y.YOND_SIDD(ARCH, PIPE, state_dict=O.smoother_state_dict(ARCH))
    ref = drv.iter_denoise_batch(torch.from_numpy(imgs).cuda(), dict(p))
    hin = torch.from_numpy(imgs).pin_memory()
    hout = torch.zeros((6, 64, 32 * 64)).pin_memory()
    res = drv.iter_denoise_host(hin, hout, dict(p), group=[3, 1, 2])
    assert torch.equal(hout, ref["raw_dns"][-1].cpu())
    assert np.array_equal(res["rounds"], ref["rounds"])
    for r in range(3):
        got = np.concatenate([np.atleast_2d(s[r]) for s in res["regs"]])
        np.testing.assert_allclose(got, ref["regs"][r], rtol=1e-10, equal_nan=True)


@pytest.mark.gpu
def test_mixed_batch_vs_oracle(Y, lut_table):
    """Two images with their own p in one call against oracle.IterDenoise run per image with that image's p."""
    rng = np.random.default_rng(21)
    imgs = np.stack([_sidd_image(rng, 128, 4.0, 6.0), _sidd_image(rng, 128, 9.0, 15.0)])
    ps = [dict(P), dict(P, wp=4095, bl=256, scale=3839.0)]
    pipe = dict(PIPE, max_iter=1)
    sd = O.smoother_state_dict(ARCH)
    drv = Y.YOND_SIDD(ARCH, pipe, state_dict=sd)
    res = drv.iter_denoise_batch(torch.from_numpy(imgs).cuda(), dict(P, wp=[1023, 4095], bl=[64, 256], scale=[959.0, 3839.0]))
    for i in range(2):
        ref = O.IterDenoise(ARCH, sd, imgs[i], dict(ps[i]), pipe, biaslut=O.BiasLUT(lut_table))
        np.testing.assert_allclose(res["regs"][0][i], np.asarray(ref["regs"][0], np.float64), rtol=TOL_EST)
        assert int(res["rounds"][i]) == len(ref["raw_dns"])
        for r in range(len(ref["raw_dns"])):
            assert float(np.abs(res["raw_dns"][r][i].cpu().numpy() - ref["raw_dns"][r]).max()) < TOL_ABS, (i, r)
