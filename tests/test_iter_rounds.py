"""IterDenoise with max_iter > 1 (YOND_SIDD.py:419-472, oracle IterDenoise): N collab rounds in the device pipeline, the live
mask chained over the rounds, the collab maps from cached noisy-frame statistics, and the host bookkeeping of N rounds."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import yond_oracle as O

ARCHS = {
    "unet": {"name": "UNetSeeInDark", "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1, "res": True, "norm": True},
    "gru": {"name": "GuidedResUnet", "guided": True, "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1, "res": True, "norm": True},
}
PIPE = {"full_est": True, "est_type": "simple+full", "k": 29, "full_dn": False, "vst_type": "exact", "bias_corr": "pre",
        "iter": "iter", "max_iter": 1}
P = {"wp": 1023, "bl": 64, "ratio": 1, "gain": 1, "sigma": 0, "scale": 959.0}
TOL_ABS = 2e-3
TOL_EST = 1e-4
REC = np.dtype([("gain", "<f4"), ("sigma", "<f4"), ("scale", "<f4"), ("lower", "<f4"), ("upper", "<f4"), ("lut_row", "<i4"),
                ("table_n", "<i4"), ("exact", "<i4")])
VST_FIELDS = ("gain", "sigma", "scale", "lower", "upper", "exact")


def _sidd_image(rng, n=128, K=4.0, S=6.0):
    return np.stack([O.synth_noisy(rng, O.synth_clean_smooth(rng, n, n), K, S) for _ in range(32)])


# ------------------------------------------------------------------ host bookkeeping (CPU)
def test_read_summary_three_rounds_mixed_stops():
    from yond_public_b200.pipeline import YOND_SIDD
    regs4 = [torch.tensor([[1e-3 * (i + 1), 2e-5, 0.959 * (i + 1), 0.1] for i in range(3)], dtype=torch.float64) + r
             for r in (0.0, 1e-4, 2e-4)]
    live = [torch.ones(3, dtype=torch.int32), torch.tensor([1, 0, 1], dtype=torch.int32), torch.tensor([1, 0, 0], dtype=torch.int32)]
    regs, rounds, gains = YOND_SIDD.read_summary({"regs4": regs4, "live": live})
    assert rounds.tolist() == [3, 1, 2]
    assert len(regs) == len(gains) == 3
    assert not np.isnan(regs[0]).any()
    assert np.isnan(regs[1][1]).all() and not np.isnan(regs[1][[0, 2]]).any()
    assert np.isnan(regs[2][[1, 2]]).all() and not np.isnan(regs[2][0]).any()
    np.testing.assert_array_equal(regs[2][0], regs4[2][0, :2].numpy())
    for r in range(3):  # (gain, sigma) are the estimates' values, not masked
        np.testing.assert_array_equal(gains[r], regs4[r][:, 2:].numpy())


@pytest.mark.parametrize("bad", [-1, 1.5, "2", None, True])
def test_max_iter_validation(bad):
    from yond_public_b200.pipeline import collab_rounds
    with pytest.raises(ValueError):
        collab_rounds(dict(PIPE, max_iter=bad))


def test_collab_rounds_count():
    from yond_public_b200.pipeline import collab_rounds
    assert [collab_rounds(dict(PIPE, max_iter=n)) for n in (0, 1, 3)] == [0, 1, 3]
    assert collab_rounds(dict(PIPE, iter="once", max_iter=3)) == 0
    assert collab_rounds(dict(PIPE, max_iter=np.int64(2))) == 2


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def Y():
    import yond_public_b200 as Y
    return Y


def _params(ch):
    return ch["params"].cpu().numpy().view(REC)


@pytest.mark.gpu
def test_liveness_chained_over_rounds(Y):
    """Four images over four rounds: all live; stops at round 2; stops at round 3 with beta1 >= 0 again at round 4; beta2 < 0 at
    round 3.  The live mask is chained, a stopped image keeps its last live round's VST parameters, gain / sigma are computed
    before the beta1 guard."""
    eng = Y.YondEngine(Y.build_net(ARCHS["gru"]), ARCHS["gru"], Y.BiasLUT())
    rounds = [
        [[4e-3, 1e-5], [3e-3, 2e-5], [5e-3, 3e-5], [2e-3, 1e-5]],
        [[4.1e-3, 1.1e-5], [-2e-3, 1e-5], [5.1e-3, 3.1e-5], [2.1e-3, 1.2e-5]],
        [[4.2e-3, 1.2e-5], [3.5e-3, 2e-5], [-1e-3, 3.2e-5], [2.2e-3, -1e-6]],
        [[4.3e-3, 1.3e-5], [3.6e-3, 2e-5], [5.3e-3, 3.3e-5], [2.3e-3, 1.4e-5]],
    ]
    fps = 2
    chains = []
    for r, regs in enumerate(rounds, start=1):
        t = torch.tensor(regs, device="cuda", dtype=torch.float64)
        chains.append(eng.chain_params(t, None, 4, fps, 959, 959.0, 959, r, "pre", "exact", prev=chains[-1] if chains else None))
    oks = [c["ok"].cpu().tolist() for c in chains]
    assert oks == [[1, 1, 1, 1], [1, 0, 1, 1], [1, 0, 0, 1], [1, 0, 0, 1]]
    last_live = {1: 0, 2: 1}  # image -> index of its last live round
    for r in range(1, 4):
        pa = _params(chains[r])
        for img, lr in last_live.items():
            if r <= lr:
                continue
            pl = _params(chains[lr])
            for f in VST_FIELDS:
                assert np.array_equal(pa[f][img * fps:(img + 1) * fps], pl[f][img * fps:(img + 1) * fps]), (r, img, f)
            assert (pa["lut_row"][img * fps:(img + 1) * fps] == -1).all()  # no bias row of this round is filled for it
        r4 = chains[r]["regs4"].cpu().numpy()
        b1 = np.array([x[0] for x in rounds[r]])
        b2 = np.array([x[1] for x in rounds[r]])
        b2g = np.where(b2 < 0, b1 * b1, b2)
        np.testing.assert_array_equal(r4[:, 0], b1)
        np.testing.assert_array_equal(r4[:, 1], b2g)
        np.testing.assert_array_equal(r4[:, 2], b1 * 959)  # before the guard: stopped images too
        np.testing.assert_array_equal(r4[:, 3], np.sqrt(b2g) * 959)


BASE_REGS = (4.2e-3, 3.9e-5)  # K = 4, sigma = 6 at scale 959: what the collab estimates of these images give, made exact


def _override(monkeypatch, forced):
    """Wraps the estimator's collab estimate: every image gets BASE_REGS, then forced = {(call index, image): beta1} (call 0 = round 2
    of the next run) — the rounds an image stays live no longer depend on the data."""
    from yond_public_b200 import nlf
    est = nlf._estimator()
    orig = type(est).estimate_collab_cached.__get__(est)  # the method itself, not an earlier wrapper
    calls = {"n": 0}

    def wrapped(*a, **k):
        regs = orig(*a, **k)
        regs[:, 0], regs[:, 1] = BASE_REGS
        for (c, img), b1 in forced.items():
            if c == calls["n"]:
                regs[img, 0] = b1
        calls["n"] += 1
        return regs
    monkeypatch.setattr(est, "estimate_collab_cached", wrapped)
    return calls


@pytest.mark.gpu
def test_stopped_images_through_the_pipeline(Y, monkeypatch):
    rng = np.random.default_rng(5)
    imgs = np.stack([_sidd_image(rng, 64) for _ in range(3)])
    drv = Y.YOND_SIDD(ARCHS["gru"], dict(PIPE, max_iter=3), state_dict=O.smoother_state_dict(ARCHS["gru"]))
    x = torch.from_numpy(imgs).cuda()
    _override(monkeypatch, {})
    base = drv.iter_denoise_batch(x, dict(P))
    assert base["rounds"].tolist() == [4, 4, 4]
    # image 1 stops at round 2, image 2 at round 3
    _override(monkeypatch, {(0, 1): -1e-3, (1, 2): -2e-3})
    res = drv.iter_denoise_batch(x, dict(P))
    assert res["rounds"].tolist() == [4, 1, 2]
    dns = res["raw_dns"]
    assert len(dns) == 4 and len(res["regs"]) == 4
    for r in (1, 2, 3):
        assert torch.equal(dns[r][1], dns[0][1]), r
    for r in (2, 3):
        assert torch.equal(dns[r][2], dns[1][2]), r
    for r in range(4):  # the other image does not notice (float64-atomic order of the fit sums aside)
        assert float((dns[r][0] - base["raw_dns"][r][0]).abs().max()) < 1e-6
    nan = [np.isnan(res["regs"][r][:, 0]).tolist() for r in range(4)]
    assert nan == [[False] * 3, [False, True, False], [False, True, True], [False, True, True]]
    # the drop-in surface: raw_dns / regs of the completed rounds; p ends with the last EVALUATED round's (gain, sigma)
    for img, forced, n_dns, r_eval in ((0, {}, 4, 3), (1, {(0, 0): -1e-3}, 1, 1), (2, {(1, 0): -2e-3}, 2, 2)):
        _override(monkeypatch, forced)
        log = []
        drv._log = lambda m: log.append(m)
        p = dict(P)
        one = drv.IterDenoise({"lr": imgs[img], "name": "x"}, {"p": p, "img_id": img})
        assert len(one["raw_dns"]) == len(one["regs"]) == n_dns
        for r in range(n_dns):
            np.testing.assert_allclose(one["raw_dns"][r], dns[r][img].cpu().numpy(), rtol=0, atol=1e-6)
        g = res["dev"]["regs4"][r_eval][img].cpu().numpy()
        np.testing.assert_allclose([p["gain"], p["sigma"]], g[2:], rtol=1e-9)
        assert sum(m.startswith("Iter ") for m in log) == r_eval
        assert sum(m.startswith("Warning") for m in log) == (1 if n_dns < 4 else 0)


def _oracle_round(arch, sd, blocks, mosaic, pp, full_dn, lut):
    """The oracle's VST denoise of one collab round with given (gain, sigma) (oracle IterDenoise.run)."""
    scale = P["wp"] - P["bl"]
    if full_dn:
        bf = O.get_bias(mosaic.max() * scale, pp["sigma"], pp["gain"]) if lut is None else None
        return O.VST_Denoiser(arch, sd, mosaic, pp, "pre", lut, bf, "exact").clip(0, 1)
    bf = O.get_bias(blocks.max() * scale, pp["sigma"], pp["gain"]) if lut is None else None
    return np.concatenate([O.VST_Denoiser(arch, sd, b, pp, "pre", lut, bf, "exact").clip(0, 1) for b in blocks], axis=-1)


@pytest.mark.gpu
@pytest.mark.parametrize("key,geom,use_lut", [("gru", "sidd", True), ("gru", "frame", True), ("unet", "sidd", True),
                                              ("unet", "frame", True), ("unet", "frame", False)])
def test_rounds_vs_oracle(Y, lut_table, key, geom, use_lut):
    """max_iter = 3 against the oracle: every collab round on identical inputs (our previous output), and end to end."""
    rng = np.random.default_rng(17)
    arch, sd = ARCHS[key], O.smoother_state_dict(ARCHS[key])
    if geom == "sidd":
        blocks = _sidd_image(rng, 128)
        pipe = dict(PIPE, max_iter=3)
        mosaic = np.concatenate(list(blocks), axis=-1)
        x = torch.from_numpy(blocks).cuda()[None]
    else:
        mosaic = O.synth_noisy(rng, O.synth_clean_smooth(rng, 384, 512), 4.0, 6.0)
        blocks = mosaic
        pipe = dict(PIPE, full_dn=True, max_iter=3)
        x = torch.from_numpy(mosaic).cuda().reshape(1, 1, *mosaic.shape)
    lut = O.BiasLUT(lut_table) if use_lut else None
    drv = Y.YOND_SIDD(arch, pipe, state_dict=sd, biaslut="default" if use_lut else None)
    res = drv.iter_denoise_dev(x, dict(P))
    dns = [d[0].cpu().numpy() for d in res["dns"]]
    r4 = [t.cpu().numpy()[0] for t in res["regs4"]]
    live = [int(t.cpu()[0]) for t in res["live"]]
    assert len(dns) == 4
    for r in range(1, 4):
        ref = O.SimpleNLF(mosaic, dns[r - 1], k=29, setting={"mode": "collab", "SIDD_256": geom == "sidd"})
        ref = (ref[0], ref[0] ** 2) if ref[1] < 0 else ref
        np.testing.assert_allclose(r4[r][:2], np.asarray(ref, np.float64), rtol=TOL_EST)
        if live[r]:
            pp = dict(P, gain=r4[r][2], sigma=r4[r][3])
            out = _oracle_round(arch, sd, blocks, mosaic, pp, geom == "frame", lut)
            assert float(np.abs(dns[r] - out).max()) < TOL_ABS, r
        else:
            assert np.array_equal(dns[r], dns[r - 1])
    ref = O.IterDenoise(arch, sd, blocks, dict(P), pipe, biaslut=lut, sidd_256=geom == "sidd")
    regs, rounds, _ = drv.read_summary(res)
    assert int(rounds[0]) == len(ref["raw_dns"])
    for r in range(int(rounds[0])):
        assert float(np.abs(dns[r] - ref["raw_dns"][r]).max()) < TOL_ABS, r
        ours, theirs = regs[r][0], np.asarray(ref["regs"][r], np.float64)
        if r == 0:
            np.testing.assert_allclose(ours, theirs, rtol=TOL_EST)
            continue
        # from round 2 on the input is our previous output, which differs from the oracle's by the bf16 conv stack, and the
        # difference compounds over the rounds: the input-drift bar of the two-round golden test, on beta1 and on sigma = sqrt(beta2)
        # (the quantity the VST uses; beta2 is the fit's intercept, whose relative drift is twice sigma's)
        np.testing.assert_allclose(ours[0], theirs[0], rtol=2e-3)
        np.testing.assert_allclose(np.sqrt(ours[1]), np.sqrt(theirs[1]), rtol=2e-3)


def _close(a, b):
    assert a["rounds"].tolist() == b["rounds"].tolist()
    assert len(a["raw_dns"]) == len(b["raw_dns"])
    for i in range(len(a["raw_dns"])):
        np.testing.assert_allclose(np.asarray(a["regs"][i]), np.asarray(b["regs"][i]), rtol=1e-10, equal_nan=True)
        assert float((a["raw_dns"][i] - b["raw_dns"][i]).abs().max()) < 1e-6, i


@pytest.mark.gpu
@pytest.mark.parametrize("geom", ["sidd", "frame"])
def test_prefix_property(Y, geom):
    """Rounds 1..k+1 of a max_iter = 3 run are a max_iter = k run."""
    rng = np.random.default_rng(8)
    if geom == "sidd":
        x = torch.from_numpy(np.stack([_sidd_image(rng, 64) for _ in range(2)])).cuda()
        pipe = dict(PIPE)
    else:
        x = torch.from_numpy(np.stack([O.synth_noisy(rng, O.synth_clean_smooth(rng, 192, 320), 4.0, 6.0 + i) for i in range(2)])[:, None]).cuda()
        pipe = dict(PIPE, full_dn=True)
    sd = O.smoother_state_dict(ARCHS["gru"])
    full = Y.YOND_SIDD(ARCHS["gru"], dict(pipe, max_iter=3), state_dict=sd).iter_denoise_batch(x, dict(P))
    assert len(full["raw_dns"]) == 4
    for k in (0, 1, 2):
        part = Y.YOND_SIDD(ARCHS["gru"], dict(pipe, max_iter=k), state_dict=sd).iter_denoise_batch(x, dict(P))
        cut = {"raw_dns": full["raw_dns"][:k + 1], "regs": full["regs"][:k + 1],
               "rounds": np.minimum(full["rounds"], k + 1)}
        _close(cut, part)


def _mode1_maps(Y, x, y, nblk, split, x_mosaic, raw=None):
    """Collab maps of the two-pass mode 1 of yond_nlf_maps_bayer / _raw16 (x, y in the given layouts, y in the mosaic layout)."""
    lib = Y._lib.load()
    from yond_public_b200._lib import check, ptr, stream_ptr
    if x_mosaic:
        nimg, H, Wm = x.shape
        W = Wm // nblk
    else:
        nimg, _, H, W = x.shape
    n = Y.nlf.NlfEstimator.collab_geometry(nimg, nblk, H, W, split)
    B, h = (nimg * nblk if split else nimg), H // 2
    w = (W // 2) if split else nblk * (W // 2)
    var, mean, lap = (torch.empty(n, device="cuda") for _ in range(3))
    work = torch.empty(int(lib.yond_nlf_work_bytes(B, h, w, 4)), device="cuda", dtype=torch.uint8)
    if raw is not None:
        check(lib.yond_nlf_maps_raw16(ptr(x), C.byref(raw), int(x_mosaic), ptr(y), 1, ptr(var), ptr(mean), ptr(lap), nimg, nblk, H, W,
                                      int(split), 29, 1, None, ptr(work), stream_ptr()))
    else:
        check(lib.yond_nlf_maps_bayer(ptr(x), int(x_mosaic), ptr(y), 1, ptr(var), ptr(mean), ptr(lap), nimg, nblk, H, W, int(split), 29, 1,
                                      None, ptr(work), stream_ptr()))
    return var, mean, lap


@pytest.mark.gpu
def test_cached_collab_maps_equal_two_pass_maps(Y):
    """The collab maps from the cached std_k(lr)^2 (self estimate's var map, or the one-pass lr_var) equal mode 1's bit for bit:
    plain mosaics, SIDD strips (blocks layout and split out of a frame) and a uint16 source."""
    rng = np.random.default_rng(2)
    est = Y.nlf._estimator()

    def check_maps(ref, got):
        for a, b, name in zip(ref, got, ("var", "mean", "lap")):
            assert torch.equal(a, b[:a.numel()]), name

    # plain mosaics of 4 blocks (one image per mosaic), lr statistics from the self estimate
    x = torch.from_numpy(np.stack([_sidd_image(rng, 64)[:4] for _ in range(2)])).cuda()  # (2, 4, 64, 64)
    y = (x.permute(0, 2, 1, 3).reshape(2, 64, 256) * 0.9).contiguous()
    n = est.collab_geometry(2, 4, 64, 64, False)
    self_var = torch.empty(n, device="cuda")
    est.estimate_dev(x, None, 29, var_map=self_var)
    lr_var = torch.empty(n, device="cuda")
    est.lr_var_dev(x, lr_var, 29)
    assert torch.equal(self_var, lr_var)
    check_maps(_mode1_maps(Y, x, y, 4, False, False), [m.clone() for m in est.collab_maps_cached(y, self_var, 4, 29)])
    # SIDD strips: blocks layout, and 32 strips of a frame (mosaic layout)
    xb = torch.from_numpy(_sidd_image(rng, 64)[None]).cuda()
    yb = (xb.permute(0, 2, 1, 3).reshape(1, 64, 32 * 64) ** 2).contiguous()
    lr_var = torch.empty(est.collab_geometry(1, 32, 64, 64, True), device="cuda")
    est.lr_var_dev(xb, lr_var, 29, split_blocks=True)
    check_maps(_mode1_maps(Y, xb, yb, 32, True, False), [m.clone() for m in est.collab_maps_cached(yb, lr_var, 32, 29, split_blocks=True)])
    xf = xb.permute(0, 2, 1, 3).reshape(1, 64, 32 * 64).contiguous()
    est.lr_var_dev(xf, lr_var, 29, split_blocks=True, x_mosaic=True, nblk=32)
    check_maps(_mode1_maps(Y, xf, yb, 32, True, True), [m.clone() for m in est.collab_maps_cached(yb, lr_var, 32, 29, split_blocks=True)])
    # uint16 sensor mosaic, plain frame and SIDD strips
    raw16 = torch.from_numpy(rng.integers(64, 1024, size=(2, 1, 96, 2048), dtype=np.uint16).view(np.int16)).cuda()
    rn = Y._lib.RawNorm(64.0, 1023.0, 1.0, 0)
    yr = torch.from_numpy(rng.uniform(0, 1, size=(2, 96, 2048)).astype(np.float32)).cuda()
    for split, nb, xr, xm in ((False, 1, raw16, False), (True, 32, raw16.reshape(2, 96, 2048), True)):
        lr_var = torch.empty(est.collab_geometry(2, nb, 96, 2048 // nb, split), device="cuda")
        est.lr_var_dev(xr, lr_var, 29, split_blocks=split, x_mosaic=xm, nblk=nb, raw=rn)
        check_maps(_mode1_maps(Y, xr, yr, nb, split, xm, raw=rn), [m.clone() for m in est.collab_maps_cached(yr, lr_var, nb, 29, split_blocks=split)])


@pytest.mark.gpu
def test_batched_equals_per_image_max_iter_2(Y):
    rng = np.random.default_rng(11)
    imgs = np.stack([_sidd_image(rng, 64, K, S) for K, S in ((2.0, 3.0), (9.0, 14.0), (5.0, 40.0))])
    drv = Y.YOND_SIDD(ARCHS["gru"], dict(PIPE, max_iter=2), state_dict=O.smoother_state_dict(ARCHS["gru"]))
    res = drv.iter_denoise_batch(torch.from_numpy(imgs).cuda(), dict(P))
    assert len(res["raw_dns"]) == 3
    for i in range(len(imgs)):
        one = drv.IterDenoise({"lr": imgs[i], "name": "x"}, {"p": dict(P), "img_id": i})
        assert len(one["raw_dns"]) == int(res["rounds"][i])
        for r in range(len(one["regs"])):
            np.testing.assert_allclose(res["regs"][r][i], np.asarray(one["regs"][r]), rtol=1e-9)
            np.testing.assert_allclose(res["raw_dns"][r][i].cpu().numpy(), one["raw_dns"][r], rtol=0, atol=1e-6)


@pytest.mark.gpu
def test_uint16_equals_float_max_iter_2(Y):
    rng = np.random.default_rng(3)
    sd = O.smoother_state_dict(ARCHS["gru"])
    cases = [(dict(PIPE, full_dn=True, max_iter=2), (2, 1, 192, 256), 512, 16383, 100, {"wp": 16383, "bl": 512, "ratio": 100, "scale": (16383 - 512) / 100}),
             (dict(PIPE, max_iter=2), (1, 32, 64, 64), 64, 1023, 1, dict(P))]
    for pipe, shape, bl, wp, ratio, p in cases:
        clean = np.stack([O.synth_clean_smooth(rng, shape[2], shape[3] * shape[1]) for _ in range(shape[0])])
        dn = clean * (wp - bl) / ratio
        raw = np.clip(rng.poisson(np.maximum(dn, 0) / 2.0) * 2.0 + rng.normal(0, 3.0, dn.shape) + bl, 0, wp).astype(np.uint16)
        raw = raw.reshape(shape[0], shape[2], shape[1], shape[3]).transpose(0, 2, 1, 3).copy()
        drv = Y.YOND_SIDD(ARCHS["gru"], pipe, state_dict=sd)
        drv.engine.max_value = 4.0
        p = dict(p, gain=1, sigma=0)
        t16 = torch.from_numpy(raw.view(np.int16)).cuda()
        a = drv.iter_denoise_batch(t16, dict(p), raw=(bl, wp, ratio))
        b = drv.iter_denoise_batch(Y.normalize_raw(t16, bl, wp, ratio), dict(p))
        assert len(a["raw_dns"]) == 3
        _close(a, b)


@pytest.mark.gpu
def test_host_path_equals_batched_max_iter_2(Y):
    rng = np.random.default_rng(13)
    imgs = np.stack([_sidd_image(rng, 64, 4.0, 6.0 + i) for i in range(5)])
    drv = Y.YOND_SIDD(ARCHS["gru"], dict(PIPE, max_iter=2), state_dict=O.smoother_state_dict(ARCHS["gru"]))
    ref = drv.iter_denoise_batch(torch.from_numpy(imgs).cuda(), dict(P))
    hin = torch.from_numpy(imgs).pin_memory()
    hout = torch.zeros((5, 64, 32 * 64)).pin_memory()
    res = drv.iter_denoise_host(hin, hout, dict(P), group=2)
    assert torch.equal(hout, ref["raw_dns"][-1].cpu())
    assert np.array_equal(res["rounds"], ref["rounds"])
    assert len(res["regs"][0]) == 3
    for r in range(3):
        got = np.concatenate([np.atleast_2d(s[r]) for s in res["regs"]])
        np.testing.assert_allclose(got, ref["regs"][r], rtol=1e-10, equal_nan=True)
