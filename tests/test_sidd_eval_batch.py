"""SIDD scoring of a whole batch (YOND_SIDD.py:635-668 for every image and round at once): sidd_eval_batch renders every image with its
own camera metadata in one launch and returns the raw / sRGB PSNR and SSIM table after one read-back.  It must give what the per-image
sidd_eval_image gives, what the oracle gives, and the same for the output of the batched pipeline; its launch count must not grow with
the number of images."""
import numpy as np
import pytest
import torch

from oracle import yond_oracle as O

PATTERNS = [[[1, 2], [2, 3]], [[2, 1], [3, 2]], [[2, 3], [1, 2]], [[3, 2], [2, 1]]]
CST = np.array([[0.8, 0.25, -0.05], [-0.3, 1.1, 0.2], [0.02, -0.2, 0.9]])
ARCH = {"name": "GuidedResUnet", "guided": True, "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1, "res": True, "norm": True}
PIPE = {"full_est": True, "est_type": "simple+full", "k": 29, "full_dn": False, "vst_type": "exact", "bias_corr": "pre",
        "iter": "iter", "max_iter": 3}
P = {"wp": 1023, "bl": 64, "ratio": 1, "gain": 1, "sigma": 0, "scale": 959.0}
BASE_REGS = (4.2e-3, 3.9e-5)


@pytest.fixture(scope="module")
def Y():
    import yond_public_b200 as Y
    return Y


def _meta(rng, pat):
    return {"bayer_2by2": PATTERNS[pat], "wb": np.array([[rng.uniform(1.5, 2.5), 1.0, rng.uniform(1.3, 2.2)]]),
            "cst2": CST + rng.normal(0, 0.03, (3, 3))}


def _workload(rng, nimg, nround, nblk=8, Hb=64):
    """Clean mosaics (nimg, Hb, nblk*Hb) and nround rounds of outputs that move towards them."""
    clean = np.stack([np.concatenate([O.synth_clean(rng, Hb, Hb) for _ in range(nblk)], -1) for _ in range(nimg)])
    noisy = O.synth_noisy(rng, clean, 2.0, 3.0).astype(np.float32)
    outs = [((1 - a) * noisy + a * clean).astype(np.float32) for a in np.linspace(0.3, 0.9, nround)]
    return clean, outs


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _assert_matches_per_image(Y, res, dns, hr, metas, rounds, nblk):
    """res (sidd_eval_batch) against sidd_eval_image on each image's completed rounds: pictures byte for byte, PSNR within 1e-12
    relative, SSIM within 1e-12 absolute, -1 / NaN exactly where the reference scores or renders nothing."""
    nround, nimg = res["psnr"].shape
    for i in range(nimg):
        one = Y.sidd_eval_image([dns[r][i] for r in range(rounds[i])], hr[i], metas[i], nblk=nblk)
        assert torch.equal(res["img_hr"][i], one["img_hr"]), i
        k = 0  # the per-image result lists the sRGB numbers of the rendered rounds only
        for r in range(nround):
            got = [res[key][r, i] for key in ("psnr", "ssim", "psnr_rgb", "ssim_rgb")]
            if r >= rounds[i]:
                assert np.isnan(got).all() and not res["rendered"][r, i], (r, i)
                continue
            if one["img_dn"][r] is None:
                assert got[:2] == [-1.0, -1.0] and one["psnr"][r] == -1.0 and np.isnan(got[2:]).all(), (r, i)
                assert not res["rendered"][r, i]
                continue
            assert res["rendered"][r, i]
            np.testing.assert_allclose(got[0], one["psnr"][r], rtol=1e-12, atol=0)
            np.testing.assert_allclose(got[1], one["ssim"][r], rtol=0, atol=1e-12)
            np.testing.assert_allclose(got[2], one["psnr_rgb"][k], rtol=1e-12, atol=0)
            np.testing.assert_allclose(got[3], one["ssim_rgb"][k], rtol=0, atol=1e-12)
            assert torch.equal(res["img_dn"][r, i], one["img_dn"][r]), (r, i)
            k += 1


@pytest.mark.gpu
def test_batch_equals_per_image(Y):
    """Five images with all four CFA patterns and their own wb / cst2, three rounds, rounds = [3, 1, 2, 3, 2], and one output of round
    2 without a positive value."""
    rng = np.random.default_rng(31)
    nimg, nround, nblk = 5, 3, 8
    clean, outs = _workload(rng, nimg, nround, nblk)
    outs[1][3] = 0.0  # image 3, round 2: all zeros
    metas = [_meta(rng, i % 4) for i in range(nimg)]
    rounds = [3, 1, 2, 3, 2]
    hr, dns = _cuda(clean), [_cuda(o) for o in outs]
    res = Y.sidd_eval_batch(dns, hr, metas, nblk=nblk, rounds=rounds)
    assert res["psnr"].shape == (nround, nimg) and res["psnr"].dtype == np.float64
    assert tuple(res["img_dn"].shape) == (nround, nimg, 64, nblk * 64, 3) and res["img_dn"].dtype == torch.uint8
    assert tuple(res["img_hr"].shape) == (nimg, 64, nblk * 64, 3) and res["img_hr"].is_cuda
    assert res["rendered"].tolist() == [[True] * 5, [True, False, True, False, True], [True, False, False, True, False]]
    assert res["psnr"][1, 3] == -1.0 and res["ssim"][1, 3] == -1.0
    _assert_matches_per_image(Y, res, dns, hr, metas, rounds, nblk)
    # raw numbers only: the same raw table (up to the order of the float64 atomics), no pictures
    raw = Y.sidd_eval_batch(dns, hr, None, nblk=nblk, rounds=rounds)
    np.testing.assert_allclose(raw["psnr"], res["psnr"], rtol=1e-12, atol=0)
    np.testing.assert_allclose(raw["ssim"], res["ssim"], rtol=0, atol=1e-12)
    assert (raw["psnr"] == -1).tolist() == (res["psnr"] == -1).tolist()
    assert np.isnan(raw["psnr_rgb"]).all() and raw["img_dn"] is None and not raw["rendered"].any()


@pytest.mark.gpu
def test_vs_oracle_sidd_shape(Y):
    """Two SIDD-shaped images (256 x 8192, 32 blocks of 256 x 256) with two CFA patterns in one call, against the oracle's render and
    per-image numbers at the bars of the per-image checks: pictures equal, PSNR 1e-9, SSIM 1e-7."""
    rng = np.random.default_rng(44)
    clean = np.stack([np.concatenate([O.synth_clean(rng, 256, 256) for _ in range(32)], -1) for _ in range(2)])
    dn = (0.85 * clean + 0.15 * O.synth_noisy(rng, clean, 3.0, 4.0)).astype(np.float32)
    metas = [_meta(rng, 1), _meta(rng, 3)]
    res = Y.sidd_eval_batch([_cuda(dn)], _cuda(clean), metas, nblk=32)
    assert res["rendered"].all()
    for i, m in enumerate(metas):
        img_hr = O.process_sidd_image(clean[i], m["bayer_2by2"], m["wb"], m["cst2"])
        img_dn = O.process_sidd_image(dn[i], m["bayer_2by2"], m["wb"], m["cst2"])
        assert np.array_equal(res["img_hr"][i].cpu().numpy(), img_hr), i
        assert np.array_equal(res["img_dn"][0, i].cpu().numpy(), img_dn), i
        p, s = O.sidd_image_metrics(dn[i], clean[i], 32)
        pr, sr = O.sidd_rgb_metrics(img_dn, img_hr, 32)
        assert abs(res["psnr"][0, i] - p) < 1e-9 and abs(res["ssim"][0, i] - s) < 1e-7
        assert abs(res["psnr_rgb"][0, i] - pr) < 1e-9 and abs(res["ssim_rgb"][0, i] - sr) < 1e-7


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
def test_from_the_pipeline(Y, monkeypatch):
    """iter_denoise_batch at max_iter = 3 with images that stop early (rounds [4, 1, 2]) scored with rounds=res['rounds']: equal to the
    per-image loop over each image's completed rounds, the repeated rounds NaN."""
    rng = np.random.default_rng(5)
    nblk, Hb = 32, 64
    clean = np.stack([np.stack([O.synth_clean_smooth(rng, Hb, Hb) for _ in range(nblk)]) for _ in range(3)])
    noisy = O.synth_noisy(rng, clean, 4.0, 6.0).astype(np.float32)
    drv = Y.YOND_SIDD(ARCH, PIPE, state_dict=O.smoother_state_dict(ARCH))
    _override(monkeypatch, {(0, 1): -1e-3, (1, 2): -2e-3})
    res = drv.iter_denoise_batch(_cuda(noisy), dict(P))
    assert res["rounds"].tolist() == [4, 1, 2]
    hr = _cuda(np.concatenate(list(clean.transpose(1, 0, 2, 3)), axis=-1))  # (3, Hb, nblk*Hb): the blocks side by side
    metas = [_meta(rng, p) for p in (0, 2, 3)]
    got = Y.sidd_eval_batch(res["raw_dns"], hr, metas, nblk=nblk, rounds=res["rounds"])
    assert got["psnr"].shape == (4, 3)
    assert np.isnan(got["psnr"][1:, 1]).all() and np.isnan(got["ssim_rgb"][2:, 2]).all()
    assert not np.isnan(got["psnr"][:, 0]).any() and got["rendered"][:, 0].all()
    _assert_matches_per_image(Y, got, res["raw_dns"], hr, metas, res["rounds"].tolist(), nblk)


@pytest.mark.gpu
def test_launch_count_does_not_grow_with_images(Y):
    rng = np.random.default_rng(8)
    counts = []
    for nimg in (2, 6):
        clean, outs = _workload(rng, nimg, 2)
        hr, dns = _cuda(clean), [_cuda(o) for o in outs]
        metas = [_meta(rng, i % 4) for i in range(nimg)]
        Y.sidd_eval_batch(dns, hr, metas, nblk=8)  # first call: the gamma table is uploaded once per device
        n0 = Y._lib.launch_count()
        Y.sidd_eval_batch(dns, hr, metas, nblk=8, rounds=[2] * (nimg - 1) + [1])
        counts.append(Y._lib.launch_count() - n0)
    assert counts[0] == counts[1], counts


def _bad_cases():
    """name -> function(hr, dns, metas) returning the arguments of a call that must raise ValueError."""
    bad_pattern = {"bayer_2by2": [[0, 1], [2, 3]], "wb": np.ones((1, 3)), "cst2": CST}
    return {
        "metas_count": lambda hr, dns, m: ((dns, hr, m[:-1]), {}),
        "rounds_count": lambda hr, dns, m: ((dns, hr, m), {"rounds": [2]}),
        "round_shape": lambda hr, dns, m: (([dns[0], dns[1][:, :, :-64].contiguous()], hr, m), {}),
        "round_count_zero": lambda hr, dns, m: (([], hr, m), {}),
        "not_cuda": lambda hr, dns, m: (([dns[0].cpu(), dns[1]], hr, m), {}),
        "not_float32": lambda hr, dns, m: ((dns, hr.double(), m), {}),
        "not_contiguous": lambda hr, dns, m: (([dns[0].transpose(1, 2).contiguous().transpose(1, 2), dns[1]], hr, m), {}),
        "meta_key": lambda hr, dns, m: ((dns, hr, [m[0], {k: v for k, v in m[1].items() if k != "wb"}]), {}),
        "bayer_pattern": lambda hr, dns, m: ((dns, hr, [m[0], bad_pattern]), {}),
        "rounds_low": lambda hr, dns, m: ((dns, hr, m), {"rounds": [0, 2]}),
        "rounds_high": lambda hr, dns, m: ((dns, hr, m), {"rounds": [3, 2]}),
        "nblk_split": lambda hr, dns, m: ((dns, hr, m), {"nblk": 3}),
        "block_small": lambda hr, dns, m: ((dns, hr, m), {"nblk": 64}),
        "too_many_blocks": lambda hr, dns, m: _too_many_blocks(m),
    }


def _too_many_blocks(metas):
    """2 images x 16384 blocks of 12 x 12 x 3 channels: more block-channels than one launch of the metric kernels takes."""
    big = torch.zeros((2, 12, 16384 * 12), device="cuda")
    return ([big, big.clone()], big, metas), {"nblk": 16384}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(_bad_cases()))
def test_errors_before_any_launch(Y, case):
    rng = np.random.default_rng(3)
    clean, outs = _workload(rng, 2, 2, nblk=8)
    hr, dns = _cuda(clean), [_cuda(o) for o in outs]
    metas = [_meta(rng, 0), _meta(rng, 1)]
    args, kw = _bad_cases()[case](hr, dns, metas)
    torch.cuda.synchronize()
    n0 = Y._lib.launch_count()
    with pytest.raises(ValueError):
        Y.sidd_eval_batch(*args, **kw)
    assert Y._lib.launch_count() == n0


def test_cpu_tensors_rejected():
    """No device needed: inputs that are not CUDA tensors are refused before the library is touched."""
    from yond_public_b200.metrics import sidd_eval_batch
    hr = torch.zeros((1, 16, 64))
    with pytest.raises(ValueError):
        sidd_eval_batch([hr.clone()], hr, nblk=4)
    with pytest.raises(ValueError):
        sidd_eval_batch([np.zeros((1, 16, 64), np.float32)], np.zeros((1, 16, 64), np.float32), nblk=4)
