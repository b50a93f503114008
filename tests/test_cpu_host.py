"""CPU tests (no GPU): the C-ABI library loads and exports every symbol include/yond_b200.h declares, the host-side
logic (state-dict layout, FLOP accounting, padding math, sharding) is right, and the product
path refuses to run without CUDA (no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import yond_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARCH_GRU = {"name": "GuidedResUnet", "guided": True, "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1, "res": True, "norm": True}
ARCH_UNET = {"name": "UNetSeeInDark", "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1, "res": True, "norm": True}
ARCH_SNR = dict(ARCH_GRU, name="SNRnet")


@pytest.fixture(scope="module")
def Y():
    from yond_public_b200 import build
    build.build()
    import yond_public_b200 as Y
    return Y


def test_library_exports_every_declared_symbol(Y):
    hdr = open(os.path.join(ROOT, "include", "yond_b200.h")).read()
    declared = set(re.findall(r"\b(yond_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"yond_vst_params"}
    lib = C.CDLL(Y._lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/yond_b200.h but not exported"
    assert declared == set(Y._lib.SIGNATURES), "ctypes binding and header disagree"
    assert C.sizeof(Y._lib.VstParams) == 32
    assert Y._lib.load().yond_version() >= 100


def test_library_is_sm100a_tcgen05():
    """The conv kernel object must contain tcgen05 / TMA machine code (UTCHMMA, UTMALDG, LDTM), not legacy HMMA."""
    from yond_public_b200 import build
    obj = os.path.join(ROOT, "yond_public_b200", "build", "conv_tc.o")
    cuda_bin = os.path.dirname(build._nvcc())  # the toolkit the library was built with, also when it is not on PATH
    sass = subprocess.run([os.path.join(cuda_bin, "cuobjdump") if cuda_bin else "cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
    if not sass:
        pytest.skip("cuobjdump not available")
    assert "UTCHMMA" in sass and "UTMALDG" in sass and "LDTM" in sass
    assert "HMMA.16816" not in sass


@pytest.mark.parametrize("arch,nparams,flops_px", [(ARCH_UNET, 7760484, 369152), (ARCH_GRU, 11173668, 403968), (ARCH_SNR, 11176612, None)])
def test_arch_plugin_state_dict_and_flops(Y, golden, arch, nparams, flops_px):
    net = getattr(Y, arch["name"])(arch)
    sd = net.state_dict()
    assert sum(v.numel() for v in sd.values()) == nparams
    assert [(k, tuple(v.shape)) for k, v in sd.items()] == net.expected_state()
    key = {"UNetSeeInDark": "unet", "GuidedResUnet": "gru", "SNRnet": "snr"}[arch["name"]]
    g = golden(f"net_{key}")
    assert list(sd.keys()) == [str(k) for k in g["keys"]]
    if flops_px:  # SURVEY.md §8(d): algorithmic FLOPs per packed pixel
        assert net.flops(1, 128, 128) == flops_px * 128 * 128
        assert net.flops(3, 1536, 2016) == flops_px * 3 * 1536 * 2016
    # same construction/init order as the reference => identical random-init tensors under a fixed seed
    torch.manual_seed(5)
    net2 = getattr(Y, arch["name"])(arch)
    Y.initialize_weights(net2)
    ref = O.init_state_dict(arch, seed=5)
    assert all(torch.equal(v, ref[k]) for k, v in net2.state_dict().items())
    Y.load_weights(net, ref, by_name=False)
    assert all(torch.equal(v, ref[k]) for k, v in net.state_dict().items())


def test_no_cpu_fallback(Y):
    net = Y.UNetSeeInDark(ARCH_UNET)
    with pytest.raises(Y._lib.YondError):
        net(torch.zeros(1, 4, 32, 32))
    if not torch.cuda.is_available():
        with pytest.raises(Y._lib.YondError):
            Y.bayer2rggb(np.zeros((4, 4), np.float32))
        with pytest.raises(Y._lib.YondError):
            Y.pack_raw_bayer(np.zeros((4, 4), np.uint16), raw_pattern=[[0, 1], [3, 2]], black_level_per_channel=[0, 0, 0, 0])
        with pytest.raises(Y._lib.YondError):
            Y.rot_bayer(np.zeros((4, 4), np.float32), [[2, 3], [1, 2]])
        with pytest.raises(Y._lib.YondError):
            Y.normalize_raw(np.zeros((4, 8), np.uint16), 512, 16383, 100)
        with pytest.raises(Y._lib.YondError):
            Y.calculate_ssim(np.zeros((16, 16), np.float32), np.zeros((16, 16), np.float32))
        with pytest.raises(Y._lib.YondError):
            Y.compare_psnr(np.zeros((16, 16), np.float32), np.ones((16, 16), np.float32))
        with pytest.raises(Y._lib.YondError):
            Y.process_sidd_image(np.zeros((8, 8), np.float32), [[1, 2], [2, 3]], np.ones((1, 3)), np.eye(3))
        with pytest.raises(Y._lib.YondError):
            Y.demosaic_ea(np.zeros((8, 8), np.uint16))
        with pytest.raises(Y._lib.YondError):
            Y.calculate_ssim(np.zeros((16, 16, 3), np.uint8), np.zeros((16, 16, 3), np.uint8))
        with pytest.raises(Y._lib.YondError):
            Y.ResUnet2(dict(ARCH_UNET, name="ResUnet2"))(torch.zeros(1, 4, 32, 32))
        with pytest.raises(Y._lib.YondError):
            Y.SelfResUNet(dict(ARCH_UNET, name="SelfResUNet"))(torch.zeros(1, 4, 32, 32))
        with pytest.raises(Y._lib.YondError):
            Y.GuidedSelfUnet(dict(ARCH_UNET, name="GuidedSelfUnet", res=False))(torch.zeros(1, 4, 32, 32), torch.tensor(0.04))


def test_synth_module_matches_reference_recipes(Y):
    """bench.py's inputs come from the product-side synth module: its random init is the reference's `initialize_weights`
    under the seed (== the oracle's, which is pinned against the reference), and its generators are deterministic."""
    from yond_public_b200 import synth
    from oracle import yond_oracle as O
    arch = {"name": "GuidedResUnet", "guided": True, "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1, "res": True, "norm": True}
    a, b = synth.random_init_state_dict(arch, seed=3), O.init_state_dict(arch, seed=3)
    assert list(a) == list(b) and all(torch.equal(a[k], b[k]) for k in a)
    r1, r2 = np.random.default_rng(9), np.random.default_rng(9)
    K1, S1 = synth.sample_noise_params(r1, logk_min=-0.5)
    K2, S2 = O.sample_noise_params(r2, logk_min=-0.5)
    assert (K1, S1) == (K2, S2)
    assert np.array_equal(synth.noisy(r1, synth.clean_smooth(r1, 32, 32), K1, S1), O.synth_noisy(r2, O.synth_clean_smooth(r2, 32, 32), K2, S2))
    for a_ in (arch, {"name": "UNetSeeInDark", "in_nc": 4, "out_nc": 4, "nf": 32, "nframes": 1, "res": True, "norm": True}):
        s1, s2 = synth.smoother_state_dict(a_), O.smoother_state_dict(a_)
        assert list(s1) == list(s2) and all(torch.equal(s1[k], s2[k]) for k in s1)
    bw = synth.bench_state_dict(arch, seed=0)
    assert all(float(v.abs().max()) > 0 for v in bw.values())  # dense: no tensor is left at zero


def test_unknown_arch_and_key_rejected(Y):
    with pytest.raises(NotImplementedError):
        Y.build_net({"name": "DnCNN"}, device="cpu")
    lib = Y._lib.load()
    h = C.c_void_p()
    assert lib.yond_net_create(1, 4, 4, 32, 1, 1, C.byref(h)) == 0
    a = np.zeros((3,), np.float32)
    shape = (C.c_int64 * 1)(3)
    assert lib.yond_net_set_tensor(h, b"not.a.key", a.ctypes.data_as(C.c_void_p), shape, 1) != 0
    assert b"not.a.key" in lib.yond_last_error()
    assert lib.yond_net_set_tensor(h, b"conv_in.bias", a.ctypes.data_as(C.c_void_p), shape, 1) != 0  # wrong shape
    assert lib.yond_net_create(7, 4, 4, 32, 1, 1, C.byref(C.c_void_p())) != 0
    assert lib.yond_net_create(1, 4, 4, 48, 1, 1, C.byref(C.c_void_p())) != 0
    lib.yond_net_destroy(h)


def test_nlf_maps_modes_checked(Y):
    """yond_nlf_maps_bayer / _raw16 take modes 0, 1 and 3 only; any other mode is refused before device work (YOND_ERR_INVALID)."""
    lib = Y._lib.load()
    buf = C.c_void_p(256)  # never dereferenced: the arguments are checked first
    nrm = Y._lib.RawNorm(64.0, 1023.0, 1.0, 0)
    for mode in (2, 4, -1):
        assert lib.yond_nlf_maps_bayer(buf, 1, buf, 1, buf, buf, buf, 1, 1, 64, 64, 0, 29, mode, None, buf, None) == 1
        assert b"mode" in lib.yond_last_error()
        assert lib.yond_nlf_maps_raw16(buf, C.byref(nrm), 1, buf, 1, buf, buf, buf, 1, 1, 64, 64, 0, 29, mode, None, buf, None) == 1
        assert b"mode" in lib.yond_last_error()


def test_host_math_matches_oracle(Y, golden):
    g = golden("p2d")
    for s, p in zip(g["shapes"], g["p2d"]):
        assert Y.get_p2d(tuple(int(v) for v in s), base=32) == tuple(int(v) for v in p)
    x_lut, sg_lut = Y.isp.lut_grids()
    ox, os_ = O.lut_grids()
    assert np.array_equal(x_lut, ox) and np.array_equal(sg_lut, os_)
    for sg in (0.0, 0.0049, 0.5, 1.0, 1.378, 9.99, 10.0):
        assert Y.isp.sigma_pos(sg_lut, sg) == O.BiasLUT.pos_interp(sg_lut, sg)
    gb = golden("getbias")
    # node positions of the fallback bias table are host index math (the values are generated on the device: GPU tests)
    assert np.array_equal(Y.isp.bias_table_nodes(np.float32(40.0)), gb["nodes2"])
    assert np.array_equal(Y.isp.bias_table_nodes(np.float32(700.0)), gb["nodes"])
    lib = Y._lib.load()
    for mx in (0.0, 3.2, 40.0, 48.5, 49.0, 333.3, 498.2, 499.0, 700.0, 961.0, 2400.0, 15871.0):
        assert lib.yond_bias_table_nodes(mx) == len(Y.isp.bias_table_nodes(np.float32(mx))), mx
    assert Y.VST(0, np.float64(5.1), gain=np.float64(3.7)) == O.VST(0, np.float64(5.1), gain=np.float64(3.7))


def test_shard_ranges():
    from yond_public_b200.parallel import shard_range, shard_sizes
    for n in (0, 1, 7, 40, 256, 1280):
        for world in (1, 2, 3, 4, 8):
            covered = []
            for r in range(world):
                a, b = shard_range(n, r, world)
                covered += list(range(a, b))
            assert covered == list(range(n))
            s = shard_sizes(n, world)
            assert max(s) - min(s) <= 1


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from yond_public_b200.parallel import run_sharded
    units = torch.arange(7 * 6, dtype=torch.float32).reshape(7, 2, 3)  # 7 units: ragged shares (4 + 3)
    out = run_sharded(units, lambda u: u * 2 + 1, dst=0)
    ok = bool(torch.equal(out, units * 2 + 1)) if rank == 0 else out is None
    # band-sharded frame: each rank "forwards" its row band (+ halo, cut at the border) and one all-gather assembles the
    # frame; the stand-in network is a 3x3 row-local box sum, so a missing or misplaced halo row would show
    from yond_public_b200.parallel import BandShardedForward, band_range
    for hp in (96, 80):  # 80: ragged last band (48 + 32)
        full = (torch.arange(hp * 20 * 4, dtype=torch.float32).reshape(1, hp, 20, 4) % 97) * 0.25

        def fake_net(z, ub, t, out=None):
            p_ = torch.nn.functional.pad(z.permute(0, 3, 1, 2), (0, 0, 1, 1))  # zero rows outside the slice, like the conv padding
            return (p_[:, :, :-2] + p_[:, :, 1:-1] + p_[:, :, 2:]).permute(0, 2, 3, 1).contiguous()
        fwd = BandShardedForward(fake_net, halo=16)
        got = fwd(full, None, None)
        ok = ok and bool(torch.equal(got, fake_net(full, None, None)))
        r0, r1, band = band_range(hp, rank, world)
        ok = ok and band % 16 == 0 and 0 <= r0 <= r1 <= hp
    q.put(ok)
    dist.destroy_process_group()


def test_image_parallel_gather_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert all(res)


def test_render_host_algebra(Y):
    """The 3x3 colour algebra of process_sidd_image stays NumPy on the host (utils/sidd_utils.py:161-170): same matrix as the oracle's,
    bit for bit; an unknown CFA pattern is rejected before anything touches the device (the reference drops into pdb there)."""
    from yond_public_b200 import render
    rng = np.random.default_rng(9)
    cst = np.array([[0.8, 0.25, -0.05], [-0.3, 1.1, 0.2], [0.02, -0.2, 0.9]]) + rng.normal(0, 0.03, (3, 3))
    m = render.cam2rgb_matrix(cst)
    assert m.dtype == np.float64 and np.array_equal(m, O.render_cam2rgb(cst))
    np.testing.assert_allclose(m.sum(axis=-1), 1.0, rtol=1e-15)
    assert render._FLIPS[render._pattern_key(np.array([[3, 2], [2, 1]]))] == (1, 1)
    with pytest.raises(ValueError):
        Y.process_sidd_image(np.zeros((8, 8), np.float32), [[0, 1], [2, 3]], np.ones((1, 3)), np.eye(3))
