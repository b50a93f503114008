"""Noise-level-function estimators (SimpleNLF / SelfNLF / CollabNLF, YOND_SIDD.py:62-124) on device.

Everything runs on the device: the box statistics (yond_nlf_maps*), then the estimator tail (yond_nlf_fit): exact
percentiles by radix select, the score3 threshold, the masked line fit with the reference's empty-mask fallbacks, in float64
following NumPy operation by operation.  The public functions read back only the final (beta1, beta2).
"""
from __future__ import annotations

import ctypes as C
import threading

import numpy as np
import torch

from . import _lib
from ._lib import check, ptr, stream_ptr
from .isp import _as_batch4, _dev, to_dev


class NlfEstimator:
    """Blind (beta1, beta2) estimation, batched over `nimg` images: every device stage runs once for the whole batch
    and the estimates stay on the device."""

    def __init__(self):
        self.lib = _lib.load()
        self._scr = {}

    def _buf(self, name, nbytes, dev):
        b = self._scr.get(name)
        if b is None or b.numel() < nbytes or b.device != dev:
            b = torch.empty(int(nbytes), device=dev, dtype=torch.uint8)
            self._scr[name] = b
        return b

    # -- maps -----------------------------------------------------------------------------------
    def maps(self, lr_rggb, hr_rggb=None, k=29):
        """lr_rggb / hr_rggb: (B,h,w,4) CUDA float32.  Returns var, mean, lap (same shape)."""
        B, h, w, _ = lr_rggb.shape
        work = self._buf("maps", self.lib.yond_nlf_work_bytes(B, h, w, 4), lr_rggb.device)
        var, mean, lap = torch.empty_like(lr_rggb), torch.empty_like(lr_rggb), torch.empty_like(lr_rggb)
        mode = 0 if hr_rggb is None else 1
        check(self.lib.yond_nlf_maps(ptr(lr_rggb), ptr(hr_rggb), ptr(var), ptr(mean), ptr(lap), B, h, w, 4, int(k), mode,
                                     ptr(work), stream_ptr()))
        return var, mean, lap

    # -- device-resident estimate (no host read-back) ----------------------------------------------
    DETAIL = 4 + 2 * 24

    def estimate_dev(self, x, y=None, k=29, split_blocks=False, x_mosaic=False, y_mosaic=False, nblk=None, seg_max=None,
                     details=False, step=5, raw=None, var_map=None):
        """SelfNLF (y None) / CollabNLF straight from Bayer frames, everything on the device.

        x: blocks layout (nimg, nblk, H, W) or, with x_mosaic, mosaic layout (nimg, H, nblk*W) (`nblk` then required; plain
        frames are nblk = 1 in either layout).  split_blocks: every block is its own image for the box filters (SIDD_256).
        seg_max (optional, (nimg,) f32 CUDA): receives max(x, 0) per image.  Returns regs (nimg, 2) float64 on the
        device [, detail (nimg, DETAIL)]; nothing is read back.  x may be the uint16 sensor mosaic (a 16-bit integer tensor) with
        raw = _lib.RawNorm(black, white, ratio, clip), or a CUDA uint8 tensor of nimg yond_raw_norm records (one per image): it is
        normalised on load (SURVEY 8(f)-1).
        var_map (self only; float32 CUDA, at least B*h*w*4 values): the var map goes there instead of the estimator's scratch, where
        no later call overwrites it — the cached noisy-frame statistics of the collab rounds (estimate_collab_cached)."""
        lib = self.lib
        if x_mosaic:
            nimg, H, Wm = x.shape
            nb = int(nblk or 1)
            W = Wm // nb
        else:
            nimg, nb, H, W = x.shape
        is_raw = x.dtype in (torch.int16, torch.uint16)
        assert x.is_cuda and x.is_contiguous() and (x.dtype == torch.float32 or (is_raw and raw is not None))
        dev = x.device
        h, wb = H // 2, W // 2
        B, w = (nimg * nb, wb) if split_blocks else (nimg, nb * wb)
        n_el = B * h * w * 4
        maps = self._buf("maps3", 3 * n_el * 4, dev).view(torch.float32)
        var, mean, lap = maps[:n_el], maps[n_el:2 * n_el], maps[2 * n_el:3 * n_el]
        if var_map is not None:
            assert y is None and var_map.dtype == torch.float32 and var_map.is_cuda and var_map.numel() >= n_el
            var = var_map.reshape(-1)[:n_el]
        work = self._buf("maps", lib.yond_nlf_work_bytes(B, h, w, 4), dev)
        mode = 0 if y is None else 1
        if y is not None:
            assert y.is_cuda and y.dtype == torch.float32 and y.is_contiguous() and y.numel() == x.numel()
        if is_raw:
            fn, nrm = _raw16_maps(lib, raw)
            check(fn(ptr(x), nrm, int(bool(x_mosaic)), ptr(y), int(bool(y_mosaic)), ptr(var), ptr(mean), ptr(lap),
                     nimg, nb, H, W, int(bool(split_blocks)), int(k), mode, ptr(seg_max), ptr(work), stream_ptr()))
        else:
            check(lib.yond_nlf_maps_bayer(ptr(x), int(bool(x_mosaic)), ptr(y), int(bool(y_mosaic)), ptr(var), ptr(mean), ptr(lap), nimg, nb,
                                          H, W, int(bool(split_blocks)), int(k), mode, ptr(seg_max), ptr(work), stream_ptr()))
        return self._fit(var, mean, lap, nimg, details, step)

    def _fit(self, var, mean, lap, nimg, details=False, step=5):
        lib, dev = self.lib, var.device
        n_el = var.numel()
        quants = np.ascontiguousarray(np.linspace(step, 100, 100 // step, endpoint=True), np.float64)
        regs = torch.empty((nimg, 2), device=dev, dtype=torch.float64)
        detail = torch.empty((nimg, self.DETAIL), device=dev, dtype=torch.float64) if details else None
        fwork = self._buf("fit", lib.yond_nlf_fit_work_bytes(nimg) + 256, dev)
        off = (-fwork.data_ptr()) % 256
        check(lib.yond_nlf_fit(ptr(var), ptr(mean), ptr(lap), n_el // nimg, nimg, quants.ctypes.data_as(C.POINTER(C.c_double)),
                               len(quants), ptr(regs), ptr(detail), ptr(fwork[off:]), stream_ptr()))
        return (regs, detail) if details else regs

    # -- the collab rounds of IterDenoise from cached noisy-frame statistics ---------------------------
    # Every collab round r >= 2 estimates on (lr, out_{r-1}) in the same geometry.  Its var map is stdfilt(lr, k)**2 -
    # stdfilt(out_{r-1}, k)**2, and the first term is the same in every round: it is computed once per batch (the self estimate's
    # var map when the geometries agree, else one lr_var_dev pass) and each round makes one box pass over out_{r-1}.
    @staticmethod
    def collab_geometry(nimg, nblk, H, W, split_blocks):
        """Number of float32 values of a map in the box-filter geometry of `nimg` images of `nblk` (H,W) blocks."""
        return (nimg * nblk if split_blocks else nimg) * (H // 2) * ((W // 2) if split_blocks else nblk * (W // 2)) * 4

    def lr_var_dev(self, x, out, k=29, split_blocks=False, x_mosaic=False, nblk=None, raw=None):
        """out <- stdfilt(x, k)**2 in the box-filter geometry (one box pass; x layouts / raw as in estimate_dev)."""
        lib = self.lib
        if x_mosaic:
            nimg, H, Wm = x.shape
            nb = int(nblk or 1)
            W = Wm // nb
        else:
            nimg, nb, H, W = x.shape
        assert x.is_cuda and x.is_contiguous() and out.is_contiguous() and out.dtype == torch.float32
        assert out.numel() >= self.collab_geometry(nimg, nb, H, W, split_blocks)
        work = self._buf("maps", lib.yond_nlf_work_bytes(1, 1, 1, 4), x.device)  # mode 3 uses no scratch
        if x.dtype in (torch.int16, torch.uint16):
            fn, nrm = _raw16_maps(lib, raw)
            check(fn(ptr(x), nrm, int(bool(x_mosaic)), None, 0, ptr(out), None, None, nimg, nb, H, W, int(bool(split_blocks)), int(k), 3,
                     None, ptr(work), stream_ptr()))
        else:
            assert x.dtype == torch.float32
            check(lib.yond_nlf_maps_bayer(ptr(x), int(bool(x_mosaic)), None, 0, ptr(out), None, None, nimg, nb, H, W,
                                          int(bool(split_blocks)), int(k), 3, None, ptr(work), stream_ptr()))
        return out

    def collab_maps_cached(self, y, lr_var, nblk, k=29, split_blocks=False, y_mosaic=True):
        """CollabNLF maps (var, mean, lap) of the float32 frames y — mosaic layout (nimg, H, nblk*W) or, y_mosaic False, blocks
        layout (nimg, nblk, H, W) — against the cached lr_var = stdfilt(lr, k)**2 (read only) in the same geometry."""
        if y_mosaic:
            nimg, H, Wm = y.shape
            W = Wm // nblk
        else:
            nimg, _, H, W = y.shape
        assert y.is_cuda and y.dtype == torch.float32 and y.is_contiguous() and lr_var.dtype == torch.float32
        n_el = self.collab_geometry(nimg, nblk, H, W, split_blocks)
        assert lr_var.numel() >= n_el
        maps = self._buf("maps3", 3 * n_el * 4, y.device).view(torch.float32)
        var, mean, lap = maps[:n_el], maps[n_el:2 * n_el], maps[2 * n_el:3 * n_el]
        check(self.lib.yond_nlf_maps_collab_cached(ptr(y), int(bool(y_mosaic)), ptr(lr_var.reshape(-1)), ptr(var), ptr(mean), ptr(lap),
                                                   nimg, nblk, H, W, int(bool(split_blocks)), int(k), stream_ptr()))
        return var, mean, lap

    def estimate_collab_cached(self, y, lr_var, nblk, k=29, split_blocks=False, y_mosaic=True, details=False, step=5):
        """CollabNLF (beta1, beta2) of a collab round from the cached lr statistics: regs (nimg, 2) float64 on the device."""
        var, mean, lap = self.collab_maps_cached(y, lr_var, nblk, k, split_blocks, y_mosaic)
        return self._fit(var, mean, lap, y.shape[0], details, step)


def _raw16_maps(lib, raw):
    """The uint16 maps entry point and its normalisation argument: one host RawNorm for every image, or the per-image device records."""
    if isinstance(raw, torch.Tensor):
        assert raw.is_cuda and raw.dtype == torch.uint8 and raw.is_contiguous()
        return lib.yond_nlf_maps_raw16_per_image, ptr(raw)
    return lib.yond_nlf_maps_raw16, C.byref(raw)


_EST = threading.local()


def _estimator():
    """One estimator (and its device scratch) per host thread: the host-pipelined path runs two lanes concurrently."""
    est = getattr(_EST, "est", None)
    if est is None:
        est = _EST.est = NlfEstimator()
    return est


def SelfNLF(lr_rggb, k=29, kwargs=None):
    kwargs = kwargs or {}
    t, _ = to_dev(lr_rggb)
    b = _as_batch4(t) if t.dim() == 3 else t
    if kwargs.get("SIDD_256"):
        B, h, w, _ = b.shape
        b = b.reshape(h, 32, w // 32, 4).permute(1, 0, 2, 3).contiguous()
    est = _estimator()
    var, mean, lap = est.maps(b, None, k)
    return est._fit(var, mean, lap, 1)[0].cpu().numpy()


def CollabNLF(lr_rggb, hr_rggb, k=29, kwargs=None):
    kwargs = kwargs or {}
    tl, _ = to_dev(lr_rggb)
    th_, _ = to_dev(hr_rggb)
    bl = _as_batch4(tl) if tl.dim() == 3 else tl
    bh = _as_batch4(th_) if th_.dim() == 3 else th_
    if kwargs.get("SIDD_256"):
        B, h, w, _ = bl.shape
        bl = bl.reshape(h, 32, w // 32, 4).permute(1, 0, 2, 3).contiguous()
        bh = bh.reshape(h, 32, w // 32, 4).permute(1, 0, 2, 3).contiguous()
    est = _estimator()
    var, mean, lap = est.maps(bl, bh, k)
    return est._fit(var, mean, lap, 1)[0].cpu().numpy()


def SimpleNLF(lr_raw, hr_raw=None, k=29, setting=None):
    """YOND_SIDD.py:117-124 — pack + dispatch.  Returns array-like (beta1, beta2), float64.  Bayer frames (H,W) in (NumPy or
    CUDA); the maps are computed straight from the mosaic and the whole estimate runs on the device (one 16-byte read-back)."""
    setting = setting or {"mode": "self"}
    sidd = bool(setting.get("SIDD_256", False))
    if setting["mode"] not in ("self", "collab"):
        raise NotImplementedError(setting["mode"])
    lr, _ = to_dev(lr_raw)
    hr = None
    if setting["mode"] == "collab":
        hr, _ = to_dev(hr_raw)
        assert hr.shape == lr.shape
    assert lr.dim() == 2
    if sidd:
        assert lr.shape[1] % 64 == 0, "SIDD_256 splits the mosaic into 32 blocks along W (YOND_SIDD.py:65,91-93)"
    regs = _estimator().estimate_dev(lr[None], None if hr is None else hr[None], k, split_blocks=sidd, x_mosaic=True, y_mosaic=True,
                                     nblk=32 if sidd else 1)
    return regs[0].cpu().numpy()
