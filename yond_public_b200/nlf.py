"""Noise-level-function estimators (SimpleNLF / SelfNLF / CollabNLF, YOND_SIDD.py:62-124) on device.

Device work: box statistics (yond_nlf_maps), exact order statistics (yond_order_stats), score3 bin occupancy
(yond_score3_bins), masked regression sums (yond_masked_sums).  Host work (a few dozen scalars, float64,
exactly like the reference): np.percentile's linear interpolation, the score argmin, the reference's guards
and the 2x2 least-squares solve.
"""
from __future__ import annotations

import ctypes as C
import threading

import numpy as np
import torch

from . import _lib
from ._lib import check, ptr, stream_ptr
from .isp import _as_batch4, _dev, bayer2rggb, to_dev


def _percentiles_from_order_stats(lo_vals, hi_vals, gamma):
    """np.percentile(method='linear') given the two bracketing order statistics (float32) and the fractional
    part gamma (float64): NumPy's _lerp — the difference is taken in float32, the lerp in float64."""
    a = lo_vals.astype(np.float32)
    b = hi_vals.astype(np.float32)
    diff = (b - a)  # float32, like np.subtract on the float32 array
    out = a + diff * gamma
    hi_side = gamma >= 0.5
    out[hi_side] = (b - diff * (1 - gamma))[hi_side]
    return np.asarray(out, dtype=np.float64)


class NlfEstimator:
    """Blind (beta1, beta2) estimation, batched over `nseg` images: every device stage runs once for the whole batch
    and the host sees three small read-backs per batch (order statistics, bin counts, regression sums)."""

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

    # -- percentiles ----------------------------------------------------------------------------
    def percentiles(self, data, quants, nseg=1):
        """np.percentile(segment.reshape(-1), quants, method='linear') for each of the `nseg` equal contiguous segments
        of `data`, from exact device order statistics.  Returns (nseg, len(quants)) float64 ((len,) when nseg == 1)."""
        n = data.numel() // nseg
        q = np.atleast_1d(np.asarray(quants, np.float64))
        qq = np.true_divide(q, 100)
        vi = (n - 1) * qq  # NumPy's virtual index for method='linear'
        lo = np.floor(vi).astype(np.int64)
        hi = np.minimum(lo + 1, n - 1)
        gamma = vi - lo
        ranks = np.concatenate([lo, hi]).astype(np.uint64)
        sel_work = self._buf("select", self.lib.yond_select_work_bytes(nseg), data.device)
        ranks_dev = torch.from_numpy(ranks.view(np.int64)).to(data.device)
        out = torch.empty((nseg, len(ranks)), device=data.device, dtype=torch.float32)
        check(self.lib.yond_order_stats(ptr(data), n, nseg, ptr(ranks_dev), len(ranks), ptr(out), ptr(sel_work), stream_ptr()))
        vals = out.cpu().numpy()
        res = np.stack([_percentiles_from_order_stats(v[:len(q)], v[len(q):], gamma) for v in vals])
        return res[0] if nseg == 1 else res

    # -- get_threshold(mode='score3'), YOND_SIDD.py:22-49 ----------------------------------------
    def threshold_score3(self, lap, mean, step=5, nseg=1):
        quants = np.linspace(step, 100, 100 // step, endpoint=True)
        ths = np.atleast_2d(self.percentiles(lap, quants, nseg))
        n = lap.numel() // nseg
        small = self._buf("bins", nseg * 1001 * 4 + 256, lap.device)
        ths_dev = torch.from_numpy(np.ascontiguousarray(ths)).to(lap.device)
        npk = torch.empty((nseg, ths.shape[1]), device=lap.device, dtype=torch.int32)
        check(self.lib.yond_score3_bins(ptr(lap), ptr(mean), n, nseg, ptr(ths_dev), ths.shape[1], ptr(npk), ptr(small),
                                        stream_ptr()))
        npeaks = npk.cpu().numpy().astype(np.float64)
        score = ths / (quants[None] * npeaks)
        idx = np.argmin(score[:, 1:], axis=1) + 1  # start_pos = 1 skips the 5 % quantile (:46-47)
        th = ths[np.arange(nseg), idx]
        info = dict(ths=ths, npeaks=npeaks, score=score)
        if nseg == 1:
            return th[0], quants[idx[0]], {k: v[0] for k, v in info.items()}
        return th, quants[idx], info

    # -- masked fit, YOND_SIDD.py:77-86 + utils/isp_algos.py:345-365 ------------------------------
    def masked_fit(self, var, mean, lap, th, nseg=1):
        n = lap.numel() // nseg
        th = np.atleast_1d(np.asarray(th, np.float64)).copy()
        sums_dev = torch.empty((nseg, 12), device=lap.device, dtype=torch.float64)

        def sums(thr):
            thr_dev = torch.from_numpy(np.ascontiguousarray(thr)).to(lap.device)
            check(self.lib.yond_masked_sums(ptr(lap), ptr(mean), ptr(var), n, nseg, ptr(thr_dev), ptr(sums_dev), stream_ptr()))
            return sums_dev.cpu().numpy()
        s = sums(th)
        empty = s[:, 0] == 0
        if empty.any():  # "no flat area": fall back to the 25th percentile (:79-84) ...
            th_backup = np.atleast_1d(self.percentiles(lap, [25.0], nseg)).reshape(nseg)
            redo = empty & (th != th_backup)
            th[redo] = th_backup[redo]
            th[empty & ~redo] = np.inf  # ... and when that IS the threshold, the reference keeps the unmasked maps
            s2 = sums(th)
            s[empty] = s2[empty]
        regs = np.zeros((nseg, 2), np.float64)
        for i in range(nseg):
            # polyfit keeps 1e-4 < x < 0.8 when that is > 1 % of the points (:348-350)
            use = s[i, 6:12] if s[i, 6] > 0.01 * s[i, 0] else s[i, 0:6]
            N, Sx, Sy, Sxx, Sxy = use[0], use[1], use[2], use[3], use[4]
            det = N * Sxx - Sx * Sx
            b1 = (N * Sxy - Sx * Sy) / det
            regs[i] = (b1, (Sy - b1 * Sx) / N)
        if nseg == 1:
            return regs[0], th[0]
        return regs, th

    # -- device-resident estimate (no host read-back) ----------------------------------------------
    DETAIL = 4 + 2 * 24

    def estimate_dev(self, x, y=None, k=29, split_blocks=False, x_mosaic=False, y_mosaic=False, nblk=None, seg_max=None,
                     details=False, step=5, raw=None, reuse_self_var=False, var_map=None):
        """SelfNLF (y None) / CollabNLF straight from Bayer frames, everything on the device.

        x: blocks layout (nimg, nblk, H, W) or, with x_mosaic, mosaic layout (nimg, H, nblk*W) (`nblk` then required; plain
        frames are nblk = 1 in either layout).  split_blocks: every block is its own image for the box filters (SIDD_256).
        seg_max (optional, (nimg,) f32 CUDA): receives max(x, 0) per image.  Returns regs (nimg, 2) float64 on the
        device [, detail (nimg, DETAIL)]; nothing is read back.  x may be the uint16 sensor mosaic (a 16-bit integer tensor) with
        raw = _lib.RawNorm(black, white, ratio, clip): it is normalised on load (SURVEY 8(f)-1).
        reuse_self_var (collab only): the previous call on this estimator was the SELF estimate of the same x in the same geometry,
        so its var map (= stdfilt(x, k)**2, exactly what CollabNLF computes first) is still in place and the pass over x is skipped.
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
        mode = 0 if y is None else (2 if reuse_self_var and getattr(self, "_self_key", None) == (x.data_ptr(), B, h, w, int(k)) else 1)
        self._self_key = (x.data_ptr(), B, h, w, int(k)) if y is None else None
        if y is not None:
            assert y.is_cuda and y.dtype == torch.float32 and y.is_contiguous() and y.numel() == x.numel()
        if is_raw:
            check(lib.yond_nlf_maps_raw16(ptr(x), C.byref(raw), int(bool(x_mosaic)), ptr(y), int(bool(y_mosaic)), ptr(var), ptr(mean), ptr(lap),
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
            check(lib.yond_nlf_maps_raw16(ptr(x), C.byref(raw), int(bool(x_mosaic)), None, 0, ptr(out), None, None, nimg, nb, H, W,
                                          int(bool(split_blocks)), int(k), 3, None, ptr(work), stream_ptr()))
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

    # -- SelfNLF / CollabNLF ----------------------------------------------------------------------
    def estimate(self, lr_rggb, hr_rggb=None, k=29, details=False, nseg=1, timings=None):
        """lr_rggb (and hr_rggb for collab): (B,h,w,4) with B = nseg * frames-per-image, image-major.  Returns the
        (beta1, beta2) of every image: (2,) for nseg == 1, else (nseg, 2)."""
        var, mean, lap = self.maps(lr_rggb, hr_rggb, k)
        th, pct, info = self.threshold_score3(lap, mean, step=5, nseg=nseg)
        reg, th = self.masked_fit(var, mean, lap, th, nseg=nseg)
        if details:
            return reg, dict(th=th, pct=pct, **info)
        return reg


_EST = threading.local()


def _estimator():
    """One estimator (and its device scratch) per host thread: the host-pipelined path runs two lanes concurrently."""
    est = getattr(_EST, "est", None)
    if est is None:
        est = _EST.est = NlfEstimator()
    return est


def _rggb_batch(raw, sidd_256):
    """Bayer (H,W) [or (B,H,W)] -> packed (B,h,w,4) device batch.  SIDD_256: the mosaic's 32 blocks become 32
    separate images, which is what stacking them on the channel axis means for a box filter (YOND_SIDD.py:65,91-93)."""
    t, _ = to_dev(raw)
    if t.dim() == 2:
        t = t[None]
    if sidd_256:
        B, H, W = t.shape
        assert B == 1 and W % 32 == 0
        t = t.reshape(H, 32, W // 32).permute(1, 0, 2).contiguous()
    return bayer2rggb(t)


def SelfNLF(lr_rggb, k=29, kwargs=None):
    kwargs = kwargs or {}
    t, _ = to_dev(lr_rggb)
    b = _as_batch4(t) if t.dim() == 3 else t
    if kwargs.get("SIDD_256"):
        B, h, w, _ = b.shape
        b = b.reshape(h, 32, w // 32, 4).permute(1, 0, 2, 3).contiguous()
    return _estimator().estimate(b, None, k)


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
    return _estimator().estimate(bl, bh, k)


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
