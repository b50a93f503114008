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

FRAME_GEOM = np.dtype([("base", "<u8"), ("H", "<i4"), ("W", "<i4"), ("off", "<i8")])  # yond_frame_geom
assert FRAME_GEOM.itemsize == 24


RAW_DTYPES = (torch.int16, torch.uint16)


def check_frames(frames, nimg=None, k=29, raw=False):
    """Bayer frames of any even sizes as a list of (H, W) CUDA float32 tensors: a sequence of them, one (n, H, W) tensor or one (H, W)
    frame.  Raises ValueError for a count other than `nimg` (when given), a frame that is not a contiguous 2-D CUDA float32 tensor, an
    odd H or W, or a packed size (H/2, W/2) not larger than the filter radius k // 2 (the box filters reflect once at the border).
    raw: the frames are int16 / uint16 sensor mosaics instead.  Also raises ValueError for a list that mixes dtypes and for a frame whose
    data pointer is not aligned for the kernels' Bayer loads (8 bytes for float32, 4 for a 16-bit mosaic)."""
    if isinstance(frames, torch.Tensor):
        if frames.dim() not in (2, 3):
            raise ValueError(f"frames: one (n, H, W) tensor or (H, W) frame expected, got shape {tuple(frames.shape)}")
        frames = [frames] if frames.dim() == 2 else list(frames.unbind(0))
    else:
        try:
            frames = list(frames)
        except TypeError:
            raise ValueError(f"frames: a sequence of (H, W) tensors or one (n, H, W) tensor expected, got {type(frames).__name__}") from None
    if not frames or (nimg is not None and len(frames) != nimg):
        raise ValueError(f"frames: {nimg if nimg is not None else 'at least one'} frame(s) expected, got {len(frames)}")
    dtypes = sorted({str(f.dtype) for f in frames if isinstance(f, torch.Tensor)})
    if len(dtypes) > 1:
        raise ValueError(f"frames: one dtype expected, the list mixes {', '.join(dtypes)}")
    for i, f in enumerate(frames):
        if not isinstance(f, torch.Tensor) or f.dim() != 2:
            raise ValueError(f"frame {i}: a 2-D (H, W) tensor expected, got {getattr(f, 'shape', type(f).__name__)}")
        H, W = f.shape
        if H % 2 or W % 2:
            raise ValueError(f"frame {i}: H and W must be even (Bayer 2x2 cells), got {H}x{W}")
        if min(H, W) // 2 <= k // 2:
            raise ValueError(f"frame {i}: packed size {H // 2}x{W // 2} must exceed the filter radius {k // 2}")
        if raw and f.dtype not in RAW_DTYPES:
            raise ValueError(f"frame {i}: raw= given, so an int16 / uint16 sensor mosaic expected, got {f.dtype}")
        if not raw and f.dtype != torch.float32:
            hint = " (a 16-bit sensor mosaic needs raw=)" if f.dtype in RAW_DTYPES else ""
            raise ValueError(f"frame {i}: float32 expected, got {f.dtype}{hint}")
        if not f.is_contiguous():
            raise ValueError(f"frame {i}: a contiguous tensor expected")
        align = 4 if raw else 8
        if f.data_ptr() % align:
            raise ValueError(f"frame {i}: data pointer {f.data_ptr():#x} is not {align}-byte aligned (the Bayer loads of the kernels)")
        if not f.is_cuda:
            raise ValueError(f"frame {i}: a CUDA tensor expected, got one on {f.device}")
    return frames


class FrameTable:
    """Frames of any even sizes as the kernels address them: one yond_frame_geom record per frame (its address, H, W and the float offset
    of its maps, which is also its offset in a flat buffer of the frames' outputs) and the fit's nframes + 1 segment offsets, copied to
    the device together with the host arrays of `extra` in one non-blocking copy from pinned memory.  The frames are not copied: the
    caller keeps them alive and unchanged while work that reads them is enqueued.
    Attributes: geom / off (host), records / seg_off (device views), extra (device byte views, one per array of `extra`), nframes,
    n_el (= off[-1]), max_H, max_W, device."""

    def __init__(self, frames, extra=()):
        from .pipeline import _upload
        off = np.concatenate([[0], np.cumsum([f.numel() for f in frames])]).astype(np.uint64)
        geom = np.zeros(len(frames), FRAME_GEOM)
        geom["base"] = [f.data_ptr() for f in frames]
        geom["H"] = [f.shape[0] for f in frames]
        geom["W"] = [f.shape[1] for f in frames]
        geom["off"] = off[:-1].astype(np.int64)
        arrays = [geom, off] + list(extra)
        buf, offs = _upload(arrays, frames[0].device)
        views = [buf[o:o + np.asarray(a).nbytes] for o, a in zip(offs, arrays)]
        self.geom, self.off = geom, off
        self.records, self.seg_off, self.extra = views[0], views[1].view(torch.int64), views[2:]
        self.nframes, self.n_el = len(frames), int(off[-1])
        self.max_H, self.max_W = int(geom["H"].max()), int(geom["W"].max())
        self.device = frames[0].device

    def records_from(self, i):
        """The device records of frames i, i + 1, ..."""
        return self.records[i * FRAME_GEOM.itemsize:]


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

    def _fit(self, var, mean, lap, nimg, details=False, step=5, segments=None):
        """segments (optional): (seg_off, max_len), the device offsets (nimg + 1 uint64) of segments of different lengths and the
        longest length; else the maps are nimg segments of equal length."""
        lib, dev = self.lib, var.device
        n_el = var.numel()
        quants = np.ascontiguousarray(np.linspace(step, 100, 100 // step, endpoint=True), np.float64)
        regs = torch.empty((nimg, 2), device=dev, dtype=torch.float64)
        detail = torch.empty((nimg, self.DETAIL), device=dev, dtype=torch.float64) if details else None
        qp = quants.ctypes.data_as(C.POINTER(C.c_double))
        if segments is None:
            fwork = self._buf("fit", lib.yond_nlf_fit_work_bytes(nimg) + 256, dev)
            off = (-fwork.data_ptr()) % 256
            check(lib.yond_nlf_fit(ptr(var), ptr(mean), ptr(lap), n_el // nimg, nimg, qp, len(quants), ptr(regs), ptr(detail),
                                   ptr(fwork[off:]), stream_ptr()))
        else:
            seg_off, max_len = segments
            fwork = self._buf("fit", lib.yond_nlf_fit_ragged_work_bytes(nimg) + 256, dev)
            off = (-fwork.data_ptr()) % 256
            check(lib.yond_nlf_fit_ragged(ptr(var), ptr(mean), ptr(lap), ptr(seg_off), int(max_len), nimg, qp, len(quants), ptr(regs),
                                          ptr(detail), ptr(fwork[off:]), stream_ptr()))
        return (regs, detail) if details else regs

    # -- the self estimate of frames of different sizes (round 1 of IterDenoise on the full-resolution frames) ----------------
    def maps_frames(self, frames, k=29, var_map=None, seg_max=None, raw=None):
        """SelfNLF maps of a list of (H, W) CUDA float32 Bayer frames of any even sizes (check_frames), every box pass one launch for
        all of them.  Returns var, mean, lap: flat float32 maps, frame i's packed (H/2, W/2, 4) maps at float offsets
        off[i]:off[i + 1] (off: the host array of the nframes + 1 offsets), then off and the device copy of the offsets (uint64).
        frames may also be a FrameTable of frames already checked and uploaded.
        var_map (optional; float32 CUDA, at least off[-1] values): the var map goes there instead of the estimator's scratch, where no
        later call overwrites it — the cached noisy-frame statistics of the collab rounds (estimate_collab_frames).
        seg_max (optional, (nframes,) f32 CUDA): receives max(x, 0) per frame.
        raw: the frames are uint16 / int16 sensor mosaics and raw the CUDA uint8 tensor of their nframes yond_raw_norm records (one per
        frame, in the order of the frames): they are normalised on load."""
        lib = self.lib
        t = frames if isinstance(frames, FrameTable) else FrameTable(check_frames(frames, None, k, raw=raw is not None))
        dev, n_el = t.device, t.n_el
        maps = self._buf("maps3", 3 * n_el * 4, dev).view(torch.float32)
        var, mean, lap = maps[:n_el], maps[n_el:2 * n_el], maps[2 * n_el:3 * n_el]
        if var_map is not None:
            assert var_map.dtype == torch.float32 and var_map.is_cuda and var_map.numel() >= n_el
            var = var_map.reshape(-1)[:n_el]
        work = self._buf("maps", n_el * 4, dev)
        args = (t.nframes, t.max_H, t.max_W, ptr(var), ptr(mean), ptr(lap), int(k))
        if raw is not None:
            assert isinstance(raw, torch.Tensor) and raw.is_cuda and raw.dtype == torch.uint8 and raw.numel() >= t.nframes * 16
            check(lib.yond_nlf_maps_frames_raw16(ptr(t.records), ptr(raw), *args, ptr(seg_max), ptr(work), stream_ptr()))
        elif seg_max is not None:
            check(lib.yond_nlf_maps_frames_max(ptr(t.records), *args, ptr(work), stream_ptr(), ptr(seg_max)))
        else:
            check(lib.yond_nlf_maps_frames(ptr(t.records), *args, ptr(work), stream_ptr()))
        return var, mean, lap, t.off, t.seg_off

    def estimate_frames(self, frames, k=29, details=False, step=5, var_map=None, seg_max=None, raw=None):
        """Batched SelfNLF (SimpleNLF 'self') of a list of (H, W) CUDA float32 Bayer frames of any even sizes, or one (n, H, W) tensor:
        regs (nframes, 2) float64 on the device [, detail (nframes, DETAIL)], nothing read back.  The maps of all frames take one launch
        per box pass and the fit one set of launches.  A frame wider than 160 - 2*(k//2) packed pixels (every full-resolution frame) gets
        the same bits as estimate_dev on it alone; a narrower one takes the wide box-filter layout too and may differ from estimate_dev,
        which packs such frames side by side, in the float64 rounding of the window sums.  var_map, seg_max, raw and a FrameTable for
        frames: see maps_frames."""
        var, mean, lap, off, seg_off = self.maps_frames(frames, k, var_map, seg_max, raw)
        return self._fit(var, mean, lap, len(off) - 1, details, step, segments=(seg_off, int(np.diff(off).max())))

    def collab_maps_frames(self, y, table, lr_var, k=29):
        """CollabNLF maps (var, mean, lap) of frames of different sizes in one box pass: y is the flat float32 buffer of the frames of
        `table` (a FrameTable; frame i at float offset off[i], the layout of the maps — a round's output of iter_denoise_frames_dev),
        lr_var the var maps of the self estimate of the same table (maps_frames' var_map, read only)."""
        n_el = table.n_el
        assert y.is_cuda and y.dtype == torch.float32 and y.is_contiguous() and y.numel() >= n_el
        assert lr_var.dtype == torch.float32 and lr_var.is_cuda and lr_var.numel() >= n_el
        maps = self._buf("maps3", 3 * n_el * 4, y.device).view(torch.float32)
        var, mean, lap = maps[:n_el], maps[n_el:2 * n_el], maps[2 * n_el:3 * n_el]
        check(self.lib.yond_nlf_maps_frames_collab_cached(ptr(y), ptr(table.records), table.nframes, table.max_H, table.max_W,
                                                          ptr(lr_var.reshape(-1)), ptr(var), ptr(mean), ptr(lap), int(k), stream_ptr()))
        return var, mean, lap

    def estimate_collab_frames(self, y, table, lr_var, k=29, details=False, step=5):
        """CollabNLF (beta1, beta2) of a collab round of frames of different sizes (collab_maps_frames + the ragged fit): regs (nframes, 2)
        float64 on the device."""
        var, mean, lap = self.collab_maps_frames(y, table, lr_var, k)
        off = table.off
        return self._fit(var, mean, lap, table.nframes, details, step, segments=(table.seg_off, int(np.diff(off).max())))

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
