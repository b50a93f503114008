"""sRGB render of the SIDD driver on the device (SURVEY 8(f)-3): `process_sidd_image` (utils/sidd_utils.py:156-180) turns a
mosaic into the 8-bit BGR picture the reference saves and scores (YOND_SIDD.py:601-607, :637-665).  The reference does it on the
CPU through NumPy and OpenCV's edge-aware demosaic; here it is ONE kernel from the float32 mosaic to the uint8 picture
(csrc/render_kernels.cu).  Same names and arguments as the reference; the 3x3 colour algebra stays NumPy float64 on the host,
exactly as the reference computes it.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check, ptr, stream_ptr
from .isp import _back, to_dev

_RGB2XYZ = np.array([[0.4124564, 0.3575761, 0.1804375], [0.2126729, 0.7151522, 0.0721750], [0.0193339, 0.1191920, 0.9503041]])
# flip_bayer (utils/sidd_utils.py:182-196): pattern -> (fliplr, flipud)
_FLIPS = {((1, 2), (2, 3)): (0, 0), ((2, 1), (3, 2)): (1, 0), ((2, 3), (1, 2)): (0, 1), ((3, 2), (2, 1)): (1, 1)}


def _pattern_key(bayer_pattern):
    key = tuple(tuple(int(v) for v in row) for row in np.asarray(bayer_pattern).tolist())
    if key not in _FLIPS:
        raise ValueError(f"Unknown Bayer pattern {bayer_pattern}")  # the reference drops into pdb here
    return key


def cam2rgb_matrix(cst):
    """utils/sidd_utils.py:161-170: row-normalised inverse of cst x rgb2xyz, float64."""
    rgb2cam = np.matmul(np.asarray(cst, np.float64), _RGB2XYZ)
    cam2rgb = np.linalg.inv(rgb2cam)
    return cam2rgb / np.sum(cam2rgb, axis=-1, keepdims=True)


# yond_render_cam / yond_render_pic (include/yond_b200.h)
CAM_REC = np.dtype([("gain", "<f8", (4,)), ("cam2rgb", "<f8", (9,)), ("flip_lr", "<i4"), ("flip_ud", "<i4")])
PIC_REC = np.dtype([("src", "<u8"), ("src_max", "<u8"), ("cam", "<i4"), ("reserved", "<i4")])
META_KEYS = ("bayer_2by2", "wb", "cst2")


def camera_records(metas):
    """One yond_render_cam per SIDD metadata dict (keys 'bayer_2by2', 'wb', 'cst2'): the flips (utils/sidd_utils.py:182-196), gains
    per 2x2 site (:249-252) and cam2rgb matrix (:161-170) the render of that image uses, in the reference's float64 NumPy arithmetic —
    the one place process_sidd_image and metrics.sidd_eval_batch take them from.  ValueError for a missing key or an unknown Bayer
    pattern."""
    rec = np.zeros(len(metas), CAM_REC)
    for i, meta in enumerate(metas):
        missing = [k for k in META_KEYS if k not in meta]
        if missing:
            raise ValueError(f"meta {i} lacks {missing}")
        rec["flip_lr"][i], rec["flip_ud"][i] = _FLIPS[_pattern_key(meta["bayer_2by2"])]
        wb = np.asarray(meta["wb"], np.float64)
        rec["gain"][i] = [1 / wb[0][0], 1 / wb[0][1], 1 / wb[0][1], 1 / wb[0][2]]
        rec["cam2rgb"][i] = cam2rgb_matrix(meta["cst2"]).reshape(-1)
    return rec


def process_sidd_image(image, bayer_pattern, wb, cst, *, save_file_rgb=None):
    """utils/sidd_utils.py:156-180.  image: (H,W) (or (B,H,W) sharing one camera) float32 mosaic, NumPy or CUDA tensor; returns the
    (H,W,3) uint8 BGR picture (NumPy in -> NumPy out, tensor in -> CUDA tensor out), in the flipped orientation the reference
    leaves it in."""
    cam = camera_records([{"bayer_2by2": bayer_pattern, "wb": wb, "cst2": cst}])[0]
    flip_lr, flip_ud = int(cam["flip_lr"]), int(cam["flip_ud"])
    gains = np.ascontiguousarray(cam["gain"][[0, 1, 3]])
    ccm = np.ascontiguousarray(cam["cam2rgb"])
    x, np_in = to_dev(image)
    batched = x.dim() == 3
    xb = x if batched else x[None]
    B, H, W = xb.shape
    out = torch.empty((B, H, W, 3), device=x.device, dtype=torch.uint8)
    check(_lib.load().yond_render_srgb(ptr(xb), ptr(out), B, H, W, flip_lr, flip_ud, gains.ctypes.data_as(C.POINTER(C.c_double)),
                                       ccm.ctypes.data_as(C.POINTER(C.c_double)), stream_ptr()))
    res = _back(out if batched else out[0], np_in)
    if save_file_rgb:
        import cv2  # file output only (the reference's cv2.imwrite)
        cv2.imwrite(save_file_rgb, res if isinstance(res, np.ndarray) else res.cpu().numpy())
    return res


def demosaic_ea(bayer_u16):
    """cv2.cvtColor(bayer, cv2.COLOR_BayerBG2RGB_EA) for uint16 mosaics (H,W) or (B,H,W): the integer stage of the render
    (utils/sidd_utils.py:244) on its own."""
    x, np_in = to_dev(np.ascontiguousarray(bayer_u16, np.uint16) if isinstance(bayer_u16, np.ndarray) else bayer_u16, dtype=torch.uint16)
    batched = x.dim() == 3
    xb = x if batched else x[None]
    B, H, W = xb.shape
    out = torch.empty((B, H, W, 3), device=x.device, dtype=torch.uint16)
    check(_lib.load().yond_demosaic_ea(ptr(xb), ptr(out), B, H, W, stream_ptr()))
    return _back(out if batched else out[0], np_in)
