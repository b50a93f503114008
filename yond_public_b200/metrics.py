"""Image-quality metrics of the SIDD driver on the device (SURVEY 8(f)-3): the reference evaluates raw PSNR and a
MATLAB-style SSIM per 256x256 block of every denoised mosaic in CPU worker threads (YOND_SIDD.py:635-697); here one call
measures every block of a batch of mosaics on the GPU.  Same names as the reference: `compare_psnr` (its alias of
skimage.metrics.peak_signal_noise_ratio), `ssim`, `calculate_ssim`; `block_metrics` is the batched form the driver uses.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check, ptr, stream_ptr
from .isp import to_dev


def gaussian_kernel(ksize=11, sigma=1.5):
    """cv2.getGaussianKernel(ksize, sigma) for sigma > 0: exp(-(i-c)^2 / (2 sigma^2)) normalised to sum 1, float64."""
    x = np.arange(ksize, dtype=np.float64) - (ksize - 1) * 0.5
    k = np.exp(-0.5 / (sigma * sigma) * x * x)
    return k * (1.0 / k.sum())


_WIN = np.ascontiguousarray(gaussian_kernel(11, 1.5))


def block_metrics(a, b, nblk=1, data_range=1.0, ssim_scale=255.0, psnr=True, ssim=True):
    """a, b: (nimg, H, nblk*Wb) (or (H, nblk*Wb)) mosaics.  Returns device tensors (psnr, ssim), each (nimg, nblk) float64 (None
    when not requested): raw PSNR and the SSIM of (a*255, b*255) of every block, like YOND_SIDD.py:649-652."""
    ta, _ = to_dev(a)
    tb, _ = to_dev(b)
    if ta.dim() == 2:
        ta, tb = ta[None], tb[None]
    ta, tb = ta.contiguous(), tb.contiguous()
    assert ta.shape == tb.shape and ta.dtype == torch.float32 and tb.dtype == torch.float32
    nimg, H, Wm = ta.shape
    out_p = torch.empty((nimg, nblk), device=ta.device, dtype=torch.float64) if psnr else None
    out_s = torch.empty((nimg, nblk), device=ta.device, dtype=torch.float64) if ssim else None
    check(_lib.load().yond_block_metrics(ptr(ta), ptr(tb), nimg, H, Wm, int(nblk), float(data_range), float(ssim_scale),
                                         _WIN.ctypes.data_as(C.POINTER(C.c_double)), ptr(out_p), ptr(out_s), stream_ptr()))
    return out_p, out_s


def _is_u8(a):
    return (isinstance(a, np.ndarray) and a.dtype == np.uint8) or (torch.is_tensor(a) and a.dtype == torch.uint8)


def block_metrics_rgb8(a, b, nblk=1, psnr=True, ssim=True):
    """a, b: (nimg, H, nblk*Wb, 3) (or (H, nblk*Wb, 3)) uint8 pictures.  Returns device tensors (psnr, ssim), each (nimg, nblk)
    float64: PSNR at data_range 255 and the channel-mean SSIM of every block, like YOND_SIDD.py:661-665."""
    ta, _ = to_dev(a, dtype=torch.uint8)
    tb, _ = to_dev(b, dtype=torch.uint8)
    if ta.dim() == 3:
        ta, tb = ta[None], tb[None]
    ta, tb = ta.contiguous(), tb.contiguous()
    assert ta.shape == tb.shape and ta.dtype == torch.uint8 and tb.dtype == torch.uint8 and ta.shape[-1] == 3
    nimg, H, Wm, _ = ta.shape
    out_p = torch.empty((nimg, nblk), device=ta.device, dtype=torch.float64) if psnr else None
    out_s = torch.empty((nimg, nblk), device=ta.device, dtype=torch.float64) if ssim else None
    check(_lib.load().yond_block_metrics_rgb8(ptr(ta), ptr(tb), nimg, H, Wm, int(nblk), _WIN.ctypes.data_as(C.POINTER(C.c_double)),
                                              ptr(out_p), ptr(out_s), stream_ptr()))
    return out_p, out_s


def compare_psnr(image_true, image_test, data_range=1):
    """skimage.metrics.peak_signal_noise_ratio: float32 images (YOND_SIDD.py:651) or uint8 (H,W,3) pictures (:663)."""
    if _is_u8(image_true) and _is_u8(image_test):
        if data_range != 255:
            raise ValueError("uint8 pictures are measured at data_range=255")
        p, _ = block_metrics_rgb8(image_true, image_test, 1, ssim=False)
    else:
        p, _ = block_metrics(image_true, image_test, 1, data_range=data_range, ssim=False)
    return float(p.cpu()[0, 0])


def ssim(prediction, target):
    """YOND_SIDD.py:679-697 on one 2-D image pair already in [0, 255]."""
    _, s = block_metrics(np.asarray(prediction, np.float32), np.asarray(target, np.float32), 1, ssim_scale=1.0, psnr=False)
    return float(s.cpu()[0, 0])


def calculate_ssim(target, ref):
    """YOND_SIDD.py:700-721: 2-D images, or (H, W, 3) / (H, W, 1) channel means."""
    if _is_u8(target) and _is_u8(ref) and target.ndim == 3 and target.shape[2] == 3:
        if tuple(target.shape) != tuple(ref.shape):
            raise ValueError("Input images must have the same dimensions.")
        _, s = block_metrics_rgb8(target, ref, 1, psnr=False)
        return float(s.cpu()[0, 0])
    img1, img2 = np.asarray(target), np.asarray(ref)
    if img1.shape != img2.shape:
        raise ValueError("Input images must have the same dimensions.")
    if img1.ndim == 2:
        return ssim(img1, img2)
    if img1.ndim == 3:
        if img1.shape[2] == 3:
            return float(np.mean([ssim(img1[:, :, i], img2[:, :, i]) for i in range(3)]))
        if img1.shape[2] == 1:
            return ssim(np.squeeze(img1), np.squeeze(img2))
    raise ValueError("Wrong input image dimensions.")


def sidd_image_metrics(outputs, hr_raw, nblk=32):
    """The per-image numbers of multiprocess_plot (YOND_SIDD.py:643-656): mean over the mosaic's blocks of raw PSNR and SSIM; an
    output whose maximum is <= 0 scores (-1, -1).  outputs / hr_raw: (H, nblk*Wb) mosaics (NumPy or CUDA)."""
    t, _ = to_dev(outputs)
    if float(t.max()) <= 0:
        return -1.0, -1.0
    p, s = block_metrics(t, hr_raw, nblk)
    return float(p.mean().cpu()), float(s.mean().cpu())


def sidd_rgb_metrics(img_dn, img_hr, nblk=32):
    """YOND_SIDD.py:660-665: mean over the picture's blocks (split along W) of the sRGB PSNR and SSIM.  (H, nblk*Wb, 3) uint8."""
    p, s = block_metrics_rgb8(img_dn, img_hr, nblk)
    return float(p.mean().cpu()), float(s.mean().cpu())


def sidd_eval_image(outputs, hr_raw, meta=None, nblk=32, rgb=True):
    """The scoring half of multiprocess_plot (YOND_SIDD.py:635-668) for one image, all on the device: for every iteration's
    mosaic in `outputs` ((n_iter, H, nblk*Wb) or a list) the raw PSNR / SSIM against `hr_raw`, and — with `meta` (keys 'bayer_2by2',
    'wb', 'cst2') and rgb=True, the reference's save_plot branch — the sRGB PSNR / SSIM of the rendered pictures.  An iteration whose
    output has no positive value scores -1 like the reference and is not rendered.  Returns {'psnr': [...], 'ssim': [...],
    'psnr_rgb': [...], 'ssim_rgb': [...], 'img_hr': CUDA uint8 picture or None, 'img_dn': [pictures]}."""
    from .render import process_sidd_image
    hr, _ = to_dev(hr_raw)
    res = {"psnr": [], "ssim": [], "psnr_rgb": [], "ssim_rgb": [], "img_hr": None, "img_dn": []}
    do_rgb = bool(rgb and meta is not None)
    if do_rgb:
        res["img_hr"] = process_sidd_image(hr, meta["bayer_2by2"], meta["wb"], meta["cst2"])
    for out in outputs:
        t, _ = to_dev(out)
        if float(t.max()) <= 0:
            res["psnr"].append(-1.0)
            res["ssim"].append(-1.0)
            res["img_dn"].append(None)
            continue
        p, s = block_metrics(t, hr, nblk)
        res["psnr"].append(float(p.mean().cpu()))
        res["ssim"].append(float(s.mean().cpu()))
        if do_rgb:
            img = process_sidd_image(t, meta["bayer_2by2"], meta["wb"], meta["cst2"])
            pr, sr = block_metrics_rgb8(img, res["img_hr"], nblk)
            res["psnr_rgb"].append(float(pr.mean().cpu()))
            res["ssim_rgb"].append(float(sr.mean().cpu()))
            res["img_dn"].append(img)
    return res


_SSIM_WIN = 11
_GRID_Z = 65535  # blocks per grid z of the metric and render kernels


def _check_mosaics(name, t):
    if not torch.is_tensor(t) or not t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous() or t.dim() != 3:
        raise ValueError(f"{name}: need a contiguous CUDA float32 (nimg, H, nblk*Wb) tensor, got "
                         f"{tuple(t.shape) if torch.is_tensor(t) else type(t).__name__}"
                         f"{'' if not torch.is_tensor(t) else f' {t.dtype} on {t.device}'}")
    if t.data_ptr() % 16:
        raise ValueError(f"{name}: the data must be 16-byte aligned")


def sidd_eval_batch(raw_dns, hr_raw, metas=None, nblk=32, rounds=None, rgb=True):
    """sidd_eval_image for every image and round of a batch in one pass (YOND_SIDD.py:635-668, the scoring half of the SIDD eval):
    raw_dns is the list of (nimg, H, nblk*Wb) CUDA float32 mosaics per round that YOND_SIDD.iter_denoise_batch returns, hr_raw the
    (nimg, H, nblk*Wb) clean mosaics, metas nimg dicts with 'bayer_2by2', 'wb', 'cst2' (None: raw numbers only), rounds the rounds each
    image completed (iter_denoise_batch's res['rounds']; None: all of them).  Every image is rendered with its own metadata.

    Returns, after one read-back: 'psnr', 'ssim', 'psnr_rgb', 'ssim_rgb': (nround, nimg) float64 NumPy arrays — the mean over the
    blocks; raw (-1, -1) and sRGB NaN where the output has no positive value (the reference neither renders nor scores it); all four
    NaN for rounds at or beyond rounds[i] (repeats of the last completed round); sRGB NaN without metas or with rgb=False.
    'img_hr': (nimg, H, W, 3) and 'img_dn': (nround, nimg, H, W, 3) uint8 CUDA BGR pictures (None without metas or with rgb=False),
    'rendered': (nround, nimg) bool; the bytes of a picture that was not rendered are unspecified.
    Raises ValueError, before anything is enqueued, for inputs of the wrong number, shape, device, dtype or layout, metadata without
    a key or with an unknown Bayer pattern, rounds outside [1, nround], Wm % nblk != 0, blocks smaller than the SSIM window, and
    more block-channels (or pictures) than one launch of the metric (or render) kernel takes."""
    from .pipeline import _upload
    from .render import PIC_REC, camera_records
    dns = list(raw_dns)
    _check_mosaics("hr_raw", hr_raw)
    nimg, H, Wm = hr_raw.shape
    nround = len(dns)
    if nround < 1:
        raise ValueError("raw_dns: need at least one round")
    for r, t in enumerate(dns):
        _check_mosaics(f"raw_dns[{r}]", t)
        if t.shape != hr_raw.shape or t.device != hr_raw.device:
            raise ValueError(f"raw_dns[{r}]: shape {tuple(t.shape)} on {t.device}, hr_raw is {tuple(hr_raw.shape)} on {hr_raw.device}")
    do_rgb = bool(rgb and metas is not None)
    if metas is not None:
        metas = list(metas)
        if len(metas) != nimg:
            raise ValueError(f"metas: {len(metas)} entries for {nimg} images")
        cams = camera_records(metas)
    if rounds is None:
        rnd = np.full(nimg, nround, np.int32)
    else:
        rnd = np.asarray(rounds)
        if rnd.shape != (nimg,):
            raise ValueError(f"rounds: need one entry per image ({nimg}), got shape {rnd.shape}")
        if not np.issubdtype(rnd.dtype, np.integer) or (rnd < 1).any() or (rnd > nround).any():
            raise ValueError(f"rounds: need integers in [1, {nround}], got {rnd.tolist()}")
        rnd = rnd.astype(np.int32)
    nblk = int(nblk)
    if nblk < 1 or Wm % nblk:
        raise ValueError(f"nblk: {Wm} columns do not split into {nblk} blocks")
    Wb = Wm // nblk
    if H < _SSIM_WIN or Wb < _SSIM_WIN:
        raise ValueError(f"blocks of {H} x {Wb} are smaller than the {_SSIM_WIN} x {_SSIM_WIN} SSIM window")
    if H % 2 or Wm % 2:
        raise ValueError(f"H and W must be even (Bayer mosaics), got {H} x {Wm}")
    if nimg * nblk * (3 if do_rgb else 1) > _GRID_Z or (do_rgb and (nround + 1) * nimg > _GRID_Z):
        raise ValueError(f"{nimg} images x {nblk} blocks x {nround} rounds: more block-channels or pictures than one launch takes "
                         f"({_GRID_Z}); split the batch")

    dev = hr_raw.device
    blk = torch.empty((4 if do_rgb else 2, nround, nimg, nblk), device=dev, dtype=torch.float64)  # per-block psnr, ssim[, _rgb]
    out_max = torch.empty((nround, nimg), device=dev, dtype=torch.float32)
    table = torch.empty((nround, nimg, 4), device=dev, dtype=torch.float64)
    pics = torch.empty((nround + 1, nimg, H, Wm, 3), device=dev, dtype=torch.uint8) if do_rgb else None
    uploads = [rnd]
    if do_rgb:  # picture (0, i) the clean mosaic of image i, (r + 1, i) round r's output; none for the rounds it did not complete
        rec = np.zeros((nround + 1, nimg), PIC_REC)
        rec["cam"] = np.arange(nimg, dtype=np.int32)
        rec["src"][0] = hr_raw.data_ptr() + np.arange(nimg, dtype=np.uint64) * (H * Wm * 4)
        for r, t in enumerate(dns):
            live = r < rnd
            rec["src"][r + 1] = np.where(live, t.data_ptr() + np.arange(nimg, dtype=np.uint64) * (H * Wm * 4), 0)
            rec["src_max"][r + 1] = out_max[r].data_ptr() + np.arange(nimg, dtype=np.uint64) * 4
        uploads += [rec, cams]
    up, offs = _upload(uploads, dev)
    at = [C.c_void_p(up.data_ptr() + o) for o in offs]
    lib, s = _lib.load(), stream_ptr()
    win = _WIN.ctypes.data_as(C.POINTER(C.c_double))
    for r, t in enumerate(dns):
        check(lib.yond_seg_max(ptr(t), H * Wm, nimg, ptr(out_max[r]), s))
    if do_rgb:
        check(lib.yond_render_srgb_cams(at[1], at[2], ptr(pics), (nround + 1) * nimg, H, Wm, s))
    for r, t in enumerate(dns):
        check(lib.yond_block_metrics(ptr(t), ptr(hr_raw), nimg, H, Wm, nblk, 1.0, 255.0, win, ptr(blk[0, r]), ptr(blk[1, r]), s))
        if do_rgb:
            check(lib.yond_block_metrics_rgb8(ptr(pics[r + 1]), ptr(pics[0]), nimg, H, Wm, nblk, win, ptr(blk[2, r]), ptr(blk[3, r]), s))
    check(lib.yond_sidd_scores(ptr(blk[0]), ptr(blk[1]), ptr(blk[2]) if do_rgb else None, ptr(blk[3]) if do_rgb else None,
                               ptr(out_max), at[0], nround, nimg, nblk, ptr(table), s))
    host = table.cpu().numpy()
    res = {k: np.ascontiguousarray(host[..., j]) for j, k in enumerate(("psnr", "ssim", "psnr_rgb", "ssim_rgb"))}
    res["rendered"] = ~np.isnan(res["psnr_rgb"])  # with pictures, a rendered one always has finite sRGB numbers
    res["img_hr"] = pics[0] if do_rgb else None
    res["img_dn"] = pics[1:] if do_rgb else None
    return res
