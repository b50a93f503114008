"""The YOND blind-denoise pipeline on B200, behind the reference driver's method surface
(YOND_SIDD.py:136-483: Simple_Denoiser, VST_Denoiser, IterDenoise) plus a batched, device-resident engine.

Per frame: pack -> noise-parameter estimate (SimpleNLF) -> bias LUT -> generalized-Anscombe VST -> normalise ->
reflect-pad -> AWGN denoiser (tcgen05 conv stack) -> crop -> de-normalise -> inverse VST -> unpack.
All per-pixel work runs in libyond_b200 kernels; the host keeps the reference's scalar logic and guards.
"""
from __future__ import annotations

import ctypes as C

import os

import numpy as np
import torch

from . import _lib, archs, isp, nlf
from ._lib import VstParams, check, ptr, stream_ptr

SIGMA_CORR_PRE = 1.03  # YOND_SIDD.py:284
RAW_REC = np.dtype([("black", "<f4"), ("white", "<f4"), ("ratio", "<f4"), ("clip", "<i4")])  # yond_raw_norm
assert RAW_REC.itemsize == C.sizeof(_lib.RawNorm)


def _per_image(v, nimg, name):
    a = np.asarray(v)
    if a.ndim > 1 or (a.ndim == 1 and a.shape[0] != nimg):
        raise ValueError(f"{name}: a scalar or {nimg} values (one per image) expected, got shape {a.shape}")
    try:
        f = a.astype(np.float64)
    except (TypeError, ValueError):
        raise ValueError(f"{name}: numbers expected, got {v!r}") from None
    if not np.isfinite(f).all():
        raise ValueError(f"{name}: non-finite value in {v!r}")
    return np.broadcast_to(a, (nimg,))


def batch_exposure(p, nimg, raw=None):
    """The exposure parameters of a batch of `nimg` images, one value per image.  p['wp'], p['bl'], p['scale'] (default wp - bl) and
    each entry of raw = (black, white, ratio[, clip]) are a scalar (every image) or a length-nimg sequence / 1-D array.
    Returns (scale_est, scale, raw_rec): float64 (nimg,) arrays scale_est = wp - bl and scale, and the (nimg,) RAW_REC records of
    raw (None without raw).  Raises ValueError for a wrong length, wp <= bl, scale <= 0, ratio <= 0, white <= black or a
    non-finite value."""
    wp, bl = _per_image(p["wp"], nimg, "p['wp']"), _per_image(p["bl"], nimg, "p['bl']")
    scale_est = (wp - bl).astype(np.float64)
    if not (scale_est > 0).all():
        raise ValueError(f"p['wp'] must exceed p['bl'] for every image: wp={p['wp']!r}, bl={p['bl']!r}")
    scale = _per_image(p["scale"], nimg, "p['scale']").astype(np.float64) if "scale" in p else scale_est
    if not (scale > 0).all():
        raise ValueError(f"p['scale'] must be positive for every image, got {p['scale']!r}")
    if raw is None:
        return scale_est, scale, None
    if not 3 <= len(raw) <= 4:
        raise ValueError(f"raw = (black, white, ratio[, clip]) expected, got {raw!r}")
    rec = np.zeros(nimg, RAW_REC)
    for field, v in zip(("black", "white", "ratio", "clip"), raw):
        a = _per_image(v, nimg, f"raw {field}")
        rec[field] = a.astype(bool) if field == "clip" else a.astype(np.float64)
    if not (rec["white"] > rec["black"]).all():
        raise ValueError(f"raw: white must exceed black for every image, got {raw!r}")
    if not (rec["ratio"] > 0).all():
        raise ValueError(f"raw: ratio must be positive for every image, got {raw!r}")
    return scale_est, scale, rec


def _upload(arrays, device):
    """One non-blocking copy of the concatenated bytes of `arrays` from pinned memory on the current stream; returns the device byte
    buffer and the byte offset of each array.  The caching allocators keep both buffers until the copy and the kernels enqueued
    after it on this stream have run, so nothing waits for the host."""
    offs, parts, n = [], [], 0
    for a in arrays:
        n = (n + 7) // 8 * 8
        offs.append(n)
        parts.append((n, np.ascontiguousarray(a).view(np.uint8).reshape(-1)))
        n += parts[-1][1].size
    host = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    h = host.numpy()
    for o, b in parts:
        h[o:o + b.size] = b
    return host.to(device, non_blocking=True), offs


def build_net(arch: dict, device="cuda"):
    """globals()[arch['name']](arch) of the reference (YOND_SIDD.py:177)."""
    cls = getattr(archs, arch["name"], None)
    if cls is None:
        raise NotImplementedError(f"arch '{arch['name']}' is outside the B200 hot path (UNetSeeInDark, GuidedResUnet, SNRnet, ResUnet2)")
    return cls(arch).to(device)


class YondEngine:
    """Batched VST-denoise of equally sized Bayer frames, device-resident."""

    def __init__(self, net, arch, biaslut=None, chunk=None):
        self.lib = _lib.load()
        self.net = net
        self.arch = arch
        self.guided = "guided" in arch
        self.biaslut = biaslut
        self.chunk = chunk
        self._bufs = {}
        self.forward = None  # optional replacement of net.forward_nhwc (parallel.BandShardedForward: one frame across ranks)

    def _buf(self, name, shape, dtype, device):
        n = int(np.prod(shape))
        b = self._bufs.get(name)
        if b is None or b.numel() < n or b.dtype != dtype or b.device != device:
            b = torch.empty(n, device=device, dtype=dtype)
            self._bufs[name] = b
        return b[:n].view(*shape)

    def default_chunk(self, B, hp, wp):
        if self.chunk:
            return min(B, int(self.chunk))
        per = max(1, hp * wp * 400)  # ~bytes of activations per frame (yond_net_workspace_bytes: ~335 B per packed pixel)
        cap = int(os.environ.get("YOND_CHUNK", "640"))
        budget = int(os.environ.get("YOND_CHUNK_GIB", "16")) << 30  # of the 180 GB: a 12 MP frame needs ~1.1 GiB
        return int(max(1, min(B, budget // per, cap)))

    # ------------------------------------------------------------------------------------------
    def make_params(self, gains, sigmas, scale, bias_corr, vst_type, frame_max, device, fixed_table=None):
        """Per-frame yond_vst_params + the bias rows they index, for CALLER-GIVEN (gain, sigma) — the function-level
        VST_Denoiser surface.  (The blind pipeline fills the same structures on the device: `chain_params`.)

        Bias source per frame, like the reference (YOND_SIDD.py:252-262, utils/isp_algos.py:196-231): only
        bias_corr == 'pre' applies a bias ('post' computes one and never uses it, :261 / :294-295); the BiasLUT row for this
        sigma/K when a LUT is loaded and sigma/K is inside its range, otherwise the fallback `get_bias` table up to this
        frame's maximum (`frame_max`: callable returning per-frame max in DN), generated on the device.  `scale`: one value or one
        per frame."""
        gains = np.asarray(gains, np.float64)
        sigmas = np.asarray(sigmas, np.float64)
        B = len(gains)
        exact = 1 if (bias_corr is None and vst_type == "exact") else 0
        row_of = np.full(B, -1, np.int32)
        table_n_of = np.zeros(B, np.int32)
        jobs = []  # (row index, kind, payload)
        if bias_corr == "pre":
            # frames come in runs sharing (K, sigma) (the 32 blocks of an image): resolve each distinct pair once
            pairs, inverse = np.unique(np.stack([gains, sigmas], 1), axis=0, return_inverse=True)
            inverse = np.asarray(inverse).reshape(-1)
            fmax, key_row = None, {}
            for u, (k, s) in enumerate(pairs):
                k, s = float(k), float(s)
                idx = np.nonzero(inverse == u)[0]
                if self.biaslut is not None and self.biaslut.in_range(k, s):
                    row_of[idx] = len(jobs)
                    jobs.append(("lut", k, s))
                    continue
                for b in idx:
                    if fixed_table is not None:
                        key = ("fixed",)
                    else:
                        if fmax is None:
                            fmax = frame_max()
                        key = ("tab", k, s, float(np.ceil(np.float32(fmax[b]))))
                    if key not in key_row:
                        key_row[key] = len(jobs)
                        jobs.append(("fixed", fixed_table) if fixed_table is not None else ("tab", k, s, np.float32(fmax[b])))
                    row_of[b] = key_row[key]
        rows = xnodes = None
        stride = 1921
        if jobs:
            lib = self.lib
            sizes = []
            for j in jobs:
                if j[0] == "lut":
                    sizes.append(1921)
                elif j[0] == "fixed":
                    sizes.append(len(j[1][0]))
                else:
                    sizes.append(int(lib.yond_bias_table_nodes(float(j[3]))))
            stride = max(1921, max(sizes))
            rows = torch.zeros((len(jobs), stride), device=device, dtype=torch.float32)
            xnodes = torch.zeros((len(jobs), stride), device=device, dtype=torch.float32)
            work = self._buf("chain1", (int(lib.yond_chain_work_bytes(1)),), torch.uint8, device)
            for i, j in enumerate(jobs):
                if j[0] == "lut":
                    self.biaslut.sigma_row(j[1], j[2], out=rows[i, :1921])
                    xnodes[i, :1921] = self.biaslut.device_table()[1]
                elif j[0] == "fixed":
                    nodes, vals = j[1]
                    xnodes[i, :len(nodes)] = torch.from_numpy(np.asarray(nodes, np.float32)).to(device)
                    rows[i, :len(vals)] = torch.from_numpy(np.asarray(vals, np.float32)).to(device)
                else:
                    check(lib.yond_bias_table(j[1], j[2], float(j[3]), ptr(xnodes[i]), ptr(rows[i]), stride, None, ptr(work), stream_ptr()))
            sz = np.asarray(sizes, np.int32)
            is_tab = np.asarray([j[0] != "lut" for j in jobs])
            table_n_of = np.where(row_of >= 0, np.where(is_tab, sz, 0)[np.maximum(row_of, 0)], 0).astype(np.int32)
        # VST(0) / VST(scale) / nsr in float64 on the host (YOND_SIDD.py:264-268), vectorised over the batch
        c0 = (3 / 8) * gains ** 2 + sigmas ** 2
        lower = 2 / gains * np.sqrt(np.maximum(c0, 0))
        upper = 2 / gains * np.sqrt(np.maximum(gains * scale + c0, 0))
        rec = np.zeros(B, dtype=np.dtype([("gain", "<f4"), ("sigma", "<f4"), ("scale", "<f4"), ("lower", "<f4"), ("upper", "<f4"),
                                          ("lut_row", "<i4"), ("table_n", "<i4"), ("exact", "<i4")]))
        assert rec.dtype.itemsize == C.sizeof(VstParams)
        rec["gain"], rec["sigma"], rec["scale"], rec["lower"], rec["upper"] = gains, sigmas, scale, lower, upper
        rec["lut_row"] = row_of
        rec["table_n"] = table_n_of
        rec["exact"] = exact
        t = (1 / (upper - lower) * (SIGMA_CORR_PRE if bias_corr == "pre" else 1.0)).astype(np.float32)  # :268, :284-285
        raw = torch.from_numpy(rec.view(np.uint8).copy()).to(device)
        return raw, rows, xnodes, stride, torch.from_numpy(t).to(device)

    # ------------------------------------------------------------------------------------------
    # The same structures filled ON THE DEVICE from the estimator's (beta1, beta2): no host read-back between the
    # estimate and the denoiser (YOND_SIDD.py:356, :438-447, :252-269, :284-285).
    BIAS_MODES = {None: 0, "pre": 1, "post": 2}
    max_value = 1.0  # upper bound of the (normalised) input data assumed when sizing fallback bias tables; raise for noclip data

    def chain_params(self, regs, seg_max, nseg, fps, scale_est, scale, bound_scale, rnd, bias_corr, vst_type, prev=None, scales_dev=None):
        """regs: (nseg,2) float64 CUDA.  Returns a dict of device buffers: params (bytes), t, rows, xnodes, stride,
        regs4 (nseg,4: beta1, beta2 after the guards, gain, sigma), ok (nseg int32: still live after this round).
        scale_est, scale, bound_scale: one value or one per image.  scales_dev (optional): the same as a (nseg,3) float64 CUDA array
        already on the device; else they are copied there.
        prev: the chain of the previous round (rnd >= 2) — its params are kept by images that are not live, and its ok is chained."""
        if bias_corr not in self.BIAS_MODES:
            raise NotImplementedError(f"bias_corr={bias_corr!r}")
        lib, dev = self.lib, regs.device
        mode = self.BIAS_MODES[bias_corr]
        exact = 1 if (bias_corr is None and vst_type == "exact") else 0
        lut = self.biaslut.device_arrays() if (self.biaslut is not None and mode == 1) else None
        scale_est, scale, bound_scale = (np.broadcast_to(np.asarray(v, np.float64), (nseg,)) for v in (scale_est, scale, bound_scale))
        if scales_dev is None:
            buf, _ = _upload([np.stack([scale_est, scale, bound_scale], 1)], dev)
            scales_dev = buf.view(torch.float64)
        stride = 1921
        rows = xnodes = None
        if mode == 1:  # rows sized for the largest bound of the batch
            cap = int(lib.yond_bias_table_nodes(float((np.float32(self.max_value) * bound_scale.astype(np.float32)).max())))
            stride = max(1921, cap) if lut is not None else max(cap, 8)
            rows = torch.empty((nseg, stride), device=dev, dtype=torch.float32)
            xnodes = torch.empty((nseg, stride), device=dev, dtype=torch.float32)
        psz = C.sizeof(VstParams)
        out = dict(params=torch.empty(nseg * fps * psz, device=dev, dtype=torch.uint8),
                   t=torch.empty(nseg * fps, device=dev, dtype=torch.float32), rows=rows, xnodes=xnodes, stride=stride,
                   regs4=torch.empty((nseg, 4), device=dev, dtype=torch.float64), ok=torch.empty(nseg, device=dev, dtype=torch.int32))
        work = self._buf("chain", (int(lib.yond_chain_work_bytes(nseg)),), torch.uint8, dev)
        # the per-image array replaces the scalar (scale_est, scale, bound_scale) arguments
        check(lib.yond_vst_params_fill(ptr(regs), ptr(seg_max), nseg, fps, 0.0, 0.0, 0.0, int(rnd), mode,
                                       exact, ptr(lut[0]) if lut else None, ptr(lut[2]) if lut else None, ptr(lut[1]) if lut else None,
                                       1921, 1101, ptr(prev["params"]) if prev is not None else None, ptr(out["params"]), ptr(out["t"]),
                                       ptr(rows), ptr(xnodes), stride, ptr(out["regs4"]), ptr(out["ok"]), ptr(work), stream_ptr(),
                                       ptr(prev["ok"]) if prev is not None else None, ptr(scales_dev)))
        return out

    def vst_denoise_dev(self, frames, chain, out, frames_per_row=1, fps=1, select=False, fallback=None, clip01=True, raw=None, shape=None):
        """VST_Denoiser for frames (B,H,W) with device-filled parameters; writes `out` (plain (B,H,W) or the mosaic layout
        (B/n, H, n*W) for frames_per_row = n).  select: frames of images with chain['ok'] == 0 copy `fallback` instead.
        raw: frames is the uint16 sensor mosaic and raw the CUDA uint8 tensor of the yond_raw_norm records of its images (fps frames
        each).
        shape = (B, H, W): frames is instead the device yond_frame_geom records (nlf.FrameTable) of B frames of that size, each read where
        it lies (uint16 mosaics with raw; fps = 1)."""
        B, H, W = frames.shape if shape is None else shape
        dev = frames.device
        h, w = H // 2, W // 2
        pl, pr, pt, pb = isp.get_p2d((B, 4, h, w), base=32)
        hp, wp = h + pt + pb, w + pl + pr
        unit = int(np.lcm(frames_per_row, fps))
        cb = max(unit, self.default_chunk(B, hp, wp) // unit * unit)
        z = self._buf("z", (cb, hp, wp, 4), torch.float32, dev)
        y = self._buf("y", (cb, hp, wp, 4), torch.float32, dev)
        ub = self._buf("ub", (cb,), torch.float32, dev)
        psz = C.sizeof(VstParams)
        st = stream_ptr()
        params, t = chain["params"], chain["t"]
        for b0 in range(0, B, cb):
            n = min(cb, B - b0)
            pch = params[b0 * psz:]
            if shape is not None:  # a table of frames of one size
                check(self.lib.yond_vst_fwd_frames(ptr(frames[b0 * nlf.FRAME_GEOM.itemsize:]),
                                                   ptr(raw[b0 * RAW_REC.itemsize:]) if raw is not None else None, ptr(z[:n]), ptr(ub[:n]),
                                                   n, H, W, pl, pr, pt, pb, ptr(pch), ptr(chain["rows"]), ptr(chain["xnodes"]),
                                                   chain["stride"], st))
            elif raw is not None:  # uint16 sensor mosaic, normalised on load with each image's record (b0 starts an image)
                check(self.lib.yond_vst_fwd_raw16(ptr(frames[b0:b0 + n]), None, ptr(z[:n]), ptr(ub[:n]), n, H, W, pl, pr, pt, pb, ptr(pch),
                                                  ptr(chain["rows"]), ptr(chain["xnodes"]), chain["stride"], st,
                                                  ptr(raw[b0 // fps * RAW_REC.itemsize:]), fps))
            else:
                check(self.lib.yond_vst_fwd(ptr(frames[b0:b0 + n]), ptr(z[:n]), ptr(ub[:n]), n, H, W, pl, pr, pt, pb, ptr(pch),
                                            ptr(chain["rows"]), ptr(chain["xnodes"]), chain["stride"], st))
            (self.forward or self.net.forward_nhwc)(z[:n], ub[:n], t[b0:b0 + n] if self.guided else None, out=y[:n])
            check(self.lib.yond_vst_inv_place(ptr(y[:n]), ptr(out), n, H, W, pl, pr, pt, pb, ptr(pch), int(clip01), frames_per_row, b0,
                                              ptr(chain["ok"]) if select else None, fps, ptr(fallback) if select else None, st))
        return out

    # ------------------------------------------------------------------------------------------
    def vst_denoise(self, bayer, gains, sigmas, scale, bias_corr="pre", vst_type="exact", clip01=True, table_bound=None, fixed_table=None, out=None):
        """VST_Denoiser (YOND_SIDD.py:250-299) for a batch: bayer (B,H,W) CUDA f32 -> (B,H,W) CUDA f32.  gains, sigmas and scale:
        one value or one per frame."""
        B, H, W = bayer.shape
        dev = bayer.device
        h, w = H // 2, W // 2
        pl, pr, pt, pb = isp.get_p2d((B, 4, h, w), base=32)
        hp, wp = h + pt + pb, w + pl + pr
        gains = np.broadcast_to(np.asarray(gains, np.float64), (B,))
        sigmas = np.broadcast_to(np.asarray(sigmas, np.float64), (B,))
        scale = np.broadcast_to(np.asarray(scale, np.float64), (B,))
        # upper bound of a fallback table: the caller's bound (YOND_SIDD.py:393-395: one table per image, up to the image
        # max) or, like VST_Denoiser / BiasLUT.get_lut on their own, each frame's max in DN (float32 product)
        if table_bound is not None:
            frame_max = lambda: np.full(B, np.float32(table_bound), np.float32)
        else:
            frame_max = lambda: (bayer.amax(dim=(1, 2)).clamp_min(0).cpu().numpy().astype(np.float32) * scale.astype(np.float32))
        params, rows, xnodes, stride, t = self.make_params(gains, sigmas, scale, bias_corr, vst_type, frame_max, dev, fixed_table)
        if out is None:
            out = torch.empty_like(bayer)
        cb = self.default_chunk(B, hp, wp)
        z = self._buf("z", (cb, hp, wp, 4), torch.float32, dev)
        y = self._buf("y", (cb, hp, wp, 4), torch.float32, dev)
        ub = self._buf("ub", (cb,), torch.float32, dev)
        psz = C.sizeof(VstParams)
        st = stream_ptr()
        for b0 in range(0, B, cb):
            n = min(cb, B - b0)
            pch = params[b0 * psz:]
            check(self.lib.yond_vst_fwd(ptr(bayer[b0:b0 + n]), ptr(z[:n]), ptr(ub[:n]), n, H, W, pl, pr, pt, pb, ptr(pch),
                                        ptr(rows), ptr(xnodes), stride, st))
            self.net.forward_nhwc(z[:n], ub[:n], t[b0:b0 + n] if self.guided else None, out=y[:n])
            check(self.lib.yond_vst_inv(ptr(y[:n]), ptr(out[b0:b0 + n]), n, H, W, pl, pr, pt, pb, ptr(pch), int(clip01), st))
        return out

    # ------------------------------------------------------------------------------------------
    # Halo-overlapped tiling of one full-resolution frame (new design; the reference forwards whole frames,
    # YOND_SIDD.py:281-290).  The receptive field of the networks is 107 (UNetSeeInDark) / 123 (GuidedResUnet, SNRnet)
    # packed pixels (SURVEY.md §5), so a 128-pixel halo with tile origins on multiples of 16 reproduces the whole-frame
    # forward; the frame-global quantities (per-sample max `ub`, guidance `t`, VST constants) are computed on the whole
    # frame BEFORE tiling and handed to every tile.
    HALO = 128

    @staticmethod
    def tile_grid(hp, wp, core):
        """Tile cores (y0, x0, ch, cw) covering the padded frame; `core` is a multiple of 16."""
        assert core % 16 == 0
        return [(y0, x0, min(core, hp - y0), min(core, wp - x0)) for y0 in range(0, hp, core) for x0 in range(0, wp, core)]

    def net_forward_tiled(self, z, ub, t, core=512, tiles=None, y=None):
        """z: (1,hp,wp,4) padded frame on device -> y (1,hp,wp,4).  Only `tiles` (default: all) are computed — a rank
        of a tile-sharded run passes its own share and the cores are gathered afterwards.

        A tile is its core plus a halo that is CUT at the frame border: the network zero-pads every feature map at the
        true border, so nothing outside the frame may be fed to it (zeros at the input would become non-zero features
        after the first bias).  Tiles therefore differ in shape (corner / edge / interior); tiles of equal shape are
        forwarded together as one batch (a 768x768 tile is as much work as 36 SIDD blocks)."""
        _, hp, wp, _ = z.shape
        halo = self.HALO
        grid = self.tile_grid(hp, wp, core)
        tiles = list(range(len(grid))) if tiles is None else list(tiles)
        if y is None:
            y = torch.zeros_like(z)
        st = stream_ptr()
        groups = {}
        for ti in tiles:
            y0, x0, ch, cw = grid[ti]
            ty0, tx0 = max(0, y0 - halo), max(0, x0 - halo)
            ty1, tx1 = min(hp, y0 + ch + halo), min(wp, x0 + cw + halo)
            groups.setdefault((ty1 - ty0, tx1 - tx0), []).append((y0, x0, ch, cw, ty0, tx0))
        max_px = 640 * 128 * 128  # same activation budget as a 640-block chunk
        for (th, tw), members in groups.items():
            per = max(1, max_px // (th * tw))
            for g0 in range(0, len(members), per):
                part = members[g0:g0 + per]
                n = len(part)
                zt = self._buf("tile_in", (n, th, tw, 4), torch.float32, z.device)
                yt = self._buf("tile_out", (n, th, tw, 4), torch.float32, z.device)
                for i, (y0, x0, ch, cw, ty0, tx0) in enumerate(part):
                    check(self.lib.yond_tile_extract(ptr(z[0]), ptr(zt[i]), hp, wp, ty0, tx0, th, tw, st))
                ubn = ub.reshape(1).expand(n).contiguous()
                tn = None if t is None else t.reshape(1).expand(n).contiguous()
                self.net.forward_nhwc(zt, ubn, tn, out=yt)
                for i, (y0, x0, ch, cw, ty0, tx0) in enumerate(part):
                    check(self.lib.yond_tile_insert(ptr(yt[i]), ptr(y[0]), hp, wp, ty0, tx0, th, tw, y0 - ty0, x0 - tx0, ch, cw, st))
        return y

    def vst_denoise_tiled(self, frame, gain, sigma, scale, bias_corr="pre", vst_type="exact", clip01=True, core=512,
                          tiles=None, return_padded=False):
        """VST_Denoiser on one full-resolution Bayer frame (H,W) with halo tiling of the network stage."""
        H, W = frame.shape
        dev = frame.device
        h, w = H // 2, W // 2
        pl, pr, pt, pb = isp.get_p2d((1, 4, h, w), base=32)
        hp, wp = h + pt + pb, w + pl + pr
        fmax = lambda: (frame.amax().clamp_min(0).reshape(1).cpu().numpy().astype(np.float32) * np.float32(scale))
        params, rows, xnodes, stride, t = self.make_params([gain], [sigma], float(scale), bias_corr, vst_type, fmax, dev)
        z = torch.empty((1, hp, wp, 4), device=dev, dtype=torch.float32)
        ub = torch.empty(1, device=dev, dtype=torch.float32)
        st = stream_ptr()
        check(self.lib.yond_vst_fwd(ptr(frame), ptr(z), ptr(ub), 1, H, W, pl, pr, pt, pb, ptr(params), ptr(rows), ptr(xnodes), stride, st))
        y = self.net_forward_tiled(z, ub, t if self.guided else None, core=core, tiles=tiles)
        if return_padded:  # a rank of a sharded run returns its partial padded output for the gather
            return y, (params, (pl, pr, pt, pb))
        out = torch.empty_like(frame)
        check(self.lib.yond_vst_inv(ptr(y), ptr(out), 1, H, W, pl, pr, pt, pb, ptr(params), int(clip01), st))
        return out

    def simple_denoise(self, bayer, out=None):
        """Simple_Denoiser (YOND_SIDD.py:238-248) for a batch (no VST; non-guided nets only, like the reference)."""
        B, H, W = bayer.shape
        dev = bayer.device
        h, w = H // 2, W // 2
        pl, pr, pt, pb = isp.get_p2d((B, 4, h, w), base=32)
        hp, wp = h + pt + pb, w + pl + pr
        if out is None:
            out = torch.empty_like(bayer)
        cb = self.default_chunk(B, hp, wp)
        z = self._buf("z", (cb, hp, wp, 4), torch.float32, dev)
        y = self._buf("y", (cb, hp, wp, 4), torch.float32, dev)
        ub = self._buf("ub", (cb,), torch.float32, dev)
        st = stream_ptr()
        for b0 in range(0, B, cb):
            n = min(cb, B - b0)
            check(self.lib.yond_pack_pad(ptr(bayer[b0:b0 + n]), ptr(z[:n]), ptr(ub[:n]), n, H, W, pl, pr, pt, pb, st))
            self.net.forward_nhwc(z[:n], ub[:n], None, out=y[:n])
            check(self.lib.yond_crop_unpack(ptr(y[:n]), ptr(out[b0:b0 + n]), n, H, W, pl, pr, pt, pb, st))
        return out


class HostJob:
    """A batch submitted with iter_denoise_host(wait=False): .result() waits for its last download and reads the numbers."""

    def __init__(self, drv, results, out_done):
        self.drv, self.results, self.out_done = drv, results, out_done

    def result(self):
        self.out_done.synchronize()
        summaries = [self.drv.read_summary(r) for r in self.results]
        return {"regs": [s_[0] for s_ in summaries], "rounds": np.concatenate([s_[1] for s_ in summaries])}


class YOND_SIDD:
    """Drop-in for the reference driver's pipeline methods.  Construct from the yml dicts:

        drv = YOND_SIDD(arch=cfg['arch'], pipe=cfg['pipeline'], state_dict=torch.load(...))
        res = drv.IterDenoise(data, {'p': p, 'img_id': k})          # same dict in / dict out as the reference
    """

    def __init__(self, arch, pipe, state_dict=None, net=None, biaslut="default", device="cuda", chunk=None, log=None):
        self.arch = dict(arch)
        self.pipe = dict(pipe)
        if self.pipe.get("bias_corr") == "none":  # YOND_SIDD.py:164-165
            self.pipe["bias_corr"] = None
        self.device = torch.device(device)
        self.net = net if net is not None else build_net(self.arch, self.device)
        if state_dict is not None:
            archs.load_weights(self.net, state_dict, by_name=False)  # YOND_SIDD.py:183-185
        self.net.eval()
        if biaslut == "default":  # the reference enables the LUT iff checkpoints/bias_lut_2d.npy exists (:171)
            biaslut = isp.BiasLUT()
        self.biaslut = biaslut
        self.engine = YondEngine(self.net, self.arch, self.biaslut, chunk=chunk)
        self.logfile = None
        self._log = log or (lambda *a, **k: None)

    # -- helpers --------------------------------------------------------------------------------
    @staticmethod
    def _as_table(bias_func):
        """A reference-style `bias_func` (scipy interp1d from get_bias) or a (nodes, values) pair -> (nodes, values)."""
        if bias_func is None:
            return None
        if isinstance(bias_func, tuple):
            return bias_func
        return np.asarray(bias_func.x), np.asarray(bias_func.y)

    # -- YOND_SIDD.py:238-248 ---------------------------------------------------------------------
    def Simple_Denoiser(self, lr_raw, denoiser="unet", p=None, show=False):
        x, np_in = isp.to_dev(lr_raw)
        out = self.engine.simple_denoise(x[None])[0]
        return out.cpu().numpy() if np_in else out

    # -- YOND_SIDD.py:250-299 ---------------------------------------------------------------------
    def VST_Denoiser(self, lr_raw, hr_raw=None, bias_corr="pre", bias_func=None, denoiser="net", p=None, show=False):
        if denoiser in ("bm3d", "fbi"):
            raise NotImplementedError("bm3d / fbi comparison denoisers are outside the B200 hot path (SURVEY §2)")
        x, np_in = isp.to_dev(lr_raw)
        # bias: LUT when loaded and sigma/K in range, else the fallback table — the caller's `bias_func` when given
        # (only consulted without a LUT, :254-257), else get_bias up to this frame's max (:256 / isp_algos.py:204-212)
        fixed = self._as_table(bias_func) if self.biaslut is None else None
        out = self.engine.vst_denoise(x[None], [p["gain"]], [p["sigma"]], p["scale"], bias_corr=bias_corr,
                                      vst_type=self.pipe.get("vst_type", "exact"), clip01=False, fixed_table=fixed)[0]
        return out.cpu().numpy() if np_in else out

    # -- YOND_SIDD.py:301-483 ---------------------------------------------------------------------
    def IterDenoise(self, data, params):
        lr = data["lr"]
        p = params["p"]
        np_in = isinstance(lr, np.ndarray)
        blocks, _ = isp.to_dev(lr)
        full = None
        if data.get("lr_full") is not None:  # the reference loads data['lr_path_full'] from disk (:339-340)
            full, _ = isp.to_dev(data["lr_full"])
        early = {}

        def grab_round1(dn1):  # D2H of the round-1 result on a side stream as soon as it is complete
            ev = torch.cuda.Event()
            ev.record()
            side = getattr(self, "_down_stream", None)
            if side is None:
                side = self._down_stream = torch.cuda.Stream(self.device)
            side.wait_event(ev)
            with torch.cuda.stream(side):
                v = isp.pinned_view("round1", dn1[0])
                v.copy_(dn1[0], non_blocking=True)
                early["done"] = torch.cuda.Event()
                early["done"].record(side)
            dn1.record_stream(side)
            early["view"] = v

        def host_round1():  # runs while the GPU works on round 2: pinned -> fresh NumPy array
            early["done"].synchronize()
            out = np.empty(tuple(early["view"].shape), np.float32)
            isp._host_copy(out, early["view"].numpy())
            early["np"] = out

        np_pipe = np_in and self.pipe["full_est"] and "simple" in self.pipe["est_type"]
        res = self.iter_denoise_device(blocks, p, lr_full=full, after_round1=grab_round1 if np_pipe else None,
                                       before_summary=host_round1 if np_pipe else None)
        if np_in:  # NumPy in -> NumPy out like the reference; the mosaic of the input never leaves the host
            if "np" in early:
                dns = [early["np"]] + isp.to_host(res["raw_dns"][1:])
            else:
                dns = isp.to_host(res["raw_dns"])
            lr_raw = np.concatenate(list(lr), axis=-1) if lr.ndim == 3 else lr
        else:
            dns, lr_raw = list(res["raw_dns"]), res["lr_raw"]()
        results = {"raw_dns": dns, "regs": res["regs"], "lr_raw": lr_raw}
        hr = data.get("hr")
        results["hr_raw"] = (np.concatenate(list(hr), axis=-1) if isinstance(hr, np.ndarray) and hr.ndim == 3 else hr)
        return results

    # -- the blind N-round pipeline, device-resident and free of host synchronisation ----------------------------
    reuse_self_var = True  # collab estimate of plain frames starts from the self estimate's var map (one box pass less)

    def iter_denoise_dev(self, x, p, lr_full=None, timings=None, raw=None, after_round1=None):
        """IterDenoise (YOND_SIDD.py:301-483, `simple` estimator) for a batch of images: x (nimg, nblk, H, W) CUDA f32 —
        SIDD images of nblk blocks, or full frames with nblk = 1.  Every stage runs once for the whole batch; the noise
        estimate, the reference's guards, the VST constants, the bias rows and the per-round selection all stay on the device,
        so nothing is read back until the caller asks for the numbers.

        Rounds: round 1 (self estimate) and, with pipe['iter'] == 'iter', pipe['max_iter'] collab rounds (:419-472).  A batch
        always runs every round on the device: an image whose beta1 < 0 stopped the reference's loop is carried through the
        later rounds by selection (its output is a copy of its last live round's, its parameters are those of that round), so
        no round needs a read-back.

        Returns device tensors: dns / regs4 / live = per-round lists of the outputs (nimg, H, nblk*W) (the reference's mosaic
        layout), (nimg, 4) float64 = (beta1, beta2 after the guards, gain, sigma), and (nimg,) int32 = the image is still live
        after this round (all ones in round 1).  dn1 / regs1 = round 1, final = the last round, regs2 / ok = round 2 (None without
        collab rounds).

        raw = (black, white, ratio[, clip]): x is the uint16 SENSOR mosaic (16-bit integer tensor) and the dataset normalisation
        (raw - black) * ratio / (white - black) of the 14-bit drivers (data_process/yond_datasets.py:955-961, :1053-1056) is applied
        on load by the estimator and the VST front end — the float32 frame never exists (SURVEY 8(f)-1).

        Exposure per image: p['wp'], p['bl'], p['scale'] and each entry of raw are a scalar (every image) or one value per image
        (batch_exposure; ValueError before anything is launched), so a batch may mix white / black levels and ratios.  They reach the
        device in one small copy; scalars take the same path.

        lr_full: the full-resolution noisy frame of every image (the shipped SIDD configuration estimates round 1 on it, :338-341) —
        a sequence of nimg (H_i, W_i) CUDA float32 frames, of any even sizes, or one (nimg, H, W) tensor.  Round 1 is then one
        estimate_frames call for the whole batch; the fallback bias-table bound stays the maximum of each image's blocks (:393), and
        the collab rounds estimate on the blocks as without lr_full (:431).  ValueError before anything is launched for a wrong number
        of frames, a malformed frame (nlf.check_frames) or lr_full together with raw, which is not supported."""
        pipe = self.pipe
        n_collab = collab_rounds(pipe)
        if lr_full is not None and raw is not None:
            raise ValueError("lr_full takes float32 frames and is not supported together with raw= (uint16 sensor input)")
        if raw is not None:
            assert x.dtype in (torch.int16, torch.uint16)
        assert pipe["full_est"] and "simple" in pipe["est_type"]
        nimg, nblk, H, W = x.shape
        dev = x.device
        eng = self.engine
        k, bias_corr, vst_type = pipe["k"], pipe["bias_corr"], pipe.get("vst_type", "exact")
        full_dn = bool(pipe["full_dn"])
        scale_est, scale, raw_rec = batch_exposure(p, nimg, raw)
        if lr_full is not None:
            lr_full = nlf.check_frames(lr_full, nimg, k)
        # (scale_est, scale, bound) per image for round 1 and for the collab rounds.  The bound of a fallback bias table: full_dn
        # round 1 = the frame's max in DN of p['scale'] (:256); everything else lr_raw.max()*(wp-bl) (:393, :449)
        scales1 = np.stack([scale_est, scale, scale if full_dn else scale_est], 1)
        scales_c = np.stack([scale_est, scale, scale_est], 1)
        buf, offs = _upload([scales1, scales_c] + ([raw_rec] if raw is not None else []), dev)
        s1_dev = buf[offs[0]:offs[1]].view(torch.float64)
        sc_dev = buf[offs[1]:offs[1] + scales_c.nbytes].view(torch.float64)
        raw = buf[offs[2]:] if raw is not None else None
        est = nlf._estimator()

        def mark(name):  # optional stage timing (synchronising; for profiling only)
            if timings is not None:
                import time
                torch.cuda.synchronize()
                now = time.perf_counter()
                timings[name] = timings.get(name, 0.0) + (now - timings.get("_t", now))
                timings["_t"] = now
        mark("start")
        if full_dn and nblk > 1:  # one network pass over the whole mosaic (:387-389): make it a frame
            x = x.permute(0, 2, 1, 3).reshape(nimg, 1, H, nblk * W).contiguous()
            mos_blocks, W, nblk = nblk, nblk * W, 1
        else:
            mos_blocks = nblk
        # Geometry of the collab estimates.  The shipped driver hard-codes SIDD_256 = True (:431): the mosaic is cut into 32 strips
        # along W that the box filters treat as separate images.  That is the SIDD layout; for plain frames (the drivers of the
        # other datasets are not in the repository) the default here is one image, `sidd_256: True` in the pipeline dict restores
        # the hard-coded behaviour (needs W % 64 == 0).
        sidd = bool(pipe.get("sidd_256", mos_blocks == 32))
        if n_collab and sidd and nblk == 1:  # a frame (or a full_dn mosaic): the 32 strips are split out of the mosaic layout
            assert W % 64 == 0, "SIDD_256 splits the packed frame into 32 strips along W (YOND_SIDD.py:91-93)"
            cx, cnb, c_mosaic = x.reshape(nimg, H, W), 32, True
        else:
            cx, cnb, c_mosaic = x, nblk, False
        # stdfilt(lr, k)**2 in the collab geometry, shared by every collab round: the self estimate's var map when it ran in the same
        # geometry (not SIDD_256, not on lr_full), else one box pass over lr in round 2
        reuse = n_collab > 0 and not sidd and lr_full is None and self.reuse_self_var
        lr_var = None
        if n_collab:
            n_el = est.collab_geometry(nimg, cnb, H, W // cnb if c_mosaic else W, sidd)
            lr_var = eng._buf("lr_var", (n_el,), torch.float32, dev)
        need_max = bias_corr == "pre"
        seg_max = torch.empty(nimg, device=dev, dtype=torch.float32) if need_max else None
        # ---- round 1: self-calibration on the mosaic (:315, :338-341) or on the full-resolution frame when given
        if lr_full is None:
            regs = est.estimate_dev(x, None, k, split_blocks=False, seg_max=seg_max, raw=raw, var_map=lr_var if reuse else None)
        else:
            regs = est.estimate_frames(lr_full, k)
            if need_max:  # the bound is the maximum of the image's blocks, not of its full frame (:393)
                check(eng.lib.yond_seg_max(ptr(x), x[0].numel(), nimg, ptr(seg_max), stream_ptr()))
        mark("estimate_self")
        ch = eng.chain_params(regs, seg_max, nimg, nblk, *scales1.T, 1, bias_corr, vst_type, scales_dev=s1_dev)
        frames = x.reshape(nimg * nblk, H, W)
        out = torch.empty((nimg, H, nblk * W), device=dev, dtype=torch.float32)
        eng.vst_denoise_dev(frames, ch, out, frames_per_row=nblk, fps=nblk, raw=raw)
        mark("denoise_round1")
        if after_round1 is not None:  # round 1 is enqueued: a caller may start downloading it under the collab rounds
            after_round1(out)
        dns, regs4, live = [out], [ch["regs4"]], [ch["ok"]]
        # ---- rounds 2 .. max_iter + 1: collab estimate on (lr, previous output) (:431), guards, VST denoise, selection (:445-447)
        for r in range(2, n_collab + 2):
            if r == 2 and not reuse:
                est.lr_var_dev(cx, lr_var, k, split_blocks=sidd, x_mosaic=c_mosaic, nblk=cnb, raw=raw)
            regs = est.estimate_collab_cached(out, lr_var, cnb, k, split_blocks=sidd, y_mosaic=True)
            mark("estimate_collab")
            ch = eng.chain_params(regs, seg_max, nimg, nblk, *scales_c.T, r, bias_corr, vst_type, prev=ch, scales_dev=sc_dev)
            prev_out, out = out, torch.empty_like(out)
            eng.vst_denoise_dev(frames, ch, out, frames_per_row=nblk, fps=nblk, select=True, fallback=prev_out, raw=raw)
            mark(f"denoise_round{r}")
            dns.append(out)
            regs4.append(ch["regs4"])
            live.append(ch["ok"])
        two = len(dns) > 1
        return {"dns": dns, "regs4": regs4, "live": live, "dn1": dns[0], "final": dns[-1], "regs1": regs4[0],
                "regs2": regs4[1] if two else None, "ok": live[1] if two else None, "lr": x, "nblk": nblk}

    @staticmethod
    def summary_async(res):
        """Enqueues (on the current stream) the download of a batch's numbers into pinned host memory; read_summary then
        needs no device synchronisation of its own beyond the event the caller waits for."""
        host = {}
        for key in ("regs4", "live"):
            host[key] = []
            for t in res[key]:
                h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
                h.copy_(t, non_blocking=True)
                host[key].append(h)
        res["host"] = host

    @staticmethod
    def host_numbers(res):
        """The per-round (nimg,4) regs4 and (nimg,) live arrays of a batch as NumPy: from the pinned copies of summary_async, else
        read back (one small copy per round and list)."""
        host = res.get("host")
        src = host if host is not None else res
        return [t.cpu().numpy() for t in src["regs4"]], [t.cpu().numpy().astype(bool) for t in src["live"]]

    @staticmethod
    def read_summary(res):
        """One read-back of the numbers of a finished batch: regs per round as (nimg,2) float64 arrays (rows of images that did
        not complete a round are NaN in it — the reference does not append them, :445-447), rounds per image (1 + the live
        collab rounds), and (gain, sigma) per round as (nimg,2) arrays (not masked: the values the estimate gave)."""
        r4, live = YOND_SIDD.host_numbers(res)
        nimg = r4[0].shape[0]
        regs = [r4[0][:, :2].copy()]
        gains = [r4[0][:, 2:].copy()]
        rounds = np.ones(nimg, np.int64)
        for r in range(1, len(r4)):
            reg = r4[r][:, :2].copy()
            reg[~live[r]] = np.nan
            regs.append(reg)
            gains.append(r4[r][:, 2:].copy())
            rounds += live[r]
        return regs, rounds, gains

    def iter_denoise_batch(self, blocks, p, log=None, timings=None, raw=None, lr_full=None):
        """IterDenoise for a BATCH of SIDD-shaped images (or full frames, nblk = 1) at once: blocks (nimg, nblk, H, W) CUDA
        f32.  Same per-image algorithm and guards as the reference (YOND_SIDD.py:301-483); every device stage runs once for
        all images and the host reads back ONE small array at the end.
        Returns {'raw_dns': [(nimg,H,nblk*W) per round, max_iter + 1 of them], 'regs': [(nimg,2) per round; NaN rows in the
        rounds an image did not complete (a beta1 < 0 guard kept its previous result)], 'rounds': (nimg,) number of denoise rounds
        each image completed}.  An image's entries of raw_dns beyond its rounds repeat its last completed round.
        lr_full (optional): the full-resolution frame of every image, sizes may differ (iter_denoise_dev): round 1 estimates on them."""
        res = self.iter_denoise_dev(blocks, p, timings=timings, raw=raw, lr_full=lr_full)
        regs, rounds, _ = self.read_summary(res)
        return {"raw_dns": list(res["dns"]), "regs": regs, "rounds": rounds, "lr_raw": None, "dev": res}

    # -- full frames of different sizes in one batch ---------------------------------------------------------------------
    def _check_frames_call(self, frames, p, raw):
        """The ValueErrors of iter_denoise_frames_dev, all raised before anything is enqueued."""
        pipe = self.pipe
        if pipe.get("sidd_256"):
            raise ValueError("iter_denoise_frames: pipe['sidd_256'] cuts blocks of a SIDD mosaic into strips; full frames of different sizes "
                             "are one image each (set sidd_256 False)")
        if not pipe["full_est"] or "simple" not in pipe["est_type"]:
            raise ValueError(f"iter_denoise_frames: the blind pipeline needs full_est and a 'simple' est_type, got full_est="
                             f"{pipe['full_est']!r}, est_type={pipe['est_type']!r}")
        n_collab = collab_rounds(pipe)
        if isinstance(frames, torch.Tensor):
            raise ValueError("iter_denoise_frames: a list of (H, W) frames expected (a stacked tensor goes to iter_denoise_batch)")
        frames = list(frames)
        if len(frames) > 65535:
            raise ValueError(f"iter_denoise_frames: at most 65535 frames per call, got {len(frames)}")
        exposure = batch_exposure(p, len(frames), raw)
        frames = nlf.check_frames(frames, None, pipe["k"], raw=raw is not None)
        return frames, n_collab, exposure

    def iter_denoise_frames_dev(self, frames, p, raw=None):
        """IterDenoise (YOND_SIDD.py:301-483, `simple` estimator) for a batch of full frames of any even sizes: each image is its frame,
        as in iter_denoise_dev with nblk = 1, and gets exactly what iter_denoise_dev gives on that frame alone.  No host synchronisation
        between the first and the last kernel; every round, liveness and selection of stopped images as in iter_denoise_dev.
        frames: a list of (H_i, W_i) CUDA tensors, float32 Bayer frames, or with raw = (black, white, ratio[, clip]) int16 / uint16 sensor
        mosaics normalised on load.  p['wp'], p['bl'], p['scale'] and the entries of raw: a scalar or one value per frame (caller order).
        ValueError before anything is enqueued for a malformed or misaligned frame (nlf.check_frames), a mix of dtypes, 16-bit frames
        without raw= or float32 frames with it, pipe['sidd_256'], a pipeline without full_est / a 'simple' est_type, the exposure errors
        of batch_exposure and more than 65535 frames.

        The frames are ordered on the host by padded size (then H, W; ties keep the caller's order), so that every size is a contiguous
        range of the DEVICE ORDER: res['order'][j] is the caller index of device row j.  The estimator and the parameter chain run once
        per round for all frames; the VST front end, the network and the inverse run once per size (and chunk).  No frame is copied: the
        kernels read each one where it lies, so the caller keeps them unchanged until the work is done.
        Returns dns / regs4 / live = per-round lists like iter_denoise_dev: dns[r][i] is caller frame i's (H_i, W_i) output (the outputs of
        a round are views into one flat buffer, res['flat'][r], in device order), regs4[r] (nimg, 4) float64 and live[r] (nimg,) int32
        rows are in DEVICE order."""
        frames, n_collab, (scale_est, scale, raw_rec) = self._check_frames_call(frames, p, raw)
        pipe, eng, est = self.pipe, self.engine, nlf._estimator()
        nimg, dev = len(frames), frames[0].device
        k, bias_corr, vst_type = pipe["k"], pipe["bias_corr"], pipe.get("vst_type", "exact")
        full_dn = bool(pipe["full_dn"])
        pads = [isp.get_p2d((1, 4, f.shape[0] // 2, f.shape[1] // 2), base=32) for f in frames]
        key = [(f.shape[0] // 2 + pd[2] + pd[3], f.shape[1] // 2 + pd[0] + pd[1], f.shape[0], f.shape[1]) for f, pd in zip(frames, pads)]
        order = np.asarray(sorted(range(nimg), key=lambda i: key[i]), np.int64)  # stable: equal sizes keep the caller's order
        groups = []  # (first, end, H, W) ranges of the device order
        for j, i in enumerate(order):
            if j and key[order[j - 1]] == key[i]:
                groups[-1][1] = j + 1
            else:
                groups.append([j, j + 1, frames[i].shape[0], frames[i].shape[1]])
        # (scale_est, scale, bound) per image for round 1 and the collab rounds, as iter_denoise_dev for nblk = 1 (:256, :393, :449)
        scales1 = np.stack([scale_est, scale, scale if full_dn else scale_est], 1)[order]
        scales_c = np.stack([scale_est, scale, scale_est], 1)[order]
        table = nlf.FrameTable([frames[i] for i in order], [scales1, scales_c] + ([raw_rec[order]] if raw is not None else []))
        s1_dev, sc_dev = (v.view(torch.float64) for v in table.extra[:2])
        raw_dev = table.extra[2] if raw is not None else None
        off = table.off.astype(np.int64)
        # round 1: one self estimate of every frame; its var map is stdfilt(lr, k)**2 of the collab rounds, its first pass gives seg_max
        lr_var = eng._buf("lr_var", (table.n_el,), torch.float32, dev) if n_collab else None
        seg_max = torch.empty(nimg, device=dev, dtype=torch.float32) if bias_corr == "pre" else None
        regs = est.estimate_frames(table, k, var_map=lr_var, seg_max=seg_max, raw=raw_dev)
        ch = eng.chain_params(regs, seg_max, nimg, 1, *scales1.T, 1, bias_corr, vst_type, scales_dev=s1_dev)
        psz = C.sizeof(VstParams)

        def denoise(ch, out, fallback=None):
            for g0, g1, H, W in groups:
                sl = slice(int(off[g0]), int(off[g1]))
                part = {key_: ch[key_] for key_ in ("rows", "xnodes", "stride")}
                part.update(params=ch["params"][g0 * psz:], t=ch["t"][g0:], ok=ch["ok"][g0:])
                eng.vst_denoise_dev(table.records_from(g0), part, out[sl].view(g1 - g0, H, W), select=fallback is not None,
                                    fallback=None if fallback is None else fallback[sl], raw=None if raw_dev is None else raw_dev[g0 * RAW_REC.itemsize:],
                                    shape=(g1 - g0, H, W))
            return out

        out = denoise(ch, torch.empty(table.n_el, device=dev, dtype=torch.float32))
        flat, regs4, live = [out], [ch["regs4"]], [ch["ok"]]
        # rounds 2 .. max_iter + 1: one collab estimate of every frame against the cached var map, the chain with prev=, selection
        for r in range(2, n_collab + 2):
            regs = est.estimate_collab_frames(out, table, lr_var, k)
            ch = eng.chain_params(regs, seg_max, nimg, 1, *scales_c.T, r, bias_corr, vst_type, prev=ch, scales_dev=sc_dev)
            out = denoise(ch, torch.empty_like(out), fallback=out)
            flat.append(out)
            regs4.append(ch["regs4"])
            live.append(ch["ok"])
        pos = np.empty(nimg, np.int64)
        pos[order] = np.arange(nimg)  # device row of caller frame i
        dns = [[o[int(off[pos[i]]):int(off[pos[i] + 1])].view(frames[i].shape) for i in range(nimg)] for o in flat]
        return {"dns": dns, "regs4": regs4, "live": live, "flat": flat, "order": order, "table": table}

    def iter_denoise_frames(self, frames, p, raw=None):
        """IterDenoise for a batch of full frames of any even sizes in one call (iter_denoise_frames_dev), float32 or, with raw=, 16-bit
        sensor mosaics.  Returns {'raw_dns': [[caller frame i's (H_i, W_i) output] per round, max_iter + 1 of them], 'regs': [(nimg, 2) per
        round, NaN rows in the rounds an image did not complete], 'rounds': (nimg,)}, everything in the caller's order, after one
        read-back at the end (read_summary)."""
        res = self.iter_denoise_frames_dev(frames, p, raw=raw)
        regs, rounds, _ = self.read_summary(res)
        pos = np.argsort(res["order"])
        return {"raw_dns": res["dns"], "regs": [r[pos] for r in regs], "rounds": rounds[pos], "dev": res}

    def iter_denoise_host(self, host_in, host_out, p, group=8, lanes=1, wait=True, raw=None):
        """End-to-end batched IterDenoise on HOST buffers: host_in (nimg,nblk,H,W) f32 pinned -> host_out (nimg,H,nblk*W) f32
        pinned (final round of every image; full frames are nblk = 1).  Images are processed in groups of `group`.

        One host thread, three streams: the H2D copy of group g+1 and the D2H copy of group g-1 run on their own streams
        while group g computes (a ring of three device staging buffers, event-ordered).  Because the pipeline itself never
        waits for the device (iter_denoise_dev), the host only enqueues; the per-image numbers are read back once, at the
        end.  wait=False returns a job whose .result() does that read-back: a caller streaming batch after batch submits
        the next batch first, so its first upload runs under the tail of this one (bench.py's e2e keeps two in flight).
        `lanes` is accepted for compatibility and ignored (round 1 needed host threads to hide the estimator's read-backs).
        raw = (black, white, ratio[, clip]): host_in holds uint16 sensor mosaics (int16 / uint16 tensor, half the H2D bytes), see
        iter_denoise_dev.  Per-image values of p / raw (one per image of host_in) are sliced for each group."""
        assert host_in.is_pinned() and host_out.is_pinned(), "pinned host buffers required for asynchronous copies"
        nimg = host_in.shape[0]
        batch_exposure(p, nimg, raw)  # malformed values raise before the first copy
        part = lambda v, a, b: v[a:b] if np.ndim(v) == 1 else v
        dev = self.device
        cur = torch.cuda.current_stream(dev)
        sizes = [min(group, nimg - a) for a in range(0, nimg, group)] if isinstance(group, int) else [int(g) for g in group]
        assert sum(sizes) == nimg and min(sizes) > 0, "group sizes must add up to the number of images"
        gmax = max(sizes)
        key = (tuple(host_in.shape[1:]), gmax, host_in.dtype)
        io = getattr(self, "_io", None)
        if io is None or io["key"] != key:
            torch.cuda.synchronize(dev)
            io = self._io = dict(key=key, s_in=torch.cuda.Stream(dev), s_out=torch.cuda.Stream(dev), seq=0,
                                 ring=[dict(buf=torch.empty((gmax,) + tuple(host_in.shape[1:]), device=dev, dtype=host_in.dtype), free=None) for _ in range(3)])
        s_in, s_out, ring = io["s_in"], io["s_out"], io["ring"]
        starts = np.concatenate([[0], np.cumsum(sizes)])
        groups = [(int(starts[i]), int(starts[i + 1])) for i in range(len(sizes))]
        seq0 = io["seq"]
        io["seq"] += len(groups)
        in_ready = {}

        def stage_in(g):
            a, b = groups[g]
            slot = ring[(seq0 + g) % 3]
            if slot["free"] is not None:
                s_in.wait_event(slot["free"])  # the staging buffer is free once the group that used it has been consumed
            with torch.cuda.stream(s_in):
                slot["buf"][:b - a].copy_(host_in[a:b], non_blocking=True)
                in_ready[g] = torch.cuda.Event()
                in_ready[g].record(s_in)

        results = []
        stage_in(0)
        for g, (a, b) in enumerate(groups):
            if g + 1 < len(groups):
                stage_in(g + 1)
            slot = ring[(seq0 + g) % 3]
            cur.wait_event(in_ready[g])
            pg = {key: part(v, a, b) if key in ("wp", "bl", "scale") else v for key, v in p.items()}
            res = self.iter_denoise_dev(slot["buf"][:b - a], pg, raw=None if raw is None else tuple(part(v, a, b) for v in raw))
            done = torch.cuda.Event()
            done.record(cur)
            slot["free"] = done
            s_out.wait_event(done)
            with torch.cuda.stream(s_out):
                host_out[a:b].copy_(res["final"], non_blocking=True)
                self.summary_async(res)
            res["final"].record_stream(s_out)
            for t in res["regs4"] + res["live"]:
                t.record_stream(s_out)
            res.pop("lr", None)  # a view of the staging buffer, which is reused
            res.pop("dns", None)  # only the final round is downloaded: the intermediate rounds' frames are released
            results.append(res)
        out_done = torch.cuda.Event()
        out_done.record(s_out)
        job = HostJob(self, results, out_done)
        return job.result() if wait else job

    def iter_denoise_device(self, blocks, p, lr_full=None, after_round1=None, before_summary=None):
        """Device-resident IterDenoise.  `blocks`: (nblk,H,W) CUDA f32 (SIDD layout) or (H,W) frame.
        Returns CUDA tensors in the reference's mosaic layout: (H, nblk*W)."""
        pipe = self.pipe
        p = p  # updated in place like the reference (p['gain'], p['sigma'])
        single = blocks.dim() == 2
        blk = blocks[None] if single else blocks
        nblk, H, W = blk.shape
        mosaic = lambda: (blk[0] if nblk == 1 else blk.permute(1, 0, 2).reshape(H, nblk * W).contiguous())  # :315
        if not pipe["full_est"]:
            # :367-378 — no estimator configured: plain network pass per block, returned as-is (not clipped)
            dn = self.engine.simple_denoise(blk)
            dn = dn[0] if nblk == 1 else dn.permute(1, 0, 2).reshape(H, nblk * W)
            return {"raw_dns": [dn], "regs": (0, 0), "lr_raw": mosaic}
        if "simple" not in pipe["est_type"]:
            raise NotImplementedError(f"est_type '{pipe['est_type']}' needs external estimate files / networks (YOND_SIDD.py:316-353)")
        res = self.iter_denoise_dev(blk[None].contiguous(), p, lr_full=None if lr_full is None else [lr_full], after_round1=after_round1)
        if before_summary is not None:  # everything is enqueued; host work placed here overlaps the collab rounds
            before_summary()
        r4, live = self.host_numbers(res)
        b1, b2, g, s_ = r4[0][0]
        self._log(f"Self Est: K={g:.4f}, b={s_:.4f} (beta1={b1:.3e}, beta2={b2:.3e})")
        p["gain"], p["sigma"] = g, s_  # :356
        raw_dns, out_regs = [res["dns"][0][0]], [r4[0][0, :2].copy()]
        # the rounds the reference evaluates: every live collab round and the first one that fails the beta1 guard
        for r in range(1, len(r4)):
            b1, b2, g, s_ = r4[r][0]
            p["gain"], p["sigma"] = g, s_  # :442 — set before the guard, like the reference
            self._log(f"Iter {r} Est: K={g:.4f}, sigma={s_:.4f} (beta1={b1:.3e}, beta2={b2:.3e})")
            if not live[r][0]:
                self._log("Warning!!! Wrong noise level! Backup to iter_0 result.")  # :445-447
                break
            raw_dns.append(res["dns"][r][0])
            out_regs.append(r4[r][0, :2].copy())
        return {"raw_dns": raw_dns, "regs": out_regs, "lr_raw": mosaic}  # lr_raw: a thunk (the mosaic copy is only made on request)


def collab_rounds(pipe):
    """Number of collab rounds IterDenoise runs after round 1 (YOND_SIDD.py:419-472): pipe['max_iter'] with pipe['iter'] == 'iter',
    else 0.  max_iter must be an integer >= 0 (ValueError otherwise)."""
    if pipe.get("iter") != "iter":
        return 0
    n = pipe.get("max_iter")
    if isinstance(n, (bool, np.bool_)) or not isinstance(n, (int, np.integer)) or n < 0:
        raise ValueError(f"pipeline max_iter must be an integer >= 0, got {n!r}")
    return int(n)
