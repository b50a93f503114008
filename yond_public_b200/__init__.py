"""yond_public_b200 — B200-native (sm_100a) implementation of YOND's per-image blind raw denoising path.

Same plugin surface as the reference (fenghansen/YOND_public): the function names of utils/isp_ops.py /
utils/isp_algos.py / YOND_SIDD.py, the yml-configured arch classes, and the driver's pipeline methods.
All per-pixel work runs in hand-written CUDA kernels behind the C-ABI of include/yond_b200.h
(libyond_b200.so, bound with ctypes in _lib.py).  There is no CPU fallback.
"""
from . import _lib, isp  # noqa: F401
from .archs import GuidedResUnet, GuidedSelfUnet, ResUnet2, SelfResUNet, SNRnet, UNetSeeInDark, initialize_weights, load_weights  # noqa: F401
from .isp import (VST, BiasLUT, bayer2rggb, bayer2rggbs, blur, get_bias_points, get_bias_table, get_p2d, inverse_VST,  # noqa: F401
                  normalize_raw, pack_raw_bayer, rggb2bayer, rggb2bayers, rot_bayer, stdfilt)
from .metrics import block_metrics, block_metrics_rgb8, calculate_ssim, compare_psnr, sidd_eval_batch, sidd_eval_image, sidd_image_metrics, sidd_rgb_metrics  # noqa: F401
from .render import demosaic_ea, process_sidd_image  # noqa: F401
from .nlf import CollabNLF, SelfNLF, SimpleNLF  # noqa: F401
from .pipeline import YOND_SIDD, YondEngine, build_net  # noqa: F401

__all__ = ["UNetSeeInDark", "GuidedResUnet", "SNRnet", "ResUnet2", "SelfResUNet", "GuidedSelfUnet", "initialize_weights", "load_weights", "bayer2rggb", "rggb2bayer",
           "bayer2rggbs", "rggb2bayers", "VST", "inverse_VST", "BiasLUT", "stdfilt", "blur", "get_p2d", "get_bias_table", "get_bias_points",
           "pack_raw_bayer", "normalize_raw", "rot_bayer", "compare_psnr", "calculate_ssim", "block_metrics", "block_metrics_rgb8", "sidd_image_metrics", "sidd_rgb_metrics", "sidd_eval_image", "sidd_eval_batch", "process_sidd_image", "demosaic_ea", "SimpleNLF", "SelfNLF", "CollabNLF", "YOND_SIDD", "YondEngine", "build_net"]
