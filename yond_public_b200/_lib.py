"""ctypes binding of libyond_b200.so (the C-ABI in include/yond_b200.h).

This is the reference-side stub a YOND maintainer would add (INTEGRATION.md): the reference is pure
Python, so its FFI is ctypes.  There is NO fallback: if the CUDA library is missing or a call fails, an
exception is raised — the product path never routes through a CPU implementation.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libyond_b200.so")


class YondError(RuntimeError):
    pass


class VstParams(C.Structure):
    """yond_vst_params (include/yond_b200.h)."""
    _fields_ = [("gain", C.c_float), ("sigma", C.c_float), ("scale", C.c_float), ("lower", C.c_float),
                ("upper", C.c_float), ("lut_row", C.c_int32), ("table_n", C.c_int32), ("exact_inverse", C.c_int32)]


class RawNorm(C.Structure):
    """yond_raw_norm (include/yond_b200.h): (float32(raw) - black) * ratio / (white - black), optional clip to [0,1]."""
    _fields_ = [("black", C.c_float), ("white", C.c_float), ("ratio", C.c_float), ("clip", C.c_int)]


_P, _I, _SZ, _D, _U64 = C.c_void_p, C.c_int, C.c_size_t, C.c_double, C.c_uint64

# name -> (restype, argtypes); every symbol include/yond_b200.h declares
SIGNATURES = {
    "yond_last_error": (C.c_char_p, []),
    "yond_version": (_I, []),
    "yond_launch_count": (_U64, []),
    "yond_prof_enable": (_I, [_I]),
    "yond_prof_read": (_I, [C.c_char_p, _SZ, _I]),
    "yond_pack": (_I, [_P, _P, _I, _I, _I, _P]),
    "yond_unpack": (_I, [_P, _P, _I, _I, _I, _P]),
    "yond_rot90": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "yond_pack_raw": (_I, [_P, _P, _I, _I, _I, C.POINTER(C.c_int), C.POINTER(C.c_float), C.c_float, _I, _I, _P]),
    "yond_ingest_mosaic": (_I, [_P, _P, _SZ, C.c_float, C.c_float, C.c_float, _I, _P]),
    "yond_block_metrics": (_I, [_P, _P, _I, _I, _I, _I, _D, C.c_float, C.POINTER(C.c_double), _P, _P, _P]),
    "yond_block_metrics_rgb8": (_I, [_P, _P, _I, _I, _I, _I, C.POINTER(C.c_double), _P, _P, _P]),
    "yond_render_srgb": (_I, [_P, _P, _I, _I, _I, _I, _I, C.POINTER(C.c_double), C.POINTER(C.c_double), _P]),
    "yond_demosaic_ea": (_I, [_P, _P, _I, _I, _I, _P]),
    "yond_render_srgb_cams": (_I, [_P, _P, _P, _I, _I, _I, _P]),
    "yond_sidd_scores": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _P, _P]),
    "yond_vst": (_I, [_P, _P, _SZ, _D, _D, _P]),
    "yond_inverse_vst": (_I, [_P, _P, _SZ, _D, _D, _I, _P]),
    "yond_lut_row": (_I, [_P, _I, _I, _D, _P, _P]),
    "yond_lut_apply": (_I, [_P, _P, _SZ, _P, _P, _I, _D, _D, _P]),
    "yond_table_apply": (_I, [_P, _P, _SZ, _P, _P, _I, _P]),
    "yond_vst_fwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _I, _P]),
    "yond_vst_fwd_raw16": (_I, [_P, C.POINTER(RawNorm), _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _I, _P, _P, _I]),
    "yond_vst_inv": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _I, _P]),
    "yond_pack_pad": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "yond_crop_unpack": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "yond_box_blur": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _P, _P]),
    "yond_nlf_work_bytes": (_SZ, [_I, _I, _I, _I]),
    "yond_nlf_maps": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _P]),
    "yond_nlf_maps_bayer": (_I, [_P, _I, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P]),
    "yond_nlf_maps_raw16": (_I, [_P, C.POINTER(RawNorm), _I, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P]),
    "yond_nlf_maps_raw16_per_image": (_I, [_P, _P, _I, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P]),
    "yond_nlf_maps_collab_cached": (_I, [_P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "yond_nlf_fit_work_bytes": (_SZ, [_I]),
    "yond_nlf_fit": (_I, [_P, _P, _P, _SZ, _I, C.POINTER(_D), _I, _P, _P, _P, _P]),
    "yond_nlf_maps_frames": (_I, [_P, _I, _I, _I, _P, _P, _P, _I, _P, _P]),
    "yond_nlf_fit_ragged_work_bytes": (_SZ, [_I]),
    "yond_nlf_fit_ragged": (_I, [_P, _P, _P, _P, _SZ, _I, C.POINTER(_D), _I, _P, _P, _P, _P]),
    "yond_seg_max": (_I, [_P, _SZ, _I, _P, _P]),
    "yond_nlf_maps_frames_max": (_I, [_P, _I, _I, _I, _P, _P, _P, _I, _P, _P, _P]),
    "yond_nlf_maps_frames_raw16": (_I, [_P, _P, _I, _I, _I, _P, _P, _P, _I, _P, _P, _P]),
    "yond_nlf_maps_frames_collab_cached": (_I, [_P, _P, _I, _I, _I, _P, _P, _P, _P, _I, _P]),
    "yond_vst_fwd_frames": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _I, _P]),
    "yond_chain_work_bytes": (_SZ, [_I]),
    "yond_bias_table_nodes": (_I, [C.c_float]),
    "yond_vst_params_fill": (_I, [_P, _P, _I, _I, _D, _D, _D, _I, _I, _I, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P]),
    "yond_bias_table": (_I, [_D, _D, C.c_float, _P, _P, _I, _P, _P, _P]),
    "yond_bias_points": (_I, [_P, _I, _D, _D, _I, _P, _P, _P]),
    "yond_vst_inv_place": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _I, _I, _I, _P, _I, _P, _P]),
    "yond_net_create": (_I, [_I, _I, _I, _I, _I, _I, C.POINTER(_P)]),
    "yond_net_destroy": (None, [_P]),
    "yond_net_set_tensor": (_I, [_P, C.c_char_p, _P, C.POINTER(C.c_int64), _I]),
    "yond_net_num_keys": (_I, [_P]),
    "yond_net_key": (C.c_char_p, [_P, _I]),
    "yond_net_key_shape": (_I, [_P, _I, C.POINTER(C.c_int64)]),
    "yond_net_missing": (_I, [_P, C.c_char_p, _SZ]),
    "yond_net_workspace_bytes": (_SZ, [_P, _I, _I, _I]),
    "yond_net_forward": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _P, _SZ, _P]),
    "yond_net_forward_nchw": (_I, [_P, _P, _P, _P, _I, _I, _I, _P, _SZ, _P]),
    "yond_net_flops": (_D, [_P, _I, _I, _I]),
    "yond_net_set_conv_impl": (_I, [_P, _I]),
    "yond_net_profile": (_I, [_P, _I]),
    "yond_net_profile_read": (_I, [_P, C.POINTER(_D), C.POINTER(_D), C.POINTER(_I), _I]),
    "yond_conv2d": (_I, [_I, _I, _I, _I, _I, _I, _I, _P, _P, _I, _P, _P, _P, _P, _I, C.c_float, _P, _P, _P, _P]),
    "yond_tile_extract": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "yond_tile_insert": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
}

_lib = None


def load():
    """Loads the library (building nothing: run `python -m yond_public_b200.build` / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise YondError(f"{LIB_PATH} not found — build it with `python -m yond_public_b200.build` "
                        "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise YondError(f"libyond_b200 error {rc}: {load().yond_last_error().decode(errors='replace')}")


def ptr(t):
    """Device pointer of a torch tensor (must be contiguous) or None."""
    if t is None:
        return None
    assert t.is_contiguous(), "libyond_b200 takes contiguous buffers"
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def prof_enable(on=True):
    check(load().yond_prof_enable(int(bool(on))))


def prof_read(reset=True):
    """{stage: {scopes, ms, bytes, flops}} accumulated by the library's live stage profiler."""
    import json
    buf = C.create_string_buffer(1 << 16)
    check(load().yond_prof_read(buf, len(buf), int(bool(reset))))
    return json.loads(buf.value.decode())


def launch_count():
    return int(load().yond_launch_count())
