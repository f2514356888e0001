"""ctypes binding of librnc.so (include/rnc.h).  No torch types cross this boundary: callers pass
``tensor.data_ptr()`` integers, plain ints and the raw ``cudaStream_t``.

The library is REQUIRED on the product path: ``lib()`` raises ``RncUnavailable`` if it cannot be loaded —
there is no CPU or PyTorch fallback for the hot path.
"""
import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RNC_LIB") or os.path.join(_HERE, "librnc.so")      # RNC_LIB: developer override (variant builds)
ABI_VERSION = 11
CONV_NO_HALO, CONV_BASE_OFFSET, CONV_SPLIT_N, CONV_NO_PAIR, CONV_AUX_BLOCKED, CONV_OUT_BLOCKED, CONV_TF32, CONV_WINDOW = 1, 2, 4, 8, 16, 32, 64, 128   # rnc_conv_umma_desc.flags

(EPI_LINEAR, EPI_RELU, EPI_SIGMOID, EPI_GRU_ZR, EPI_GRU_Q, EPI_RELU_FLOW, EPI_RELU_ADD_RELU, EPI_TANH_RELU,
 EPI_FLOW_DELTA) = range(9)
CONV_NO_HALO, CONV_BASE_OFFSET = 1, 2

_vp, _i, _f = C.c_void_p, C.c_int, C.c_float


class RncUnavailable(RuntimeError):
    pass


class RncError(RuntimeError):
    pass


class ConvDesc(C.Structure):
    """Mirror of rnc_conv_desc (include/rnc.h)."""
    _fields_ = [("in0", _vp), ("c0", _i), ("ld0", _i),
                ("in1", _vp), ("c1", _i), ("ld1", _i),
                ("weight", _vp), ("bias", _vp),
                ("out", _vp), ("ldo", _i),
                ("h", _vp), ("ldh", _i),
                ("aux0", _vp), ("ldaux", _i),
                ("B", _i), ("H", _i), ("W", _i),
                ("cout", _i), ("kh", _i), ("kw", _i), ("epilogue", _i)]


class UmmaConvDesc(C.Structure):
    """Mirror of rnc_conv_umma_desc (include/rnc.h)."""
    _fields_ = [("in0_hi", _vp), ("in0_lo", _vp), ("c0", _i), ("ld0", _i),
                ("in1_hi", _vp), ("in1_lo", _vp), ("c1", _i), ("ld1", _i),
                ("w_hi", _vp), ("w_lo", _vp), ("ktot", _i), ("coutpad", _i),
                ("bias", _vp), ("unscale", _f),
                ("out_f32", _vp), ("ldo_f32", _i),
                ("out_hi", _vp), ("out_lo", _vp), ("ldo_split", _i),
                ("h", _vp), ("ldh", _i),
                ("aux0", _vp), ("ldaux", _i),
                ("B", _i), ("H", _i), ("W", _i),
                ("cout", _i), ("kh", _i), ("kw", _i), ("epilogue", _i),
                ("stride", _i), ("hin", _i), ("win", _i),
                ("res", _vp), ("ldres", _i), ("flags", _i), ("stats", _vp), ("add", _vp), ("ldadd", _i), ("win_pitch", _i)]


# name -> (restype, argtypes); every symbol include/rnc.h declares
SIGNATURES = {
    "rnc_abi_version": (_i, []),
    "rnc_build_info": (C.c_char_p, []),
    "rnc_status_string": (C.c_char_p, [_i]),
    "rnc_last_cuda_error": (_i, []),
    "rnc_launch_count": (C.c_longlong, []),
    "rnc_launch_count_reset": (None, []),
    "rnc_pyramid_offset": (C.c_size_t, [_i, _i, _i, _i, _i]),
    "rnc_fmap_prepare": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "rnc_corr_lookup_fwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _i, _i, _vp]),
    "rnc_corr_lookup_split_fwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp]),
    "rnc_corr_lookup_umma_workspace_bytes": (C.c_size_t, [_i, _i, _i]),
    "rnc_corr_lookup_umma_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, C.c_size_t, _vp]),
    "rnc_f32_to_f16": (_i, [_vp, _vp, C.c_size_t, _vp]),
    "rnc_conv2d_cl_fwd": (_i, [C.POINTER(ConvDesc), _vp]),
    "rnc_conv_umma_tiles": (C.c_longlong, [_i, _i, _i, _i, _i, _i, _i]),
    "rnc_conv2d_umma_fwd": (_i, [C.POINTER(UmmaConvDesc), _vp]),
    "rnc_f32_to_split": (_i, [_vp, _i, _i, C.c_longlong, _vp, _vp, _i, _i, _vp]),
    "rnc_f32_to_tf32_split": (_i, [_vp, _i, _i, C.c_longlong, _vp, _vp, _i, _i, _vp]),
    "rnc_stem_conv7x7s2_fwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "rnc_stem_window_prep": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "rnc_instnorm_stats": (_i, [_vp, _i, _i, _i, _f, _vp, _vp, _vp]),
    "rnc_instnorm_finalize": (_i, [_vp, _i, _i, _i, _f, _vp, _vp]),
    "rnc_instnorm_apply": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "rnc_add_relu_split": (_i, [_vp, _vp, C.c_size_t, _vp, _vp, _vp, _vp]),
    "rnc_fmap_pyramid": (_i, [_vp, _i, _i, _i, _i, _i, _vp]),
    "rnc_conv_flow7x7_split_fwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _i, _vp]),
    "rnc_conv_flow7x7_fwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _i, _vp]),
    "rnc_flow_head2_fwd": (_i, [_vp, _i, _i, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "rnc_flow_im2col7_split_fwd": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _vp]),
    "rnc_flow_tap_gather_fwd": (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "rnc_forward_interpolate_fwd": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "rnc_coords_init": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "rnc_coords_to_flow": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "rnc_nchw_to_cl": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _vp]),
    "rnc_cl_to_nchw": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "rnc_convex_upsample_fwd": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "rnc_flow_x2_fwd": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "rnc_ncup_guidance_fwd": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _i, _vp]),
    "rnc_ncup_guidance_split_fwd": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp]),
    "rnc_conf_head_fwd": (_i, [_vp, _i, _i, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "rnc_ncup_fwd": (_i, [_vp, _vp, C.POINTER(_f), _i, _i, _i, _f, _vp, _vp]),
    "rnc_bilinear_sample_fwd": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "rnc_nconv2d_fwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _f, _vp, _vp, _vp]),
    "rnc_corr_lookup_bwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "rnc_pyramid_pool_bwd": (_i, [_vp, _i, _i, _i, _i, _i, _vp]),
    "rnc_conv2d_cl_wgrad": (_i, [_vp, _i, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _vp, _vp]),
    "rnc_conv2d_umma_wgrad_workspace_bytes": (C.c_size_t, [_i, _i, _i, _i, _i, _i, _i, _i]),
    "rnc_conv2d_umma_wgrad": (_i, [_vp, _i, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _vp, _vp, C.c_size_t, _vp]),
    "rnc_nconv2d_bwd_workspace_bytes": (C.c_size_t, [_i, _i, _i, _i]),
    "rnc_nconv2d_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _f, _vp, _vp, _vp, _vp, C.c_size_t, _vp]),
}

_lib = None
_lock = threading.Lock()


def lib():
    """Load librnc.so once; raise loudly if it is missing or stale."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RncUnavailable(
                f"{LIB_PATH} not found: build it with `python raft-ncup_b200/rnc/build.py` "
                "(the RAFT-NCUP hot path has no CPU/PyTorch fallback)")
        try:
            handle = C.CDLL(LIB_PATH)
        except OSError as e:
            raise RncUnavailable(f"cannot load {LIB_PATH}: {e}") from e
        for name, (res, args) in SIGNATURES.items():
            try:
                fn = getattr(handle, name)
            except AttributeError as e:
                raise RncUnavailable(f"{LIB_PATH} does not export {name} (stale build?)") from e
            fn.restype = res
            fn.argtypes = args
        if handle.rnc_abi_version() != ABI_VERSION:
            raise RncUnavailable(f"librnc ABI {handle.rnc_abi_version()} != expected {ABI_VERSION}; rebuild")
        _lib = handle
    return _lib


def check(status, what=""):
    """Translate a negative rnc_status into a Python exception (the reference's error channel, SURVEY §8b)."""
    if status == 0:
        return
    l = lib()
    msg = l.rnc_status_string(status).decode()
    if status == -4:
        msg += f" (cudaError {l.rnc_last_cuda_error()})"
    if status in (-1, -3):
        raise ValueError(f"rnc {what}: {msg}")
    raise RncError(f"rnc {what}: {msg}")


def launch_count():
    return int(lib().rnc_launch_count())


def launch_count_reset():
    lib().rnc_launch_count_reset()
