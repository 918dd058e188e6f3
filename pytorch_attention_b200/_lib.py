"""ctypes binding of libpa_b200.so (C ABI in include/pa_b200.h).  No CPU fallback: if the library is missing
or a call fails, an exception is raised."""
from __future__ import annotations

import ctypes as C
import os
import threading

from . import build as _build

PA_DTYPE_F16, PA_DTYPE_BF16, PA_DTYPE_F32 = 0, 1, 2
PA_ERR_BAD_SHAPE, PA_ERR_UNSUPPORTED, PA_ERR_MISALIGNED, PA_ERR_WORKSPACE = -1, -2, -3, -4
PA_ERR_CUDA, PA_ERR_DEVICE, PA_ERR_NULL = -5, -6, -7

_vp, _i, _ll, _f = C.c_void_p, C.c_int, C.c_longlong, C.c_float


class GemmArgs(C.Structure):
    _fields_ = [("a_dtype", _i), ("b_dtype", _i), ("out_dtype", _i),
                ("M", _i), ("N", _i), ("K", _i), ("Z", _i),
                ("A", _vp), ("lda", _ll), ("a_batch", _ll),
                ("B", _vp), ("ldb", _ll), ("b_batch", _ll),
                ("D", _vp), ("ldd", _ll), ("d_batch", _ll),
                ("bias", _vp), ("bias_mode", _i), ("block_n", _i),
                ("residual", _vp), ("ldr", _ll), ("r_batch", _ll), ("res_dtype", _i), ("cluster", _i)]


class AttnArgs(C.Structure):
    _fields_ = [("G", _i), ("H", _i), ("n_q", _i), ("n_k", _i),
                ("q", _vp), ("ldq", _ll), ("q_group", _ll), ("q_col0", _i),
                ("kv", _vp), ("ldkv", _ll), ("kv_group", _ll), ("k_col0", _i), ("v_col0", _i),
                ("o", _vp), ("ldo", _ll), ("o_group", _ll), ("o_col0", _i),
                ("scale", _f), ("head_dim", _i)]


class VitArgs(C.Structure):
    _fields_ = [("dtype", _i), ("out_dtype", _i), ("B", _i), ("N", _i), ("C", _i), ("H", _i),
                ("scale", _f),
                ("x", _vp), ("qkv_weight", _vp), ("qkv_bias", _vp), ("proj_weight", _vp), ("proj_bias", _vp),
                ("y", _vp), ("topk", _i)]


class VitBlockArgs(C.Structure):
    _fields_ = [("attn", VitArgs), ("ln_weight", _vp), ("ln_bias", _vp), ("ln_eps", _f)]


class BvitArgs(C.Structure):
    _fields_ = [("dtype", _i), ("out_dtype", _i), ("B", _i), ("N", _i), ("C", _i), ("H", _i), ("dim_head", _i), ("scale", _f),
                ("x", _vp), ("qkv_weight", _vp), ("out_weight", _vp), ("out_bias", _vp), ("qkv", _vp), ("y", _vp)]


class PvtArgs(C.Structure):
    _fields_ = [("dtype", _i), ("out_dtype", _i), ("B", _i), ("N", _i), ("C", _i), ("H", _i),
                ("Himg", _i), ("Wimg", _i), ("sr", _i), ("scale", _f),
                ("x", _vp), ("q_weight", _vp), ("q_bias", _vp), ("kv_weight", _vp), ("kv_bias", _vp),
                ("proj_weight", _vp), ("proj_bias", _vp), ("sr_weight_t", _vp), ("sr_scale", _vp), ("sr_shift", _vp),
                ("y", _vp),
                ("sr_mode", _i), ("sr_dense_weight", _vp), ("sr_dense_bias", _vp), ("rel_pos", _vp),
                ("kv_tokens", _vp), ("kv_count", _i)]


class P2tArgs(C.Structure):
    _fields_ = [("attn", PvtArgs), ("n_levels", _i), ("pool_h", _i * 4), ("pool_w", _i * 4),
                ("dconv_weight_t", _vp * 4), ("dconv_bias", _vp * 4), ("norm_weight", _vp), ("norm_bias", _vp), ("norm_eps", _f)]


class PvtBlockArgs(C.Structure):
    _fields_ = [("attn", PvtArgs), ("ln_weight", _vp), ("ln_bias", _vp), ("ln_eps", _f)]


class CvtArgs(C.Structure):
    _fields_ = [("dtype", _i), ("out_dtype", _i), ("B", _i), ("C", _i), ("H", _i), ("Himg", _i), ("Wimg", _i), ("ks", _i),
                ("scale", _f),
                ("x", _vp), ("dw_weight", _vp), ("dw_scale", _vp), ("dw_shift", _vp), ("qkv_weight", _vp), ("qkv_bias", _vp),
                ("proj_weight", _vp), ("proj_bias", _vp), ("y", _vp), ("residual", _vp)]


class XcitArgs(C.Structure):
    _fields_ = [("dtype", _i), ("out_dtype", _i), ("B", _i), ("N", _i), ("C", _i), ("H", _i), ("scale", _f),
                ("x", _vp), ("qkv_weight", _vp), ("qkv_bias", _vp), ("proj_weight", _vp), ("proj_bias", _vp),
                ("temperature", _vp), ("y", _vp)]


class XcaBlockArgs(C.Structure):
    _fields_ = [("attn", XcitArgs), ("ln_weight", _vp), ("ln_bias", _vp), ("ln_eps", _f)]


class LepeArgs(C.Structure):
    _fields_ = [("B", _i), ("L", _i), ("C", _i), ("H", _i), ("resolution", _i), ("idx", _i), ("split_size", _i),
                ("scale", _f),
                ("q", _vp), ("k", _vp), ("v", _vp), ("ld", _ll), ("batch_stride", _ll),
                ("get_v_weight_t", _vp), ("get_v_bias", _vp),
                ("out", _vp), ("ldo", _ll), ("out_batch_stride", _ll)]


class CswinBlockArgs(C.Structure):
    _fields_ = [("dtype", _i), ("out_dtype", _i), ("B", _i), ("L", _i), ("C", _i), ("H", _i),
                ("reso", _i), ("split_size", _i), ("last_stage", _i), ("residual", _i), ("scale", _f), ("ln_eps", _f),
                ("x", _vp), ("norm1_weight", _vp), ("norm1_bias", _vp), ("qkv_weight", _vp), ("qkv_bias", _vp),
                ("proj_weight", _vp), ("proj_bias", _vp), ("get_v_weight_t", _vp * 2), ("get_v_bias", _vp * 2),
                ("y", _vp)]


class DilateArgs(C.Structure):
    _fields_ = [("dtype", _i), ("out_dtype", _i), ("B", _i), ("Himg", _i), ("Wimg", _i), ("C", _i), ("H", _i),
                ("kernel_size", _i), ("n_dilation", _i), ("dilation", _i * 8), ("scale", _f),
                ("x", _vp), ("qkv_weight", _vp), ("qkv_bias", _vp), ("proj_weight", _vp), ("proj_bias", _vp), ("y", _vp)]


class DilateBlockArgs(C.Structure):
    _fields_ = [("attn", DilateArgs), ("ln_weight", _vp), ("ln_bias", _vp), ("ln_eps", _f)]


# name -> (restype, argtypes); every symbol declared in include/pa_b200.h must be listed here
# (tests/test_abi.py cross-checks this table against the header).
SYMBOLS = {
    "pa_version": (_i, []),
    "pa_last_error": (C.c_char_p, []),
    "pa_device_check": (_i, [_i]),
    "pa_launch_count": (C.c_ulonglong, []),
    "pa_reload_env": (None, []),
    "pa_debug_cosched_occupancy": (_i, [_i, C.POINTER(_i)]),
    "pa_gemm_tn": (_i, [C.POINTER(GemmArgs), _vp]),
    "pa_cast_f32": (_i, [_vp, _vp, _ll, _i, _vp]),
    "pa_debug_set_gemm_trace": (None, [_vp]),
    "pa_attn_core": (_i, [C.POINTER(AttnArgs), _vp]),
    "pa_vit_workspace_bytes": (C.c_size_t, [C.POINTER(VitArgs)]),
    "pa_last_vit_path": (_i, []),
    "pa_vit_fwd": (_i, [C.POINTER(VitArgs), _vp, C.c_size_t, _vp]),
    "pa_vit_block_attn_workspace_bytes": (C.c_size_t, [C.POINTER(VitBlockArgs)]),
    "pa_vit_block_attn_fwd": (_i, [C.POINTER(VitBlockArgs), _vp, C.c_size_t, _vp]),
    "pa_bvit_workspace_bytes": (C.c_size_t, [C.POINTER(BvitArgs)]),
    "pa_bvit_fwd": (_i, [C.POINTER(BvitArgs), _vp, C.c_size_t, _vp]),
    "pa_pvt_workspace_bytes": (C.c_size_t, [C.POINTER(PvtArgs)]),
    "pa_pvt_fwd": (_i, [C.POINTER(PvtArgs), _vp, C.c_size_t, _vp]),
    "pa_p2t_workspace_bytes": (C.c_size_t, [C.POINTER(P2tArgs)]),
    "pa_p2t_fwd": (_i, [C.POINTER(P2tArgs), _vp, C.c_size_t, _vp]),
    "pa_pvt_block_attn_workspace_bytes": (C.c_size_t, [C.POINTER(PvtBlockArgs)]),
    "pa_pvt_block_attn_fwd": (_i, [C.POINTER(PvtBlockArgs), _vp, C.c_size_t, _vp]),
    "pa_cvt_workspace_bytes": (C.c_size_t, [C.POINTER(CvtArgs)]),
    "pa_cvt_fwd": (_i, [C.POINTER(CvtArgs), _vp, C.c_size_t, _vp]),
    "pa_xca_workspace_bytes": (C.c_size_t, [C.POINTER(XcitArgs)]),
    "pa_xca_fwd": (_i, [C.POINTER(XcitArgs), _vp, C.c_size_t, _vp]),
    "pa_xca_block_attn_workspace_bytes": (C.c_size_t, [C.POINTER(XcaBlockArgs)]),
    "pa_xca_block_attn_fwd": (_i, [C.POINTER(XcaBlockArgs), _vp, C.c_size_t, _vp]),
    "pa_class_attn_workspace_bytes": (C.c_size_t, [C.POINTER(XcitArgs)]),
    "pa_class_attn_fwd": (_i, [C.POINTER(XcitArgs), _vp, C.c_size_t, _vp]),
    "pa_cswin_lepe_fwd": (_i, [C.POINTER(LepeArgs), _vp]),
    "pa_cswin_block_attn_workspace_bytes": (C.c_size_t, [C.POINTER(CswinBlockArgs)]),
    "pa_cswin_block_attn_fwd": (_i, [C.POINTER(CswinBlockArgs), _vp, C.c_size_t, _vp]),
    "pa_dilate_workspace_bytes": (C.c_size_t, [C.POINTER(DilateArgs)]),
    "pa_dilate_fwd": (_i, [C.POINTER(DilateArgs), _vp, C.c_size_t, _vp]),
    "pa_dilate_core": (_i, [C.POINTER(DilateArgs), _vp, _vp, _vp]),
    "pa_dilate_block_attn_workspace_bytes": (C.c_size_t, [C.POINTER(DilateBlockArgs)]),
    "pa_dilate_block_attn_fwd": (_i, [C.POINTER(DilateBlockArgs), _vp, C.c_size_t, _vp]),
}

_lock = threading.Lock()
_lib = None


class PaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libpa_b200 error {code}: {msg}")
        self.code = code


def lib_path():
    return _build.LIB_PATH


def load():
    """Load (building first if the sources are newer and nvcc is available) and return the CDLL."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = _build.LIB_PATH
        stale_error = None
        if _build.is_stale():
            try:
                _build.build_lib()
            except Exception as e:  # no nvcc, or compile error
                if not os.path.exists(path):
                    raise RuntimeError(
                        f"libpa_b200.so is not built ({path}) and could not be built: {e}. "
                        "This package has no CPU / PyTorch fallback.") from e
                stale_error = e
        lib = C.CDLL(path)
        for name, (res, args) in SYMBOLS.items():
            try:
                fn = getattr(lib, name)
            except AttributeError as e:
                raise RuntimeError(f"{path} does not export {name}: the library is older than the sources"
                                   + (f" and the rebuild failed: {stale_error}" if stale_error else "")) from e
            fn.restype = res
            fn.argtypes = args
        if stale_error is not None:
            # an older library is in use although the sources are newer (e.g. the GPU box has no nvcc in PATH): say so, and
            # refuse outright if its ABI version differs from the header this package was written against
            import warnings
            want = _build.header_version()
            if want is not None and int(lib.pa_version()) != want:
                raise RuntimeError(f"{path} reports ABI version {lib.pa_version()} but include/pa_b200.h declares {want}, "
                                   f"and the rebuild failed: {stale_error}")
            warnings.warn(f"libpa_b200.so is older than its sources and could not be rebuilt ({stale_error}); using it as is",
                          RuntimeWarning)
        _lib = lib
        return lib


def check(rc):
    if rc != 0:
        msg = load().pa_last_error()
        msg = msg.decode() if msg else ""
        if rc in (PA_ERR_BAD_SHAPE,):
            raise AssertionError(msg)         # the reference raises AssertionError on shape violations
        if rc in (PA_ERR_UNSUPPORTED, PA_ERR_MISALIGNED, PA_ERR_NULL, PA_ERR_WORKSPACE):
            raise ValueError(msg)
        raise PaError(rc, msg)


def launch_count():
    return int(load().pa_launch_count())


def reload_env():
    """The library caches the PA_* environment switches at its first call; re-read them after changing os.environ."""
    load().pa_reload_env()
