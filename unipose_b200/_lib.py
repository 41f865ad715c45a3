"""ctypes binding of libunipose_b200.so (the C-ABI declared in include/unipose_b200.h).

There is NO fallback: if the shared object is missing or a call fails, this raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_void_p

from . import build as _build

UP_BF16, UP_FP16, UP_SPLIT = 0, 1, 2
UP_RESIZE_OUT_U8, UP_RESIZE_OUT_F32 = 8, 9
UP_FLAG_RELU, UP_FLAG_RESIDUAL, UP_FLAG_OUT_NCHW_F32, UP_FLAG_STATS, UP_FLAG_PROJ = 1, 2, 4, 8, 16


class UpConvDesc(ctypes.Structure):
    _fields_ = [
        ("n", c_int32), ("h", c_int32), ("w", c_int32),
        ("ho", c_int32), ("wo", c_int32),
        ("cin", c_int32), ("cout", c_int32),
        ("kh", c_int32), ("kw", c_int32),
        ("stride", c_int32), ("dil", c_int32),
        ("pad_h", c_int32), ("pad_w", c_int32),
        ("x_cstride", c_int32), ("x_coff", c_int32),
        ("x_groups", c_int32), ("x_group_nstride", c_int32),
        ("y_cstride", c_int32), ("y_coff", c_int32),
        ("r_cstride", c_int32), ("r_coff", c_int32),
        ("dtype", c_int32), ("flags", c_int32),
        ("cout_valid", c_int32), ("out_c_total", c_int32),
        ("x_cextent", c_int32), ("x_wpitch", c_int32),
        ("x_plane_stride", c_int64), ("y_plane_stride", c_int64),
        ("r_plane_stride", c_int64), ("w_plane_stride", c_int64),
        ("proj_cin", c_int32), ("proj_stride", c_int32),
    ]


class UpPackJob(ctypes.Structure):
    _fields_ = [("w", c_void_p), ("out", c_void_p), ("row_scale", c_void_p),
                ("plane_stride", c_int64), ("tile_start", c_int64),
                ("kh", c_int32), ("kw", c_int32), ("rows", c_int32), ("cols", c_int32),
                ("cout_real", c_int32), ("cin_total", c_int32), ("ci_off", c_int32), ("cin_slice", c_int32),
                ("scale_period", c_int32), ("dtype", c_int32), ("transpose", c_int32), ("reserved", c_int32)]


class UpEpilogueJob(ctypes.Structure):
    _fields_ = [("gamma", c_void_p), ("beta", c_void_p), ("mean", c_void_p), ("var", c_void_p), ("bias", c_void_p),
                ("fold_scale", c_void_p), ("scale", c_void_p), ("shift", c_void_p),
                ("eps", c_float), ("c_bn", c_int32), ("bias_len", c_int32), ("cout_real", c_int32), ("cout", c_int32),
                ("fold_into_weights", c_int32), ("reserved", c_int32 * 2)]


class UpImageJob(ctypes.Structure):
    _fields_ = [("src", c_void_p), ("h", c_int32), ("w", c_int32), ("pitch", c_int32), ("flip", c_int32)]


class UpWaspChainDesc(ctypes.Structure):
    _fields_ = [("n", c_int32), ("h", c_int32), ("w", c_int32), ("cin", c_int32), ("dil", c_int32 * 3),
                ("dtype", c_int32), ("conv1_cin", c_int32)]


class UpBneckChainDesc(ctypes.Structure):
    _fields_ = [("n", c_int32), ("h", c_int32), ("w", c_int32), ("planes", c_int32), ("nblocks", c_int32),
                ("dil", c_int32), ("dtype", c_int32)]


class UpBneckTailDesc(ctypes.Structure):
    _fields_ = [("n", c_int32), ("h", c_int32), ("w", c_int32), ("planes", c_int32), ("dil", c_int32), ("dtype", c_int32),
                ("proj_cin", c_int32), ("next_planes", c_int32)]


class UpBneckChainWeights(ctypes.Structure):
    _fields_ = [("w1", c_void_p), ("w2", c_void_p), ("w3", c_void_p), ("shift1", c_void_p), ("shift2", c_void_p),
                ("shift3", c_void_p)]


class UpWaspChainWeights(ctypes.Structure):
    _fields_ = [("aspp", c_void_p * 4), ("shift", c_void_p * 4), ("conv1", c_void_p), ("shift1", c_void_p),
                ("gap_t", c_void_p), ("shift_gap", c_void_p), ("conv1_pool_t", c_void_p)]


_P = c_void_p
_I = c_int
_L = c_int64
_F = c_float
_D = ctypes.c_double

# name -> argtypes (restype is always int unless listed in _RESTYPES)
_SIGNATURES = {
    "up_version": [],
    "up_device_info": [POINTER(c_int), POINTER(c_int), POINTER(c_int)],
    "up_conv2d_fwd": [POINTER(UpConvDesc), _P, _P, _P, _P, _P, _P, _P, _P],
    "up_pack_conv_weight": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _L, _P],
    "up_bn_fold": [_P, _P, _P, _P, _F, _P, _P, _I, _I, _P],
    "up_pack_input_s2d": [_P, _P, _I, _I, _I, _I, _L, _I, _I, _P],
    "up_pack_input_u8_s2d": [_P, _P, _I, _I, _I, _I, _L, _I, _I, _F, _F, _P],
    "up_resize_pack_u8": [POINTER(UpImageJob), _P, _I, _I, _I, _I, _P, _L, _I, _I, _F, _F, _P],
    "up_gaussian_labels": [_P, _P, _I, _I, _I, _I, _F, _F, _I, _I, _P],
    "up_nchw_f32_to_nhwc": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _L, _P],
    "up_nhwc_to_nchw_f32": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _L, _P],
    "up_maxpool3x3s2": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _L, _L, _P],
    "up_upsample_bilinear_ac": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _L, _L, _P],
    "up_global_avgpool": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _L, _L, _P],
    "up_broadcast_hw": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _L, _L, _P],
    "up_global_sumpool": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _L, _L, _P],
    "up_upsample_bilinear_ac_nchw_f32": [_P, _P, _I, _I, _I, _I, _I, _I, _P],
    "up_avgpool9s8p1_f32": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "up_convlstm_cell0_fwd": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P],
    "up_convlstm_cell_fwd": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P],
    "up_convlstm_cell_bwd": [_P] * 17 + [_I, _I, _I, _I, _I, _P],
    "up_argmax2d": [_P, _P, _P, _P, _I, _I, _I, _I, _P],
    "up_calc_dists": [_P, _P, _P, _I, _I, _D, _D, _P],
    "up_dist_acc": [_P, _P, _I, _I, _D, _P],
    "up_mse_fwd_bwd": [_P, _P, _P, _P, _P, _L, _F, _P],
    "up_adam_step": [_P, _P, _P, _P, _L, _F, _F, _F, _F, _I, _P],
    "up_debug_conv_timing": [_P],
    "up_debug_chain_timing": [_P],
    "up_conv2d_wgrad": [POINTER(UpConvDesc), _P, _P, _P, _I, _I, _P, _L, _I, _P],
    "up_bn_stats": [_P, _L, _I, _I, _P, _P],
    "up_bn_finalize": [_P, _L, _P, _P, _P, _P, _F, _F, _P, _P, _P, _P, _I, _I, _P],
    "up_bn_stats_finalize": [_P, _L, _I, _I, _P, _P, _P, _P, _P, _F, _F, _P, _P, _P, _P, _I, _P],
    "up_bn_eval_prepare": [_P, _P, _P, _P, _F, _P, _P, _P, _P, _I, _I, _P],
    "up_scale_shift_act": [_P, _P, _P, _P, _P, _P, _L, _I, _I, _I, _P],
    "up_bn_bwd": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _I, _I, _I, _P, _P, _P],
    "up_ew_mul": [_P, _P, _P, _L, _I, _I, _I, _I, _P],
    "up_maxpool3x3s2_bwd": [_P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _P],
    "up_upsample_bilinear_ac_bwd": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "up_add_broadcast": [_P, _P, _I, _I, _I, _F, _I, _I, _P],
    "up_zero_insert2x": [_P, _P, _I, _I, _I, _I, _I, _P],
    "up_pack_conv_weights": [_P, _I, _L, _P],
    "up_wasp_chain_supported": [POINTER(UpWaspChainDesc)],
    "up_bneck_chain_supported": [POINTER(UpBneckChainDesc)],
    "up_bneck_tail_supported": [POINTER(UpBneckTailDesc)],
    "up_bneck_tail_fwd": [POINTER(UpBneckTailDesc), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "up_bneck_chain_fwd": [POINTER(UpBneckChainDesc), POINTER(UpBneckChainWeights), _P, _P, _P, _P, _L, _P],
    "up_debug_bneck_timing": [_P],
    "up_wasp_chain_fwd": [POINTER(UpWaspChainDesc), POINTER(UpWaspChainWeights), _P, _P, _P, _P, _L, _P],
    "up_epilogue_consts": [_P, _I, _I, _P],
}
_RESTYPES = {"up_conv2d_wgrad_scratch_bytes": (c_int64, [POINTER(UpConvDesc)]),
             "up_bn_work_doubles": (c_int64, [_I]),
             "up_pack_job_tiles": (c_int64, [POINTER(UpPackJob)]),
             "up_wasp_chain_workspace_bytes": (c_int64, [POINTER(UpWaspChainDesc)]),
             "up_bneck_chain_workspace_bytes": (c_int64, [POINTER(UpBneckChainDesc)])}


class UpView(ctypes.Structure):
    _fields_ = [("ptr", c_void_p), ("cstride", c_int32), ("coff", c_int32), ("plane_stride", c_int64)]

# Every symbol include/unipose_b200.h declares (tests check the .so exports all of them).
DECLARED_SYMBOLS = ["up_last_error"] + list(_SIGNATURES) + list(_RESTYPES)

_lib = None


def lib_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = True) -> ctypes.CDLL:
    """Load (building first if the .so is absent or stale and nvcc is available)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    override = os.environ.get("UNIPOSE_B200_LIB")     # A/B testing of kernel builds (tools only)
    if override:
        build_if_missing = False
        path = override
    if build_if_missing:
        try:
            path = _build.build_library()
        except Exception:
            if not os.path.exists(path):
                raise
    if not os.path.exists(path):
        raise RuntimeError(
            "unipose_b200: %s is missing - run `python -m unipose_b200.build` (needs nvcc). "
            "There is no CPU / PyTorch fallback." % path)
    lib = ctypes.CDLL(path)
    lib.up_last_error.restype = c_char_p
    lib.up_last_error.argtypes = []
    for name, args in _SIGNATURES.items():
        fn = getattr(lib, name, None)
        if fn is None:
            continue  # reported by the symbol test; calling it raises below
        fn.argtypes = args
        fn.restype = c_int
    for name, (res, args) in _RESTYPES.items():
        fn = getattr(lib, name, None)
        if fn is not None:
            fn.argtypes = args
            fn.restype = res
    _lib = lib
    return lib


def call(name: str, *args) -> None:
    """Invoke a C-ABI entry point; raise RuntimeError(up_last_error()) on a non-zero status."""
    lib = load()
    fn = getattr(lib, name, None)
    if fn is None:
        raise RuntimeError("unipose_b200: symbol %s not exported by %s" % (name, lib_path()))
    rc = fn(*args)
    if rc != 0:
        raise RuntimeError("unipose_b200.%s failed (%d): %s" % (name, rc, lib.up_last_error().decode()))
