"""ctypes binding of libb2u.so — the C-ABI declared in include/b2u.h.

There is no CPU fallback: if the library is missing it is built with nvcc, and if that fails the import raises.
Every wrapper raises `B2UError` with the library's message on a non-zero status.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
MAX_TAPS = 16
MAX_VIEWS = 4

EPI_RELU = 1
EPI_STATS = 2
EPI_OUT_F32 = 4
EPI_HEAD = 8
EPI_HEAD_ONLY = 16

DT_F32, DT_U8, DT_U16, DT_I16 = 0, 1, 2, 3     # b2u.h B2U_DT_*: element type of raw input tiles / rasters


class B2UError(RuntimeError):
    pass


class View(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("C", C.c_int32), ("W", C.c_int32), ("H", C.c_int32), ("N", C.c_int32),
                ("sW", C.c_int64), ("sH", C.c_int64), ("sN", C.c_int64)]


class BNFin(C.Structure):
    _fields_ = [("counter", C.c_void_p), ("count", C.c_double), ("gamma", C.c_void_p), ("beta", C.c_void_p),
                ("eps", C.c_float), ("momentum", C.c_float), ("running_mean", C.c_void_p),
                ("running_var", C.c_void_p), ("mean", C.c_void_p), ("invstd", C.c_void_p), ("scale", C.c_void_p),
                ("shift", C.c_void_p)]


class ConvDesc(C.Structure):
    _fields_ = [
        ("a", View * MAX_VIEWS), ("num_a", C.c_int32), ("out", View),
        ("w", C.c_void_p), ("w_rows", C.c_int32), ("w_taps", C.c_int32), ("w_cin", C.c_int32), ("w_cinp", C.c_int32),
        ("num_taps", C.c_int32),
        ("tap_a", C.c_int8 * MAX_TAPS), ("tap_dy", C.c_int8 * MAX_TAPS), ("tap_dx", C.c_int8 * MAX_TAPS),
        ("tap_w", C.c_int8 * MAX_TAPS),
        ("scale", C.c_void_p), ("shift", C.c_void_p),
        ("res", View), ("res_mask", View), ("zmask", View),
        ("flags", C.c_uint32), ("stats", C.c_void_p), ("stats_ld", C.c_int32),
        ("out_f32", C.c_void_p), ("out_f32_ld", C.c_int32),
        ("fin", BNFin),
        ("num_out", C.c_int32), ("out_nt", View * 4),
        ("w_batch_rows", C.c_int32),
        ("head_w", C.c_void_p), ("head_b", C.c_void_p), ("head_n", C.c_int32), ("head_ld", C.c_int32),
    ]


class ConvInfo(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("m_tiles", "n_tiles", "block_n", "tile_w", "tile_h", "tile_n", "stages",
                                         "k_chunks", "grid", "stats_rows", "fused_finalize")]


class WgradDesc(C.Structure):
    _fields_ = [
        ("dy", View), ("a", View * MAX_VIEWS), ("num_a", C.c_int32), ("num_taps", C.c_int32),
        ("tap_a", C.c_int8 * MAX_TAPS), ("tap_dy", C.c_int8 * MAX_TAPS), ("tap_dx", C.c_int8 * MAX_TAPS),
        ("Cout", C.c_int32), ("Cin", C.c_int32), ("want_bias", C.c_int32),
        ("partial", C.c_void_p), ("partial_bytes", C.c_size_t),
    ]


class WStageItem(C.Structure):
    _fields_ = [("w", C.c_void_p), ("bias", C.c_void_p), ("row_of_co", C.c_void_p), ("wf", C.c_void_p),
                ("wd", C.c_void_p), ("bias_rows", C.c_void_p), ("Cout", C.c_int32), ("Cin", C.c_int32),
                ("kk", C.c_int32), ("wf_cinp", C.c_int32), ("wd_coutp", C.c_int32), ("scale", C.c_float),
                ("block_start", C.c_int32), ("dscale", C.c_void_p)]


class WgradInfo(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("splits", "co_pad", "ci_pad", "taps_per_unit", "units", "grid", "k_steps",
                                         "block_n", "stages")] + [("partial_bytes", C.c_size_t)]


_lib = None


def lib_path() -> Path:
    # B2U_LIB: a diagnostic build of the same sources (tools/conv_timeline.py builds one with -DB2U_TIMELINE)
    override = os.environ.get("B2U_LIB")
    return Path(override) if override else _HERE / "libb2u.so"


def load():
    """Load (building first if necessary) libb2u.so. Raises if it cannot be produced — no fallback path exists."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not path.exists():
        from . import build as _build
        _build.build()
    if not path.exists():
        raise B2UError(f"{path} is missing and could not be built; the CUDA extension is mandatory")
    lib = C.CDLL(str(path))
    lib.b2u_last_error.restype = C.c_char_p
    _declare(lib)
    _lib = lib
    return lib


def _declare(lib):
    vp, i32, i64, f32, f64, u8p = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double, C.c_void_p
    sigs = {
        "b2u_version": [],
        "b2u_device_check": [],
        "b2u_conv_query": [C.POINTER(ConvDesc), C.POINTER(ConvInfo)],
        "b2u_conv_plan_create": [C.POINTER(ConvDesc), C.POINTER(vp)],
        "b2u_conv_plan_info": [vp, C.POINTER(ConvInfo)],
        "b2u_conv_run": [vp, vp],
        "b2u_wgrad_query": [C.POINTER(WgradDesc), C.POINTER(WgradInfo)],
        "b2u_wgrad_plan_create": [C.POINTER(WgradDesc), C.POINTER(vp)],
        "b2u_wgrad_run": [vp, vp],
        "b2u_wgrad_reduce": [vp, i32, i32, i32, i32, i32, i32, i32, vp, vp, f32, vp, vp, i32, vp],
        "b2u_stage_weights": [vp, i32, i32, vp],
        "b2u_bn_stats": [vp, i32, i64, i32, vp, i32, i32, vp],
        "b2u_bn_finalize": [vp, i32, i32, i32, f64, vp, vp, f32, f32, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp],
        "b2u_bn_eval_affine": [i32, vp, vp, vp, vp, f32, vp, vp, vp],
        "b2u_bn_apply": [vp, i32, vp, vp, vp, i32, vp, vp, i32, vp, i32, i64, i32, vp],
        "b2u_bn_bwd_reduce": [vp, i32, vp, i32, vp, i32, vp, vp, vp, vp, i32, i64, i32, vp, i32, i32, vp],
        "b2u_bn_bwd_finalize": [vp, i32, i32, i32, f64, vp, vp, vp, vp, vp, C.c_size_t, vp],
        "b2u_bn_bwd_apply": [vp, i32, vp, i32, vp, i32, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp, i32, i64, i32, vp],
        "b2u_bn_bwd_fused": [vp, i32, vp, i32, vp, i32, vp, vp, vp, vp, vp, i32, i32, vp, i32, i64, i32, vp, i32, i32, f64,
                             vp, vp, vp, vp, vp, vp],
        "b2u_maxpool_fwd": [vp, vp, u8p, i32, i32, i32, i32, i32, vp],
        "b2u_maxpool_bwd": [vp, u8p, vp, i32, i32, i32, i32, i32, i32, vp],
        "b2u_shuffle_cat_fwd": [vp, i32, i32, i32, vp, i32, i32, vp, vp, i32, vp, i32, i32, i32, i32, vp],
        "b2u_shuffle_bwd": [vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, vp],
        "b2u_shuffle_bwd_from_cat": [vp, vp, i32, vp, i32, i32, i32, i32, i32, vp],
        "b2u_copy_lanes": [vp, i32, i32, vp, i32, i32, i32, i64, vp],
        "b2u_shuffle_cat_fwd_crop": [vp, i32, i32, i32, vp, i32, i32, vp, vp, i32, vp, i32, i32, i32, i32, i32, i32, vp],
        "b2u_shuffle_bwd_crop": [vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp],
        "b2u_pad_even_fwd": [vp, vp, i32, i32, i32, i32, vp],
        "b2u_spectral_norm": [vp, i32, i32, vp, vp, i32, vp, vp],
        "b2u_spectral_norm_bwd": [vp, vp, i32, i32, vp, vp, vp, vp],
        "b2u_softmax_dim1": [vp, vp, vp, i32, i32, i32, vp],
        "b2u_softmax_dim1_bwd": [vp, vp, vp, vp, i32, i32, i32, vp],
        "b2u_transpose_bnc": [vp, i32, vp, i32, i32, i32, i32, vp],
        "b2u_attn_out": [vp, vp, vp, vp, i64, vp],
        "b2u_attn_out_bwd": [vp, vp, vp, vp, vp, vp, i64, vp],
        "b2u_pad_even_bwd": [vp, vp, i32, i32, i32, i32, i32, vp],
        "b2u_nchw_to_nhwc": [vp, i32, f32, f32, vp, i32, i32, i32, i32, i32, i32, i32, vp],
        "b2u_pointwise_smallk": [vp, i32, i32, vp, i32, vp, i32, vp, i32, i64, i32, vp],
        "b2u_im2col": [vp, i32, i32, i32, i32, i32, i32, i32, i32, vp, i32, vp],
        "b2u_crop_tiles": [vp, i32, f32, f32, i32, i64, i64, vp, vp, i32, i32, vp, i32, vp],
        "b2u_crop_train_batch": [vp, i32, i32, i64, i64, vp, i32, vp, vp, vp, i32, i32, vp, vp, vp],
        "b2u_nhwc_to_nchw_f32": [vp, i32, i32, vp, i32, i32, i32, i32, vp],
        "b2u_ce_weight_sum": [u8p, i64, vp, i32, vp, i32, vp],
        "b2u_ce_fwd_bwd": [vp, i32, u8p, i64, i32, vp, vp, i32, vp, i32, vp, i32, f32, vp],
        "b2u_ce_finalize": [vp, i32, vp, i32, vp, vp],
        "b2u_focal_fwd_bwd": [vp, i32, u8p, i64, i32, vp, f32, i32, vp, i32, vp, i32, f32, vp],
        "b2u_dice_stats": [vp, i32, u8p, i32, i64, i32, i32, vp, i32, vp],
        "b2u_dice_bwd": [vp, i32, u8p, i32, i64, i32, i32, vp, i32, f32, i32, vp, i32, vp, f32, vp],
        "b2u_mse_fwd_bwd": [vp, i32, vp, i64, vp, i32, vp, i32, f32, vp],
        "b2u_mse_finalize": [vp, i32, i64, vp, vp],
        "b2u_regression_sums": [vp, i32, vp, i64, vp, i32, vp, vp, vp],
        "b2u_dice_counts": [vp, i32, u8p, i64, i32, vp, vp],
        "b2u_cast_f32_bf16": [vp, vp, i64, vp],
        "b2u_cast_bf16_f32": [vp, vp, i64, vp],
        "b2u_sgd_step": [vp, vp, i64, f32, f32, vp],
        "b2u_adam_step": [vp, vp, vp, vp, i64, vp, vp, vp, i32, vp, vp],
        "b2u_stitch_accumulate": [vp, i32, i32, i32, i32, i32, vp, vp, vp, i32, vp, u8p, i64, i64, i64, i64, vp],
        "b2u_stitch_finalize": [vp, u8p, i32, i64, i64, u8p, vp],
        "b2u_stitch_accumulate_q31": [vp, i32, i32, i32, i32, i32, vp, vp, vp, i32, vp, u8p, i64, i64, i64, i64, vp],
        "b2u_stitch_finalize_q31": [vp, u8p, i32, i64, i64, u8p, vp],
        "b2u_stitch_accumulate_dev": [vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, i32, i32, vp, u8p, i64, i64, i64, i64, vp],
        "b2u_stitch_accumulate_raw": [vp, i32, i32, i32, i32, i32, vp, vp, vp, i32, vp, u8p, i64, i64, i64, i64, vp],
        "b2u_stitch_finalize_mean": [vp, u8p, i32, i64, i64, f32, vp, vp],
        "b2u_softmax_nchw": [vp, i32, i32, i64, i32, i32, vp, u8p, vp],
        "b2u_confusion_counts": [u8p, i64, i64, u8p, i64, i64, i32, i32, i32, i32, vp, vp, vp, vp],
    }
    for name, args in sigs.items():
        fn = getattr(lib, name, None)
        if fn is None:
            continue  # tests assert that every declared symbol is exported; tolerate here for partial builds
        fn.argtypes = args
        fn.restype = C.c_int
    lib.b2u_conv_plan_destroy.argtypes = [vp]
    lib.b2u_conv_plan_destroy.restype = None
    lib.b2u_wgrad_plan_destroy.argtypes = [vp]
    lib.b2u_wgrad_plan_destroy.restype = None


def check(status: int, what: str = ""):
    if status != 0:
        msg = load().b2u_last_error().decode(errors="replace")
        raise B2UError(f"{what or 'b2u call'} failed ({status}): {msg}")


def call(name: str, *args):
    lib = load()
    check(getattr(lib, name)(*args), name)
