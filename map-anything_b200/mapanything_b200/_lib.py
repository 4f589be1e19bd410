"""ctypes binding of the C-ABI CUDA library (include/mapanything_b200.h).

There is deliberately NO fallback: if the shared object is missing or a call fails, the caller gets an
exception.  Nothing in this package computes on the CPU or through PyTorch library kernels instead.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("MAPANYTHING_B200_LIB", _HERE / "libmapanything_b200.so"))

MA_OK = 0
MA_BF16, MA_F32 = 0, 1
MA_ACT_NONE, MA_ACT_GELU, MA_ACT_RELU = 0, 1, 2
MA_GEMM_ACT_AFTER_RESIDUAL, MA_GEMM_RELU_OUT_BEFORE_RESIDUAL = 1, 2


class MapAnythingB200Error(RuntimeError):
    pass


class GemmEpilogue(C.Structure):
    _fields_ = [
        ("out", C.c_void_p),
        ("ldo", C.c_int64),
        ("out_dtype", C.c_int32),
        ("act", C.c_int32),
        ("bias", C.c_void_p),
        ("colscale", C.c_void_p),
        ("residual", C.c_void_p),
        ("ldr", C.c_int64),
        ("residual_dtype", C.c_int32),
        ("residual_row_mod", C.c_int32),
        ("out_relu", C.c_void_p),
        ("ldo_relu", C.c_int64),
        ("rows_per_group_in", C.c_int32),
        ("rows_per_group_out", C.c_int32),
        ("row_offset_out", C.c_int32),
        ("flags", C.c_int32),
        ("head_w", C.c_void_p),
        ("head_bias", C.c_void_p),
        ("head_out", C.c_void_p),
    ]


MA_ATTN_MAX_SEGMENTS, MA_ATTN_STATE_IN, MA_ATTN_STATE_OUT = 16, 1, 2


class AttnExt(C.Structure):
    _fields_ = [
        ("n_segments", C.c_int32),
        ("flags", C.c_int32),
        ("seg_row0", C.c_int32 * MA_ATTN_MAX_SEGMENTS),
        ("seg_len", C.c_int32 * MA_ATTN_MAX_SEGMENTS),
        ("state_o", C.c_void_p),
        ("ld_state_o", C.c_int64),
        ("state_m", C.c_void_p),
        ("kv_split", C.c_int32),
        ("kv_split_from", C.c_int32),
        ("split_stride_o", C.c_int64),
        ("split_stride_m", C.c_int64),
    ]


class DecodeSpec(C.Structure):
    """ma_decode_spec (include/mapanything_b200.h)."""
    _fields_ = [("rep", C.c_int), ("has_conf", C.c_int), ("has_mask", C.c_int), ("point_mode", C.c_int),
                ("use_factored", C.c_int), ("conf_vmin", C.c_float)]


class JpegInfo(C.Structure):
    """ma_jpeg_info (include/mapanything_b200.h)."""
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("ncomp", C.c_int32), ("h_samp", C.c_int32),
                ("v_samp", C.c_int32), ("restart_interval", C.c_int32), ("nsegments", C.c_int32), ("nsubseq", C.c_int32),
                ("nblocks", C.c_int64), ("plane_bytes", C.c_int64), ("blob_bytes", C.c_int64)]


MA_REP = {"pointmap": 0, "raymap+depth": 1, "raydirs+depth+pose": 2, "campointmap+pose": 3, "pointmap+raydirs+depth+pose": 4}
MA_PTS = {"linear": 0, "exp": 1, "z_exp": 2}

# name -> (restype, argtypes); must list every symbol include/mapanything_b200.h declares.
_i, _i64, _p, _f = C.c_int, C.c_int64, C.c_void_p, C.c_float
SIGNATURES = {
    "ma_last_error": (C.c_char_p, []),
    "ma_abi_version": (_i, []),
    "ma_device_info": (_i, [C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "ma_set_pdl": (_i, [_i]),
    "ma_set_stream_k": (_i, [_i]),
    "ma_last_gemm_block": (_i, []),
    "ma_last_attention_kernel": (_i, []),
    "ma_last_resample_kernel": (_i, []),
    "ma_gemm_bf16": (_i, [_p, _i64, _p, _i64, _i, _i, _i, C.POINTER(GemmEpilogue), _i, _p]),
    "ma_conv3x3_bf16": (_i, [_p, _i, _i, _i, _i, _p, _i64, _i, C.POINTER(GemmEpilogue), _i, _p]),
    "ma_attention_fwd": (_i, [_p, _i64, _i64, _i, _p, _i64, _i64, _i, _p, _i64, _i, _p, _i64, _i, _i, _i, _i, _i, _i64,
                              _i64, _f, _p]),
    "ma_attention_fwd_ex": (_i, [_p, _i64, _i64, _i, _p, _i64, _i64, _i, _p, _i64, _i, _p, _i64, _i, _i, _i, _i, _i, _i64,
                                 _i64, _f, C.POINTER(AttnExt), _p]),
    "ma_attention_merge": (_i, [_p, _i64, _i64, _p, _i64, _i, _i64, _i, _f, _p, _i64, _i, _p]),
    "ma_patchify": (_i, [_p, _p, _i, _i, _i, _i, _i, _p]),
    "ma_layernorm": (_i, [_p, _i, _i64, _p, _i, _i64, _p, _p, _i, _i, _f, _i, _i64, _i64, _i64, _i64, _p]),
    "ma_fill_f32": (_i, [_p, _i64, _f, _p]),
    "ma_set_rows": (_i, [_p, _i64, _i, _i64, _i64, _p, _p, _i, _p]),
    "ma_im2col3x3": (_i, [_p, _p, _i, _i, _i, _i, _i, _p]),
    "ma_pixel_shuffle": (_i, [_p, _p, _i, _i, _i, _i, _i, _p]),
    "ma_pixel_shuffle_f32": (_i, [_p, _i64, _p, _i64, _i, _i, _i, _i, _i, _p]),
    "ma_bilinear_align_corners": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "ma_token_mean": (_i, [_p, _p, _i, _i, _i, _p]),
    "ma_decode_dense": (_i, [_p, _i, _p, _p, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "ma_decode_scene": (_i, [C.POINTER(DecodeSpec), _p, _i, _p, _p, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "ma_head_linear_small": (_i, [_p, _i64, _p, _i64, _p, _p, _i64, _i64, _i, _i, _p]),
    "ma_split_bf16x3": (_i, [_p, _i64, _p, _i, _i, _p]),
    "ma_token_mean_f32": (_i, [_p, _p, _i, _i, _i, _p]),
    "ma_linear_rows_f32": (_i, [_p, _i64, _p, _i64, _p, _i, _p, _i64, _i, _i, _i, _p]),
    "ma_rays_from_intrinsics": (_i, [_p, _p, _i, _i, _i, _p]),
    "ma_normalize_rays": (_i, [_p, _p, _i64, _p]),
    "ma_depth_z_to_along_ray": (_i, [_p, _p, _p, _i64, _p]),
    "ma_pose_to_quat_trans": (_i, [_p, _p, _p, _i, _p]),
    "ma_unshuffle_split": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p]),
    "ma_depth_factor": (_i, [_p, _i, _i64, _p, _p, _p]),
    "ma_pose_inputs": (_i, [_p, _p, _p, _i, _p, _p, _p, _p]),
    "ma_fuse_add": (_i, [_p, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "ma_denorm_image":(_i, [_p, _p, _i, _i, _i, C.POINTER(_f), C.POINTER(_f), _p]),
    "ma_intrinsics_from_rays": (_i, [_p, _p, _i, _i, _i, _p]),
    "ma_pose_matrices": (_i, [_p, _p, _p, _i, _p]),
    "ma_edge_mask": (_i, [_p, _p, _i, _p, _p, _p, _p, _p, _p, _i, _i, _i, _f, _f, _p]),
    "ma_apply_mask": (_i, [_p, _i, _i, _p, _p, _i64, _i, _p]),
    "ma_quantile_mask": (_i, [_p, _p, _p, _i, _i64, _f, _p]),
    "ma_mask_and": (_i, [_p, _p, _p, _i64, _p]),
    "ma_depthmap_to_world": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _p]),
    "ma_resample_coeffs": (_i, [_i, _i, _i, C.POINTER(_i), _p, _p]),
    "ma_resample_h_u8rgb": (_i, [_p, _i64, _i64, _i, _i, _i, _i, _i, _p, _p, _p, _i, _i, _i, _i, _p, _p]),
    "ma_resample_pack_coeffs": (_i, [_p, _i, _i, _p]),
    "ma_gather_rows_cols_f32": (_i, [_p, _i64, _p, _p, _i, _i, _p, _p]),
    "ma_f32_to_u8": (_i, [_p, _i64, _f, _p, _p]),
    "ma_resample_v_norm_u8rgb": (_i, [_p, _i, _i, _i, _i, _p, _p, _i, _i, _i, _i, _p, _p, _p, _p, _p]),
    "ma_jpeg_parse": (_i, [_p, _i64, C.POINTER(JpegInfo), _p, _i64]),
    "ma_jpeg_workspace": (_i, [C.POINTER(JpegInfo), _i, C.POINTER(_i64)]),
    "ma_jpeg_decode": (_i, [_p, C.POINTER(_i64), C.POINTER(JpegInfo), _i, C.POINTER(_p), C.POINTER(C.c_int32), _p, _i64, _p,
                            _p]),
}

_lib = None


def load() -> C.CDLL:
    """Loads the library (once). Raises if it has not been built: there is no other compute path."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise MapAnythingB200Error(
            f"{LIB_PATH} not found. Build it with `python map-anything_b200/build.py` "
            "(nvcc, sm_100a). This package has no CPU / PyTorch fallback."
        )
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so is stale / missing a symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != MA_OK:
        msg = load().ma_last_error().decode("utf-8", "replace")
        raise MapAnythingB200Error(f"{what} failed (status {rc}): {msg}")
