"""ctypes binding of libpwa_b200.so (C ABI in include/pwa.h).

There is NO CPU fallback and no alternative backend: if the shared library is missing the
import fails loudly with the build command; device entry points raise on a machine without a GPU.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpwa_b200.so")

PWA_F32, PWA_BF16, PWA_F16 = 0, 1, 2


class PwaGeom(C.Structure):
    _fields_ = [
        ("dims", C.c_int32 * 3), ("ws", C.c_int32 * 3), ("shift", C.c_int32 * 3), ("pads", C.c_int32 * 6),
        ("sp", C.c_int32 * 3), ("nwin", C.c_int32 * 3), ("data_lo", C.c_int32 * 3), ("crop_lo", C.c_int32 * 3),
        ("P", C.c_int32), ("N", C.c_int32), ("masked", C.c_int32), ("padded", C.c_int32),
    ]


class PwaAttnShape(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("P", C.c_int32), ("C", C.c_int32), ("heads", C.c_int32), ("I", C.c_int32),
        ("ws", C.c_int32 * 3), ("scale", C.c_float), ("p_drop", C.c_float),
        ("seed", C.c_uint64), ("offset", C.c_uint64), ("ld_qkv", C.c_int32), ("ld_p", C.c_int32),
        ("seed_dev", C.c_void_p), ("sel_table", C.c_void_p), ("work", C.c_void_p),
    ]


class PwaDenseAttn(C.Structure):                     # struct pwa_dense_attn
    _fields_ = [
        ("B", C.c_int32), ("P", C.c_int32), ("heads", C.c_int32), ("dh", C.c_int32), ("nq", C.c_int32), ("nk", C.c_int32),
        ("ld_q", C.c_int32), ("ld_k", C.c_int32), ("ld_v", C.c_int32),
        ("bias_stride", C.c_int64 * 4), ("mask_stride", C.c_int64 * 4),
        ("scale", C.c_float), ("p_drop", C.c_float), ("seed_dev", C.c_void_p),
    ]


class PwaError(RuntimeError):
    pass


def _load():
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA extension is not built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` (or `make -C <package>/csrc`). "
            "This package has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, f32p, u8p = C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p
    gp, sp = C.POINTER(PwaGeom), C.POINTER(PwaAttnShape)
    lib.pwa_version.restype = i32
    lib.pwa_last_error.restype = C.c_char_p
    lib.pwa_geometry.argtypes = [C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), gp]
    lib.pwa_region_ids.argtypes = [gp, vp]
    lib.pwa_index_map.argtypes = [gp, i32, vp]
    lib.pwa_attn_sel_table.argtypes = [vp, i32, i32, vp]
    lib.pwa_attn_sel_table.restype = i32
    lib.pwa_partition.argtypes = [vp, vp, i32, i32, gp, i32, i32, vp]
    lib.pwa_reverse.argtypes = [vp, vp, i32, i32, gp, i32, i32, vp]
    lib.pwa_reverse_add.argtypes = [vp, vp, vp, i32, i32, gp, i32, i32, vp]
    lib.pwa_reverse_add.restype = i32
    lib.pwa_gather_rows.argtypes = [vp, vp, vp, vp, i32, C.c_int64, C.c_int64, i32, i32, vp]
    lib.pwa_gather_rows.restype = i32
    lib.pwa_colsum_f32.argtypes = [f32p, f32p, i32, C.c_int64, vp]
    lib.pwa_colsum_f32.restype = i32
    lib.pwa_colsum_rows.argtypes = [vp, f32p, C.c_int64, i32, i32, vp]
    lib.pwa_colsum_rows.restype = i32
    lib.pwa_dropout.argtypes = [vp, vp, C.c_int64, C.c_float, vp, i32, vp]
    lib.pwa_dropout.restype = i32
    lib.pwa_dropout_colsum.argtypes = [vp, vp, C.c_int64, i32, C.c_float, vp, vp, i32, vp]
    lib.pwa_dropout_colsum.restype = i32
    lib.pwa_token_gemm_supported.argtypes = [i32, i32]
    lib.pwa_token_gemm_supported.restype = i32
    lib.pwa_token_gemm_fwd.argtypes = [vp] * 11 + [C.c_int64, i32, i32, C.c_float, C.c_float, vp, vp]
    lib.pwa_token_gemm_fwd.restype = i32
    lib.pwa_token_gemm_fwd_dt.argtypes = [vp] * 11 + [C.c_int64, i32, i32, C.c_float, C.c_float, vp, i32, vp]
    lib.pwa_token_gemm_fwd_dt.restype = i32
    if hasattr(lib, "pwa_debug_fwd_timeline"):          # debug builds only (make TIMELINE=1, include/pwa_debug.h)
        lib.pwa_debug_fwd_timeline.argtypes = [vp, i32]
        lib.pwa_debug_fwd_timeline.restype = i32
    lib.pwa_attn_tc_supported.argtypes = [sp, i32]
    dp = C.POINTER(PwaDenseAttn)
    lib.pwa_attn_dense_fwd.argtypes = [vp] * 7 + [dp, i32, vp]
    lib.pwa_attn_dense_bwd.argtypes = [vp] * 13 + [dp, i32, vp]
    lib.pwa_attn_dense_fwd.restype = lib.pwa_attn_dense_bwd.restype = i32
    lib.pwa_attn_fwd.argtypes = [vp] * 5 + [f32p] * 4 + [u8p, vp, f32p, sp, i32, i32, vp]
    lib.pwa_attn_bwd.argtypes = [vp] * 5 + [f32p] * 4 + [u8p, vp, f32p, vp] + [vp] * 3 + [f32p] * 7 + [sp, i32, i32, vp]
    i64, f32 = C.c_int64, C.c_float
    lib.pwa_ln_fwd.argtypes = [vp, vp, f32p, f32p, vp, vp, f32p, f32p, i64, i32, f32, i32, vp]
    lib.pwa_ln_bwd.argtypes = [vp, vp, f32p, f32p, f32p, vp, vp, f32p, f32p, i64, i32, i32, vp]
    lib.pwa_ln_bwd2.argtypes = [vp, vp, f32p, f32p, f32p, vp, vp, f32p, f32p, f32p, f32p, i64, i32, i32, vp]
    lib.pwa_ln_fwd.restype = lib.pwa_ln_bwd.restype = lib.pwa_ln_bwd2.restype = i32
    i32p = C.POINTER(i32)
    lib.pwa_bias_tables_fwd.argtypes = [f32p] * 8 + [f32p] * 4 + [i32, i32, i32p, i32p, i32, vp]
    lib.pwa_bias_tables_bwd.argtypes = [f32p] * 8 + [f32p] * 4 + [f32p] * 8 + [i32, i32, i32p, i32p, i32, vp]
    lib.pwa_bias_tables_fwd.restype = lib.pwa_bias_tables_bwd.restype = i32
    for name in ("pwa_geometry", "pwa_region_ids", "pwa_index_map", "pwa_partition", "pwa_reverse",
                 "pwa_attn_tc_supported", "pwa_attn_fwd", "pwa_attn_bwd"):
        getattr(lib, name).restype = i32
    return lib


lib = _load()

EXPORTED_SYMBOLS = ("pwa_version", "pwa_last_error", "pwa_geometry", "pwa_region_ids", "pwa_index_map", "pwa_attn_sel_table",
                    "pwa_partition", "pwa_reverse", "pwa_reverse_add", "pwa_gather_rows", "pwa_colsum_f32", "pwa_colsum_rows", "pwa_dropout", "pwa_dropout_colsum", "pwa_token_gemm_supported", "pwa_token_gemm_fwd", "pwa_token_gemm_fwd_dt", "pwa_attn_fwd", "pwa_attn_bwd", "pwa_attn_tc_supported", "pwa_attn_dense_fwd", "pwa_attn_dense_bwd",
                    "pwa_ln_fwd", "pwa_ln_bwd", "pwa_ln_bwd2", "pwa_bias_tables_fwd", "pwa_bias_tables_bwd")


def check(rc: int, what: str):
    if rc != 0:
        msg = lib.pwa_last_error().decode("utf-8", "replace")
        if rc == -1 and "not compatible with the number of heads" in msg:
            raise ValueError(msg)                      # same exception type as window_attention.py:19-22
        if rc == -2:
            raise NotImplementedError(f"{what}: {msg}")
        raise PwaError(f"{what} failed (rc={rc}): {msg}")
