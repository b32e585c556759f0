"""ctypes binding of liboffk.so (the C ABI declared in include/offk.h).

There is deliberately NO fallback: if the shared library is missing or a call
fails, a RuntimeError is raised.  PyTorch is used by the callers only for
device memory, streams and torch.distributed.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("OFFK_LIB") or os.path.join(_HERE, "liboffk.so")   # OFFK_LIB: bring-up builds only

PREC_TF32, PREC_TF32X3 = 1, 2
INDEX_REFERENCE_FLAT, INDEX_ALIGNED = 0, 1
DROP_NONE, DROP_MASK, DROP_SEED = 0, 1, 2
POOL_MAX, POOL_AVG = 0, 1
LOAD_VEC_K, LOAD_VEC_ROW = 2, 3


class OffkIdx(C.Structure):
    _fields_ = [("off", C.c_int32), ("y", C.c_int16), ("x", C.c_int16)]


class OffkGemm(C.Structure):
    """Mirror of offk_gemm_t."""
    _fields_ = [
        ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32),
        ("a_src", C.c_void_p), ("a_row", C.c_void_p), ("a_col", C.c_void_p),
        ("a_h", C.c_int32), ("a_w", C.c_int32), ("a_ones_row", C.c_int32), ("a_mode", C.c_int32),
        ("b_src", C.c_void_p), ("b_row", C.c_void_p), ("b_col", C.c_void_p), ("b_mode", C.c_int32),
        ("out", C.c_void_p), ("out_row", C.c_void_p), ("out_col", C.c_void_p),
        ("bias", C.c_void_p), ("relu_pre_cols", C.c_int32),
        ("gate", C.c_void_p), ("gate_col0", C.c_int32), ("gate_first", C.c_int32),
        ("addend", C.c_void_p), ("add_row", C.c_void_p), ("add_col", C.c_void_p),
        ("relu_post", C.c_int32), ("atomic_out", C.c_int32),
        ("ones_row_out", C.c_void_p),
        ("split_k", C.c_int32), ("tile_n", C.c_int32), ("out_vec", C.c_int32), ("reserved", C.c_int32),
        ("finish_counter", C.c_void_p), ("aux_out", C.c_void_p), ("aux_row", C.c_void_p), ("aux_addend", C.c_void_p),
    ]


class OffkTGemm(C.Structure):
    """Mirror of offk_tgemm_t."""
    _fields_ = [
        ("g", OffkGemm),
        ("a_kind", C.c_int32), ("lda", C.c_int32), ("a_coff", C.c_int32),
        ("n_img", C.c_int32), ("hin", C.c_int32), ("win", C.c_int32), ("ctot", C.c_int32), ("cin", C.c_int32),
        ("kh", C.c_int32), ("kw", C.c_int32), ("stride", C.c_int32), ("pad", C.c_int32), ("hout", C.c_int32),
        ("wout", C.c_int32),
        ("b_kind", C.c_int32), ("ldb", C.c_int32), ("prepared", C.c_int32), ("geom_flags", C.c_int32),
        ("pad_w", C.c_int32), ("precision", C.c_int32), ("bk", C.c_int32), ("reserved", C.c_int32),
        ("b_lo_delta", C.c_int64),
        ("out_ld", C.c_int32), ("out_c0", C.c_int32),
        ("tmap_a", C.c_uint64 * 16), ("tmap_b", C.c_uint64 * 16), ("tmap_c", C.c_uint64 * 16),
        ("c_mode", C.c_int32), ("reserved3", C.c_int32),
    ]


TMA_A_DENSE, TMA_A_IM2COL, TMA_A_NCHW, TMA_A_NCHW_T, TMA_A_IM2COL_T = 0, 1, 2, 3, 4
TMA_B_DENSE, TMA_B_DENSE_T = 0, 1
TGEMM_FREE_GEOM = 1


class OffkStencil(C.Structure):
    """Mirror of offk_stencil_t."""
    _fields_ = [
        ("B", C.c_int32), ("L", C.c_int32), ("Cg", C.c_int32), ("Cs", C.c_int32), ("K", C.c_int32),
        ("H", C.c_int32), ("W", C.c_int32),
        ("g_fs", C.c_int64), ("d_fs", C.c_int64), ("g_ps", C.c_int32), ("d_ps", C.c_int32),
        ("out_ctot", C.c_int32), ("out_coff", C.c_int32),
        ("index_mode", C.c_int32), ("drop_mode", C.c_int32),
        ("keep_scale", C.c_float), ("drop_p", C.c_float),
        ("seed", C.c_uint64), ("keep_mask", C.c_void_p), ("seed_dev", C.c_void_p),
    ]


class OffkStencilIO(C.Structure):
    """Mirror of offk_stencil_io_t."""
    _fields_ = [
        ("g", C.c_void_p), ("d", C.c_void_p), ("w", C.c_void_p), ("bias", C.c_void_p), ("out", C.c_void_p),
        ("dout", C.c_void_p), ("dg", C.c_void_p), ("dg_fs", C.c_int64), ("dd", C.c_void_p), ("dd_fs", C.c_int64),
        ("dw", C.c_void_p), ("dbias", C.c_void_p),
    ]


class OffkPermute(C.Structure):
    """Mirror of offk_permute_t."""
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("cout", C.c_int32), ("cin", C.c_int32), ("kh", C.c_int32),
                ("kw", C.c_int32)]


_P = C.c_void_p
_PROTOS = {
    "offk_version": (C.c_int, []),
    "offk_last_error_string": (C.c_char_p, []),
    "offk_device_info": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                   C.POINTER(C.c_longlong)]),
    "offk_gather_gemm": (C.c_int, [C.POINTER(OffkGemm), C.c_int, _P]),
    "offk_tma_gemm_prepare": (C.c_int, [C.POINTER(OffkTGemm)]),
    "offk_tma_gemm": (C.c_int, [C.POINTER(OffkTGemm), _P]),
    "offk_stencil_diff_fwd": (C.c_int, [C.POINTER(OffkStencil), _P, _P, _P, _P, _P, _P]),
    "offk_stencil_diff_bwd": (C.c_int, [C.POINTER(OffkStencil), _P, _P, _P, _P, _P, C.c_int64, _P, C.c_int64,
                                        _P, _P, _P]),
    "offk_stencil_diff_fwd_batch": (C.c_int, [C.c_int, C.POINTER(OffkStencil), C.POINTER(OffkStencilIO), _P]),
    "offk_stencil_diff_bwd_batch": (C.c_int, [C.c_int, C.POINTER(OffkStencil), C.POINTER(OffkStencilIO), _P]),
    "offk_avgpool_drop_fwd": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_uint64, _P,
                                        C.c_float, C.c_float, _P, _P]),
    "offk_head_fwd": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_uint64, _P, C.c_float,
                                C.c_float, _P, _P, C.c_int, C.c_int, _P, _P, _P, _P]),
    "offk_head_bwd": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_uint64, _P, C.c_float,
                                C.c_float, _P, C.c_int, C.c_int, _P, _P, C.c_int, _P, _P, _P, _P]),
    "offk_seed_set": (C.c_int, [_P, C.c_uint64, _P]),
    "offk_pool3_nhwc": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                  _P, C.c_int, C.c_int, _P]),
    "offk_segment_mean_fwd": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, _P]),
    "offk_segment_mean_bwd": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, _P]),
    "offk_fill_zero": (C.c_int, [_P, C.c_longlong, _P]),
    "offk_relu_gate": (C.c_int, [_P, _P, C.c_longlong, _P, _P]),
    "offk_gate_copy": (C.c_int, [_P, C.c_int, C.c_int, _P, C.c_int, C.c_int, _P, C.c_int, C.c_int, C.c_int, C.c_int,
                                 C.c_int, _P]),
    "offk_bias_act": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "offk_add_relu_slice": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "offk_nchw_to_nhwc": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "offk_image_to_nhwc": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "offk_gather_copy": (C.c_int, [_P, _P, _P, C.c_longlong, _P]),
    "offk_tf32_residual": (C.c_int, [_P, _P, C.c_longlong, _P]),
    "offk_permute_weight_batch": (C.c_int, [C.c_int, C.POINTER(OffkPermute), C.c_int, _P]),
    "offk_drop_keep_host": (C.c_int, [C.c_uint64, C.c_uint64, C.c_float]),
    "offk_ce_loss_fwd_bwd": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_float, _P, _P, _P]),
    "offk_grad_sumsq": (C.c_int, [_P, C.c_longlong, _P, _P]),
    "offk_clip_adam_step": (C.c_int, [_P, _P, _P, _P, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong), C.c_int, C.c_float,
                                      C.c_float, C.c_float, C.c_float, C.c_float, C.c_int, C.c_float, _P, _P]),
}

_lib = None


def exported_symbols():
    """Names include/offk.h declares (used by the CPU test that checks the .so exports them all)."""
    return list(_PROTOS)


def lib():
    """Load liboffk.so once.  Raises RuntimeError when it has not been built -- there is no CPU path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"liboffk.so not found at {LIB_PATH}: build it with `python -c 'import __graft_entry__ as g; "
                f"g.build()'` (nvcc, sm_100a). The OFF path has no CPU / PyTorch fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(code: int, what: str = "offk"):
    if code != 0:
        msg = lib().offk_last_error_string()
        raise RuntimeError(f"{what} failed with code {code}: {msg.decode() if msg else ''}")
