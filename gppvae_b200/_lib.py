"""ctypes binding of libgppvae_b200.so (the C ABI declared in include/gppvae_b200.h).

There is no CPU or torch fallback behind this module: if the shared library is absent and cannot
be built, importing the ops raises.  The library itself contains no torch types.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_uint32, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgppvae_b200.so")

GPP_WANT_BINV = 1
GPP_PLANES_COLSQ, GPP_PLANES_UNIT_BOUND = 1, 2
# scalar slots (enum gpp_scalar_slot)
S_V0, S_VN, S_LOGDETB, S_TRBINV, S_WNORM2, S_ROWCONST, S_XB2, S_QUAD, NSCAL = range(9)

GPP_MAX_DESIGNS = 16
# factored designs over one slot index (enum gpp_effect_kind)
EFFECT_KINDS = {"kr": 0, "object": 1, "view": 2}

_PF = c_void_p   # device pointers travel as void*
# HOST arrays (the k-design entries): of device pointers, of int64 leading dimensions, of int32 column counts
_PH, _I64H, _I32H = ctypes.POINTER(c_void_p), ctypes.POINTER(c_int64), ctypes.POINTER(c_int32)


def host_ptrs(ptrs):
    """HOST array of device pointers (None entries become NULL)."""
    return (c_void_p * len(ptrs))(*ptrs)


def host_i64(vals):
    return (c_int64 * len(vals))(*[int(v) for v in vals])


def host_i32(vals):
    return (c_int32 * len(vals))(*[int(v) for v in vals])


_SIGNATURES = {
    "gpp_version": (c_int, []),
    "gpp_last_error": (c_char_p, []),
    "gpp_gemm_engine": (c_char_p, []),
    "gpp_launch_count": (ctypes.c_uint64, []),
    "gpp_normalize_rows_fwd": (c_int, [_PF, c_int64, c_int64, _PF, c_void_p]),
    "gpp_normalize_rows_bwd": (c_int, [_PF, _PF, c_int64, c_int64, _PF, c_void_p]),
    "gpp_khatri_rao_fwd": (c_int, [_PF, c_int64, c_int32, _PF, c_int64, c_int32, _PF, _PF, c_int64, _PF, c_int64,
                                   c_void_p]),
    "gpp_khatri_rao_bwd": (c_int, [_PF, c_int64, _PF, c_int64, c_int32, _PF, c_int64, c_int32, _PF, _PF, c_int64,
                                   _PF, _PF, c_void_p]),
    "gpp_gram_workspace_bytes": (c_size_t, [c_int64, c_int32, c_int32]),
    "gpp_gram_vtz": (c_int, [_PF, c_int64, _PF, c_int64, c_int64, c_int32, c_int32, _PF, c_int64, _PF, c_size_t,
                             c_void_p]),
    "gpp_gram_vtz_simt": (c_int, [_PF, c_int64, _PF, c_int64, c_int64, c_int32, c_int32, _PF, c_int64, _PF, c_size_t,
                                  c_void_p]),
    "gpp_factor_state_bytes": (c_size_t, [c_int32]),
    "gpp_solve_workspace_bytes": (c_size_t, [c_int32, c_int32]),
    "gpp_factor": (c_int, [_PF, c_int64, c_int32, _PF, c_uint32, _PF, _PF, _PF, c_size_t, c_void_p]),
    "gpp_solve_w": (c_int, [_PF, c_int64, c_int32, c_int32, c_int32, c_int64, _PF, c_int64, _PF, _PF, c_size_t,
                            _PF, c_size_t, c_void_p]),
    "gpp_factor_solve": (c_int, [_PF, c_int64, c_int32, c_int32, _PF, c_int64, c_uint32, _PF, c_int64, _PF, _PF,
                                 _PF, c_size_t, c_void_p]),
    "gpp_xb_workspace_bytes": (c_size_t, [c_int64, c_int32, c_int32]),
    "gpp_xb_nll": (c_int, [_PF, c_int64, _PF, c_int64, _PF, c_int64, c_int64, c_int32, c_int32, _PF, _PF, c_int64,
                           _PF, _PF, c_size_t, c_void_p]),
    "gpp_vbs": (c_int, [_PF, c_int64, c_int32, c_int32, _PF, c_void_p]),
    "gpp_vb_workspace_bytes": (c_size_t, [c_int64, c_int32, c_int32]),
    "gpp_vb": (c_int, [_PF, c_int64, _PF, c_int64, _PF, _PF, c_int64, _PF, c_int64, c_int32, c_int32, c_int32, _PF,
                       c_int64, _PF, c_size_t, c_void_p]),
    "gpp_rows_workspace_bytes": (c_size_t, []),
    "gpp_x_minus_am": (c_int, [_PF, c_int64, _PF, c_int64, _PF, c_int64, c_int64, c_int32, c_int32, c_float, _PF,
                               c_int64, _PF, c_size_t, c_void_p]),
    "gpp_atb_workspace_bytes": (c_size_t, [c_int64, c_int32, c_int32]),
    "gpp_atb": (c_int, [_PF, c_int64, _PF, c_int64, c_int64, c_int32, c_int32, _PF, c_int64, _PF, c_size_t,
                        c_void_p]),
    "gpp_planes_bytes": (c_size_t, [c_int64, c_int32]),
    "gpp_split_workspace_bytes": (c_size_t, [c_int64, c_int32]),
    "gpp_planes_supported": (c_int, [c_int64, c_int32, c_int32]),
    "gpp_split_planes": (c_int, [_PF, c_int64, c_int64, c_int32, c_uint32, _PF, c_size_t, _PF, c_size_t, c_void_p]),
    "gpp_khatri_rao_fwd_planes": (c_int, [_PF, c_int64, c_int32, _PF, c_int64, c_int32, _PF, _PF, c_int64, _PF, c_int64,
                                          _PF, c_size_t, _PF, c_size_t, c_void_p]),
    "gpp_gram_planes_workspace_bytes": (c_size_t, [c_int64, c_int32, c_int32]),
    "gpp_gram_vtz_planes": (c_int, [_PF, _PF, c_int64, c_int32, c_int32, c_int32, _PF, c_int64, _PF, c_size_t,
                                    c_void_p]),
    "gpp_atb_planes": (c_int, [_PF, _PF, c_int64, c_int32, c_int32, _PF, c_int64, _PF, c_size_t, c_void_p]),
    "gpp_xb_planes_workspace_bytes": (c_size_t, [c_int64, c_int32, c_int32]),
    "gpp_xb_nll_planes": (c_int, [_PF, _PF, c_int64, _PF, c_int64, c_int64, c_int32, c_int32, _PF, _PF, c_int64, _PF,
                                  _PF, c_size_t, c_void_p]),
    "gpp_vb_planes_workspace_bytes": (c_size_t, [c_int64, c_int32, c_int32]),
    "gpp_vb_planes": (c_int, [_PF, _PF, c_int64, _PF, _PF, c_int64, _PF, c_int64, c_int32, c_int32, c_int32, _PF, c_int64,
                              _PF, c_size_t, c_void_p]),
    "gpp_am": (c_int, [_PF, c_int64, _PF, c_int64, c_int64, c_int32, c_int32, c_float, _PF, c_int64, _PF, c_size_t,
                       c_void_p]),
    "gpp_kr_slot_sums": (c_int, [_PF, c_int64, _PF, _PF, _PF, c_int64, c_int32, c_int32, c_int32, c_int32, _PF, c_int64,
                                 c_void_p]),
    "gpp_kr_slot_sums_planes": (c_int, [_PF, c_int64, c_int64, _PF, _PF, _PF, c_int64, c_int32, c_int32, c_int32, c_int32,
                                        c_int32, _PF, c_size_t, c_void_p]),
    "gpp_am_planes": (c_int, [_PF, _PF, c_int64, c_int32, c_int32, c_float, _PF, c_int64, _PF, c_size_t, c_void_p]),
    "gpp_kr_assemble_gc": (c_int, [_PF, c_int64, _PF, c_int32, c_int32, c_int32, c_int32, c_int32, _PF, c_int64,
                                   c_void_p]),
    "gpp_kr_assemble_m": (c_int, [_PF, c_int64, _PF, c_int32, c_int32, c_int32, c_int32, _PF, c_int64, c_void_p]),
    "gpp_kr_xb_workspace_bytes": (c_size_t, [c_int64]),
    "gpp_kr_xb_nll": (c_int, [_PF, c_int64, _PF, c_int64, _PF, _PF, c_int64, c_int64, c_int32, c_int32, _PF, _PF,
                              c_int64, _PF, _PF, c_size_t, c_void_p]),
    "gpp_kr_grad_rhs": (c_int, [_PF, c_int64, _PF, c_int64, _PF, c_int32, c_int32, c_int32, c_int32, c_double, _PF,
                                c_int64, c_void_p]),
    "gpp_kr_grad_views_workspace_bytes": (c_size_t, [c_int32, c_int32, c_int32]),
    "gpp_kr_grad_views": (c_int, [_PF, c_int64, _PF, c_int64, _PF, c_int64, _PF, c_int32, c_int32, c_int32, c_int32,
                                  c_double, _PF, c_int64, _PF, c_size_t, c_void_p]),
    "gpp_kr_view_sums_workspace_bytes": (c_size_t, [c_int64, c_int32, c_int32, c_int32, c_int32]),
    "gpp_kr_view_sums": (c_int, [_PF, c_int64, _PF, _PF, _PF, c_int64, c_int32, c_int32, c_int32, c_int32, _PF, c_int64,
                                 _PF, c_size_t, c_void_p]),
    "gpp_kr_assemble_gc_blocks": (c_int, [_PF, c_int64, _PF, c_int64, _PF, c_int32, c_int32, c_int32, c_int32, c_int32,
                                          _I32H, c_int32, _PF, c_int64, c_void_p]),
    "gpp_kr_assemble_m_blocks": (c_int, [_PF, c_int64, _PF, c_int32, c_int32, c_int32, c_int32, c_int32, _I32H, _PF,
                                         c_int64, _PF, c_int64, c_void_p]),
    "gpp_kr_xb_nll_views": (c_int, [_PF, c_int64, _PF, c_int64, _PF, c_int64, _PF, _PF, c_int64, c_int64, c_int32,
                                    c_int32, _PF, _PF, c_int64, _PF, _PF, c_size_t, c_void_p]),
    "gpp_kr_predict_views": (c_int, [_PF, c_int64, _PF, c_int32, c_int32, c_int32, c_int32, _I32H, _PF, c_int64, _PF,
                                     _PF, c_void_p]),
    "gpp_kr_predict_rows": (c_int, [_PF, c_int64, _PF, c_int64, _PF, c_int64, _PF, _PF, _PF, _PF, _PF, c_int64, c_int64,
                                    c_int32, c_int32, c_int32, _PF, _PF, c_int64, _PF, c_void_p]),
    "gpp_rows_dot": (c_int, [_PF, c_int64, _PF, c_int64, c_int64, c_int32, _PF, _PF, c_void_p]),
    "gpp_taylor_expansion_fwd": (c_int, [_PF, c_int64, _PF, c_int64, _PF, c_int64, _PF, c_int64, c_int64, c_int32,
                                         c_int32, _PF, _PF, _PF, c_void_p]),
    "gpp_taylor_expansion_bwd": (c_int, [_PF, _PF, c_int64, _PF, c_int64, c_int64, c_int32, c_int32, _PF, _PF, _PF,
                                         c_int64, _PF, c_int64, _PF, c_void_p]),
    "gpp_split_stacked_workspace_bytes": (c_size_t, [c_int64, c_int32, _I32H]),
    "gpp_split_planes_stacked": (c_int, [c_int32, _PH, _I64H, _I32H, c_int64, c_uint32, _PF, c_size_t, _PF, c_size_t,
                                         c_void_p]),
    "gpp_factor_blocks_state_bytes": (c_size_t, [c_int32, c_int32]),
    "gpp_factor_blocks": (c_int, [_PF, c_int64, c_int32, _I32H, _PF, c_uint32, _PF, _PF, _PF, _PF, c_size_t, c_void_p]),
    "gpp_solve_blocks_workspace_bytes": (c_size_t, [c_int32, c_int32, c_int32]),
    "gpp_solve_w_blocks": (c_int, [_PF, c_int64, c_int32, _I32H, c_int32, c_int32, c_int64, _PF, c_int64, _PF, _PF, _PF,
                                   c_size_t, _PF, c_size_t, c_void_p]),
    "gpp_vbs_blocks": (c_int, [_PF, _PF, _PF, c_int32, _I32H, c_int64, c_int32, _PF, c_void_p]),
    "gpp_taylor_expansion_fwd_multi": (c_int, [_PF, c_int64, _PF, c_int64, c_int32, _PH, _I64H, _PH, _I64H, _I32H, c_int64,
                                               c_int32, _PF, _PF, _PF, c_void_p]),
    "gpp_taylor_expansion_bwd_multi": (c_int, [_PF, _PF, c_int64, c_int32, _PH, _I64H, _I32H, c_int64, c_int32, _PF, _PF,
                                               _PF, c_int64, _PH, _I64H, _PF, c_void_p]),
    "gpp_host_ctx_create": (c_int, [ctypes.POINTER(c_void_p)]),
    "gpp_host_ctx_destroy": (c_int, [c_void_p]),
    "gpp_gp_term_host_submit": (c_int, [c_void_p, _PF, c_int64, c_int32, _PF, c_int64, c_int32, _PF, _PF, _PF, c_int64,
                                        c_int32, _PF, _PF, _PF, _PF, ctypes.POINTER(c_int32)]),
    "gpp_gp_term_host_wait": (c_int, [c_void_p, c_int32]),
    "gpp_gp_term_host": (c_int, [c_void_p, _PF, c_int64, c_int32, _PF, c_int64, c_int32, _PF, _PF, _PF, c_int64,
                                 c_int32, _PF, _PF, _PF, _PF]),
}
EXPORTED_SYMBOLS = tuple(sorted(_SIGNATURES))

_lib = None


class GppError(RuntimeError):
    """A libgppvae_b200 call returned a negative status; carries the C-side message."""


def load(build_if_missing: bool = True) -> ctypes.CDLL:
    """Load (and on first use, if needed, build) the shared library.  Raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if not build_if_missing:
            raise ImportError(f"{LIB_PATH} is missing; run `python -m gppvae_b200.build`")
        from . import build as _build   # compiles with nvcc; raises if nvcc is absent
        _build.build()
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load().gpp_last_error()
        raise GppError(f"{what} failed with status {status}: {msg.decode() if msg else '?'}")


def launch_count() -> int:
    return int(load().gpp_launch_count())


def gemm_engine() -> str:
    return load().gpp_gemm_engine().decode()
