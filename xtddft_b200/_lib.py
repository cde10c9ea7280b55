"""ctypes binding of libxtdsigma.so (include/xtd_sigma.h).  Fails loudly: there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libxtdsigma.so")

XTD_FXC_NONE, XTD_FXC_UKS, XTD_FXC_ALDA0, XTD_FXC_MCOL, XTD_FXC_UKS_TAU, XTD_FXC_MCOL_TAU = 0, 1, 2, 3, 4, 5
XTD_SIDE_RIGHT, XTD_SIDE_LEFT, XTD_SIDE_LEFT_T, XTD_SIDE_RIGHT_T = 0, 1, 2, 3
T_NAMES = ["pack", "xc_gemm", "xc_stream", "k1", "k2", "j", "local", "unpack", "total", "k2_slice", "xc_slice"]


class XtdError(RuntimeError):
    pass


ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_long)


class XtdSolverOpts(C.Structure):
    _fields_ = [("tol", C.c_double), ("tol_residual", C.c_double), ("lindep", C.c_double), ("level_shift", C.c_double),
                ("max_cycle", C.c_int), ("max_space", C.c_int), ("pick_positive", C.c_int), ("allreduce", ALLREDUCE_FN),
                ("allreduce_ctx", C.c_void_p)]


class XtdStats(C.Structure):
    _fields_ = [("flops_gemm", C.c_double), ("launches", C.c_ulonglong), ("ms", C.c_double * 12), ("flops", C.c_double * 12)]


_P = C.c_void_p
_I, _L, _D = C.c_int, C.c_long, C.c_double

# every symbol include/xtd_sigma.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "xtd_last_error": (C.c_char_p, []),
    "xtd_version": (_I, []),
    "xtd_create": (_I, [C.POINTER(_P), _I, _L]),
    "xtd_destroy": (_I, [_P]),
    "xtd_set_stream": (_I, [_P, _P]),
    "xtd_set_mo": (_I, [_P, _I, _P, _L, _I]),
    "xtd_add_channel": (_I, [_P, _I, _P, _I, _I, _P, _I, _P, _I, _P, _I]),
    "xtd_channel_layout": (_I, [_P, _I, _I, C.POINTER(_L), C.POINTER(_L), C.POINTER(_L)]),
    "xtd_add_kterm": (_I, [_P, _I, _I, _P, _I, _I]),
    "xtd_add_kterm_t": (_I, [_P, _I, _I, _D]),
    "xtd_add_jblock": (_I, [_P, _I, _I, _I, _I, _I]),
    "xtd_set_jmix": (_I, [_P, _P, _I]),
    "xtd_set_exchange_emulation": (_I, [_P, _I]),
    "xtd_set_open_orbitals": (_I, [_P, _I, _P, _I]),
    "xtd_get_kopen": (_I, [_P, _P, _L]),
    "xtd_df_begin": (_I, [_P, _I, _L]),
    "xtd_df_add": (_I, [_P, _I, _P, _L, _L, _L, _I]),
    "xtd_jblock_diag": (_I, [_P, _I, _P]),
    "xtd_set_grid": (_I, [_P, _P, _I, _L, _L, _L, _P]),
    "xtd_set_fxc": (_I, [_P, _I, _P]),
    "xtd_grid_commit": (_I, [_P]),
    "xtd_add_local_gemm": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _I, _I, _D]),
    "xtd_add_rank1": (_I, [_P, _I, _P, _I, _P]),
    "xtd_add_diag": (_I, [_P, _I, _P]),
    "xtd_set_gather": (_I, [_P, _I, _P, _P, _P, _L]),
    "xtd_set_scatter": (_I, [_P, _L, _P, _P, _P, _P, _L]),
    "xtd_finalize": (_I, [_P, _I]),
    "xtd_sigma": (_I, [_P, _I, _P, _P]),
    "xtd_sigma_partial": (_I, [_P, _I, _P]),
    "xtd_partial_buffer": (_I, [_P, _I, C.POINTER(_P), C.POINTER(_L)]),
    "xtd_sigma_finish": (_I, [_P, _I, _P]),
    "xtd_sigma_host": (_I, [_P, _I, _P, _P]),
    "xtd_get_stats": (_I, [_P, C.POINTER(XtdStats)]),
    "xtd_reset_stats": (_I, [_P]),
    "xtd_xc_split_form": (_I, [_P, _I]),
    "xtd_last_chunks": (_I, [_P, C.POINTER(_L), C.POINTER(_L)]),
    "xtd_enable_block_response": (_I, [_P]),
    "xtd_block_response": (_I, [_P, _P, _P, _P, _P, _P]),
    "xtd_block_response_batch": (_I, [_P, _I, _P, _P, _P, _P, _P]),
    "xtd_last_density_batches": (_I, [_P, C.POINTER(_L)]),
    "xtd_vec_dots": (_I, [_P, _P, _I, _P, _L, _I, _P, _L, _I, _L]),
    "xtd_vec_lincomb": (_I, [_P, _P, _L, _P, _L, _P, _I, _I, _I, _L, _D]),
    "xtd_vec_residual": (_I, [_P, _P, _P, _P, _L, _P, _P, _I, _L]),
    "xtd_vec_precond": (_I, [_P, _P, _L, _P, _P, _P, _I, _L]),
    "xtd_vec_scale": (_I, [_P, _P, _L, _P, _I, _L]),
    "xtd_davidson": (_I, [_P, _I, C.POINTER(XtdSolverOpts), _P, _P, _I, _P, _P, _P, C.POINTER(_I), C.POINTER(_I)]),
    "xtd_host_sym_eig": (_I, [_P, _I, _P]),
    "xtd_host_gs_coefficients": (_I, [_P, _I, _D, _P]),
    "xtd_dgemm_tn": (_I, [_P, _I, _I, _I, _D, _P, _L, _P, _L, _P, _L, _I]),
    "xtd_dgemm": (_I, [_P, _I, _I, _I, _D, _P, _L, _I, _P, _L, _I, _P, _L, _I]),
    "xtd_ozaki_gemm": (_I, [_P, _I, _I, _I, _I, _I, _I, _P, _L, _L, _P, _L, _L, _P, _L, _D, _I, _P]),
    "xtd_launch_count": (C.c_ulonglong, []),
}

_lib = None


def load(path: str = LIB_PATH):
    """Load the shared library and bind every declared symbol; raises if the library or a symbol is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(path):
        raise XtdError(f"{path} not found: build it with `python -m xtddft_b200.build` (nvcc, sm_100a). "
                       "There is no CPU fallback for the sigma path.")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)           # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc < 0:
        msg = load().xtd_last_error()
        raise XtdError(f"{what} failed with code {rc}: {msg.decode() if msg else ''}")
    return rc
