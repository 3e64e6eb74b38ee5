"""ctypes binding of libkrylov_b200.so (include/krylov_b200.h).

The library is the product; this module only declares its signatures.  It is
built in-tree by `make -C krylov.jl_b200` (see __graft_entry__.build()).
Loading fails loudly if the shared object is missing -- there is no fallback.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_PKG)                      # krylov.jl_b200/
SO_PATH = os.environ.get("KB200_LIB") or os.path.join(ROOT, "lib", "libkrylov_b200.so")   # KB200_LIB: A/B builds

KRYLOV_FLOAT32, KRYLOV_FLOAT64 = 0, 1
KRYLOV_CPU, KRYLOV_CUDA = 0, 1
KRYLOV_CG, KRYLOV_MINRES, KRYLOV_GMRES, KRYLOV_BICGSTAB = 0, 3, 8, 10
KRYLOV_FOM, KRYLOV_FGMRES, KRYLOV_CGS, KRYLOV_B200_CG_LANCZOS = 7, 9, 11, 100
KRYLOV_CR, KRYLOV_DIOM, KRYLOV_DQGMRES = 1, 5, 6
SOLVER_IDS = {"cg": KRYLOV_CG, "minres": KRYLOV_MINRES, "gmres": KRYLOV_GMRES, "bicgstab": KRYLOV_BICGSTAB,
              "fom": KRYLOV_FOM, "fgmres": KRYLOV_FGMRES, "cgs": KRYLOV_CGS, "cg_lanczos": KRYLOV_B200_CG_LANCZOS,
              "cr": KRYLOV_CR, "diom": KRYLOV_DIOM, "dqgmres": KRYLOV_DQGMRES}

MATVEC = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p, C.c_void_p)
BLOCK_MATVEC = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p)
CALLBACK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p)


class KrylovWorkspaceOptions(C.Structure):
    _fields_ = [("memory", C.c_int), ("window", C.c_int)]


class KrylovOptions(C.Structure):
    _fields_ = [("atol", C.c_double), ("rtol", C.c_double), ("itmax", C.c_int), ("verbose", C.c_int),
                ("lambda_", C.c_double), ("tau", C.c_double), ("nu", C.c_double), ("timemax", C.c_double),
                ("radius", C.c_double), ("restart", C.c_int), ("reorthogonalization", C.c_int),
                ("linesearch", C.c_int)]


class KrylovB200Options(C.Structure):
    _fields_ = [("history", C.c_int), ("ldiv", C.c_int), ("etol", C.c_double), ("conlim", C.c_double),
                ("fused", C.c_int), ("batch", C.c_int), ("callback", CALLBACK), ("callback_user", C.c_void_p),
                ("time_kernels", C.c_int), ("check_curvature", C.c_int), ("cr_gamma", C.c_double)]


class KrylovB200Stats(C.Structure):
    _fields_ = [("niter", C.c_int), ("solved", C.c_int), ("inconsistent", C.c_int), ("indefinite", C.c_int),
                ("npcCount", C.c_int), ("nresiduals", C.c_int), ("nAresiduals", C.c_int), ("nAcond", C.c_int),
                ("allocation_timer", C.c_double), ("timer", C.c_double), ("status", C.c_char * 96),
                ("Anorm", C.c_double)]


# every symbol include/krylov_b200.h declares: name -> (restype, argtypes)
_P, _I, _D, _LL = C.c_void_p, C.c_int, C.c_double, C.c_longlong
SIGNATURES = {
    "krylov_workspace_create": (_I, [_I, _I, _I, _I, _I, C.POINTER(KrylovWorkspaceOptions), C.POINTER(_P)]),
    "krylov_default_workspace_options": (KrylovWorkspaceOptions, []),
    "krylov_default_options": (KrylovOptions, []),
    "krylov_get_version": (None, [C.POINTER(_I)] * 3),
    "krylov_solve": (_I, [_P, MATVEC, MATVEC, MATVEC, MATVEC, _P, _P, _P, C.POINTER(KrylovOptions)]),
    "krylov_get_x": (_I, [_P, _P, _I]),
    "krylov_get_y": (_I, [_P, _P, _I]),
    "krylov_is_solved": (_I, [_P]),
    "krylov_niter": (_I, [_P]),
    "krylov_elapsed_time": (_D, [_P]),
    "krylov_warm_start": (_I, [_P, _P, _I]),
    "krylov_warm_start2": (_I, [_P, _P, _P, _I, _I]),
    "krylov_workspace_free": (_I, [_P]),
    "krylov_block_workspace_create": (_I, [_I, _I, _I, _I, _I, _I, C.POINTER(KrylovWorkspaceOptions), C.POINTER(_P)]),
    "krylov_block_solve": (_I, [_P, BLOCK_MATVEC, BLOCK_MATVEC, BLOCK_MATVEC, _P, _P, C.POINTER(KrylovOptions)]),
    "krylov_block_get_X": (_I, [_P, _P, _I, _I]),
    "krylov_block_is_solved": (_I, [_P]),
    "krylov_block_niter": (_I, [_P]),
    "krylov_block_elapsed_time": (_D, [_P]),
    "krylov_block_warm_start": (_I, [_P, _P, _I, _I]),
    "krylov_block_workspace_free": (_I, [_P]),
    "krylov_b200_block_qr_fallbacks": (_LL, [_P]),
    "krylov_b200_device_count": (_I, []),
    "krylov_b200_set_device": (_I, [_I]),
    "krylov_b200_last_error": (C.c_char_p, []),
    "krylov_b200_set_operator_csr": (_I, [_P, _I, _LL, _P, _P, _P, _I, _I, _I]),
    "krylov_b200_share_operator": (_I, [_P, _P]),
    "krylov_b200_attach_csr": (_I, [_P, _P]),
    "krylov_b200_operator_encoding": (_I, [_P]),
    "krylov_b200_set_preconditioner_diag": (_I, [_P, _I, _P, _I]),
    "krylov_b200_set_preconditioner_blockdiag": (C.c_int, [_P, C.c_int, C.c_int, _P, C.c_int]),
    "krylov_b200_default_options": (KrylovB200Options, []),
    "krylov_b200_set_options": (_I, [_P, C.POINTER(KrylovB200Options)]),
    "krylov_b200_get_stats": (_I, [_P, C.POINTER(KrylovB200Stats)]),
    "krylov_b200_get_history": (_I, [_P, _I, C.POINTER(_D), _I]),
    "krylov_b200_get_vector": (_I, [_P, C.c_char_p, C.POINTER(_P)]),
    "krylov_b200_get_kernel_times": (_I, [_P, C.POINTER(_D)]),
    "krylov_b200_launch_count": (_LL, [_P]),
    "krylov_b200_stream": (_P, [_P]),
    "krylov_b200_wait_stream": (C.c_int, [_P, _P]),
    "krylov_b200_dist_handle_bytes": (_I, []),
    "krylov_b200_dist_init": (_I, [_P, _I, _I, _I, _P, _P]),
    "krylov_b200_dist_set_push": (_I, [_P, _I, _P, _P]),
    "krylov_b200_dist_set_sendlist": (_I, [_P, _I, _P, _P, _P, _P, _LL]),
    "krylov_b200_dist_export": (_I, [_P, _P]),
    "krylov_b200_dist_import": (_I, [_P, _P]),
    "kb200_ctx_create": (_P, [_I]),
    "kb200_ctx_destroy": (None, [_P]),
    "kb200_sync": (_I, [_P]),
    "kb200_alloc": (_P, [_LL]),
    "kb200_free": (_I, [_P]),
    "kb200_h2d": (_I, [_P, _P, _LL]),
    "kb200_d2h": (_I, [_P, _P, _LL]),
    "kb200_dot": (_I, [_P, _I, _I, _P, _P, C.POINTER(_D)]),
    "kb200_nrm2": (_I, [_P, _I, _I, _P, C.POINTER(_D)]),
    "kb200_axpy": (_I, [_P, _I, _I, _D, _P, _P]),
    "kb200_axpby": (_I, [_P, _I, _I, _D, _P, _D, _P]),
    "kb200_scal": (_I, [_P, _I, _I, _D, _P]),
    "kb200_copy": (_I, [_P, _I, _I, _P, _P]),
    "kb200_scalcopy": (_I, [_P, _I, _I, _P, _D, _P]),
    "kb200_divcopy": (_I, [_P, _I, _I, _P, _P, _D]),
    "kb200_fill": (_I, [_P, _I, _I, _P, _D]),
    "kb200_csr_create": (_P, [_P, _I, _I, _LL, _P, _P, _P, _I, _I, _I]),
    "kb200_csr_destroy": (None, [_P]),
    "kb200_csr_read_mtx": (_P, [_P, C.c_char_p, _I]),
    "kb200_csr_transpose": (_P, [_P, _P]),
    "kb200_csr_info": (_I, [_P, C.POINTER(_I), C.POINTER(_LL)]),
    "kb200_csr_download": (_I, [_P, _P, _P, _P, _P]),
    "kb200_mtx_read": (_I, [C.c_char_p, C.POINTER(_I), C.POINTER(_LL), _P, _P, _P]),
    "kb200_host_householder": (_I, [_I, _I, _P, _P, _P, _I]),
    "kb200_host_cholqr_factors": (_I, [_I, _P, _P, _P]),
    "kb200_host_householder_signs": (_I, [_I, _P, _P]),
    "kb200_spmv_csr": (_I, [_P, _P, _P, _P, _I]),
    "kb200_csr_plan": (_I, [_P, C.POINTER(_LL)]),
}

_LIB = None


def build(verbose: bool = False) -> str:
    """Compile the CUDA extension for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", ROOT, "-j8"] + ([] if verbose else ["-s"])
    subprocess.check_call(cmd)
    return SO_PATH


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU fallback)")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            try:
                fn = getattr(L, name)
            except AttributeError:
                if os.environ.get("KB200_LIB"):      # an older A/B build may lack newer entry points
                    continue
                raise
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB


def last_error() -> str:
    return lib().krylov_b200_last_error().decode("utf-8", "replace")
