"""ctypes binding of libcgx_b200.so (the C ABI declared in include/cgx.h).

There is no CPU fallback: if the shared library cannot be loaded, or no CUDA device is
visible when a context is created, the call raises.  The library is built in-tree by
``new_cg_variants_b200.build`` (nvcc, sm_100a) and loaded from this directory.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)

OK, ERR_ARG, ERR_CUDA, ERR_BREAKDOWN, ERR_UNSUPPORTED = 0, 1, 2, 3, 4

VARIANT_IDS = {"hs": 0, "cg": 1, "gv": 2, "pr": 3, "m": 4, "pipe_pr": 5, "pipe_p": 6,
               "pipe_pr_m": 7, "pipe_p_m": 8}
HIST_NAMES = ("error_A_norm", "residual_2_norm", "error_2_norm", "updated_residual_2_norm")
HIST_BITS = {name: 1 << i for i, name in enumerate(HIST_NAMES)}
PATHS = {"auto": 0, "stream": 1, "persistent": 2}


class CgxInfo(C.Structure):
    _fields_ = [("loop_ms", C.c_double), ("setup_ms", C.c_double), ("h2d_bytes", C.c_double),
                ("d2h_bytes", C.c_double), ("kernel_launches", C.c_int64),
                ("iterations", C.c_int32), ("breakdown_iter", C.c_int32), ("path", C.c_int32),
                ("stop_iter", C.c_int32)]

    def as_dict(self):
        return {f: getattr(self, f) for f, _ in self._fields_}


class CgxError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libcgx_b200 error {code}: {msg}")
        self.code = code


# name -> (restype, argtypes); must list every function declared in include/cgx.h
# (tests/test_abi.py parses the header and checks this table and the .so against it).
_P = C.c_void_p
PROTOTYPES = {
    "cgx_version": (C.c_int, []),
    "cgx_last_error": (C.c_char_p, []),
    "cgx_device_count": (C.c_int, []),
    "cgx_ctx_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "cgx_ctx_destroy": (C.c_int, [_P]),
    "cgx_set_csr_host": (C.c_int, [_P, C.c_int64, C.c_int64, c_int32_p, c_int32_p, c_double_p]),
    "cgx_set_stencil": (C.c_int, [_P, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_double, C.c_double]),
    "cgx_set_stencil_coef_host": (C.c_int, [_P, C.c_int, C.c_int64, C.c_int64, C.c_int64, c_double_p, c_double_p,
                                            c_double_p, c_double_p]),
    "cgx_set_jacobi_host": (C.c_int, [_P, c_double_p, C.c_int64]),
    "cgx_load_problem_host": (C.c_int, [_P, c_double_p, c_double_p, c_double_p, C.c_int64]),
    "cgx_load_problem_dev": (C.c_int, [_P, _P, _P, _P, C.c_int64]),
    "cgx_run": (C.c_int, [_P, C.c_int, C.c_int, C.c_uint, C.c_int, C.POINTER(CgxInfo)]),
    "cgx_begin": (C.c_int, [_P, C.c_int, C.c_int, C.c_uint, C.c_int]),
    "cgx_advance": (C.c_int, [_P, C.c_int]),
    "cgx_get_info": (C.c_int, [_P, C.POINTER(CgxInfo)]),
    "cgx_get_scalars": (C.c_int, [_P, c_double_p]),
    "cgx_set_option": (C.c_int, [_P, C.c_char_p, C.c_int]),
    "cgx_set_tolerance": (C.c_int, [_P, C.c_double]),
    "cgx_debug_times": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "cgx_set_profile": (C.c_int, [_P, C.c_int]),
    "cgx_get_profile": (C.c_int, [_P, C.c_int, c_double_p, C.POINTER(C.c_int64)]),
    "cgx_profile_class_name": (C.c_char_p, [C.c_int]),
    "cgx_profile_class_count": (C.c_int, []),
    "cgx_fetch_host": (C.c_int, [_P, c_double_p, c_double_p]),
    "cgx_fetch_dev": (C.c_int, [_P, _P, _P]),
    "cgx_fetch_vector_host": (C.c_int, [_P, C.c_char_p, c_double_p]),
    "cgx_set_csr_part_host": (C.c_int, [_P, C.c_int64, C.c_int64, C.c_int64, c_int32_p, c_int32_p, c_double_p, C.c_int, C.c_int,
                                        c_int32_p, c_int32_p, c_int32_p, c_int32_p, c_int32_p]),
    "cgx_set_capture": (C.c_int, [_P, C.c_uint]),
    "cgx_fetch_capture_host": (C.c_int, [_P, C.c_int, c_double_p]),
    "cgx_set_gv_replace": (C.c_int, [_P, C.POINTER(C.c_uint8), C.c_int]),
    "cgx_advance_stages": (C.c_int, [_P, C.c_int]),
    "cgx_gv_replace_now": (C.c_int, [_P]),
    "cgx_solve_host": (C.c_int, [_P, C.c_int, c_double_p, c_double_p, c_double_p, C.c_int64, C.c_int,
                                 C.c_uint, C.c_int, c_double_p, c_double_p, C.POINTER(CgxInfo)]),
    "cgx_set_stencil_slab": (C.c_int, [_P, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_double, C.c_double]),
    "cgx_dist_ipc_handle": (C.c_int, [_P, _P]),
    "cgx_dist_attach_ipc": (C.c_int, [_P, C.c_int, _P]),
    "cgx_dist_attach_ctx": (C.c_int, [_P, C.c_int, _P]),
    "cgx_dist_nccl_unique_id": (C.c_int, [C.c_char_p, _P]),
    "cgx_dist_commit": (C.c_int, [_P, C.c_int, C.c_char_p, _P]),
    "cgx_group_load_problem_host": (C.c_int, [C.POINTER(_P), C.c_int, c_double_p, c_double_p, c_double_p, C.c_int64]),
    "cgx_group_begin": (C.c_int, [C.POINTER(_P), C.c_int, C.c_int, C.c_int, C.c_uint, C.c_int]),
    "cgx_group_advance": (C.c_int, [C.POINTER(_P), C.c_int, C.c_int]),
    "cgx_batch_run": (C.c_int, [C.POINTER(_P), C.c_int, c_int32_p, c_int32_p, C.c_uint, C.POINTER(CgxInfo)]),
    "cgx_spmv_host": (C.c_int, [_P, c_double_p, c_double_p, C.c_int64]),
    "cgx_dot_host": (C.c_int, [_P, c_double_p, c_double_p, C.c_int64, c_double_p]),
}

_lib = None


def lib_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = True):
    """Load (building first if needed) the shared library; raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path) and not build_if_missing:
        raise CgxError(ERR_CUDA, f"{path} is missing; run `python -m new_cg_variants_b200.build`")
    # never load a binary older than its sources: rebuild when a compiler is here (a no-op when the
    # source stamp matches), otherwise refuse a stale library
    try:
        _build.build()
    except RuntimeError as e:
        if "nvcc not found" not in str(e):
            raise
        stamp = open(_build.STAMP).read().strip() if os.path.exists(_build.STAMP) else ""
        if not os.path.exists(path) or stamp != _build._fingerprint():
            raise CgxError(ERR_CUDA, f"{path} is missing or older than csrc/ and nvcc is not available to rebuild it")
    lib = C.CDLL(path)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)   # AttributeError here = ABI mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, allow_breakdown: bool = False) -> int:
    if rc == OK or (allow_breakdown and rc == ERR_BREAKDOWN):
        return rc
    msg = load().cgx_last_error()
    raise CgxError(rc, msg.decode() if msg else "")


def check_tol(tol) -> float:
    """A relative tolerance as cgx_set_tolerance takes it: 0 (off) or 0 < tol < 1, else ValueError."""
    t = float(tol)
    if not (t == 0.0 or 0.0 < t < 1.0):
        raise ValueError(f"tol must be 0 (off) or satisfy 0 < tol < 1, got {tol!r}")
    return t


def dptr(a: np.ndarray | None):
    """float64 C-contiguous host array -> double* (None -> NULL)."""
    if a is None:
        return None
    assert a.dtype == np.float64 and a.flags.c_contiguous
    return a.ctypes.data_as(c_double_p)


def iptr(a: np.ndarray):
    assert a.dtype == np.int32 and a.flags.c_contiguous
    return a.ctypes.data_as(c_int32_p)
