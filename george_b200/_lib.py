# -*- coding: utf-8 -*-
"""
ctypes binding of the C ABI in ``include/bgp.h`` (``george_b200/lib/libbgp_b200.so``).

There is NO CPU fallback: if the shared library is missing, or no sm_100 device is visible when a compute
entry point is called, the call raises.  Status codes are mapped to the exception types the reference raises
for the same conditions (SURVEY.md §8b): ``numpy.linalg.LinAlgError`` for a non positive-definite matrix
(what ``scipy.linalg.cholesky`` raises in ``solvers/basic.py:68``), ``ValueError`` for an invalid kernel
(``std::invalid_argument``, ``parser.h:16``), ``RuntimeError`` for dimension mismatch / not-computed
(``exceptions.h:8-18``), ``IndexError`` for out-of-range access (``_hodlr.cpp:26``).
"""

import ctypes as C
import os

import numpy as np

from ._spec import HodlrNodeInfo, HodlrOpts, KernelSpec

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libbgp_b200.so")

BGP_OK, BGP_ERR_INVALID, BGP_ERR_DIM, BGP_ERR_NOT_COMPUTED, BGP_ERR_LINALG = 0, 1, 2, 3, 4
BGP_ERR_CUDA, BGP_ERR_NO_DEVICE, BGP_ERR_RANK_CAPACITY, BGP_ERR_INDEX, BGP_ERR_NOMEM = 5, 6, 7, 8, 9


class BGPError(RuntimeError):
    """CUDA / device failure inside libbgp_b200 (there is no fallback path)."""


class RankCapacityError(BGPError):
    """The ACA rank of a node exceeded the configured per-level capacity."""


_lib = None

_p = C.c_void_p
_dp = C.POINTER(C.c_double)
_i64 = C.c_int64
_i32 = C.c_int32
_specp = C.POINTER(KernelSpec)

# name -> (restype, argtypes); must list every symbol include/bgp.h declares (tests/test_abi.py checks it)
SIGNATURES = {
    "bgp_last_error": (C.c_char_p, []),
    "bgp_version": (C.c_int, []),
    "bgp_device_count": (C.c_int, []),
    "bgp_set_device": (C.c_int, [C.c_int]),
    "bgp_launch_count": (C.c_uint64, []),
    "bgp_spec_validate": (C.c_int, [_specp]),
    "bgp_spec_num_params": (C.c_int, [_specp, C.POINTER(C.c_int)]),
    "bgp_kmat_symmetric": (C.c_int, [_specp, _p, _i64, _p]),
    "bgp_kmat_general": (C.c_int, [_specp, _p, _i64, _p, _i64, _p]),
    "bgp_kmat_diagonal": (C.c_int, [_specp, _p, _p, _i64, _p]),
    "bgp_kmat_gradient_symmetric": (C.c_int, [_specp, _p, _p, _i64, _p]),
    "bgp_kmat_gradient_general": (C.c_int, [_specp, _p, _p, _i64, _p, _i64, _p]),
    "bgp_kmat_x1_gradient_general": (C.c_int, [_specp, _p, _i64, _p, _i64, _p]),
    "bgp_kmat_x2_gradient_general": (C.c_int, [_specp, _p, _i64, _p, _i64, _p]),
    "bgp_kmat_matvec": (C.c_int, [_specp, _p, _i64, _p, _i64, _p, _p, _i64, _p]),
    "bgp_kmat_gradient_contract": (C.c_int, [_specp, _p, _p, _i64, _p, _p]),
    "bgp_dense_grad_terms": (C.c_int, [_p, _p, _p, _p, _p, _p]),
    "bgp_hodlr_grad_terms": (C.c_int, [_p, _p, _p, _p, _p, _p]),
    "bgp_dense_create": (C.c_int, [C.POINTER(_p)]),
    "bgp_dense_destroy": (None, [_p]),
    "bgp_dense_compute": (C.c_int, [_p, _specp, _p, _i64, _i32, _p]),
    "bgp_dense_log_determinant": (C.c_int, [_p, _dp]),
    "bgp_dense_apply_inverse": (C.c_int, [_p, _p, _i64, _i64]),
    "bgp_dense_dot_solve": (C.c_int, [_p, _p, _dp]),
    "bgp_dense_apply_sqrt": (C.c_int, [_p, _p, _i64, _p]),
    "bgp_dense_get_inverse": (C.c_int, [_p, _p]),
    "bgp_dense_export_factor": (C.c_int, [_p, _p]),
    "bgp_dense_import_factor": (C.c_int, [_p, _p, _i64, C.c_double]),
    "bgp_dense_last_timing": (C.c_int, [_p, _dp]),
    "bgp_hodlr_default_opts": (None, [C.POINTER(HodlrOpts)]),
    "bgp_hodlr_create": (C.c_int, [C.POINTER(_p)]),
    "bgp_hodlr_destroy": (None, [_p]),
    "bgp_hodlr_compute": (C.c_int, [_p, _specp, _p, _i64, _i32, _p, C.POINTER(HodlrOpts)]),
    "bgp_hodlr_compute_dev": (C.c_int, [_p, _specp, _p, _i64, _i32, _p, C.POINTER(HodlrOpts)]),
    "bgp_hodlr_computed": (C.c_int, [_p]),
    "bgp_hodlr_log_determinant": (C.c_int, [_p, _dp]),
    "bgp_hodlr_apply_inverse": (C.c_int, [_p, _p, _i64, _i64]),
    "bgp_hodlr_dot_solve": (C.c_int, [_p, _p, _dp]),
    "bgp_hodlr_dot_solve_dev": (C.c_int, [_p, _p, _dp]),
    "bgp_hodlr_get_inverse": (C.c_int, [_p, _p]),
    "bgp_hodlr_num_nodes": (C.c_int, [_p, C.POINTER(_i64)]),
    "bgp_hodlr_node_info": (C.c_int, [_p, C.POINTER(HodlrNodeInfo)]),
    "bgp_hodlr_node_pivots": (C.c_int, [_p, _i64, _p, _p]),
    "bgp_hodlr_last_timing": (C.c_int, [_p, _dp]),
    "bgp_hodlr_last_work": (C.c_int, [_p, _dp]),
    "bgp_hodlr_set_profiling": (C.c_int, [_p, C.c_int]),
    "bgp_hodlr_last_aca_profile": (C.c_int, [_p, _dp]),
    "bgp_selftest_lu": (C.c_int, [_i32, _i32, _p, _p, _p]),
    "bgp_selftest_gemm": (C.c_int, [_i32, _i32, _i32, _i32, _i32, _p, _i64, _p, _i64, _p, _i64, _i32]),
    "bgp_comm_unique_id": (C.c_int, [_p, C.c_char_p]),
    "bgp_comm_init": (C.c_int, [_p, C.c_int, C.c_int, C.c_char_p]),
    "bgp_comm_destroy": (C.c_int, []),
    "bgp_dev_alloc": (C.c_int, [C.POINTER(_p), C.c_size_t]),
    "bgp_dev_free": (C.c_int, [_p]),
    "bgp_dev_upload": (C.c_int, [_p, _p, C.c_size_t]),
    "bgp_host_alloc_pinned": (C.c_int, [C.POINTER(_p), C.c_size_t]),
    "bgp_host_free_pinned": (C.c_int, [_p]),
}


def load():
    """Load libbgp_b200.so (once).  Raises ImportError loudly if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "george_b200: the CUDA library {0} is missing. Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
            "There is no CPU fallback.".format(LIB_PATH))
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means the .so is stale w.r.t. include/bgp.h
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    msg = load().bgp_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(status):
    """Translate a non-zero status into the reference's exception type."""
    if status == BGP_OK:
        return
    msg = last_error()
    if status == BGP_ERR_INVALID:
        raise ValueError(msg or "invalid kernel")
    if status in (BGP_ERR_DIM, BGP_ERR_NOT_COMPUTED):
        raise RuntimeError(msg or "dimension mismatch")
    if status == BGP_ERR_LINALG:
        raise np.linalg.LinAlgError(msg or "matrix is not positive definite")
    if status == BGP_ERR_INDEX:
        raise IndexError(msg)
    if status == BGP_ERR_NOMEM:
        raise MemoryError(msg)
    if status == BGP_ERR_RANK_CAPACITY:
        raise RankCapacityError(msg)
    raise BGPError("libbgp_b200 status {0}: {1}".format(status, msg))


def ptr(a):
    """Raw data pointer of a numpy array (must stay alive for the duration of the call)."""
    return C.c_void_p(a.ctypes.data)
