"""ctypes binding of libtaxidispatch.so (include/taxidispatch.h).  No CPU fallback: importing the
compute surface without the built library raises, and every compute call without a CUDA device
returns TD_ERR_NO_DEVICE which is raised as TaxiDispatchError."""
from __future__ import annotations

import ctypes
import os

from . import build as _build

TD_OK = 0
TD_ERR_INVALID = -1
TD_ERR_CUDA = -2
TD_ERR_WORKSPACE = -3
TD_ERR_CAPACITY = -4
TD_ERR_NO_DEVICE = -5
TD_ERR_NOT_CONVERGED = -6
INT32_MAX = 2**31 - 1
BIG_COST = 250000
PAIRS_EXACT_MAX_N = 4096    # TD_PAIRS_EXACT_MAX_N
PAIRS_BATCH_MAX_N = 4096    # TD_PAIRS_BATCH_MAX_N
POOL_BATCH_MAX_N = 512      # TD_POOL_BATCH_MAX_N
BATCH_LARGE_MAX_N = 2048    # TD_BATCH_LARGE_MAX_N
STANDS_MAX_S = 128          # TD_STANDS_MAX_S
POOL_REC_W = 9
PROF_COST, PROF_LCM, PROF_ASSIGN, PROF_POOL_ENUM, PROF_POOL_SELECT = range(5)

c_i32p = ctypes.c_void_p
c_vp = ctypes.c_void_p


class LcmParams(ctypes.Structure):
    _fields_ = [("mask_value", ctypes.c_int32), ("stop_above", ctypes.c_int32), ("stop_at_value", ctypes.c_int32),
                ("sum_below", ctypes.c_int32), ("residual_size", ctypes.c_int32), ("max_iters", ctypes.c_int32)]


class AssignStats(ctypes.Structure):
    _fields_ = [("objective", ctypes.c_int64), ("rows_scanned", ctypes.c_int64), ("auction_rounds", ctypes.c_int32),
                ("phases", ctypes.c_int32), ("search_steps", ctypes.c_int32), ("augmentations", ctypes.c_int32),
                ("unassigned_after_auction", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class AssignCertificate(ctypes.Structure):
    _fields_ = [("min_reduced_cost", ctypes.c_int64), ("max_matched_slack", ctypes.c_int64), ("dual_objective", ctypes.c_int64),
                ("matched_real_cost", ctypes.c_int64), ("sign_violations", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class PoolStats(ctypes.Structure):
    _fields_ = [("evaluated", ctypes.c_int64), ("feasible", ctypes.c_int64), ("kept", ctypes.c_int64),
                ("rounds", ctypes.c_int32), ("passes", ctypes.c_int32)]


class TaxiDispatchError(RuntimeError):
    def __init__(self, code: int, where: str, detail: str = ""):
        self.code = code
        super().__init__("%s failed: %s (code %d)%s" % (where, strerror(code), code, (" -- " + detail) if detail else ""))


# every symbol include/taxidispatch.h declares: name -> (restype, argtypes)
_I = ctypes.c_int
_SIGNATURES = {
    "td_version": (ctypes.c_char_p, []),
    "td_strerror": (ctypes.c_char_p, [_I]),
    "td_last_cuda_error": (ctypes.c_char_p, []),
    "td_device_count": (_I, []),
    "td_launch_count": (ctypes.c_int64, []),
    "td_launch_count_reset": (None, []),
    "td_prof_enable": (None, [_I]),
    "td_prof_reset": (None, []),
    "td_prof_read": (_I, [_I, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64)]),
    "td_cost_matrix": (_I, [c_vp, _I, c_vp, _I, c_vp, _I, ctypes.c_int32, ctypes.c_int32, c_vp, c_vp]),
    "td_cost_matrix_rows": (_I, [c_vp, _I, c_vp, _I, c_vp, _I, ctypes.c_int32, ctypes.c_int32, _I, _I, c_vp, c_vp]),
    "td_lcm_workspace_bytes": (ctypes.c_size_t, [_I]),
    "td_lcm": (_I, [c_vp, _I, ctypes.POINTER(LcmParams), c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, ctypes.c_size_t, c_vp]),
    "td_assign_workspace_bytes": (ctypes.c_size_t, [_I]),
    "td_assign_exact": (_I, [c_vp, _I, c_vp, c_vp, c_vp, ctypes.POINTER(AssignStats), c_vp, ctypes.c_size_t, c_vp]),
    "td_assign_rect_workspace_bytes": (ctypes.c_size_t, [_I, _I, _I]),
    "td_assign_exact_rect": (_I, [c_vp, _I, _I, _I, c_vp, c_vp, c_vp, ctypes.POINTER(AssignStats), c_vp, ctypes.c_size_t, c_vp]),
    "td_assign_read_duals": (_I, [c_vp, _I, _I, _I, c_vp, c_vp, c_vp]),
    "td_assign_certify_workspace_bytes": (ctypes.c_size_t, [_I]),
    "td_assign_certify": (_I, [c_vp, _I, _I, _I, c_vp, c_vp, c_vp, c_vp, c_vp, ctypes.c_size_t, c_vp]),
    "td_assign_exact_batch": (_I, [c_vp, c_vp, c_vp, _I, _I, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "td_lcm_batch": (_I, [c_vp, c_vp, c_vp, _I, _I, ctypes.POINTER(LcmParams), c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "td_assign_exact_batch_cluster": (_I, [c_vp, c_vp, c_vp, _I, _I, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "td_lcm_batch_cluster": (_I, [c_vp, c_vp, c_vp, _I, _I, ctypes.POINTER(LcmParams), c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "td_assign_exact_batch_large": (_I, [c_vp, c_vp, c_vp, _I, _I, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "td_lcm_batch_large": (_I, [c_vp, c_vp, c_vp, _I, _I, ctypes.POINTER(LcmParams), c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "td_pool_workspace_bytes":(ctypes.c_size_t, [_I, _I, _I, ctypes.c_int64]),
    "td_pool_find": (_I, [c_vp, _I, c_vp, _I, _I, _I, _I, c_vp, ctypes.c_int32, c_vp, ctypes.POINTER(PoolStats),
                          c_vp, ctypes.c_size_t, ctypes.c_int64, c_vp]),
    "td_pool_shards_workspace_bytes": (ctypes.c_size_t, [_I, _I, _I, _I, ctypes.c_int64]),
    "td_pool_find_shards": (_I, [c_vp, _I, c_vp, _I, _I, _I, _I, _I, c_vp, ctypes.c_int32, c_vp, ctypes.POINTER(PoolStats),
                                 c_vp, ctypes.c_size_t, ctypes.c_int64, c_vp]),
    "td_pool_find_shards_headed": (_I, [c_vp, _I, c_vp, _I, _I, _I, _I, _I, c_vp, ctypes.c_int32, c_vp, ctypes.c_size_t,
                                       ctypes.c_int64, c_vp]),
    "td_pool_merge_headed": (_I, [c_vp, c_vp, _I, _I, _I, _I, c_vp, c_vp, c_vp, ctypes.c_size_t, c_vp]),
    "td_pool_pairs_workspace_bytes": (ctypes.c_size_t, [_I]),
    "td_pool_pairs": (_I, [c_vp, c_vp, _I, c_vp, _I, _I, ctypes.c_double, c_vp, ctypes.c_int32, c_vp, c_vp, ctypes.c_size_t, c_vp]),
    "td_pool_read_stats": (_I, [c_vp, _I, ctypes.POINTER(PoolStats), ctypes.POINTER(ctypes.c_int), c_vp]),
    "td_pool_read_stats_bytes": (ctypes.c_size_t, []),
    "td_pool_merge_workspace_bytes": (ctypes.c_size_t, [_I, _I]),
    "td_pool_merge": (_I, [c_vp, _I, _I, _I, c_vp, c_vp, c_vp, ctypes.c_size_t, c_vp]),
    "td_pool_merge_padded": (_I, [c_vp, c_vp, c_vp, _I, _I, _I, _I, c_vp, c_vp, c_vp, ctypes.c_size_t, c_vp]),
    "td_pool_pairs_exact_workspace_bytes": (ctypes.c_size_t, [_I, _I]),
    "td_pool_pairs_exact_batch": (_I, [c_vp, c_vp, c_vp, c_vp, _I, _I, c_vp, _I, _I, ctypes.c_double, c_vp, c_vp, c_vp, c_vp,
                                       ctypes.c_size_t, c_vp]),
    "td_pool_pairs_batch": (_I, [c_vp, c_vp, c_vp, c_vp, _I, _I, c_vp, _I, _I, ctypes.c_double, c_vp, c_vp, c_vp, c_vp]),
    "td_pool_batch_workspace_bytes": (ctypes.c_size_t, [_I, _I, ctypes.c_int64]),
    "td_pool_find_all_batch": (_I, [c_vp, c_vp, c_vp, _I, _I, c_vp, _I, _I, _I, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                    ctypes.c_size_t, ctypes.c_int64, c_vp]),
    "td_assign_stands_workspace_bytes": (ctypes.c_size_t, [_I, _I, _I]),
    "td_assign_stands_batch": (_I, [c_vp, _I, ctypes.c_int32, ctypes.c_int32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, _I, _I,
                                    c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, ctypes.c_size_t, c_vp]),
    "tdh_assign_stands": (_I, [c_vp, _I, c_vp, _I, c_vp, _I, ctypes.c_int32, ctypes.c_int32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "tdh_pool_pairs_exact": (_I, [c_vp, c_vp, _I, c_vp, _I, _I, ctypes.c_double, c_vp, c_vp, c_vp]),
    "tdh_pool_pairs": (_I, [c_vp, c_vp, _I, c_vp, _I, _I, ctypes.c_double, c_vp, c_vp, c_vp]),
    "tdh_cost_matrix": (_I, [c_vp, _I, c_vp, _I, c_vp, _I, ctypes.c_int32, ctypes.c_int32, c_vp]),
    "tdh_lcm": (_I, [c_vp, _I, ctypes.POINTER(LcmParams), c_vp, c_vp, c_vp, c_vp, c_vp]),
    "tdh_assign_exact": (_I, [c_vp, _I, c_vp, c_vp, c_vp, ctypes.POINTER(AssignStats)]),
    "tdh_assign_exact_rect": (_I, [c_vp, _I, _I, _I, c_vp, c_vp, c_vp, ctypes.POINTER(AssignStats)]),
    "tdh_pool_find": (_I, [c_vp, _I, c_vp, _I, _I, _I, _I, c_vp, ctypes.c_int32, c_vp, ctypes.POINTER(PoolStats)]),
    "tdh_pool_find_all": (_I, [c_vp, _I, c_vp, _I, _I, _I, c_vp, ctypes.c_int32, c_vp, ctypes.POINTER(PoolStats)]),
}

_lib = None


def library_path() -> str:
    return _build.SO


def lib() -> ctypes.CDLL:
    """Loads the shared library (building it first if the sources are newer).  Raises when it
    cannot be had -- there is deliberately no other implementation to fall back to."""
    global _lib
    if _lib is None:
        path = _build.SO
        if _build.needs_build():
            try:
                _build.build()
            except Exception as e:  # keep an existing, older .so usable on boxes without nvcc
                if not os.path.exists(path):
                    raise ImportError("libtaxidispatch.so is missing and could not be built: %s" % e) from e
        l = ctypes.CDLL(path)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(l, name)  # AttributeError = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def strerror(code: int) -> str:
    return lib().td_strerror(code).decode()


def check(code: int, where: str):
    if code != TD_OK:
        detail = lib().td_last_cuda_error().decode() if code == TD_ERR_CUDA else ""
        raise TaxiDispatchError(code, where, detail)
