"""ctypes binding of libbn_b200.so (include/bn_b200.h).

The product has no CPU path: if the shared library is missing it is built with
nvcc (``bayesnetworks_b200.build``); if that fails, or no CUDA device is
present when a compute entry point is called, the error is raised -- nothing
falls back to the oracle or to numpy.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

# status codes (include/bn_b200.h)
BN_OK, BN_ERR_BAD_ARG, BN_ERR_CUDA, BN_ERR_OOM = 0, 1, 2, 3
BN_ERR_NO_LEGAL_PROPOSAL, BN_ERR_NO_DEVICE, BN_ERR_CAPACITY, BN_ERR_UNSUPPORTED = 4, 5, 6, 7
BN_RNG_WH, BN_RNG_RMT, BN_RNG_REPLAY = 0, 1, 2

EXPORTED_SYMBOLS = (
    "bn_last_error", "bn_abi_version", "bn_device_count", "bn_create", "bn_create_from_device",
    "bn_create_from_stats", "bn_block_colsum_device", "bn_block_gram_device", "bn_create_from_stats_device",
    "bn_destroy", "bn_trim_pool", "bn_set_stream", "bn_set_default_stream", "bn_get_stats", "bn_get_gram_ms",
    "bn_get_launch_count", "bn_score_nodes", "bn_score_all_proposals",
    "bn_score_all_proposals_device", "bn_run", "bn_main_fun", "bn_score_state_len",
)

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


class BnError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"libbn_b200 status {status}: {message}")
        self.status = status


class Trace(C.Structure):
    _fields_ = [("capacity", C.c_int), ("n_rows", _ip), ("iter", _ip), ("changed_node", _ip),
                ("movetype", _ip), ("global_ll", _dp), ("additions", _ip), ("deletions", _ip),
                ("fn", _ip), ("fp", _ip)]


class ChainStats(C.Structure):
    _fields_ = [("uniforms", C.c_int64), ("valid_iters", C.c_int64), ("proposed", C.c_int * 3),
                ("reject", C.c_int * 3), ("n_nonpd", C.c_int), ("total_edges", C.c_int),
                ("status", C.c_int), ("windows", C.c_int), ("alg_bytes", C.c_int64),
                ("phase_cycles", C.c_int64 * 12), ("slots_simulated", C.c_int64), ("kernel_cycles", C.c_int64)]


import numpy as _np
CHAIN_STATS_DTYPE = _np.dtype([("uniforms", "<i8"), ("valid_iters", "<i8"), ("proposed", "<i4", (3,)),
                               ("reject", "<i4", (3,)), ("n_nonpd", "<i4"), ("total_edges", "<i4"),
                               ("status", "<i4"), ("windows", "<i4"), ("alg_bytes", "<i8"),
                               ("phase_cycles", "<i8", (12,)), ("slots_simulated", "<i8"), ("kernel_cycles", "<i8")],
                              align=True)
assert CHAIN_STATS_DTYPE.itemsize == C.sizeof(ChainStats)


class RunArgs(C.Structure):
    _fields_ = [("n_chains", C.c_int), ("rng_kind", C.c_int), ("seeds", _ip), ("replay", _dp),
                ("replay_len", C.c_int64), ("initial_network", C.c_int), ("drop", C.c_int),
                ("n_iter", C.c_int), ("output_every", C.c_int), ("device_outputs", C.c_int),
                ("moves_capacity", C.c_int), ("n_moves", _ip), ("moves", _ip), ("edge_freq", _ip),
                ("npar_freq", _ip), ("mt_state_in", _ip), ("mt_state_out", _ip),
                ("start_parents", _ip), ("start_n_par", _ip), ("state_in", C.c_void_p), ("state_out", C.c_void_p),
                ("score_state_in", _dp), ("score_state_out", _dp), ("anc_freq", _ip),
                ("best_parents", _ip), ("best_n_par", _ip), ("best", C.c_void_p), ("mb_freq", _ip)]


class BestGraphC(C.Structure):
    """bn_best_graph"""
    _fields_ = [("log_post", C.c_double), ("log_lik", C.c_double), ("log_prior", C.c_double),
                ("iter", C.c_int64), ("total_edges", C.c_int), ("found", C.c_int)]


class ChainStateC(C.Structure):
    """bn_chain_state"""
    _fields_ = [("iter", C.c_int64), ("valid", C.c_int), ("total_edges_member", C.c_int),
                ("additions", C.c_int), ("deletions", C.c_int), ("wh_state", C.c_int * 3), ("uniforms", C.c_int64)]


_lib = None


def lib() -> C.CDLL:
    """Load (building if needed) libbn_b200.so; raises if it cannot be had."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("BN_B200_LIB") or _build.LIB   # (BN_B200_LIB: another build of the same library, for A/B runs)
    if not os.path.exists(path):
        _build.build()
    L = C.CDLL(path)
    L.bn_last_error.restype = C.c_char_p
    L.bn_get_launch_count.restype = C.c_int64
    L.bn_get_launch_count.argtypes = [C.c_void_p]
    L.bn_destroy.argtypes = [C.c_void_p]
    L.bn_destroy.restype = None
    L.bn_create.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                            C.c_int, C.c_double, C.c_double, C.c_int, C.POINTER(C.c_void_p)]
    L.bn_create_from_device.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                        C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_int,
                                        C.POINTER(C.c_void_p)]
    L.bn_create_from_stats.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_int,
                                       C.POINTER(C.c_void_p)]
    L.bn_block_colsum_device.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    L.bn_block_gram_device.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                       C.c_void_p, C.POINTER(C.c_float)]
    L.bn_create_from_stats_device.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_int,
                                              C.POINTER(C.c_void_p)]
    L.bn_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    L.bn_set_default_stream.argtypes = [C.c_void_p]
    L.bn_get_stats.argtypes = [C.c_void_p] * 5
    L.bn_get_gram_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
    L.bn_score_nodes.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.bn_score_all_proposals.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 5
    L.bn_score_all_proposals_device.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 5 + [C.POINTER(C.c_float)]
    L.bn_run.argtypes = [C.c_void_p, C.POINTER(RunArgs), C.POINTER(Trace), C.c_void_p, C.c_void_p,
                         C.c_void_p, C.POINTER(C.c_float)]
    L.bn_score_state_len.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
    L.bn_main_fun.argtypes = ([C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                               C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int,
                               C.c_int, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 10)
    _lib = L
    return L


def check(status: int) -> None:
    if status != BN_OK:
        raise BnError(status, lib().bn_last_error().decode("utf-8", "replace"))


def ptr(a):
    """Raw pointer of a numpy array (or None)."""
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def as_i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)
