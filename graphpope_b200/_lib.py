"""ctypes binding of libgraphpope_b200.so (the C ABI in include/graphpope_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` (``make -C
graphpope_b200/csrc``).  There is no CPU fallback: if the shared object is
missing, or no CUDA device is visible when a compute entry point is called, the
product raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_uint32, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgraphpope_b200.so")

GP_OK = 0
GP_ERR_INVALID = 1
GP_ERR_CUDA = 2
GP_ERR_OOM = 3
GP_ERR_INDEX_RANGE = 4
GP_ERR_LEVEL_OVERFLOW = 5
GP_ERR_UNSUPPORTED = 6
GP_ERR_NOT_CONVERGED = 7
GP_ERR_NO_DEVICE = 8

GP_CSR_SYMMETRIZE = 0x1
GP_UNREACHABLE_U16 = 0xFFFF

CDIST_MODES = {"distance": 0, "similarity": 1, "euclidean": 2}  # dist_map keys, utils.py:158-162


class GraphpopeError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"graphpope_b200 [{status}]: {message}")
        self.status = status


class CsrInfo(ctypes.Structure):
    _fields_ = [("num_nodes", c_int64), ("num_input_edges", c_int64), ("num_edges", c_int64),
                ("max_out_degree", c_int64), ("is_symmetric", c_int32), ("reserved", c_int32)]


class MsbfsStats(ctypes.Structure):
    _fields_ = [("num_anchors", c_int64), ("lane_words", c_int64), ("max_level", c_int32),
                ("levels_run", c_int32), ("pull_levels", c_int32), ("push_levels", c_int32),
                ("edges_examined", c_int64), ("grid_blocks", c_int64)]

    def as_dict(self):
        return {name: int(getattr(self, name)) for name, _ in self._fields_}


# name -> (restype, argtypes); every function include/graphpope_b200.h declares
SIGNATURES = {
    "gp_abi_version": (c_int, []),
    "gp_last_error": (c_char_p, []),
    "gp_status_string": (c_char_p, [c_int]),
    "gp_device_info": (c_int, [POINTER(c_int32), POINTER(c_int32), POINTER(c_int32), c_char_p, c_int64]),
    "gp_launch_count": (c_int64, []),
    "gp_msbfs_kernel_ms": (c_int, [c_void_p, POINTER(ctypes.c_float)]),
    "gp_msbfs_set_stage_events": (c_int, [c_void_p, c_int32]),
    "gp_msbfs_kernel_device_ns": (c_int, [c_void_p, POINTER(c_uint64), c_void_p]),
    "gp_pipeline_stage_ms": (c_int, [c_void_p, POINTER(ctypes.c_float)]),
    "gp_msbfs_trace": (c_int, [c_void_p, c_void_p, c_int64, POINTER(c_int32), POINTER(c_int32)]),
    "gp_csr_create": (c_int, [c_int64, c_int64, c_uint32, POINTER(c_void_p)]),
    "gp_csr_build": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "gp_csr_info": (c_int, [c_void_p, POINTER(CsrInfo), c_void_p]),
    "gp_csr_export": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "gp_csr_trace_ms": (c_int, [c_void_p, POINTER(ctypes.c_float), c_int32, POINTER(c_int32)]),
    "gp_csr_free": (c_int, [c_void_p]),
    "gp_msbfs_create": (c_int, [c_void_p, c_int64, POINTER(c_void_p)]),
    "gp_msbfs_run": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "gp_msbfs_hops_u16": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "gp_msbfs_features": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_void_p]),
    "gp_msbfs_set_push": (c_int, [c_void_p, c_int32]),
    "gp_msbfs_stats": (c_int, [c_void_p, POINTER(MsbfsStats), c_void_p]),
    "gp_msbfs_free": (c_int, [c_void_p]),
    "gp_geodesic_run": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int64,
                                c_void_p, c_int64, c_int64, c_void_p]),
    "gp_concat_x": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64, c_void_p]),
    "gp_msbfs_planes": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_int64), POINTER(c_int32),
                                POINTER(c_int32), POINTER(c_int32), c_void_p]),
    "gp_decode_gathered": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_int64, c_int32, c_int32, c_int32,
                                   c_int64, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_void_p]),
    "gp_msbfs_pack": (c_int, [c_void_p, c_int32, POINTER(c_void_p), POINTER(c_int64), POINTER(c_int32),
                              POINTER(c_int32), POINTER(c_void_p), c_void_p]),
    "gp_geodesic_run_packed": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int32, c_void_p]),
    "gp_msbfs_packed_info": (c_int, [c_void_p, c_int32, POINTER(c_void_p), POINTER(c_int64), POINTER(c_int32),
                                     POINTER(c_int32), POINTER(c_void_p)]),
    "gp_msbfs_ipc_export": (c_int, [c_void_p, c_void_p, POINTER(c_int64)]),
    "gp_ipc_open": (c_int, [c_void_p, POINTER(c_void_p)]),
    "gp_ipc_close": (c_int, [c_void_p]),
    "gp_decode_peers": (c_int, [c_void_p, c_int32, c_int64, c_int64, c_int32, c_int32, c_int64, c_void_p, c_int64,
                                c_int64, c_void_p, c_int64, c_int64, c_void_p]),
    "gp_exchange_create": (c_int, [c_void_p, c_int32, c_int32, POINTER(c_void_p)]),
    "gp_exchange_ipc_export": (c_int, [c_void_p, c_void_p]),
    "gp_exchange_local_ptr": (c_int, [c_void_p, POINTER(c_void_p)]),
    "gp_exchange_set_peer": (c_int, [c_void_p, c_int32, c_void_p]),
    "gp_geodesic_run_exchange": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p,
                                         c_int64, c_int64, c_void_p, c_int64, c_int64, c_void_p]),
    "gp_exchange_run": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_void_p]),
    "gp_exchange_status": (c_int, [c_void_p, POINTER(c_int32), c_void_p]),
    "gp_exchange_set_grid": (c_int, [c_void_p, c_int32]),
    "gp_exchange_trace": (c_int, [c_void_p, c_void_p]),
    "gp_exchange_free": (c_int, [c_void_p]),
    "gp_fstore_layout": (c_int, [c_void_p, POINTER(c_int32), POINTER(c_int64), c_void_p]),
    "gp_fstore_pack": (c_int, [c_void_p, c_void_p, c_int32, c_void_p]),
    "gp_fstore_merge": (c_int, [c_void_p, c_int32, c_int64, c_int64, c_int64, c_int32, c_int64, c_void_p, c_void_p]),
    "gp_fstore_gather": (c_int, [c_void_p, c_int64, c_int64, c_int32, c_void_p, c_int64, c_void_p, c_int64, c_int64,
                                 c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "gp_normalize_into": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64, c_int64, c_void_p]),
    "gp_geodesic_embed_host": (c_int, [c_void_p, c_int64, c_int64, c_uint32, c_void_p, c_int64, c_void_p,
                                       c_int64, c_void_p, c_int64, c_int64, c_void_p, POINTER(MsbfsStats)]),
    "gp_ctx_create": (c_int, [POINTER(c_void_p)]),
    "gp_ctx_free": (c_int, [c_void_p]),
    "gp_geodesic_embed_host_ctx": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_uint32, c_void_p, c_int64, c_void_p,
                                           c_int64, c_void_p, c_int64, c_int64, c_void_p, POINTER(MsbfsStats)]),
    "gp_host_concat": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_void_p, c_int64]),
    "gp_block_to_host": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_void_p]),
    "gp_degree": (c_int, [c_void_p, c_void_p, c_void_p]),
    "gp_pagerank": (c_int, [c_void_p, c_double, c_double, c_int32, c_void_p, POINTER(c_int32), c_void_p]),
    "gp_closeness": (c_int, [c_void_p, c_void_p, c_void_p]),
    "gp_clustering": (c_int, [c_void_p, c_void_p, c_void_p]),
    "gp_betweenness": (c_int, [c_void_p, c_void_p, c_void_p]),
    "gp_eigenvector": (c_int, [c_void_p, c_double, c_int32, c_void_p, POINTER(c_int32), c_void_p]),
    "gp_kmeans_plusplus": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int64, c_uint64, c_void_p, c_void_p, c_void_p,
                                   c_void_p]),
    "gp_kmeans_assign": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p]),
    "gp_kmeans_update": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_void_p, c_void_p]),
    "gp_topk_stable_i32": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "gp_topk_stable_f64": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "gp_cdist_minmax": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int32, c_int32, c_void_p,
                                c_int64, c_int64, c_void_p]),
}

_lib = None


def load():
    """Load the shared library (no GPU needed to load it)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C graphpope_b200/csrc`). graphpope_b200 has no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        if lib.gp_abi_version() != 1:
            raise ImportError("libgraphpope_b200.so has an unexpected ABI version")
        _lib = lib
    return _lib


def check(status: int, iterations: int | None = None):
    """Raise the Python exception the reference would have raised for ``status``.  ``iterations`` is the
    iteration budget of a power-iteration call (reported by PowerIterationFailedConvergence)."""
    if status == GP_OK:
        return
    msg = (load().gp_last_error() or b"").decode("utf-8", "replace")
    if status == GP_ERR_INDEX_RANGE:
        raise IndexError(f"graphpope_b200: {msg}")
    if status == GP_ERR_LEVEL_OVERFLOW:
        raise OverflowError(f"graphpope_b200: {msg}")
    if status == GP_ERR_OOM:
        raise MemoryError(f"graphpope_b200: {msg}")
    if status == GP_ERR_NOT_CONVERGED:
        try:
            import networkx as nx
            raise nx.PowerIterationFailedConvergence(100 if iterations is None else int(iterations))  # utils.py:28
        except ImportError:
            pass
    raise GraphpopeError(status, msg)


def require_cuda():
    """Fail loudly when there is no device: the product has no CPU path."""
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError("graphpope_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return load()
