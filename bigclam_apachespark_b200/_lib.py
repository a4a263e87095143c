"""ctypes binding of libbigclam_b200.so (C ABI declared in include/bigclam_b200.h).

The library is the product: there is no Python or CPU fallback.  Importing this module never
needs a GPU (so the symbol table can be checked on a CPU box), but every compute call fails
loudly when the shared library is missing or no CUDA device is usable.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libbigclam_b200.so")

OK, EINVAL, ECUDA, ENOMEM, EIO, EUNSUPPORTED = 0, -1, -2, -3, -4, -5
F_TIME_KERNELS = 1
F_RECORD_ACCEPTED = 2
F_SPARSE_ROWS = 4
F_LS_EXHAUSTIVE = 8


class Params(C.Structure):
    """`bigclam_params` — one field per script-level variable of codes/bigclam4-7.scala:16-43."""

    _fields_ = [
        ("k", C.c_int32),
        ("max_inter", C.c_int32),
        ("alpha", C.c_double),
        ("beta", C.c_double),
        ("min_p", C.c_double),
        ("max_p", C.c_double),
        ("min_f", C.c_double),
        ("max_f", C.c_double),
        ("device", C.c_int32),
        ("flags", C.c_int32),
    ]


class Graph(C.Structure):
    """`bigclam_graph` — CSR produced by the edge-list reader."""

    _fields_ = [
        ("n", C.c_int64),
        ("nnz", C.c_int64),
        ("rowptr", C.POINTER(C.c_int64)),
        ("col", C.POINTER(C.c_int32)),
        ("ids", C.POINTER(C.c_int64)),
        ("n_edge_lines", C.c_int64),
    ]


class BigclamError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"bigclam_b200 error {code}: {msg}")
        self.code = code


# Every symbol include/bigclam_b200.h declares: name -> (restype, argtypes)
_vp, _i64, _i32, _dbl = C.c_void_p, C.c_int64, C.c_int32, C.c_double
_pd, _pi64 = C.POINTER(C.c_double), C.POINTER(C.c_int64)
SIGNATURES = {
    "bigclam_default_params": (C.c_int, [C.POINTER(Params), _i32]),
    "bigclam_step_sizes": (C.c_int, [_dbl, _i32, _vp]),
    "bigclam_create": (C.c_int, [C.POINTER(_vp), _i64, _vp, _vp, C.POINTER(Params)]),
    "bigclam_destroy": (None, [_vp]),
    "bigclam_last_error": (C.c_char_p, [_vp]),
    "bigclam_set_F": (C.c_int, [_vp, _vp]),
    "bigclam_set_sumF": (C.c_int, [_vp, _vp]),
    "bigclam_get_F": (C.c_int, [_vp, _vp]),
    "bigclam_get_sumF": (C.c_int, [_vp, _vp]),
    "bigclam_step": (C.c_int, [_vp, _vp, _pd, _pi64]),
    "bigclam_loglikelihood": (C.c_int, [_vp, _pd]),
    "bigclam_run": (C.c_int, [_vp, _i32, _dbl, _i64, _pd, _pi64, _vp, _i64]),
    "bigclam_get_accepted": (C.c_int, [_vp, _vp]),
    "bigclam_get_kernel_time": (C.c_int, [_vp, _pd, _pi64, _pi64]),
    "bigclam_get_tile_stats": (C.c_int, [_vp, _pi64, _pi64, _pi64, _pi64, _pi64]),
    "bigclam_get_ls_stats": (C.c_int, [_vp, _pi64, _pi64]),
    "bigclam_set_holdout": (C.c_int, [_vp, _vp, _vp, _vp]),
    "bigclam_holdout_loglikelihood": (C.c_int, [_vp, _pd, _pi64]),
    "bigclam_retile": (C.c_int, [_vp]),
    "bigclam_set_stream": (C.c_int, [_vp, _vp]),
    "bigclam_device_state": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), _pi64]),
    "bigclam_device_accepted": (C.c_int, [_vp, C.POINTER(_vp)]),
    "bigclam_set_owned_nodes": (C.c_int, [_vp, _vp, _i64]),
    "bigclam_set_owned_range": (C.c_int, [_vp, _i64, _i64]),
    "bigclam_set_uset": (C.c_int, [_vp, _vp]),
    "bigclam_step_local": (C.c_int, [_vp, C.POINTER(_vp)]),
    "bigclam_finish_local": (C.c_int, [_vp, _pd, _pi64]),
    "bigclam_collect_timing": (C.c_int, [_vp]),
    "bigclam_llh_local": (C.c_int, [_vp, C.POINTER(_vp)]),
    "bigclam_rollback": (C.c_int, [_vp]),
    "bigclam_ipc_export": (C.c_int, [_vp, _vp]),
    "bigclam_ipc_open_peers": (C.c_int, [_vp, _i32, _i32, _vp]),
    "bigclam_mark_all_changed": (C.c_int, [_vp]),
    "bigclam_ipc_handle_count": (C.c_int, [_vp]),
    "bigclam_xchg_export": (C.c_int, [_vp, _i32, _i32, _vp]),
    "bigclam_xchg_open_peers": (C.c_int, [_vp, _vp]),
    "bigclam_llh_finish_local": (C.c_int, [_vp, _pd]),
    "bigclam_multi_create": (C.c_int, [C.POINTER(_vp), _i64, _vp, _vp, C.POINTER(Params), _i32, _vp]),
    "bigclam_multi_destroy": (None, [_vp]),
    "bigclam_multi_last_error": (C.c_char_p, [_vp]),
    "bigclam_multi_world": (C.c_int, [_vp]),
    "bigclam_multi_set_F": (C.c_int, [_vp, _vp]),
    "bigclam_multi_set_F_csr": (C.c_int, [_vp, _vp, _vp, _vp]),
    "bigclam_multi_set_sumF": (C.c_int, [_vp, _vp]),
    "bigclam_multi_get_F": (C.c_int, [_vp, _i32, _vp]),
    "bigclam_multi_get_sumF": (C.c_int, [_vp, _i32, _vp]),
    "bigclam_multi_get_F_nnz": (C.c_int, [_vp, _pi64]),
    "bigclam_multi_get_F_csr": (C.c_int, [_vp, _vp, _vp, _vp]),
    "bigclam_multi_step": (C.c_int, [_vp, _vp, _pd, _pi64]),
    "bigclam_multi_loglikelihood": (C.c_int, [_vp, _pd]),
    "bigclam_multi_run": (C.c_int, [_vp, _i32, _dbl, _i64, _pd, _pi64, _vp, _i64]),
    "bigclam_multi_get_kernel_time": (C.c_int, [_vp, _pd, _pi64]),
    "bigclam_multi_get_ls_stats": (C.c_int, [_vp, _pi64, _pi64]),
    "bigclam_set_F_csr": (C.c_int, [_vp, _vp, _vp, _vp]),
    "bigclam_get_F_nnz": (C.c_int, [_vp, _pi64]),
    "bigclam_get_F_csr": (C.c_int, [_vp, _vp, _vp, _vp]),
    "bigclam_set_pool_region": (C.c_int, [_vp, _i64, _i64]),
    "bigclam_get_pool_capacity": (C.c_int, [_vp, _pi64]),
    "bigclam_graph_read_edgelist": (C.c_int, [C.c_char_p, _i32, C.POINTER(Graph), C.c_char_p, _i64]),
    "bigclam_graph_free": (None, [C.POINTER(Graph)]),
    "bigclam_extract": (C.c_int, [_vp, _dbl, _vp, _vp]),
    "bigclam_conductance_seeds": (C.c_int, [_i64, _vp, _vp, _vp, _vp, _pi64]),
    "bigclam_conductance_seeds_gpu": (C.c_int, [_i64, _vp, _vp, _i32, _vp, _vp, _pi64]),
    "bigclam_init_neighbor_com_F": (C.c_int, [_i64, _vp, _vp, _i32, _vp, _i64, _i32, C.c_uint64, _vp]),
    "bigclam_device_count": (C.c_int, []),
    "bigclam_version": (C.c_char_p, []),
}

_lib = None


def load() -> C.CDLL:
    """Load the shared library; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  bigclam_apachespark_b200 has no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError == header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int, ctx=None):
    if rc != OK:
        msg = load().bigclam_last_error(ctx)
        raise BigclamError(rc, msg.decode() if msg else "unknown error")


def sparse_node_words(ld: int) -> int:
    """Worst-case 8-byte words one node can take in a sparse-row output pool: a full row block and a full delta
    block (csrc/bigclam_sparse.cuh: sp_words(ld) each) — the unit bigclam_set_pool_region is sized in."""
    return 2 * (((ld + 1) & ~1) + ((ld + 7) & ~7) // 4)
