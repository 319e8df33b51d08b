"""ctypes binding of ``libscs_b200.so`` (C ABI: ``include/scs_b200.h``).

There is no CPU fallback: if the library has not been built, or no CUDA device is usable, the
functions here raise.  The binding mirrors the header one to one; `INTEGRATION.md` shows the
same stub for a maintainer of the reference.
"""

from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_size_t, c_uint8, c_uint64, c_void_p
from pathlib import Path

LIB_PATH = Path(__file__).resolve().parent / "libscs_b200.so"

SCS_OK = 0
SCS_ERR_INVALID = -1
SCS_ERR_CUDA = -2
SCS_ERR_NO_DEVICE = -3
SCS_ERR_TOO_SMALL = -4
SCS_ERR_NO_CONVERGE = -5
SCS_ERR_INPUT = -6
SCS_ERR_EMPTY = -7
SCS_ERR_PEER = -8
IPC_HANDLE_BYTES = 64


class NodeStats(ctypes.Structure):
    """``scs_node_stats`` of include/scs_b200.h."""

    _fields_ = [
        ("n_components", c_int32),
        ("contracted_size", c_int32),
        ("spectral_ran", c_int32),
        ("solver", c_int32),
        ("matvecs", c_int32),
        ("restarts", c_int32),
        ("tie_flag", c_int32),
        ("kmeans_stable_splits", c_int32),
        ("eig", c_double * 3),
        ("residual", c_double),
        ("margin", c_double),
        ("kmeans_runner_up", c_double),
    ]

    def as_dict(self) -> dict:
        return {
            "n_components": self.n_components,
            "contracted_size": self.contracted_size,
            "spectral_ran": bool(self.spectral_ran),
            "solver": self.solver,
            "matvecs": self.matvecs,
            "restarts": self.restarts,
            "tie_flag": self.tie_flag,
            "eig": [self.eig[0], self.eig[1], self.eig[2]],
            "residual": self.residual,
            "margin": self.margin,
            "kmeans_stable_splits": self.kmeans_stable_splits,
            "kmeans_runner_up": self.kmeans_runner_up,
        }


class LibraryMissingError(RuntimeError):
    """``libscs_b200.so`` is not built: the CUDA path is the only path."""


_P = c_void_p  # every array argument is passed as a raw address

# name -> (restype, argtypes); one entry per function declared in include/scs_b200.h
SIGNATURES: dict[str, tuple] = {
    "scs_version": (c_int, []),
    "scs_status_string": (c_char_p, [c_int]),
    "scs_last_error": (c_char_p, [_P]),
    "scs_ctx_create": (c_int, [c_int, _P, POINTER(_P)]),
    "scs_ctx_destroy": (c_int, [_P]),
    "scs_ctx_synchronize": (c_int, [_P]),
    "scs_ctx_launch_count": (c_int64, [_P]),
    "scs_ctx_io_bytes": (c_int, [_P, POINTER(c_int64), POINTER(c_int64)]),
    "scs_ctx_timer_start": (c_int, [_P]),
    "scs_ctx_timer_stop": (c_int, [_P, POINTER(c_double)]),
    "scs_ctx_set_small_node_limit": (c_int, [_P, c_int]),
    "scs_ctx_set_medium_node_limit": (c_int, [_P, c_int]),
    "scs_ctx_set_device_forest": (c_int, [_P, c_int]),
    "scs_ctx_set_wide_entries": (c_int, [_P, c_int]),
    "scs_ctx_set_full_rows": (c_int, [_P, c_int]),
    "scs_ctx_stage_seconds": (c_int, [_P, _P, c_int]),
    "scs_ctx_flush_l2": (c_int, [_P]),
    "scs_ctx_profile_enable": (c_int, [_P, c_int]),
    "scs_ctx_profile_read": (c_int, [_P, c_int, POINTER(c_int64), POINTER(c_double), POINTER(c_double), POINTER(c_double)]),
    "scs_bit_words": (c_int, [c_int]),
    "scs_pcg_build_dev": (c_int, [_P, c_int, c_int, c_int64] + [_P] * 12),
    "scs_pcg_build_rows_dev": (c_int, [_P, c_int, c_int, c_int64, _P, _P, _P, _P, _P, _P, c_int, c_int, _P, _P, _P, _P, _P]),
    "scs_components_dev": (c_int, [_P, c_int, _P, _P, POINTER(c_int32)]),
    "scs_contract_dev": (c_int, [_P, c_int, _P, _P, _P, _P, POINTER(c_int32), _P, _P]),
    "scs_spectral_bipartition_dev": (c_int, [_P, c_int, _P, _P, c_uint64, _P, POINTER(NodeStats)]),
    "scs_normalized_matvec_dev": (c_int, [_P, c_int, _P, _P, _P, _P]),
    "scs_node_split_host": (
        c_int,
        [_P, c_int, c_int, c_int64, _P, _P, _P, _P, _P, _P, c_int, c_uint64, _P, POINTER(NodeStats)],
    ),
    "scs_node_split_dev": (
        c_int,
        [_P, c_int, c_int, c_int64, _P, _P, _P, _P, _P, _P, c_int, c_uint64, _P, POINTER(NodeStats)],
    ),
    "scs_node_last_buffers": (c_int, [_P, POINTER(c_int), POINTER(c_int)] + [POINTER(_P)] * 7),
    "scs_dev_alloc": (c_int, [_P, c_size_t, POINTER(_P)]),
    "scs_dev_free": (c_int, [_P, _P]),
    "scs_memcpy_h2d": (c_int, [_P, _P, _P, c_size_t]),
    "scs_memcpy_d2h": (c_int, [_P, _P, _P, c_size_t]),
    "scs_set_host_threads": (c_int, [c_int]),
    "scs_forest_create": (c_int, [c_int, _P, _P, _P, _P, _P, _P, c_int, POINTER(_P)]),
    "scs_forest_create_view": (c_int, [c_int, _P, _P, _P, _P, _P, _P, c_int, POINTER(_P)]),
    "scs_forest_destroy": (c_int, [_P]),
    "scs_forest_parse_newick": (c_int, [c_char_p, c_size_t, POINTER(_P), POINTER(_P), POINTER(c_size_t), POINTER(c_int)]),
    "scs_newick_last_error": (c_char_p, []),
    "scs_forest_last_error": (c_char_p, []),
    "scs_flat_tree_newick": (c_int, [c_int64, _P, _P, c_char_p, c_size_t, c_int, POINTER(_P), POINTER(c_size_t)]),
    "scs_flat_tree_newick_values": (
        c_int,
        [c_int64, _P, _P, c_char_p, c_size_t, c_int, _P, c_int, POINTER(_P), POINTER(c_size_t)],
    ),
    "scs_supertree_support": (c_int, [_P, _P, c_int64, _P, _P, _P, _P, _P]),
    "scs_supertree_triplets": (c_int, [_P, _P, c_int64, _P, _P, _P]),
    "scs_supertree_taxon_triplets": (c_int, [_P, _P, c_int64, _P, _P, _P, _P]),
    "scs_supertree_mrp": (c_int, [_P, _P, c_int64, _P, _P, _P]),
    "scs_forest_pairwise_rf": (c_int, [_P, _P, _P, _P, _P]),
    "scs_profiler_range": (c_int, [c_int]),
    "scs_debug_small_cycles": (c_int, [_P, _P, c_int]),
    "scs_free": (None, [_P]),
    "scs_forest_num_trees": (c_int, [_P]),
    "scs_forest_num_nodes": (c_int64, [_P]),
    "scs_forest_num_leaves": (c_int64, [_P]),
    "scs_forest_num_taxa": (c_int, [_P]),
    "scs_forest_pair_visits": (c_int64, [_P]),
    "scs_forest_tree_info": (c_int, [_P, c_int, POINTER(c_int64), POINTER(c_double), POINTER(c_int32)]),
    "scs_forest_tree": (c_int, [_P, c_int, _P, _P, _P, _P]),
    "scs_forest_taxa": (c_int, [_P, _P]),
    "scs_forest_induce": (c_int, [_P, _P, POINTER(_P)]),
    "scs_forest_induce_parts": (c_int, [_P, _P, c_int, _P, _P]),
    "scs_forest_tours": (c_int, [_P, c_int, _P, _P, _P, _P, _P, _P, _P]),
    "scs_forest_split": (
        c_int,
        [_P, _P, c_int, c_int, c_uint64, POINTER(c_int32), _P, _P, POINTER(NodeStats)],
    ),
    "scs_nodes_split_small_host": (
        c_int,
        [_P, c_int, _P, c_int64, c_int64, _P, _P, _P, _P, _P, _P, c_int, _P, _P],
    ),
    "scs_nodes_split_small_dev": (c_int, [_P, c_int, _P, _P, _P, _P, _P, _P, _P, c_int, _P, _P]),
    "scs_supertree_build": (c_int, [_P, _P, c_int, c_int, c_uint64, c_int, POINTER(_P)]),
    "scs_supertree_build_sharded": (c_int, [_P, _P, c_int, c_int, c_uint64, c_int, c_int, c_int, POINTER(_P)]),
    "scs_supertree_shared_prefix": (c_int64, [_P]),
    "scs_supertree_shared_records": (c_int64, [_P]),
    "scs_supertree_wave_info": (c_int, [_P, _P, _P]),
    "scs_supertree_wave_seconds": (c_int, [_P, _P]),
    "scs_supertree_destroy": (c_int, [_P]),
    "scs_supertree_num_nodes": (c_int64, [_P]),
    "scs_supertree_nodes": (c_int, [_P, _P, _P]),
    "scs_supertree_counters": (c_int, [_P, POINTER(c_int64), POINTER(c_int64), POINTER(c_int64), POINTER(c_int64)]),
    "scs_device_forest_create": (c_int, [_P, _P, c_int, POINTER(_P)]),
    "scs_device_forest_destroy": (c_int, [_P]),
    "scs_device_forest_bytes": (c_int64, [_P]),
    "scs_supertree_build_resident": (c_int, [_P, _P, c_int, c_uint64, c_int, c_int, c_int, POINTER(_P)]),
    "scs_supertree_record_wave": (c_int, [_P, c_int64]),
    "scs_nodes_split_medium_dev": (c_int, [_P, c_int, _P, _P, _P, _P, c_int, c_int64, _P, _P, _P, _P, _P, _P, c_int, _P, _P, _P]),
    "scs_supertree_medium_info": (c_int, [_P, POINTER(c_int64), POINTER(c_int64), POINTER(ctypes.c_double)]),
    "scs_supertree_seconds": (c_int, [_P, _P]),
    "scs_supertree_num_records": (c_int64, [_P]),
    "scs_supertree_record_size": (c_int, [_P, c_int64]),
    "scs_supertree_record": (c_int, [_P, c_int64, _P, _P, POINTER(NodeStats)]),
    "scs_shard_create": (c_int, [_P, c_int, c_int, c_int, _P]),
    "scs_shard_connect_ipc": (c_int, [_P, _P]),
    "scs_shard_window": (c_int, [_P, POINTER(_P), POINTER(c_size_t)]),
    "scs_shard_connect_ptrs": (c_int, [_P, _P]),
    "scs_shard_engage": (c_int, [_P, c_int]),
    "scs_shard_configure": (c_int, [_P, c_int, c_double]),
    "scs_shard_barrier": (c_int, [_P]),
    "scs_shard_nodes": (c_int64, [_P]),
    "scs_shard_destroy": (c_int, [_P]),
}

_LIB: ctypes.CDLL | None = None


def load() -> ctypes.CDLL:
    """The loaded library with every signature set; raises if it is missing."""
    global _LIB  # noqa: PLW0603
    if _LIB is not None:
        return _LIB
    if not LIB_PATH.is_file():
        msg = (
            f"{LIB_PATH} is missing: build it with `python -m spectralclustersupertree_b200.build` "
            "(there is no CPU fallback for the CUDA path)"
        )
        raise LibraryMissingError(msg)
    # Row-sharded nodes wait on the device for kernels of other contexts; a kernel whose code is loaded lazily at
    # its first launch can block behind such a wait when the contexts share a process (the in-process multi-rank
    # tests), so ask for all kernels up front.  Only effective before the CUDA runtime initialises.
    os.environ.setdefault("CUDA_MODULE_LOADING", "EAGER")
    # Idle OpenMP threads of the host-side helpers (tree validation, uploads) should sleep rather than spin: the
    # recursion's own driver threads, and the other ranks of a multi-GPU job, need the cores.  Only effective if the
    # OpenMP runtime has not been loaded yet (bench.py sets it before importing anything).
    os.environ.setdefault("OMP_WAIT_POLICY", "passive")
    lib = ctypes.CDLL(str(LIB_PATH))
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    _LIB = lib
    return lib


def ptr(array) -> int | None:
    """Address of a C-contiguous numpy array (None for None)."""
    if array is None:
        return None
    if not array.flags["C_CONTIGUOUS"]:
        msg = "array must be C-contiguous"
        raise ValueError(msg)
    return array.ctypes.data


__all__ = ["LIB_PATH", "SIGNATURES", "LibraryMissingError", "NodeStats", "c_uint8", "load", "ptr"]
