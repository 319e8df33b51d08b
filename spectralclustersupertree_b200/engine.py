"""Host-side handles over the C ABI: a GPU context (``Engine``) and a source-tree store (``Forest``).

``Engine`` owns one ``scs_ctx`` (one CUDA stream + workspace on one GPU).  ``Forest`` owns one
``scs_forest``: the flat-array form of the list of source trees the reference's recursion
carries (ref: src/sc_supertree/scs.py:18-25, 411-455).  Everything numeric happens inside
``libscs_b200.so``; this module only moves numpy arrays across the boundary.
"""

from __future__ import annotations

import ctypes
import os
from collections.abc import Sequence

import numpy as np

from . import _lib
from ._lib import NodeStats, ptr

WEIGHTINGS = ("one", "branch", "depth", "bootstrap")  # codes of scs_forest_tours


class ScsError(RuntimeError):
    """A call into libscs_b200.so failed."""

    def __init__(self, status: int, detail: str = "") -> None:
        self.status = status
        text = _lib.load().scs_status_string(status).decode()
        super().__init__(f"libscs_b200: {text}" + (f" ({detail})" if detail else ""))


def _check(status: int, ctx=None) -> None:
    if status == _lib.SCS_OK:
        return
    detail = ""
    if ctx is not None:
        detail = _lib.load().scs_last_error(ctx).decode()
    raise ScsError(status, detail)


class Engine:
    """One GPU context.  Not thread-safe; use one per thread per GPU."""

    def __init__(self, device: int | None = None) -> None:
        self._lib = _lib.load()
        if device is None:
            device = int(os.environ.get("SCS_B200_DEVICE", os.environ.get("LOCAL_RANK", "0")))
        handle = ctypes.c_void_p()
        status = self._lib.scs_ctx_create(device, None, ctypes.byref(handle))
        if status != _lib.SCS_OK:
            raise ScsError(status, f"scs_ctx_create(device={device}); the CUDA path has no CPU fallback")
        self._ctx = handle
        self.device = device

    # -- lifetime ----------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_ctx", None):
            self._lib.scs_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self) -> None:  # pragma: no cover - interpreter shutdown order
        try:
            self.close()
        except Exception:  # noqa: BLE001, S110
            pass

    def __enter__(self) -> "Engine":
        return self

    def __exit__(self, *exc) -> None:
        self.close()

    @property
    def handle(self):
        return self._ctx

    @property
    def launch_count(self) -> int:
        return int(self._lib.scs_ctx_launch_count(self._ctx))

    def synchronize(self) -> None:
        _check(self._lib.scs_ctx_synchronize(self._ctx), self._ctx)

    def io_bytes(self) -> tuple[int, int]:
        """(host->device, device->host) bytes copied by the host-buffer entry points so far."""
        h2d, d2h = ctypes.c_int64(0), ctypes.c_int64(0)
        _check(self._lib.scs_ctx_io_bytes(self._ctx, ctypes.byref(h2d), ctypes.byref(d2h)), self._ctx)
        return h2d.value, d2h.value

    def timer_start(self) -> None:
        _check(self._lib.scs_ctx_timer_start(self._ctx), self._ctx)

    def timer_stop(self) -> float:
        """Milliseconds since ``timer_start`` on the context's stream (CUDA events)."""
        ms = ctypes.c_double(0.0)
        _check(self._lib.scs_ctx_timer_stop(self._ctx, ctypes.byref(ms)), self._ctx)
        return ms.value

    def set_small_node_limit(self, limit: int) -> None:
        """Largest recursion node (vertices) that takes the one-CTA path; 0 forces the staged path."""
        _check(self._lib.scs_ctx_set_small_node_limit(self._ctx, limit), self._ctx)

    def set_medium_node_limit(self, limit: int) -> None:
        """Nodes above the small-node limit with at most ``limit`` vertices (max 4096) go through the batched
        medium-node path of the native driver; 0 sends them down the per-node staged path."""
        _check(self._lib.scs_ctx_set_medium_node_limit(self._ctx, limit), self._ctx)

    def set_device_forest(self, on: bool) -> None:
        """Native single-GPU build: keep the source trees on the device for the whole recursion (default) or on
        the host (restriction by the host threads, tours copied per wave)."""
        _check(self._lib.scs_ctx_set_device_forest(self._ctx, int(bool(on))), self._ctx)

    def set_wide_entries(self, on: bool) -> None:
        """Graph build with the 8-byte bucket entries of nodes with >= 65 536 taxa at every size (tests)."""
        _check(self._lib.scs_ctx_set_wide_entries(self._ctx, int(on)), self._ctx)

    def set_full_rows(self, on: bool) -> None:
        """Graph build: every row CTA visits all its leaf pairs instead of the pairs beyond the diagonal + mirror (tests)."""
        _check(self._lib.scs_ctx_set_full_rows(self._ctx, int(on)), self._ctx)

    def stage_seconds(self, reset: bool = True) -> dict:
        """Host wall clock per stage of the staged node path (``scs_ctx_stage_seconds``)."""
        out = np.zeros(8)
        _check(self._lib.scs_ctx_stage_seconds(self._ctx, ptr(out), int(reset)), self._ctx)
        keys = ("enqueue_graph", "wait_graph", "enqueue_contract", "spectral", "result_copy", "lanczos_in_spectral",
                "tour_components")  # fmt: skip
        return dict(zip(keys, out[:7].tolist(), strict=True))

    def flush_l2(self) -> None:
        _check(self._lib.scs_ctx_flush_l2(self._ctx), self._ctx)

    def profile(self, on: bool) -> None:
        _check(self._lib.scs_ctx_profile_enable(self._ctx, int(on)), self._ctx)

    def profile_read(self, kind: int) -> dict:
        """Summed per-launch event timings of one kernel kind (0 matvec, 1 graph-build rows)."""
        n, ms, nbytes, units = ctypes.c_int64(0), ctypes.c_double(0), ctypes.c_double(0), ctypes.c_double(0)
        status = self._lib.scs_ctx_profile_read(
            self._ctx, kind, ctypes.byref(n), ctypes.byref(ms), ctypes.byref(nbytes), ctypes.byref(units)
        )
        _check(status, self._ctx)
        return {"launches": n.value, "ms": ms.value, "bytes": nbytes.value, "units": units.value}

    # -- raw device memory (tests, bench) -------------------------------------------------------
    def alloc(self, nbytes: int) -> int:
        out = ctypes.c_void_p()
        _check(self._lib.scs_dev_alloc(self._ctx, nbytes, ctypes.byref(out)), self._ctx)
        return out.value

    def free(self, dev: int) -> None:
        _check(self._lib.scs_dev_free(self._ctx, dev), self._ctx)

    def to_device(self, array: np.ndarray) -> int:
        array = np.ascontiguousarray(array)
        dev = self.alloc(max(array.nbytes, 16))
        if array.nbytes:
            _check(self._lib.scs_memcpy_h2d(self._ctx, dev, ptr(array), array.nbytes), self._ctx)
        return dev

    def to_host(self, dev: int, shape, dtype) -> np.ndarray:
        out = np.empty(shape, dtype=dtype)
        if out.nbytes:
            _check(self._lib.scs_memcpy_d2h(self._ctx, ptr(out), dev, out.nbytes), self._ctx)
        return out

    # -- one recursion node from host tours (ref: scs.py:110-134) --------------------------------
    def node_split(self, tours, contract_edges: bool = True, seed: int = 0):
        """``(part, stats)`` for the leaf tours of one recursion node (``flatten.LeafTours``)."""
        part = np.empty(tours.n, dtype=np.int32)
        stats = NodeStats()
        status = self._lib.scs_node_split_host(
            self._ctx, tours.n, tours.num_trees, tours.num_leaves, ptr(tours.leaf_offsets), ptr(tours.leaf_taxon),
            ptr(tours.adj_depth), ptr(tours.adj_val), ptr(tours.root_depth), ptr(tours.tree_weight),
            int(bool(contract_edges)), seed & 0xFFFFFFFFFFFFFFFF, ptr(part), ctypes.byref(stats),
        )  # fmt: skip
        _check(status, self._ctx)
        return part, stats

    def forest_split(self, forest: "Forest", weighting: str, contract_edges: bool = True, seed: int = 0):
        """``(taxa, part, stats)``: the vertices (global taxon ids, ascending) of the recursion node
        holding ``forest`` and, per vertex, its component index or spectral side."""
        cap = max(forest.num_taxa, 1)
        taxa = np.empty(cap, dtype=np.int32)
        part = np.empty(cap, dtype=np.int32)
        n = ctypes.c_int32(0)
        stats = NodeStats()
        status = self._lib.scs_forest_split(
            self._ctx, forest.handle, WEIGHTINGS.index(weighting), int(bool(contract_edges)),
            seed & 0xFFFFFFFFFFFFFFFF, ctypes.byref(n), ptr(taxa), ptr(part), ctypes.byref(stats),
        )  # fmt: skip
        if status == _lib.SCS_ERR_INPUT and weighting == "bootstrap":
            # the reference multiplies a missing support by the tree weight (ref: scs.py:655-657)
            msg = "unsupported operand type(s) for *: 'NoneType' and 'float'"
            raise TypeError(msg)
        _check(status, self._ctx)
        return taxa[: n.value].copy(), part[: n.value].copy(), stats

    # -- the whole recursion, natively (csrc/driver.cu) --------------------------------------------
    def supertree_build(self, forest: "Forest", weighting: str, contract_edges: bool = True, seed: int = 0,
                        record: bool = False, rank: int = 0, world: int = 1) -> dict:
        """``scs_supertree_build``: the supertree as flat arrays (``parent[i] < i``, ``taxon`` = global
        taxon id for tips, -1 otherwise), the driver's counters and, if ``record``, one
        ``(taxa, part, stats)`` per recursion node that reached the GPU."""
        handle = ctypes.c_void_p()
        status = self._lib.scs_supertree_build_sharded(
            self._ctx, forest.handle, WEIGHTINGS.index(weighting), int(bool(contract_edges)),
            seed & 0xFFFFFFFFFFFFFFFF, int(bool(record)), rank, world, ctypes.byref(handle),
        )  # fmt: skip
        if status == _lib.SCS_ERR_INPUT and weighting == "bootstrap":
            msg = "unsupported operand type(s) for *: 'NoneType' and 'float'"
            raise TypeError(msg)
        if status == _lib.SCS_ERR_EMPTY:  # ref: scs.py:63-65, reached through the recursion
            msg = "There must be at least one tree to make a supertree."
            raise ValueError(msg)
        _check(status, self._ctx)
        return self._collect_supertree(handle, record)

    def device_forest(self, forest: "Forest", weighting: str) -> "DeviceForest":
        """``scs_device_forest_create``: the source trees uploaded once, to be kept in HBM between builds."""
        handle = ctypes.c_void_p()
        _check(self._lib.scs_device_forest_create(self._ctx, forest.handle, WEIGHTINGS.index(weighting),
                                                  ctypes.byref(handle)), self._ctx)  # fmt: skip
        return DeviceForest(handle, weighting)

    def supertree_build_resident(self, resident: "DeviceForest", contract_edges: bool = True, seed: int = 0,
                                 record: bool = False, rank: int = 0, world: int = 1) -> dict:
        """``scs_supertree_build_resident``: the build of ``supertree_build`` from trees already in HBM."""
        handle = ctypes.c_void_p()
        status = self._lib.scs_supertree_build_resident(
            self._ctx, resident.handle, int(bool(contract_edges)), seed & 0xFFFFFFFFFFFFFFFF, int(bool(record)), rank,
            world, ctypes.byref(handle),
        )  # fmt: skip
        if status == _lib.SCS_ERR_INPUT and resident.weighting == "bootstrap":
            msg = "unsupported operand type(s) for *: 'NoneType' and 'float'"
            raise TypeError(msg)
        if status == _lib.SCS_ERR_EMPTY:
            msg = "There must be at least one tree to make a supertree."
            raise ValueError(msg)
        _check(status, self._ctx)
        return self._collect_supertree(handle, record)

    def supertree_support(self, forest: "Forest", parent, taxon) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """``scs_supertree_support``: per node of the flat supertree (``parent[i] < i``, ``taxon`` = the forest's taxon
        id on tips) the support / conflict / permitted counts ``[n, 3]`` (int32) and their sums over the tree weights
        ``[n, 3]``; per source tree ``[T, 4]``: shared, source and supertree clusters, Robinson-Foulds distance."""
        parent = np.ascontiguousarray(parent, dtype=np.int32)
        taxon = np.ascontiguousarray(taxon, dtype=np.int32)
        n = len(parent)
        if len(taxon) != n:
            msg = "parent and taxon must have the same length"
            raise ValueError(msg)
        counts = np.zeros((n, 3), dtype=np.int32)
        weighted = np.zeros((n, 3), dtype=np.float64)
        per_tree = np.zeros((forest.num_trees, 4), dtype=np.int32)
        status = self._lib.scs_supertree_support(self._ctx, forest.handle, n, ptr(parent), ptr(taxon), ptr(counts),
                                                 ptr(weighted), ptr(per_tree))  # fmt: skip
        _check(status, self._ctx)
        return counts, weighted, per_tree

    def supertree_triplets(self, forest: "Forest", parent, taxon) -> np.ndarray:
        """``scs_supertree_triplets``: per source tree ``[T, 5]`` (int64): shared taxa, triplets resolved in the
        restricted source tree, triplets resolved in the restricted supertree, agreeing and contradicting triplets."""
        parent = np.ascontiguousarray(parent, dtype=np.int32)
        taxon = np.ascontiguousarray(taxon, dtype=np.int32)
        n = len(parent)
        if len(taxon) != n:
            msg = "parent and taxon must have the same length"
            raise ValueError(msg)
        per_tree = np.zeros((forest.num_trees, 5), dtype=np.int64)
        status = self._lib.scs_supertree_triplets(self._ctx, forest.handle, n, ptr(parent), ptr(taxon), ptr(per_tree))
        _check(status, self._ctx)
        return per_tree

    def supertree_taxon_triplets(self, forest: "Forest", parent, taxon) -> tuple[np.ndarray, np.ndarray]:
        """``scs_supertree_taxon_triplets``: per taxon id of ``forest`` ``[num_taxa, 6]`` (int64): source trees sharing
        it with at least two other taxa, triplets containing it, and those of them resolved in the restricted source
        tree, resolved in the restricted supertree, agreeing and contradicting; ``[num_taxa, 3]``: the resolved-source,
        agreeing and contradicting counts summed with the tree weights in tree order."""
        parent = np.ascontiguousarray(parent, dtype=np.int32)
        taxon = np.ascontiguousarray(taxon, dtype=np.int32)
        n = len(parent)
        if len(taxon) != n:
            msg = "parent and taxon must have the same length"
            raise ValueError(msg)
        per_taxon = np.zeros((forest.num_taxa, 6), dtype=np.int64)
        weighted = np.zeros((forest.num_taxa, 3), dtype=np.float64)
        status = self._lib.scs_supertree_taxon_triplets(self._ctx, forest.handle, n, ptr(parent), ptr(taxon),
                                                        ptr(per_taxon), ptr(weighted))  # fmt: skip
        _check(status, self._ctx)
        return per_taxon, weighted

    def supertree_mrp(self, forest: "Forest", parent, taxon) -> np.ndarray:
        """``scs_supertree_mrp``: per source tree ``[T, 4]`` (int64): shared taxa, MRP characters (the non-trivial
        clusters of the restricted source tree), their summed parsimony length on the supertree (steps), and the
        characters of length 1."""
        parent = np.ascontiguousarray(parent, dtype=np.int32)
        taxon = np.ascontiguousarray(taxon, dtype=np.int32)
        n = len(parent)
        if len(taxon) != n:
            msg = "parent and taxon must have the same length"
            raise ValueError(msg)
        per_tree = np.zeros((forest.num_trees, 4), dtype=np.int64)
        status = self._lib.scs_supertree_mrp(self._ctx, forest.handle, n, ptr(parent), ptr(taxon), ptr(per_tree))
        _check(status, self._ctx)
        return per_tree

    def forest_pairwise_rf(self, forest: "Forest") -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """``scs_forest_pairwise_rf``: for every pair of source trees, restricted to the taxa they share, three
        ``[T, T]`` int32 matrices: the shared taxa, the non-trivial clusters of row tree i's restriction (not
        symmetric) and the clusters the two restrictions have in common."""
        T = forest.num_trees
        shared = np.zeros((T, T), dtype=np.int32)
        clusters = np.zeros((T, T), dtype=np.int32)
        common = np.zeros((T, T), dtype=np.int32)
        status = self._lib.scs_forest_pairwise_rf(self._ctx, forest.handle, ptr(shared), ptr(clusters), ptr(common))
        _check(status, self._ctx)
        return shared, clusters, common

    def _collect_supertree(self, handle, record: bool) -> dict:
        try:
            count = self._lib.scs_supertree_num_nodes(handle)
            parent = np.empty(count, dtype=np.int32)
            taxon = np.empty(count, dtype=np.int32)
            _check(self._lib.scs_supertree_nodes(handle, ptr(parent), ptr(taxon)), self._ctx)
            small, large, waves, pairs = (ctypes.c_int64(0) for _ in range(4))
            self._lib.scs_supertree_counters(handle, ctypes.byref(small), ctypes.byref(large), ctypes.byref(waves),
                                             ctypes.byref(pairs))  # fmt: skip
            seconds = np.zeros(4)
            self._lib.scs_supertree_seconds(handle, ptr(seconds))
            medium, rerun, medium_s = ctypes.c_int64(0), ctypes.c_int64(0), ctypes.c_double(0.0)
            self._lib.scs_supertree_medium_info(handle, ctypes.byref(medium), ctypes.byref(rerun), ctypes.byref(medium_s))
            wave_tasks = np.zeros(max(waves.value, 1), dtype=np.int32)
            wave_max_n = np.zeros(max(waves.value, 1), dtype=np.int32)
            self._lib.scs_supertree_wave_info(handle, ptr(wave_tasks), ptr(wave_max_n))
            wave_seconds = np.zeros((max(waves.value, 1), 3))
            self._lib.scs_supertree_wave_seconds(handle, ptr(wave_seconds))
            out = {"parent": parent, "taxon": taxon, "nodes_small": small.value, "nodes_large": large.value,
                   "nodes_medium": medium.value, "nodes_rerun": rerun.value, "medium_seconds": medium_s.value,
                   "waves": waves.value, "pair_visits": pairs.value, "records": [],
                   "shared_prefix": int(self._lib.scs_supertree_shared_prefix(handle)),
                   "shared_records": int(self._lib.scs_supertree_shared_records(handle)),
                   "wave_tasks": wave_tasks[: waves.value].tolist(), "wave_max_n": wave_max_n[: waves.value].tolist(),
                   "wave_seconds": wave_seconds[: waves.value].tolist(),
                   "seconds": dict(zip(("large_nodes", "small_batches", "restrict", "tours"), seconds.tolist(), strict=True))}  # fmt: skip
            if record:
                for i in range(self._lib.scs_supertree_num_records(handle)):
                    n = self._lib.scs_supertree_record_size(handle, i)
                    taxa = np.empty(n, dtype=np.int32)
                    part = np.empty(n, dtype=np.int32)
                    stats = NodeStats()
                    self._lib.scs_supertree_record(handle, i, ptr(taxa), ptr(part), ctypes.byref(stats))
                    out["records"].append((taxa, part, stats))
                out["record_waves"] = [int(self._lib.scs_supertree_record_wave(handle, i))
                                       for i in range(len(out["records"]))]
            return out
        finally:
            self._lib.scs_supertree_destroy(handle)

    # -- one node over several GPUs (csrc/shard.cu) -------------------------------------------------
    def shard_create(self, rank: int, world: int, n_max: int) -> bytes:
        """Allocate this rank's exchange window; returns its IPC handle (64 opaque bytes) for the peers."""
        handle = (ctypes.c_ubyte * _lib.IPC_HANDLE_BYTES)()
        _check(self._lib.scs_shard_create(self._ctx, rank, world, n_max, ctypes.addressof(handle)), self._ctx)
        return bytes(handle)

    def shard_connect(self, handles: Sequence[bytes]) -> None:
        """Map the peers' windows from their IPC handles (all ranks' handles, in rank order)."""
        blob = b"".join(handles)
        buf = (ctypes.c_ubyte * len(blob)).from_buffer_copy(blob)
        _check(self._lib.scs_shard_connect_ipc(self._ctx, ctypes.addressof(buf)), self._ctx)

    def shard_window(self) -> int:
        out, size = ctypes.c_void_p(), ctypes.c_size_t(0)
        _check(self._lib.scs_shard_window(self._ctx, ctypes.byref(out), ctypes.byref(size)), self._ctx)
        return out.value

    def shard_connect_local(self, windows: Sequence[int]) -> None:
        """Peers in this process (one Engine per GPU, or several on one GPU): raw window pointers."""
        arr = (ctypes.c_void_p * len(windows))(*windows)
        _check(self._lib.scs_shard_connect_ptrs(self._ctx, ctypes.addressof(arr)), self._ctx)

    def shard_engage(self, on: bool = True) -> None:
        _check(self._lib.scs_shard_engage(self._ctx, int(on)), self._ctx)

    def shard_configure(self, min_n: int = 0, timeout_seconds: float = 0.0) -> None:
        _check(self._lib.scs_shard_configure(self._ctx, int(min_n), float(timeout_seconds)), self._ctx)

    def shard_barrier(self) -> None:
        _check(self._lib.scs_shard_barrier(self._ctx), self._ctx)

    @property
    def shard_nodes(self) -> int:
        return int(self._lib.scs_shard_nodes(self._ctx))

    def shard_destroy(self) -> None:
        _check(self._lib.scs_shard_destroy(self._ctx), self._ctx)

    # -- single stages on explicit device buffers (parity tests, profiling, bench) ---------------
    def upload_tours(self, tours) -> dict:
        """Device copies of a ``LeafTours`` (free with ``free_tours``)."""
        return {
            "n": tours.n, "T": tours.num_trees, "L": tours.num_leaves,
            "leaf_offsets": self.to_device(tours.leaf_offsets), "leaf_taxon": self.to_device(tours.leaf_taxon),
            "adj_depth": self.to_device(tours.adj_depth), "adj_val": self.to_device(tours.adj_val),
            "root_depth": self.to_device(tours.root_depth), "tree_weight": self.to_device(tours.tree_weight),
        }  # fmt: skip

    def free_tours(self, dev: dict) -> None:
        for key in ("leaf_offsets", "leaf_taxon", "adj_depth", "adj_val", "root_depth", "tree_weight"):
            self.free(dev[key])

    def node_split_dev(self, dev: dict, part_dev: int, contract_edges: bool = True, seed: int = 0) -> NodeStats:
        """One recursion node on tours already resident in HBM (``upload_tours``)."""
        stats = NodeStats()
        status = self._lib.scs_node_split_dev(
            self._ctx, dev["n"], dev["T"], dev["L"], dev["leaf_offsets"], dev["leaf_taxon"], dev["adj_depth"],
            dev["adj_val"], dev["root_depth"], dev["tree_weight"], int(bool(contract_edges)),
            seed & 0xFFFFFFFFFFFFFFFF, part_dev, ctypes.byref(stats),
        )  # fmt: skip
        _check(status, self._ctx)
        return stats

    def pcg_build(self, tours, want_counts: bool = True) -> dict:
        """``scs_pcg_build_dev`` on fresh device buffers; returns host copies of every output."""
        n = tours.n
        words = self._lib.scs_bit_words(n)
        dev = self.upload_tours(tours)
        bufs = {
            "W": self.alloc(8 * n * n), "C": self.alloc(4 * n * n) if want_counts else None,
            "occ": self.alloc(4 * n), "adj_bits": self.alloc(4 * n * words), "max_bits": self.alloc(4 * n * words),
            "degree": self.alloc(8 * n),
        }  # fmt: skip
        try:
            # poison the outputs: an entry the build forgets to write must not look right by accident
            poison = np.full(n * max(n, words) * 8, 0xFF, dtype=np.uint8)
            for key, nbytes in (("W", 8 * n * n), ("adj_bits", 4 * n * words), ("max_bits", 4 * n * words), ("degree", 8 * n)):
                _check(self._lib.scs_memcpy_h2d(self._ctx, bufs[key], ptr(poison), nbytes), self._ctx)
            status = self._lib.scs_pcg_build_dev(
                self._ctx, n, dev["T"], dev["L"], dev["leaf_offsets"], dev["leaf_taxon"], dev["adj_depth"],
                dev["adj_val"], dev["root_depth"], dev["tree_weight"], bufs["W"], bufs["C"], bufs["occ"],
                bufs["adj_bits"], bufs["max_bits"], bufs["degree"],
            )  # fmt: skip
            _check(status, self._ctx)
            self.synchronize()
            out = {
                "W": self.to_host(bufs["W"], (n, n), np.float64),
                "occ": self.to_host(bufs["occ"], (n,), np.int32),
                "adj_bits": self.to_host(bufs["adj_bits"], (n, words), np.uint32),
                "max_bits": self.to_host(bufs["max_bits"], (n, words), np.uint32),
                "degree": self.to_host(bufs["degree"], (n,), np.float64),
            }
            if want_counts:
                out["C"] = self.to_host(bufs["C"], (n, n), np.int32)
            return out
        finally:
            self.free_tours(dev)
            for b in bufs.values():
                if b:
                    self.free(b)

    def components(self, bits: np.ndarray, n: int) -> tuple[np.ndarray, int]:
        """``scs_components_dev``: (label = smallest vertex of the component, number of components)."""
        d_bits = self.to_device(bits)
        d_label = self.alloc(4 * n)
        count = ctypes.c_int32(0)
        try:
            _check(self._lib.scs_components_dev(self._ctx, n, d_bits, d_label, ctypes.byref(count)), self._ctx)
            return self.to_host(d_label, (n,), np.int32), count.value
        finally:
            self.free(d_bits)
            self.free(d_label)

    def contract(self, W: np.ndarray, adj_bits: np.ndarray, max_bits: np.ndarray):
        """``scs_contract_dev``: (group, m, Wc[m, m], degree_c[m])."""
        n = W.shape[0]
        d_W, d_adj, d_max = self.to_device(W), self.to_device(adj_bits), self.to_device(max_bits)
        d_group, d_Wc, d_deg = self.alloc(4 * n), self.alloc(8 * n * n), self.alloc(8 * n)
        m = ctypes.c_int32(0)
        try:
            status = self._lib.scs_contract_dev(self._ctx, n, d_W, d_adj, d_max, d_group, ctypes.byref(m), d_Wc, d_deg)
            _check(status, self._ctx)
            m = m.value
            group = self.to_host(d_group, (n,), np.int32)
            if m == n:
                return group, m, W.copy(), W.sum(axis=1)
            return group, m, self.to_host(d_Wc, (m, m), np.float64), self.to_host(d_deg, (m,), np.float64)
        finally:
            for d in (d_W, d_adj, d_max, d_group, d_Wc, d_deg):
                self.free(d)

    def spectral_bipartition(self, W: np.ndarray, seed: int = 0, degree: np.ndarray | None = None):
        """``scs_spectral_bipartition_dev``: (side[m], stats)."""
        W = np.ascontiguousarray(W, dtype=np.float64)
        m = W.shape[0]
        d_W = self.to_device(W)
        d_deg = None if degree is None else self.to_device(np.ascontiguousarray(degree, dtype=np.float64))
        d_side = self.alloc(4 * max(m, 1))
        stats = NodeStats()
        try:
            status = self._lib.scs_spectral_bipartition_dev(
                self._ctx, m, d_W, d_deg, seed & 0xFFFFFFFFFFFFFFFF, d_side, ctypes.byref(stats)
            )
            _check(status, self._ctx)
            return self.to_host(d_side, (m,), np.int32), stats
        finally:
            self.free(d_W)
            self.free(d_side)
            if d_deg:
                self.free(d_deg)

    def normalized_matvec(self, W: np.ndarray, inv_sqrt_deg: np.ndarray, x: np.ndarray) -> np.ndarray:
        """``scs_normalized_matvec_dev``: D^-1/2 W D^-1/2 x."""
        m = W.shape[0]
        d_W, d_s, d_x, d_y = self.to_device(W), self.to_device(inv_sqrt_deg), self.to_device(x), self.alloc(8 * m)
        try:
            _check(self._lib.scs_normalized_matvec_dev(self._ctx, m, d_W, d_s, d_x, d_y), self._ctx)
            return self.to_host(d_y, (m,), np.float64)
        finally:
            for d in (d_W, d_s, d_x, d_y):
                self.free(d)

    def last_node_pointers(self) -> dict:
        """Device addresses and shape of the node most recently split (``scs_node_last_buffers``): for checks that
        cannot afford host copies of whole matrices."""
        n, m = ctypes.c_int(0), ctypes.c_int(0)
        ptrs = [ctypes.c_void_p() for _ in range(7)]
        _check(
            self._lib.scs_node_last_buffers(self._ctx, ctypes.byref(n), ctypes.byref(m), *[ctypes.byref(p) for p in ptrs]),
            self._ctx,
        )
        names = ("W", "adj_bits", "max_bits", "occ", "degree", "Wc", "group")
        out = {k: p.value for k, p in zip(names, ptrs, strict=True)}
        out.update({"n": n.value, "m": m.value})
        return out

    def last_node_rows(self, row_lo: int, row_hi: int) -> tuple[np.ndarray, np.ndarray]:
        """Rows [row_lo, row_hi) of W and of the adjacency bits of the node most recently split."""
        p = self.last_node_pointers()
        n = p["n"]
        words = self._lib.scs_bit_words(n)
        W = self.to_host(p["W"] + 8 * row_lo * n, (row_hi - row_lo, n), np.float64)
        bits = self.to_host(p["adj_bits"] + 4 * row_lo * words, (row_hi - row_lo, words), np.uint32)
        return W, bits

    def matvec_on_device(self, m: int, W_dev: int, isd_dev: int, x: np.ndarray) -> np.ndarray:
        """y = D^-1/2 W D^-1/2 x with W and 1/sqrt(d) already on the device (``scs_normalized_matvec_dev``)."""
        d_x = self.to_device(np.ascontiguousarray(x, dtype=np.float64))
        d_y = self.alloc(8 * m)
        try:
            _check(self._lib.scs_normalized_matvec_dev(self._ctx, m, W_dev, isd_dev, d_x, d_y), self._ctx)
            return self.to_host(d_y, (m,), np.float64)
        finally:
            self.free(d_x)
            self.free(d_y)

    def last_node_buffers(self) -> dict:
        """Host copies of the device buffers of the node most recently split (parity tests)."""
        n, m = ctypes.c_int(0), ctypes.c_int(0)
        ptrs = [ctypes.c_void_p() for _ in range(7)]
        _check(
            self._lib.scs_node_last_buffers(self._ctx, ctypes.byref(n), ctypes.byref(m), *[ctypes.byref(p) for p in ptrs]),
            self._ctx,
        )
        n, m = n.value, m.value
        words = self._lib.scs_bit_words(n)
        W, adj, mx, occ, deg, Wc, group = (p.value for p in ptrs)
        out = {"n": n, "m": m}
        out["W"] = self.to_host(W, (n, n), np.float64)
        out["adj_bits"] = self.to_host(adj, (n, words), np.uint32)
        out["occ"] = self.to_host(occ, (n,), np.int32)
        out["degree"] = self.to_host(deg, (n,), np.float64)
        if mx:
            out["max_bits"] = self.to_host(mx, (n, words), np.uint32)
        if m and m != n and Wc and group:
            out["Wc"] = self.to_host(Wc, (m, m), np.float64)
            out["group"] = self.to_host(group, (n,), np.int32)
        return out


def merge_sharded(parts: list[tuple[np.ndarray, np.ndarray, int]]) -> tuple[np.ndarray, np.ndarray]:
    """Join the outputs of ``supertree_build(rank=r, world=N)`` for r = 0..N-1.

    ``parts[r] = (parent, taxon, shared_prefix)``.  Nodes ``[0, shared_prefix)`` are identical on
    every rank; each rank's remaining nodes hang below its own sub-problems, so they are appended
    with their parent indices shifted."""
    parent0, taxon0, prefix = parts[0]
    parents = [np.asarray(parent0, dtype=np.int32)]
    taxa = [np.asarray(taxon0, dtype=np.int32)]
    # a tip placed into a shared slot by its owner (a sub-problem that resolved to a single tip) must win
    head_taxon = taxa[0][:prefix].copy()
    offset = len(parent0)
    for parent, taxon, p in parts[1:]:
        if p != prefix:
            msg = f"ranks disagree on the shared prefix ({p} != {prefix})"
            raise ValueError(msg)
        parent = np.asarray(parent, dtype=np.int32)
        taxon = np.asarray(taxon, dtype=np.int32)
        head_taxon = np.maximum(head_taxon, taxon[:prefix])
        tail = parent[prefix:].copy()
        tail[tail >= prefix] += offset - prefix
        parents.append(tail)
        taxa.append(taxon[prefix:])
        offset += len(tail)
    taxa[0] = np.concatenate([head_taxon, taxa[0][prefix:]])
    return np.concatenate(parents), np.concatenate(taxa)


def set_host_threads(threads: int) -> None:
    """Host threads for tree restriction / flattening / the recursion driver (0 = OpenMP default)."""
    status = _lib.load().scs_set_host_threads(int(threads))
    if status != _lib.SCS_OK:
        raise ScsError(status, "scs_set_host_threads")


_DEFAULT: Engine | None = None


_FASTFLATTEN = None


def _fastflatten():
    """The CPython accelerator of ``Forest.from_trees`` (csrc/fastflatten.c), built on first use; None if it cannot be
    built or imported (the Python loop below is then used: host-side glue, not compute)."""
    global _FASTFLATTEN  # noqa: PLW0603
    if _FASTFLATTEN is None:
        try:
            from . import build as _build

            _build.build_fastflatten()
            from . import _fastflatten as module

            _FASTFLATTEN = module
        except Exception:  # noqa: BLE001
            _FASTFLATTEN = False
    return _FASTFLATTEN or None


def default_engine() -> Engine:
    """The process-wide engine used by ``construct_supertree`` (device from ``SCS_B200_DEVICE``)."""
    global _DEFAULT  # noqa: PLW0603
    if _DEFAULT is None:
        _DEFAULT = Engine()
    return _DEFAULT


def unpack_bits(bits: np.ndarray, n: int) -> np.ndarray:
    """Bit matrix (n x words uint32, bit b of word j = column 32 j + b) -> boolean n x n."""
    as_bytes = bits.view(np.uint8).reshape(bits.shape[0], -1)
    return np.unpackbits(as_bytes, axis=1, bitorder="little")[:, :n].astype(bool)


class DeviceForest:
    """Source trees resident on the device (owner of one ``scs_device_forest``)."""

    def __init__(self, handle, weighting: str) -> None:
        self._lib = _lib.load()
        self.handle = handle
        self.weighting = weighting

    @property
    def nbytes(self) -> int:
        return int(self._lib.scs_device_forest_bytes(self.handle))

    def close(self) -> None:
        if self.handle:
            self._lib.scs_device_forest_destroy(self.handle)
            self.handle = None


class Forest:
    """Flat source trees + weights (owner of one ``scs_forest``)."""

    def __init__(self, handle, names: Sequence[str]) -> None:
        self._lib = _lib.load()
        self._handle = handle
        self.names = names  # global taxon id -> name (sorted)

    # -- construction --------------------------------------------------------------------------
    @classmethod
    def from_arrays(cls, node_offsets, parent, length, support, taxon, weights, names: Sequence[str],
                    copy: bool = False) -> "Forest":
        """Flat source trees (pre-order nodes per tree) as a forest.  By default the per-node arrays are not copied
        (``scs_forest_create_view``): the forest refers to them and this object keeps them alive -- do not modify them
        while it exists; ``copy=True`` makes the library own a copy (``scs_forest_create``)."""
        lib = _lib.load()
        node_offsets = np.ascontiguousarray(node_offsets, dtype=np.int64)
        parent = np.ascontiguousarray(parent, dtype=np.int32)
        taxon = np.ascontiguousarray(taxon, dtype=np.int32)
        length = None if length is None else np.ascontiguousarray(length, dtype=np.float64)
        support = None if support is None else np.ascontiguousarray(support, dtype=np.float64)
        weights = np.ascontiguousarray(weights, dtype=np.float64)
        handle = ctypes.c_void_p()
        create = lib.scs_forest_create if copy else lib.scs_forest_create_view
        status = create(
            len(weights), ptr(node_offsets), ptr(parent), ptr(length), ptr(support), ptr(taxon), ptr(weights),
            len(names), ctypes.byref(handle),
        )  # fmt: skip
        if status != _lib.SCS_OK:
            raise ScsError(status, "scs_forest_create: " + lib.scs_forest_last_error().decode())
        forest = cls(handle, names)
        if not copy:
            forest._borrowed = (parent, length, support, taxon)  # the library reads these until the forest is closed
        return forest

    @classmethod
    def from_trees(cls, trees: Sequence, weights: Sequence[float], names: Sequence[str] | None = None) -> "Forest":
        """Flatten tree objects exposing the PhyloNode surface (children iteration, ``name``,
        ``length``, ``support``; ref: scs.py:570,624-631,560-564)."""
        fast = _fastflatten()
        if fast is not None:
            # csrc/fastflatten.c: one C-level walk over the node objects; tips numbered in first-seen order there,
            # renumbered here by rank in the sorted name list (global taxon id = rank of the name)
            raw_off, raw_par, raw_len, raw_sup, raw_tax, seen = fast.flatten(list(trees))
            if names is None:
                names = sorted(seen)
            taxon_id = {name: i for i, name in enumerate(names)}
            remap = np.fromiter((taxon_id[name] for name in seen), dtype=np.int32, count=len(seen))
            taxon = np.frombuffer(raw_tax, dtype=np.int32)
            if len(remap):
                taxon = np.where(taxon >= 0, remap[np.maximum(taxon, 0)], -1).astype(np.int32)
            return cls.from_arrays(np.frombuffer(raw_off, dtype=np.int64), np.frombuffer(raw_par, dtype=np.int32),
                                   np.frombuffer(raw_len, dtype=np.float64), np.frombuffer(raw_sup, dtype=np.float64),
                                   taxon, list(weights), names)  # fmt: skip
        if names is None:
            found: set[str] = set()
            for tree in trees:
                found.update(tree.get_tip_names())
            names = sorted(found)
        taxon_id = {name: i for i, name in enumerate(names)}
        offsets = [0]
        parent: list[int] = []
        length: list[float] = []
        support: list[float] = []
        taxon: list[int] = []
        nan = float("nan")
        for tree in trees:
            base = len(parent)
            stack = [(tree, -1)]
            while stack:
                node, up = stack.pop()
                k = len(parent) - base
                parent.append(up)
                ln, sp = node.length, getattr(node, "support", None)
                length.append(nan if ln is None else float(ln))
                support.append(nan if sp is None else float(sp))
                kids = list(node)
                if kids:
                    taxon.append(-1)
                    stack.extend((child, k) for child in reversed(kids))
                else:
                    taxon.append(taxon_id[node.name])
            offsets.append(len(parent))
        return cls.from_arrays(offsets, parent, length, support, taxon, list(weights), names)

    @classmethod
    def from_newick(cls, text: bytes | str) -> "Forest":
        """Line-separated Newick text straight into the flat store (``scs_forest_parse_newick``): no node
        objects.  Raises ``NewickError`` on a syntax error, like ``make_tree``."""
        from .tree import NewickError

        lib = _lib.load()
        data = text.encode("utf-8") if isinstance(text, str) else bytes(text)
        handle, names_ptr = ctypes.c_void_p(), ctypes.c_void_p()
        names_bytes, num_taxa = ctypes.c_size_t(), ctypes.c_int()
        status = lib.scs_forest_parse_newick(data, len(data), ctypes.byref(handle), ctypes.byref(names_ptr),
                                             ctypes.byref(names_bytes), ctypes.byref(num_taxa))  # fmt: skip
        if status == _lib.SCS_ERR_INPUT:
            raise NewickError(lib.scs_newick_last_error().decode())
        if status != _lib.SCS_OK:
            raise ScsError(status, "scs_forest_parse_newick")
        try:
            raw = ctypes.string_at(names_ptr, names_bytes.value)
        finally:
            lib.scs_free(names_ptr)
        names = [part.decode("utf-8") for part in raw.split(b"\0")[: num_taxa.value]]
        return cls(handle, names)

    def close(self) -> None:
        if getattr(self, "_handle", None):
            self._lib.scs_forest_destroy(self._handle)
            self._handle = None

    def __del__(self) -> None:  # pragma: no cover
        try:
            self.close()
        except Exception:  # noqa: BLE001, S110
            pass

    # -- queries -------------------------------------------------------------------------------
    @property
    def handle(self):
        return self._handle

    @property
    def num_trees(self) -> int:
        return self._lib.scs_forest_num_trees(self._handle)

    @property
    def num_nodes(self) -> int:
        return self._lib.scs_forest_num_nodes(self._handle)

    @property
    def num_leaves(self) -> int:
        return self._lib.scs_forest_num_leaves(self._handle)

    @property
    def num_taxa(self) -> int:
        return self._lib.scs_forest_num_taxa(self._handle)

    @property
    def pair_visits(self) -> int:
        return self._lib.scs_forest_pair_visits(self._handle)

    def taxa(self) -> np.ndarray:
        """Global ids of the taxa present, ascending (ref: scs.py:708-725)."""
        present = np.zeros(max(self.num_taxa, 1), dtype=np.uint8)
        n = self._lib.scs_forest_taxa(self._handle, ptr(present))
        if n < 0:
            raise ScsError(n, "scs_forest_taxa")
        return np.flatnonzero(present[: self.num_taxa]).astype(np.int32)

    def tree_arrays(self, t: int):
        """``(parent, length, support, taxon)`` of tree ``t`` (pre-order)."""
        count = ctypes.c_int64(0)
        status = self._lib.scs_forest_tree_info(self._handle, t, ctypes.byref(count), None, None)
        if status != _lib.SCS_OK:
            raise ScsError(status, "scs_forest_tree_info")
        m = count.value
        parent = np.empty(m, dtype=np.int32)
        length = np.empty(m, dtype=np.float64)
        support = np.empty(m, dtype=np.float64)
        taxon = np.empty(m, dtype=np.int32)
        status = self._lib.scs_forest_tree(self._handle, t, ptr(parent), ptr(length), ptr(support), ptr(taxon))
        if status != _lib.SCS_OK:
            raise ScsError(status, "scs_forest_tree")
        return parent, length, support, taxon

    def weights(self) -> np.ndarray:
        out = np.empty(self.num_trees, dtype=np.float64)
        w = ctypes.c_double(0.0)
        for t in range(self.num_trees):
            self._lib.scs_forest_tree_info(self._handle, t, None, ctypes.byref(w), None)
            out[t] = w.value
        return out

    # -- operations ----------------------------------------------------------------------------
    def induce(self, keep_ids: np.ndarray) -> "Forest":
        """Restrict every tree to the given global taxon ids (ref: scs.py:411-455)."""
        keep = np.zeros(max(self.num_taxa, 1), dtype=np.uint8)
        keep[keep_ids] = 1
        handle = ctypes.c_void_p()
        status = self._lib.scs_forest_induce(self._handle, ptr(keep), ctypes.byref(handle))
        if status != _lib.SCS_OK:
            raise ScsError(status, "scs_forest_induce")
        return Forest(handle, self.names)

    def induce_parts(self, part_of_taxon: np.ndarray, count: int) -> tuple[list["Forest"], np.ndarray]:
        """All restrictions of one recursion node at once (ref: scs.py:139-155): forest ``c`` keeps the
        taxa with ``part_of_taxon[x] == c``.  Also returns the taxa still present in some restricted tree."""
        part = np.ascontiguousarray(part_of_taxon, dtype=np.int32)
        if len(part) < self.num_taxa:
            msg = "part_of_taxon needs one entry per global taxon id"
            raise ValueError(msg)
        handles = (ctypes.c_void_p * max(count, 1))()
        present = np.zeros(max(self.num_taxa, 1), dtype=np.uint8)
        status = self._lib.scs_forest_induce_parts(self._handle, ptr(part), count, ctypes.addressof(handles), ptr(present))
        if status != _lib.SCS_OK:
            raise ScsError(status, "scs_forest_induce_parts")
        forests = [Forest(ctypes.c_void_p(handles[c]), self.names) for c in range(count)]
        return forests, np.flatnonzero(present[: self.num_taxa]).astype(np.int32)

    def tours(self, weighting: str, local_id: np.ndarray | None = None):
        """Leaf tours (``flatten.LeafTours``) with vertex ids = rank among the taxa present."""
        from .flatten import LeafTours

        present = self.taxa()
        if local_id is None:
            local_id = np.full(max(self.num_taxa, 1), -1, dtype=np.int32)
            local_id[present] = np.arange(len(present), dtype=np.int32)
        T, L = self.num_trees, self.num_leaves
        out = LeafTours(
            n=len(present),
            leaf_offsets=np.zeros(T + 1, dtype=np.int64),
            leaf_taxon=np.zeros(L, dtype=np.int32),
            adj_depth=np.zeros(L, dtype=np.int32),
            adj_val=np.zeros(L, dtype=np.float64),
            root_depth=np.zeros(T, dtype=np.int32),
            tree_weight=np.zeros(T, dtype=np.float64),
        )
        status = self._lib.scs_forest_tours(
            self._handle, WEIGHTINGS.index(weighting), ptr(local_id), ptr(out.leaf_offsets), ptr(out.leaf_taxon),
            ptr(out.adj_depth), ptr(out.adj_val), ptr(out.root_depth), ptr(out.tree_weight),
        )  # fmt: skip
        if status == _lib.SCS_ERR_INPUT and weighting == "bootstrap":
            msg = "unsupported operand type(s) for *: 'NoneType' and 'float'"
            raise TypeError(msg)
        if status != _lib.SCS_OK:
            raise ScsError(status, "scs_forest_tours")
        return out
