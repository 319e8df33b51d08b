"""GPU: one recursion node row-sharded over several ranks (csrc/shard.cu) must give, bit for bit, what
one GPU gives -- W rows, components, contraction and the Lanczos iterates are the same arithmetic
whoever owns the row.

Two set-ups: ranks as host threads of this process (one context each; on a 1-GPU box they share the
GPU, with 2+ GPUs they sit on different devices with peer access), and ranks as separate processes
over CUDA IPC (the production layout: one process per GPU; needs 2 GPUs)."""

from __future__ import annotations

import os
import subprocess
import sys
import threading
from pathlib import Path

import numpy as np
import pytest

from spectralclustersupertree_b200.engine import Engine, Forest, merge_sharded
from spectralclustersupertree_b200.synthetic import make_problem

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def device_count() -> int:
    import torch

    return torch.cuda.device_count()


def forest_of(arrays) -> Forest:
    return Forest.from_arrays(arrays["node_offsets"], arrays["parent"], arrays["length"], arrays["support"],
                              arrays["taxon"], arrays["weights"], arrays["names"])  # fmt: skip


class Ranks:
    """`world` contexts in this process, their exchange windows connected by pointer."""

    def __init__(self, world: int, n_max: int, min_n: int) -> None:
        gpus = max(device_count(), 1)
        self.world = world
        self.engines = [Engine(r % gpus) for r in range(world)]
        for r, eng in enumerate(self.engines):
            eng.shard_create(r, world, n_max)
            eng.shard_configure(min_n=min_n, timeout_seconds=30.0)
        windows = [eng.shard_window() for eng in self.engines]
        for eng in self.engines:
            eng.shard_connect_local(windows)

    def run(self, fn):
        """fn(rank, engine) on one thread per rank; re-raises the first failure."""
        out = [None] * self.world
        errors = []

        def work(r):
            try:
                out[r] = fn(r, self.engines[r])
            except BaseException as exc:  # noqa: BLE001
                errors.append(exc)

        threads = [threading.Thread(target=work, args=(r,)) for r in range(self.world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        return out

    def close(self) -> None:
        for eng in self.engines:
            eng.synchronize()
        for eng in self.engines:
            eng.close()


@pytest.mark.parametrize(
    ("n", "trees", "weighting", "world", "contract"),
    [(600, 60, "branch", 2, True), (600, 60, "depth", 3, True), (900, 80, "one", 2, False),
     (5000, 160, "branch", 2, True)],
)  # fmt: skip
def test_sharded_node_equals_single_gpu(engine, n, trees, weighting, world, contract):
    arrays = make_problem(n, trees, weighting, 77 + n, tree_weights=weighting == "branch").forest_arrays()
    forest = forest_of(arrays)
    tours = forest.tours(weighting)
    # descend to the first connected node so that contraction and the spectral step run
    want_part, want = engine.node_split(tours, contract_edges=contract, seed=5)
    while want.n_components != 1:
        sizes = np.bincount(want_part)
        forest = forest.induce(forest.taxa()[want_part == np.argmax(sizes)])
        tours = forest.tours(weighting)
        want_part, want = engine.node_split(tours, contract_edges=contract, seed=5)
    assert want.spectral_ran and tours.n >= 64

    ranks = Ranks(world, n_max=tours.n, min_n=64)
    try:
        # first un-engaged (grows every workspace without a peer waiting), then cooperatively
        ranks.run(lambda r, eng: eng.node_split(tours, contract_edges=contract, seed=5))
        for eng in ranks.engines:
            eng.shard_engage(True)
        got = ranks.run(lambda r, eng: eng.node_split(tours, contract_edges=contract, seed=5))
        for eng in ranks.engines:
            assert eng.shard_nodes == 1
        for part, stats in got:
            assert np.array_equal(part, want_part)
            assert stats.contracted_size == want.contracted_size
            assert stats.matvecs == want.matvecs
            assert stats.eig[1] == want.eig[1]  # bit for bit: the same arithmetic whoever owns a row
            assert stats.residual == want.residual
            assert stats.tie_flag == want.tie_flag
    finally:
        ranks.close()


def test_sharded_disconnected_node_labels_components(engine):
    arrays = make_problem(700, 40, "depth", 4242).forest_arrays()
    tours = forest_of(arrays).tours("depth")
    want_part, want = engine.node_split(tours, seed=1)
    ranks = Ranks(2, n_max=tours.n, min_n=64)
    try:
        ranks.run(lambda r, eng: eng.node_split(tours, seed=1))
        for eng in ranks.engines:
            eng.shard_engage(True)
        for part, stats in ranks.run(lambda r, eng: eng.node_split(tours, seed=1)):
            assert stats.n_components == want.n_components
            assert np.array_equal(part, want_part)
    finally:
        ranks.close()


@pytest.mark.parametrize("shared_upload", [False, True])
def test_sharded_build_equals_single_gpu_build(engine, monkeypatch, shared_upload):
    """The native recursion with the large nodes shared out and the frontier dealt out afterwards; with
    shared_upload every rank sends only its slice of the source trees over PCIe and gathers the rest from the
    peers' windows (csrc/devforest.cu: devforest_upload, cooperative)."""
    if shared_upload:
        monkeypatch.setenv("SCS_SHARED_UPLOAD_MIN_NODES", "0")
    arrays = make_problem(1500, 120, "branch", 99, tree_weights=True).forest_arrays()
    single = engine.supertree_build(forest_of(arrays), "branch")
    ranks = Ranks(2, n_max=1500, min_n=256)
    try:
        ranks.run(lambda r, eng: eng.supertree_build(forest_of(arrays), "branch"))  # warm-up, alone
        built = ranks.run(lambda r, eng: eng.supertree_build(forest_of(arrays), "branch", rank=r, world=2))
        assert all(eng.shard_nodes > 0 for eng in ranks.engines)
        parent, taxon = merge_sharded([(b["parent"], b["taxon"], b["shared_prefix"]) for b in built])
    finally:
        ranks.close()
    from helpers import rf
    from spectralclustersupertree_b200.scs import _tree_from_flat

    a = _tree_from_flat(single["parent"], single["taxon"], arrays["names"])
    b = _tree_from_flat(parent, taxon, arrays["names"])
    assert sorted(b.get_tip_names()) == sorted(a.get_tip_names())
    assert rf(a, b) == 0


def test_peer_timeout_is_an_error_not_a_hang(engine):
    """A rank whose peer never shows up gets SCS_ERR_PEER after the configured timeout."""
    from spectralclustersupertree_b200 import _lib
    from spectralclustersupertree_b200.engine import ScsError

    ranks = Ranks(2, n_max=256, min_n=64)
    try:
        ranks.engines[0].shard_configure(timeout_seconds=0.5)
        with pytest.raises(ScsError) as err:
            ranks.engines[0].shard_barrier()  # rank 1 never arrives
        assert err.value.status == _lib.SCS_ERR_PEER
    finally:
        ranks.close()


def test_two_processes_over_cuda_ipc():
    """One process per rank, windows mapped through cudaIpc handles exchanged with torch.distributed.  With a
    single GPU both ranks share it (the worker takes LOCAL_RANK modulo the device count): CUDA IPC works between
    processes on one device, and the device-side waits make progress because the two processes' kernels are
    time-sliced; every wait is bounded (SCS_ERR_PEER after the configured timeout), so a stall fails, not hangs."""
    env = dict(os.environ, PYTHONPATH=str(ROOT))
    # --standalone: the rendezvous takes a free local port, so a busy fixed port cannot fail the test
    cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nnodes=1", "--nproc-per-node=2",
           str(ROOT / "tests" / "mp_sharded_worker.py")]  # fmt: skip
    done = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=300, check=False)
    assert done.returncode == 0, done.stdout[-3000:] + done.stderr[-3000:]
    assert "SHARDED-OK" in done.stdout
