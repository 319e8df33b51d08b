"""GPU: a batch of small recursion nodes through ``scs_nodes_split_small_host`` (both capacities of the one-CTA
kernel, launched heaviest first) against the same nodes one at a time through ``scs_node_split_host``."""

from __future__ import annotations

import ctypes

import numpy as np
import pytest

from spectralclustersupertree_b200 import _lib
from spectralclustersupertree_b200._lib import NodeStats, ptr
from spectralclustersupertree_b200.flatten import flatten_trees
from spectralclustersupertree_b200.tree import make_tree

pytestmark = pytest.mark.gpu

SMALL_NODE = np.dtype([("n", np.int32), ("num_trees", np.int32), ("leaf_base", np.int64), ("tree_base", np.int64),
                       ("vertex_base", np.int64)])  # fmt: skip


def _random_newick(names, rng) -> str:
    def sub(xs):
        if len(xs) == 1:
            return f"{xs[0]}:{rng.uniform(0.1, 2.0):.3f}"
        cut = int(rng.integers(1, len(xs)))
        return f"({sub(xs[:cut])},{sub(xs[cut:])}):{rng.uniform(0.1, 2.0):.3f}"

    xs = list(rng.permutation(names))
    cut = int(rng.integers(1, len(xs)))
    return f"({sub(xs[:cut])},{sub(xs[cut:])});"


def _caterpillar(names, rng) -> str:
    xs = list(rng.permutation(names))
    s = f"({xs[0]}:1,{xs[1]}:1)"
    for x in xs[2:]:
        s = f"({s}:{rng.uniform(0.1, 2.0):.3f},{x}:1)"
    return s + ";"


def _node(n, num_trees, rng, *, caterpillars=0):
    """Leaf tours of one node: n taxa, trees on random subsets (the first one on all n taxa, so k_t = n occurs)."""
    names = [f"t{i}" for i in range(n)]
    lines = [_random_newick(names, rng)]
    for i in range(num_trees - 1):
        if i < caterpillars:
            lines.append(_caterpillar(names, rng))
            continue
        k = int(rng.integers(2, n + 1))
        lines.append(_random_newick(list(rng.choice(names, size=k, replace=False)), rng))
    weights = rng.uniform(0.5, 2.0, size=len(lines))
    return flatten_trees([make_tree(s) for s in lines], weights, "branch", {x: i for i, x in enumerate(names)})


def _split_one(engine, tours):
    part, stats = engine.node_split(tours, contract_edges=True, seed=0)
    return part, stats


def _same_partition(a, b) -> bool:
    return np.array_equal(a, b) or (a.max() <= 1 and b.max() <= 1 and np.array_equal(a, 1 - b))


def test_small_batch_matches_per_node_path(engine):
    """Node sizes 3..64 in mixed order, a node with more trees than one staging chunk, caterpillars deeper than 32
    levels, k_t = n at every node.  Against the per-node one-CTA path (graph from pcg_rows_kernel, small limit 64):
    every stat bit for bit.  Against the staged path (small limit 0): components, contracted size, Fiedler value to
    1e-9, partition unless tie-flagged."""
    rng = np.random.default_rng(20261022)
    sizes = [17, 3, 64, 9, 40, 32, 5, 33, 24, 48, 12, 31, 57, 4, 20]
    nodes = []
    for b, n in enumerate(sizes):
        trees = 300 if b == 1 else 600 if b == 5 else int(rng.integers(2, 40))
        nodes.append(_node(n, trees, rng, caterpillars=3 if n > 34 else 0))
    desc = np.zeros(len(nodes), dtype=SMALL_NODE)
    offsets, L, T, N = [], 0, 0, 0
    for b, t in enumerate(nodes):
        desc[b] = (t.n, t.num_trees, L, T, N)
        offsets.append(t.leaf_offsets)
        L += t.num_leaves
        T += t.num_trees
        N += t.n
    assert max(t.num_leaves for t in nodes) > 1024  # more than one chunk at either capacity

    def cat(field, dtype):
        return np.ascontiguousarray(np.concatenate([getattr(t, field) for t in nodes]), dtype=dtype)

    leaf_offsets = np.ascontiguousarray(np.concatenate(offsets), dtype=np.int64)
    taxon, depth, val = cat("leaf_taxon", np.int32), cat("adj_depth", np.int32), cat("adj_val", np.float64)
    root, weight = cat("root_depth", np.int32), cat("tree_weight", np.float64)
    part = np.full(N, -7, dtype=np.int32)
    stats = (NodeStats * len(nodes))()
    lib = _lib.load()
    status = lib.scs_nodes_split_small_host(
        engine.handle, len(nodes), ptr(desc), L, T, ptr(leaf_offsets), ptr(taxon), ptr(depth), ptr(val), ptr(root),
        ptr(weight), 1, ptr(part), ctypes.cast(stats, ctypes.c_void_p),
    )  # fmt: skip
    assert status == _lib.SCS_OK

    engine.set_small_node_limit(64)
    try:
        jacobi = [_split_one(engine, t) for t in nodes]
        engine.set_small_node_limit(0)
        staged = [_split_one(engine, t) for t in nodes]
    finally:
        engine.set_small_node_limit(32)
    spectral = 0
    for b, t in enumerate(nodes):
        got_part = part[desc[b]["vertex_base"] : desc[b]["vertex_base"] + t.n]
        got = stats[b]
        jpart, jst = jacobi[b]
        assert np.array_equal(got_part, jpart), b
        assert bytes(got) == bytes(jst), b
        spart, sst = staged[b]
        assert got.n_components == sst.n_components, b
        assert got.contracted_size == sst.contracted_size, b
        if got.n_components == 1 and got.contracted_size > 2:
            spectral += 1
            assert abs(got.eig[1] - sst.eig[1]) <= 1e-9, (b, got.eig[1], sst.eig[1])
        if not got.tie_flag and not sst.tie_flag:
            assert _same_partition(got_part, spart), b
    assert spectral >= 5
