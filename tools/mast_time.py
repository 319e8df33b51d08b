"""Time ``scs_supertree_mast`` (csrc/triplets.cu) on the synthetic workloads of bench.py.

    python tools/mast_time.py [--workload c4|c5] [--steps 5] [--warmup 1] [--taxa]

The supertree is built through the product path (``Engine.supertree_build``) from the same seeded forest, then the
MAST pass is timed with CUDA events on the context's stream after one warm-up call (the call includes uploading the
source forest and copying the results back).  The per-tree triplet pass is timed the same way in the same run, for
scale.  ``cells`` is the number of table cells the pass fills, sum_t I_t * I_s over the trees with k >= 3 (internal
nodes of the two restrictions), next to its bound sum_t (k_t - 1)^2.  With ``--taxa`` ``scs_supertree_mast_taxa``
(the same pass plus the traceback of one agreement set per tree) is timed the same way in the same run, and its
per-tree counts are checked against ``scs_supertree_mast``'s.  ``--warmup 0`` skips the warm-up calls (C5's MAST call
takes minutes).  Prints one JSON line with the card name and power limit."""

from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from triplet_time import gpu_info  # noqa: E402


def internal_counts(arrays: dict, parent, taxon):
    """Per source tree: k, the internal nodes of t' and of s'.  Every taxon of these forests is a tip of the supertree,
    so t' is t with its unary nodes collapsed; s' has one internal node per distinct LCA in S of S-consecutive taxa."""
    import numpy as np

    offsets = np.asarray(arrays["node_offsets"], dtype=np.int64)
    local = np.asarray(arrays["parent"], dtype=np.int64)
    ftaxon = np.asarray(arrays["taxon"], dtype=np.int64)
    T = len(offsets) - 1
    tree_of = np.repeat(np.arange(T), np.diff(offsets))
    has_parent = local >= 0
    kids = np.bincount((local + offsets[tree_of])[has_parent], minlength=len(local))
    i_t = np.bincount(tree_of, weights=kids >= 2, minlength=T).astype(np.int64)
    # S in depth-first pre-order: the LCA of pre-order nodes a < b is the parent of the shallowest node in (a, b]
    n = len(parent)
    children = [[] for _ in range(n)]
    for v in range(1, n):
        children[parent[v]].append(v)
    order, stack = [], [0]
    while stack:
        v = stack.pop()
        order.append(v)
        stack.extend(reversed(children[v]))
    order = np.asarray(order)
    rank = np.empty(n, dtype=np.int64)
    rank[order] = np.arange(n)
    depth = np.zeros(n, dtype=np.int64)
    for v in order[1:]:
        depth[v] = depth[parent[v]] + 1
    pre_depth, pre_parent = depth[order], rank[np.asarray(parent)[order].clip(0)]
    table = [np.arange(n)]
    while (1 << len(table)) <= n:
        prev, half = table[-1], 1 << (len(table) - 1)
        a, b = prev[:-half], prev[half:]
        table.append(np.where(pre_depth[b] < pre_depth[a], b, a))
    taxon_rank = np.full(int(ftaxon.max()) + 1, -1, dtype=np.int64)
    tips = np.flatnonzero(np.asarray(taxon) >= 0)
    taxon_rank[np.asarray(taxon)[tips]] = rank[tips]
    leaf = ftaxon >= 0
    t_of, r = tree_of[leaf], taxon_rank[ftaxon[leaf]]
    k = np.bincount(t_of, minlength=T)
    sort = np.lexsort((r, t_of))
    t_of, r = t_of[sort], r[sort]
    same = t_of[1:] == t_of[:-1]
    lo, hi = r[:-1][same] + 1, r[1:][same]
    level = np.floor(np.log2(hi - lo + 1)).astype(np.int64)
    best = np.empty(len(lo), dtype=np.int64)
    for l in np.unique(level):
        sel = level == l
        x, y = table[l][lo[sel]], table[l][hi[sel] - (1 << l) + 1]
        best[sel] = np.where(pre_depth[y] < pre_depth[x], y, x)
    lca = pre_parent[best]
    pairs = np.unique(t_of[1:][same] * n + lca)
    i_s = np.bincount(pairs // n, minlength=T)
    return k, i_t, i_s


def main() -> None:
    import numpy as np

    from bench import WORKLOADS, POOLED_WORKLOADS
    from spectralclustersupertree_b200.engine import Engine, Forest
    from spectralclustersupertree_b200.synthetic import make_forest_arrays, make_problem

    parser = argparse.ArgumentParser()
    parser.add_argument("--workload", default="c4", choices=["c4", "c5"])
    parser.add_argument("--steps", type=int, default=5)
    parser.add_argument("--warmup", type=int, default=1)
    parser.add_argument("--taxa", action="store_true", help="also time scs_supertree_mast_taxa")
    args = parser.parse_args()
    n, t, weighting, seed, tw = WORKLOADS[args.workload]
    t0 = time.perf_counter()
    if args.workload in POOLED_WORKLOADS:
        arrays = make_forest_arrays(n, t, weighting, seed, tree_weights=tw, workers=32)
    else:
        arrays = make_problem(n, t, weighting, seed, tree_weights=tw).forest_arrays()
    forest = Forest.from_arrays(arrays["node_offsets"], arrays["parent"], arrays["length"], arrays["support"],
                                arrays["taxon"], arrays["weights"], arrays["names"])  # fmt: skip
    gen_s = time.perf_counter() - t0
    engine = Engine(0)
    t0 = time.perf_counter()
    built = engine.supertree_build(forest, weighting)
    build_s = time.perf_counter() - t0
    parent, taxon = built["parent"], built["taxon"]

    def timed(call):
        for _ in range(args.warmup):  # modules loaded, allocator primed
            call(forest, parent, taxon)
            print(f"{call.__name__}: warmed up", file=sys.stderr, flush=True)
        ms = []
        for _ in range(args.steps):
            engine.timer_start()
            out = call(forest, parent, taxon)
            ms.append(engine.timer_stop())
            print(f"{call.__name__}: {ms[-1]:.1f} ms", file=sys.stderr, flush=True)
        return out, ms

    per_tree, ms = timed(engine.supertree_mast)
    extra = {}
    if args.taxa:
        (taxa_per_tree, tip_state, per_taxon, _weighted), taxa_ms = timed(engine.supertree_mast_taxa)
        assert taxa_per_tree.tobytes() == per_tree.tobytes()
        assert per_taxon[:, 0].sum() == per_tree[:, 0].sum()
        assert per_taxon[:, 1].sum() == (per_tree[:, 0] - per_tree[:, 1]).sum()
        extra = {"mast_taxa_ms_median": float(np.median(taxa_ms)), "mast_taxa_ms": taxa_ms,
                 "kept_tips": int((tip_state == 1).sum()), "pruned_tips": int((tip_state == 0).sum()),
                 "taxa_most_pruned": int(per_taxon[:, 1].max())}  # fmt: skip
    _triplets, triplet_ms = timed(engine.supertree_triplets)
    k, i_t, i_s = internal_counts(arrays, np.asarray(parent), np.asarray(taxon))
    assert np.array_equal(k, per_tree[:, 0])
    big = k >= 3
    depth = np.zeros(len(parent), dtype=np.int64)
    for i in range(1, len(parent)):
        depth[i] = depth[parent[i]] + 1
    shared, agreement = int(per_tree[:, 0].sum()), int(per_tree[:, 1].sum())
    print(json.dumps({
        "tool": "mast_time", "workload": args.workload, "taxa": n, "trees": t, "supertree_nodes": int(len(parent)),
        "supertree_depth": int(depth.max()), "source_leaves": int(forest.num_leaves),
        "max_shared": int(per_tree[:, 0].max()), "shared": shared, "agreement": agreement,
        "pruned": shared - agreement, "trees_agreeing": int((per_tree[:, 0] == per_tree[:, 1]).sum()),
        "cells": int((i_t[big] * i_s[big]).sum()), "cells_bound": int(((k[big] - 1) ** 2).sum()),
        "mast_ms_median": float(np.median(ms)), "mast_ms_min": float(min(ms)), "mast_ms": ms,
        **extra, "triplets_ms_median": float(np.median(triplet_ms)), "triplets_ms": triplet_ms,
        "build_s_first": build_s, "generate_s": gen_s, **gpu_info(),
    }))  # fmt: skip
    engine.close()


if __name__ == "__main__":
    main()
