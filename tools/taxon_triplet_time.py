"""Time ``scs_supertree_taxon_triplets`` (csrc/triplets.cu) on the synthetic workloads of bench.py, next to the
per-tree call ``scs_supertree_triplets`` on the same supertree.

    python tools/taxon_triplet_time.py [--workload c4|c5] [--steps 5]

The supertree is built through the product path (``Engine.supertree_build``) from the same seeded forest, then each
call is timed with CUDA events on the context's stream after one warm-up call (a call includes uploading the source
forest and copying the results back).  The two calls alternate step by step.  Prints one JSON line with the card
name and power limit, and checks that every triplet is credited to its three taxa."""

from __future__ import annotations

import argparse
import json
import sys
import time
from math import comb
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from triplet_time import gpu_info  # noqa: E402


def main() -> None:
    import numpy as np

    from bench import POOLED_WORKLOADS, WORKLOADS
    from spectralclustersupertree_b200.engine import Engine, Forest
    from spectralclustersupertree_b200.synthetic import make_forest_arrays, make_problem

    parser = argparse.ArgumentParser()
    parser.add_argument("--workload", default="c4", choices=["c4", "c5"])
    parser.add_argument("--steps", type=int, default=5)
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
    built = engine.supertree_build(forest, weighting)
    parent, taxon = built["parent"], built["taxon"]
    engine.supertree_triplets(forest, parent, taxon)  # warm-up: modules loaded, allocator primed
    engine.supertree_taxon_triplets(forest, parent, taxon)
    tree_ms, taxon_ms = [], []
    for _ in range(args.steps):
        engine.timer_start()
        per_tree = engine.supertree_triplets(forest, parent, taxon)
        tree_ms.append(engine.timer_stop())
        engine.timer_start()
        per_taxon, weighted = engine.supertree_taxon_triplets(forest, parent, taxon)
        taxon_ms.append(engine.timer_stop())
    shared = per_tree[:, 0]
    depth = np.zeros(len(parent), dtype=np.int64)
    for i in range(1, len(parent)):
        depth[i] = depth[parent[i]] + 1
    credited = all(int(per_taxon[:, 2 + f].sum()) == 3 * int(per_tree[:, 1 + f].sum()) for f in range(4))
    credited = credited and int(per_taxon[:, 1].sum()) == 3 * sum(comb(int(k), 3) for k in shared)
    fit = per_taxon[:, 4] / np.maximum(per_taxon[:, 2], 1)
    print(json.dumps({
        "tool": "taxon_triplet_time", "workload": args.workload, "taxa": n, "trees": t,
        "supertree_nodes": int(len(parent)), "supertree_depth": int(depth.max()), "source_leaves": int(forest.num_leaves),
        "pair_work": int((shared.astype(np.float64) ** 2).sum()), "max_shared": int(shared.max()),
        "taxon_triplets_ms_median": float(np.median(taxon_ms)), "taxon_triplets_ms_min": float(min(taxon_ms)),
        "taxon_triplets_ms": taxon_ms, "triplets_ms_median": float(np.median(tree_ms)), "triplets_ms": tree_ms,
        "every_triplet_credited_three_times": bool(credited), "lowest_taxon_fit": float(fit[per_taxon[:, 0] >= 5].min()),
        "weighted_agree_sum": float(weighted[:, 1].sum()), "generate_s": gen_s, **gpu_info(),
    }))  # fmt: skip
    engine.close()


if __name__ == "__main__":
    main()
