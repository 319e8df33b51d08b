"""Time ``scs_supertree_mrp`` (csrc/triplets.cu) on the synthetic workloads of bench.py.

    python tools/mrp_time.py [--workload c4|c5] [--steps 5]

The supertree is built through the product path (``Engine.supertree_build``) from the same seeded forest, then the
MRP pass is timed with CUDA events on the context's stream after one warm-up call (the call includes uploading the
source forest and copying the results back).  The per-tree triplet pass is timed the same way in the same run, for
comparison.  Prints one JSON line with the card name and power limit."""

from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from triplet_time import gpu_info  # noqa: E402


def main() -> None:
    import numpy as np

    from bench import WORKLOADS, POOLED_WORKLOADS
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
    t0 = time.perf_counter()
    built = engine.supertree_build(forest, weighting)
    build_s = time.perf_counter() - t0
    parent, taxon = built["parent"], built["taxon"]

    def timed(call):
        call(forest, parent, taxon)  # warm-up: modules loaded, allocator primed
        ms = []
        for _ in range(args.steps):
            engine.timer_start()
            out = call(forest, parent, taxon)
            ms.append(engine.timer_stop())
        return out, ms

    per_tree, ms = timed(engine.supertree_mrp)
    _triplets, triplet_ms = timed(engine.supertree_triplets)
    depth = np.zeros(len(parent), dtype=np.int64)
    for i in range(1, len(parent)):
        depth[i] = depth[parent[i]] + 1
    characters, steps = int(per_tree[:, 1].sum()), int(per_tree[:, 2].sum())
    print(json.dumps({
        "tool": "mrp_time", "workload": args.workload, "taxa": n, "trees": t, "supertree_nodes": int(len(parent)),
        "supertree_depth": int(depth.max()), "source_leaves": int(forest.num_leaves),
        "max_shared": int(per_tree[:, 0].max()), "characters": characters, "steps": steps,
        "exact": int(per_tree[:, 3].sum()), "ci": characters / steps if steps else None,
        "mrp_ms_median": float(np.median(ms)), "mrp_ms_min": float(min(ms)), "mrp_ms": ms,
        "triplets_ms_median": float(np.median(triplet_ms)), "triplets_ms": triplet_ms,
        "build_s_first": build_s, "generate_s": gen_s, **gpu_info(),
    }))  # fmt: skip
    engine.close()


if __name__ == "__main__":
    main()
