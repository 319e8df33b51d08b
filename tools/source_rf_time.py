"""Time ``scs_forest_pairwise_rf`` (csrc/pairwise.cu) on the synthetic workloads of bench.py.

    python tools/source_rf_time.py [--workload c4|c5] [--steps 5]

The seeded source forest of the workload is generated, then the pairwise pass is timed with CUDA events on the
context's stream after one warm-up call (the call includes uploading the forest, the tours and copying the three
T x T matrices back).  No supertree is involved.  Prints one JSON line with the card name and power limit, the pairs,
the pairs sharing at least three taxa (comparable), the sum of their shared taxa, and the median and minimum of the
timed calls."""

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
    shared, clusters, common = engine.forest_pairwise_rf(forest)  # warm-up: modules loaded, allocator primed
    ms = []
    for _ in range(args.steps):
        engine.timer_start()
        again = engine.forest_pairwise_rf(forest)
        ms.append(engine.timer_stop())
    same = all(np.array_equal(a, b) for a, b in zip((shared, clusters, common), again, strict=True))
    upper = np.triu_indices(len(shared), 1)
    k = shared[upper]
    comparable = k >= 3
    rf = (clusters + clusters.T - 2 * common)[upper][comparable]
    print(json.dumps({
        "tool": "source_rf_time", "workload": args.workload, "taxa": n, "trees": t,
        "source_leaves": int(forest.num_leaves), "pairs": int(len(k)), "comparable_pairs": int(comparable.sum()),
        "sum_shared_comparable": int(k[comparable].sum(dtype=np.int64)), "max_shared": int(k.max()) if len(k) else 0,
        "sum_rf": int(rf.sum(dtype=np.int64)), "repeat_identical": bool(same),
        "pairwise_ms_median": float(np.median(ms)), "pairwise_ms_min": float(min(ms)), "pairwise_ms": ms,
        "generate_s": gen_s, **gpu_info(),
    }))  # fmt: skip
    engine.close()


if __name__ == "__main__":
    main()
