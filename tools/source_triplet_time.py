"""Time ``scs_forest_pairwise_triplets`` (csrc/pairwise.cu) on the synthetic workloads of bench.py.

    python tools/source_triplet_time.py [--workload c4|c5] [--steps 3]

The seeded source forest of the workload is generated, then the pairwise triplet pass is timed with CUDA events on
the context's stream after one warm-up call (the call includes uploading the forest, the tours and copying the four
T x T matrices back).  No supertree is involved.  Prints one JSON line with the card name and power limit, the pairs,
the pairs sharing at least three taxa (comparable), the sums of their k and k^2 (a pair costs O(k^2 log D)), the
summed counts, whether every timed call returned the warm-up call's bits, and the median and minimum of the timed
calls."""

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
    parser.add_argument("--steps", type=int, default=3)
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
    first = engine.forest_pairwise_triplets(forest)  # warm-up: modules loaded, allocator primed
    ms, same = [], True
    for _ in range(args.steps):
        engine.timer_start()
        again = engine.forest_pairwise_triplets(forest)
        ms.append(engine.timer_stop())
        same = same and all(np.array_equal(a, b) for a, b in zip(first, again, strict=True))
    shared, resolved, agree, contradict = first
    upper = np.triu_indices(len(shared), 1)
    k = shared[upper].astype(np.int64)
    comparable = k >= 3
    kc = k[comparable]
    distance = (resolved + resolved.T - 2 * agree - contradict)[upper][comparable]
    print(json.dumps({
        "tool": "source_triplet_time", "workload": args.workload, "taxa": n, "trees": t,
        "source_leaves": int(forest.num_leaves), "pairs": int(len(k)), "comparable_pairs": int(comparable.sum()),
        "sum_shared_comparable": int(kc.sum()), "sum_shared_sq_comparable": int((kc * kc).sum()),
        "max_shared": int(k.max()) if len(k) else 0,
        "sum_resolved": int(resolved[upper][comparable].sum() + resolved.T[upper][comparable].sum()),
        "sum_agree": int(agree[upper][comparable].sum()), "sum_contradict": int(contradict[upper][comparable].sum()),
        "sum_distance": int(distance.sum()), "repeat_identical": bool(same),
        "pairwise_ms_median": float(np.median(ms)), "pairwise_ms_min": float(min(ms)), "pairwise_ms": ms,
        "generate_s": gen_s, **gpu_info(),
    }))  # fmt: skip
    engine.close()


if __name__ == "__main__":
    main()
