"""Time ``scs_supertree_triplets`` (csrc/triplets.cu) on the synthetic workloads of bench.py.

    python tools/triplet_time.py [--workload c4|c5] [--steps 5]

The supertree is built through the product path (``Engine.supertree_build``) from the same seeded forest, then the
triplet pass is timed with CUDA events on the context's stream after one warm-up call (the call includes uploading
the source forest and copying the results back).  Prints one JSON line with the card name and power limit."""

from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))


def gpu_info() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, check=False, timeout=30).stdout.strip().splitlines()  # fmt: skip
        name, power = (x.strip() for x in out[0].split(","))
        return {"gpu": name, "power_limit": power}
    except Exception:  # noqa: BLE001
        return {"gpu": "unknown", "power_limit": "unknown"}


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
    engine.supertree_triplets(forest, parent, taxon)  # warm-up: modules loaded, allocator primed
    ms = []
    for _ in range(args.steps):
        engine.timer_start()
        per_tree = engine.supertree_triplets(forest, parent, taxon)
        ms.append(engine.timer_stop())
    shared = per_tree[:, 0].astype(np.float64)
    depth = np.zeros(len(parent), dtype=np.int64)
    for i in range(1, len(parent)):
        depth[i] = depth[parent[i]] + 1
    print(json.dumps({
        "tool": "triplet_time", "workload": args.workload, "taxa": n, "trees": t, "supertree_nodes": int(len(parent)),
        "supertree_depth": int(depth.max()), "source_leaves": int(forest.num_leaves),
        "pair_work": int((shared * shared).sum()), "max_shared": int(per_tree[:, 0].max()),
        "triplets_ms_median": float(np.median(ms)), "triplets_ms_min": float(min(ms)), "triplets_ms": ms,
        "build_s_first": build_s, "generate_s": gen_s,
        "resolved_source": int(per_tree[:, 1].sum()), "agree": int(per_tree[:, 3].sum()),
        "contradict": int(per_tree[:, 4].sum()), "fit": float(per_tree[:, 3].sum() / max(1, per_tree[:, 1].sum())),
        **gpu_info(),
    }))  # fmt: skip
    engine.close()


if __name__ == "__main__":
    main()
