"""Time the large recursion nodes of a workload and dump every recursion record (run on the GPU box).

    python tools/large_node_time.py [workload] [--records PATH]

The build runs from the device-resident forest as bench.py's ``value`` does: two warm-up builds, then one build
with recording on.  Reported:
* the whole build, between CUDA events on the context's stream;
* every wave whose largest node takes the per-node path (above the medium limit): the wave's GPU time and its
  largest node's size;
* the per-node path's stage clocks summed over those nodes (host wall clock around work that ends in a stream
  synchronise): tour components, graph build, contraction, Lanczos and the rest of the spectral step.
``--records`` writes every recursion record -- n, components, contracted size m, the eigenvalues as hex floats,
matvecs, residual (hex) and tie flag -- as JSON, so that the records of two builds can be diffed bit for bit."""

from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402
from spectralclustersupertree_b200.engine import Engine, Forest  # noqa: E402

MEDIUM_LIMIT = 4096  # the default medium limit: larger nodes take the per-node path


def record_json(taxa, stats) -> dict:
    return {"n": int(len(taxa)), "first_taxon": int(taxa[0]), "components": int(stats.n_components),
            "m": int(stats.contracted_size), "eig": [float(x).hex() for x in stats.eig], "matvecs": int(stats.matvecs),
            "residual": float(stats.residual).hex(), "tie_flag": int(stats.tie_flag)}  # fmt: skip


def main() -> None:
    parser = argparse.ArgumentParser()
    parser.add_argument("workload", nargs="?", default="c4")
    parser.add_argument("--records", type=Path, default=None)
    args = parser.parse_args()
    a = bench.make_workload(args.workload)
    engine = Engine(0)
    forest = Forest.from_arrays(a["node_offsets"], a["parent"], a["length"], a["support"], a["taxon"], a["weights"],
                                a["names"])  # fmt: skip
    resident = engine.device_forest(forest, a["weighting"])
    for _ in range(2):
        engine.supertree_build_resident(resident)
    engine.stage_seconds(reset=True)
    engine.timer_start()
    built = engine.supertree_build_resident(resident, record=True)
    total_ms = engine.timer_stop()
    stages = engine.stage_seconds(reset=True)
    resident.close()

    print(f"{args.workload}: build {total_ms:.2f} ms (CUDA events), {len(built['records'])} records, "
          f"{built['nodes_large']} nodes on the per-node path")
    print("wave  largest n  wave GPU ms")
    for w, (max_n, sec) in enumerate(zip(built["wave_max_n"], built["wave_seconds"], strict=True)):
        if max_n > MEDIUM_LIMIT:
            print(f"{w:4d}  {max_n:9d}  {1e3 * sec[0]:11.2f}")
    graph = stages["enqueue_graph"] + stages["wait_graph"]
    tours = stages.get("tour_components", 0.0)
    lanczos = stages["lanczos_in_spectral"]
    print(f"per-node path, summed: tour components {1e3 * tours:.2f} ms, graph build and its "
          f"components {1e3 * graph:.2f} ms, contraction {1e3 * stages['enqueue_contract']:.2f} ms, Lanczos "
          f"{1e3 * lanczos:.2f} ms, rest of the spectral step {1e3 * (stages['spectral'] - lanczos):.2f} ms")
    large = [(taxa, stats) for taxa, _, stats in built["records"] if len(taxa) > MEDIUM_LIMIT]
    for taxa, stats in large:
        print(f"  n {len(taxa):6d}  components {stats.n_components:3d}  m {stats.contracted_size:6d}  "
              f"matvecs {stats.matvecs:3d}  eig {stats.eig[1]!r}")
    if args.records:
        args.records.parent.mkdir(parents=True, exist_ok=True)
        args.records.write_text(json.dumps([record_json(taxa, stats) for taxa, _, stats in built["records"]]) + "\n")
        print("records ->", args.records)
    engine.close()


if __name__ == "__main__":
    main()
