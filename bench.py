"""Benchmark of the supertree hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4] [--impl reference] [--dump-outputs DIR]

One *step* is one complete ``construct_supertree`` job on the named synthetic workload (default
``c4``: 10 000 taxa x 1 000 source trees, depth weighting -- the configuration BASELINE.json's metric
is quoted on).  Three clocks are reported in one JSON line:

* ``value``  -- the hot path alone with inputs resident in HBM: the whole recursion of the job
  (``scs_supertree_build_resident``) from source trees that were uploaded before the timed region -- tours, graph
  build, components, contraction, spectral split and the restriction of the trees to the children, all on the
  device, wave by wave; CUDA events around the build.
* ``e2e``    -- the same job through the public host-buffer path over the C ABI
  (``scs_forest_create_view`` + ``scs_supertree_build``): flat source trees in host memory in, flat
  supertree out; validation of the trees, H2D of the forest, the recursion, D2H of partitions inside the timed
  region.  With N > 1 the large recursion nodes are row-sharded over the GPUs, smaller sub-problems are dealt out
  over the ranks (no data-path collective) and the outputs are all-gathered.
* ``roofline`` -- the Laplacian matvec (the kernel BASELINE.json's metric names), timed per launch
  with CUDA events inside the timed steps, against the measured HBM peak.

``--impl reference`` times the CPU oracle port of the reference (oracle/: the reference is pure Python
and needs cogent3, which is not installable here -- DESIGN.md) on the WHOLE job: every step is one full
``construct_supertree`` recursion of the same workload on the host cores (C graph build, numpy components
and contraction, sklearn ``SpectralClustering`` called as the reference calls it, Python tree restriction;
independent sub-problems spread over a pool of worker processes).  Nothing is extrapolated: the value is a
measured wall time.  Because one such run takes minutes at c4, the number of timed runs is capped by
``--reference-budget-s`` (at least one is always timed; ``steps_timed`` says how many).
``cpu_baseline`` in the GPU arm's line is the same measurement when the whole job fits the bounded-sample
budget (c1-c3), else the job's top-level recursion node alone, reported as what it is: a lower bound.
"""

from __future__ import annotations

import os

# idle OpenMP threads of the library's host-side helpers must sleep, not spin: with one process per GPU they would
# take the cores the other ranks' driver threads need (read by the OpenMP runtime when it is first loaded)
os.environ.setdefault("OMP_WAIT_POLICY", "passive")

import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

METRIC = "construct_supertree wall-time at 10k taxa/1k trees"
PROFILE_MIN_N = 4096  # csrc/common.cuh kProfileMinSize: launches timed one by one (matrices larger than L2)
# dram__bytes_read.sum + dram__bytes_write.sum of one matvec launch, read from the summary tools/ncu_summary.py
# writes from this round's `ncu --set full` capture (null when no capture has been summarised)
NCU_TRAFFIC_FILE = ROOT / "profiles" / "r02_ncu_matvec_traffic.json"

# name -> (taxa, trees, weighting, seed, tree weights)   (BASELINE.json configs; seed = 1000 * index)
WORKLOADS = {
    "c1": (100, 30, "depth", 1000, False),
    "c2": (500, 50, "branch", 2000, False),
    "c3": (1000, 100, "branch", 3000, True),
    "c4": (10000, 1000, "depth", 4000, False),
    # not a bench line: tools/run_workload.py runs it at 1/2/4/8 GPUs
    "c5": (50000, 5000, "branch", 5000, False),
}
# generated with one random stream per source tree by a pool of processes (synthetic.make_forest_arrays)
POOLED_WORKLOADS = {"c5"}


def describe(workload: str) -> str:
    n, t, weighting, seed, tw = WORKLOADS[workload]
    extra = ", tree weights U[0.5,2]" if tw else ""
    streams = ", one random stream per source tree" if workload in POOLED_WORKLOADS else ""
    return (
        f"{workload}: {n} taxa x {t} source trees (birth-death model tree, SMIDGen-style subsets, 5% NNI noise), "
        f"pcg_weighting={weighting}{extra}, seed {seed}{streams}"
    )


def make_workload(workload: str) -> dict:
    from spectralclustersupertree_b200.synthetic import make_forest_arrays, make_problem

    n, t, weighting, seed, tw = WORKLOADS[workload]
    if workload in POOLED_WORKLOADS:
        world = max(1, int(os.environ.get("WORLD_SIZE", "1")))  # every rank generates the same trees
        arrays = make_forest_arrays(n, t, weighting, seed, tree_weights=tw,
                                    workers=max(1, min(32, (os.cpu_count() or 1) // world)))
    else:
        arrays = make_problem(n, t, weighting, seed, tree_weights=tw).forest_arrays()
    arrays["weighting"] = weighting
    return arrays


def measured_peak_gbs() -> tuple[float, str]:
    path = ROOT / "MEASURED_PEAKS.json"
    if path.is_file():
        try:
            return float(json.loads(path.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except (KeyError, ValueError):
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    FIELDS = (
        "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
        "clocks_event_reasons.sw_power_cap"
    )

    def __init__(self, device: int) -> None:
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(device)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )  # fmt: skip
        except OSError:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, sm_max, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.splitlines():
            cells = [c.strip() for c in line.split(",")]
            if len(cells) < 7:
                continue
            try:
                sm.append(float(cells[0]))
                sm_max.append(float(cells[1]))
            except ValueError:
                continue
            for name, cell in zip(names, cells[3:7], strict=True):
                if cell.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {
            "sm_mhz": statistics.median(sm),
            "sm_max_mhz": max(sm_max),
            "reasons": sorted(reasons),
            "samples": len(sm),
        }


# ---------------------------------------------------------------------------------------------
# the CPU oracle on a bounded sample (cpu_baseline and --impl reference)
# ---------------------------------------------------------------------------------------------
def oracle_children_csr(arrays: dict):
    """The flat pre-order forest as the child lists oracle/pcg_oracle.c reads (vectorised)."""
    offsets = arrays["node_offsets"]
    parent = arrays["parent"].astype(np.int64)
    tree_of = np.repeat(np.arange(len(offsets) - 1), np.diff(offsets))
    base = offsets[:-1][tree_of]
    is_root = parent < 0
    gparent = np.where(is_root, -1, parent + base)
    order = np.argsort(gparent, kind="stable")  # children of a node, in pre-order = child order
    order = order[gparent[order] >= 0]
    counts = np.bincount(gparent[order], minlength=len(parent))
    child_ptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    child_idx = order.astype(np.int64)
    weighting = arrays["weighting"]
    if weighting == "branch":
        own = np.where(np.isnan(arrays["length"]), 1.0, arrays["length"])
    elif weighting == "bootstrap":
        own = arrays["support"].copy()
    else:
        own = np.zeros(len(parent))
    return offsets[:-1].astype(np.int64), child_ptr, child_idx, arrays["taxon"].astype(np.int32), own.astype(np.float64)


def oracle_top_node(arrays: dict) -> dict:
    """Time the CPU oracle on the job's top-level recursion node (ref: scs.py:110-134)."""
    from oracle import scs_oracle

    n = len(arrays["names"])
    roots, child_ptr, child_idx, tip_taxon, own = oracle_children_csr(arrays)
    scs_oracle._c_lib()  # build / load outside the timed region
    t0 = time.perf_counter()
    W, C, occ = scs_oracle.pcg_dense_c_arrays(
        n, roots, child_ptr, child_idx, tip_taxon, own, arrays["weights"], arrays["weighting"]
    )
    t1 = time.perf_counter()
    label = scs_oracle.graph_components(C > 0)
    n_comp = len(np.unique(label))
    t2 = time.perf_counter()
    spectral_n = 0
    if n_comp == 1:
        _, Wc, _ = scs_oracle.contract_dense(W, C, occ)
        spectral_n = Wc.shape[0]
        scs_oracle.spectral_bipartition(Wc, np.random.RandomState(0))
    t3 = time.perf_counter()
    return {
        "seconds": t3 - t0,
        "pcg_s": t1 - t0,
        "components_s": t2 - t1,
        "spectral_s": t3 - t2,
        "n": n,
        "n_components": n_comp,
        "spectral_n": int(spectral_n),
    }


def cpu_threads() -> int:
    return os.cpu_count() or 1


def oracle_whole_job(workload: str) -> dict:
    """One full ``construct_supertree`` recursion of the workload on the CPU oracle port, measured.

    The trees are handed over as ``PhyloNode`` objects (built outside the timed region, as the reference
    receives them); the top of the recursion runs in this process (its BLAS calls use every core), components of
    at most 1 500 taxa are solved by a pool of forked worker processes, one per host core."""
    from oracle import scs_oracle
    from spectralclustersupertree_b200.synthetic import make_problem

    n, t, weighting, seed, tw = WORKLOADS[workload]
    prob = make_problem(n, t, weighting, seed, tree_weights=tw)
    trees = prob.phylonodes()
    weights = [1.0] * len(trees) if prob.weights is None else list(prob.weights)
    scs_oracle._c_lib()
    timers: dict = {}
    info: dict = {}
    t0 = time.perf_counter()
    tree = scs_oracle.construct_supertree_parallel(trees, weights, weighting, workers=cpu_threads(),
                                                   defer_max_taxa=1500, timers=timers, info=info)  # fmt: skip
    seconds = time.perf_counter() - t0
    return {"seconds": seconds, "top_stage_seconds": timers, "tips": len(tree.get_tip_names()), **info}


def whole_job_sample(workload: str, detail: dict) -> str:
    top = ", ".join(f"{k} {v:.1f}" for k, v in detail["top_stage_seconds"].items())
    return (
        f"the whole {workload} job, measured: every one of its {detail['recursion_nodes']} recursion nodes "
        f"({detail['spectral_nodes']} through sklearn SpectralClustering) on the CPU oracle port -- C graph build, "
        f"numpy components/contraction, Python tree restriction; serial part (nodes > 1500 taxa) [{top}] s, "
        f"{detail['deferred_subproblems']} sub-problems over {detail['workers']} worker processes"
    )


def reference_line(args) -> dict:
    """``--impl reference``: the CPU oracle port on the whole job; every step is a full measured run."""
    times = []
    detail = {}
    budget = args.reference_budget_s
    started = time.perf_counter()
    first = oracle_whole_job(args.workload)  # doubles as the warm-up when there is time for more
    runs_fit = int(budget // max(first["seconds"], 1e-9))
    if args.warmup == 0 or runs_fit < 2:
        times.append(first["seconds"])
        detail = first
    for _ in range(args.steps - len(times)):
        if time.perf_counter() - started + first["seconds"] > budget:
            break
        detail = oracle_whole_job(args.workload)
        times.append(detail["seconds"])
    value = statistics.mean(times)
    sample = whole_job_sample(args.workload, detail) + f"; {len(times)} full run(s) timed within the {budget:.0f} s budget"
    cores = cpu_threads()
    return {
        "metric": METRIC, "value": value, "unit": "s", "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
        "steps_timed": len(times), "warmup": args.warmup, "ms_per_step": value * 1e3, "higher_is_better": False,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": describe(args.workload)},
        "cpu_baseline": {"value": value, "unit": "s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }  # fmt: skip


# ---------------------------------------------------------------------------------------------
# the GPU arm
# ---------------------------------------------------------------------------------------------
def dump_outputs(out_dir: Path, arrays: dict) -> None:
    """``--dump-outputs``: each array as ``out_dir/<name>.npy`` in float64 (the int32 node arrays convert exactly), so
    that two builds of the project can be compared output for output on the same seeded workload.  A supertree has
    fewer than 2 nodes per taxon: the largest workload (c5, 50 000 taxa) writes under 4 MB in all."""
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", np.asarray(a, dtype=np.float64))


def gather_supertree(dist, built: dict, local_rank: int):
    """All ranks' flat outputs joined on every rank (tiny: 2 int32 per output node)."""
    import torch

    from spectralclustersupertree_b200.engine import merge_sharded

    device = torch.device("cuda", local_rank)
    world = dist.get_world_size()
    size = torch.tensor([len(built["parent"]), built["shared_prefix"]], device=device, dtype=torch.int64)
    sizes = [torch.zeros_like(size) for _ in range(world)]
    dist.all_gather(sizes, size)
    longest = int(max(int(s[0]) for s in sizes))
    mine = torch.full((2, longest), -2, device=device, dtype=torch.int32)
    mine[0, : len(built["parent"])] = torch.from_numpy(built["parent"]).to(device)
    mine[1, : len(built["taxon"])] = torch.from_numpy(built["taxon"]).to(device)
    everyone = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(everyone, mine)
    parts = []
    for r in range(world):
        count, prefix = int(sizes[r][0]), int(sizes[r][1])
        host = everyone[r].cpu().numpy()
        parts.append((host[0, :count], host[1, :count], prefix))
    return merge_sharded(parts)


def profile_step(args, arrays: dict) -> dict:
    """One product-path job inside a cudaProfilerStart/Stop bracket (the step ncu captures)."""
    from spectralclustersupertree_b200 import _lib
    from spectralclustersupertree_b200.engine import Engine, Forest, set_host_threads

    engine = Engine(0)
    if args.small_limit >= 0:
        engine.set_small_node_limit(args.small_limit)
    set_host_threads(max(1, min(16, os.cpu_count() or 1)))
    lib = _lib.load()

    def forest():
        return Forest.from_arrays(arrays["node_offsets"], arrays["parent"], arrays["length"], arrays["support"],
                                  arrays["taxon"], arrays["weights"], arrays["names"])  # fmt: skip

    engine.supertree_build(forest(), arrays["weighting"])  # warm-up: workspaces sized, modules loaded
    engine.synchronize()
    before = engine.launch_count
    lib.scs_profiler_range(1)
    t0 = time.perf_counter()
    built = engine.supertree_build(forest(), arrays["weighting"])
    engine.synchronize()
    seconds = time.perf_counter() - t0
    lib.scs_profiler_range(0)
    cycles = np.zeros(2, dtype=np.uint64)
    lib.scs_debug_small_cycles(engine.handle, cycles.ctypes.data, 0)
    out = {"workload": describe(args.workload), "step_seconds_under_profiler": seconds,
           "small_kernel_cycles_since_start": {"graph_build": int(cycles[0]), "after_build": int(cycles[1])},
           "gpu_launches_in_step": int(engine.launch_count - before), "waves": built["waves"],
           "nodes_small": built["nodes_small"], "nodes_large": built["nodes_large"]}  # fmt: skip
    engine.close()
    return out


def gpu_line(args, arrays: dict) -> dict:
    from spectralclustersupertree_b200.engine import Engine, Forest
    from spectralclustersupertree_b200.scs import supertree_of_forest

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod

        torch.cuda.set_device(local_rank)
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist = dist_mod
    engine = Engine(local_rank)
    if args.small_limit >= 0:
        engine.set_small_node_limit(args.small_limit)
    weighting = arrays["weighting"]
    # torchrun exports OMP_NUM_THREADS=1; give every rank its share of the host cores instead
    from spectralclustersupertree_b200.engine import set_host_threads

    host_threads = max(1, min(16, (os.cpu_count() or 1) // world))
    set_host_threads(host_threads)
    if dist is not None and args.shard_min_n > 0:
        # exchange windows for the nodes that are row-sharded over the GPUs (csrc/shard.cu): every rank
        # exports its window as a CUDA IPC handle, all-gathered here, mapped by every peer
        handles = [None] * world
        dist.all_gather_object(handles, engine.shard_create(rank, world, len(arrays["names"])))
        engine.shard_connect(handles)
        engine.shard_configure(min_n=args.shard_min_n, timeout_seconds=30.0)
        dist.barrier()

    def new_forest():
        return Forest.from_arrays(arrays["node_offsets"], arrays["parent"], arrays["length"], arrays["support"],
                                  arrays["taxon"], arrays["weights"], arrays["names"])  # fmt: skip

    def e2e_step():
        """The product path: flat host arrays in, flat supertree out (joined over the ranks)."""
        built = engine.supertree_build(new_forest(), weighting, rank=rank, world=world)
        if dist is None:
            return built, (built["parent"], built["taxon"])
        return built, gather_supertree(dist, built, local_rank)

    # one untimed build with records: what the job consists of
    traced = engine.supertree_build(new_forest(), weighting, record=True, rank=rank, world=world)
    sharing = dist is not None and args.shard_min_n > 0
    spectral = [st for _, _, st in traced["records"] if st.n_components == 1]
    sizes = [len(taxa) for taxa, _, _ in traced["records"]]
    job = {
        "recursion_nodes_this_rank": len(traced["records"]),
        "spectral_nodes_this_rank": len(spectral),
        "largest_spectral_m": max((st.contracted_size for st in spectral), default=0),
        "lanczos_matvecs_this_rank": sum(st.matvecs for st in spectral if st.solver == 3),
        "tie_nodes_this_rank": sum(1 for st in spectral if st.tie_flag & 3),
        "pair_visits_this_rank": int(traced["pair_visits"]),
        "waves": traced["waves"],
        "wave_tasks": traced["wave_tasks"],
        "wave_max_n": traced["wave_max_n"],
        "nodes_small_one_launch_per_wave": traced["nodes_small"],
        "nodes_medium_batched_per_wave": traced["nodes_medium"],
        "nodes_medium_rerun_per_node": traced["nodes_rerun"],
        "nodes_large_per_node": traced["nodes_large"],
        "nodes_row_sharded_over_gpus": int(sum(1 for n in sizes[: traced["shared_records"]] if sharing and n >= args.shard_min_n)),
    }
    if world == 1:
        job["recursion_nodes"] = len(traced["records"])
    resident = engine.device_forest(new_forest(), weighting)
    job["resident_forest_bytes"] = resident.nbytes

    def barrier():
        engine.synchronize()
        if dist is not None:
            dist.barrier()

    def device_step():
        """The hot path with its inputs resident in HBM: the whole recursion from the device forest."""
        return engine.supertree_build_resident(resident, rank=rank, world=world)

    for _ in range(args.warmup):
        e2e_step()
        device_step()
    engine.synchronize()

    sampler = ClockSampler(local_rank)
    # ---- timed: the recursion from the device-resident forest (value), per-launch matvec / row-kernel timing --------
    engine.profile(True)
    launches_before = engine.launch_count
    dev_ms = []
    for _ in range(args.steps):
        engine.flush_l2()
        barrier()
        engine.timer_start()
        dev_built = device_step()
        dev_ms.append(engine.timer_stop())
        barrier()
    gpu_launches = engine.launch_count - launches_before
    engine.profile(False)
    matvec = engine.profile_read(0)
    rows = engine.profile_read(1)
    # ---- timed: end to end from host buffers (e2e) -----------------------------------------------
    h2d0, d2h0 = engine.io_bytes()
    e2e_s = []
    host_split = dict.fromkeys(("large_nodes", "small_batches", "restrict", "tours"), 0.0)
    for _ in range(args.steps):
        engine.flush_l2()
        barrier()
        t0 = time.perf_counter()
        built, merged = e2e_step()
        engine.synchronize()
        e2e_s.append(time.perf_counter() - t0)
        for k in built["seconds"]:
            host_split[k] += built["seconds"][k] / args.steps
        host_split["medium_batches"] = host_split.get("medium_batches", 0.0) + built["medium_seconds"] / args.steps
        barrier()
    h2d1, d2h1 = engine.io_bytes()
    clocks = sampler.stop()
    resident.close()
    tips = int((merged[1] >= 0).sum())
    if args.dump_outputs and rank == 0:
        dump_outputs(Path(args.dump_outputs), {
            "resident_parent": dev_built["parent"], "resident_taxon": dev_built["taxon"],
            "e2e_parent": merged[0], "e2e_taxon": merged[1],
        })  # fmt: skip

    value_s = statistics.mean(dev_ms) / 1e3
    e2e_value = statistics.mean(e2e_s)
    if dist is not None:
        import torch

        both = torch.tensor([value_s, e2e_value], device=f"cuda:{local_rank}", dtype=torch.float64)
        dist.all_reduce(both, op=dist.ReduceOp.MAX)
        value_s, e2e_value = both.tolist()

    peak, peak_src = measured_peak_gbs()
    roofline = {"bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": None,
                "kernel": "matvec_rows<256> (y = D^-1/2 W D^-1/2 x, fp64; the launches with m >= 4096: W exceeds the 126 MB L2)", "peak_source": peak_src}  # fmt: skip
    if sharing:
        # every launch of that size is then the row-sharded kernel: its time includes the all-gather of the
        # result over NVLink and the wait for the slowest rank
        roofline["kernel"] = ("matvec_rows_allgather<256> (this rank's row block of y = D^-1/2 W D^-1/2 x fused with the "
                              "all-gather of y into every peer's window and the barrier; m >= 4096)")
    if matvec["launches"] and matvec["ms"] > 0:
        achieved = matvec["bytes"] / (matvec["ms"] * 1e-3) / 1e9
        roofline.update({
            "achieved": achieved, "frac": achieved / peak, "launches": matvec["launches"],
            "avg_launch_us": 1e3 * matvec["ms"] / matvec["launches"],
            "bytes_per_launch": matvec["bytes"] / matvec["launches"],
            "share_of_step": matvec["ms"] / sum(dev_ms),
        })  # fmt: skip
        # DRAM bytes of one launch as ncu measured them (dram__bytes_read.sum + dram__bytes_write.sum of this
        # round's `ncu --set full` capture of the largest matvec launch of this workload); null without a capture
        if NCU_TRAFFIC_FILE.is_file():
            captured = json.loads(NCU_TRAFFIC_FILE.read_text())
            # the capture is of the job's largest launch (grid = m rows); `achieved` averages launches of several
            # sizes, so the measured bytes are scaled by the ratio measured / algorithmic of the captured launch
            m_cap = int(str(captured.get("grid", "(0")).strip("()").split(",")[0] or 0)
            algorithmic = 8.0 * m_cap * m_cap + 24.0 * m_cap
            ratio = captured["dram_bytes_per_launch"] / algorithmic if algorithmic else None
            captured["algorithmic_bytes_of_captured_launch"] = algorithmic
            captured["measured_over_algorithmic"] = ratio
            roofline["traffic"] = roofline["bytes_per_launch"] * ratio if ratio else captured["dram_bytes_per_launch"]
            roofline["traffic_detail"] = captured
    roofline_rows = None
    if rows["launches"] and rows["ms"] > 0:
        visits = rows["units"]
        roofline_rows = {
            "kernel": "pcg_rows_kernel (leaf-pair LCA weighting -> W rows, adjacency bits, degree), n >= 4096",
            "bound": "shared-memory / issue (not HBM): ordered leaf-pair visits per second",
            "pair_visits_per_s": visits / (rows["ms"] * 1e-3),
            "write_GBps": rows["bytes"] / (rows["ms"] * 1e-3) / 1e9,
            "launches": rows["launches"],
            "share_of_step": rows["ms"] / sum(dev_ms),
        }
    line = {
        "metric": METRIC, "value": value_s, "unit": "s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": value_s * 1e3, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {
            "workload": describe(args.workload),
            "l2": "flushed between timed steps (256 MB write); the top-level W (0.8 GB) exceeds L2 by itself",
            "value_is": "the whole recursion from source trees already resident in HBM (scs_supertree_build_resident: tours, "
                        "node splits and tree restriction on the device, wave by wave; per wave the nodes > 4096 taxa one "
                        "by one, the nodes of 33..4096 taxa as one batch, the nodes <= 32 taxa in one launch); CUDA "
                        "events around the build; max over ranks",
            "e2e_is": "scs_forest_create_view (the caller's flat arrays validated in place, not copied) + "
                      "scs_supertree_build over the C ABI from flat host arrays to the flat "
                      "supertree (wall clock: validation of the trees, H2D of the forest, the recursion as in value, D2H "
                      "of partitions and bookkeeping; for N > 1 recursion nodes with >= --shard-min-n taxa are "
                      "row-sharded over the GPUs (every leaf pair once over all ranks, the halves exchanged over NVLink; "
                      "fused matvec + all-gather over peer windows), smaller "
                      "sub-problems are dealt out over the ranks and the outputs are all-gathered)",
            "e2e_host_seconds": host_split,
            "e2e_step_seconds": [round(x, 4) for x in e2e_s],
            "host_threads_per_rank": host_threads,
            "supertree_tips": tips,
            "job": job,
        },
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "s", "h2d_bytes_per_step": (h2d1 - h2d0) // args.steps,
                "d2h_bytes_per_step": (d2h1 - d2h0) // args.steps},
        "gpu_launches": int(gpu_launches),
        "roofline": roofline,
        "roofline_pcg_rows": roofline_rows,
    }  # fmt: skip
    if rank == 0 and world == 1 and args.workload != "c5":
        # the drop-in itself: construct_supertree(list of tree objects) -- C-level flattening of the node objects,
        # native build, node objects of the result (the objects themselves are built outside the timed call)
        from spectralclustersupertree_b200 import construct_supertree
        from spectralclustersupertree_b200.synthetic import make_problem

        n_, t_, w_, seed_, tw_ = WORKLOADS[args.workload]
        problem = make_problem(n_, t_, w_, seed_, tree_weights=tw_)
        objects = problem.phylonodes()
        construct_supertree(objects, problem.weights, w_, engine=engine)  # warm
        t0 = time.perf_counter()
        result = construct_supertree(objects, problem.weights, w_, engine=engine)
        line["e2e_python_api"] = {"value": time.perf_counter() - t0, "unit": "s",
                                  "call": "construct_supertree(list[PhyloNode], weights, pcg_weighting) -> PhyloNode",
                                  "tips": len(result.get_tip_names())}  # fmt: skip
        del objects, problem
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        if args.workload in ("c1", "c2", "c3"):
            # the whole job fits the bounded-sample budget: measured end to end
            detail = oracle_whole_job(args.workload)
            line["cpu_baseline"] = {"value": detail["seconds"], "unit": "s", "cores": cpu_threads(), "kind": "port",
                                    "sample": whole_job_sample(args.workload, detail)}  # fmt: skip
        else:
            detail = oracle_top_node(arrays)
            line["cpu_baseline"] = {
                "value": detail["seconds"], "unit": "s", "cores": cpu_threads(), "kind": "port",
                "sample": (
                    f"LOWER BOUND -- one of the job's {job.get('recursion_nodes', '?')} recursion nodes only: the top-level node of "
                    f"{args.workload} on the CPU oracle port (C graph build {detail['pcg_s']:.1f} s, components "
                    f"{detail['components_s']:.1f} s, contraction + sklearn SpectralClustering on {detail['spectral_n']} "
                    f"vertices {detail['spectral_s']:.1f} s), measured; the whole job is measured by "
                    f"`bench.py --impl reference` (profiles/README.md)"
                ),
            }  # fmt: skip
    if dist is not None:
        engine.synchronize()
        dist.barrier()  # nobody may unmap a window a peer is still using
    engine.close()
    if dist is not None:
        dist.destroy_process_group()
    return line if rank == 0 else {}


def main() -> None:
    parser = argparse.ArgumentParser()
    parser.add_argument("--gpus", type=int, default=1)
    parser.add_argument("--steps", type=int, default=3)
    parser.add_argument("--warmup", type=int, default=3)
    parser.add_argument("--impl", default="b200", choices=["b200", "reference"])
    parser.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    parser.add_argument("--no-cpu-baseline", action="store_true")
    parser.add_argument("--reference-budget-s", type=float, default=240.0,
                        help="--impl reference: stop starting new full CPU runs after this many seconds "
                             "(one run is always timed)")
    parser.add_argument("--small-limit", type=int, default=-1,
                        help="tuning: nodes up to this many taxa take the one-CTA small-node path (default: the "
                             "library's, 32; capacity 64); larger ones up to 4096 the batched medium path")
    parser.add_argument("--profile-step", action="store_true",
                        help="for ncu: no recording pass, no replay, no CPU baseline -- one warm-up job, then exactly "
                             "one scs_supertree_build bracketed by cudaProfilerStart/Stop "
                             "(ncu --profile-from-start off captures that step only)")
    parser.add_argument("--shard-min-n", type=int, default=4096,
                        help="N > 1: recursion nodes with at least this many taxa are row-sharded over the GPUs "
                             "(0: never; the ranks then only share out the independent sub-problems)")
    parser.add_argument("--dump-outputs", metavar="DIR", default="",
                        help="after the timed steps, write the supertree of the last timed step of each clock as "
                             "DIR/<name>.npy (float64): resident_parent / resident_taxon (value's build; with N > 1 "
                             "rank 0's share) and e2e_parent / e2e_taxon (e2e's build, joined over the ranks)")
    args = parser.parse_args()
    if args.steps < 1 or args.warmup < 0:
        parser.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl == "reference" or args.profile_step):
        parser.error("--dump-outputs writes what the GPU arm's timed steps computed")
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        if rank != 0:
            return
        print(json.dumps(reference_line(args)), flush=True)
        return
    if args.profile_step:
        print(json.dumps(profile_step(args, make_workload(args.workload))), flush=True)
        return
    line = gpu_line(args, make_workload(args.workload))
    if rank == 0:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
