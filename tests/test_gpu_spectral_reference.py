"""GPU: everything the spectral step reports, on every solver path, against the fp64 reference
(oracle/spectral_oracle.py) or the values recorded from the reference's own runs (tests/golden).

One contract for every path (solver 2 = dense Jacobi in the small batch, 3 = Lanczos per node or in the medium batch):

* ``eig[1]`` within 1e-10 of lambda_2 (Lanczos: with a true residual below 1e-10);
* ``eig[2]``: Jacobi within 1e-10 of lambda_3; Lanczos never below lambda_3 - 1e-10 (a Ritz value of N never exceeds
  the eigenvalue it approximates, so 1 - theta_2 is an upper estimate of lambda_3);
* ``tie_flag`` bit 0: Jacobi sets it exactly when lambda_3 - lambda_2 < 1e-7 (1e-9 either side of the threshold is
  not judged); Lanczos never sets it without such a gap, but may miss a repeated eigenvalue (test at the end);
* ``margin`` within 1e-6 of the reference wherever the partitions agree and lambda_3 - lambda_2 >= 1e-4;
* bit 1, bit 4, ``kmeans_stable_splits`` and ``kmeans_runner_up`` as the exact 2-means of the reference embedding
  gives them, except where a sorted key lies within 1e-9 of the range from a split's centroid midpoint (counted);
* the partition: the reference's best split up to label swap wherever there is no tie.

Where a test targets a path it asserts on ``solver``, ``restarts``, ``nodes_medium`` and ``nodes_rerun`` that the
input took it."""

from __future__ import annotations

import math

import numpy as np
import pytest

from helpers import (CASES, compare_with_ctrace, compare_with_reference_trace, ctrace_key, ctrace_part_hash,
                     flat_clades, load_case, load_ctrace, node_graphs, parse)  # fmt: skip
from oracle import scs_oracle
from oracle.spectral_oracle import fiedler_reference, normalized_operator, two_means_1d
from spectralclustersupertree_b200.engine import Forest

pytestmark = pytest.mark.gpu

GAP_TIE = 1e-7
NEAR = 1e-9
CLEAR_GAP = 1e-4  # eigengap above which the embedding (margin, stable splits, partition) is well determined
SMALL_DEFAULT, MEDIUM_DEFAULT = 32, 4096


def check_bit0(stats, gap: float) -> None:
    bit0 = bool(stats.tie_flag & 1)
    if stats.solver == 2:
        if abs(gap - GAP_TIE) > NEAR:
            assert bit0 == (gap < GAP_TIE), (gap, stats.tie_flag)
    else:
        assert not bit0 or gap < GAP_TIE + NEAR, (gap, stats.tie_flag)  # no false positives


def check_eigenvalues(stats, lam2: float, lam3: float) -> None:
    assert stats.solver in (2, 3), stats.solver
    assert abs(stats.eig[1] - lam2) <= 1e-10, (stats.eig[1], lam2)
    if stats.solver == 2:
        assert abs(stats.eig[2] - lam3) <= 1e-10, (stats.eig[2], lam3)
    else:
        assert stats.residual < 1e-10, stats.residual
        assert stats.eig[2] >= lam3 - 1e-10, (stats.eig[2], lam3)
    check_bit0(stats, lam3 - lam2)


def check_against_reference(side: np.ndarray, stats, W: np.ndarray) -> dict:
    """The whole contract for one spectral step with side[m] per vertex of the graph W.  Returns what was compared."""
    lam2, lam3, u = fiedler_reference(W)
    check_eigenvalues(stats, lam2, lam3)
    r = two_means_1d(u)
    out = {"partition": False, "kmeans": False}
    if lam3 - lam2 < CLEAR_GAP:
        return out
    same = np.array_equal(side, r["side"]) or np.array_equal(side, 1 - r["side"])
    if r["margin"] >= 1e-6:
        assert same, "partition differs from the reference's best split"
        out["partition"] = True
    if same:
        assert abs(stats.margin - r["margin"]) < 1e-6, (stats.margin, r["margin"])
    if r["closest"] >= NEAR:
        assert stats.kmeans_stable_splits == r["stable_splits"], (stats.kmeans_stable_splits, r["stable_splits"])
        assert bool(stats.tie_flag & 16) == (r["stable_splits"] > 1)
        assert abs(stats.kmeans_runner_up - r["runner_up"]) < 1e-6, (stats.kmeans_runner_up, r["runner_up"])
        assert bool(stats.tie_flag & 2) == (r["margin"] < 1e-9)
        out["kmeans"] = True
    return out


# ---- a. matrix level: scs_spectral_bipartition_dev (per-node Lanczos) ------------------------------------------------
def planted(m: int, seed: int, spread: bool = False) -> np.ndarray:
    """Dense two-community graph (cross weights x 0.05); ``spread``: weights also scaled by 10^U(-6, 6)."""
    rng = np.random.RandomState(seed)
    A = np.triu(rng.uniform(0.5, 1.5, (m, m)), 1)
    if spread:
        A *= 10.0 ** np.triu(rng.uniform(-6, 6, (m, m)), 1)
    A += A.T
    h = max(m // 2, 1)
    A[:h, h:] *= 0.05
    A[h:, :h] *= 0.05
    return A


# both sides of every kernel switch: warp- / CTA-per-row matvec at 2048, lanczos_tail / the lanczos_step cluster above
# 4096, two_means_1d / two_means_staged + sort_tile / sort_far above 8192 keys (m = 8193 sorts 8191 +inf pads)
@pytest.mark.parametrize("m", [3, 4, 33, 2047, 2048, 2049, 4095, 4096, 4097, 8192, 8193, 9973])
def test_planted_graph_on_both_sides_of_every_kernel_switch(engine, m):
    W = planted(m, m)
    side, stats = engine.spectral_bipartition(W, seed=7)
    assert stats.solver == 3 and stats.restarts == 0
    done = check_against_reference(side, stats, W)
    assert done["partition"] and done["kmeans"]
    assert stats.tie_flag == 0


@pytest.mark.parametrize("m", [40, 700, 5000])
def test_weights_spanning_twelve_decades(engine, m):
    W = planted(m, 100 + m, spread=True)
    side, stats = engine.spectral_bipartition(W, seed=3)
    assert stats.solver == 3 and not stats.tie_flag & 12
    check_against_reference(side, stats, W)


def test_isolated_vertex(engine):
    W = planted(60, 5)
    W[17, :] = W[:, 17] = 0.0
    side, stats = engine.spectral_bipartition(W, seed=1)
    vals, _ = scs_oracle.normalized_affinity_eigs(W, 3)  # scipy's rule: a vertex of degree 0 is scaled by 1
    assert abs(stats.eig[1] - vals[1]) <= 1e-10
    assert not stats.tie_flag & 8  # a zero degree is not a bad one
    done = check_against_reference(side, stats, W)
    assert done["partition"]


def test_given_degree_and_a_negative_one(engine):
    # integer weights: the row sums are exact in any order, so the given degrees are the ones the kernel computes
    rng = np.random.RandomState(2)
    W = np.triu(rng.randint(0, 9, (300, 300)).astype(float), 1)
    W += W.T
    W[:150, 150:] = np.floor(W[:150, 150:] / 8)
    W[150:, :150] = W[:150, 150:].T
    a_side, a = engine.spectral_bipartition(W, seed=4)
    b_side, b = engine.spectral_bipartition(W, seed=4, degree=W.sum(axis=1))
    assert np.array_equal(a_side, b_side)
    assert bytes(a) == bytes(b)
    check_against_reference(a_side, a, W)
    degree = W.sum(axis=1)
    degree[10] = -1.0
    _, c = engine.spectral_bipartition(W, seed=4, degree=degree)
    assert c.tie_flag & 8


def test_two_seeds_give_the_same_partition(engine):
    W = planted(500, 9)
    a_side, a = engine.spectral_bipartition(W, seed=0)
    b_side, b = engine.spectral_bipartition(W, seed=12345)
    assert np.array_equal(a_side, b_side) or np.array_equal(a_side, 1 - b_side)
    assert abs(a.eig[1] - b.eig[1]) <= 1e-10
    assert check_against_reference(a_side, a, W)["partition"]


@pytest.mark.parametrize("m", [5, 5000])
def test_complete_graph_takes_the_deflated_second_run(engine, m):
    """K_m: lambda_2 = ... = lambda_m = m / (m - 1).  The Krylov space closes after one step, so the solver runs
    again deflated by the Fiedler vector -- on lanczos_tail at m = 5, on the lanczos_step cluster at m = 5000."""
    W = np.ones((m, m)) - np.eye(m)
    side, stats = engine.spectral_bipartition(W, seed=2)
    assert stats.solver == 3
    assert abs(stats.eig[1] - m / (m - 1)) <= 1e-10
    assert stats.tie_flag & 1
    assert abs(stats.eig[2] - stats.eig[1]) <= 1e-10
    assert 0 < side.sum() < m


# numpy copy of the documented restart scheme (csrc/spectral.cu: lanczos_largest, csrc/spectral_dev.cuh): Lanczos
# with full re-orthogonalisation against q0 = sqrt(d) / |sqrt(d)| and the basis, checks every 4 steps and at the last
# one, converged when beta_j <= 1e-11 or |beta_j s_j| <= 1e-12, explicit restart from the Ritz vector after
# kMaxBasis = 256 steps, at most kMaxRestarts = 8 restarts.
def lanczos_restarts(W: np.ndarray, seed: int = 0, max_basis: int = 256, max_restarts: int = 8):
    """(restarts, converged, theta_1) of the scheme above from a random start."""
    from threadpoolctl import threadpool_limits

    with threadpool_limits(limits=1):  # thousands of small products: threads only add overhead
        return _lanczos_restarts(W, seed, max_basis, max_restarts)


def _lanczos_restarts(W, seed, max_basis, max_restarts):
    from scipy.linalg import eigh_tridiagonal

    N, _ = normalized_operator(W)
    d = W.sum(axis=1)
    q0 = np.sqrt(d) / math.sqrt(d.sum())
    m = len(d)
    jmax = min(m - 1, max_basis)
    V = np.zeros((jmax + 2, m))
    V[0] = q0
    v = np.random.RandomState(seed).uniform(-1, 1, m)
    theta = float("nan")
    for attempt in range(max_restarts + 1):

        def orth(w, k):
            h1 = V[:k] @ w
            w = w - V[:k].T @ h1
            h2 = V[:k] @ w
            return w - V[:k].T @ h2, h1 + h2

        w, _ = orth(v, 1)
        V[1] = w / np.linalg.norm(w)
        alpha, beta = np.zeros(jmax), np.zeros(jmax)
        latched = 0
        for j in range(1, jmax + 1):
            w, h = orth(N @ V[j], j + 1)
            alpha[j - 1], beta[j - 1] = h[j], np.linalg.norm(w)
            if beta[j - 1] <= 1e-11 and not latched:
                latched = j
            V[j + 1] = w / beta[j - 1] if beta[j - 1] > 0 else w
            if j % 4 == 0 or j == jmax:
                k = latched or j
                th, S = eigh_tridiagonal(alpha[:k], beta[: k - 1])
                theta = float(th[-1])
                if beta[k - 1] <= 1e-11 or abs(beta[k - 1] * S[-1, -1]) <= 1e-12:
                    return attempt, True, theta
        y = V[1 : k + 1].T @ S[:, -1]
        v = y / np.linalg.norm(y)
    return max_restarts, False, theta


def weighted_path(m: int, seed: int) -> np.ndarray:
    w = np.random.RandomState(seed).uniform(0.5, 2.0, m - 1)
    W = np.zeros((m, m))
    i = np.arange(m - 1)
    W[i, i + 1] = W[i + 1, i] = w
    return W


def test_explicit_restart_after_the_basis_is_full(engine):
    """A weighted path of 300 vertices: lambda_3 - lambda_2 = 1.5e-4, so 256 steps (of a 299-dimensional space) do not
    reach the residual; the restarted runs do (the numpy copy needs 3 restarts)."""
    W = weighted_path(300, 1)
    restarts, converged, _ = lanczos_restarts(W, seed=1)
    assert converged and 1 <= restarts < 8
    lam2, lam3, _ = fiedler_reference(W)
    side, stats = engine.spectral_bipartition(W, seed=1)
    assert stats.solver == 3 and stats.restarts >= 1
    assert not stats.tie_flag & 4
    assert stats.matvecs > 256
    check_against_reference(side, stats, W)


def test_restart_limit(engine):
    """A weighted path of 1 000 vertices (lambda_3 - lambda_2 = 1.3e-5): nine runs of 256 steps stop short of the
    residual.  The pair is accepted and flagged (bit 2); its Ritz value still bounds lambda_2 from above."""
    W = weighted_path(1000, 0)
    restarts, converged, _ = lanczos_restarts(W, seed=0)
    assert not converged and restarts == 8
    lam2, _, _ = fiedler_reference(W)
    side, stats = engine.spectral_bipartition(W, seed=0)
    assert stats.solver == 3 and stats.restarts == 8
    assert stats.tie_flag & 4
    assert stats.eig[1] >= lam2 - 1e-12
    assert 0 < side.sum() < len(side)


# ---- b. the batched paths against the recorded traces ---------------------------------------------------------------
LIMITS = [(64, 4096), (SMALL_DEFAULT, MEDIUM_DEFAULT), (0, 4096), (0, 0)]
UNTIDY = ["branch", "bootstrap", "depth", "nocontract", "caterpillar"]
UNTIDY_MISMATCHES = {"caterpillar": 2}  # see tests/test_gpu_untidy.py
_GRAPHS: dict = {}


def build_with_limits(engine, forest_of, weighting, small, medium, contract=True):
    engine.set_small_node_limit(small)
    engine.set_medium_node_limit(medium)
    try:
        built = engine.supertree_build(forest_of(), weighting, contract_edges=contract, record=True)
    finally:
        engine.set_small_node_limit(SMALL_DEFAULT)
        engine.set_medium_node_limit(MEDIUM_DEFAULT)
    solvers = {int(s.solver) for _, _, s in built["records"] if s.spectral_ran and s.contracted_size >= 3}
    assert solvers <= {2, 3}, solvers
    if small == 0:
        assert 2 not in solvers
    if medium == 0:
        assert built["nodes_medium"] == 0
    sizes = [len(t) for t, _, s in built["records"] if s.spectral_ran and s.contracted_size >= 3]
    if small and any(n <= small for n in sizes):
        assert 2 in solvers
    if medium and any(max(small, 2) < n <= medium for n in sizes):
        assert built["nodes_medium"] > 0
    return built


def check_record_stats(stats, lam2, lam3, margin, same, stable=None, runner=None) -> bool:
    """The contract on one record against recorded values; the 2-means fields only where the recorded embedding is
    well determined.  Returns whether they were compared."""
    check_eigenvalues(stats, lam2, lam3)
    if lam3 - lam2 < CLEAR_GAP:
        return False
    if same and margin is not None:
        assert abs(stats.margin - margin) < 1e-6, (stats.margin, margin)
        if margin > 2e-9:
            assert not stats.tie_flag & 2
        elif margin < 5e-10:
            assert stats.tie_flag & 2
    if stable is None:
        return False
    assert stats.kmeans_stable_splits == stable, (stats.kmeans_stable_splits, stable)
    assert bool(stats.tie_flag & 16) == (stable > 1)
    if runner is not None:
        assert abs(stats.kmeans_runner_up - runner) < 1e-6, (stats.kmeans_runner_up, runner)
    return True


@pytest.mark.parametrize("limits", LIMITS, ids=lambda v: f"small{v[0]}-medium{v[1]}")
@pytest.mark.parametrize("name", list(CASES))
def test_golden_cases_on_every_path(engine, name, limits):
    case = load_case(name)
    names = case["names"]
    trees = parse(case["lines"])
    built = build_with_limits(engine, lambda: Forest.from_trees(trees, case["weights"], names), case["weighting"],
                              *limits)  # fmt: skip
    if name not in _GRAPHS:
        _GRAPHS[name] = node_graphs(case)
    graphs = _GRAPHS[name]
    trace = []
    for taxa, part, stats in built["records"]:
        rec = {"names": sorted(names[t] for t in taxa), "n_components": int(stats.n_components)}
        if stats.spectral_ran:
            rec["contracted_size"] = int(stats.contracted_size)
            rec["partition"] = [sorted(names[t] for t in taxa[part == s]) for s in (0, 1)]
        trace.append((rec, stats))
    compare_with_reference_trace([r for r, _ in trace], case["nodes"], name)
    by_names = {tuple(n["names"]): n for n in case["nodes"]}
    checked = kmeans = skipped = 0
    for rec, stats in trace:
        ref = by_names.get(tuple(rec["names"]))
        if ref is None or "eigenvalues" not in ref or rec.get("contracted_size", 0) < 3:
            continue
        checked += 1
        # the recorded margin is measured on sklearn's own split (before a steered node was replaced)
        sklearn = ref.get("partition_seed0", ref["partition"])
        same = {frozenset(p) for p in rec["partition"]} == {frozenset(p) for p in sklearn}
        e, km = ref["eigenvalues"], ref["kmeans"]
        W = graphs.get(tuple(rec["names"]))
        near = W is None or two_means_1d(fiedler_reference(W)[2])["closest"] < NEAR
        skipped += near
        stable = None if near else km["stable_splits"]
        kmeans += check_record_stats(stats, e[1], e[2], ref["margin"], same, stable, km.get("second_best_relative", 0.0))
    if any("eigenvalues" in n and n["contracted_size"] >= 3 for n in case["nodes"]):
        assert checked > 0
    print(name, limits, "checked", checked, "2-means fields", kmeans, "near a midpoint", skipped)


def check_ctrace(records, ctrace, expected_mismatches=0) -> tuple[int, int]:
    compare_with_ctrace(records, ctrace, expected_mismatches=expected_mismatches)
    by_key = {node["key"]: node for node in ctrace["nodes"]}
    checked = kmeans = 0
    for taxa, part, stats in records:
        ref = by_key.get(ctrace_key(taxa))
        if ref is None or "eig" not in ref or ref["m"] < 3:
            continue
        checked += 1
        lam2, lam3 = ref["eig"]
        same = ctrace_part_hash(part) == ref.get("nat", ref["part"])  # the split the recorded margin is measured on
        # the compact trace keeps the stable count only where it exceeds 1; the margin stands in for the embedding
        well = ref["margin"] >= 1e-6
        stable = ((ref.get("km") or {}).get("stable", 1)) if well else None
        kmeans += check_record_stats(stats, lam2, lam3, ref["margin"], same, stable)
    return checked, kmeans


@pytest.mark.parametrize("limits", LIMITS, ids=lambda v: f"small{v[0]}-medium{v[1]}")
@pytest.mark.parametrize("case", UNTIDY)
def test_untidy_cases_on_every_path(engine, case, limits):
    ctrace = load_ctrace(f"untidy_{case}")
    trees = parse(ctrace["lines"])
    names = sorted({x for t in trees for x in t.get_tip_names()})
    built = build_with_limits(engine, lambda: Forest.from_trees(trees, ctrace["weights"], names), ctrace["weighting"],
                              *limits, contract=ctrace.get("contract_edges", True))  # fmt: skip
    checked, kmeans = check_ctrace(built["records"], ctrace, UNTIDY_MISMATCHES.get(case, 0))
    assert checked > 0
    print(case, limits, "checked", checked, "2-means fields", kmeans)


def test_c4_large_nodes(engine):
    """The C4 workload with the default limits: its largest nodes run the lanczos_step cluster and, above 8192
    contracted vertices, the staged 2-means sort."""
    import bench

    ctrace = load_ctrace("c4")
    arrays = bench.make_workload("c4")
    forest = Forest.from_arrays(arrays["node_offsets"], arrays["parent"], arrays["length"], arrays["support"],
                                arrays["taxon"], arrays["weights"], arrays["names"])  # fmt: skip
    built = engine.supertree_build(forest, arrays["weighting"], record=True)
    big = [s.contracted_size for _, _, s in built["records"] if s.spectral_ran]
    assert max(big) > 8192 and sum(m > 4096 for m in big) >= 2
    checked, kmeans = check_ctrace(built["records"], ctrace)
    assert checked > 1000
    print("c4 checked", checked, "2-means fields", kmeans)


# ---- c. the medium batch's re-run of a node through the per-node path ----------------------------------------------
def three_clades(size: int):
    """Three clades G1, G2, G3 of ``size`` taxa (same shape) in the trees ((G1,G2),G3), ((G2,G3),G1), ((G1,G3),G2)
    with equal weights: each clade contracts to one vertex and the node becomes an equal-weight K3 (lambda_2 =
    lambda_3 = 1.5)."""
    groups = [[f"{g}{i:02d}" for i in range(size)] for g in "abc"]

    def clade(taxa):
        text = taxa[-1]
        for x in reversed(taxa[:-1]):
            text = f"({x},{text})"
        return text

    a, b, c = (clade(g) for g in groups)
    lines = [f"(({a},{b}),{c});", f"(({b},{c}),{a});", f"(({a},{c}),{b});"]
    names = sorted(x for g in groups for x in g)
    return parse(lines), names, groups


def _top_record(built, n):
    return next((taxa, part, stats) for taxa, part, stats in built["records"] if len(taxa) == n)


def test_medium_node_with_a_repeated_fiedler_value_is_rerun(engine):
    trees, names, groups = three_clades(20)

    def forest():
        return Forest.from_trees(trees, [1.0] * 3, names)

    built = engine.supertree_build(forest(), "one", record=True)
    assert built["nodes_medium"] >= 1 and built["nodes_rerun"] >= 1
    taxa, part, stats = _top_record(built, 60)
    assert stats.contracted_size == 3 and stats.solver == 3
    assert stats.tie_flag & 1
    assert abs(stats.eig[1] - 1.5) <= 1e-10 and abs(stats.eig[2] - 1.5) <= 1e-10
    side = dict(zip((names[t] for t in taxa), part.tolist(), strict=True))
    for g in groups:
        assert len({side[x] for x in g}) == 1
    assert len(set(side.values())) == 2
    engine.set_medium_node_limit(0)
    try:
        per_node = engine.supertree_build(forest(), "one", record=True)
    finally:
        engine.set_medium_node_limit(MEDIUM_DEFAULT)
    assert per_node["nodes_medium"] == 0
    assert flat_clades(built["parent"], built["taxon"]) == flat_clades(per_node["parent"], per_node["taxon"])


def test_small_node_with_a_repeated_fiedler_value(engine):
    trees, names, groups = three_clades(8)
    built = engine.supertree_build(Forest.from_trees(trees, [1.0] * 3, names), "one", record=True)
    taxa, part, stats = _top_record(built, 24)
    assert stats.solver == 2 and stats.contracted_size == 3
    assert stats.tie_flag & 1
    assert abs(stats.eig[1] - 1.5) <= 1e-10 and abs(stats.eig[2] - 1.5) <= 1e-10
    side = dict(zip((names[t] for t in taxa), part.tolist(), strict=True))
    for g in groups:
        assert len({side[x] for x in g}) == 1


# ---- d. the multiplicity a single-vector Krylov space cannot see ---------------------------------------------------
def block_circulant(size: int = 60, seed: int = 4) -> np.ndarray:
    """Three copies of one random graph joined pairwise by the same weak symmetric block: N commutes with the cyclic
    shift of the copies, so every eigenvalue of its antisymmetric sector is double -- lambda_2 = lambda_3 among
    them."""
    rng = np.random.RandomState(seed)
    A = np.triu(rng.uniform(0, 1, (size, size)), 1)
    A += A.T
    B = 0.01 * rng.uniform(0, 1, (size, size))
    B = B + B.T
    return np.block([[A, B, B], [B, A, B], [B, B, A]])


def test_block_circulant_fiedler_value(engine):
    W = block_circulant()
    lam2, lam3, _ = fiedler_reference(W)
    assert lam3 - lam2 < 1e-12
    side, stats = engine.spectral_bipartition(W, seed=5)
    assert stats.solver == 3
    assert abs(stats.eig[1] - lam2) <= 1e-10 and stats.residual < 1e-10


@pytest.mark.xfail(strict=True, reason="single-vector Lanczos: the Krylov space never closes on a repeated Fiedler "
                   "eigenvalue, so the deflated second run does not happen and bit 0 stays clear")  # fmt: skip
def test_block_circulant_repeated_fiedler_value_is_flagged(engine):
    side, stats = engine.spectral_bipartition(block_circulant(), seed=5)
    assert stats.tie_flag & 1
