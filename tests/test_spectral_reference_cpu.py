"""CPU: the fp64 reference of the spectral step (oracle/spectral_oracle.py) that tests/test_gpu_spectral_reference.py
holds the kernels to -- its exact 1-D 2-means against brute force and Lloyd's iteration, its eigen routes against each
other, and the two together against the spectral nodes recorded from the unmodified reference (tests/golden)."""

from __future__ import annotations

import numpy as np
import pytest

from helpers import GAP_TIE, load_case, node_graphs
from oracle.spectral_oracle import fiedler_reference, two_means_1d


def brute_force_2means(u: np.ndarray) -> tuple[int, np.ndarray]:
    """(split count of the least within-cluster sum of squares, that SSE for every split) of the sorted signed keys."""
    keys = np.sort(u)
    sse = np.array([((keys[:i] - keys[:i].mean()) ** 2).sum() + ((keys[i:] - keys[i:].mean()) ** 2).sum()
                    for i in range(1, len(keys))])  # fmt: skip
    return int(np.argmin(sse)) + 1, sse


def lloyd_fixed_point(keys: np.ndarray, i: int) -> int | None:
    """Lloyd's iteration from the split after ``i`` sorted keys: the split it stops at, or None if a key is ever
    equidistant from the two centroids (no strict fixed point) or a cluster empties."""
    for _ in range(4 * len(keys)):
        c0, c1 = keys[:i].mean(), keys[i:].mean()
        d0, d1 = np.abs(keys - c0), np.abs(keys - c1)
        if np.any(d0 == d1):
            return None
        lower = d0 < d1
        j = int(lower.sum())
        if not (np.array_equal(lower[:j], np.ones(j, bool)) and 0 < j < len(keys)):
            return None
        if j == i:
            return i
        i = j
    return None


def _inputs():
    rng = np.random.RandomState(5)
    out = [rng.standard_normal(m) for m in (3, 4, 5, 17, 64, 301)]
    out += [rng.uniform(-1, 1, m) ** 3 for m in (7, 40)]
    # heavy ties: few distinct values, duplicate keys on both sides of the cut
    out += [rng.randint(-3, 4, m).astype(float) for m in (6, 9, 25, 200)]
    out += [np.repeat([-1.0, 0.25, 2.0], [5, 7, 3]), np.array([1.0, 1.0, -2.0, -2.0, 0.5]), np.array([0.0, 1.0, 2.0])]
    # two clusters that are nearly tied
    out += [np.concatenate([rng.normal(-1, 0.1, 30), rng.normal(1, 0.1, 30)])]
    return out


@pytest.mark.parametrize("k", range(len(_inputs())))
def test_two_means_matches_brute_force(k):
    u0 = _inputs()[k]
    r = two_means_1d(u0)
    m = len(u0)
    # sign flip: the first entry of largest magnitude is positive
    arg = int(np.flatnonzero(np.abs(u0) == np.abs(u0).max())[0])
    assert r["u"][arg] > 0 or u0[arg] == 0
    assert np.array_equal(np.abs(r["u"]), np.abs(u0))
    keys = r["sorted"]
    best, sse = brute_force_2means(r["u"])
    scale = max(((keys - keys.mean()) ** 2).sum(), 1e-300)
    # the chosen split has the least SSE (to rounding), and no smaller split is strictly better
    assert sse[r["best"] - 1] <= sse.min() + 1e-12 * scale
    assert all(sse[i - 1] > sse.min() + 1e-12 * scale for i in range(1, r["best"]) if i != best)
    # never between two equal keys, so the side rule puts exactly the upper `m - best` keys on side 1
    assert keys[r["best"] - 1] < keys[r["best"]]
    assert int(r["side"].sum()) == m - r["best"]
    assert np.array_equal(r["side"], (r["u"] >= keys[r["best"]]).astype(np.int32))
    # margin: the closest key to the centroid midpoint of the chosen split, over the range
    mid = 0.5 * (keys[: r["best"]].mean() + keys[r["best"] :].mean())
    assert abs(r["margin"] - np.abs(r["u"] - mid).min() / np.ptp(keys)) < 1e-12
    # stable splits and runner-up
    stable = [i for i in range(1, m) if lloyd_fixed_point(keys, i) == i]
    assert r["stable_splits"] == len(stable)
    scores = {i: scale - sse[i - 1] for i in stable}  # between-cluster sum of squares
    others = [scores[i] for i in stable if i != r["best"]]
    expected = max(others) / (scale - sse[r["best"] - 1]) if others else 0.0
    assert abs(r["runner_up"] - expected) < 1e-9


@pytest.mark.parametrize("seed", range(6))
def test_stable_count_equals_lloyd_fixed_points(seed):
    """Every Lloyd run from every split ends at a stable split, and every stable split is one such end."""
    rng = np.random.RandomState(100 + seed)
    u = np.concatenate([rng.normal(c, 0.15, rng.randint(3, 12)) for c in rng.uniform(-2, 2, 4)])
    r = two_means_1d(u)
    ends = {lloyd_fixed_point(r["sorted"], i) for i in range(1, len(u))} - {None}
    assert len(ends) == r["stable_splits"]
    assert r["best"] in ends


# cases with spectral nodes (dcm and dcm_iq split into components only)
SPECTRAL_CASES = ["supertriplets", "c1_100x30_depth", "c2_500x50_branch", "c3_1000x100_branch_weighted",
                  "s_200x40_bootstrap", "s_300x40_branch_weighted", "s_150x40_one"]  # fmt: skip


@pytest.mark.parametrize("name", SPECTRAL_CASES)
def test_reference_reproduces_the_recorded_spectral_nodes(name):
    """Top-level graphs of the golden cases are disconnected, so the spectral nodes below them are rebuilt by the
    oracle and their recorded eigenvalues, margin, stable splits and runner-up reproduced."""
    case = load_case(name)
    by_names = {tuple(n["names"]): n for n in case["nodes"] if "eigenvalues" in n}
    compared = skipped = 0
    for names, Wc in node_graphs(case).items():
        ref = by_names.get(names)
        if ref is None or Wc.shape[0] < 3:
            continue
        lam2, lam3, u = fiedler_reference(Wc)
        assert abs(lam2 - ref["eigenvalues"][1]) < 1e-12, names[:4]
        assert abs(lam3 - ref["eigenvalues"][2]) < 1e-12, names[:4]
        if lam3 - lam2 < 1e-4:
            skipped += 1  # the embedding is ill-determined
            continue
        r = two_means_1d(u)
        km = ref["kmeans"]
        if r["closest"] < 1e-9:
            skipped += 1  # the stable count depends on rounding
            continue
        compared += 1
        assert r["stable_splits"] == km["stable_splits"], names[:4]
        assert abs(r["runner_up"] - km.get("second_best_relative", 0.0)) < 1e-9, names[:4]
        if km["reference_is_optimal"]:
            # the recorded margin is measured on sklearn's partition, here the optimum
            assert abs(r["margin"] - ref["margin"]) < 1e-9, names[:4]
    assert compared >= 10
    print(name, "compared", compared, "skipped", skipped)


def test_dense_and_lanczos_routes_agree():
    rng = np.random.RandomState(3)
    m = 1500
    A = rng.uniform(0, 1, (m, m)) * (rng.random_sample((m, m)) < 0.3)
    A = np.triu(A, 1)
    A = A + A.T
    A[: m // 2, m // 2 :] *= 0.05
    A[m // 2 :, : m // 2] *= 0.05
    d2, d3, du = fiedler_reference(A, dense=True)
    l2, l3, lu = fiedler_reference(A, dense=False)
    assert d3 - d2 > GAP_TIE
    assert abs(d2 - l2) < 1e-12 and abs(d3 - l3) < 1e-12
    du, lu = du / np.linalg.norm(du), lu / np.linalg.norm(lu)
    assert min(np.abs(du - lu).max(), np.abs(du + lu).max()) < 1e-8
    assert np.array_equal(two_means_1d(du)["side"], two_means_1d(lu)["side"])
