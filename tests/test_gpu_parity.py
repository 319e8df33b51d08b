"""GPU: the CUDA path, called through the C ABI, against the golden vectors recorded from the
reference and against the CPU oracle on the same seeded inputs.

Bars (BASELINE.json north_star): W, adjacency, occurrences, component labels, contraction groups
and contracted weights bit-exact (for every weighting -- the row kernel sums in tree input order
with separately rounded multiply and add, like the reference); Fiedler eigenvalue within 1e-6;
partitions identical up to label swap wherever the eigengap / 2-means margin is not a tie."""

from __future__ import annotations

import numpy as np
import pytest

from helpers import CASES, load_case, parse
from oracle import scs_oracle
from spectralclustersupertree_b200.engine import Forest, unpack_bits
from spectralclustersupertree_b200.flatten import flatten_trees

pytestmark = pytest.mark.gpu


def tours_of(case, weighting=None):
    trees = parse(case["lines"])
    tid = {x: i for i, x in enumerate(case["names"])}
    return flatten_trees(trees, case["weights"], weighting or case["weighting"], tid)


@pytest.mark.parametrize("name", list(CASES))
def test_pcg_build_bit_exact(engine, name):
    case = load_case(name)
    ref = case["pcg"]
    n = len(case["names"])
    out = engine.pcg_build(tours_of(case), want_counts=True)
    assert np.array_equal(out["W"], ref["W"])
    assert np.array_equal(out["W"], out["W"].T)
    assert np.array_equal(out["C"], ref["C"])
    assert np.array_equal(out["occ"], ref["occ"])
    assert np.array_equal(unpack_bits(out["adj_bits"], n), ref["C"] > 0)
    top = np.maximum(ref["occ"][:, None], ref["occ"][None, :])
    assert np.array_equal(unpack_bits(out["max_bits"], n), (ref["C"] > 0) & (ref["C"] == top))
    assert np.allclose(out["degree"], ref["W"].sum(axis=1), rtol=1e-13, atol=0)
    # without the count matrix the other outputs are unchanged
    lean = engine.pcg_build(tours_of(case), want_counts=False)
    for key in ("W", "occ", "adj_bits", "max_bits", "degree"):
        assert np.array_equal(lean[key], out[key]), key


@pytest.mark.parametrize("name", ["supertriplets", "c1_100x30_depth"])
def test_pcg_other_weightings_match_oracle(engine, name):
    case = load_case(name)
    trees = parse(case["lines"])
    tid = {x: i for i, x in enumerate(case["names"])}
    for weighting in ("one", "depth", "branch"):
        W, C, occ = scs_oracle.pcg_dense_c(trees, case["weights"], weighting, tid)
        out = engine.pcg_build(flatten_trees(trees, case["weights"], weighting, tid))
        assert np.array_equal(out["W"], W), weighting
        assert np.array_equal(out["C"], C), weighting
        assert np.array_equal(out["occ"], occ), weighting


@pytest.mark.parametrize("name", list(CASES))
def test_components_bit_exact(engine, name):
    case = load_case(name)
    ref = case["pcg"]
    n = len(case["names"])
    out = engine.pcg_build(tours_of(case), want_counts=False)
    label, count = engine.components(out["adj_bits"], n)
    assert np.array_equal(label, ref["label"])
    assert count == len(np.unique(ref["label"]))


@pytest.mark.parametrize("name", list(CASES))
def test_contraction_bit_exact(engine, name):
    case = load_case(name)
    ref = case["pcg"]
    out = engine.pcg_build(tours_of(case), want_counts=False)
    group, m, Wc, deg = engine.contract(out["W"], out["adj_bits"], out["max_bits"])
    assert np.array_equal(group, ref["group"])
    assert m == int(ref["group"].max()) + 1
    assert np.array_equal(Wc, ref["Wc"][:m, :m])
    assert np.allclose(deg, ref["Wc"][:m, :m].sum(axis=1), rtol=1e-13, atol=0)


def random_affinity(n, density, seed):
    rng = np.random.RandomState(seed)
    A = rng.uniform(0, 10, size=(n, n)) * (rng.random_sample((n, n)) < density)
    A = np.triu(A, 1)
    return A + A.T


@pytest.mark.parametrize(("n", "density", "seed"), [(3, 1.0, 1), (5, 0.9, 2), (17, 0.8, 3), (64, 0.5, 4),
                                                    (257, 0.8, 5), (1000, 0.6, 6), (2500, 0.8, 7)])  # fmt: skip
def test_spectral_eigenvalue_and_partition(engine, n, density, seed):
    A = random_affinity(n, density, seed)
    # two planted communities so the Fiedler vector is well separated
    half = n // 2
    A[:half, half:] *= 0.05
    A[half:, :half] *= 0.05
    side, stats = engine.spectral_bipartition(A, seed=11)
    vals, emb = scs_oracle.normalized_affinity_eigs(A, 3)
    assert abs(stats.eig[1] - vals[1]) < 1e-6 * max(1.0, abs(vals[1]))
    assert stats.residual < 1e-9
    if n > 3 and vals[2] - vals[1] > 1e-6:
        ref = scs_oracle.spectral_bipartition(A, np.random.RandomState(0))
        assert np.array_equal(side, ref) or np.array_equal(side, 1 - ref)
        assert stats.tie_flag == 0


def test_spectral_matches_oracle_on_reference_graphs(engine):
    """The contracted graphs the reference hands to sklearn at the spectral nodes of c1."""
    case = load_case("c1_100x30_depth")
    trees = parse(case["lines"])
    checked = 0
    for node in case["nodes"]:
        if "eigenvalues" not in node or len(node["names"]) < 3:
            continue
        names = node["names"]
        keep = set(names)
        sub = [t.get_sub_tree(keep, ignore_missing=True, as_rooted=True) for t in trees
               if len(keep & set(t.get_tip_names())) >= 2]  # fmt: skip
        tid = {x: i for i, x in enumerate(names)}
        W, C, occ = scs_oracle.pcg_dense_c(sub, [1.0] * len(sub), case["weighting"], tid)
        _, Wc, _ = scs_oracle.contract_dense(W, C, occ)
        if Wc.shape[0] < 3:
            continue
        side, stats = engine.spectral_bipartition(Wc, seed=3)
        assert abs(stats.eig[1] - node["eigenvalues"][1]) < 1e-6
        checked += 1
    assert checked >= 10


def test_spectral_tiny_and_degenerate(engine):
    side, stats = engine.spectral_bipartition(np.array([[0.0, 2.0], [2.0, 0.0]]))
    assert sorted(side.tolist()) == [0, 1]
    assert stats.solver == 1
    # path a-b-c: the middle vertex sits exactly on the boundary -> reported as a tie
    P = np.array([[0.0, 1.0, 0.0], [1.0, 0.0, 1.0], [0.0, 1.0, 0.0]])
    side, stats = engine.spectral_bipartition(P)
    assert side[0] != side[2]
    assert abs(stats.eig[1] - 1.0) < 1e-9
    # complete graph K3: lambda_2 == lambda_3 -> tie flagged
    K = np.ones((3, 3)) - np.eye(3)
    side, stats = engine.spectral_bipartition(K)
    assert stats.tie_flag & 1
    assert 0 < side.sum() < 3
    from spectralclustersupertree_b200.engine import ScsError

    with pytest.raises(ScsError):
        engine.spectral_bipartition(np.zeros((1, 1)))


@pytest.mark.parametrize("m", [2, 3, 31, 100, 1001, 2047, 2048, 2049, 3001, 4097, 8193])  # warp / CTA per row at 2048
def test_normalized_matvec(engine, m):
    A = random_affinity(m, 0.7, m)
    d = A.sum(axis=1)
    isd = np.where(d > 0, 1.0 / np.sqrt(np.where(d > 0, d, 1.0)), 1.0)
    x = np.random.RandomState(m).uniform(-1, 1, m)
    y = engine.normalized_matvec(A, isd, x)
    ref = isd * (A @ (isd * x))
    assert np.allclose(y, ref, rtol=1e-12, atol=1e-14)


def test_node_split_host_components_and_sides(engine):
    case = load_case("dcm")  # disconnected at the top level: part = component index by smallest member
    part, stats = engine.node_split(tours_of(case))
    ref_label = case["pcg"]["label"]
    _, expected = np.unique(ref_label, return_inverse=True)
    assert stats.n_components == len(np.unique(ref_label))
    assert np.array_equal(part, expected)
    bufs = engine.last_node_buffers()
    assert np.array_equal(bufs["W"], case["pcg"]["W"])
    assert np.array_equal(bufs["occ"], case["pcg"]["occ"])


def test_forest_split_matches_node_split(engine):
    case = load_case("s_300x40_branch_weighted")
    trees = parse(case["lines"])
    forest = Forest.from_trees(trees, case["weights"], case["names"])
    taxa, part, stats = engine.forest_split(forest, "branch")
    part2, stats2 = engine.node_split(tours_of(case))
    assert np.array_equal(taxa, np.arange(len(case["names"])))
    assert np.array_equal(part, part2)
    assert stats.n_components == stats2.n_components


def test_large_graph_properties(engine):
    """Size-independent properties at a size the Python oracle cannot reach quickly: symmetry,
    determinism (two builds are bit-identical), degree = row sums, occ = leaf counts, integer
    weights for unit-weight depth weighting, and agreement with the C oracle."""
    from spectralclustersupertree_b200.synthetic import make_problem

    prob = make_problem(3000, 120, "depth", 4242)
    trees = prob.phylonodes()
    names = sorted({x for t in trees for x in t.get_tip_names()})
    tid = {x: i for i, x in enumerate(names)}
    tours = flatten_trees(trees, [1.0] * len(trees), "depth", tid)
    a = engine.pcg_build(tours, want_counts=False)
    b = engine.pcg_build(tours, want_counts=False)
    assert np.array_equal(a["W"], b["W"])
    assert np.array_equal(a["W"], a["W"].T)
    assert np.array_equal(a["W"], np.round(a["W"]))
    assert np.array_equal(a["degree"], a["W"].sum(axis=1))  # integers: any order is exact
    assert np.array_equal(a["occ"], np.bincount(tours.leaf_taxon, minlength=len(names)))
    W, C, occ = scs_oracle.pcg_dense_c(trees, [1.0] * len(trees), "depth", tid)
    assert np.array_equal(a["W"], W)
    assert np.array_equal(unpack_bits(a["adj_bits"], len(names)), C > 0)


def _caterpillar(names, rng, lengths=True):
    """A maximally deep tree over ``names`` (every internal node has one leaf child), leaves in random order."""
    order = list(rng.permutation(names))
    fmt = (lambda: f":{rng.uniform(0.01, 3.0):.6f}") if lengths else (lambda: "")
    s = f"({order[0]}{fmt()},{order[1]}{fmt()})"
    for x in order[2:]:
        s = f"({s}{fmt()},{x}{fmt()})" if rng.rand() < 0.5 else f"({x}{fmt()},{s}{fmt()})"
    return s + ";"


def _bushy(names, rng, lengths=True):
    """Random tree with polytomies over ``names``."""
    fmt = (lambda: f":{rng.uniform(0.01, 3.0):.6f}") if lengths else (lambda: "")
    items = [f"{x}{fmt()}" for x in rng.permutation(names)]
    while len(items) > 1:
        k = min(len(items), int(rng.choice([2, 2, 2, 3, 5])))
        picked = [items.pop(int(rng.randint(len(items)))) for _ in range(k)]
        inner = "(" + ",".join(picked) + ")"
        items.append(inner + (fmt() if len(items) > 0 else ""))
    return items[0].rsplit(")", 1)[0] + ");"


@pytest.mark.parametrize("weighting", ["branch", "depth", "one"])
def test_pcg_deep_trees_bit_exact(engine, weighting):
    """Leaves with far more ancestors than one round of the row kernel's chain walk holds (15 a side), on
    either side of the leaf, together with polytomies: the continuation rounds must visit every pair once,
    in tree order."""
    rng = np.random.RandomState(77)
    names = [f"x{i:03d}" for i in range(140)]
    lines, weights = [], []
    for t in range(24):
        sub = list(rng.choice(names, size=int(rng.randint(3, 120)), replace=False))
        make = _caterpillar if t % 3 else _bushy
        lines.append(make(sub, rng, lengths=weighting == "branch"))
        weights.append(float(rng.uniform(0.5, 2.0)))
    trees = parse(lines)
    tid = {x: i for i, x in enumerate(names)}
    W, C, occ = scs_oracle.pcg_dense_c(trees, weights, weighting, tid)
    out = engine.pcg_build(flatten_trees(trees, weights, weighting, tid))
    assert np.array_equal(out["W"], W)
    assert np.array_equal(out["C"], C)
    assert np.array_equal(out["occ"], occ)
    assert np.array_equal(unpack_bits(out["adj_bits"], len(names)), C > 0)


def test_pcg_rows_in_column_chunks_bit_exact(engine):
    """More taxa than one CTA's shared memory holds columns for (10 080 at two CTAs per SM): every row is built
    by several chunk CTAs, each reading only its own buckets of every tree."""
    rng = np.random.RandomState(5)
    n = 10500
    names = [f"x{i:05d}" for i in range(n)]
    lines, weights = [], []
    for t in range(16):
        sub = list(rng.choice(names, size=int(rng.randint(50, 700)), replace=False))
        lines.append((_bushy if t % 2 else _caterpillar)(sub, rng))
        weights.append(float(rng.uniform(0.5, 2.0)))
    # one tree that covers both ends of the taxon range, so that pairs across chunks exist
    lines.append(_bushy(names[:40] + names[-40:], rng))
    weights.append(1.25)
    trees = parse(lines)
    tid = {x: i for i, x in enumerate(names)}
    W, C, occ = scs_oracle.pcg_dense_c(trees, weights, "branch", tid)
    out = engine.pcg_build(flatten_trees(trees, weights, "branch", tid), want_counts=False)
    assert np.array_equal(out["W"], W)
    assert np.array_equal(out["occ"], occ)
    assert np.array_equal(unpack_bits(out["adj_bits"], n), C > 0)
    top = np.maximum(occ[:, None], occ[None, :])
    assert np.array_equal(unpack_bits(out["max_bits"], n), (C > 0) & (C == top))


def test_pcg_wide_bucket_entries_bit_exact(engine):
    """Nodes with 65 536 taxa or more keep {tour position, slot} in 8-byte entries; the same path at a size the
    oracle can check."""
    case = load_case("c2_500x50_branch")
    ref = case["pcg"]
    engine.set_wide_entries(True)
    try:
        out = engine.pcg_build(tours_of(case), want_counts=True)
        lean = engine.pcg_build(tours_of(case), want_counts=False)  # upper triangle + mirror
    finally:
        engine.set_wide_entries(False)
    assert np.array_equal(out["W"], ref["W"])
    assert np.array_equal(out["C"], ref["C"])
    assert np.array_equal(out["occ"], ref["occ"])
    for key in ("W", "occ", "adj_bits", "max_bits", "degree"):
        assert np.array_equal(lean[key], out[key]), key


def test_full_size_workload_against_the_c_oracle(engine):
    """BASELINE's 10 000-taxon x 1 000-tree workload, top-level recursion node: the whole W (10^8 entries), the
    occurrences and the adjacency against the C oracle, plus the size-independent properties (symmetry, degree =
    row sums, determinism of a second build)."""
    import bench

    arrays = bench.make_workload("c4")
    n = len(arrays["names"])
    roots, child_ptr, child_idx, tip_taxon, own = bench.oracle_children_csr(arrays)
    W, C, occ = scs_oracle.pcg_dense_c_arrays(n, roots, child_ptr, child_idx, tip_taxon, own, arrays["weights"],
                                              arrays["weighting"])  # fmt: skip
    forest = Forest.from_arrays(arrays["node_offsets"], arrays["parent"], arrays["length"], arrays["support"],
                                arrays["taxon"], arrays["weights"], arrays["names"])  # fmt: skip
    try:
        taxa, part, stats = engine.forest_split(forest, arrays["weighting"], seed=0)
        got = engine.last_node_buffers()
        assert np.array_equal(taxa, np.arange(n))
        assert np.array_equal(got["W"], W)
        assert np.array_equal(got["occ"], occ)
        adjacency = unpack_bits(got["adj_bits"], n)
        assert np.array_equal(adjacency, C > 0)
        del C, adjacency
        assert np.array_equal(got["W"], got["W"].T)
        assert np.array_equal(got["degree"], W.sum(axis=1))  # depth weighting, unit weights: integers, any order
        from scipy.sparse import csr_matrix
        from scipy.sparse.csgraph import connected_components

        # depth >= 1 wherever an edge exists; scipy numbers components by their smallest vertex, like the library
        count, label = connected_components(csr_matrix(W > 0), directed=False)
        assert stats.n_components == count
        if count > 1:
            assert np.array_equal(part, label)
        engine.forest_split(forest, arrays["weighting"], seed=0)
        again = engine.last_node_buffers()
        assert np.array_equal(again["W"], got["W"])
        assert np.array_equal(again["adj_bits"], got["adj_bits"])
    finally:
        forest.close()


def test_more_than_65535_source_trees(engine):
    """The co-occurrence counts of the small-node path are 16 bits wide (csrc/small.cu); nodes covered by more source
    trees than that must be routed to the paths with 32-bit counts -- by the per-node entry point and by both
    recursion drivers -- instead of wrapping.  65 536 trees ((a,b),(c,d)) and 1 000 trees ((a,c),(b,d)): a wrapped
    count of 65 536 is 0 and would delete the edges a-b and c-d."""
    t1, t2 = 65536, 1000
    trees = t1 + t2
    parent = np.tile(np.array([-1, 0, 1, 1, 0, 4, 4], dtype=np.int32), trees)
    taxon = np.concatenate([np.tile(np.array([-1, -1, 0, 1, -1, 2, 3], dtype=np.int32), t1),
                            np.tile(np.array([-1, -1, 0, 2, -1, 1, 3], dtype=np.int32), t2)])  # fmt: skip
    offsets = np.arange(trees + 1, dtype=np.int64) * 7
    nan = np.full(7 * trees, np.nan)
    weights = np.ones(trees)
    names = ["a", "b", "c", "d"]

    def forest():
        return Forest.from_arrays(offsets, parent, nan, nan, taxon, weights, names)

    taxa, part, stats = engine.forest_split(forest(), "one", seed=3)
    got = engine.last_node_buffers()
    want = np.array([[0, t1, t2, 0], [t1, 0, 0, t2], [t2, 0, 0, t1], [0, t2, t1, 0]], dtype=np.float64)
    assert np.array_equal(got["W"], want)
    assert np.array_equal(got["occ"], np.full(4, trees, dtype=np.int32))
    assert stats.n_components == 1 and stats.contracted_size == 4  # no pair is together in every tree
    assert part[0] == part[1] and part[2] == part[3] and part[0] != part[2]
    for device_forest in (True, False):
        engine.set_device_forest(device_forest)
        try:
            built = engine.supertree_build(forest(), "one", record=True)
        finally:
            engine.set_device_forest(True)
        top = built["records"][0]
        assert top[2].n_components == 1 and top[2].contracted_size == 4
        assert top[1][0] == top[1][1] and top[1][2] == top[1][3] and top[1][0] != top[1][2]
        assert sorted(built["taxon"][built["taxon"] >= 0]) == [0, 1, 2, 3]
