"""GPU: ``source_tree_distances`` (csrc/pairwise.cu) against the set-based oracle (oracle/pairwise_oracle.py), every
entry of the three counted matrices exactly, on the golden fixtures, the synthetic C1-C3 problems, the untidy golden
cases with the caterpillar, random trees with taxa missing on either side, one and two trees, trees sharing fewer
than three taxa and skipped entries; the 1 000-tree workload against a numpy taxon product and ``clade_support`` with
source trees as the supertree, for symmetry and for determinism; caterpillars 20 000 levels deep; a planted outlier
tree; the ``scs --source-rf-out`` command."""

from __future__ import annotations

import numpy as np
import pytest

from helpers import CASES, load_case, load_ctrace, parse
from oracle import pairwise_oracle
from spectralclustersupertree_b200 import clade_support, source_tree_distances
from spectralclustersupertree_b200.engine import Forest
from spectralclustersupertree_b200.synthetic import make_problem
from spectralclustersupertree_b200.tree import NotCompleted, make_tree
from test_pairwise_cpu import random_forest

pytestmark = pytest.mark.gpu

COUNTS = ("shared_taxa", "clusters", "common", "rf")


def check(engine, trees):
    got = source_tree_distances(trees, engine=engine)
    kept = [i for i, tree in enumerate(trees) if not isinstance(tree, NotCompleted)]
    want = pairwise_oracle.pairwise_rf([trees[i] for i in kept])
    for key in COUNTS:
        assert np.array_equal(getattr(got, key)[np.ix_(kept, kept)], np.array(want[key]).reshape(len(kept), -1)), key
    return got


@pytest.mark.parametrize("case", sorted(CASES))
def test_golden_fixtures(engine, case):
    check(engine, parse(load_case(case)["lines"]))


@pytest.mark.parametrize("shape", [(100, 30, "depth", 1000), (500, 50, "branch", 2000), (1000, 100, "branch", 3000)])
def test_synthetic_problems(engine, shape):
    n, t, weighting, seed = shape
    got = check(engine, make_problem(n, t, weighting, seed, tree_weights=True).phylonodes())
    assert (np.triu(got.shared_taxa, 1) >= 3).sum() > 0 and got.common.sum() > 0


@pytest.mark.parametrize("case", ["branch", "bootstrap", "depth", "nocontract", "caterpillar"])
def test_untidy_golden_cases(engine, case):
    check(engine, parse(load_ctrace(f"untidy_{case}")["lines"]))


@pytest.mark.parametrize("seed", range(3))
def test_random_trees_with_taxa_missing_on_either_side(engine, seed):
    check(engine, random_forest(seed, 40, pool=30))


def test_one_tree_and_two_trees(engine):
    got = check(engine, [make_tree("((a,b),((c,d),e));")])
    assert got.shared_taxa.tolist() == [[5]] and got.clusters.tolist() == [[3]] and got.rf.tolist() == [[0]]
    got = check(engine, [make_tree("((a,b),(c,d));"), make_tree("((a,c),(b,d));")])
    assert got.rf.tolist() == [[0, 4], [4, 0]] and got.normalized_rf[0, 1] == 1.0


def test_trees_sharing_fewer_than_three_taxa(engine):
    trees = [make_tree(s) for s in ("((a,b),(c,d));", "((a,b),(x,y));", "a;", "(x,y);", "((q,r),s);", "(a,(c,d));",
                                    "(((a,b)),c);")]  # fmt: skip
    got = check(engine, trees)
    assert got.shared_taxa[0].tolist() == [4, 2, 1, 0, 0, 3, 3]
    assert np.isnan(got.normalized_rf[0, 1]) and got.rf[0, 1] == 0
    assert got.comparable.tolist() == [2, 0, 0, 0, 0, 1, 1]


def test_not_completed_entries_are_skipped(engine):
    trees = [make_tree("((a,b),(c,d));"), NotCompleted("ERROR", "x", "failed"), make_tree("((a,c),(b,d));")]
    got = check(engine, trees)
    assert got.rf.tolist() == [[0, -1, 4], [-1, -1, -1], [4, -1, 0]]
    assert got.comparable.tolist() == [1, -1, 1]
    assert np.isnan(got.normalized_rf[1]).all() and np.isnan(got.mean_normalized_rf[1])


def test_c4_full_size_against_clade_support(engine):
    problem = make_problem(10000, 1000, "depth", 4000)
    trees = problem.phylonodes()
    got = source_tree_distances(trees, engine=engine)
    again = source_tree_distances(trees, engine=engine)
    for key in (*COUNTS, "normalized_rf", "comparable", "mean_normalized_rf"):
        assert getattr(got, key).tobytes() == getattr(again, key).tobytes(), key
    names = sorted(set().union(*(tree.get_tip_names() for tree in trees)))
    index = {name: x for x, name in enumerate(names)}
    B = np.zeros((len(trees), len(names)), dtype=np.int64)
    for t, tree in enumerate(trees):
        B[t, [index[name] for name in tree.get_tip_names()]] = 1
    assert np.array_equal(got.shared_taxa, B @ B.T)
    assert np.array_equal(got.shared_taxa, got.shared_taxa.T) and np.array_equal(got.common, got.common.T)
    assert np.array_equal(np.diag(got.clusters), np.diag(got.common)) and (np.diag(got.rf) == 0).all()
    assert (got.rf >= 0).all() and (got.common <= np.minimum(got.clusters, got.clusters.T)).all()
    size = B.sum(axis=1)
    rows = sorted({0, int(np.argmax(size)), int(np.argmin(size)), 17, 500, 999})
    for i in rows:
        support = clade_support(trees[i], trees, engine=engine)
        assert np.array_equal(support.rf, got.rf[i])
        assert np.array_equal(support.shared, got.common[i])
        assert np.array_equal(support.source_clusters, got.clusters[:, i])
        assert np.array_equal(support.supertree_clusters, got.clusters[i])
    assert got.comparable.max() > 100


def caterpillar_arrays(k: int, reverse: bool) -> tuple[np.ndarray, np.ndarray]:
    """Flat pre-order caterpillar ((((x0, x1), x2), ...), x{k-1}) on taxon ids 0..k-1 (k-1 - x with ``reverse``): its
    clusters are the prefixes {x0..xm}, 1 <= m <= k - 2, and its deepest tips lie k - 1 levels down."""
    parent = np.full(2 * k - 1, -1, dtype=np.int32)
    taxon = np.full(2 * k - 1, -1, dtype=np.int32)
    for i in range(k - 1):  # internal node 2i holds tip k-1-i and internal node 2i + 2
        parent[2 * i + 1] = 2 * i
        taxon[2 * i + 1] = k - 1 - i
        parent[2 * i + 2] = 2 * i
    taxon[2 * k - 2] = 0
    if reverse:
        taxon[taxon >= 0] = k - 1 - taxon[taxon >= 0]
    return parent, taxon


def test_deep_caterpillars(engine):
    k = 20000
    names = [f"x{i:05d}" for i in range(k)]
    ahead, behind = caterpillar_arrays(k, False), caterpillar_arrays(k, True)
    for second, common in ((ahead, k - 2), (behind, 0)):
        forest = Forest.from_arrays([0, 2 * k - 1, 4 * k - 2], np.concatenate([ahead[0], second[0]]), None, None,
                                    np.concatenate([ahead[1], second[1]]), [1.0, 1.0], names, copy=True)  # fmt: skip
        shared, clusters, both = engine.forest_pairwise_rf(forest)
        assert shared.tolist() == [[k, k], [k, k]]
        assert clusters.tolist() == [[k - 2, k - 2], [k - 2, k - 2]]
        assert both[0, 1] == both[1, 0] == common
        assert both[0, 0] == both[1, 1] == k - 2
        assert clusters[0, 1] + clusters[1, 0] - 2 * both[0, 1] == 2 * (k - 2 - common)


def test_planted_outlier(engine):
    problem = make_problem(1000, 100, "branch", 3000, tree_weights=True)
    trees = problem.phylonodes()
    before = source_tree_distances(trees, engine=engine)
    outlier = int(np.argmax(before.comparable))
    permuted = problem.phylonodes()[outlier]
    tips = list(permuted.iter_tips())
    labels = [tip.name for tip in tips]
    for tip, name in zip(tips, np.random.RandomState(9).permutation(labels).tolist(), strict=True):
        tip.name = name
    trees[outlier] = permuted
    after = check(engine, trees)
    assert after.mean_normalized_rf[outlier] > before.mean_normalized_rf[outlier]
    ranked = np.flatnonzero(after.comparable >= 10)
    assert outlier in ranked
    assert ranked[np.argmax(after.mean_normalized_rf[ranked])] == outlier


def test_cli_source_rf_out(engine, tmp_path):
    from click.testing import CliRunner

    from spectralclustersupertree_b200.cli import scs

    problem = make_problem(300, 40, "branch", 21)
    src = tmp_path / "trees.nwk"
    src.write_text("\n".join(problem.newick_lines()) + "\n")
    plain, main, tsv, fit = tmp_path / "plain.nwk", tmp_path / "main.nwk", tmp_path / "rf.tsv", tmp_path / "mrp.tsv"
    runner = CliRunner()
    assert runner.invoke(scs, ["-i", str(src), "-o", str(plain)]).exit_code == 0
    result = runner.invoke(scs, ["-i", str(src), "-o", str(main), "--source-rf-out", str(tsv)])
    assert result.exit_code == 0, result.output
    assert main.read_bytes() == plain.read_bytes()
    got = source_tree_distances(parse(problem.newick_lines()), engine=engine)
    assert tsv.read_text() == got.tsv()
    rows = [line.split("\t") for line in tsv.read_text().splitlines()]
    assert rows[0] == ["tree_a", "tree_b", "shared", "clusters_a", "clusters_b", "common", "rf"]
    pairs = [(int(r[0]), int(r[1])) for r in rows[1:]]
    assert pairs == sorted(pairs) and all(a < b for a, b in pairs)
    assert pairs == [(a, b) for a, b in zip(*np.nonzero(np.triu(got.shared_taxa >= 3, 1)), strict=True)]
    assert all(int(r[2]) >= 3 for r in rows[1:])
    result = runner.invoke(scs, ["-i", str(src), "-o", str(main), "--source-rf-out", str(tsv), "--mrp-out", str(fit)])
    assert result.exit_code == 0, result.output
    assert main.read_bytes() == plain.read_bytes()
    assert tsv.read_text() == got.tsv() and fit.read_text().strip()
