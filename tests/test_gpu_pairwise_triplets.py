"""GPU: ``source_tree_triplet_distances`` (csrc/pairwise.cu, pw_triplets) against the oracle
(oracle/pairwise_triplet_oracle.py), every entry of the four counted matrices exactly, on the golden fixtures, the
synthetic C1-C3 problems, the untidy golden cases with the caterpillar, random trees with taxa missing on either
side, one and two trees, trees sharing fewer than three taxa and skipped entries; rows against ``triplet_fit`` with a
source tree as the supertree; the 1 000-tree workload for determinism and against ``source_tree_distances`` and
``triplet_fit``; caterpillars 20 000 levels deep, and one too deep; a planted outlier tree; the
``scs --source-triplets-out`` command."""

from __future__ import annotations

from math import comb

import numpy as np
import pytest

from helpers import CASES, load_case, load_ctrace, parse
from oracle import pairwise_triplet_oracle
from spectralclustersupertree_b200 import source_tree_distances, source_tree_triplet_distances, triplet_fit
from spectralclustersupertree_b200.engine import Forest, ScsError
from spectralclustersupertree_b200.synthetic import make_problem
from spectralclustersupertree_b200.tree import NotCompleted, make_tree
from test_gpu_pairwise import caterpillar_arrays
from test_pairwise_cpu import random_forest

pytestmark = pytest.mark.gpu

COUNTS = ("shared_taxa", "resolved", "agree", "contradict", "distance")
# the oracle is cubic in the shared taxa: on these inputs it compares the pairs of the first 12 trees
LARGE = {"c3_1000x100_branch_weighted", "supertriplets"}


def check(engine, trees, subset=None):
    """Every pair of ``trees`` (of ``subset`` of them, if given) against the oracle."""
    got = source_tree_triplet_distances(trees, engine=engine)
    kept = [i for i, tree in enumerate(trees) if not isinstance(tree, NotCompleted)]
    if subset is not None:
        kept = [i for i in kept if i in set(subset)]
    want = pairwise_triplet_oracle.pairwise_triplets([trees[i] for i in kept])
    for key in COUNTS:
        assert np.array_equal(getattr(got, key)[np.ix_(kept, kept)], np.array(want[key]).reshape(len(kept), -1)), key
    return got


def check_rows(engine, trees, got, rows):
    """Row i against ``triplet_fit`` with tree i as the supertree."""
    for i in rows:
        fit = triplet_fit(trees[i], trees, engine=engine)
        assert np.array_equal(fit.shared, got.shared_taxa[i]), i
        assert np.array_equal(fit.resolved_source, got.resolved[:, i]), i
        assert np.array_equal(fit.resolved_supertree, got.resolved[i]), i
        assert np.array_equal(fit.agree, got.agree[i]), i
        assert np.array_equal(fit.contradict, got.contradict[i]), i


@pytest.mark.parametrize("case", sorted(CASES))
def test_golden_fixtures(engine, case):
    trees = parse(load_case(case)["lines"])
    got = check(engine, trees, range(12) if case in LARGE else None)
    if case in LARGE:
        check_rows(engine, trees, got, sorted({0, 17, len(trees) - 1, int(np.argmax(np.diag(got.shared_taxa)))}))


@pytest.mark.parametrize("shape", [(100, 30, "depth", 1000), (500, 50, "branch", 2000), (1000, 100, "branch", 3000)])
def test_synthetic_problems(engine, shape):
    n, t, weighting, seed = shape
    trees = make_problem(n, t, weighting, seed, tree_weights=True).phylonodes()
    got = check(engine, trees, range(12) if n > 500 else None)
    assert (np.triu(got.shared_taxa, 1) >= 3).sum() > 0 and got.agree.sum() > 0 and got.contradict.sum() > 0


@pytest.mark.parametrize("case", ["branch", "bootstrap", "depth", "nocontract", "caterpillar"])
def test_untidy_golden_cases(engine, case):
    trees = parse(load_ctrace(f"untidy_{case}")["lines"])
    if case != "caterpillar":
        check(engine, trees)
        return
    # the caterpillars (tours over 700 levels deep) cost the oracle k^3 per pair: two of them with the small trees,
    # and every row with at least three tips against triplet_fit
    tips = [len(tree.get_tip_names()) for tree in trees]
    deep = sorted(range(len(trees)), key=lambda i: -tips[i])[:2]
    got = check(engine, trees, sorted(set(deep) | {i for i in range(len(trees)) if tips[i] < 100}))
    check_rows(engine, trees, got, [i for i in range(len(trees)) if tips[i] >= 3])


@pytest.mark.parametrize("seed", range(3))
def test_random_trees_with_taxa_missing_on_either_side(engine, seed):
    got = check(engine, random_forest(seed, 40, pool=30))
    assert got.contradict.sum() > 0


def test_one_tree_and_two_trees(engine):
    got = check(engine, [make_tree("((a,b),((c,d),e));")])
    assert got.shared_taxa.tolist() == [[5]] and got.resolved.tolist() == [[comb(5, 3)]]
    assert got.distance.tolist() == [[0]]
    got = check(engine, [make_tree("((a,b),(c,d));"), make_tree("((a,c),(b,d));")])
    assert got.distance.tolist() == [[0, 4], [4, 0]] and got.contradict[0, 1] == 4
    assert got.normalized_distance[0, 1] == 1.0


def test_trees_sharing_fewer_than_three_taxa(engine):
    trees = [make_tree(s) for s in ("((a,b),(c,d));", "((a,b),(x,y));", "a;", "(x,y);", "((q,r),s);", "(a,(c,d));",
                                    "(((a,b)),c);")]  # fmt: skip
    got = check(engine, trees)
    assert got.shared_taxa[0].tolist() == [4, 2, 1, 0, 0, 3, 3]
    assert np.isnan(got.normalized_distance[0, 1]) and got.distance[0, 1] == 0
    assert got.comparable.tolist() == [2, 0, 0, 0, 0, 1, 1]


def test_not_completed_entries_are_skipped(engine):
    trees = [make_tree("((a,b),(c,d));"), NotCompleted("ERROR", "x", "failed"), make_tree("((a,c),(b,d));")]
    got = check(engine, trees)
    assert got.distance.tolist() == [[0, -1, 4], [-1, -1, -1], [4, -1, 0]]
    assert got.comparable.tolist() == [1, -1, 1]
    assert np.isnan(got.normalized_distance[1]).all() and np.isnan(got.mean_normalized_distance[1])


def test_c4_full_size(engine):
    trees = make_problem(10000, 1000, "depth", 4000).phylonodes()
    got = source_tree_triplet_distances(trees, engine=engine)
    again = source_tree_triplet_distances(trees, engine=engine)
    for key in (*COUNTS, "normalized_distance", "comparable", "mean_normalized_distance"):
        assert getattr(got, key).tobytes() == getattr(again, key).tobytes(), key
    assert np.array_equal(got.shared_taxa, source_tree_distances(trees, engine=engine).shared_taxa)
    assert np.array_equal(got.agree, got.agree.T) and np.array_equal(got.contradict, got.contradict.T)
    assert np.array_equal(np.diag(got.resolved), np.diag(got.agree)) and (np.diag(got.contradict) == 0).all()
    k = got.shared_taxa.astype(np.int64)
    assert (got.resolved <= k * (k - 1) * (k - 2) // 6).all()
    assert (np.minimum(got.resolved, got.resolved.T) >= got.agree + got.contradict).all()
    assert (got.distance >= 0).all() and got.contradict.sum() > 0
    size = np.diag(got.shared_taxa)
    check_rows(engine, trees, got, sorted({0, int(np.argmax(size)), int(np.argmin(size)), 17, 500, 999}))
    assert got.comparable.max() > 100


def caterpillar_forest(k: int, reverse: bool) -> Forest:
    """The caterpillar on k taxa and the same (or the reversed) caterpillar as a forest of two trees."""
    ahead, second = caterpillar_arrays(k, False), caterpillar_arrays(k, reverse)
    names = [f"x{i:05d}" for i in range(k)]
    return Forest.from_arrays([0, 2 * k - 1, 4 * k - 2], np.concatenate([ahead[0], second[0]]), None, None,
                              np.concatenate([ahead[1], second[1]]), [1.0, 1.0], names, copy=True)  # fmt: skip


def test_deep_caterpillars(engine):
    k = 20000
    full = comb(k, 3)
    assert full > 2**31
    shared, resolved, agree, contradict = engine.forest_pairwise_triplets(caterpillar_forest(k, False))
    assert shared.tolist() == [[k, k], [k, k]]
    assert resolved.tolist() == agree.tolist() == [[full, full], [full, full]]
    assert contradict.tolist() == [[0, 0], [0, 0]]
    shared, resolved, agree, contradict = engine.forest_pairwise_triplets(caterpillar_forest(k, True))
    assert resolved.tolist() == [[full, full], [full, full]]
    assert agree.tolist() == [[full, 0], [0, full]]
    assert contradict.tolist() == [[0, full], [full, 0]]


def test_caterpillar_beyond_the_fenwick_tree_is_refused(engine):
    forest = caterpillar_forest(40000, False)
    before = engine.launch_count
    with pytest.raises(ScsError, match="too deep"):
        engine.forest_pairwise_triplets(forest)
    assert engine.launch_count == before


def test_planted_outlier(engine):
    problem = make_problem(1000, 100, "branch", 3000, tree_weights=True)
    trees = problem.phylonodes()
    before = source_tree_triplet_distances(trees, engine=engine)
    outlier = int(np.argmax(before.comparable))
    permuted = problem.phylonodes()[outlier]
    tips = list(permuted.iter_tips())
    labels = [tip.name for tip in tips]
    for tip, name in zip(tips, np.random.RandomState(9).permutation(labels).tolist(), strict=True):
        tip.name = name
    trees[outlier] = permuted
    after = source_tree_triplet_distances(trees, engine=engine)
    assert after.mean_normalized_distance[outlier] > before.mean_normalized_distance[outlier]
    ranked = np.flatnonzero(after.comparable >= 10)
    assert outlier in ranked
    assert ranked[np.argmax(after.mean_normalized_distance[ranked])] == outlier


def test_cli_source_triplets_out(engine, tmp_path):
    from click.testing import CliRunner

    from spectralclustersupertree_b200.cli import scs

    problem = make_problem(300, 40, "branch", 21)
    src = tmp_path / "trees.nwk"
    src.write_text("\n".join(problem.newick_lines()) + "\n")
    plain, main, tsv, rf = tmp_path / "plain.nwk", tmp_path / "main.nwk", tmp_path / "triplets.tsv", tmp_path / "rf.tsv"
    runner = CliRunner()
    assert runner.invoke(scs, ["-i", str(src), "-o", str(plain)]).exit_code == 0
    result = runner.invoke(scs, ["-i", str(src), "-o", str(main), "--source-triplets-out", str(tsv)])
    assert result.exit_code == 0, result.output
    assert main.read_bytes() == plain.read_bytes()
    got = source_tree_triplet_distances(parse(problem.newick_lines()), engine=engine)
    assert tsv.read_text() == got.tsv()
    rows = [line.split("\t") for line in tsv.read_text().splitlines()]
    assert rows[0] == ["tree_a", "tree_b", "shared", "resolved_a", "resolved_b", "agree", "contradict", "distance"]
    pairs = [(int(r[0]), int(r[1])) for r in rows[1:]]
    assert pairs == [(a, b) for a, b in zip(*np.nonzero(np.triu(got.shared_taxa >= 3, 1)), strict=True)]
    assert all(int(r[2]) >= 3 for r in rows[1:])
    result = runner.invoke(scs, ["-i", str(src), "-o", str(main), "--source-triplets-out", str(tsv),
                                 "--source-rf-out", str(rf)])  # fmt: skip
    assert result.exit_code == 0, result.output
    assert main.read_bytes() == plain.read_bytes()
    assert tsv.read_text() == got.tsv()
    assert rf.read_text() == source_tree_distances(parse(problem.newick_lines()), engine=engine).tsv()
