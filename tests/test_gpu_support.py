"""GPU: ``clade_support`` (csrc/support.cu) against the set-based oracle (oracle/support_oracle.py): integer outputs
exactly, weighted sums to 1e-12 relative, on built supertrees, model trees, random trees, the untidy golden cases
(the caterpillar case has leaf tours more than 1 024 levels deep), supertrees and sources with taxa the other lacks,
one tree, trees sharing fewer than two taxa, and the 10 000-taxon workload; determinism; the ``scs --support-out``
command."""

from __future__ import annotations

import numpy as np
import pytest

from helpers import CASES, load_case, load_ctrace, parse
from oracle import support_oracle
from spectralclustersupertree_b200 import clade_support, construct_supertree
from spectralclustersupertree_b200.engine import Forest
from spectralclustersupertree_b200.synthetic import make_problem
from spectralclustersupertree_b200.tree import NotCompleted, PhyloNode, make_tree

pytestmark = pytest.mark.gpu

INTS = ("support", "conflict", "permitted", "irrelevant", "rf", "shared", "source_clusters", "supertree_clusters")
FLOATS = ("weighted_support", "weighted_conflict", "weighted_permitted")


def check(engine, supertree, trees, weights=None):
    got = clade_support(supertree, trees, weights, engine=engine)
    want = support_oracle.clade_support(supertree, trees, weights)
    for key in INTS:
        assert np.array_equal(getattr(got, key), np.asarray(want[key])), key
    for key in FLOATS:
        np.testing.assert_allclose(getattr(got, key), np.asarray(want[key]), rtol=1e-12, atol=0, err_msg=key)
    np.testing.assert_allclose(got.v, np.asarray(want["v"]), rtol=1e-12, atol=1e-15, equal_nan=True)
    return got


def random_tree(names, seed: int) -> PhyloNode:
    """A random rooted binary tree on ``names`` (random joins)."""
    rng = np.random.RandomState(seed)
    nodes = [PhyloNode(name) for name in names]
    while len(nodes) > 1:
        i, j = sorted(rng.choice(len(nodes), size=2, replace=False))
        b, a = nodes.pop(j), nodes.pop(i)
        nodes.append(PhyloNode("", [a, b]))
    return nodes[0]


@pytest.mark.parametrize("case", sorted(CASES))
def test_golden_fixtures(engine, case):
    data = load_case(case)
    trees = parse(data["lines"])
    supertree = construct_supertree(trees, data["weights"], data["weighting"], engine=engine)
    check(engine, supertree, parse(data["lines"]), data["weights"])


@pytest.mark.parametrize("weighting", ["one", "branch", "depth", "bootstrap"])
@pytest.mark.parametrize("shape", [(100, 30, 1000), (500, 50, 2000), (1000, 100, 3000)])
def test_synthetic_problems(engine, shape, weighting):
    n, t, seed = shape
    problem = make_problem(n, t, weighting, seed, tree_weights=True)
    trees = problem.phylonodes()
    supertree = construct_supertree(trees, problem.weights, weighting, engine=engine)
    got = check(engine, supertree, problem.phylonodes(), problem.weights)
    assert (got.support > 0).any()


def test_model_tree_and_a_random_tree(engine):
    problem = make_problem(500, 50, "one", 2000)
    model = problem.model.to_phylonode()
    got = check(engine, model, problem.phylonodes())
    assert got.support.sum() > got.conflict.sum()
    rand = random_tree(sorted(model.get_tip_names()), seed=7)
    got = check(engine, rand, problem.phylonodes())
    assert got.conflict.sum() > got.support.sum()


@pytest.mark.parametrize("case", ["branch", "bootstrap", "depth", "nocontract", "caterpillar"])
def test_untidy_golden_cases(engine, case):
    ctrace = load_ctrace(f"untidy_{case}")
    trees = parse(ctrace["lines"])
    supertree = make_tree(ctrace["supertree"])
    check(engine, supertree, trees, ctrace["weights"])
    # one of the source trees (unary chains, polytomies) as the supertree
    check(engine, trees[-1], trees, None)


def test_taxa_missing_on_either_side(engine):
    problem = make_problem(300, 40, "one", 11)
    trees = problem.phylonodes()
    supertree = construct_supertree(trees, None, "one", engine=engine)
    extra = make_tree(f"({supertree.get_newick()[:-1]},(zz1,zz2));")  # supertree taxa no source has
    check(engine, extra, problem.phylonodes())
    names = sorted(supertree.get_tip_names())
    dropped = set(names[::3])
    pruned = supertree.get_sub_tree([x for x in names if x not in dropped], as_rooted=True)
    check(engine, pruned, problem.phylonodes())  # sources with taxa the supertree lacks


def test_one_tree_and_trees_sharing_fewer_than_two_taxa(engine):
    supertree = make_tree("(((a,b),c),(d,(e,f)));")
    check(engine, supertree, [make_tree("((a,c),(b,(d,e)));")])
    sources = [make_tree("(a,(x,y));"), make_tree("(x,y);"), make_tree("a;"), make_tree("((a,f),(b,e));"),
               make_tree("(q,r,s);")]  # fmt: skip
    got = check(engine, supertree, sources, [1.0, 2.0, 3.0, 4.0, 5.0])
    assert got.rf.tolist()[:3] == [0, 0, 0]


def test_not_completed_entries_are_skipped(engine):
    supertree = make_tree("((a,b),(c,d));")
    trees = [make_tree("((a,b),(c,d));"), NotCompleted("ERROR", "x", "failed"), make_tree("((a,c),(b,d));")]
    got = clade_support(supertree, trees, engine=engine)
    assert got.rf.tolist() == [0, -1, 4]
    assert got.support.tolist() == [0, 1, 1] and got.conflict.tolist() == [0, 1, 1]
    assert got.irrelevant.tolist() == [2, 0, 0]
    assert [node.support for node in got.annotated().iter_nontips(include_self=True)] == [None, 0.0, 0.0]


def test_c4_full_size_and_determinism(engine):
    problem = make_problem(10000, 1000, "depth", 4000)
    trees = problem.phylonodes()
    supertree = construct_supertree(trees, None, "depth", engine=engine)
    check(engine, supertree, trees[:50])
    got = clade_support(supertree, trees, engine=engine)
    again = clade_support(supertree, trees, engine=engine)
    for key in (*INTS, *FLOATS, "v"):
        assert getattr(got, key).tobytes() == getattr(again, key).tobytes(), key
    s_tips = set(supertree.get_tip_names())
    for t, tree in enumerate(trees):
        X = s_tips.intersection(tree.get_tip_names())
        a = {c for c in supertree.get_sub_tree(X, ignore_missing=True, as_rooted=True).clade_sets() if len(c) < len(X)}
        b = {c for c in tree.get_sub_tree(X, ignore_missing=True, as_rooted=True).clade_sets() if len(c) < len(X)}
        assert got.rf[t] == len(a ^ b), t


def test_cli_support_out(engine, tmp_path):
    from click.testing import CliRunner

    from spectralclustersupertree_b200.cli import scs

    problem = make_problem(300, 40, "branch", 21)
    src = tmp_path / "trees.nwk"
    src.write_text("\n".join(problem.newick_lines()) + "\n")
    plain, with_support, labelled = tmp_path / "plain.nwk", tmp_path / "main.nwk", tmp_path / "support.nwk"
    runner = CliRunner()
    assert runner.invoke(scs, ["-i", str(src), "-o", str(plain)]).exit_code == 0
    result = runner.invoke(scs, ["-i", str(src), "-o", str(with_support), "--support-out", str(labelled)])
    assert result.exit_code == 0, result.output
    assert with_support.read_bytes() == plain.read_bytes()
    supertree = make_tree(plain.read_text().strip())
    got = clade_support(supertree, parse(problem.newick_lines()), engine=engine)
    annotated = make_tree(labelled.read_text().strip())
    labels = [node.support for node in annotated.iter_nontips(include_self=True)]
    expected = [None if np.isnan(v) else round(float(v), 3) for v in got.v]
    expected[0] = None  # the root carries no label
    assert labels == expected
    assert annotated.clade_sets() == supertree.clade_sets()
