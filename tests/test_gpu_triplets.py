"""GPU: ``triplet_fit`` (csrc/triplets.cu) against the brute-force oracle (oracle/triplet_oracle.py): every count
exactly, ``weighted_fit`` to 1e-12 relative, on built supertrees, model trees, random trees, the untidy golden cases
(the caterpillar case has leaf tours more than 1 024 levels deep), supertrees and sources with taxa the other lacks,
one tree, trees sharing fewer than three taxa, skipped entries and the 10 000-taxon workload; determinism; agreement
with the Robinson-Foulds distance of ``clade_support``; the ``scs --triplets-out`` command."""

from __future__ import annotations

from math import comb

import numpy as np
import pytest

from helpers import CASES, load_case, load_ctrace, parse
from oracle import triplet_oracle
from spectralclustersupertree_b200 import clade_support, construct_supertree, triplet_fit
from spectralclustersupertree_b200.synthetic import make_problem
from spectralclustersupertree_b200.tree import NotCompleted, PhyloNode, make_tree

pytestmark = pytest.mark.gpu

INTS = ("shared", "resolved_source", "resolved_supertree", "agree", "contradict")


def check(engine, supertree, trees, weights=None):
    got = triplet_fit(supertree, trees, weights, engine=engine)
    want = triplet_oracle.triplet_fit(supertree, trees, weights)
    for key in INTS:
        assert np.array_equal(getattr(got, key), np.asarray(want[key])), key
    assert np.array_equal(got.unresolved, got.resolved_source - got.agree - got.contradict)
    np.testing.assert_allclose(got.weighted_fit, want["weighted_fit"], rtol=1e-12, atol=0, equal_nan=True)
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
    keep = slice(None) if n <= 500 else slice(0, 25)  # the oracle is cubic in the shared taxa
    got = check(engine, supertree, problem.phylonodes()[keep], problem.weights[keep])
    assert got.agree.sum() > 0


def test_model_tree_and_a_random_tree(engine):
    problem = make_problem(500, 50, "one", 2000)
    model = problem.model.to_phylonode()
    got = check(engine, model, problem.phylonodes())
    assert got.weighted_fit > 0.9
    rand = random_tree(sorted(model.get_tip_names()), seed=7)
    got = check(engine, rand, problem.phylonodes())
    assert got.contradict.sum() > got.agree.sum()


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


def test_one_tree_and_trees_sharing_fewer_than_three_taxa(engine):
    supertree = make_tree("(((a,b),c),(d,(e,f)));")
    check(engine, supertree, [make_tree("((a,c),(b,(d,e)));")])
    sources = [make_tree("(a,(x,y));"), make_tree("(x,y);"), make_tree("a;"), make_tree("((a,f),(x,e));"),
               make_tree("(q,r,s);"), make_tree("((a,b),(c,y));")]  # fmt: skip
    got = check(engine, supertree, sources, [1.0, 2.0, 3.0, 4.0, 5.0, 6.0])
    assert got.shared.tolist() == [1, 0, 1, 3, 0, 3]
    assert got.resolved_source.tolist()[:5] == [0, 0, 0, 1, 0]


def test_not_completed_entries_are_skipped(engine):
    supertree = make_tree("((a,b),(c,d));")
    trees = [make_tree("((a,b),(c,d));"), NotCompleted("ERROR", "x", "failed"), make_tree("((a,c),(b,d));")]
    got = triplet_fit(supertree, trees, [1.0, 100.0, 3.0], engine=engine)
    assert got.agree.tolist() == [4, -1, 0] and got.contradict.tolist() == [0, -1, 4]
    assert got.unresolved.tolist() == [0, -1, 0]
    assert got.fit[0] == 1.0 and np.isnan(got.fit[1]) and got.fit[2] == 0.0
    assert got.weighted_fit == 4.0 / 16.0
    with pytest.raises(ValueError, match="must match"):
        triplet_fit(supertree, trees, [1.0], engine=engine)


def test_c4_full_size_and_determinism(engine):
    problem = make_problem(10000, 1000, "depth", 4000)
    trees = problem.phylonodes()
    supertree = construct_supertree(trees, None, "depth", engine=engine)
    got = triplet_fit(supertree, trees, engine=engine)
    again = triplet_fit(supertree, trees, engine=engine)
    for key in (*INTS, "unresolved", "fit"):
        assert getattr(got, key).tobytes() == getattr(again, key).tobytes(), key
    assert got.weighted_fit == again.weighted_fit
    smallest = np.argsort(got.shared, kind="stable")[:4]
    check(engine, supertree, [trees[t] for t in smallest])
    bound = np.array([comb(int(k), 3) for k in got.shared], dtype=np.int64)
    assert (bound >= got.resolved_source).all() and (bound >= got.resolved_supertree).all()
    assert (got.resolved_source >= got.agree + got.contradict).all()
    assert (got.resolved_supertree >= got.agree + got.contradict).all()
    rf = clade_support(supertree, trees, engine=engine).rf
    same = (got.agree == got.resolved_source) & (got.agree == got.resolved_supertree)
    assert np.array_equal(rf == 0, same)


def test_cli_triplets_out(engine, tmp_path):
    from click.testing import CliRunner

    from spectralclustersupertree_b200.cli import scs

    problem = make_problem(300, 40, "branch", 21)
    src = tmp_path / "trees.nwk"
    src.write_text("\n".join(problem.newick_lines()) + "\n")
    plain, main, tsv = tmp_path / "plain.nwk", tmp_path / "main.nwk", tmp_path / "fit.tsv"
    labelled = tmp_path / "support.nwk"
    runner = CliRunner()
    assert runner.invoke(scs, ["-i", str(src), "-o", str(plain)]).exit_code == 0
    result = runner.invoke(scs, ["-i", str(src), "-o", str(main), "--triplets-out", str(tsv)])
    assert result.exit_code == 0, result.output
    assert main.read_bytes() == plain.read_bytes()
    supertree = make_tree(plain.read_text().strip())
    got = triplet_fit(supertree, parse(problem.newick_lines()), engine=engine)
    assert tsv.read_text() == got.tsv()
    rows = [line.split("\t") for line in tsv.read_text().splitlines()]
    assert rows[0] == ["tree", "shared", "resolved_source", "resolved_supertree", "agree", "contradict"]
    assert len(rows) == 1 + len(problem.newick_lines())
    result = runner.invoke(scs, ["-i", str(src), "-o", str(main), "--triplets-out", str(tsv), "--support-out",
                                 str(labelled)])  # fmt: skip
    assert result.exit_code == 0, result.output
    assert main.read_bytes() == plain.read_bytes()
    assert tsv.read_text() == got.tsv()
    assert labelled.read_text().strip()
