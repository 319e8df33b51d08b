"""GPU: ``taxon_triplet_fit`` (csrc/triplets.cu) against the per-taxon oracle (oracle/taxon_triplet_oracle.py): every count
exactly and the three weighted sums bit for bit, on built supertrees, the untidy golden cases (the caterpillar case
included), source trees with unary chains or polytomies as the supertree, taxa missing on either side, one tree, trees
sharing fewer than three taxa and skipped entries; a planted rogue taxon; the 10 000-taxon workload against
``triplet_fit``; the ``scs --taxon-triplets-out`` command."""

from __future__ import annotations

import re
from math import comb

import numpy as np
import pytest

from helpers import CASES, load_case, load_ctrace, parse
from oracle import taxon_triplet_oracle
from spectralclustersupertree_b200 import construct_supertree, taxon_triplet_fit, triplet_fit
from spectralclustersupertree_b200.synthetic import make_problem
from spectralclustersupertree_b200.tree import NotCompleted, make_tree

pytestmark = pytest.mark.gpu

COUNTS = ("trees", "triplets", "resolved_source", "resolved_supertree", "agree", "contradict")
SUMS = ("weighted_resolved_source", "weighted_agree", "weighted_contradict")


def check(engine, supertree, trees, weights=None):
    got = taxon_triplet_fit(supertree, trees, weights, engine=engine)
    want = taxon_triplet_oracle.taxon_fit(supertree, trees, weights)
    assert got.names == want["names"]
    for key in COUNTS:
        assert np.array_equal(getattr(got, key), want[key]), key
    for f, key in enumerate(SUMS):
        assert getattr(got, key).tobytes() == np.ascontiguousarray(want["weighted"][:, f]).tobytes(), key
    assert got.weighted_fit.tobytes() == want["weighted_fit"].tobytes()
    assert np.array_equal(got.unresolved, got.resolved_source - got.agree - got.contradict)
    return got


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
    keep = slice(None) if n <= 100 else slice(0, 12)  # the oracle is cubic in the shared taxa
    got = check(engine, supertree, problem.phylonodes()[keep], problem.weights[keep])
    assert got.agree.sum() > 0


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
    trees = problem.phylonodes()[:15]
    supertree = construct_supertree(problem.phylonodes(), None, "one", engine=engine)
    extra = make_tree(f"({supertree.get_newick()[:-1]},(zz1,zz2));")  # supertree taxa no source has
    got = check(engine, extra, trees)
    assert got.trees[got.names.index("zz1")] == 0
    names = sorted(supertree.get_tip_names())
    dropped = set(names[::3])
    pruned = supertree.get_sub_tree([x for x in names if x not in dropped], as_rooted=True)
    check(engine, pruned, trees)  # sources with taxa the supertree lacks


def test_one_tree_and_trees_sharing_fewer_than_three_taxa(engine):
    supertree = make_tree("(((a,b),c),(d,(e,f)));")
    check(engine, supertree, [make_tree("((a,c),(b,(d,e)));")])
    sources = [make_tree("(a,(x,y));"), make_tree("(x,y);"), make_tree("a;"), make_tree("((a,f),(x,e));"),
               make_tree("(q,r,s);"), make_tree("((a,b),(c,y));")]  # fmt: skip
    got = check(engine, supertree, sources, [1.0, 2.0, 3.0, 4.0, 5.0, 6.0])
    assert got.trees.tolist() == [2, 1, 1, 0, 1, 1]  # a b c d e f
    got = check(engine, make_tree("((a,b),(c,d));"), [make_tree("((a,c),(b,d));")])
    assert got.agree.tolist() == [0, 0, 0, 0] and got.contradict.tolist() == [3, 3, 3, 3]
    got = check(engine, make_tree("(((a,b),c),d);"), [make_tree("(((a,b),d),c);")])
    assert got.agree.tolist() == [2, 2, 1, 1] and got.contradict.tolist() == [1, 1, 2, 2]


def test_not_completed_entries_are_skipped(engine):
    supertree = make_tree("((a,b),(c,d));")
    trees = [make_tree("((a,b),(c,d));"), NotCompleted("ERROR", "x", "failed"), make_tree("((a,c),(b,d));")]
    got = taxon_triplet_fit(supertree, trees, [1.0, 100.0, 3.0], engine=engine)
    want = check(engine, supertree, [trees[0], trees[2]], [1.0, 3.0])
    for key in (*COUNTS, *SUMS):
        assert getattr(got, key).tobytes() == getattr(want, key).tobytes(), key
    assert got.trees.tolist() == [2, 2, 2, 2] and got.weighted_fit.tolist() == [0.25] * 4
    every = taxon_triplet_fit(supertree, [trees[1]], engine=engine)
    assert every.trees.tolist() == [0, 0, 0, 0] and np.isnan(every.fit).all()
    with pytest.raises(ValueError, match="must match"):
        taxon_triplet_fit(supertree, trees, [1.0], engine=engine)


def regraft(tree, taxon: str, onto: str):
    """``tree`` with ``taxon`` pruned and regrafted as the sibling of tip ``onto``."""
    rest = [x for x in tree.get_tip_names() if x != taxon]
    text = tree.get_sub_tree(rest, as_rooted=True).get_newick()
    text, count = re.subn(rf"(?<=[(,]){re.escape(onto)}(?=[,)])", f"({onto},{taxon})", text)
    assert count == 1
    return make_tree(text)


def test_planted_rogue(engine):
    problem = make_problem(100, 30, "one", 5)
    model = problem.model.to_phylonode()
    trees = problem.phylonodes()
    tips = [node.name for node in model.iter_tips()]
    held = {name: sum(name in tree.get_tip_names() for tree in trees) for name in tips}
    rogue = max(tips, key=lambda name: held[name])
    onto = tips[-1] if tips.index(rogue) < len(tips) // 2 else tips[0]  # far away in the model tree
    planted = regraft(model, rogue, onto)
    before = check(engine, model, trees)
    after = check(engine, planted, trees)
    r = after.names.index(rogue)
    often = np.flatnonzero(after.trees >= 5)
    assert r in often and after.fit[r] == after.fit[often].min()
    assert np.sum(after.fit[often] == after.fit[r]) == 1
    assert after.contradict[r] > before.contradict[r]
    # the other taxa change only through the triplets that hold the rogue too
    with_rogue = np.zeros(len(after.names), dtype=np.int64)
    index = {name: i for i, name in enumerate(after.names)}
    for tree in trees:
        shared = set(tree.get_tip_names()) & set(tips)
        if rogue in shared and len(shared) >= 3:
            for name in shared - {rogue}:
                with_rogue[index[name]] += len(shared) - 2
    others = np.arange(len(after.names)) != r
    assert np.array_equal(after.resolved_source, before.resolved_source)
    for key in ("resolved_supertree", "agree", "contradict"):
        change = np.abs(getattr(after, key) - getattr(before, key))
        assert (change[others] <= with_rogue[others]).all(), key
        assert (change[others][with_rogue[others] == 0] == 0).all(), key


def test_c4_full_size_and_determinism(engine):
    problem = make_problem(10000, 1000, "depth", 4000)
    trees = problem.phylonodes()
    supertree = construct_supertree(trees, None, "depth", engine=engine)
    got = taxon_triplet_fit(supertree, trees, engine=engine)
    again = taxon_triplet_fit(supertree, trees, engine=engine)
    for key in (*COUNTS, *SUMS, "fit", "weighted_fit"):
        assert getattr(got, key).tobytes() == getattr(again, key).tobytes(), key
    per_tree = triplet_fit(supertree, trees, engine=engine)
    for key in ("resolved_source", "resolved_supertree", "agree", "contradict"):
        assert getattr(got, key).sum() == 3 * getattr(per_tree, key).sum(), key
    assert got.triplets.sum() == 3 * sum(comb(int(k), 3) for k in per_tree.shared)
    assert got.trees.sum() == per_tree.shared[per_tree.shared >= 3].sum()


def test_cli_taxon_triplets_out(engine, tmp_path):
    from click.testing import CliRunner

    from spectralclustersupertree_b200.cli import scs

    problem = make_problem(300, 40, "branch", 21)
    src = tmp_path / "trees.nwk"
    src.write_text("\n".join(problem.newick_lines()) + "\n")
    plain, main, tsv, fit_tsv = (tmp_path / name for name in ("plain.nwk", "main.nwk", "taxa.tsv", "fit.tsv"))
    labelled = tmp_path / "support.nwk"
    runner = CliRunner()
    assert runner.invoke(scs, ["-i", str(src), "-o", str(plain)]).exit_code == 0
    result = runner.invoke(scs, ["-i", str(src), "-o", str(main), "--taxon-triplets-out", str(tsv)])
    assert result.exit_code == 0, result.output
    assert main.read_bytes() == plain.read_bytes()
    supertree = make_tree(plain.read_text().strip())
    got = taxon_triplet_fit(supertree, parse(problem.newick_lines()), engine=engine)
    assert tsv.read_text() == got.tsv()
    rows = [line.split("\t") for line in tsv.read_text().splitlines()]
    assert rows[0] == ["taxon", "trees", "triplets", "resolved_source", "resolved_supertree", "agree", "contradict"]
    assert [row[0] for row in rows[1:]] == sorted(supertree.get_tip_names())
    result = runner.invoke(scs, ["-i", str(src), "-o", str(main), "--taxon-triplets-out", str(tsv), "--triplets-out",
                                 str(fit_tsv), "--support-out", str(labelled)])  # fmt: skip
    assert result.exit_code == 0, result.output
    assert main.read_bytes() == plain.read_bytes()
    assert tsv.read_text() == got.tsv()
    assert fit_tsv.read_text() == triplet_fit(supertree, parse(problem.newick_lines()), engine=engine).tsv()
    assert labelled.read_text().strip()
