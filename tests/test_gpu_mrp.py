"""GPU: ``mrp_score`` (csrc/triplets.cu) against the MRP oracle (oracle/mrp_oracle.py): every per-tree count exactly
and ``weighted_steps`` to 1e-12 relative, on the inputs of the triplet tests (built supertrees, model and random
trees, the untidy golden cases with the caterpillar, taxa missing on either side, one tree, trees sharing fewer than
three taxa, skipped entries); a source tree as the supertree; the 10 000-taxon workload against ``clade_support`` and
for determinism; a caterpillar supertree within and beyond the depth of the shared-memory stack; the ``scs --mrp-out``
command."""

from __future__ import annotations

import numpy as np
import pytest

from helpers import CASES, load_case, load_ctrace, parse
from oracle import mrp_oracle
from spectralclustersupertree_b200 import clade_support, construct_supertree, mrp_score
from spectralclustersupertree_b200.engine import Forest, ScsError
from spectralclustersupertree_b200.synthetic import make_problem
from spectralclustersupertree_b200.tree import NotCompleted, PhyloNode, make_tree

pytestmark = pytest.mark.gpu

INTS = ("shared", "characters", "steps", "exact")


def check(engine, supertree, trees, weights=None, route="s'"):
    """``route="s'"`` scores on the restricted supertree, which the CPU tests pin to the unrestricted one and is much
    faster in the oracle."""
    got = mrp_score(supertree, trees, weights, engine=engine)
    want = mrp_oracle.mrp_score(supertree, trees, weights, route=route)
    for key in INTS:
        assert np.array_equal(getattr(got, key), np.asarray(want[key])), key
    assert np.array_equal(got.extra, got.steps - got.characters)
    assert (got.steps >= got.characters).all()
    np.testing.assert_allclose(got.weighted_steps, want["weighted_steps"], rtol=1e-12, atol=0)
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
    assert got.exact.sum() > 0


def test_model_tree_and_a_random_tree(engine):
    problem = make_problem(500, 50, "one", 2000)
    model = problem.model.to_phylonode()
    got = check(engine, model, problem.phylonodes())
    assert got.total_ci > 0.9
    rand = random_tree(sorted(model.get_tip_names()), seed=7)
    got = check(engine, rand, problem.phylonodes())
    assert got.total_ci < 0.5


@pytest.mark.parametrize("case", ["branch", "bootstrap", "depth", "nocontract", "caterpillar"])
def test_untidy_golden_cases(engine, case):
    ctrace = load_ctrace(f"untidy_{case}")
    trees = parse(ctrace["lines"])
    supertree = make_tree(ctrace["supertree"])
    check(engine, supertree, trees, ctrace["weights"])
    # one of the source trees (unary chains, polytomies) as the supertree: all its clusters cost one step
    got = check(engine, trees[-1], trees, None)
    assert got.steps[-1] == got.characters[-1] == got.exact[-1]


def test_taxa_missing_on_either_side(engine):
    problem = make_problem(300, 40, "one", 11)
    trees = problem.phylonodes()
    supertree = construct_supertree(trees, None, "one", engine=engine)
    extra = make_tree(f"({supertree.get_newick()[:-1]},(zz1,zz2));")  # supertree taxa no source has
    check(engine, extra, problem.phylonodes())
    names = sorted(supertree.get_tip_names())
    dropped = set(names[::3])
    pruned = supertree.get_sub_tree([x for x in names if x not in dropped], as_rooted=True)
    check(engine, pruned, problem.phylonodes(), route="S")  # sources with taxa the supertree lacks


def test_one_tree_and_trees_sharing_fewer_than_three_taxa(engine):
    supertree = make_tree("(((a,b),c),(d,(e,f)));")
    check(engine, supertree, [make_tree("((a,c),(b,(d,e)));")], route="S")
    sources = [make_tree("(a,(x,y));"), make_tree("(x,y);"), make_tree("a;"), make_tree("((a,f),(x,e));"),
               make_tree("(q,r,s);"), make_tree("((a,b),(c,y));"), make_tree("(a,b,c,d,e,f);")]  # fmt: skip
    got = check(engine, supertree, sources, [1.0, 2.0, 3.0, 4.0, 5.0, 6.0, 7.0], route="S")
    assert got.shared.tolist() == [1, 0, 1, 3, 0, 3, 6]
    assert got.characters.tolist() == [0, 0, 0, 1, 0, 1, 0]
    assert got.steps.tolist() == [0, 0, 0, 2, 0, 1, 0]


def test_not_completed_entries_are_skipped(engine):
    supertree = make_tree("((a,b),(c,d));")
    trees = [make_tree("((a,b),(c,d));"), NotCompleted("ERROR", "x", "failed"), make_tree("((a,c),(b,d));")]
    got = mrp_score(supertree, trees, [1.0, 100.0, 3.0], engine=engine)
    assert got.steps.tolist() == [2, -1, 4] and got.characters.tolist() == [2, -1, 2]
    assert got.exact.tolist() == [2, -1, 0] and got.extra.tolist() == [0, -1, 2]
    assert got.ci[0] == 1.0 and np.isnan(got.ci[1]) and got.ci[2] == 0.5
    assert got.total_steps == 6 and got.total_characters == 4 and got.weighted_steps == 14.0
    with pytest.raises(ValueError, match="must match"):
        mrp_score(supertree, trees, [1.0], engine=engine)


def test_c4_full_size_against_clade_support(engine):
    problem = make_problem(10000, 1000, "depth", 4000)
    trees = problem.phylonodes()
    supertree = construct_supertree(trees, None, "depth", engine=engine)
    got = mrp_score(supertree, trees, engine=engine)
    again = mrp_score(supertree, trees, engine=engine)
    for key in (*INTS, "extra", "ci"):
        assert getattr(got, key).tobytes() == getattr(again, key).tobytes(), key
    assert got.weighted_steps == again.weighted_steps
    support = clade_support(supertree, trees, engine=engine)
    assert np.array_equal(got.exact, support.shared)
    assert np.array_equal(got.characters, support.source_clusters)
    assert (got.steps >= got.characters).all() and got.total_steps > got.total_characters
    smallest = np.argsort(got.shared, kind="stable")[:4]
    check(engine, supertree, [trees[t] for t in smallest])


def caterpillar(n: int) -> tuple[list[str], np.ndarray, np.ndarray]:
    """Flat caterpillar ((((t0, t1), t2), ...), t{n-1}) seen from the root: tip n - 1 hangs off the root and tips 0
    and 1 lie n - 1 levels deep."""
    names = [f"t{i}" for i in range(n)]
    parent = np.full(2 * n - 1, -1, dtype=np.int32)
    taxon = np.full(2 * n - 1, -1, dtype=np.int32)
    for i in range(n - 1):  # internal node 2i holds tip n - 1 - i and internal node 2i + 2 (tip 0 at the bottom)
        parent[2 * i + 1] = 2 * i
        taxon[2 * i + 1] = n - 1 - i
        parent[2 * i + 2] = 2 * i
    taxon[2 * n - 2] = 0
    return names, parent, taxon


def caterpillar_tree(names: list[str]) -> PhyloNode:
    node = PhyloNode(names[0])
    for name in names[1:]:
        node = PhyloNode("", [node, PhyloNode(name)])
    return node


def deep_sources(names: list[str]) -> list[PhyloNode]:
    rng = np.random.RandomState(5)
    picks = [[0, 1, 2, 3], [0, len(names) - 1, len(names) // 2, 5, 9], list(range(0, len(names), len(names) // 40))]
    picks += [sorted(rng.choice(len(names), size=30, replace=False)) for _ in range(3)]
    return [random_tree([names[i] for i in pick], seed=s) for s, pick in enumerate(picks)]


def test_deep_caterpillar_supertree(engine):
    names, parent, taxon = caterpillar(4000)
    sources = deep_sources(names)
    forest = Forest.from_trees(sources, [1.0] * len(sources), names=names)
    per_tree = engine.supertree_mrp(forest, parent, taxon)
    want = mrp_oracle.mrp_score(caterpillar_tree(names), sources, route="s'")
    for c, key in enumerate(INTS):
        assert per_tree[:, c].tolist() == want[key], key


def test_caterpillar_beyond_the_stack_is_refused(engine):
    names, parent, taxon = caterpillar(40000)
    sources = deep_sources(names)
    forest = Forest.from_trees(sources, [1.0] * len(sources), names=names)
    with pytest.raises(ScsError, match="too deep"):
        engine.supertree_mrp(forest, parent, taxon)


def test_cli_mrp_out(engine, tmp_path):
    from click.testing import CliRunner

    from spectralclustersupertree_b200.cli import scs

    problem = make_problem(300, 40, "branch", 21)
    src = tmp_path / "trees.nwk"
    src.write_text("\n".join(problem.newick_lines()) + "\n")
    plain, main, tsv = tmp_path / "plain.nwk", tmp_path / "main.nwk", tmp_path / "mrp.tsv"
    labelled, fit, per_taxon = tmp_path / "support.nwk", tmp_path / "fit.tsv", tmp_path / "taxa.tsv"
    runner = CliRunner()
    assert runner.invoke(scs, ["-i", str(src), "-o", str(plain)]).exit_code == 0
    result = runner.invoke(scs, ["-i", str(src), "-o", str(main), "--mrp-out", str(tsv)])
    assert result.exit_code == 0, result.output
    assert main.read_bytes() == plain.read_bytes()
    supertree = make_tree(plain.read_text().strip())
    got = mrp_score(supertree, parse(problem.newick_lines()), engine=engine)
    assert tsv.read_text() == got.tsv()
    rows = [line.split("\t") for line in tsv.read_text().splitlines()]
    assert rows[0] == ["tree", "shared", "characters", "steps", "exact"]
    assert len(rows) == 1 + len(problem.newick_lines())
    result = runner.invoke(scs, ["-i", str(src), "-o", str(main), "--mrp-out", str(tsv), "--support-out",
                                 str(labelled), "--triplets-out", str(fit), "--taxon-triplets-out", str(per_taxon)])  # fmt: skip
    assert result.exit_code == 0, result.output
    assert main.read_bytes() == plain.read_bytes()
    assert tsv.read_text() == got.tsv()
    assert labelled.read_text().strip() and fit.read_text().strip() and per_taxon.read_text().strip()
