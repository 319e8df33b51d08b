"""GPU: ``mast_fit`` (csrc/triplets.cu) against the agreement-subtree oracle (oracle/mast_oracle.py): every per-tree
count exactly and ``weighted_pruned`` to 1e-12 relative, on the inputs of the MRP tests (built supertrees, model and
random trees, the untidy golden cases, taxa missing on either side, one tree, trees sharing up to two taxa, skipped
entries); polytomies of degree >= 3 on both sides, up to wider than a warp, for the Hungarian path; a star supertree;
symmetry; caterpillars thousands of levels deep; the 10 000-taxon workload against ``clade_support`` and for
determinism; a tree whose table is above the cap; the ``scs --mast-out`` command."""

from __future__ import annotations

import random

import numpy as np
import pytest

from helpers import CASES, load_case, load_ctrace, parse
from oracle import mast_oracle
from spectralclustersupertree_b200 import clade_support, construct_supertree, mast_fit
from spectralclustersupertree_b200.engine import Forest, ScsError
from spectralclustersupertree_b200.synthetic import make_problem
from spectralclustersupertree_b200.tree import NotCompleted, PhyloNode, make_tree

pytestmark = pytest.mark.gpu

INTS = ("shared", "agreement", "pruned")


def check(engine, supertree, trees, weights=None):
    got = mast_fit(supertree, trees, weights, engine=engine)
    want = mast_oracle.mast_fit(supertree, trees, weights)
    for key in INTS:
        assert np.array_equal(getattr(got, key), np.asarray(want[key])), key
    assert ((got.agreement >= np.minimum(got.shared, 1)) & (got.agreement <= got.shared)).all()
    np.testing.assert_allclose(got.weighted_pruned, want["weighted_pruned"], rtol=1e-12, atol=0)
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


def polytomy_tree(names, seed: int, widest: int) -> PhyloNode:
    """A random rooted tree on ``names`` whose nodes have 2 to ``widest`` children."""
    rng = random.Random(seed)
    nodes = [PhyloNode(name) for name in names]
    while len(nodes) > 1:
        k = rng.randint(2, min(widest, len(nodes)))
        rng.shuffle(nodes)
        group, nodes = nodes[:k], nodes[k:]
        nodes.append(PhyloNode("", group))
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
    assert got.total_agreement > 0


def test_model_tree_and_a_random_tree(engine):
    problem = make_problem(500, 50, "one", 2000)
    model = problem.model.to_phylonode()
    got = check(engine, model, problem.phylonodes())
    assert got.total_agreement / got.total_shared > 0.8
    rand = random_tree(sorted(model.get_tip_names()), seed=7)
    got = check(engine, rand, problem.phylonodes())
    assert got.total_agreement / got.total_shared < 0.3


@pytest.mark.parametrize("case", ["branch", "bootstrap", "depth", "nocontract", "caterpillar"])
def test_untidy_golden_cases(engine, case):
    ctrace = load_ctrace(f"untidy_{case}")
    trees = parse(ctrace["lines"])
    supertree = make_tree(ctrace["supertree"])
    check(engine, supertree, trees, ctrace["weights"])
    # one of the source trees (unary chains, polytomies) as the supertree agrees with itself on every shared taxon
    got = check(engine, trees[-1], trees, None)
    assert got.agreement[-1] == got.shared[-1] and got.pruned[-1] == 0


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


def test_one_tree_and_trees_sharing_up_to_two_taxa(engine):
    supertree = make_tree("(((a,b),c),(d,(e,f)));")
    got = check(engine, supertree, [make_tree("((a,c),(b,(d,e)));")])
    assert got.shared.tolist() == [5] and got.agreement.tolist() == [4]
    sources = [make_tree("(a,(x,y));"), make_tree("(x,y);"), make_tree("a;"), make_tree("((a,f),(x,e));"),
               make_tree("(q,r,s);"), make_tree("((a,b),(c,y));"), make_tree("(a,b,c,d,e,f);"),
               make_tree("(b,x);")]  # fmt: skip
    got = check(engine, supertree, sources, [1.0, 2.0, 3.0, 4.0, 5.0, 6.0, 7.0, 8.0])
    assert got.shared.tolist() == [1, 0, 1, 3, 0, 3, 6, 1]
    assert got.agreement.tolist() == [1, 0, 1, 2, 0, 3, 2, 1]
    assert got.weighted_pruned == 4.0 * 1 + 7.0 * 4


def test_not_completed_entries_are_skipped(engine):
    supertree = make_tree("((a,b),(c,d));")
    trees = [make_tree("((a,b),(c,d));"), NotCompleted("ERROR", "x", "failed"), make_tree("((a,c),(b,d));")]
    got = mast_fit(supertree, trees, [1.0, 100.0, 3.0], engine=engine)
    assert got.shared.tolist() == [4, -1, 4] and got.agreement.tolist() == [4, -1, 2]
    assert got.pruned.tolist() == [0, -1, 2]
    assert got.fraction[0] == 1.0 and np.isnan(got.fraction[1]) and got.fraction[2] == 0.5
    assert got.total_shared == 8 and got.total_agreement == 6 and got.weighted_pruned == 6.0
    with pytest.raises(ValueError, match="must match"):
        mast_fit(supertree, trees, [1.0], engine=engine)


def test_polytomies_on_both_sides(engine):
    names = [f"t{i}" for i in range(60)]
    supertrees = [polytomy_tree(names, seed, widest) for seed, widest in enumerate((3, 5, 8, 12))]
    rng = random.Random(3)
    sources = [polytomy_tree(rng.sample(names, rng.randint(10, 60)), 100 + s, rng.choice((3, 4, 6, 9)))
               for s in range(12)]  # fmt: skip
    for supertree in supertrees:
        check(engine, supertree, sources)


def test_polytomies_wider_than_a_warp_on_both_sides(engine):
    rng = random.Random(9)
    names = [f"t{i}" for i in range(120)]
    pairs = []
    for s in range(4):
        a, b = names[:], names[:]
        rng.shuffle(a)
        rng.shuffle(b)
        # root polytomies of 40 to 100 children, some of them small clades, on both sides
        S = make_tree("((" + ",".join(a[:3]) + "),(" + ",".join(a[3:7]) + ")," + ",".join(a[7:80 + 10 * s]) + ");")
        t = make_tree("((" + ",".join(b[:2]) + "),(" + ",".join(b[2:40]) + ")," + ",".join(b[40:]) + ");")
        pairs.append((S, t))
    for S, t in pairs:
        got = check(engine, S, [t])
        assert got.agreement[0] == check(engine, t, [S]).agreement[0]


def test_star_supertree_gives_at_most_two(engine):
    names = [f"t{i}" for i in range(200)]
    star = make_tree("(" + ",".join(names) + ");")
    rng = np.random.RandomState(1)
    sources = [random_tree(list(rng.choice(names, size=k, replace=False)), seed=k) for k in (1, 2, 3, 5, 40, 200)]
    got = check(engine, star, sources)
    assert got.agreement.tolist() == [min(int(k), 2) for k in got.shared]


def test_symmetry(engine):
    names = [f"t{i}" for i in range(150)]
    for seed in range(3):
        a, b = polytomy_tree(names, 2 * seed, 5), polytomy_tree(names, 2 * seed + 1, 4)
        one = check(engine, a, [b])
        other = check(engine, b, [a])
        assert one.agreement.tolist() == other.agreement.tolist()


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


def test_deep_caterpillar_supertree(engine):
    names, parent, taxon = caterpillar(4000)
    rng = np.random.RandomState(5)
    picks = [[0, 1, 2, 3], [0, len(names) - 1, len(names) // 2, 5, 9], list(range(0, len(names), len(names) // 40))]
    picks += [sorted(rng.choice(len(names), size=30, replace=False)) for _ in range(3)]
    sources = [random_tree([names[i] for i in pick], seed=s) for s, pick in enumerate(picks)]
    sources.append(caterpillar_tree([names[i] for i in range(0, 4000, 7)]))  # agrees on all of its taxa
    forest = Forest.from_trees(sources, [1.0] * len(sources), names=names)
    per_tree = engine.supertree_mast(forest, parent, taxon)
    want = mast_oracle.mast_fit(caterpillar_tree(names), sources)
    assert per_tree[:, 0].tolist() == want["shared"]
    assert per_tree[:, 1].tolist() == want["agreement"]
    assert per_tree[-1, 1] == per_tree[-1, 0] == 572


def test_caterpillar_source_against_reversed_caterpillar(engine):
    names = [f"t{i}" for i in range(2000)]
    source = caterpillar_tree(names)
    reversed_supertree = caterpillar_tree(names[::-1])
    got = check(engine, reversed_supertree, [source])
    assert got.shared.tolist() == [2000] and got.agreement.tolist() == [2]
    moved = names[:700] + names[701:] + [names[700]]  # one taxon moved to the top: drop it and they agree
    got = mast_fit(caterpillar_tree(moved), [source], engine=engine)
    assert got.agreement.tolist() == [1999]


def test_table_above_the_cap_is_refused_before_any_launch(engine):
    n = 34000  # (n - 1)^2 ints pass 4 GiB
    names, parent, taxon = caterpillar(n)
    forest = Forest.from_arrays(np.array([0, len(parent)]), parent, None, None, taxon, [1.0], names, copy=True)
    launches = engine.launch_count
    with pytest.raises(ScsError, match="above the cap"):
        engine.supertree_mast(forest, parent, taxon)
    assert engine.launch_count == launches


def test_c4_full_size_against_clade_support(engine):
    problem = make_problem(10000, 1000, "depth", 4000)
    trees = problem.phylonodes()
    supertree = construct_supertree(trees, None, "depth", engine=engine)
    got = mast_fit(supertree, trees, engine=engine)
    again = mast_fit(supertree, trees, engine=engine)
    for key in (*INTS, "fraction"):
        assert getattr(got, key).tobytes() == getattr(again, key).tobytes(), key
    assert got.weighted_pruned == again.weighted_pruned
    support = clade_support(supertree, trees, engine=engine)
    assert np.array_equal(got.agreement == got.shared, support.rf == 0)
    assert ((got.agreement >= 1) & (got.agreement <= got.shared)).all()
    smallest = np.argsort(got.shared, kind="stable")[:4]
    check(engine, supertree, [trees[t] for t in smallest])


def test_cli_mast_out(engine, tmp_path):
    from click.testing import CliRunner

    from spectralclustersupertree_b200.cli import scs

    problem = make_problem(300, 40, "branch", 21)
    src = tmp_path / "trees.nwk"
    src.write_text("\n".join(problem.newick_lines()) + "\n")
    plain, main, tsv = tmp_path / "plain.nwk", tmp_path / "main.nwk", tmp_path / "mast.tsv"
    labelled, fit, per_taxon = tmp_path / "support.nwk", tmp_path / "fit.tsv", tmp_path / "taxa.tsv"
    mrp = tmp_path / "mrp.tsv"
    runner = CliRunner()
    assert runner.invoke(scs, ["-i", str(src), "-o", str(plain)]).exit_code == 0
    result = runner.invoke(scs, ["-i", str(src), "-o", str(main), "--mast-out", str(tsv)])
    assert result.exit_code == 0, result.output
    assert main.read_bytes() == plain.read_bytes()
    supertree = make_tree(plain.read_text().strip())
    got = mast_fit(supertree, parse(problem.newick_lines()), engine=engine)
    assert tsv.read_text() == got.tsv()
    rows = [line.split("\t") for line in tsv.read_text().splitlines()]
    assert rows[0] == ["tree", "shared", "agreement", "pruned"]
    assert len(rows) == 1 + len(problem.newick_lines())
    result = runner.invoke(scs, ["-i", str(src), "-o", str(main), "--mast-out", str(tsv), "--support-out",
                                 str(labelled), "--triplets-out", str(fit), "--taxon-triplets-out", str(per_taxon),
                                 "--mrp-out", str(mrp)])  # fmt: skip
    assert result.exit_code == 0, result.output
    assert main.read_bytes() == plain.read_bytes()
    assert tsv.read_text() == got.tsv()
    assert labelled.read_text().strip() and fit.read_text().strip() and per_taxon.read_text().strip()
    assert mrp.read_text().strip()
