"""GPU: the agreement sets of ``mast_taxa`` (``scs_supertree_mast_taxa``, csrc/triplets.cu) on every input family of
the MAST tests: per tree the counts are bit for bit those of ``scs_supertree_mast``, the node states mark exactly the
shared tips, the kept taxa form an agreement set of the MAST size (tests/mast_set_oracle.py) and, for k <= 9, one of the
maximum sets found by brute force; the per-taxon counts are those of the states.  Also: cases whose maximum set is
unique (a taxon moved in a 2 000-tip caterpillar, a rogue taxon planted at the root of the model tree), a 4 000-level
caterpillar supertree, the 10 000-taxon workload for determinism and the two identities, a tree above the table cap,
and the ``scs --mast-taxa-out`` command."""

from __future__ import annotations

import random

import numpy as np
import pytest

from helpers import CASES, load_case, load_ctrace, parse
import mast_set_oracle
from spectralclustersupertree_b200 import construct_supertree, mast_fit, mast_taxa
from spectralclustersupertree_b200.engine import Forest, ScsError
from spectralclustersupertree_b200.mast import _node_arrays
from spectralclustersupertree_b200.scs import _is_not_completed
from spectralclustersupertree_b200.support import _flat_supertree
from spectralclustersupertree_b200.synthetic import make_problem
from spectralclustersupertree_b200.tree import NotCompleted, PhyloNode, make_tree
from test_gpu_mast import caterpillar, caterpillar_tree, polytomy_tree, random_tree

pytestmark = pytest.mark.gpu


def check_states(forest, names, supertree, trees, per_tree, tip_state, brute: bool = True):
    """Per tree of ``forest`` (source ``trees``): the states mark exactly its shared tips and the kept ones are an
    agreement set of the MAST size; returns the kept sets."""
    in_s = frozenset(supertree.get_tip_names())
    _node_taxon, offsets = _node_arrays(forest)
    sets = []
    for j, tree in enumerate(trees):
        states = tip_state[offsets[j]:offsets[j + 1]]
        tx = forest.tree_arrays(j)[3]
        assert (states[tx < 0] == -1).all()
        shared = {names[x] for x in tx if x >= 0 and names[x] in in_s}
        assert {names[x] for x, s in zip(tx, states, strict=True) if s >= 0} == shared
        Y = frozenset(names[x] for x, s in zip(tx, states, strict=True) if s == 1)
        assert per_tree[j, 0] == len(shared) and per_tree[j, 1] == len(Y)
        assert mast_set_oracle.is_agreement_set(tree, supertree, Y, size=int(per_tree[j, 1])), j
        if brute and len(shared) <= 9:
            assert Y in mast_set_oracle.maximum_sets(tree, supertree), j
        sets.append(Y)
    return sets


def check(engine, supertree, trees, weights=None):
    got = mast_taxa(supertree, trees, weights, engine=engine)
    fit = mast_fit(supertree, trees, weights, engine=engine)
    for key in ("shared", "agreement", "pruned"):
        assert np.array_equal(getattr(got, key), getattr(fit, key)), key
    assert got.trees.sum() == fit.total_shared and got.taxon_pruned.sum() == fit.total_pruned
    if weights is None:
        weights = [1.0] * len(trees)
    kept = [i for i, tree in enumerate(trees) if not _is_not_completed(tree)]
    _nodes, names, parent, taxon = _flat_supertree(supertree, [trees[i] for i in kept])
    forest = Forest.from_trees([trees[i] for i in kept], [float(weights[i]) for i in kept], names=names)
    per_tree, tip_state, per_taxon, weighted = engine.supertree_mast_taxa(forest, parent, taxon)
    assert per_tree.tobytes() == engine.supertree_mast(forest, parent, taxon).tobytes()
    node_taxon, offsets = _node_arrays(forest)
    want, want_weighted = mast_set_oracle.taxon_counts(tip_state, node_taxon, offsets, forest.weights(),
                                                       forest.num_taxa)
    assert np.array_equal(per_taxon, want) and weighted.tobytes() == want_weighted.tobytes()
    sets = check_states(forest, names, supertree, [trees[i] for i in kept], per_tree, tip_state)
    for j, t in enumerate(kept):
        shared = frozenset(trees[t].get_tip_names()) & frozenset(supertree.get_tip_names())
        assert got.pruned_taxa[t] == tuple(sorted(shared - sets[j]))
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
    supertree = construct_supertree(problem.phylonodes(), problem.weights, weighting, engine=engine)
    check(engine, supertree, problem.phylonodes(), problem.weights)


def test_model_tree_and_a_random_tree(engine):
    problem = make_problem(500, 50, "one", 2000)
    model = problem.model.to_phylonode()
    check(engine, model, problem.phylonodes())
    check(engine, random_tree(sorted(model.get_tip_names()), seed=7), problem.phylonodes())


@pytest.mark.parametrize("case", ["branch", "bootstrap", "depth", "nocontract", "caterpillar"])
def test_untidy_golden_cases(engine, case):
    ctrace = load_ctrace(f"untidy_{case}")
    trees = parse(ctrace["lines"])
    check(engine, make_tree(ctrace["supertree"]), trees, ctrace["weights"])
    got = check(engine, trees[-1], trees, None)
    assert got.pruned_taxa[-1] == ()


def test_taxa_missing_on_either_side(engine):
    problem = make_problem(300, 40, "one", 11)
    supertree = construct_supertree(problem.phylonodes(), None, "one", engine=engine)
    extra = make_tree(f"({supertree.get_newick()[:-1]},(zz1,zz2));")
    got = check(engine, extra, problem.phylonodes())
    assert got.trees[got.names.index("zz1")] == 0 and np.isnan(got.fraction[got.names.index("zz1")])
    names = sorted(supertree.get_tip_names())
    dropped = set(names[::3])
    pruned = supertree.get_sub_tree([x for x in names if x not in dropped], as_rooted=True)
    check(engine, pruned, problem.phylonodes())


def test_trees_sharing_up_to_two_taxa_and_skipped_entries(engine):
    supertree = make_tree("(((a,b),c),(d,(e,f)));")
    sources = [make_tree("(a,(x,y));"), make_tree("(x,y);"), make_tree("a;"), make_tree("((a,f),(x,e));"),
               make_tree("(q,r,s);"), NotCompleted("ERROR", "x", "failed"), make_tree("((a,b),(c,y));"),
               make_tree("(a,b,c,d,e,f);"), make_tree("(b,x);"), make_tree("((a,c),(b,(d,e)));")]  # fmt: skip
    got = check(engine, supertree, sources, [1.0, 2.0, 3.0, 4.0, 5.0, 100.0, 6.0, 7.0, 8.0, 9.0])
    assert [len(p) for p in got.pruned_taxa if p is not None] == [0, 0, 0, 1, 0, 0, 4, 0, 1]
    assert got.pruned_taxa[5] is None and got.shared[5] == -1


def test_polytomies_on_both_sides(engine):
    names = [f"t{i}" for i in range(60)]
    supertrees = [polytomy_tree(names, seed, widest) for seed, widest in enumerate((3, 5, 8, 12))]
    rng = random.Random(3)
    sources = [polytomy_tree(rng.sample(names, rng.randint(4, 60)), 100 + s, rng.choice((3, 4, 6, 9)))
               for s in range(16)]  # fmt: skip
    for supertree in supertrees:
        check(engine, supertree, sources)


def test_polytomies_wider_than_a_warp_on_both_sides(engine):
    rng = random.Random(9)
    names = [f"t{i}" for i in range(120)]
    for s in range(4):
        a, b = names[:], names[:]
        rng.shuffle(a)
        rng.shuffle(b)
        S = make_tree("((" + ",".join(a[:3]) + "),(" + ",".join(a[3:7]) + ")," + ",".join(a[7:80 + 10 * s]) + ");")
        t = make_tree("((" + ",".join(b[:2]) + "),(" + ",".join(b[2:40]) + ")," + ",".join(b[40:]) + ");")
        check(engine, S, [t])
        check(engine, t, [S])


def test_star_supertree(engine):
    names = [f"t{i}" for i in range(200)]
    star = make_tree("(" + ",".join(names) + ");")
    rng = np.random.RandomState(1)
    sources = [random_tree(list(rng.choice(names, size=k, replace=False)), seed=k) for k in (1, 2, 3, 5, 9, 40, 200)]
    got = check(engine, star, sources)
    assert [len(p) for p in got.pruned_taxa] == [max(int(k) - 2, 0) for k in got.shared]


def test_moved_taxon_of_a_caterpillar_is_the_only_one_pruned(engine):
    names = [f"t{i}" for i in range(2000)]
    moved = names[:700] + names[701:] + [names[700]]
    got = mast_taxa(caterpillar_tree(moved), [caterpillar_tree(names)], engine=engine)
    assert got.pruned_taxa == [("t700",)]
    assert got.taxon_pruned.sum() == 1 and got.taxon_pruned[got.names.index("t700")] == 1


def test_planted_rogue_taxon(engine):
    problem = make_problem(500, 50, "one", 2000)
    model = problem.model.to_phylonode()
    names = sorted(model.get_tip_names())
    rng = random.Random(17)
    x = rng.choice(names)
    rest = model.get_sub_tree([y for y in names if y != x], as_rooted=True)
    S = PhyloNode("", [*rest.children, PhyloNode(x)])  # x re-attached as a child of the root
    sources = [model.get_sub_tree(sorted({*rng.sample(names, rng.randint(20, 120)), x}), as_rooted=True)
               for _ in range(40)]  # fmt: skip
    sources += [model.get_sub_tree(rng.sample(names, 50), as_rooted=True) for _ in range(5)]
    got = check(engine, S, sources)
    exact = 0
    for t, source in enumerate(sources):
        if x not in source.get_tip_names():
            continue
        side = next(c for c in source.children if x in c.get_tip_names())
        inside = len(side.get_tip_names()) - 1
        if inside >= 2 and len(source.get_tip_names()) - inside - 1 >= 2:
            assert got.pruned_taxa[t] == (x,), t
            exact += 1
    assert exact >= 10
    top = got.names.index(x)
    assert all(got.taxon_pruned[top] > p for i, p in enumerate(got.taxon_pruned) if i != top)


def test_deep_caterpillar_supertree(engine):
    names, parent, taxon = caterpillar(4000)
    rng = np.random.RandomState(5)
    picks = [[0, 1, 2, 3], [0, len(names) - 1, len(names) // 2, 5, 9], list(range(0, len(names), len(names) // 40))]
    picks += [sorted(rng.choice(len(names), size=30, replace=False)) for _ in range(3)]
    sources = [random_tree([names[i] for i in pick], seed=s) for s, pick in enumerate(picks)]
    sources.append(caterpillar_tree([names[i] for i in range(0, 4000, 7)]))
    forest = Forest.from_trees(sources, [1.0] * len(sources), names=names)
    per_tree, tip_state, _per_taxon, _weighted = engine.supertree_mast_taxa(forest, parent, taxon)
    assert per_tree.tobytes() == engine.supertree_mast(forest, parent, taxon).tobytes()
    sets = check_states(forest, names, caterpillar_tree(names), sources, per_tree, tip_state)
    assert len(sets[-1]) == 572


def test_c4_full_size(engine):
    problem = make_problem(10000, 1000, "depth", 4000)
    trees = problem.phylonodes()
    supertree = construct_supertree(trees, None, "depth", engine=engine)
    _nodes, names, parent, taxon = _flat_supertree(supertree, trees)
    forest = Forest.from_trees(trees, [1.0] * len(trees), names=names)
    first = engine.supertree_mast_taxa(forest, parent, taxon)
    again = engine.supertree_mast_taxa(forest, parent, taxon)
    for a, b in zip(first, again, strict=True):
        assert a.tobytes() == b.tobytes()
    per_tree, tip_state, per_taxon, _weighted = first
    fit = mast_fit(supertree, trees, engine=engine)
    assert np.array_equal(per_tree[:, 0], fit.shared) and np.array_equal(per_tree[:, 1], fit.agreement)
    assert per_taxon[:, 0].sum() == fit.total_shared and per_taxon[:, 1].sum() == fit.total_pruned
    smallest = np.argsort(per_tree[:, 0], kind="stable")[:50]
    drawn = np.random.RandomState(4).choice(len(trees), size=50, replace=False)
    pick = sorted(set(smallest.tolist()) | set(drawn.tolist()))
    sub = Forest.from_trees([trees[t] for t in pick], [1.0] * len(pick), names=names)
    sub_tree, sub_state, _, _ = engine.supertree_mast_taxa(sub, parent, taxon)
    assert np.array_equal(sub_tree, per_tree[pick])
    _node_taxon, offsets = _node_arrays(forest)
    _sub_taxon, sub_offsets = _node_arrays(sub)
    for j, t in enumerate(pick):  # a tree's states do not depend on the other trees of the forest
        assert np.array_equal(sub_state[sub_offsets[j]:sub_offsets[j + 1]], tip_state[offsets[t]:offsets[t + 1]])
    check_states(sub, names, supertree, [trees[t] for t in pick], sub_tree, sub_state, brute=False)


def test_table_above_the_cap_is_refused_before_any_launch(engine):
    n = 34000
    names, parent, taxon = caterpillar(n)
    forest = Forest.from_arrays(np.array([0, len(parent)]), parent, None, None, taxon, [1.0], names, copy=True)
    launches = engine.launch_count
    with pytest.raises(ScsError, match="scs_supertree_mast_taxa: source tree 0 .* above the cap"):
        engine.supertree_mast_taxa(forest, parent, taxon)
    assert engine.launch_count == launches


def test_cli_mast_taxa_out(engine, tmp_path):
    from click.testing import CliRunner

    from spectralclustersupertree_b200.cli import scs

    problem = make_problem(300, 40, "branch", 21)
    src = tmp_path / "trees.nwk"
    src.write_text("\n".join(problem.newick_lines()) + "\n")
    plain, main, tsv, mast = tmp_path / "plain.nwk", tmp_path / "main.nwk", tmp_path / "taxa.tsv", tmp_path / "m.tsv"
    runner = CliRunner()
    assert runner.invoke(scs, ["-i", str(src), "-o", str(plain)]).exit_code == 0
    result = runner.invoke(scs, ["-i", str(src), "-o", str(main), "--mast-taxa-out", str(tsv), "--mast-out", str(mast)])
    assert result.exit_code == 0, result.output
    assert main.read_bytes() == plain.read_bytes()
    supertree = make_tree(plain.read_text().strip())
    trees = parse(problem.newick_lines())
    assert tsv.read_text() == mast_taxa(supertree, trees, engine=engine).tsv()
    assert mast.read_text() == mast_fit(supertree, trees, engine=engine).tsv()
    rows = [line.split("\t") for line in tsv.read_text().splitlines()]
    assert rows[0] == ["taxon", "trees", "pruned"] and len(rows) == 1 + len(supertree.get_tip_names())
