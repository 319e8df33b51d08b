"""CPU: the agreement-subtree oracle (oracle/mast_oracle.py) against a brute force over taxon subsets and on
hand-worked cases, its ties to the clade support oracle and its symmetry, and the derived fields, skipped entries and
TSV of ``MastFit`` (host code only: no GPU is touched)."""

from __future__ import annotations

import math
import random

import numpy as np
import pytest

from oracle import mast_oracle, support_oracle
from spectralclustersupertree_b200.mast import MAST_TSV_HEADER, _fit
from spectralclustersupertree_b200.tree import PhyloNode, make_tree

# supertree, source: (shared, agreement)
CASES = {
    "quartets": ("((a,b),(c,d));", "((a,c),(b,d));", (4, 2)),
    "caterpillars": ("(((a,b),c),d);", "(((a,b),d),c);", (4, 3)),
    "star_against_binary": ("(a,b,c,d,e,f);", "(((a,b),c),((d,e),f));", (6, 2)),
    "identical": ("((a,b),(c,d));", "((b,a),(d,c));", (4, 4)),
    "unary_chains": ("((((a,b))),(c,d));", "(((a,b)),((c),d));", (4, 4)),
    "polytomy_refined": ("((a,b,c),d);", "(((a,b),c),d);", (4, 3)),
    "missing_on_both_sides": ("(((a,b),x),(c,d));", "((a,(b,y)),(c,d));", (4, 4)),
    "two_shared": ("((a,b),(c,d));", "((a,x),(c,y));", (2, 2)),
    "lone_tip": ("((a,b),(c,d));", "a;", (1, 1)),
    "nothing_shared": ("((a,b),(c,d));", "(x,(y,z));", (0, 0)),
}


def random_tree(names, rng: random.Random, unary: bool = True, widest: int = 4):
    """A random rooted tree on ``names`` with polytomies of up to ``widest`` children and, optionally, unary nodes."""
    nodes = list(names)
    while len(nodes) > 1:
        k = rng.randint(2, min(widest, len(nodes)))
        rng.shuffle(nodes)
        group, nodes = nodes[:k], nodes[k:]
        text = "(" + ",".join(group) + ")"
        if unary and rng.random() < 0.2:
            text = "(" + text + ")"
        nodes.append(text)
    return make_tree(nodes[0] + ";")


def random_pairs(seed: int, count: int, most: int = 8):
    """(supertree, source) pairs with taxa missing on either side."""
    rng = random.Random(seed)
    for _ in range(count):
        names = [f"t{i}" for i in range(rng.randint(2, most))]
        source = rng.sample([*names, "x1", "x2"], rng.randint(2, min(most, len(names) + 2)))
        yield random_tree(names, rng), random_tree(source, rng)


def caterpillar(names) -> PhyloNode:
    node = PhyloNode(names[0])
    for name in names[1:]:
        node = PhyloNode("", [node, PhyloNode(name)])
    return node


@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_known_answers(case):
    supertree, source, want = CASES[case]
    S, t = make_tree(supertree), make_tree(source)
    assert mast_oracle.tree_fit(S, t) == want
    assert mast_oracle.tree_fit(t, S) == want


def test_recurrence_equals_brute_force():
    checked = 0
    for S, t in random_pairs(1, 300):
        k, m = mast_oracle.tree_fit(S, t)
        assert m == mast_oracle.mast_brute(t, S), (S.get_newick(), t.get_newick())
        checked += k >= 4
    assert checked > 80


def test_star_against_any_binary_tree_gives_two():
    rng = random.Random(4)
    for k in range(2, 12):
        names = [f"t{i}" for i in range(k)]
        star = make_tree("(" + ",".join(names) + ");")
        binary = random_tree(names, rng, unary=False, widest=2)
        assert mast_oracle.tree_fit(star, binary) == (k, 2)


def test_caterpillar_against_its_reverse_gives_two():
    names = [f"t{i}" for i in range(60)]
    assert mast_oracle.tree_fit(caterpillar(names[::-1]), caterpillar(names)) == (60, 2)
    moved = names[:30] + names[31:] + [names[30]]
    assert mast_oracle.tree_fit(caterpillar(moved), caterpillar(names)) == (60, 59)


def test_wide_polytomies_on_both_sides():
    rng = random.Random(9)
    names = [f"t{i}" for i in range(40)]
    for _ in range(5):
        a, b = names[:], names[:]
        rng.shuffle(a)
        rng.shuffle(b)
        # two polytomies of 35 children each, five taxa grouped differently below them
        S = make_tree("((" + ",".join(a[:3]) + ")," + ",".join(a[3:5]) + "," + ",".join(a[5:]) + ");")
        t = make_tree("((" + ",".join(b[:2]) + ")," + ",".join(b[2:6]) + "," + ",".join(b[6:]) + ");")
        k, m = mast_oracle.tree_fit(S, t)
        assert k == 40 and m == mast_oracle.tree_fit(t, S)[1]
        # dropping the five grouped taxa leaves the same star on 35
        assert 35 <= m < 40


def test_full_agreement_exactly_when_rf_is_zero_and_symmetry():
    both = 0
    for S, t in random_pairs(3, 200, most=10):
        k, m = mast_oracle.tree_fit(S, t)
        rf = support_oracle.clade_support(S, [t])["rf"][0]
        assert (m == k) == (rf == 0)
        assert mast_oracle.tree_fit(t, S) == (k, m)
        assert 0 < m <= k or k == 0
        both += m == k and k >= 3
    assert both > 5


def test_oracle_weighted_pruned_in_tree_order():
    out = mast_oracle.mast_fit(make_tree("((a,b),(c,d));"), [make_tree("((a,b),(c,d));"), make_tree("((a,c),(b,d));"),
                                                            make_tree("(a,b);")], [0.1, 0.2, 5.0])  # fmt: skip
    assert out["agreement"] == [4, 2, 2] and out["pruned"] == [0, 2, 0]
    assert out["weighted_pruned"] == (0.0 + 0.1 * 0) + 0.2 * 2 + 5.0 * 0


def test_fit_derived_values_and_skipped_entries():
    per_tree = np.array([[4, 3], [-1, -1], [0, 0], [5, 5], [7, 2]], dtype=np.int64)
    weights = [0.1, 7.0, 1.0, 0.2, 0.3]
    fit = _fit(per_tree, weights, [0, 2, 3, 4])
    assert fit.pruned.tolist() == [1, -1, 0, 0, 5]
    assert fit.fraction[0] == 0.75 and math.isnan(fit.fraction[1]) and math.isnan(fit.fraction[2])
    assert fit.fraction[3] == 1.0 and fit.fraction[4] == 2 / 7
    assert fit.total_shared == 16 and fit.total_agreement == 10 and fit.total_pruned == 6
    want = 0.0
    for t in (0, 2, 3, 4):
        want += weights[t] * int(per_tree[t, 0] - per_tree[t, 1])
    assert fit.weighted_pruned == want
    empty = _fit(per_tree[[1]], [1.0], [])
    assert empty.total_pruned == 0 and empty.weighted_pruned == 0.0 and empty.pruned.tolist() == [-1]


def test_tsv_formatting():
    per_tree = np.array([[4, 3], [-1, -1], [2, 2]], dtype=np.int64)
    text = _fit(per_tree, [1.0, 1.0, 1.0], [0, 2]).tsv()
    assert text == f"{MAST_TSV_HEADER}\n0\t4\t3\t1\n1\t-1\t-1\t-1\n2\t2\t2\t0\n"
    assert MAST_TSV_HEADER == "tree\tshared\tagreement\tpruned"
