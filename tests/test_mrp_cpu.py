"""CPU: the MRP oracle (oracle/mrp_oracle.py) on hand-worked known answers, its supertree route against its restricted
route and against the brute-force minimum, its tie to the clade support oracle, and the derived fields and TSV of
``MrpScore`` (host code only: no GPU is touched)."""

from __future__ import annotations

import math
import random

import numpy as np
import pytest

from oracle import mrp_oracle, support_oracle
from spectralclustersupertree_b200.mrp import MRP_TSV_HEADER, _score
from spectralclustersupertree_b200.tree import make_tree

QUARTET = "((a,b),(c,d));"

# supertree, source: (shared, characters, steps, exact)
CASES = {
    "cherry": ("((a,b),c);", "((a,b),c);", (3, 1, 1, 1)),
    "identical": (QUARTET, QUARTET, (4, 2, 2, 2)),
    "hard_polytomy": ("(a,b,c,d);", QUARTET, (4, 2, 4, 0)),
    "contradicting": (QUARTET, "((a,c),(b,d));", (4, 2, 4, 0)),
    "caterpillar_against_balanced": ("(((a,b),c),d);", QUARTET, (4, 2, 3, 1)),
    "star_source": (QUARTET, "(a,b,c,d);", (4, 0, 0, 0)),
    "unary_chain_supertree": ("((((a,b))),c);", "((a,b),c);", (3, 1, 1, 1)),
    "unary_chain_source": (QUARTET, "((((a,b))),(c,d));", (4, 2, 2, 2)),
    "source_taxon_missing_from_supertree": (QUARTET, "((a,x),(b,c));", (3, 1, 2, 0)),
    "supertree_taxon_missing_from_source": ("(((a,b),e),(c,d));", QUARTET, (4, 2, 2, 2)),
    "two_tips": (QUARTET, "(a,b);", (2, 0, 0, 0)),
    "lone_tip": (QUARTET, "a;", (1, 0, 0, 0)),
    "nothing_shared": (QUARTET, "(x,(y,z));", (0, 0, 0, 0)),
}


def random_tree(names, rng: random.Random, unary: bool = True):
    """A random rooted tree on ``names`` with polytomies of up to four children and, optionally, unary nodes."""
    nodes = list(names)
    while len(nodes) > 1:
        k = rng.randint(2, min(4, len(nodes)))
        rng.shuffle(nodes)
        group, nodes = nodes[:k], nodes[k:]
        text = "(" + ",".join(group) + ")"
        if unary and rng.random() < 0.2:
            text = "(" + text + ")"
        nodes.append(text)
    return make_tree(nodes[0] + ";")


def random_pairs(seed: int, count: int, most: int = 9):
    """(supertree, source) pairs with taxa missing on either side."""
    rng = random.Random(seed)
    for _ in range(count):
        names = [f"t{i}" for i in range(rng.randint(3, most))]
        source = rng.sample([*names, "x1", "x2"], rng.randint(2, min(most, len(names) + 2)))
        yield random_tree(names, rng), random_tree(source, rng)


@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_known_answers(case):
    supertree, source, want = CASES[case]
    S, t = make_tree(supertree), make_tree(source)
    assert mrp_oracle.tree_score(S, t) == want
    assert mrp_oracle.tree_score(S, t, route="s'") == want


def test_hard_polytomy_pair_costs_two():
    star = make_tree("(a,b,c,d);")
    assert mrp_oracle.hartigan_length(star, frozenset("ab"), frozenset("cd")) == 2
    assert mrp_oracle.brute_length(star, frozenset("ab"), frozenset("cd")) == 2


def test_supertree_route_equals_restricted_route():
    for S, t in random_pairs(1, 200):
        assert mrp_oracle.character_lengths(S, t) == mrp_oracle.character_lengths(S, t, route="s'")


def test_hartigan_equals_brute_force_minimum():
    checked = 0
    for S, t in random_pairs(2, 200):
        if sum(1 for node in S.preorder() if node.children) > 10:
            continue
        X, chars = mrp_oracle.characters(frozenset(S.get_tip_names()), t)
        for c in chars:
            assert mrp_oracle.hartigan_length(S, c, X - c) == mrp_oracle.brute_length(S, c, X - c)
            checked += 1
    assert checked > 100


def test_every_character_costs_a_step_and_exact_ones_are_supertree_clusters():
    pairs = list(random_pairs(3, 150, most=12))
    for S, t in pairs:
        X, chars = mrp_oracle.characters(frozenset(S.get_tip_names()), t)
        if not chars:
            continue
        restricted = S.get_sub_tree(X, ignore_missing=True, as_rooted=True)
        s_clusters = restricted.clade_sets()
        for c, length in zip(chars, mrp_oracle.character_lengths(S, t)[1], strict=True):
            assert length >= 1
            assert (length == 1) == (c in s_clusters)
    supertrees, trees = [S for S, _t in pairs], [t for _S, t in pairs]
    for S, t in zip(supertrees, trees, strict=True):
        support = support_oracle.clade_support(S, [t])
        score = mrp_oracle.mrp_score(S, [t])
        assert score["exact"] == support["shared"]
        assert score["characters"] == support["source_clusters"]


def test_oracle_weighted_steps_in_tree_order():
    out = mrp_oracle.mrp_score(make_tree(QUARTET), [make_tree(QUARTET), make_tree("((a,c),(b,d));"),
                                                    make_tree("(a,b);")], [0.1, 0.2, 5.0])  # fmt: skip
    assert out["steps"] == [2, 4, 0]
    assert out["weighted_steps"] == (0.0 + 0.1 * 2) + 0.2 * 4 + 5.0 * 0


def test_score_derived_values_and_skipped_entries():
    per_tree = np.array([[4, 2, 3, 1], [-1, -1, -1, -1], [2, 0, 0, 0], [5, 3, 3, 3]], dtype=np.int64)
    weights = [0.1, 7.0, 1.0, 0.2]
    score = _score(per_tree, weights, [0, 2, 3])
    assert score.extra.tolist() == [1, -1, 0, 0]
    assert score.ci[0] == 2 / 3 and math.isnan(score.ci[1]) and math.isnan(score.ci[2]) and score.ci[3] == 1.0
    assert score.total_steps == 6 and score.total_characters == 5 and score.total_ci == 5 / 6
    want = 0.0
    for t in (0, 2, 3):
        want += weights[t] * int(per_tree[t, 2])
    assert score.weighted_steps == want
    empty = _score(per_tree[[2]], [1.0], [0])
    assert empty.total_steps == 0 and math.isnan(empty.total_ci) and empty.weighted_steps == 0.0


def test_tsv_formatting():
    per_tree = np.array([[4, 2, 3, 1], [-1, -1, -1, -1], [2, 0, 0, 0]], dtype=np.int64)
    text = _score(per_tree, [1.0, 1.0, 1.0], [0, 2]).tsv()
    assert text == f"{MRP_TSV_HEADER}\n0\t4\t2\t3\t1\n1\t-1\t-1\t-1\t-1\n2\t2\t0\t0\t0\n"
    assert MRP_TSV_HEADER == "tree\tshared\tcharacters\tsteps\texact"
