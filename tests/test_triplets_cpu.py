"""CPU: the brute-force triplet oracle (oracle/triplet_oracle.py) on hand-worked known answers, and the TSV that
``scs --triplets-out`` writes (host code only: no GPU is touched)."""

from __future__ import annotations

import math

import numpy as np
import pytest

from oracle.triplet_oracle import tree_fit, triplet_fit
from spectralclustersupertree_b200.triplets import TSV_HEADER, _fit, triplet_tsv
from spectralclustersupertree_b200.tree import make_tree

QUARTET = "((a,b),(c,d));"

# supertree, source: (shared, resolved_source, resolved_supertree, agree, contradict)
CASES = {
    "identical": (QUARTET, QUARTET, (4, 4, 4, 4, 0)),
    "contradicting": (QUARTET, "((a,c),(b,d));", (4, 4, 4, 0, 4)),
    "star_source": (QUARTET, "(a,b,c,d);", (4, 0, 4, 0, 0)),
    "polytomy_source": ("(((a,b),c),d);", "((a,b,c),d);", (4, 3, 4, 3, 0)),
    "source_taxa_missing_from_supertree": (QUARTET, "((a,x),(b,(c,d)));", (4, 4, 4, 2, 2)),
    "supertree_taxa_missing_from_source": ("(((a,b),e),(c,d));", QUARTET, (4, 4, 4, 4, 0)),
    "unary_chain_source": (QUARTET, "((((a,b))),(c,d));", (4, 4, 4, 4, 0)),
    "unary_root_source": (QUARTET, "(((a,b),(c,d)));", (4, 4, 4, 4, 0)),
    "unary_chain_supertree": ("(((a,b)),(c,d));", QUARTET, (4, 4, 4, 4, 0)),
    "caterpillar_against_balanced": ("(((a,b),c),d);", QUARTET, (4, 4, 4, 2, 2)),
    "three_taxa_shared": (QUARTET, "((a,b),(c,y));", (3, 1, 1, 1, 0)),
    "two_tips": (QUARTET, "(a,b);", (2, 0, 0, 0, 0)),
    "lone_tip": (QUARTET, "a;", (1, 0, 0, 0, 0)),
    "nothing_shared": (QUARTET, "(x,(y,z));", (0, 0, 0, 0, 0)),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_known_answers(case):
    supertree, source, want = CASES[case]
    assert tree_fit(make_tree(supertree), make_tree(source)) == want


def test_oracle_counts_every_triplet_once():
    # a caterpillar against its mirror image: every one of the C(6, 3) triplets is resolved in both
    s = make_tree("(((((a,b),c),d),e),f);")
    t = make_tree("(a,(b,(c,(d,(e,f)))));")
    k, rs, rsup, agree, contradict = tree_fit(s, t)
    assert (k, rs, rsup) == (6, 20, 20)
    assert agree + contradict == 20 and contradict > agree


def test_oracle_weighted_fit_in_tree_order():
    out = triplet_fit(make_tree(QUARTET), [make_tree(QUARTET), make_tree("((a,c),(b,d));"), make_tree("(a,b);")],
                      [2.0, 1.0, 5.0])  # fmt: skip
    assert out["agree"] == [4, 0, 0] and out["resolved_source"] == [4, 4, 0]
    assert out["weighted_fit"] == 8.0 / 12.0


def test_fit_derived_values_and_skipped_entries():
    per_tree = np.array([[4, 4, 4, 2, 2], [-1, -1, -1, -1, -1], [2, 0, 0, 0, 0], [4, 3, 4, 3, 0]], dtype=np.int64)
    fit = _fit(per_tree, [1.0, 7.0, 1.0, 3.0], [0, 2, 3])
    assert fit.unresolved.tolist() == [0, -1, 0, 0]
    assert fit.fit[0] == 0.5 and math.isnan(fit.fit[1]) and math.isnan(fit.fit[2]) and fit.fit[3] == 1.0
    assert fit.weighted_fit == (1.0 * 2 + 3.0 * 3) / (1.0 * 4 + 3.0 * 3)
    assert math.isnan(_fit(per_tree[[2]], [1.0], [0]).weighted_fit)


def test_tsv_formatting():
    per_tree = np.array([[4, 4, 4, 2, 2], [2, 0, 0, 0, 0]], dtype=np.int64)
    text = triplet_tsv(per_tree)
    assert text == f"{TSV_HEADER}\n0\t4\t4\t4\t2\t2\n1\t2\t0\t0\t0\t0\n"
    assert TSV_HEADER == "tree\tshared\tresolved_source\tresolved_supertree\tagree\tcontradict"
    assert _fit(per_tree, [1.0, 1.0], [0, 1]).tsv() == text
