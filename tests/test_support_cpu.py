"""CPU: the set-based clade-support oracle (oracle/support_oracle.py) on hand-built known answers, one per class and
one per untidy shape, and ``scs_flat_tree_newick_values`` (host code only: no GPU is touched)."""

from __future__ import annotations

import math

import numpy as np
import pytest

from oracle.support_oracle import clade_support
from spectralclustersupertree_b200.engine import Forest
from spectralclustersupertree_b200.scs import flat_newick
from spectralclustersupertree_b200.support import flat_newick_values
from spectralclustersupertree_b200.tree import make_tree

QUARTET = "((a,b),(c,d));"


def score(supertree: str, sources: list[str], weights=None) -> dict:
    return clade_support(make_tree(supertree), [make_tree(s) for s in sources], weights)


def per_tree(out: dict, t: int = 0) -> tuple[int, int, int, int]:
    return out["shared"][t], out["source_clusters"][t], out["supertree_clusters"][t], out["rf"][t]


# supertree, source, per internal node of the supertree in pre-order: class, per-tree (shared, source, supertree, rf)
CASES = {
    "identical": (QUARTET, QUARTET, ["irrelevant", "support", "support"], (2, 2, 2, 0)),
    "contradicting": (QUARTET, "((a,c),(b,d));", ["irrelevant", "conflict", "conflict"], (0, 2, 2, 4)),
    "star": (QUARTET, "(a,b,c,d);", ["irrelevant", "permitted", "permitted"], (0, 0, 2, 2)),
    "one_taxon_in_tree": (QUARTET, "(a,(c,d));", ["irrelevant", "irrelevant", "support"], (1, 1, 1, 0)),
    "unary_chain_source": (QUARTET, "((((a,b))),(c,d));", ["irrelevant", "support", "support"], (2, 2, 2, 0)),
    "unary_root_source": ("((a,b),c);", "(((a,b),c));", ["irrelevant", "support"], (1, 1, 1, 0)),
    "polytomy_source": ("(((a,b),c),d);", "((a,b,c),d);", ["irrelevant", "support", "permitted"], (1, 1, 2, 1)),
    "two_tips": (QUARTET, "(a,b);", ["irrelevant", "irrelevant", "irrelevant"], (0, 0, 0, 0)),
    "lone_tip": (QUARTET, "a;", ["irrelevant", "irrelevant", "irrelevant"], (0, 0, 0, 0)),
    "source_taxa_missing_from_supertree": (QUARTET, "((a,x),(b,(c,d)));", ["irrelevant", "conflict", "support"],
                                           (1, 2, 2, 2)),  # fmt: skip
    "supertree_taxa_missing_from_source": ("(((a,b),e),(c,d));", "((a,b),(c,d));",
                                           ["irrelevant", "support", "support", "support"], (2, 2, 2, 0)),  # fmt: skip
    "unary_chain_supertree": ("(((a,b)),(c,d));", QUARTET, ["irrelevant", "support", "support", "support"], (2, 2, 2, 0)),
    "caterpillar_against_balanced": ("(((a,b),c),d);", QUARTET, ["irrelevant", "conflict", "support"], (1, 2, 2, 2)),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_known_answers(case):
    supertree, source, classes, rows = CASES[case]
    out = score(supertree, [source])
    for i, cls in enumerate(classes):
        got = [key for key in ("support", "conflict", "permitted", "irrelevant") if out[key][i] == 1]
        assert got == [cls], (case, i, got)
    assert per_tree(out) == rows


def test_oracle_weighted_sums_and_v():
    out = score(QUARTET, [QUARTET, "((a,c),(b,d));", "(a,b,c,d);"], [2.0, 1.0, 5.0])
    assert out["support"] == [0, 1, 1]
    assert out["conflict"] == [0, 1, 1]
    assert out["permitted"] == [0, 1, 1]
    assert out["irrelevant"] == [3, 0, 0]
    assert out["weighted_support"] == [0.0, 2.0, 2.0]
    assert out["weighted_conflict"] == [0.0, 1.0, 1.0]
    assert out["weighted_permitted"] == [0.0, 5.0, 5.0]
    assert math.isnan(out["v"][0])
    assert out["v"][1:] == [1 / 3, 1 / 3]
    assert out["rf"] == [0, 4, 2]


NAMES = ["a", "b", "c", "d"]
PARENT = np.array([-1, 0, 0, 1, 1, 2, 2], dtype=np.int32)
TAXON = np.array([-1, -1, -1, 0, 1, 2, 3], dtype=np.int32)


def test_newick_values_read_back_as_supports():
    value = np.array([0.25, 0.123456, -0.5, 9.0, 9.0, 9.0, 9.0])
    text = flat_newick_values(PARENT, TAXON, NAMES, value, digits=3)
    assert text == "((a,b)0.123,(c,d)-0.500);"
    forest = Forest.from_newick(text + "\n")
    try:
        _parent, _length, support, taxon = forest.tree_arrays(0)
        internal = support[taxon < 0]
        assert math.isnan(internal[0])  # the root carries no label
        assert sorted(internal[1:].tolist()) == [round(-0.5, 3), round(0.123456, 3)]
    finally:
        forest.close()


def test_newick_values_nan_means_no_label():
    value = np.array([np.nan, np.nan, 0.75, np.nan, np.nan, np.nan, np.nan])
    assert flat_newick_values(PARENT, TAXON, NAMES, value, digits=2) == "((a,b),(c,d)0.75);"


def test_newick_values_all_nan_is_the_plain_text():
    value = np.full(len(PARENT), np.nan)
    assert flat_newick_values(PARENT, TAXON, NAMES, value) == flat_newick(PARENT, TAXON, NAMES)
