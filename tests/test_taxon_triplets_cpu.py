"""CPU: the per-taxon triplet oracle (oracle/taxon_triplet_oracle.py) on hand-worked cases, the row/column route of
csrc/triplets.cu restated in numpy against the brute force by definition, the fields derived on the host and the TSV
that ``scs --taxon-triplets-out`` writes (no GPU is touched)."""

from __future__ import annotations

import math
from math import comb

import numpy as np
import pytest

from oracle.taxon_triplet_oracle import TAXON_FIELDS, row_column_counts, taxon_fit
from oracle.triplet_oracle import tree_fit
from spectralclustersupertree_b200.triplets import TAXON_TSV_HEADER, _taxon_fit
from spectralclustersupertree_b200.tree import PhyloNode, make_tree


def untidy_tree(names, rng: np.random.RandomState) -> PhyloNode:
    """A random rooted tree on ``names`` with polytomies and unary chains."""
    nodes = [PhyloNode(name) for name in names]
    while len(nodes) > 1:
        m = min(len(nodes), 3 if rng.rand() < 0.3 else 2)
        picked = sorted(rng.choice(len(nodes), size=m, replace=False), reverse=True)
        kids = [nodes.pop(i) for i in picked]
        node = PhyloNode("", kids)
        for _ in range(rng.randint(0, 3) if rng.rand() < 0.25 else 0):
            node = PhyloNode("", [node])
        nodes.append(node)
    return nodes[0]


def test_hand_worked_cases():
    got = taxon_fit(make_tree("((a,b),(c,d));"), [make_tree("((a,c),(b,d));")])
    assert got["agree"].tolist() == [0, 0, 0, 0] and got["contradict"].tolist() == [3, 3, 3, 3]
    got = taxon_fit(make_tree("(((a,b),c),d);"), [make_tree("(((a,b),d),c);")])
    assert got["names"] == ["a", "b", "c", "d"]
    assert got["agree"].tolist() == [2, 2, 1, 1] and got["contradict"].tolist() == [1, 1, 2, 2]
    assert got["trees"].tolist() == [1, 1, 1, 1] and got["triplets"].tolist() == [3, 3, 3, 3]


@pytest.mark.parametrize("seed", range(12))
def test_row_column_route_equals_the_brute_force(seed):
    rng = np.random.RandomState(seed)
    pool = [f"t{i}" for i in range(14)]
    s_names = list(rng.choice(pool, size=rng.randint(8, 14), replace=False))
    supertree = untidy_tree(s_names, rng)
    trees, weights = [], []
    for _ in range(6):  # taxa missing on either side, some trees sharing fewer than three taxa
        names = list(rng.choice(pool + ["x1", "x2"], size=rng.randint(2, 13), replace=False))
        trees.append(untidy_tree(names, rng))
        weights.append(float(rng.choice([0.5, 1.0, 1.0 / 3.0, 7.25])))
    brute = taxon_fit(supertree, trees, weights)
    route = taxon_fit(supertree, trees, weights, route=row_column_counts)
    for key in TAXON_FIELDS:
        assert np.array_equal(brute[key], route[key]), key
    assert brute["weighted"].tobytes() == route["weighted"].tobytes()
    # every triplet is credited to its three taxa
    per_tree = [tree_fit(supertree, t) for t in trees]
    for f, key in enumerate(("resolved_source", "resolved_supertree", "agree", "contradict")):
        assert brute[key].sum() == 3 * sum(row[1 + f] for row in per_tree), key
    assert brute["triplets"].sum() == 3 * sum(comb(row[0], 3) for row in per_tree)
    assert brute["trees"].sum() == sum(row[0] for row in per_tree if row[0] >= 3)


def test_derived_fields():
    names = ["c", "a", "b", "d"]
    per_taxon = np.array([[2, 6, 4, 5, 2, 1], [1, 3, 0, 3, 0, 0], [0, 0, 0, 0, 0, 0], [1, 3, 3, 3, 3, 0]])
    weighted = np.array([[3.0, 1.5, 0.5], [0.0, 0.0, 0.0], [0.0, 0.0, 0.0], [2.0, 2.0, 0.0]])
    fit = _taxon_fit(names, per_taxon, weighted)
    assert fit.names == ["a", "b", "c", "d"]
    assert fit.trees.tolist() == [1, 0, 2, 1]
    assert fit.unresolved.tolist() == [0, 0, 1, 0]
    assert math.isnan(fit.fit[0]) and math.isnan(fit.fit[1]) and fit.fit[2] == 0.5 and fit.fit[3] == 1.0
    assert math.isnan(fit.weighted_fit[0]) and math.isnan(fit.weighted_fit[1])
    assert fit.weighted_fit[2] == 0.5 and fit.weighted_fit[3] == 1.0


def test_tsv_formatting():
    fit = _taxon_fit(["b", "a"], np.array([[2, 6, 4, 5, 2, 1], [1, 3, 0, 3, 0, 0]]), np.zeros((2, 3)))
    assert TAXON_TSV_HEADER == "taxon\ttrees\ttriplets\tresolved_source\tresolved_supertree\tagree\tcontradict"
    assert fit.tsv() == f"{TAXON_TSV_HEADER}\na\t1\t3\t0\t3\t0\t0\nb\t2\t6\t4\t5\t2\t1\n"
