"""CPU: the agreement-set oracle (tests/mast_set_oracle.py) against every maximum set found by brute force, and the
per-tree and per-taxon fields, skipped entries, weights, identities and TSV of ``MastTaxa`` from hand-made node
states (host code only: no GPU is touched)."""

from __future__ import annotations

import math

import numpy as np

import mast_set_oracle
from oracle import mast_oracle
from spectralclustersupertree_b200.mast import MAST_TAXA_TSV_HEADER, _fit, _taxa
from spectralclustersupertree_b200.tree import make_tree
from test_mast_cpu import random_pairs


def test_agreement_set_is_one_of_the_maximum_sets():
    checked = 0
    for S, t in random_pairs(5, 300):
        Y = mast_set_oracle.agreement_set(t, S)
        sets = mast_set_oracle.maximum_sets(t, S)
        assert Y in sets, (S.get_newick(), t.get_newick(), sorted(Y))
        assert mast_set_oracle.is_agreement_set(t, S, Y)
        assert len(Y) == mast_oracle.tree_fit(S, t)[1]
        checked += len(sets) > 1
    assert checked > 50  # pairs with more than one maximum set


def test_is_agreement_set_rejects():
    S, t = make_tree("(((a,b),c),(d,e));"), make_tree("(((a,c),b),(d,e));")
    assert mast_oracle.tree_fit(S, t) == (5, 4)
    assert mast_set_oracle.is_agreement_set(t, S, {"a", "c", "d", "e"})
    assert not mast_set_oracle.is_agreement_set(t, S, {"a", "b", "c", "d"})  # disagree on a, b, c
    assert not mast_set_oracle.is_agreement_set(t, S, {"a", "d", "e"})  # too small
    assert not mast_set_oracle.is_agreement_set(t, S, {"a", "c", "d", "x"})  # not shared
    assert sorted(map(sorted, mast_set_oracle.maximum_sets(t, S))) == [["a", "b", "d", "e"], ["a", "c", "d", "e"],
                                                                   ["b", "c", "d", "e"]]  # fmt: skip


def forest_states():
    """Three kept trees of a five-taxon problem (ids: a0 b1 c2 d3 x4; the supertree lacks x), as node arrays in
    pre-order with their states, and the per-tree counts they imply."""
    # tree 0: ((a,b),(c,d)) keeps a, b, d; tree 1: (a,x) keeps a; tree 2: lone tip c
    node_taxon = np.array([-1, -1, 0, 1, -1, 2, 3, -1, 0, 4, 2], dtype=np.int32)
    tip_state = np.array([-1, -1, 1, 1, -1, 0, 1, -1, 1, -1, 1], dtype=np.int8)
    offsets = np.array([0, 7, 10, 11], dtype=np.int64)
    per_tree = np.array([[4, 3], [1, 1], [1, 1]], dtype=np.int64)
    return node_taxon, tip_state, offsets, per_tree


def test_taxa_fields_with_skipped_entries_and_weights():
    names = ["a", "b", "c", "d", "x"]
    node_taxon, tip_state, offsets, per_tree = forest_states()
    tree_weights = [0.5, 9.0, 2.0, 0.25]  # input tree 1 is skipped
    kept = [0, 2, 3]
    kept_weights = [tree_weights[t] for t in kept]
    per_taxon, weighted = mast_set_oracle.taxon_counts(tip_state, node_taxon, offsets, kept_weights, 5)
    assert per_taxon.tolist() == [[2, 0], [1, 0], [2, 1], [1, 0], [0, 0]]
    assert weighted.tolist() == [0.0, 0.0, 0.5, 0.0, 0.0]
    got = _taxa(names, [3, 0, 2, 1], per_tree, tip_state, node_taxon, offsets, per_taxon, weighted, kept, 4)
    assert got.shared.tolist() == [4, -1, 1, 1] and got.agreement.tolist() == [3, -1, 1, 1]
    assert got.pruned.tolist() == [1, -1, 0, 0]
    assert got.pruned_taxa == [("c",), None, (), ()]
    assert got.names == ["a", "b", "c", "d"]
    assert got.trees.tolist() == [2, 1, 2, 1] and got.taxon_pruned.tolist() == [0, 0, 1, 0]
    assert got.weighted_pruned.tolist() == [0.0, 0.0, 0.5, 0.0]
    assert got.fraction.tolist() == [0.0, 0.0, 0.5, 0.0]
    fit = _fit(np.stack([got.shared, got.agreement], axis=1), tree_weights, kept)
    assert got.trees.sum() == fit.total_shared and got.taxon_pruned.sum() == fit.total_pruned
    assert got.tsv() == f"{MAST_TAXA_TSV_HEADER}\na\t2\t0\nb\t1\t0\nc\t2\t1\nd\t1\t0\n"
    assert MAST_TAXA_TSV_HEADER == "taxon\ttrees\tpruned"


def test_taxa_weights_add_in_tree_order_and_unshared_tips_are_nan():
    # four cherries (a,b), two of which drop b; a supertree tip z that no tree has
    names = ["a", "b", "z"]
    node_taxon = np.tile(np.array([-1, 0, 1], dtype=np.int32), 4)
    tip_state = np.array([-1, 1, 1, -1, 1, 0, -1, 1, 1, -1, 1, 0], dtype=np.int8)
    offsets = np.arange(0, 13, 3, dtype=np.int64)
    weights = [0.1, 0.2, 1e16, 0.3]
    per_taxon, weighted = mast_set_oracle.taxon_counts(tip_state, node_taxon, offsets, weights, 3)
    assert weighted[1] == (0.0 + 0.2) + 0.3 and per_taxon[1].tolist() == [4, 2]
    per_tree = np.array([[2, 2], [2, 1], [2, 2], [2, 1]], dtype=np.int64)
    got = _taxa(names, [2, 1, 0], per_tree, tip_state, node_taxon, offsets, per_taxon, weighted, range(4), 4)
    assert got.names == ["a", "b", "z"] and got.trees.tolist() == [4, 4, 0]
    assert got.fraction[1] == 0.5 and math.isnan(got.fraction[2])
    assert got.pruned_taxa == [(), ("b",), (), ("b",)]


def test_taxa_with_nothing_kept():
    got = _taxa(["a"], [0], np.zeros((0, 2)), np.zeros(0), np.zeros(0), np.zeros(1), np.zeros((1, 2)), np.zeros(1),
                [], 2)  # fmt: skip
    assert got.shared.tolist() == [-1, -1] and got.pruned_taxa == [None, None]
    assert got.trees.tolist() == [0] and math.isnan(got.fraction[0])
