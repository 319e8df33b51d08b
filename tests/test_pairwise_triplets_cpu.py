"""CPU: the source-tree triplet distance oracle (oracle/pairwise_triplet_oracle.py) on hand-worked known answers and
against the triplet-fit oracle with every source tree used as the supertree, and the derived fields, skipped-entry
convention, int64 range and TSV of ``SourceTreeTripletDistances`` (host code only: no GPU is touched)."""

from __future__ import annotations

import math

import numpy as np
import pytest

from oracle import pairwise_triplet_oracle, triplet_oracle
from spectralclustersupertree_b200.distances import (
    SOURCE_TRIPLET_TSV_HEADER,
    _triplet_distances,
    source_tree_triplet_distances,
)
from spectralclustersupertree_b200.tree import NotCompleted, make_tree
from test_pairwise_cpu import random_forest

# a, b: (shared, resolved in a, resolved in b, agree, contradict, distance)
CASES = {
    "quartets_contradicting": ("((a,b),(c,d));", "((a,c),(b,d));", (4, 4, 4, 0, 4, 4)),
    "star_against_cherry": ("(a,b,c);", "((a,b),c);", (3, 0, 1, 0, 0, 1)),
    "extra_taxon_drops_out": ("((a,b),c);", "((a,b),(c,d));", (3, 1, 1, 1, 0, 0)),
    "unary_chain_against_itself": ("(((a,b)),c);", "(((a,b)),c);", (3, 1, 1, 1, 0, 0)),
    "unary_chain_against_cherry": ("(((a,b)),c);", "((a,b),c);", (3, 1, 1, 1, 0, 0)),
    "fan_of_four_against_caterpillar": ("(a,b,c,d);", "(((a,b),c),d);", (4, 0, 4, 0, 0, 4)),
    "two_shared_taxa": ("((a,b),(c,d));", "((a,b),(x,y));", (2, 0, 0, 0, 0, 0)),
    "nothing_shared": ("((a,b),c);", "((x,y),z);", (0, 0, 0, 0, 0, 0)),
}


def dense(out: dict) -> list[np.ndarray]:
    return [np.array(out[key], dtype=dtype) for key, dtype in
            (("shared_taxa", np.int32), ("resolved", np.int64), ("agree", np.int64), ("contradict", np.int64))]  # fmt: skip


@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_known_answers(case):
    a, b, (k, ra, rb, agree, contradict, distance) = CASES[case]
    out = pairwise_triplet_oracle.pairwise_triplets([make_tree(a), make_tree(b)])
    assert out["shared_taxa"][0][1] == out["shared_taxa"][1][0] == k
    assert out["resolved"][0][1] == ra and out["resolved"][1][0] == rb
    assert out["agree"][0][1] == out["agree"][1][0] == agree
    assert out["contradict"][0][1] == out["contradict"][1][0] == contradict
    assert out["distance"][0][1] == out["distance"][1][0] == distance
    for t in range(2):  # the diagonal: a tree against itself
        assert out["shared_taxa"][t][t] == len(make_tree((a, b)[t]).get_tip_names())
        assert out["resolved"][t][t] == out["agree"][t][t] and out["contradict"][t][t] == 0
        assert out["distance"][t][t] == 0
    got = _triplet_distances(*dense(out), np.ones(2, dtype=bool))
    if k >= 3:
        assert got.normalized_distance[0, 1] == distance / math.comb(k, 3)
    else:
        assert np.isnan(got.normalized_distance[0, 1]) and got.distance[0, 1] == 0


def test_known_answer_normalized():
    out = pairwise_triplet_oracle.pairwise_triplets([make_tree(s) for s in CASES["quartets_contradicting"][:2]])
    assert _triplet_distances(*dense(out), np.ones(2, dtype=bool)).normalized_distance[0, 1] == 1.0


def test_oracle_against_triplet_fit_with_each_tree_as_the_supertree():
    for seed in range(4):
        trees = random_forest(seed, 9)
        out = pairwise_triplet_oracle.pairwise_triplets(trees)
        for i, supertree in enumerate(trees):
            fit = triplet_oracle.triplet_fit(supertree, trees)
            for j in range(len(trees)):
                assert fit["shared"][j] == out["shared_taxa"][i][j]
                assert fit["resolved_source"][j] == out["resolved"][j][i]
                assert fit["resolved_supertree"][j] == out["resolved"][i][j]
                assert fit["agree"][j] == out["agree"][i][j]
                assert fit["contradict"][j] == out["contradict"][i][j]
        assert any(out["contradict"][i][j] for i in range(9) for j in range(9))


def test_derived_fields():
    # three trees: 0 and 1 share 4 taxa, 0 and 2 share 3, 1 and 2 share 2 (nothing comparable)
    shared = np.array([[5, 4, 3], [4, 4, 2], [3, 2, 3]], dtype=np.int32)
    resolved = np.array([[10, 4, 1], [3, 4, 0], [1, 0, 1]], dtype=np.int64)
    agree = np.array([[10, 2, 1], [2, 4, 0], [1, 0, 1]], dtype=np.int64)
    contradict = np.array([[0, 1, 0], [1, 0, 0], [0, 0, 0]], dtype=np.int64)
    got = _triplet_distances(shared, resolved, agree, contradict, np.ones(3, dtype=bool))
    assert got.distance.tolist() == [[0, 2, 0], [2, 0, 0], [0, 0, 0]]
    assert got.normalized_distance[0, 1] == got.normalized_distance[1, 0] == 0.5
    assert got.normalized_distance[0, 2] == 0.0 and got.normalized_distance[0, 0] == 0.0
    assert np.isnan(got.normalized_distance[1, 2]) and np.isnan(got.normalized_distance[2, 1])
    assert got.comparable.tolist() == [2, 1, 1]
    assert got.mean_normalized_distance.tolist() == [0.25, 0.5, 0.0]
    assert got.distance.dtype == np.int64 and got.normalized_distance.dtype == np.float64
    lonely = _triplet_distances(np.array([[3, 0], [0, 2]], dtype=np.int32), np.array([[1, 0], [0, 0]], dtype=np.int64),
                                np.array([[1, 0], [0, 0]], dtype=np.int64), np.zeros((2, 2), dtype=np.int64),
                                np.ones(2, dtype=bool))  # fmt: skip
    assert lonely.comparable.tolist() == [0, 0] and np.isnan(lonely.mean_normalized_distance).all()


def test_counts_above_int32():
    k = 20000
    full = math.comb(k, 3)
    assert full > 2**31
    shared = np.full((2, 2), k, dtype=np.int32)
    resolved = np.full((2, 2), full, dtype=np.int64)
    reversed_pair = _triplet_distances(shared.copy(), resolved.copy(), np.array([[full, 0], [0, full]]),
                                       np.array([[0, full], [full, 0]]), np.ones(2, dtype=bool))  # fmt: skip
    assert reversed_pair.distance.tolist() == [[0, full], [full, 0]]
    assert reversed_pair.normalized_distance[0, 1] == 1.0
    same = _triplet_distances(shared.copy(), resolved.copy(), resolved.copy(), np.zeros((2, 2), dtype=np.int64),
                              np.ones(2, dtype=bool))  # fmt: skip
    assert (same.distance == 0).all() and (same.normalized_distance == 0.0).all()
    assert same.tsv() == f"{SOURCE_TRIPLET_TSV_HEADER}\n0\t1\t{k}\t{full}\t{full}\t{full}\t0\t0\n"


def test_skipped_entries():
    shared = np.array([[4, 7, 4], [7, 7, 7], [4, 7, 4]], dtype=np.int32)
    resolved = np.array([[4, 9, 4], [9, 9, 9], [4, 9, 4]], dtype=np.int64)
    agree = np.array([[4, 9, 0], [9, 9, 9], [0, 9, 4]], dtype=np.int64)
    contradict = np.array([[0, 9, 4], [9, 0, 9], [4, 9, 0]], dtype=np.int64)
    got = _triplet_distances(shared, resolved, agree, contradict, np.array([True, False, True]))
    for key in ("shared_taxa", "resolved", "agree", "contradict", "distance"):
        matrix = getattr(got, key)
        assert (matrix[1] == -1).all() and (matrix[:, 1] == -1).all(), key
    assert np.isnan(got.normalized_distance[1]).all() and np.isnan(got.normalized_distance[:, 1]).all()
    assert got.distance[0, 2] == 4 and got.normalized_distance[0, 2] == 1.0
    assert got.comparable.tolist() == [1, -1, 1]
    assert got.mean_normalized_distance[0] == 1.0 and math.isnan(got.mean_normalized_distance[1])
    everything_skipped = source_tree_triplet_distances([NotCompleted("ERROR", "x", "failed")] * 2)
    assert everything_skipped.shared_taxa.tolist() == [[-1, -1], [-1, -1]]
    assert everything_skipped.resolved.dtype == np.int64
    assert everything_skipped.comparable.tolist() == [-1, -1]
    assert np.isnan(everything_skipped.normalized_distance).all()
    assert np.isnan(everything_skipped.mean_normalized_distance).all()


def test_tsv_formatting():
    shared = np.array([[4, 4, 2, 3], [4, 5, 0, 3], [2, 0, 2, 2], [3, 3, 2, 3]], dtype=np.int32)
    resolved = np.array([[4, 4, 0, 1], [3, 10, 0, 0], [0, 0, 0, 0], [1, 1, 0, 1]], dtype=np.int64)
    agree = np.array([[4, 2, 0, 1], [2, 10, 0, 0], [0, 0, 0, 0], [1, 0, 0, 1]], dtype=np.int64)
    contradict = np.array([[0, 1, 0, 0], [1, 0, 0, 0], [0, 0, 0, 0], [0, 0, 0, 0]], dtype=np.int64)
    text = _triplet_distances(shared, resolved, agree, contradict, np.array([True, True, True, True])).tsv()
    assert text == (f"{SOURCE_TRIPLET_TSV_HEADER}\n"
                    "0\t1\t4\t4\t3\t2\t1\t2\n"
                    "0\t3\t3\t1\t1\t1\t0\t0\n"
                    "1\t3\t3\t0\t1\t0\t0\t1\n")  # fmt: skip
    assert SOURCE_TRIPLET_TSV_HEADER == "tree_a\ttree_b\tshared\tresolved_a\tresolved_b\tagree\tcontradict\tdistance"
    skipped = _triplet_distances(shared.copy(), resolved.copy(), agree.copy(), contradict.copy(),
                                 np.array([True, False, True, True])).tsv()  # fmt: skip
    assert skipped == f"{SOURCE_TRIPLET_TSV_HEADER}\n0\t3\t3\t1\t1\t1\t0\t0\n"
