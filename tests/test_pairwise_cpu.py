"""CPU: the source-tree distance oracle (oracle/pairwise_oracle.py) on hand-worked known answers and against the clade
support oracle with every source tree used as the supertree, and the derived fields, skipped-entry convention and TSV
of ``SourceTreeDistances`` (host code only: no GPU is touched)."""

from __future__ import annotations

import math
import random

import numpy as np
import pytest

from oracle import pairwise_oracle, support_oracle
from spectralclustersupertree_b200.distances import SOURCE_RF_TSV_HEADER, _distances, source_tree_distances
from spectralclustersupertree_b200.tree import NotCompleted, make_tree

# a, b: (shared, clusters of a, clusters of b, common, rf)
CASES = {
    "quartets_contradicting": ("((a,b),(c,d));", "((a,c),(b,d));", (4, 2, 2, 0, 4)),
    "extra_taxon_drops_out": ("((a,b),c);", "((a,b),(c,d));", (3, 1, 1, 1, 0)),
    "star_against_cherry": ("(a,b,c);", "((a,b),c);", (3, 0, 1, 0, 1)),
    "both_restrict_to_the_same": ("((a,(b,e)),(c,d));", "((a,b),(c,(d,f)));", (4, 2, 2, 2, 0)),
    "unary_chain": ("(((a,b)),c);", "((a,b),c);", (3, 1, 1, 1, 0)),
    "unary_chain_against_itself": ("(((a,b)),c);", "(((a,b)),c);", (3, 1, 1, 1, 0)),
    "two_shared_taxa": ("((a,b),(c,d));", "((a,b),(x,y));", (2, 0, 0, 0, 0)),
    "nothing_shared": ("((a,b),c);", "((x,y),z);", (0, 0, 0, 0, 0)),
}


def random_tree(names, rng: random.Random):
    """A random rooted tree on ``names`` with polytomies of up to four children and unary nodes."""
    nodes = list(names)
    while len(nodes) > 1:
        k = rng.randint(2, min(4, len(nodes)))
        rng.shuffle(nodes)
        group, nodes = nodes[:k], nodes[k:]
        text = "(" + ",".join(group) + ")"
        if rng.random() < 0.2:
            text = "(" + text + ")"
        nodes.append(text)
    return make_tree(nodes[0] + ";")


def random_forest(seed: int, count: int, pool: int = 12):
    """``count`` trees on random subsets of a pool of taxa, so that taxa are missing on either side of a pair."""
    rng = random.Random(seed)
    names = [f"t{i}" for i in range(pool)]
    return [random_tree(rng.sample(names, rng.randint(2, pool)), rng) for _ in range(count)]


@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_known_answers(case):
    a, b, (k, ca, cb, both, rf) = CASES[case]
    assert pairwise_oracle.pair_counts(make_tree(a), make_tree(b)) == (k, ca, cb, both)
    out = pairwise_oracle.pairwise_rf([make_tree(a), make_tree(b)])
    assert out["rf"][0][1] == out["rf"][1][0] == rf
    assert out["clusters"][0][1] == ca and out["clusters"][1][0] == cb
    assert out["shared_taxa"][0][0] == len(make_tree(a).get_tip_names())
    assert out["rf"][0][0] == out["rf"][1][1] == 0


def test_known_answers_normalized():
    trees = [make_tree(CASES[c][i]) for c in ("quartets_contradicting", "nothing_shared") for i in range(2)]
    out = pairwise_oracle.pairwise_rf(trees)
    got = _distances(*(np.array(out[key], dtype=np.int32) for key in ("shared_taxa", "clusters", "common")),
                     np.ones(4, dtype=bool))  # fmt: skip
    assert got.normalized_rf[0, 1] == 1.0
    assert np.isnan(got.normalized_rf[2, 3]) and np.isnan(got.normalized_rf[0, 3])
    assert got.rf[2, 3] == 0 and got.shared_taxa[2, 3] == 0


def test_oracle_against_clade_support_with_each_tree_as_the_supertree():
    for seed in range(4):
        trees = random_forest(seed, 9)
        out = pairwise_oracle.pairwise_rf(trees)
        for i, supertree in enumerate(trees):
            support = support_oracle.clade_support(supertree, trees)
            for j in range(len(trees)):
                assert support["rf"][j] == out["rf"][i][j]
                assert support["shared"][j] == out["common"][i][j]
                assert support["source_clusters"][j] == out["clusters"][j][i]
                assert support["supertree_clusters"][j] == out["clusters"][i][j]


def test_derived_fields():
    # three trees: 0 and 1 share 4 taxa, 0 and 2 share 3, 1 and 2 share 2 (nothing comparable)
    shared = np.array([[5, 4, 3], [4, 4, 2], [3, 2, 3]], dtype=np.int32)
    clusters = np.array([[3, 2, 1], [2, 2, 0], [0, 0, 0]], dtype=np.int32)
    common = np.array([[3, 1, 0], [1, 2, 0], [0, 0, 0]], dtype=np.int32)
    got = _distances(shared, clusters, common, np.ones(3, dtype=bool))
    assert got.rf.tolist() == [[0, 2, 1], [2, 0, 0], [1, 0, 0]]
    assert got.normalized_rf[0, 1] == got.normalized_rf[1, 0] == 0.5
    assert got.normalized_rf[0, 2] == got.normalized_rf[2, 0] == 1.0
    assert np.isnan(got.normalized_rf[1, 2]) and np.isnan(got.normalized_rf[2, 2])
    assert got.normalized_rf[0, 0] == 0.0
    assert got.comparable.tolist() == [2, 1, 1]
    assert got.mean_normalized_rf.tolist() == [0.75, 0.5, 1.0]
    lonely = _distances(np.array([[3, 0], [0, 2]], dtype=np.int32), np.array([[1, 0], [0, 0]], dtype=np.int32),
                        np.array([[1, 0], [0, 0]], dtype=np.int32), np.ones(2, dtype=bool))  # fmt: skip
    assert lonely.comparable.tolist() == [0, 0] and np.isnan(lonely.mean_normalized_rf).all()


def test_skipped_entries():
    shared = np.array([[4, 7, 4], [7, 7, 7], [4, 7, 4]], dtype=np.int32)
    clusters = np.array([[2, 9, 2], [9, 9, 9], [2, 9, 2]], dtype=np.int32)
    common = np.array([[2, 9, 0], [9, 9, 9], [0, 9, 2]], dtype=np.int32)
    got = _distances(shared, clusters, common, np.array([True, False, True]))
    for key in ("shared_taxa", "clusters", "common", "rf"):
        matrix = getattr(got, key)
        assert (matrix[1] == -1).all() and (matrix[:, 1] == -1).all(), key
    assert np.isnan(got.normalized_rf[1]).all() and np.isnan(got.normalized_rf[:, 1]).all()
    assert got.rf[0, 2] == 4 and got.normalized_rf[0, 2] == 1.0
    assert got.comparable.tolist() == [1, -1, 1]
    assert got.mean_normalized_rf[0] == 1.0 and math.isnan(got.mean_normalized_rf[1])
    everything_skipped = source_tree_distances([NotCompleted("ERROR", "x", "failed")] * 2)
    assert everything_skipped.shared_taxa.tolist() == [[-1, -1], [-1, -1]]
    assert everything_skipped.comparable.tolist() == [-1, -1]
    assert np.isnan(everything_skipped.normalized_rf).all() and np.isnan(everything_skipped.mean_normalized_rf).all()


def test_tsv_formatting():
    shared = np.array([[4, 4, 2, 3], [4, 5, 0, 3], [2, 0, 2, 2], [3, 3, 2, 3]], dtype=np.int32)
    clusters = np.array([[2, 2, 0, 1], [1, 3, 0, 0], [0, 0, 0, 0], [1, 1, 0, 1]], dtype=np.int32)
    common = np.array([[2, 1, 0, 1], [1, 3, 0, 0], [0, 0, 0, 0], [1, 0, 0, 1]], dtype=np.int32)
    text = _distances(shared, clusters, common, np.array([True, True, True, True])).tsv()
    assert text == (f"{SOURCE_RF_TSV_HEADER}\n"
                    "0\t1\t4\t2\t1\t1\t1\n"
                    "0\t3\t3\t1\t1\t1\t0\n"
                    "1\t3\t3\t0\t1\t0\t1\n")  # fmt: skip
    assert SOURCE_RF_TSV_HEADER == "tree_a\ttree_b\tshared\tclusters_a\tclusters_b\tcommon\trf"
    skipped = _distances(shared.copy(), clusters.copy(), common.copy(), np.array([True, False, True, True])).tsv()
    assert skipped == f"{SOURCE_RF_TSV_HEADER}\n0\t3\t3\t1\t1\t1\t0\n"
