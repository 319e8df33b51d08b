"""Oracle of the triplet distances between source trees (spectralclustersupertree_b200.distances), written from the
definition: every pair is ``triplet_oracle.tree_fit`` with one tree of the pair as the supertree, which restricts both
trees to the taxa they share with ``get_sub_tree(..., ignore_missing=True, as_rooted=True)`` and classifies every
triplet from its LCA depths.  It sits beside ``pairwise_oracle``, the Robinson-Foulds oracle of the same pairs.  Test
infrastructure only (cubic in the shared taxa of each pair)."""

from __future__ import annotations

from collections.abc import Sequence

from oracle import triplet_oracle
from spectralclustersupertree_b200.tree import PhyloNode

FIELDS = ("shared_taxa", "resolved", "agree", "contradict", "distance")


def pairwise_triplets(trees: Sequence[PhyloNode]) -> dict[str, list[list[int]]]:
    """``shared_taxa``, ``resolved`` (row i: triplets resolved in tree i on the taxa it shares with tree j), ``agree``,
    ``contradict`` and ``distance`` as T x T nested lists, the diagonal included: per pair i <= j
    ``tree_fit(supertree=t_j, tree=t_i)``."""
    T = len(trees)
    out = {key: [[0] * T for _ in range(T)] for key in FIELDS}
    for i in range(T):
        for j in range(i, T):
            k, ri, rj, agree, contradict = triplet_oracle.tree_fit(supertree=trees[j], tree=trees[i])
            distance = ri + rj - 2 * agree - contradict
            for key, value, mirror in (("shared_taxa", k, k), ("resolved", ri, rj), ("agree", agree, agree),
                                       ("contradict", contradict, contradict), ("distance", distance, distance)):  # fmt: skip
                out[key][i][j] = value
                out[key][j][i] = mirror
    return out
