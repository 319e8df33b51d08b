"""Set-based oracle of the distances between source trees (spectralclustersupertree_b200.distances), written from the
definitions, literally: every pair of trees is restricted to the taxa it shares with ``get_sub_tree(...,
ignore_missing=True, as_rooted=True)`` and every cluster is a frozenset of names.  Test infrastructure only (one
restriction per pair and side)."""

from __future__ import annotations

from collections.abc import Sequence

from spectralclustersupertree_b200.tree import PhyloNode


def restricted_clusters(tree: PhyloNode, X: frozenset) -> set[frozenset]:
    """The non-trivial clusters (2 <= |c| < |X|) of ``tree`` restricted to ``X``; none when |X| < 3."""
    if len(X) < 3:
        return set()
    restricted = tree.get_sub_tree(X, ignore_missing=True, as_rooted=True)
    return {c for c in restricted.clade_sets() if 2 <= len(c) < len(X)}


def pair_counts(a: PhyloNode, b: PhyloNode) -> tuple[int, int, int, int]:
    """(k, |C_a|, |C_b|, |C_a & C_b|) for the pair restricted to the taxa it shares."""
    X = frozenset(a.get_tip_names()) & frozenset(b.get_tip_names())
    ca, cb = restricted_clusters(a, X), restricted_clusters(b, X)
    return len(X), len(ca), len(cb), len(ca & cb)


def pairwise_rf(trees: Sequence[PhyloNode]) -> dict[str, list[list[int]]]:
    """``shared_taxa``, ``clusters`` (row i: tree i's clusters on the taxa it shares with tree j), ``common`` and
    ``rf`` as T x T nested lists, the diagonal included."""
    T = len(trees)
    out = {key: [[0] * T for _ in range(T)] for key in ("shared_taxa", "clusters", "common", "rf")}
    for i in range(T):
        for j in range(i, T):
            k, ci, cj, both = pair_counts(trees[i], trees[j])
            for key, value, mirror in (("shared_taxa", k, k), ("clusters", ci, cj), ("common", both, both),
                                       ("rf", ci + cj - 2 * both, ci + cj - 2 * both)):  # fmt: skip
                out[key][i][j] = value
                out[key][j][i] = mirror
    return out
