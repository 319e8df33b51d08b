"""Set-based oracle of the clade support of a supertree (spectralclustersupertree_b200.support), written from the
definitions, literally: every source tree is restricted with ``get_sub_tree(..., ignore_missing=True,
as_rooted=True)`` and every clade is a frozenset of names.  Test infrastructure only (quadratic and slow)."""

from __future__ import annotations

import math
from collections.abc import Sequence

from spectralclustersupertree_b200.tree import PhyloNode

SUPPORT, CONFLICT, PERMITTED, IRRELEVANT = "support", "conflict", "permitted", "irrelevant"


def _below(tree: PhyloNode) -> dict[int, frozenset[str]]:
    below: dict[int, frozenset[str]] = {}
    for node in tree.postorder():
        if not node.children:
            below[id(node)] = frozenset((node.name,))
        else:
            below[id(node)] = frozenset().union(*(below[id(c)] for c in node.children))
    return below


def classify(A: frozenset, X: frozenset, clusters: set[frozenset], containing: dict[str, list[frozenset]]) -> str:
    """The class of clade A (already restricted to X) against the non-trivial clusters of a tree on X;
    ``containing[x]`` lists the clusters that hold x (only those can meet A)."""
    if len(A) < 2 or len(A) == len(X):
        return IRRELEVANT
    if A in clusters:
        return SUPPORT
    if any(A & B and A - B and B - A for x in A for B in containing[x]):
        return CONFLICT
    return PERMITTED


def clade_support(supertree: PhyloNode, trees: Sequence[PhyloNode], weights: Sequence[float] | None = None) -> dict:
    """Per internal node of ``supertree`` (pre-order, root first): counts and weighted sums of the four classes and V;
    per tree: shared, source_clusters, supertree_clusters, rf."""
    if weights is None:
        weights = [1.0] * len(trees)
    below = _below(supertree)
    internal = [node for node in supertree.preorder() if node.children]
    s_tips = frozenset(below[id(supertree)])
    out = {key: [0] * len(internal) for key in (SUPPORT, CONFLICT, PERMITTED, IRRELEVANT)}
    wsum = {key: [0.0] * len(internal) for key in (SUPPORT, CONFLICT, PERMITTED)}
    per_tree = {"shared": [], "source_clusters": [], "supertree_clusters": [], "rf": []}
    for tree, w in zip(trees, weights, strict=True):
        X = frozenset(tree.get_tip_names()) & s_tips
        if len(X) < 2:
            clusters: set[frozenset] = set()
        else:
            restricted = tree.get_sub_tree(X, ignore_missing=True, as_rooted=True)
            clusters = {c for c in restricted.clade_sets() if 2 <= len(c) < len(X)}
        containing: dict[str, list[frozenset]] = {x: [] for x in X}
        for B in clusters:
            for x in B:
                containing[x].append(B)
        s_clusters = set()
        for i, node in enumerate(internal):
            A = below[id(node)] & X
            cls = classify(A, X, clusters, containing)
            out[cls][i] += 1
            if cls != IRRELEVANT:
                wsum[cls][i] += float(w)
                s_clusters.add(A)
        shared = len(s_clusters & clusters)
        per_tree["shared"].append(shared)
        per_tree["source_clusters"].append(len(clusters))
        per_tree["supertree_clusters"].append(len(s_clusters))
        per_tree["rf"].append(len(clusters) + len(s_clusters) - 2 * shared)
    v = []
    for ws, wc in zip(wsum[SUPPORT], wsum[CONFLICT], strict=True):
        v.append((ws - wc) / (ws + wc) if ws + wc != 0 else math.nan)
    return {
        "support": out[SUPPORT], "conflict": out[CONFLICT], "permitted": out[PERMITTED], "irrelevant": out[IRRELEVANT],
        "weighted_support": wsum[SUPPORT], "weighted_conflict": wsum[CONFLICT], "weighted_permitted": wsum[PERMITTED],
        "v": v, **per_tree,
    }  # fmt: skip
