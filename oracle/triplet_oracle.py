"""Rooted triplet fit of a supertree against its source trees (spectralclustersupertree_b200.triplets), written from
the definition: both trees are restricted to the shared taxa X with ``get_sub_tree(X, ignore_missing=True,
as_rooted=True)``, and every triplet {a, b, c} of X is classified in each restricted tree from its three pairwise LCA
depths (ab|c when LCA(a, b) lies strictly below the other two, a fan when none does).  Vectorised over the triplets
of one fixed taxon with numpy.  Test infrastructure only (cubic in the shared taxa)."""

from __future__ import annotations

from collections.abc import Sequence

import numpy as np

from spectralclustersupertree_b200.tree import PhyloNode

FIELDS = ("shared", "resolved_source", "resolved_supertree", "agree", "contradict")


def lca_depths(tree: PhyloNode, order: Sequence[str]) -> np.ndarray:
    """[k, k] depth of the LCA of every pair of the tips named in ``order`` (the diagonal is unused)."""
    index = {name: i for i, name in enumerate(order)}
    D = np.zeros((len(order), len(order)), dtype=np.int64)
    depth = {id(tree): 0}
    for node in tree.preorder():
        for child in node.children:
            depth[id(child)] = depth[id(node)] + 1
    below: dict[int, np.ndarray] = {}
    for node in tree.postorder():
        if not node.children:
            below[id(node)] = np.array([index[node.name]])
            continue
        parts = [below.pop(id(c)) for c in node.children]
        for i, p in enumerate(parts):
            for q in parts[i + 1 :]:
                D[np.ix_(p, q)] = depth[id(node)]
                D[np.ix_(q, p)] = depth[id(node)]
        below[id(node)] = np.concatenate(parts)
    return D


def _classify(dab: np.ndarray, dac: np.ndarray, dbc: np.ndarray) -> np.ndarray:
    """0 = fan, 1 = ab|c, 2 = ac|b, 3 = bc|a."""
    return np.select([dab > dac, dac > dab, dbc > dab], [1, 2, 3], 0)


def tree_fit(supertree: PhyloNode, tree: PhyloNode) -> tuple[int, int, int, int, int]:
    """(shared, resolved_source, resolved_supertree, agree, contradict) of one source tree."""
    X = sorted(set(tree.get_tip_names()) & set(supertree.get_tip_names()))
    k = len(X)
    if k < 3:
        return k, 0, 0, 0, 0
    Dt = lca_depths(tree.get_sub_tree(X, ignore_missing=True, as_rooted=True), X)
    Ds = lca_depths(supertree.get_sub_tree(X, ignore_missing=True, as_rooted=True), X)
    out = np.zeros(4, dtype=np.int64)
    for a in range(k - 2):
        rest = np.arange(a + 1, k)
        j, l = np.triu_indices(len(rest), 1)
        b, c = rest[j], rest[l]
        ct = _classify(Dt[a, b], Dt[a, c], Dt[b, c])
        cs = _classify(Ds[a, b], Ds[a, c], Ds[b, c])
        out += [(ct > 0).sum(), (cs > 0).sum(), ((ct > 0) & (ct == cs)).sum(), ((ct > 0) & (cs > 0) & (ct != cs)).sum()]
    return (k, *(int(v) for v in out))


def triplet_fit(supertree: PhyloNode, trees: Sequence[PhyloNode], weights: Sequence[float] | None = None) -> dict:
    """Per tree: the five counts of ``tree_fit``; ``weighted_fit`` = sum w agree / sum w resolved_source in tree order."""
    if weights is None:
        weights = [1.0] * len(trees)
    out: dict = {key: [] for key in FIELDS}
    num = den = 0.0
    for tree, w in zip(trees, weights, strict=True):
        row = tree_fit(supertree, tree)
        for key, value in zip(FIELDS, row, strict=True):
            out[key].append(value)
        num += float(w) * row[3]
        den += float(w) * row[1]
    out["weighted_fit"] = num / den if den != 0 else float("nan")
    return out
