"""Oracle of the agreement-subtree fit of a supertree (spectralclustersupertree_b200.mast), written from the
definitions: the source tree and the supertree are both restricted to their shared taxa X with ``get_sub_tree(...,
ignore_missing=True, as_rooted=True)``, and the size of their maximum agreement subtree follows the recurrence of
Steel & Warnow (1993), the maximum-weight matching of two child lists taken by
``scipy.optimize.linear_sum_assignment``.  ``mast_brute`` tries every subset of X instead (k <= 8 or so).  Test
infrastructure only (slow)."""

from __future__ import annotations

import itertools
from collections.abc import Sequence

import numpy as np
from scipy.optimize import linear_sum_assignment

from spectralclustersupertree_b200.tree import PhyloNode


def restrict(tree: PhyloNode, X: frozenset) -> PhyloNode:
    return tree.get_sub_tree(X, ignore_missing=True, as_rooted=True)


def _nodes(tree: PhyloNode) -> tuple[list[PhyloNode], dict[int, int], list[frozenset]]:
    order = list(tree.postorder())
    index = {id(node): i for i, node in enumerate(order)}
    below: list[frozenset] = []
    for node in order:
        below.append(frozenset((node.name,)) if not node.children else
                     frozenset().union(*(below[index[id(c)]] for c in node.children)))  # fmt: skip
    return order, index, below


def mast_restricted(a: PhyloNode, b: PhyloNode) -> int:
    """The MAST size of two rooted trees on the same taxa (any degree; unary nodes pass their child through)."""
    na, ia, la = _nodes(a)
    nb, ib, lb = _nodes(b)
    ca = [[ia[id(c)] for c in node.children] for node in na]
    cb = [[ib[id(c)] for c in node.children] for node in nb]
    table = [[0] * len(nb) for _ in na]
    for u in range(len(na)):
        row = table[u]
        for v in range(len(nb)):
            if not ca[u] or not cb[v]:  # a leaf against anything: is it in the other side's leaf set
                leaf, other = (la[u], lb[v]) if not ca[u] else (lb[v], la[u])
                row[v] = int(next(iter(leaf)) in other)
                continue
            best = max(max(table[x][v] for x in ca[u]), max(row[y] for y in cb[v]))
            weights = [[table[x][y] for y in cb[v]] for x in ca[u]]
            if len(weights) == 2 and len(cb[v]) == 2:  # two by two: the better of the two matchings
                matched = max(weights[0][0] + weights[1][1], weights[0][1] + weights[1][0])
            else:
                w = np.array(weights, dtype=np.int64)
                rows, cols = linear_sum_assignment(w, maximize=True)
                matched = int(w[rows, cols].sum())
            row[v] = max(best, matched)
    return table[len(na) - 1][len(nb) - 1]


def same_rooted_tree(a: PhyloNode, b: PhyloNode) -> bool:
    return set(a.clade_sets()) == set(b.clade_sets())


def mast_brute(source: PhyloNode, supertree: PhyloNode) -> int:
    """The largest Y in the shared taxa on which both restrictions are the same rooted tree, by trying every subset
    from the largest down."""
    X = sorted(frozenset(source.get_tip_names()) & frozenset(supertree.get_tip_names()))
    for size in range(len(X), 2, -1):
        for Y in itertools.combinations(X, size):
            if same_rooted_tree(restrict(source, frozenset(Y)), restrict(supertree, frozenset(Y))):
                return size
    return min(len(X), 2)


def tree_fit(supertree: PhyloNode, tree: PhyloNode) -> tuple[int, int]:
    """(shared, agreement) of one source tree."""
    X = frozenset(tree.get_tip_names()) & frozenset(supertree.get_tip_names())
    if len(X) <= 2:
        return len(X), len(X)
    return len(X), mast_restricted(restrict(tree, X), restrict(supertree, X))


def mast_fit(supertree: PhyloNode, trees: Sequence[PhyloNode], weights: Sequence[float] | None = None) -> dict:
    """Per tree: shared, agreement, pruned; and weighted_pruned = sum_t w_t pruned_t in tree order."""
    if weights is None:
        weights = [1.0] * len(trees)
    out = {"shared": [], "agreement": [], "pruned": []}
    weighted = 0.0
    for tree, w in zip(trees, weights, strict=True):
        k, m = tree_fit(supertree, tree)
        out["shared"].append(k)
        out["agreement"].append(m)
        out["pruned"].append(k - m)
        weighted += float(w) * (k - m)
    return {**out, "weighted_pruned": weighted}
