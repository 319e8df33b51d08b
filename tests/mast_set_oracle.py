"""Oracle of the agreement sets of ``spectralclustersupertree_b200.mast.mast_taxa``, on top of the agreement-subtree
oracle (oracle/mast_oracle.py): a CPU traceback of its table, every maximum set by brute force, a check that a taxon
set is a maximum agreement set, and the per-taxon counts of given node states.  Test infrastructure only (slow)."""

from __future__ import annotations

import itertools

import numpy as np
from scipy.optimize import linear_sum_assignment

from oracle.mast_oracle import _nodes, restrict, same_rooted_tree, tree_fit
from spectralclustersupertree_b200.tree import PhyloNode


def _shared(tree: PhyloNode, supertree: PhyloNode) -> frozenset:
    return frozenset(tree.get_tip_names()) & frozenset(supertree.get_tip_names())


def agreement_set(tree: PhyloNode, supertree: PhyloNode) -> frozenset:
    """One maximum agreement set of ``tree`` and ``supertree`` on their shared taxa: the table of ``mast_restricted``
    read back from the roots.  A cell descends into a child cell of the same value, else into every matched pair of
    positive weight of a maximum-weight matching of the children (its tie rule may differ from the GPU's)."""
    X = _shared(tree, supertree)
    if len(X) <= 2:
        return X
    a, b = restrict(tree, X), restrict(supertree, X)
    na, ia, la = _nodes(a)
    nb, ib, lb = _nodes(b)
    ca = [[ia[id(c)] for c in node.children] for node in na]
    cb = [[ib[id(c)] for c in node.children] for node in nb]
    table = [[0] * len(nb) for _ in na]
    matching: dict[tuple[int, int], list[tuple[int, int]]] = {}
    for u in range(len(na)):
        for v in range(len(nb)):
            if not ca[u] or not cb[v]:
                leaf, other = (la[u], lb[v]) if not ca[u] else (lb[v], la[u])
                table[u][v] = int(next(iter(leaf)) in other)
                continue
            w = np.array([[table[x][y] for y in cb[v]] for x in ca[u]], dtype=np.int64)
            rows, cols = linear_sum_assignment(w, maximize=True)
            matching[u, v] = [(ca[u][i], cb[v][j]) for i, j in zip(rows, cols, strict=True) if w[i, j] > 0]
            best = max(max(table[x][v] for x in ca[u]), max(table[u][y] for y in cb[v]))
            table[u][v] = max(best, int(w[rows, cols].sum()))
    kept: set = set()
    stack = [(len(na) - 1, len(nb) - 1)]
    while stack:
        u, v = stack.pop()
        m = table[u][v]
        if not ca[u] or not cb[v]:
            kept |= la[u] if not ca[u] else lb[v]
            continue
        down = [(x, v) for x in ca[u] if table[x][v] == m] + [(u, y) for y in cb[v] if table[u][y] == m]
        stack.extend(down[:1] if down else matching[u, v])
    return frozenset(kept)


def maximum_sets(tree: PhyloNode, supertree: PhyloNode) -> list[frozenset]:
    """Every maximum agreement set of the two trees on their shared taxa, by trying every subset from the largest down
    (k <= 9 or so)."""
    X = sorted(_shared(tree, supertree))
    if len(X) <= 2:
        return [frozenset(X)]
    for size in range(len(X), 2, -1):
        found = [frozenset(Y) for Y in itertools.combinations(X, size)
                 if same_rooted_tree(restrict(tree, frozenset(Y)), restrict(supertree, frozenset(Y)))]  # fmt: skip
        if found:
            return found
    return [frozenset(Y) for Y in itertools.combinations(X, 2)]


def is_agreement_set(tree: PhyloNode, supertree: PhyloNode, Y, size: int | None = None) -> bool:
    """Y lies in the shared taxa, has the MAST size (``size`` when the caller knows it, else the recurrence's), and
    both trees restricted to Y are the same rooted tree."""
    Y = frozenset(Y)
    X = _shared(tree, supertree)
    if size is None:
        size = tree_fit(supertree, tree)[1]
    if not Y <= X or len(Y) != size:
        return False
    return len(Y) <= 2 or same_rooted_tree(restrict(tree, Y), restrict(supertree, Y))


def taxon_counts(tip_state, node_taxon, node_offsets, weights, num_taxa: int) -> tuple[np.ndarray, np.ndarray]:
    """Per taxon id, from the per-node states of the agreement sets (1 kept, 0 dropped, -1 neither): [num_taxa, 2] the
    trees sharing it and those dropping it, and [num_taxa] the weights of the dropping trees added in tree order."""
    per_taxon = np.zeros((num_taxa, 2), dtype=np.int64)
    weighted = np.zeros(num_taxa, dtype=np.float64)
    for t in range(len(node_offsets) - 1):
        for i in range(int(node_offsets[t]), int(node_offsets[t + 1])):
            if tip_state[i] < 0:
                continue
            x = int(node_taxon[i])
            per_taxon[x, 0] += 1
            if tip_state[i] == 0:
                per_taxon[x, 1] += 1
                weighted[x] = weighted[x] + float(weights[t])
    return per_taxon, weighted
