"""Oracle of the MRP score of a supertree (spectralclustersupertree_b200.mrp), written from the definitions: every
source tree is restricted with ``get_sub_tree(..., ignore_missing=True, as_rooted=True)``, its non-trivial clusters
are frozensets of names (as in ``support_oracle``), and each is one binary character whose length is found by
Hartigan's pass on the supertree with the other tips missing and an all-0 outgroup above the root.  ``route="s'"``
runs the same pass on the supertree restricted to the shared taxa instead, and ``brute_length`` minimises over every
assignment of internal states.  Test infrastructure only (slow)."""

from __future__ import annotations

import itertools
from collections.abc import Sequence

from spectralclustersupertree_b200.tree import PhyloNode

BOTH = frozenset((0, 1))


def characters(supertree_tips: frozenset, tree: PhyloNode) -> tuple[frozenset, list[frozenset]]:
    """X_t and the characters of ``tree``: the clusters c of t restricted to X_t with 2 <= |c| < |X_t|."""
    X = frozenset(tree.get_tip_names()) & supertree_tips
    if len(X) < 3:
        return X, []
    restricted = tree.get_sub_tree(X, ignore_missing=True, as_rooted=True)
    return X, sorted((c for c in restricted.clade_sets() if 2 <= len(c) < len(X)), key=sorted)


def hartigan_length(tree: PhyloNode, ones: frozenset, zeros: frozenset) -> int:
    """Hartigan's length of the character (1 on ``ones``, 0 on ``zeros``, missing on the other tips) on ``tree``,
    polytomies hard, unary nodes passing their child's set up, with 0 fixed above the root."""
    state: dict[int, frozenset] = {}
    cost = 0
    for node in tree.postorder():
        if not node.children:
            state[id(node)] = frozenset((1,)) if node.name in ones else frozenset((0,)) if node.name in zeros else BOTH
            continue
        n = [sum(s in state[id(c)] for c in node.children) for s in (0, 1)]
        best = max(n)
        state[id(node)] = frozenset(s for s in (0, 1) if n[s] == best)
        cost += len(node.children) - best
    return cost + (0 not in state[id(tree)])


def brute_length(tree: PhyloNode, ones: frozenset, zeros: frozenset) -> int:
    """The minimum number of changes over all internal state assignments, the state above the root being 0
    (exponential: trees of up to about 10 internal nodes)."""
    internal = [node for node in tree.preorder() if node.children]
    best = None
    for bits in itertools.product((0, 1), repeat=len(internal)):
        at = {id(node): b for node, b in zip(internal, bits, strict=True)}
        changes = at[id(tree)] != 0
        for node in internal:
            for child in node.children:
                if child.children:
                    changes += at[id(child)] != at[id(node)]
                elif child.name in ones or child.name in zeros:
                    changes += (child.name in ones) != at[id(node)]
        best = changes if best is None else min(best, changes)
    return int(best)


def character_lengths(supertree: PhyloNode, tree: PhyloNode, route: str = "S") -> tuple[int, list[int]]:
    """k = |X_t| and the length of every character of ``tree`` on ``supertree`` (``route="S"``) or on the supertree
    restricted to X_t (``route="s'"``)."""
    X, chars = characters(frozenset(supertree.get_tip_names()), tree)
    if not chars:
        return len(X), []
    on = supertree if route == "S" else supertree.get_sub_tree(X, ignore_missing=True, as_rooted=True)
    return len(X), [hartigan_length(on, c, X - c) for c in chars]


def tree_score(supertree: PhyloNode, tree: PhyloNode, route: str = "S") -> tuple[int, int, int, int]:
    """(shared, characters, steps, exact) of one source tree."""
    k, lengths = character_lengths(supertree, tree, route)
    return k, len(lengths), sum(lengths), sum(length == 1 for length in lengths)


def mrp_score(supertree: PhyloNode, trees: Sequence[PhyloNode], weights: Sequence[float] | None = None,
              route: str = "S") -> dict:  # fmt: skip
    """Per tree: shared, characters, steps, exact; and weighted_steps = sum_t w_t steps_t in tree order."""
    if weights is None:
        weights = [1.0] * len(trees)
    out = {"shared": [], "characters": [], "steps": [], "exact": []}
    weighted = 0.0
    for tree, w in zip(trees, weights, strict=True):
        for key, value in zip(out, tree_score(supertree, tree, route), strict=True):
            out[key].append(value)
        weighted += float(w) * out["steps"][-1]
    return {**out, "weighted_steps": weighted}
