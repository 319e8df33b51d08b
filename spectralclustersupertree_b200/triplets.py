"""Rooted triplet fit of a supertree against its source trees.

For every source tree t, let X_t be the taxa it shares with the supertree S.  Both trees are restricted to X_t (as
the recursion restricts trees), and every three-taxon statement of X_t is compared: a triplet {a, b, c} is resolved
as ab|c in a tree when LCA(a, b) lies strictly below LCA(a, b, c), and is a fan otherwise.  Per source tree:

==================  ======================================================================
shared              k = |X_t|
resolved_source     triplets of X_t resolved in the restricted source tree
resolved_supertree  triplets of X_t resolved in the restricted supertree
agree               resolved in both, the same way
contradict          resolved in both, differently
unresolved          resolved_source - agree - contradict: source triplets S shows as fans
fit                 agree / resolved_source (NaN where no triplet is resolved)
==================  ======================================================================

``weighted_fit`` = sum_t w_t agree_t / sum_t w_t resolved_source_t, summed in tree order.  The counts run on the
GPU (``scs_supertree_triplets``, csrc/triplets.cu) in O(k^2 log D) per tree for a supertree of depth D, and are
exact.
"""

from __future__ import annotations

from collections.abc import Sequence
from dataclasses import dataclass

import numpy as np

from .engine import Engine, Forest, default_engine
from .scs import _is_not_completed
from .support import _flat_supertree
from .tree import PhyloNode

TSV_HEADER = "tree\tshared\tresolved_source\tresolved_supertree\tagree\tcontradict"


@dataclass
class TripletFit:
    """Per input tree (-1, or NaN for ``fit``, for skipped entries) and over all of them."""

    shared: np.ndarray
    resolved_source: np.ndarray
    resolved_supertree: np.ndarray
    agree: np.ndarray
    contradict: np.ndarray
    unresolved: np.ndarray
    fit: np.ndarray
    weighted_fit: float

    def tsv(self) -> str:
        """One line per tree in input order under ``TSV_HEADER`` (what ``scs --triplets-out`` writes)."""
        return triplet_tsv(np.stack([self.shared, self.resolved_source, self.resolved_supertree, self.agree,
                                     self.contradict], axis=1))  # fmt: skip


def triplet_tsv(per_tree: np.ndarray) -> str:
    """``per_tree`` [T, 5] (shared, resolved_source, resolved_supertree, agree, contradict) as TSV text."""
    lines = [TSV_HEADER]
    lines += ["\t".join(str(int(v)) for v in (t, *row)) for t, row in enumerate(per_tree)]
    return "\n".join(lines) + "\n"


def _fit(per_tree: np.ndarray, weights: Sequence[float], kept: Sequence[int]) -> TripletFit:
    per_tree = np.asarray(per_tree, dtype=np.int64)
    resolved, agree = per_tree[:, 1], per_tree[:, 3]
    fit = np.full(len(per_tree), np.nan)
    kept_arr = np.asarray(kept, dtype=np.int64)
    has = kept_arr[resolved[kept_arr] > 0]
    fit[has] = agree[has] / resolved[has]
    num = den = 0.0
    for t in kept:  # tree order
        num += float(weights[t]) * int(agree[t])
        den += float(weights[t]) * int(resolved[t])
    unresolved = np.where(resolved >= 0, resolved - agree - per_tree[:, 4], -1)
    return TripletFit(
        shared=per_tree[:, 0].copy(),
        resolved_source=resolved.copy(),
        resolved_supertree=per_tree[:, 2].copy(),
        agree=agree.copy(),
        contradict=per_tree[:, 4].copy(),
        unresolved=unresolved,
        fit=fit,
        weighted_fit=num / den if den != 0 else float("nan"),
    )


def flat_triplet_fit(forest: Forest, parent, taxon, *, engine: Engine | None = None) -> TripletFit:
    """Triplet fit of the flat supertree ``parent`` / ``taxon`` (as the native build returns it: ``parent[i] < i``,
    taxon ids of ``forest``) against the trees of ``forest``, weighted with the forest's tree weights (the
    ``scs --triplets-out`` route)."""
    if engine is None:
        engine = default_engine()
    per_tree = engine.supertree_triplets(forest, parent, taxon)
    return _fit(per_tree, forest.weights(), range(len(per_tree)))


def triplet_fit(supertree: PhyloNode, trees: Sequence, weights: Sequence[float] | None = None, *,
                engine: Engine | None = None) -> TripletFit:  # fmt: skip
    """Score ``supertree`` against its source ``trees`` (see the module docstring).  ``NotCompleted`` entries are
    skipped, as ``construct_supertree`` skips them: their per-tree values are -1 and they stay out of
    ``weighted_fit``."""
    if weights is None:
        weights = [1.0] * len(trees)
    if len(trees) != len(weights):
        msg = f"The number of trees ({len(trees)}) and tree weights ({len(weights)}) must match."
        raise ValueError(msg)
    kept = [i for i, tree in enumerate(trees) if not _is_not_completed(tree)]
    _nodes, names, parent, taxon = _flat_supertree(supertree, [trees[i] for i in kept])
    per_tree = np.full((len(trees), 5), -1, dtype=np.int64)
    if kept:
        if engine is None:
            engine = default_engine()
        forest = Forest.from_trees([trees[i] for i in kept], [float(weights[i]) for i in kept], names=names)
        per_tree[kept] = engine.supertree_triplets(forest, parent, taxon)
    return _fit(per_tree, weights, kept)


__all__ = ["TSV_HEADER", "TripletFit", "flat_triplet_fit", "triplet_fit", "triplet_tsv"]
