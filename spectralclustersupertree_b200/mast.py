"""Agreement-subtree fit of a supertree: per source tree, the largest set of shared taxa on which it and the supertree
agree.

Every source tree t and the supertree S are restricted to the taxa X_t they share (as the recursion restricts trees:
unary nodes collapse, polytomies stay).  Their maximum agreement subtree (MAST) is the largest Y in X_t on which the
two restrictions are the same rooted tree.  Per source tree:

=========  ======================================================================
shared     k = |X_t|
agreement  |Y|, the size of a maximum agreement subtree (k when k <= 2)
pruned     shared - agreement: the fewest taxa to drop before t and S agree
fraction   agreement / shared (NaN where nothing is shared)
=========  ======================================================================

The cluster and triplet measures count what a misplaced taxon breaks; ``pruned`` counts the taxa themselves, so one
rogue taxon costs exactly one.  agreement = shared exactly when ``clade_support``'s ``rf`` is 0 for that tree.
``shared``, ``agreement`` and ``pruned`` also sum over all kept trees, and ``weighted_pruned`` = sum_t w_t pruned_t is
added in tree order.  The sizes are computed on the GPU (``scs_supertree_mast``, csrc/triplets.cu) with the
recurrence of Steel & Warnow (1993) over every pair of internal nodes of the two restrictions.
"""

from __future__ import annotations

from collections.abc import Sequence
from dataclasses import dataclass

import numpy as np

from .engine import Engine, Forest, default_engine
from .scs import _is_not_completed
from .support import _flat_supertree
from .tree import PhyloNode

MAST_TSV_HEADER = "tree\tshared\tagreement\tpruned"


@dataclass
class MastFit:
    """Per input tree (-1, or NaN for ``fraction``, for skipped entries) and over all of them."""

    shared: np.ndarray
    agreement: np.ndarray
    pruned: np.ndarray
    fraction: np.ndarray
    total_shared: int
    total_agreement: int
    total_pruned: int
    weighted_pruned: float

    def tsv(self) -> str:
        """One line per tree in input order under ``MAST_TSV_HEADER`` (what ``scs --mast-out`` writes)."""
        lines = [MAST_TSV_HEADER]
        rows = zip(self.shared, self.agreement, self.pruned, strict=True)
        lines += ["\t".join(str(int(v)) for v in (t, *row)) for t, row in enumerate(rows)]
        return "\n".join(lines) + "\n"


def _fit(per_tree: np.ndarray, weights: Sequence[float], kept: Sequence[int]) -> MastFit:
    per_tree = np.asarray(per_tree, dtype=np.int64).reshape(-1, 2)
    shared, agreement = per_tree[:, 0].copy(), per_tree[:, 1].copy()
    kept_arr = np.asarray(kept, dtype=np.int64)
    pruned = np.full(len(per_tree), -1, dtype=np.int64)
    pruned[kept_arr] = shared[kept_arr] - agreement[kept_arr]
    fraction = np.full(len(per_tree), np.nan)
    has = kept_arr[shared[kept_arr] > 0]
    fraction[has] = agreement[has] / shared[has]
    weighted = 0.0
    for t in kept:  # tree order
        weighted += float(weights[t]) * int(pruned[t])
    return MastFit(
        shared=shared,
        agreement=agreement,
        pruned=pruned,
        fraction=fraction,
        total_shared=int(shared[kept_arr].sum()) if len(kept_arr) else 0,
        total_agreement=int(agreement[kept_arr].sum()) if len(kept_arr) else 0,
        total_pruned=int(pruned[kept_arr].sum()) if len(kept_arr) else 0,
        weighted_pruned=weighted,
    )


def flat_mast_fit(forest: Forest, parent, taxon, *, engine: Engine | None = None) -> MastFit:
    """Agreement-subtree fit of the flat supertree ``parent`` / ``taxon`` (as the native build returns it:
    ``parent[i] < i``, taxon ids of ``forest``) against the trees of ``forest``, weighted with the forest's tree
    weights (the ``scs --mast-out`` route)."""
    if engine is None:
        engine = default_engine()
    per_tree = engine.supertree_mast(forest, parent, taxon)
    return _fit(per_tree, forest.weights(), range(len(per_tree)))


def mast_fit(supertree: PhyloNode, trees: Sequence, weights: Sequence[float] | None = None, *,
             engine: Engine | None = None) -> MastFit:  # fmt: skip
    """Fit ``supertree`` to each of its source ``trees`` by their maximum agreement subtree (see the module
    docstring).  ``NotCompleted`` entries are skipped, as ``construct_supertree`` skips them: their per-tree values are
    -1 and they stay out of the totals."""
    if weights is None:
        weights = [1.0] * len(trees)
    if len(trees) != len(weights):
        msg = f"The number of trees ({len(trees)}) and tree weights ({len(weights)}) must match."
        raise ValueError(msg)
    kept = [i for i, tree in enumerate(trees) if not _is_not_completed(tree)]
    _nodes, names, parent, taxon = _flat_supertree(supertree, [trees[i] for i in kept])
    per_tree = np.full((len(trees), 2), -1, dtype=np.int64)
    if kept:
        if engine is None:
            engine = default_engine()
        forest = Forest.from_trees([trees[i] for i in kept], [float(weights[i]) for i in kept], names=names)
        per_tree[kept] = engine.supertree_mast(forest, parent, taxon)
    return _fit(per_tree, weights, kept)


__all__ = ["MAST_TSV_HEADER", "MastFit", "flat_mast_fit", "mast_fit"]
