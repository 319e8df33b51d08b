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

``taxon_triplet_fit`` credits the same triplets to their taxa, to find the taxa the source trees place differently
from the supertree.  For every tip p of the supertree, over the source trees t with p in X_t and k_t >= 3:

==================  ======================================================================
trees               the number of such trees
triplets            sum_t C(k_t - 1, 2): the triplets of X_t that contain p
resolved_source     those of them resolved in the restricted source tree
resolved_supertree  those of them resolved in the restricted supertree
agree               resolved in both, the same way
contradict          resolved in both, differently
unresolved          resolved_source - agree - contradict
fit                 agree / resolved_source (NaN where no triplet is resolved)
weighted_fit        sum_t w_t agree / sum_t w_t resolved_source (NaN where the denominator is 0)
==================  ======================================================================

``weighted_resolved_source``, ``weighted_agree`` and ``weighted_contradict`` are the sums over the same trees of
w_t times the count, added in tree order.

The counts run on the GPU (``scs_supertree_taxon_triplets``) at about the cost of the per-tree pass.
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
TAXON_TSV_HEADER = "taxon\ttrees\ttriplets\tresolved_source\tresolved_supertree\tagree\tcontradict"


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


@dataclass
class TaxonTripletFit:
    """Per tip of the supertree, in sorted-name order (``names``); see the module docstring."""

    names: list[str]
    trees: np.ndarray
    triplets: np.ndarray
    resolved_source: np.ndarray
    resolved_supertree: np.ndarray
    agree: np.ndarray
    contradict: np.ndarray
    unresolved: np.ndarray
    fit: np.ndarray
    weighted_resolved_source: np.ndarray
    weighted_agree: np.ndarray
    weighted_contradict: np.ndarray
    weighted_fit: np.ndarray

    def tsv(self) -> str:
        """One line per tip under ``TAXON_TSV_HEADER`` (what ``scs --taxon-triplets-out`` writes)."""
        columns = (self.trees, self.triplets, self.resolved_source, self.resolved_supertree, self.agree, self.contradict)
        lines = [TAXON_TSV_HEADER]
        lines += ["\t".join([name, *(str(int(c[i])) for c in columns)]) for i, name in enumerate(self.names)]
        return "\n".join(lines) + "\n"


def _ratio(num: np.ndarray, den: np.ndarray) -> np.ndarray:
    out = np.full(len(num), np.nan)
    has = den != 0
    out[has] = num[has] / den[has]
    return out


def _taxon_fit(names: Sequence[str], per_taxon: np.ndarray, weighted: np.ndarray) -> TaxonTripletFit:
    """``per_taxon`` [n, 6] (trees, triplets, resolved_source, resolved_supertree, agree, contradict) and ``weighted``
    [n, 3] (resolved_source, agree, contradict) of the tips ``names``, put in sorted-name order."""
    order = sorted(range(len(names)), key=lambda i: names[i])
    per_taxon = np.asarray(per_taxon, dtype=np.int64).reshape(-1, 6)[order]
    weighted = np.asarray(weighted, dtype=np.float64).reshape(-1, 3)[order]
    resolved, agree, contradict = per_taxon[:, 2], per_taxon[:, 4], per_taxon[:, 5]
    return TaxonTripletFit(
        names=[names[i] for i in order],
        trees=per_taxon[:, 0].copy(),
        triplets=per_taxon[:, 1].copy(),
        resolved_source=resolved.copy(),
        resolved_supertree=per_taxon[:, 3].copy(),
        agree=agree.copy(),
        contradict=contradict.copy(),
        unresolved=resolved - agree - contradict,
        fit=_ratio(agree.astype(np.float64), resolved.astype(np.float64)),
        weighted_resolved_source=weighted[:, 0].copy(),
        weighted_agree=weighted[:, 1].copy(),
        weighted_contradict=weighted[:, 2].copy(),
        weighted_fit=_ratio(weighted[:, 1], weighted[:, 0]),
    )


def flat_taxon_triplet_fit(forest: Forest, parent, taxon, *, engine: Engine | None = None) -> TaxonTripletFit:
    """Per-taxon triplet fit of the flat supertree ``parent`` / ``taxon`` (as the native build returns it) against the
    trees of ``forest``, weighted with the forest's tree weights (the ``scs --taxon-triplets-out`` route)."""
    if engine is None:
        engine = default_engine()
    per_taxon, weighted = engine.supertree_taxon_triplets(forest, parent, taxon)
    tips = np.asarray(taxon, dtype=np.int64)
    tips = tips[tips >= 0]
    return _taxon_fit([forest.names[x] for x in tips], per_taxon[tips], weighted[tips])


def taxon_triplet_fit(supertree: PhyloNode, trees: Sequence, weights: Sequence[float] | None = None, *,
                      engine: Engine | None = None) -> TaxonTripletFit:  # fmt: skip
    """Credit the triplet fit of ``supertree`` against its source ``trees`` to the supertree's tips (see the module
    docstring).  ``NotCompleted`` entries are skipped, as ``construct_supertree`` skips them."""
    if weights is None:
        weights = [1.0] * len(trees)
    if len(trees) != len(weights):
        msg = f"The number of trees ({len(trees)}) and tree weights ({len(weights)}) must match."
        raise ValueError(msg)
    kept = [i for i, tree in enumerate(trees) if not _is_not_completed(tree)]
    _nodes, names, parent, taxon = _flat_supertree(supertree, [trees[i] for i in kept])
    tips = taxon[taxon >= 0].astype(np.int64)
    per_taxon = np.zeros((len(names), 6), dtype=np.int64)
    weighted = np.zeros((len(names), 3), dtype=np.float64)
    if kept:
        if engine is None:
            engine = default_engine()
        forest = Forest.from_trees([trees[i] for i in kept], [float(weights[i]) for i in kept], names=names)
        per_taxon, weighted = engine.supertree_taxon_triplets(forest, parent, taxon)
    return _taxon_fit([names[x] for x in tips], per_taxon[tips], weighted[tips])


__all__ = ["TAXON_TSV_HEADER", "TSV_HEADER", "TaxonTripletFit", "TripletFit", "flat_taxon_triplet_fit",
           "flat_triplet_fit", "taxon_triplet_fit", "triplet_fit", "triplet_tsv"]
