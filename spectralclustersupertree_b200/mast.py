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

``mast_taxa`` names the taxa: per source tree one maximum agreement set, read back from the same table on the GPU
(``scs_supertree_mast_taxa``), and per supertree tip how many trees share it and how many of their sets drop it (see
``MastTaxa``).
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
MAST_TAXA_TSV_HEADER = "taxon\ttrees\tpruned"


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


@dataclass
class MastTaxa:
    """One maximum agreement set per input tree, and how often each supertree tip is dropped from them.

    Per input tree (-1, and None for ``pruned_taxa``, for skipped entries): ``shared``, ``agreement`` and ``pruned`` as
    in ``MastFit``, and ``pruned_taxa``, the sorted names of the shared taxa the returned set drops.  Per tip of the
    supertree, in sorted-name order (``names``), over the kept trees that share it: ``trees``, the number of them;
    ``taxon_pruned``, those whose set drops it; ``weighted_pruned``, the weights of the latter summed in tree order;
    ``fraction`` = taxon_pruned / trees (NaN where trees = 0).  A maximum agreement set is generally not unique: the
    sets are read back from the table by a fixed rule (DESIGN.md §3.18), and another maximum set of a tree could move
    the per-tip counts.  sum(trees) = ``MastFit.total_shared`` and sum(taxon_pruned) = ``MastFit.total_pruned``."""

    shared: np.ndarray
    agreement: np.ndarray
    pruned: np.ndarray
    pruned_taxa: list[tuple[str, ...] | None]
    names: list[str]
    trees: np.ndarray
    taxon_pruned: np.ndarray
    weighted_pruned: np.ndarray
    fraction: np.ndarray

    def tsv(self) -> str:
        """One line per supertree tip under ``MAST_TAXA_TSV_HEADER`` (what ``scs --mast-taxa-out`` writes)."""
        lines = [MAST_TAXA_TSV_HEADER]
        lines += [f"{name}\t{int(n)}\t{int(p)}" for name, n, p in zip(self.names, self.trees, self.taxon_pruned,
                                                                      strict=True)]  # fmt: skip
        return "\n".join(lines) + "\n"


def _taxa(names: Sequence[str], tips, per_tree: np.ndarray, tip_state: np.ndarray, node_taxon: np.ndarray,
          node_offsets: np.ndarray, per_taxon: np.ndarray, weighted: np.ndarray, kept: Sequence[int],
          count: int) -> MastTaxa:  # fmt: skip
    """``MastTaxa`` of ``count`` input trees from the native pass over the ``kept`` ones: ``per_tree`` [len(kept), 2],
    ``tip_state`` / ``node_taxon`` over the forest's nodes (tree j at ``node_offsets[j]``), ``per_taxon`` [taxa, 2]
    and ``weighted`` [taxa] by taxon id (``names`` indexed by taxon id); ``tips`` are the supertree's taxon ids."""
    rows = np.full((count, 2), -1, dtype=np.int64)
    kept = list(kept)
    if kept:
        rows[kept] = np.asarray(per_tree, dtype=np.int64).reshape(-1, 2)
    pruned = np.full(count, -1, dtype=np.int64)
    pruned[kept] = rows[kept, 0] - rows[kept, 1]
    tip_state = np.asarray(tip_state)
    node_taxon = np.asarray(node_taxon)
    pruned_taxa: list[tuple[str, ...] | None] = [None] * count
    for j, t in enumerate(kept):
        b, e = int(node_offsets[j]), int(node_offsets[j + 1])
        dropped = node_taxon[b:e][tip_state[b:e] == 0]
        pruned_taxa[t] = tuple(sorted(names[x] for x in dropped))
    tips = [int(x) for x in tips]
    order = sorted(tips, key=lambda x: names[x])
    per_taxon = np.asarray(per_taxon, dtype=np.int64).reshape(-1, 2)[order] if order else np.zeros((0, 2), np.int64)
    weighted = np.asarray(weighted, dtype=np.float64)[order] if order else np.zeros(0)
    fraction = np.full(len(order), np.nan)
    has = per_taxon[:, 0] > 0
    fraction[has] = per_taxon[has, 1] / per_taxon[has, 0]
    return MastTaxa(
        shared=rows[:, 0].copy(),
        agreement=rows[:, 1].copy(),
        pruned=pruned,
        pruned_taxa=pruned_taxa,
        names=[names[x] for x in order],
        trees=per_taxon[:, 0].copy(),
        taxon_pruned=per_taxon[:, 1].copy(),
        weighted_pruned=weighted.copy(),
        fraction=fraction,
    )


def _node_arrays(forest: Forest) -> tuple[np.ndarray, np.ndarray]:
    """The taxon of every node of ``forest`` and the node offsets of its trees."""
    taxa = [forest.tree_arrays(t)[3] for t in range(forest.num_trees)]
    offsets = np.zeros(len(taxa) + 1, dtype=np.int64)
    offsets[1:] = np.cumsum([len(x) for x in taxa])
    return (np.concatenate(taxa) if taxa else np.zeros(0, dtype=np.int32)), offsets


def flat_mast_taxa(forest: Forest, parent, taxon, *, engine: Engine | None = None) -> MastTaxa:
    """Agreement sets of the flat supertree ``parent`` / ``taxon`` (as the native build returns it: ``parent[i] < i``,
    taxon ids of ``forest``) against the trees of ``forest``, weighted with the forest's tree weights (the
    ``scs --mast-taxa-out`` route)."""
    if engine is None:
        engine = default_engine()
    per_tree, tip_state, per_taxon, weighted = engine.supertree_mast_taxa(forest, parent, taxon)
    node_taxon, offsets = _node_arrays(forest)
    tips = np.asarray(taxon, dtype=np.int64)
    return _taxa(forest.names, tips[tips >= 0], per_tree, tip_state, node_taxon, offsets, per_taxon, weighted,
                 range(len(per_tree)), len(per_tree))  # fmt: skip


def mast_taxa(supertree: PhyloNode, trees: Sequence, weights: Sequence[float] | None = None, *,
              engine: Engine | None = None) -> MastTaxa:  # fmt: skip
    """One maximum agreement set of ``supertree`` and each of its source ``trees``, and how often each supertree tip
    is dropped (see ``MastTaxa``).  ``NotCompleted`` entries are skipped, as ``construct_supertree`` skips them: their
    per-tree values are -1 and None, and they count for no taxon."""
    if weights is None:
        weights = [1.0] * len(trees)
    if len(trees) != len(weights):
        msg = f"The number of trees ({len(trees)}) and tree weights ({len(weights)}) must match."
        raise ValueError(msg)
    kept = [i for i, tree in enumerate(trees) if not _is_not_completed(tree)]
    _nodes, names, parent, taxon = _flat_supertree(supertree, [trees[i] for i in kept])
    tips = taxon[taxon >= 0].astype(np.int64)
    per_tree = np.zeros((0, 2), dtype=np.int64)
    tip_state = np.zeros(0, dtype=np.int8)
    node_taxon, offsets = np.zeros(0, dtype=np.int32), np.zeros(1, dtype=np.int64)
    per_taxon = np.zeros((len(names), 2), dtype=np.int64)
    weighted = np.zeros(len(names), dtype=np.float64)
    if kept:
        if engine is None:
            engine = default_engine()
        forest = Forest.from_trees([trees[i] for i in kept], [float(weights[i]) for i in kept], names=names)
        per_tree, tip_state, per_taxon, weighted = engine.supertree_mast_taxa(forest, parent, taxon)
        node_taxon, offsets = _node_arrays(forest)
    return _taxa(names, tips, per_tree, tip_state, node_taxon, offsets, per_taxon, weighted, kept, len(trees))


__all__ = ["MAST_TAXA_TSV_HEADER", "MAST_TSV_HEADER", "MastFit", "MastTaxa", "flat_mast_fit", "flat_mast_taxa",
           "mast_fit", "mast_taxa"]
