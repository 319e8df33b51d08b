"""How far the source trees are from each other: the rooted Robinson-Foulds distance of every pair of source trees on
the taxa they share.

For trees t_i and t_j let X_ij be the taxa both contain and k_ij = |X_ij|.  t_i|X_ij is t_i restricted to X_ij as the
recursion restricts trees (unary nodes collapse, polytomies stay), and C_i(j) its non-trivial clusters (2 <= |c| <
k_ij; none when k_ij < 3).  Per pair:

==================  ====================================================================================
shared_taxa[i, j]   k_ij; symmetric, the diagonal is the tree's own tip count
clusters[i, j]      |C_i(j)|: row i counts tree i's clusters on the taxa it shares with tree j (not symmetric)
common[i, j]        |C_i(j) & C_j(i)|; symmetric
rf                  clusters + clusters.T - 2 common
normalized_rf       rf / (clusters + clusters.T), NaN where that is 0 (k_ij < 3, or both restrictions unresolved)
==================  ====================================================================================

Per tree, ``comparable[i]`` counts the trees j != i with a finite ``normalized_rf[i, j]`` and ``mean_normalized_rf[i]``
is the mean of those values (NaN when there are none): a tree far from every tree it can be compared with is an
outlier (misrooted, paralogous, mislabelled), and a natural candidate for a low weight in ``construct_supertree``.
The diagonal is the pair (i, i): ``clusters[i, i] = common[i, i]`` are the non-trivial clusters of t_i, ``rf[i, i] =
0``.  With t_i as the supertree, ``clade_support(t_i, trees)`` reports for tree j ``rf[i, j]``, ``common[i, j]`` (its
``shared``), ``clusters[j, i]`` (``source_clusters``) and ``clusters[i, j]`` (``supertree_clusters``).  Every count is
an exact integer and tree weights do not enter.

The counts run on the GPU (``scs_forest_pairwise_rf``, csrc/pairwise.cu).  The results are dense T x T matrices on
the host: at 5 000 trees each int32 matrix takes 100 MB (three come back from the GPU) and each float64 one 200 MB.
"""

from __future__ import annotations

from collections.abc import Sequence
from dataclasses import dataclass

import numpy as np

from .engine import Engine, Forest, default_engine
from .scs import _is_not_completed

SOURCE_RF_TSV_HEADER = "tree_a\ttree_b\tshared\tclusters_a\tclusters_b\tcommon\trf"


@dataclass
class SourceTreeDistances:
    """Per pair of input trees ``[T, T]`` and per input tree ``[T]``; rows and columns of skipped entries are -1 in
    the integer fields and NaN in the float ones."""

    shared_taxa: np.ndarray
    clusters: np.ndarray
    common: np.ndarray
    rf: np.ndarray
    normalized_rf: np.ndarray
    comparable: np.ndarray
    mean_normalized_rf: np.ndarray

    def tsv(self) -> str:
        """One line per pair a < b sharing at least three taxa, in (a, b) order, under ``SOURCE_RF_TSV_HEADER`` (what
        ``scs --source-rf-out`` writes)."""
        a, b = np.nonzero(np.triu(self.shared_taxa >= 3, 1))
        rows = np.stack([a, b, self.shared_taxa[a, b], self.clusters[a, b], self.clusters[b, a], self.common[a, b],
                         self.rf[a, b]], axis=1).astype(np.int64)  # fmt: skip
        lines = [SOURCE_RF_TSV_HEADER, *("\t".join(map(str, row)) for row in rows.tolist())]
        return "\n".join(lines) + "\n"


def _distances(shared: np.ndarray, clusters: np.ndarray, common: np.ndarray, kept: np.ndarray) -> SourceTreeDistances:
    """The derived fields from the three counted matrices; ``kept`` marks the trees that were counted."""
    skipped = ~kept
    for matrix in (shared, clusters, common):
        matrix[skipped, :] = -1
        matrix[:, skipped] = -1
    both = clusters + clusters.T
    rf = both - 2 * common
    with np.errstate(invalid="ignore", divide="ignore"):
        normalized = np.where(both > 0, rf / np.where(both > 0, both, 1), np.nan)
    normalized[skipped, :] = np.nan
    normalized[:, skipped] = np.nan
    rf[skipped, :] = -1
    rf[:, skipped] = -1
    finite = np.isfinite(normalized)
    np.fill_diagonal(finite, False)
    comparable = finite.sum(axis=1).astype(np.int64)
    total = np.where(finite, normalized, 0.0).sum(axis=1)
    mean = np.where(comparable > 0, total / np.maximum(comparable, 1), np.nan)
    comparable[skipped] = -1
    return SourceTreeDistances(shared_taxa=shared, clusters=clusters, common=common, rf=rf, normalized_rf=normalized,
                               comparable=comparable, mean_normalized_rf=mean)  # fmt: skip


def flat_source_tree_distances(forest: Forest, *, engine: Engine | None = None) -> SourceTreeDistances:
    """Distances between the trees of ``forest``, without node objects (the ``scs --source-rf-out`` route)."""
    if engine is None:
        engine = default_engine()
    shared, clusters, common = engine.forest_pairwise_rf(forest)
    return _distances(shared, clusters, common, np.ones(len(shared), dtype=bool))


def source_tree_distances(trees: Sequence, *, engine: Engine | None = None) -> SourceTreeDistances:
    """Distances between every pair of ``trees`` (see the module docstring).  ``NotCompleted`` entries are skipped, as
    ``construct_supertree`` skips them."""
    T = len(trees)
    kept = np.array([not _is_not_completed(tree) for tree in trees], dtype=bool)
    shared = np.zeros((T, T), dtype=np.int32)
    clusters = np.zeros((T, T), dtype=np.int32)
    common = np.zeros((T, T), dtype=np.int32)
    index = np.flatnonzero(kept)
    if len(index):
        if engine is None:
            engine = default_engine()
        chosen = [trees[i] for i in index]
        names = sorted(set().union(*(tree.get_tip_names() for tree in chosen)))
        forest = Forest.from_trees(chosen, [1.0] * len(chosen), names=names)
        got = engine.forest_pairwise_rf(forest)
        for full, part in zip((shared, clusters, common), got, strict=True):
            full[np.ix_(index, index)] = part
    return _distances(shared, clusters, common, kept)


__all__ = ["SOURCE_RF_TSV_HEADER", "SourceTreeDistances", "flat_source_tree_distances", "source_tree_distances"]
