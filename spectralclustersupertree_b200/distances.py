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

RF is coarse: one misplaced taxon breaks every cluster on its path.  ``source_tree_triplet_distances`` gives the
graded alternative, the rooted triplet distance.  A triplet {a, b, c} of X_ij is resolved as ab|c in a restricted tree
when LCA(a, b) lies strictly below LCA(a, b, c), a fan otherwise.  Per pair:

=====================  =================================================================================
shared_taxa[i, j]      k_ij, as above
resolved[i, j]         the triplets of X_ij resolved in t_i|X_ij: row i counts tree i (not symmetric)
agree[i, j]            those resolved the same way in both restrictions; symmetric
contradict[i, j]       those resolved in both, but differently; symmetric
distance               resolved + resolved.T - 2 agree - contradict: the triplets whose resolution differs,
                       a fan in one tree against a resolved triplet in the other included
normalized_distance    distance / C(k_ij, 3), NaN where k_ij < 3
=====================  =================================================================================

``comparable`` and ``mean_normalized_distance`` follow from ``normalized_distance`` as above.  The diagonal has
``resolved[i, i] = agree[i, i]`` and ``contradict[i, i] = 0``.  With t_i as the supertree, ``triplet_fit(t_i, trees)``
reports for tree j ``shared_taxa[i, j]``, ``resolved[j, i]`` (``resolved_source``), ``resolved[i, j]``
(``resolved_supertree``), ``agree[i, j]`` and ``contradict[i, j]``.  The counts are exact int64 values (C(k, 3)
exceeds int32 from k = 2 350) from ``scs_forest_pairwise_triplets``: four T x T matrices come back from the GPU, 700 MB
at 5 000 trees.
"""

from __future__ import annotations

from collections.abc import Sequence
from dataclasses import dataclass

import numpy as np

from .engine import Engine, Forest, default_engine
from .scs import _is_not_completed

SOURCE_RF_TSV_HEADER = "tree_a\ttree_b\tshared\tclusters_a\tclusters_b\tcommon\trf"
SOURCE_TRIPLET_TSV_HEADER = "tree_a\ttree_b\tshared\tresolved_a\tresolved_b\tagree\tcontradict\tdistance"


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


def _skip(kept: np.ndarray, *matrices: np.ndarray) -> np.ndarray:
    """Sets the rows and columns of the trees not ``kept`` to -1 in every integer matrix; returns the skipped mask."""
    skipped = ~kept
    for matrix in matrices:
        matrix[skipped, :] = -1
        matrix[:, skipped] = -1
    return skipped


def _per_tree(normalized: np.ndarray, skipped: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    """Sets the rows and columns of skipped trees to NaN in ``normalized``; returns, per tree, the other trees with a
    finite normalized distance (-1 for skipped trees) and the mean of those distances (NaN when there are none)."""
    normalized[skipped, :] = np.nan
    normalized[:, skipped] = np.nan
    finite = np.isfinite(normalized)
    np.fill_diagonal(finite, False)
    comparable = finite.sum(axis=1).astype(np.int64)
    total = np.where(finite, normalized, 0.0).sum(axis=1)
    mean = np.where(comparable > 0, total / np.maximum(comparable, 1), np.nan)
    comparable[skipped] = -1
    return comparable, mean


def _distances(shared: np.ndarray, clusters: np.ndarray, common: np.ndarray, kept: np.ndarray) -> SourceTreeDistances:
    """The derived fields from the three counted matrices; ``kept`` marks the trees that were counted."""
    skipped = _skip(kept, shared, clusters, common)
    both = clusters + clusters.T
    rf = both - 2 * common
    with np.errstate(invalid="ignore", divide="ignore"):
        normalized = np.where(both > 0, rf / np.where(both > 0, both, 1), np.nan)
    rf[skipped, :] = -1
    rf[:, skipped] = -1
    comparable, mean = _per_tree(normalized, skipped)
    return SourceTreeDistances(shared_taxa=shared, clusters=clusters, common=common, rf=rf, normalized_rf=normalized,
                               comparable=comparable, mean_normalized_rf=mean)  # fmt: skip


def _counted(trees: Sequence, engine: Engine | None, method: str, dtypes: Sequence) -> tuple[list, np.ndarray]:
    """The T x T matrices of ``engine.<method>`` over the trees that are not ``NotCompleted``, placed in full-size
    zero matrices of ``dtypes``, and the mask of those trees."""
    T = len(trees)
    kept = np.array([not _is_not_completed(tree) for tree in trees], dtype=bool)
    full = [np.zeros((T, T), dtype=dtype) for dtype in dtypes]
    index = np.flatnonzero(kept)
    if len(index):
        if engine is None:
            engine = default_engine()
        chosen = [trees[i] for i in index]
        names = sorted(set().union(*(tree.get_tip_names() for tree in chosen)))
        forest = Forest.from_trees(chosen, [1.0] * len(chosen), names=names)
        got = getattr(engine, method)(forest)
        for matrix, part in zip(full, got, strict=True):
            matrix[np.ix_(index, index)] = part
    return full, kept


def flat_source_tree_distances(forest: Forest, *, engine: Engine | None = None) -> SourceTreeDistances:
    """Distances between the trees of ``forest``, without node objects (the ``scs --source-rf-out`` route)."""
    if engine is None:
        engine = default_engine()
    shared, clusters, common = engine.forest_pairwise_rf(forest)
    return _distances(shared, clusters, common, np.ones(len(shared), dtype=bool))


def source_tree_distances(trees: Sequence, *, engine: Engine | None = None) -> SourceTreeDistances:
    """Distances between every pair of ``trees`` (see the module docstring).  ``NotCompleted`` entries are skipped, as
    ``construct_supertree`` skips them."""
    (shared, clusters, common), kept = _counted(trees, engine, "forest_pairwise_rf", (np.int32, np.int32, np.int32))
    return _distances(shared, clusters, common, kept)


@dataclass
class SourceTreeTripletDistances:
    """Per pair of input trees ``[T, T]`` and per input tree ``[T]``; rows and columns of skipped entries are -1 in
    the integer fields and NaN in the float ones."""

    shared_taxa: np.ndarray
    resolved: np.ndarray
    agree: np.ndarray
    contradict: np.ndarray
    distance: np.ndarray
    normalized_distance: np.ndarray
    comparable: np.ndarray
    mean_normalized_distance: np.ndarray

    def tsv(self) -> str:
        """One line per pair a < b sharing at least three taxa, in (a, b) order, under
        ``SOURCE_TRIPLET_TSV_HEADER`` (what ``scs --source-triplets-out`` writes)."""
        a, b = np.nonzero(np.triu(self.shared_taxa >= 3, 1))
        rows = np.stack([a, b, self.shared_taxa[a, b], self.resolved[a, b], self.resolved[b, a], self.agree[a, b],
                         self.contradict[a, b], self.distance[a, b]], axis=1).astype(np.int64)  # fmt: skip
        lines = [SOURCE_TRIPLET_TSV_HEADER, *("\t".join(map(str, row)) for row in rows.tolist())]
        return "\n".join(lines) + "\n"


def _triplet_distances(shared: np.ndarray, resolved: np.ndarray, agree: np.ndarray, contradict: np.ndarray,
                       kept: np.ndarray) -> SourceTreeTripletDistances:  # fmt: skip
    """The derived fields from the four counted matrices; ``kept`` marks the trees that were counted."""
    skipped = _skip(kept, shared, resolved, agree, contradict)
    distance = resolved + resolved.T - 2 * agree - contradict
    k = shared.astype(np.int64)
    triplets = k * (k - 1) * (k - 2) // 6
    with np.errstate(invalid="ignore", divide="ignore"):
        normalized = np.where(k >= 3, distance / np.where(k >= 3, triplets, 1), np.nan)
    distance[skipped, :] = -1
    distance[:, skipped] = -1
    comparable, mean = _per_tree(normalized, skipped)
    return SourceTreeTripletDistances(shared_taxa=shared, resolved=resolved, agree=agree, contradict=contradict,
                                      distance=distance, normalized_distance=normalized, comparable=comparable,
                                      mean_normalized_distance=mean)  # fmt: skip


def flat_source_tree_triplet_distances(forest: Forest, *, engine: Engine | None = None) -> SourceTreeTripletDistances:
    """Triplet distances between the trees of ``forest``, without node objects (the ``scs --source-triplets-out``
    route)."""
    if engine is None:
        engine = default_engine()
    shared, resolved, agree, contradict = engine.forest_pairwise_triplets(forest)
    return _triplet_distances(shared, resolved, agree, contradict, np.ones(len(shared), dtype=bool))


def source_tree_triplet_distances(trees: Sequence, *, engine: Engine | None = None) -> SourceTreeTripletDistances:
    """Triplet distances between every pair of ``trees`` (see the module docstring).  ``NotCompleted`` entries are
    skipped, as ``construct_supertree`` skips them."""
    matrices, kept = _counted(trees, engine, "forest_pairwise_triplets", (np.int32, np.int64, np.int64, np.int64))
    return _triplet_distances(*matrices, kept)


__all__ = ["SOURCE_RF_TSV_HEADER", "SOURCE_TRIPLET_TSV_HEADER", "SourceTreeDistances", "SourceTreeTripletDistances",
           "flat_source_tree_distances", "flat_source_tree_triplet_distances", "source_tree_distances",
           "source_tree_triplet_distances"]
