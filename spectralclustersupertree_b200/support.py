"""How well the source trees back each clade of a supertree, and how far each source tree is from it.

For every internal node u of the supertree and every source tree t, the clade of u restricted to the taxa X_t that t
shares with the supertree is classified against t restricted to X_t (as the recursion restricts trees):

==========  =========================================================================================
irrelevant  fewer than 2 of its taxa are in X_t, or all of X_t are
support     it is a cluster of the restricted source tree
conflict    it overlaps a non-trivial cluster B of the restricted source tree: A & B, A - B, B - A all non-empty
permitted   otherwise (compatible, but the source tree does not resolve it)
==========  =========================================================================================

Per node the counts and their sums over the tree weights are reported, with V = (ws - wc) / (ws + wc) (Wilkinson et
al., Syst. Biol. 2005; NaN where no tree supports or contradicts the clade).  Per source tree the rooted
Robinson-Foulds distance between it and the supertree, both restricted to X_t, falls out of the same pass.  The
classification runs on the GPU (``scs_supertree_support``, csrc/support.cu).
"""

from __future__ import annotations

import ctypes
from collections.abc import Sequence
from dataclasses import dataclass

import numpy as np

from . import _lib
from .engine import Engine, Forest, default_engine
from .scs import _is_not_completed
from .tree import PhyloNode


def _v_index(weighted: np.ndarray) -> np.ndarray:
    ws, wc = weighted[:, 0], weighted[:, 1]
    total = ws + wc
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(total != 0, (ws - wc) / np.where(total != 0, total, 1.0), np.nan)


@dataclass
class FlatCladeSupport:
    """Support of every node of a flat supertree (indexed like its ``parent`` / ``taxon`` arrays; tips count 0) and the
    per-source-tree distances, with the supertree as Newick text labelled with V."""

    counts: np.ndarray  # [n, 3] int32: support, conflict, permitted
    weighted: np.ndarray  # [n, 3] float64: the same summed with the tree weights, in tree order
    v: np.ndarray  # [n] float64, NaN where the weighted support and conflict are both 0
    per_tree: np.ndarray  # [T, 4] int32: shared, source_clusters, supertree_clusters, rf
    newick: str


def flat_newick_values(parent, taxon, names: Sequence[str], value, digits: int = 3) -> str:
    """Newick text of a flat tree with ``value[i]`` ("%.{digits}f") after every internal non-root node where it is
    finite (``scs_flat_tree_newick_values``)."""
    lib = _lib.load()
    blob = b"".join(name.encode("utf-8") + b"\0" for name in names)
    parent = np.ascontiguousarray(parent, dtype=np.int32)
    taxon = np.ascontiguousarray(taxon, dtype=np.int32)
    value = np.ascontiguousarray(value, dtype=np.float64)
    if len(value) != len(parent):
        msg = "one value per node is needed"
        raise ValueError(msg)
    text, size = ctypes.c_void_p(), ctypes.c_size_t()
    status = lib.scs_flat_tree_newick_values(len(parent), _lib.ptr(parent), _lib.ptr(taxon), blob, len(blob),
                                             len(names), _lib.ptr(value), int(digits), ctypes.byref(text),
                                             ctypes.byref(size))  # fmt: skip
    if status != 0:
        msg = f"scs_flat_tree_newick_values failed with status {status}"
        raise RuntimeError(msg)
    try:
        return ctypes.string_at(text.value, size.value).decode("utf-8")
    finally:
        lib.scs_free(text)


def flat_clade_support(forest: Forest, parent, taxon, *, digits: int = 3, engine: Engine | None = None) -> FlatCladeSupport:
    """Support of the flat supertree ``parent`` / ``taxon`` (as the native build returns it: ``parent[i] < i``, taxon
    ids of ``forest``) from the trees of ``forest``, without node objects (the ``scs --support-out`` route)."""
    if engine is None:
        engine = default_engine()
    counts, weighted, per_tree = engine.supertree_support(forest, parent, taxon)
    v = _v_index(weighted)
    newick = flat_newick_values(parent, taxon, forest.names, v, digits)
    return FlatCladeSupport(counts=counts, weighted=weighted, v=v, per_tree=per_tree, newick=newick)


@dataclass
class CladeSupport:
    """Per internal node of ``supertree`` (pre-order, root first) and per input tree (-1 for skipped entries)."""

    supertree: PhyloNode
    support: np.ndarray
    conflict: np.ndarray
    permitted: np.ndarray
    irrelevant: np.ndarray
    weighted_support: np.ndarray
    weighted_conflict: np.ndarray
    weighted_permitted: np.ndarray
    v: np.ndarray
    rf: np.ndarray
    shared: np.ndarray
    source_clusters: np.ndarray
    supertree_clusters: np.ndarray

    def annotated(self, digits: int = 3) -> PhyloNode:
        """A copy of the supertree whose internal nodes carry V, rounded to ``digits``, as ``support`` (None where V
        is NaN)."""
        copy = self.supertree.copy()
        for node, value in zip(copy.iter_nontips(include_self=True), self.v.tolist(), strict=True):
            node.support = None if np.isnan(value) else round(value, digits)
        return copy


def _flat_supertree(supertree: PhyloNode, trees: Sequence[PhyloNode]) -> tuple[list, list[str], np.ndarray, np.ndarray]:
    """The supertree as flat pre-order arrays (parent before child) over one joint sorted name list of its tips and
    those of ``trees``: (nodes, names, parent, taxon)."""
    nodes = list(supertree.preorder())
    names = sorted({n.name for n in nodes if not n.children}.union(*(tree.get_tip_names() for tree in trees)))
    taxon_id = {name: i for i, name in enumerate(names)}
    index = {id(node): i for i, node in enumerate(nodes)}
    parent = np.array([-1 if node.parent is None or id(node.parent) not in index else index[id(node.parent)]
                       for node in nodes], dtype=np.int32)  # fmt: skip
    parent[0] = -1
    taxon = np.array([-1 if node.children else taxon_id[node.name] for node in nodes], dtype=np.int32)
    return nodes, names, parent, taxon


def clade_support(supertree: PhyloNode, trees: Sequence, weights: Sequence[float] | None = None, *,
                  engine: Engine | None = None) -> CladeSupport:  # fmt: skip
    """Score ``supertree`` against its source ``trees`` (see the module docstring).  ``NotCompleted`` entries are
    skipped, as ``construct_supertree`` skips them; their per-tree values are -1."""
    if weights is None:
        weights = [1.0] * len(trees)
    if len(trees) != len(weights):
        msg = f"The number of trees ({len(trees)}) and tree weights ({len(weights)}) must match."
        raise ValueError(msg)
    kept = [i for i, tree in enumerate(trees) if not _is_not_completed(tree)]
    nodes, names, parent, taxon = _flat_supertree(supertree, [trees[i] for i in kept])
    internal = np.array([i for i, node in enumerate(nodes) if node.children], dtype=np.int64)

    T = len(trees)
    per_tree = np.full((T, 4), -1, dtype=np.int32)
    counts = np.zeros((len(nodes), 3), dtype=np.int32)
    weighted = np.zeros((len(nodes), 3), dtype=np.float64)
    if kept:
        if engine is None:
            engine = default_engine()
        forest = Forest.from_trees([trees[i] for i in kept], [float(weights[i]) for i in kept], names=names)
        counts, weighted, rows = engine.supertree_support(forest, parent, taxon)
        per_tree[kept] = rows
    counts, weighted = counts[internal], weighted[internal]
    return CladeSupport(
        supertree=supertree,
        support=counts[:, 0].copy(),
        conflict=counts[:, 1].copy(),
        permitted=counts[:, 2].copy(),
        irrelevant=(len(kept) - counts.sum(axis=1)).astype(np.int32),
        weighted_support=weighted[:, 0].copy(),
        weighted_conflict=weighted[:, 1].copy(),
        weighted_permitted=weighted[:, 2].copy(),
        v=_v_index(weighted),
        rf=per_tree[:, 3].copy(),
        shared=per_tree[:, 0].copy(),
        source_clusters=per_tree[:, 1].copy(),
        supertree_clusters=per_tree[:, 2].copy(),
    )


__all__ = ["CladeSupport", "FlatCladeSupport", "clade_support", "flat_clade_support", "flat_newick_values"]
