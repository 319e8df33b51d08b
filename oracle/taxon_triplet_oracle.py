"""Per-taxon rooted triplet fit of a supertree against its source trees
(spectralclustersupertree_b200.triplets.taxon_triplet_fit): every triplet of the shared taxa X of a source tree is
credited to its three taxa.  Two routes over the LCA depth matrices of both trees restricted to X (as in
oracle/triplet_oracle.py): ``brute_taxon_counts`` classifies every triplet (the definition), ``row_column_counts``
restates the row/column identity csrc/triplets.cu counts by.  Test infrastructure only (cubic in the shared taxa)."""

from __future__ import annotations

from collections.abc import Sequence
from math import comb

import numpy as np

from oracle.triplet_oracle import _classify, lca_depths
from spectralclustersupertree_b200.tree import PhyloNode

TAXON_FIELDS = ("trees", "triplets", "resolved_source", "resolved_supertree", "agree", "contradict")


def _restricted_depths(supertree: PhyloNode, tree: PhyloNode) -> tuple[list[str], np.ndarray, np.ndarray]:
    """The shared tips X (sorted) and the LCA depth matrices of the source tree and the supertree restricted to X."""
    X = sorted(set(tree.get_tip_names()) & set(supertree.get_tip_names()))
    if len(X) < 3:
        return X, np.zeros((0, 0), np.int64), np.zeros((0, 0), np.int64)
    Dt = lca_depths(tree.get_sub_tree(X, ignore_missing=True, as_rooted=True), X)
    Ds = lca_depths(supertree.get_sub_tree(X, ignore_missing=True, as_rooted=True), X)
    return X, Dt, Ds


def brute_taxon_counts(Dt: np.ndarray, Ds: np.ndarray) -> np.ndarray:
    """[k, 4] per taxon: resolved_source, resolved_supertree, agree, contradict over the triplets containing it, by
    classifying every triplet (the definition)."""
    k = len(Dt)
    out = np.zeros((k, 4), dtype=np.int64)
    for a in range(k - 2):
        rest = np.arange(a + 1, k)
        j, l = np.triu_indices(len(rest), 1)
        b, c = rest[j], rest[l]
        ct = _classify(Dt[a, b], Dt[a, c], Dt[b, c])
        cs = _classify(Ds[a, b], Ds[a, c], Ds[b, c])
        flags = np.stack([ct > 0, cs > 0, (ct > 0) & (ct == cs), (ct > 0) & (cs > 0) & (ct != cs)], axis=1)
        flags = flags.astype(np.int64)
        out[a] += flags.sum(axis=0)
        for members in (b, c):
            for f in range(4):
                out[:, f] += np.bincount(members, weights=flags[:, f], minlength=k).astype(np.int64)
    return out


def row_column_counts(Dt: np.ndarray, Ds: np.ndarray) -> np.ndarray:
    """The same [k, 4] by the route of csrc/triplets.cu: in row a every point x != a gets f_alpha, f_beta, c, d over
    the other points y (alpha / beta = LCA depths with a in the source tree / supertree); R = row sums, C = column
    sums over the other rows; resolved and agree = (R / 2 + C) / 2, contradict = R / 2 + C."""
    k = len(Dt)
    R = np.zeros((k, 4), dtype=np.int64)
    C = np.zeros((k, 4), dtype=np.int64)
    for a in range(k):
        points = np.flatnonzero(np.arange(k) != a)
        alpha, beta = Dt[a, points], Ds[a, points]
        da = alpha[:, None] - alpha[None, :]
        db = beta[:, None] - beta[None, :]
        f = np.stack([(da != 0).sum(1), (db != 0).sum(1), (da * db > 0).sum(1), (da * db < 0).sum(1)], axis=1)
        R[a] = f.sum(axis=0)
        C[points] += f
    assert (R % 2 == 0).all()
    out = np.empty((k, 4), dtype=np.int64)
    out[:, :3] = (R[:, :3] // 2 + C[:, :3]) // 2
    out[:, 3] = R[:, 3] // 2 + C[:, 3]
    return out


def taxon_fit(supertree: PhyloNode, trees: Sequence[PhyloNode], weights: Sequence[float] | None = None,
              route=brute_taxon_counts) -> dict:  # fmt: skip
    """Per tip of ``supertree`` (``names``, sorted): the ``TAXON_FIELDS`` summed over the trees sharing it with at
    least two other tips, and ``weighted`` [n, 3] = resolved_source, agree, contradict summed as acc = acc + w * count
    in tree order; ``weighted_fit`` = weighted agree / weighted resolved_source (NaN where that is 0)."""
    if weights is None:
        weights = [1.0] * len(trees)
    names = sorted(supertree.get_tip_names())
    index = {name: i for i, name in enumerate(names)}
    counts = np.zeros((len(names), 6), dtype=np.int64)
    weighted = [[0.0, 0.0, 0.0] for _ in names]
    for tree, w in zip(trees, weights, strict=True):
        X, Dt, Ds = _restricted_depths(supertree, tree)
        if len(X) < 3:
            continue
        per = route(Dt, Ds)
        for name, row in zip(X, per.tolist(), strict=True):
            i = index[name]
            counts[i] += [1, comb(len(X) - 1, 2), *row]
            acc = weighted[i]
            for f, count in enumerate((row[0], row[2], row[3])):
                acc[f] = acc[f] + float(w) * float(count)
    out: dict = {"names": names, "weighted": np.array(weighted, dtype=np.float64).reshape(-1, 3)}
    for f, key in enumerate(TAXON_FIELDS):
        out[key] = counts[:, f]
    out["weighted_fit"] = np.array([acc[1] / acc[0] if acc[0] != 0 else float("nan") for acc in weighted])
    return out
