"""MRP score of a supertree: the parsimony length of the supertree on the matrix representation of its source trees.

Every source tree t is restricted to the taxa X_t it shares with the supertree S (as the recursion restricts trees),
and every non-trivial cluster c of the restricted tree (2 <= |c| < k_t) is one binary character in Baum-Ragan
coding: 1 on the taxa of c, 0 on the rest of X_t, missing on every other tip of S.  A cluster that appears in two
trees is two characters.  The length of a character is its minimum number of state changes on S under
Fitch/Hartigan parsimony, polytomies of S being hard ones, with an all-0 outgroup above the root.  Per source tree:

==========  ======================================================================
shared      k = |X_t|
characters  the non-trivial clusters of t restricted to X_t
steps       the summed length of its characters on S
exact       its characters of length 1: those that are clusters of S restricted to X_t
extra       steps - characters
ci          characters / steps, the consistency index (NaN where there is no character)
==========  ======================================================================

Every character has length at least 1, so ``exact`` equals ``clade_support``'s ``shared`` and ``characters`` its
``source_clusters``.  ``steps`` and ``characters`` also sum over all kept trees, ``weighted_steps`` = sum_t w_t
steps_t is added in tree order, and ``ci`` = characters / steps over all of them.  The lengths run on the GPU
(``scs_supertree_mrp``, csrc/triplets.cu), with a character costing the leaves of the smallest clade of the
restricted supertree that holds it.
"""

from __future__ import annotations

from collections.abc import Sequence
from dataclasses import dataclass

import numpy as np

from .engine import Engine, Forest, default_engine
from .scs import _is_not_completed
from .support import _flat_supertree
from .tree import PhyloNode

MRP_TSV_HEADER = "tree\tshared\tcharacters\tsteps\texact"


@dataclass
class MrpScore:
    """Per input tree (-1, or NaN for ``ci``, for skipped entries) and over all of them."""

    shared: np.ndarray
    characters: np.ndarray
    steps: np.ndarray
    exact: np.ndarray
    extra: np.ndarray
    ci: np.ndarray
    total_steps: int
    total_characters: int
    weighted_steps: float
    total_ci: float

    def tsv(self) -> str:
        """One line per tree in input order under ``MRP_TSV_HEADER`` (what ``scs --mrp-out`` writes)."""
        lines = [MRP_TSV_HEADER]
        rows = zip(self.shared, self.characters, self.steps, self.exact, strict=True)
        lines += ["\t".join(str(int(v)) for v in (t, *row)) for t, row in enumerate(rows)]
        return "\n".join(lines) + "\n"


def _score(per_tree: np.ndarray, weights: Sequence[float], kept: Sequence[int]) -> MrpScore:
    per_tree = np.asarray(per_tree, dtype=np.int64).reshape(-1, 4)
    characters, steps = per_tree[:, 1], per_tree[:, 2]
    ci = np.full(len(per_tree), np.nan)
    kept_arr = np.asarray(kept, dtype=np.int64)
    has = kept_arr[steps[kept_arr] > 0]
    ci[has] = characters[has] / steps[has]
    weighted = 0.0
    for t in kept:  # tree order
        weighted += float(weights[t]) * int(steps[t])
    total_steps = int(steps[kept_arr].sum()) if len(kept_arr) else 0
    total_characters = int(characters[kept_arr].sum()) if len(kept_arr) else 0
    return MrpScore(
        shared=per_tree[:, 0].copy(),
        characters=characters.copy(),
        steps=steps.copy(),
        exact=per_tree[:, 3].copy(),
        extra=np.where(steps >= 0, steps - characters, -1),
        ci=ci,
        total_steps=total_steps,
        total_characters=total_characters,
        weighted_steps=weighted,
        total_ci=total_characters / total_steps if total_steps else float("nan"),
    )


def flat_mrp_score(forest: Forest, parent, taxon, *, engine: Engine | None = None) -> MrpScore:
    """MRP score of the flat supertree ``parent`` / ``taxon`` (as the native build returns it: ``parent[i] < i``,
    taxon ids of ``forest``) against the trees of ``forest``, weighted with the forest's tree weights (the
    ``scs --mrp-out`` route)."""
    if engine is None:
        engine = default_engine()
    per_tree = engine.supertree_mrp(forest, parent, taxon)
    return _score(per_tree, forest.weights(), range(len(per_tree)))


def mrp_score(supertree: PhyloNode, trees: Sequence, weights: Sequence[float] | None = None, *,
              engine: Engine | None = None) -> MrpScore:  # fmt: skip
    """Score ``supertree`` against the matrix representation of its source ``trees`` (see the module docstring).
    ``NotCompleted`` entries are skipped, as ``construct_supertree`` skips them: their per-tree values are -1 and they
    stay out of the totals."""
    if weights is None:
        weights = [1.0] * len(trees)
    if len(trees) != len(weights):
        msg = f"The number of trees ({len(trees)}) and tree weights ({len(weights)}) must match."
        raise ValueError(msg)
    kept = [i for i, tree in enumerate(trees) if not _is_not_completed(tree)]
    _nodes, names, parent, taxon = _flat_supertree(supertree, [trees[i] for i in kept])
    per_tree = np.full((len(trees), 4), -1, dtype=np.int64)
    if kept:
        if engine is None:
            engine = default_engine()
        forest = Forest.from_trees([trees[i] for i in kept], [float(weights[i]) for i in kept], names=names)
        per_tree[kept] = engine.supertree_mrp(forest, parent, taxon)
    return _score(per_tree, weights, kept)


__all__ = ["MRP_TSV_HEADER", "MrpScore", "flat_mrp_score", "mrp_score"]
