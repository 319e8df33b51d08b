"""Spectral Cluster Supertree on B200: the reference's public surface over a CUDA hot path.

``construct_supertree`` and ``load_trees`` keep the reference's signatures
(ref: src/sc_supertree/__init__.py:6-12); the ``scs`` command lives in ``.cli``.  ``clade_support`` scores a
supertree against its source trees (per-clade support and conflict, per-tree Robinson-Foulds distance),
``triplet_fit`` compares their rooted triplets, ``taxon_triplet_fit`` credits those triplets to the taxa and
``mrp_score`` gives the parsimony length of the supertree on the matrix representation of the source trees.
``source_tree_distances`` compares the source trees with each other: the rooted Robinson-Foulds distance of every
pair on the taxa they share, the yardstick for the per-tree distances above and a basis for tree weights.
Importing the package does not touch the GPU; the first ``construct_supertree`` call loads
``libscs_b200.so`` and raises if it (or a CUDA device) is missing -- there is no CPU fallback.
"""

__version__ = "2025.12.9+b200.1"

from .distances import SourceTreeDistances, source_tree_distances  # noqa: E402
from .load import load_trees  # noqa: E402
from .mrp import MrpScore, mrp_score  # noqa: E402
from .scs import construct_supertree  # noqa: E402
from .support import CladeSupport, clade_support  # noqa: E402
from .triplets import TaxonTripletFit, TripletFit, taxon_triplet_fit, triplet_fit  # noqa: E402

__all__ = ["CladeSupport", "MrpScore", "SourceTreeDistances", "TaxonTripletFit", "TripletFit", "__version__",
           "clade_support", "construct_supertree", "load_trees", "mrp_score", "source_tree_distances",
           "taxon_triplet_fit", "triplet_fit"]
