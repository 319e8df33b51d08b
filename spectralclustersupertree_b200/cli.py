"""Command line front end, ``scs``.

Drop-in for the reference's command (ref: src/sc_supertree/cli.py:8-39): same options, defaults, help strings and
behaviour (``no_args_is_help``, ``--version``, case-insensitive weighting choice); the supertree is written to the
output file as Newick.  The work itself takes the flat route: the input file is parsed natively into the
source-tree store, the native recursion runs on the GPU, and the result is written as Newick natively -- no node
object is built at either end (``run``).
"""

from __future__ import annotations

from pathlib import Path
from typing import Literal

import click

from . import __version__
from .distances import flat_source_tree_distances
from .load import load_forest
from .engine import default_engine
from .mrp import flat_mrp_score
from .scs import flat_newick, supertree_newick_of_forest
from .support import flat_clade_support
from .triplets import flat_taxon_triplet_fit, flat_triplet_fit


def run(in_file: str, out_file: str, weighting: str = "branch", contract_edges: bool = True,
        support_out: str | None = None, triplets_out: str | None = None,
        taxon_triplets_out: str | None = None, mrp_out: str | None = None,
        source_rf_out: str | None = None) -> None:
    """``load_trees`` + ``construct_supertree`` + ``write`` of the reference's command (ref: cli.py:33-39).  With
    ``support_out`` the supertree is also written there with the V support index of every internal non-root node
    (``support.flat_clade_support``) as its label; with ``triplets_out`` the triplet fit of every source tree
    (``triplets.flat_triplet_fit``) is written there as TSV, and with ``taxon_triplets_out`` that of every tip of the
    supertree (``triplets.flat_taxon_triplet_fit``); with ``mrp_out`` the MRP score of every source tree
    (``mrp.flat_mrp_score``) is written there as TSV; with ``source_rf_out`` the Robinson-Foulds distance of every pair
    of source trees that share at least three taxa (``distances.flat_source_tree_distances``) is written there as
    TSV.  The supertree is built once either way."""
    forest = load_forest(in_file)
    if forest.num_trees == 0:  # what construct_supertree says about an empty list (ref: scs.py:63-65)
        msg = "There must be at least one tree to make a supertree."
        raise ValueError(msg)
    extras = (support_out, triplets_out, taxon_triplets_out, mrp_out, source_rf_out)
    if all(path is None for path in extras):
        text = supertree_newick_of_forest(forest, weighting.lower(), contract_edges=contract_edges)
        Path(out_file).write_text(text + "\n")
        return
    engine = default_engine()
    built = engine.supertree_build(forest, weighting.lower(), contract_edges=contract_edges)
    Path(out_file).write_text(flat_newick(built["parent"], built["taxon"], forest.names) + "\n")
    if support_out is not None:
        scored = flat_clade_support(forest, built["parent"], built["taxon"], engine=engine)
        Path(support_out).write_text(scored.newick + "\n")
    if triplets_out is not None:
        fit = flat_triplet_fit(forest, built["parent"], built["taxon"], engine=engine)
        Path(triplets_out).write_text(fit.tsv())
    if taxon_triplets_out is not None:
        per_taxon = flat_taxon_triplet_fit(forest, built["parent"], built["taxon"], engine=engine)
        Path(taxon_triplets_out).write_text(per_taxon.tsv())
    if mrp_out is not None:
        score = flat_mrp_score(forest, built["parent"], built["taxon"], engine=engine)
        Path(mrp_out).write_text(score.tsv())
    if source_rf_out is not None:
        distances = flat_source_tree_distances(forest, engine=engine)
        Path(source_rf_out).write_text(distances.tsv())


@click.command(no_args_is_help=True)
@click.version_option(__version__)
@click.option("-i", "--in-file", required=True, help="File containing source trees.")
@click.option("-o", "--out-file", required=True, help="Output file.")
@click.option(
    "-p",
    "--pcg-weighting",
    help="Proper cluster graph weighting strategy.",
    default="branch",
    type=click.Choice(["one", "depth", "branch", "bootstrap"], case_sensitive=False),
)
@click.option(
    "--disable-contraction",
    help="Disable edge contraction (not recommended).",
    default=False,
    is_flag=True,
)
@click.option(
    "--support-out",
    help="Also write the supertree with the V support index of each clade from the source trees.",
    default=None,
)
@click.option(
    "--triplets-out",
    help="Also write, per source tree, the rooted triplets the supertree agrees with and contradicts (TSV).",
    default=None,
)
@click.option(
    "--taxon-triplets-out",
    help="Also write, per supertree taxon, the rooted triplets containing it that the source trees agree with and "
    "contradict (TSV).",
    default=None,
)
@click.option(
    "--mrp-out",
    help="Also write, per source tree, the parsimony steps its clusters need on the supertree (MRP score, TSV).",
    default=None,
)
@click.option(
    "--source-rf-out",
    help="Also write the rooted Robinson-Foulds distance between every pair of source trees on the taxa they share "
    "(TSV).",
    default=None,
)
def scs(
    in_file: str,
    out_file: str,
    pcg_weighting: Literal["one", "depth", "branch", "bootstrap"],
    *,
    disable_contraction: bool,
    support_out: str | None,
    triplets_out: str | None,
    taxon_triplets_out: str | None,
    mrp_out: str | None,
    source_rf_out: str | None,
) -> None:
    """Run spectral cluster supertree over the given set of source trees."""
    run(in_file, out_file, pcg_weighting, contract_edges=not disable_contraction, support_out=support_out,
        triplets_out=triplets_out, taxon_triplets_out=taxon_triplets_out, mrp_out=mrp_out,
        source_rf_out=source_rf_out)


if __name__ == "__main__":
    scs()
