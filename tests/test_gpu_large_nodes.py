"""GPU: the per-node path of the recursion drivers for large nodes.

A node above the small limit is first split into the components of its leaf tours; only a connected node gets
its graph built (csrc/context.cu: node_split, csrc/components.cu: tour_components_async).  Lowering the medium
limit to the small limit sends every node that the medium batch would take (graph-based components) down this
path instead, so the two ways of finding components meet on the same nodes: the recursion records and the
supertree must not change.  The public single-node entry points keep building the graph of every node."""

from __future__ import annotations

import re

import numpy as np
import pytest

from helpers import compare_with_ctrace, flat_clades, load_ctrace, parse
from spectralclustersupertree_b200.engine import Forest, merge_sharded
from spectralclustersupertree_b200.synthetic import make_problem
from test_gpu_sharded_nodes import Ranks, forest_of

pytestmark = pytest.mark.gpu

SMALL_LIMIT = 32  # scs_ctx's default small limit


def _build_both_ways(engine, make_forest, weighting, contract=True):
    """(default limits, medium limit lowered to the small limit) builds, both drivers of the latter."""
    default = engine.supertree_build(make_forest(), weighting, contract_edges=contract, record=True)
    engine.set_medium_node_limit(SMALL_LIMIT)
    try:
        lowered = engine.supertree_build(make_forest(), weighting, contract_edges=contract, record=True)
        engine.set_device_forest(False)
        try:
            on_host = engine.supertree_build(make_forest(), weighting, contract_edges=contract, record=True)
        finally:
            engine.set_device_forest(True)
    finally:
        engine.set_medium_node_limit(4096)
    assert lowered["nodes_medium"] == 0 and lowered["nodes_large"] > default["nodes_large"]
    clades = flat_clades(default["parent"], default["taxon"])
    for built in (lowered, on_host):
        # the same tree; the order in which the driver emits its nodes depends on which path took them
        assert flat_clades(built["parent"], built["taxon"]) == clades
        assert sorted(built["taxon"].tolist()) == sorted(default["taxon"].tolist())
        _same_components(built["records"], default["records"])
    return default, lowered


def _same_components(records, reference):
    """Every node: the same component count and, for a disconnected node, the same labels."""
    ref = {tuple(taxa.tolist()): (part, stats) for taxa, part, stats in reference}
    assert len(records) == len(ref)
    for taxa, part, stats in records:
        want_part, want = ref[tuple(taxa.tolist())]
        assert stats.n_components == want.n_components, len(taxa)
        if stats.n_components != 1:
            assert np.array_equal(part, want_part), len(taxa)


def test_c3_tour_components_against_the_oracle_trace(engine):
    import bench

    arrays = bench.make_workload("c3")
    ctrace = load_ctrace("c3")

    def make_forest():
        return Forest.from_arrays(arrays["node_offsets"], arrays["parent"], arrays["length"], arrays["support"],
                                  arrays["taxon"], arrays["weights"], arrays["names"])  # fmt: skip

    _, lowered = _build_both_ways(engine, make_forest, arrays["weighting"])
    report = compare_with_ctrace(lowered["records"], ctrace)
    report.pop("divergent_sets")
    assert report["compared"] + report["orphans"] == len(lowered["records"])


@pytest.mark.parametrize("case", ["branch", "bootstrap", "depth", "nocontract", "caterpillar"])
def test_untidy_trees_tour_components(engine, case):
    """Unary roots and chains, two-tip trees and lone tips, caterpillars deeper than 1 024 levels."""
    ctrace = load_ctrace(f"untidy_{case}")
    contract = ctrace.get("contract_edges", True)
    trees = parse(ctrace["lines"])
    names = sorted({x for t in trees for x in t.get_tip_names()})
    _build_both_ways(engine, lambda: Forest.from_trees(trees, ctrace["weights"], names), ctrace["weighting"],
                     contract)  # fmt: skip


def test_many_components_and_trees_under_one_root_child(engine):
    """Six groups of taxa that no tree links (a top node of six or more components), trees whose
    leaves all sit under one child of the root, and a two-tip tree."""
    lines = []
    for g in range(6):
        prob = make_problem(90 + 20 * g, 12, "depth", 500 + g)
        lines += [re.sub(r"\bt(\d+)", rf"g{g}_\1", line) for line in prob.newick_lines()]
    lines.append("((g0_1,g0_2,(g0_3,g0_4)));")
    lines.append("(((g1_5,(g1_6,g1_7)),g1_8));")
    lines.append("(g2_1,g2_2);")
    trees = parse(lines)
    names = sorted({x for t in trees for x in t.get_tip_names()})
    default, _ = _build_both_ways(engine, lambda: Forest.from_trees(trees, [1.0] * len(trees), names), "depth")
    top = max(default["records"], key=lambda r: len(r[0]))
    assert len(top[0]) == len(names) and top[2].n_components >= 6


def test_public_split_of_a_disconnected_node_still_builds_w(engine):
    arrays = make_problem(700, 40, "depth", 4242).forest_arrays()
    tours = forest_of(arrays).tours("depth")
    dev = engine.upload_tours(tours)
    part_dev = engine.alloc(4 * tours.n)
    try:
        stats = engine.node_split_dev(dev, part_dev, seed=1)
        engine.synchronize()
        bufs = engine.last_node_buffers()
    finally:
        engine.free(part_dev)
        engine.free_tours(dev)
    assert stats.n_components > 1 and tours.n > SMALL_LIMIT
    want = engine.pcg_build(tours, want_counts=False)
    assert bufs["n"] == tours.n
    assert np.array_equal(bufs["W"], want["W"])
    assert np.array_equal(bufs["adj_bits"], want["adj_bits"])


def test_sharded_build_with_a_disconnected_large_node(engine):
    """Every rank finds the components from the same tours: none of them enters the sharded node path for the
    disconnected node, and the build completes and equals one rank's."""
    arrays = make_problem(700, 40, "depth", 4242).forest_arrays()
    single = engine.supertree_build(forest_of(arrays), "depth", record=True)
    top = max(single["records"], key=lambda r: len(r[0]))
    assert top[2].n_components > 1 and len(top[0]) >= 256
    ranks = Ranks(2, n_max=700, min_n=256)
    try:
        ranks.run(lambda r, eng: eng.supertree_build(forest_of(arrays), "depth"))  # warm-up, alone
        built = ranks.run(lambda r, eng: eng.supertree_build(forest_of(arrays), "depth", rank=r, world=2))
        parent, taxon = merge_sharded([(b["parent"], b["taxon"], b["shared_prefix"]) for b in built])
    finally:
        ranks.close()
    from helpers import rf
    from spectralclustersupertree_b200.scs import _tree_from_flat

    a = _tree_from_flat(single["parent"], single["taxon"], arrays["names"])
    b = _tree_from_flat(parent, taxon, arrays["names"])
    assert sorted(b.get_tip_names()) == sorted(a.get_tip_names())
    assert rf(a, b) == 0
