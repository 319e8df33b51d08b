"""GPU: the device-resident forest's tours and restriction (csrc/devforest.cu) against the host-forest driver, on forests
built to reach each of their paths: trees walked by a warp and trees walked by a CTA in the same wave, trees of more
than one CTA chunk, deep caterpillars whose restrictions leave long unary chains to merge (missing lengths included),
bootstrap weighting, and a node split into so many parts that the restriction's workspace bound passes its cap and the
exact size is read back.  Both drivers must take the same recursion, node for node, to the same supertree."""

from __future__ import annotations

import numpy as np
import pytest

from helpers import flat_clades, parse
from spectralclustersupertree_b200.engine import Forest

pytestmark = pytest.mark.gpu


def random_tree(tips: list[str], rng: np.random.RandomState, weighting: str, unary: float = 0.0,
                missing: float = 0.0) -> str:  # fmt: skip
    """A random rooted binary tree on ``tips`` (random halvings), with unary chains above some nodes, some lengths
    missing (``branch``) and a support on every internal node (``bootstrap``)."""

    def edge(text: str, internal: bool) -> str:
        if weighting == "bootstrap" and internal:
            text += str(int(rng.randint(50, 101)))
        if weighting == "branch" and rng.random_sample() >= missing:
            text += f":{rng.uniform(0.05, 1.0)!r}"
        while rng.random_sample() < unary:  # a chain of unary nodes on this branch
            text = edge(f"({text})", True)
        return text

    def sub(names: list[str]) -> str:
        if len(names) == 1:
            return edge(names[0], False)
        cut = int(rng.randint(1, len(names)))
        return edge(f"({sub(names[:cut])},{sub(names[cut:])})", True)

    names = list(tips)
    rng.shuffle(names)
    cut = int(rng.randint(1, len(names)))
    return f"({sub(names[:cut])},{sub(names[cut:])});"


def caterpillar(tips: list[str], rng: np.random.RandomState, unary: float, missing: float) -> str:
    """((((a,b),c),d),...) with unary nodes and missing lengths along the spine (branch weighting)."""

    def length() -> str:
        return "" if rng.random_sample() < missing else f":{rng.uniform(0.05, 1.0)!r}"

    text = f"({tips[0]}{length()},{tips[1]}{length()})"
    for x in tips[2:]:
        text += length()
        if rng.random_sample() < unary:
            text = f"({text}){length()}"
        text = f"({text},{x}{length()})"
    return text + ";"


def case_lines(case: str) -> tuple[list[str], str]:
    rng = np.random.RandomState({"mixed": 11, "huge": 12, "caterpillar": 13, "bootstrap": 14, "many_parts": 15}[case])
    if case == "mixed":  # 20 to 1 200 tips: both sides of the warp / CTA threshold in every early wave
        taxa = [f"t{i}" for i in range(1500)]
        lines = [random_tree(list(rng.choice(taxa, size=int(k), replace=False)), rng, "branch", 0.1, 0.1)
                 for k in np.linspace(20, 1200, 36)]  # fmt: skip
        return lines, "branch"
    if case == "huge":  # two trees of 20 000 tips: twenty chunks of a CTA each
        taxa = [f"t{i}" for i in range(20000)]
        lines = [random_tree(taxa, rng, "depth") for _ in range(2)]
        lines += [random_tree(list(rng.choice(taxa, size=2000, replace=False)), rng, "depth") for _ in range(6)]
        return lines, "depth"
    if case == "caterpillar":  # spines thousands of levels deep, unary chains on them, missing lengths
        taxa = [f"t{i}" for i in range(3000)]
        lines = [caterpillar(list(rng.choice(taxa, size=2500, replace=False)), rng, 0.3, 0.1) for _ in range(4)]
        lines += [random_tree(list(rng.choice(taxa, size=int(k), replace=False)), rng, "branch", 0.15, 0.1)
                  for k in rng.randint(100, 1500, size=10)]  # fmt: skip
        return lines, "branch"
    if case == "bootstrap":
        taxa = [f"t{i}" for i in range(800)]
        lines = [random_tree(list(rng.choice(taxa, size=int(k), replace=False)), rng, "bootstrap", 0.1)
                 for k in rng.randint(30, 800, size=30)]  # fmt: skip
        return lines, "bootstrap"
    # many_parts: 64 groups of taxa that no tree mixes, two trees per group: the top node splits into 64 parts
    lines = []
    for g in range(64):
        group = [f"g{g}_{i}" for i in range(300)]
        lines += [random_tree(group, rng, "depth") for _ in range(2)]
    return lines, "depth"


@pytest.mark.parametrize("case", ["mixed", "huge", "caterpillar", "bootstrap", "many_parts"])
def test_device_restriction_matches_host_forest(engine, case):
    lines, weighting = case_lines(case)
    trees = parse(lines)
    names = sorted({x for t in trees for x in t.get_tip_names()})
    weights = list(np.random.RandomState(7).uniform(0.5, 2.0, size=len(trees)))

    def build():
        return engine.supertree_build(Forest.from_trees(trees, weights, names), weighting, record=True)

    on_device = build()
    engine.set_device_forest(False)
    try:
        on_host = build()
    finally:
        engine.set_device_forest(True)
    if case == "many_parts":
        # the top node's restriction: a bound of parts x (nodes + trees) scratch entries, past the cap of
        # max(4 (nodes + trees), 2^22): the exact size is read back before the workspace is sized
        nodes = sum(len(list(t.preorder())) for t in trees)
        assert on_device["records"][0][2].n_components == 64
        assert 64 * (nodes + len(trees)) > max(4 * (nodes + len(trees)), 1 << 22)
    assert len(on_device["records"]) == len(on_host["records"])
    by_taxa = {taxa.tobytes(): (part, stats) for taxa, part, stats in on_host["records"]}
    for taxa, part, stats in on_device["records"]:
        opart, ostats = by_taxa[taxa.tobytes()]
        assert stats.n_components == ostats.n_components and stats.contracted_size == ostats.contracted_size
        assert np.array_equal(part, opart), len(taxa)
        if stats.n_components == 1 and stats.contracted_size >= 3:
            if case == "huge":  # below a 20 000-taxon node the Fiedler value varies in its last bits from run to run
                assert abs(stats.eig[1] - ostats.eig[1]) <= 1e-12 * abs(ostats.eig[1]), (len(taxa), stats.eig[1])
            else:
                assert stats.eig[1] == ostats.eig[1], (len(taxa), stats.eig[1], ostats.eig[1])
    assert flat_clades(on_device["parent"], on_device["taxon"]) == flat_clades(on_host["parent"], on_host["taxon"])
    assert sorted(on_device["taxon"][on_device["taxon"] >= 0].tolist()) == list(range(len(names)))
