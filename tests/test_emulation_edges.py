"""The edge cases of tests/edge_cases.py through the CPU emulation of the kernels (tests/emul) against the oracle port: lists
and states bit for bit. This checks the case builders and their expected values without a device -- the stats of the
emulated tree program confirm that each builder makes what it claims (the widest op, chain segments on the deep trees) --
and it covers the shared host code (tree_program.cpp: chunks, chain cuts, per-op counter widths) at those edges. The device
half, with what the emulation does not model (metadata windows, cp.async stages, the MAXB instantiation, schedules and
grids, directory tags), is test_gpu_edges.py."""
import numpy as np
import pytest

from oracle.oracle import random_tree
from tests import edge_cases as E
from tests.emul.emul import Emulator


@pytest.fixture(scope="module")
def emu():
    return Emulator()


@pytest.fixture(scope="module")
def trees():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = E.shapes()[name]()
        return cache[name]

    return get


def _emul_chunk(chunk_nodes):
    return chunk_nodes if chunk_nodes > 0 else 8  # 0 = the library's choice; 8 is its floor, and what it picks for these sizes


def _check(emu, port, tree, algo, block, codes, pc, ro, fr, lp, chunk_nodes, inline_nodes, level_mode, what):
    want, want_states = port.run(tree, algo, codes, pc, ro, fr, lp, block, n_threads=4, want_states=True)
    rc, got, states, stats = emu.run(tree, algo, codes, pc, ro, fr, lp, block, chunk_nodes=chunk_nodes, col_base=E.COL_BASE,
                                     inline_nodes=inline_nodes, level_mode=level_mode)
    assert rc == 0, (what, rc)
    want.pos = want.pos + E.COL_BASE
    assert got.same_as(want), (what, "lists")
    assert np.array_equal(states, want_states), (what, "states")
    return stats


def test_pairwise_cases(emu, port, trees):
    cases = E.pairwise_cases()
    assert 80 <= len(cases) <= 120
    for c in cases:
        tree = trees(c["shape"])
        codes, pc, ro, fr, lp = E.case_inputs(tree, c)
        _check(emu, port, tree, c["algo"], int(c["mode"] == "block"), codes, pc, ro, fr, lp, _emul_chunk(c["chunk_nodes"]),
               c["inline_nodes"], 1 - c["schedule"], E.case_id(c))


def test_builders_make_what_they_claim(emu, port, trees):
    codes1 = lambda t: np.zeros((t.n_leaves, 1), np.uint8)
    for a in E.ARITIES:
        t = E.star(a, 3)
        _, _, _, stats = emu.run(t, 1, codes1(t), np.zeros(1, np.uint8), chunk_nodes=8)
        assert stats[3] == a and E.op_arities(t).max() == a, a
    for refs in (47, 48, 49):
        t = E.spine(40, refs - 1)
        _, _, _, stats = emu.run(t, 0, codes1(t), np.zeros(1, np.uint8), chunk_nodes=64)
        assert stats[3] == refs
    t = E.mixed_classes()
    _, _, _, stats = emu.run(t, 1, codes1(t), np.zeros(1, np.uint8), chunk_nodes=8)
    assert stats[3] == 300 and sorted(E.op_arities(t)[E.op_arities(t) > 0]) == [3, 15, 200, 260, 300]
    for name in E.DEEP_SHAPES:
        t = trees(name)
        assert t.n_nodes - t.n_leaves >= 299, name
        for chunk_nodes in (2, 5, 16):
            _, _, _, stats = emu.run(t, 0, codes1(t), np.zeros(1, np.uint8), chunk_nodes=chunk_nodes)
            assert stats[4] > 0, (name, chunk_nodes, "expected chain segments")
    for name in ("star256", "star1000", "mixed"):  # wide trees have no deep path to cut
        _, _, _, stats = emu.run(trees(name), 0, codes1(trees(name)), np.zeros(1, np.uint8), chunk_nodes=2)
        assert stats[4] == 0, name
    # presence builders
    rng = np.random.default_rng(0)
    assert E.presence("none", 50, rng) is None
    assert E.presence("one", 50, rng).sum() == 1
    lp = E.presence("clade", 60, rng)
    z = np.flatnonzero(lp == 0)
    assert len(z) == 20 and z[-1] - z[0] == 19
    assert 0 < E.presence("p70", 1000, rng).mean() < 0.8
    # every allowed pair of values is covered, and nothing forbidden is drawn
    cases = E.all_pairs()
    names = list(E.PAIRWISE_DIMS)
    for i in range(len(names)):
        for j in range(i + 1, len(names)):
            seen = {(c[names[i]], c[names[j]]) for c in cases}
            for a in E.PAIRWISE_DIMS[names[i]]:
                for b in E.PAIRWISE_DIMS[names[j]]:
                    if E.case_allowed({names[i]: a, names[j]: b}):
                        assert (a, b) in seen, (names[i], a, names[j], b)
    assert all(E.case_allowed(c) for c in cases)


@pytest.mark.parametrize("algo", [0, 1])
def test_arity_classes(emu, port, algo):
    """Every arity of the list, nucleotide and block mode, all leaves present and 70 % present (omitted children are NONE in
    the counters), plus the tree with one op of each width class. The spread columns drive the per-state counters to the
    op's arity and one below it: an op whose counter is one bit too narrow for its arity wraps there."""
    rng = np.random.default_rng(50 + algo)
    trees = [(a, E.star(a, min(a // 3, 5), seed=a)) for a in E.ARITIES] + [("mixed", E.mixed_classes())]
    for name, tree in trees:
        for block in (0, 1):
            for pm in ("none", "p70"):
                codes, pc, ro, fr, lp = E.make_inputs(tree, algo, block, pm, "none", 0, 67, 0.02, rng, spread=True)
                _check(emu, port, tree, algo, block, codes, pc, ro, fr, lp, 8, 3, 0, (name, algo, block, pm))


def test_deep_trees_with_omitted_leaves(emu, port):
    """Spine and caterpillar trees of at least 2000 leaves cut into chain segments, with leaves omitted (the forward pass
    then does not speculate and waits on the segment below), in nucleotide and block mode, both algorithms."""
    rng = np.random.default_rng(61)
    trees = [("spine", E.spine(700, 3, seed=12)), ("caterpillar", random_tree(2000, 13, "caterpillar"))]
    n = 0
    for name, tree in trees:
        assert tree.n_leaves >= 2000
        for pm in ("p70", "one", "clade"):
            for block in (0, 1):
                for algo in (0, 1):
                    codes, pc, ro, fr, lp = E.make_inputs(tree, algo, block, pm, ["none", "some"][n % 2], 0, [33, 130][n % 2],
                                                          E.NOISE[n % 3], rng)
                    for chunk_nodes, level_mode in ((2, 0), (5, 1), (16, 0)):
                        stats = _check(emu, port, tree, algo, block, codes, pc, ro, fr, lp, chunk_nodes, n % 2 * 3, level_mode,
                                       (name, pm, block, algo, chunk_nodes))
                        assert stats[4] > 0
                    n += 1
