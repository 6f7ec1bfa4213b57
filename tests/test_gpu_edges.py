"""The CUDA pass against the oracle port where its code paths split (cases from tests/edge_cases.py), bit for bit on lists and
states. What only the device can get wrong is placed on purpose: the shared-memory metadata windows (48 references and 32 leaf
entries per warp) refilled in the middle of a chunk, the counter width of each op inside the kernel instantiated for the
widest one, chain segments waiting on each other when leaves are omitted, persistent kernels on a grid of one SM, and the
13-bit run tag of the staging directories crossing its wrap."""
import numpy as np
import pytest

import panman_b200 as pb
from oracle.oracle import random_tree
from tests import edge_cases as E

pytestmark = pytest.mark.gpu

DEFAULTS = {"chunk_nodes": 0, "inline_nodes": 3, "schedule": 1, "lanes": 1, "overlap": 1, "grid_pct": 0, "reserve_sms": 0,
            "bwd_tail": 20}


def _options(c, **kw):
    for k, v in dict(DEFAULTS, **kw).items():
        c.set_option(k, v)


@pytest.fixture(scope="module")
def ctx():
    c = pb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def trees():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = E.shapes()[name]()
        return cache[name]

    return get


def _same(res, want):
    return (np.array_equal(res.node_offsets, want.node_offsets) and np.array_equal(res.pos, want.pos)
            and np.array_equal(res.type_code, want.type_code))


def _run(c, tree, algo, block, codes, pc, ro, fr, lp, entry, col_base=E.COL_BASE):
    """One pass through one entry of the C ABI; the Result (states where the entry returns them)."""
    n_rows, width = codes.shape
    flags = pb.FLAG_BLOCK_MODE if block else 0
    c4 = pb.pack_nibbles(codes)
    if entry == "codes":
        return c.run_codes(tree, algo, codes, pc, ro, fr, lp, block, want_states=True, col_base=col_base)
    if entry == "runs":
        runs = pb.Runs.of_tree(tree, width, c4, pc)
        try:
            return c.run_runs(algo, runs, pc, ro, fr, lp, col_base=col_base, flags=flags | pb.FLAG_WANT_STATES)
        finally:
            runs.close()
    c.upload(width, n_rows, c4, c4.shape[1], pc, ro, fr, lp, col_base=col_base)
    if entry == "resident":
        c.run_resident(algo, flags | pb.FLAG_WANT_STATES)
    else:
        assert entry == "async"
        for _ in range(3):  # on two lanes where the problem is eligible (small, no chain segments)
            c.run_resident_async(algo, flags)
    return c.download()


def _check(c, port, tree, algo, block, codes, pc, ro, fr, lp, entry, what):
    want, want_states = port.run(tree, algo, codes, pc, ro, fr, lp, block, n_threads=8, want_states=True)
    res = _run(c, tree, algo, block, codes, pc, ro, fr, lp, entry)
    want.pos = want.pos + E.COL_BASE
    assert _same(res, want), (what, entry, "lists")
    if entry != "async":
        assert res.states is not None and np.array_equal(res.states, want_states), (what, entry, "states")


def test_pairwise_cases(ctx, port, trees):
    for case in E.pairwise_cases():
        tree = trees(case["shape"])
        codes, pc, ro, fr, lp = E.case_inputs(tree, case)
        _options(ctx, chunk_nodes=case["chunk_nodes"], inline_nodes=case["inline_nodes"], schedule=case["schedule"])
        ctx.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
        _check(ctx, port, tree, case["algo"], int(case["mode"] == "block"), codes, pc, ro, fr, lp, case["entry"], E.case_id(case))
    _options(ctx)


@pytest.mark.parametrize("algo", [0, 1])
def test_arity_classes(ctx, port, algo):
    """Every arity of the list x {nucleotide, block} x {all present, 70 % present: omitted children are NONE}, plus the tree
    with one op of each counter width under a 300-reference op. Columns spread over all states drive the counters to the
    op's arity; a counter one bit too narrow wraps there."""
    rng = np.random.default_rng(70 + algo)
    trees = [(a, E.star(a, min(a // 3, 5), seed=a)) for a in E.ARITIES] + [("mixed", E.mixed_classes())]
    _options(ctx)
    n = 0
    for name, tree in trees:
        ctx.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
        for block in (0, 1):
            for pm in ("none", "p70"):
                codes, pc, ro, fr, lp = E.make_inputs(tree, algo, block, pm, "none", 0, [67, 1025][n % 2], 0.02, rng, spread=True)
                _check(ctx, port, tree, algo, block, codes, pc, ro, fr, lp, "codes", (name, block, pm))
                n += 1


@pytest.mark.parametrize("algo", [0, 1])
def test_window_edges(ctx, port, algo):
    """Backbones whose ops have 47 / 48 / 49 references (the forward window holds 48) or 31 / 32 / 33 leaf children (the
    backward window holds 32 leaf entries), in chunks of 64 ops: the windows are refilled in the middle of a chunk, and
    consecutive ops straddle their ends at every offset."""
    rng = np.random.default_rng(80 + algo)
    _options(ctx, chunk_nodes=64)
    n = 0
    for rib in (46, 47, 48, 31, 32, 33):
        tree = E.spine(90, rib, seed=rib)
        assert E.op_arities(tree).max() == rib + 1
        ctx.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
        for block in (0, 1):
            for pm in ("none", "p70"):
                fr = int(algo == 0 and not block and n % 2 == 0)
                codes, pc, ro, fr, lp = E.make_inputs(tree, algo, block, pm, ["none", "some"][n % 2], fr, [40, 1025][n % 2],
                                                      E.NOISE[n % 3], rng)
                _check(ctx, port, tree, algo, block, codes, pc, ro, fr, lp, ["codes", "resident"][n % 2], (rib, block, pm))
                n += 1
    _options(ctx)


@pytest.mark.parametrize("algo", [0, 1])
def test_deep_trees_with_omitted_leaves(ctx, port, algo):
    """Deep trees (at least 2000 leaves) cut into chain segments with leaves omitted: the forward pass does not speculate and
    waits on the segment below (REF_CHAIN), the backward pass does not speculate either; nucleotide and block mode, both
    schedules, three chunk sizes. This is the PanGraph flow over a deep backbone (blocks that some sequences lack)."""
    rng = np.random.default_rng(90 + algo)
    trees = [("spine", E.spine(700, 3, seed=12)), ("caterpillar", random_tree(2000, 13, "caterpillar"))]
    n = 0
    for name, tree in trees:
        assert tree.n_leaves >= 2000
        ctx.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
        for pm in ("p70", "one", "clade"):
            for block in (0, 1):
                codes, pc, ro, fr, lp = E.make_inputs(tree, algo, block, pm, ["none", "some"][n % 2], 0, [300, 1025][n % 2],
                                                      E.NOISE[n % 3], rng)
                want, want_states = port.run(tree, algo, codes, pc, ro, fr, lp, block, n_threads=8, want_states=True)
                want.pos = want.pos + E.COL_BASE
                for chunk_nodes in (2, 5, 16):
                    for schedule in (0, 1):
                        _options(ctx, chunk_nodes=chunk_nodes, schedule=schedule)
                        res = ctx.run_codes(tree, algo, codes, pc, ro, fr, lp, block, want_states=True, col_base=E.COL_BASE)
                        what = (name, pm, block, chunk_nodes, schedule)
                        assert _same(res, want), what
                        assert np.array_equal(res.states, want_states), what
                n += 1
    _options(ctx)


@pytest.mark.parametrize("bwd_tail", [0, 200])
def test_small_grids(port, bwd_tail):
    """Persistent kernels on one SM (reserve_sms = all but one, grid_pct = 1): both ticket orders are topological, so a pass
    needs no two items resident at once -- the lists equal the oracle's on a tree cut into chain segments and on a wide one,
    synchronously and asynchronously."""
    import torch

    n_sms = torch.cuda.get_device_properties(0).multi_processor_count
    rng = np.random.default_rng(100 + bwd_tail)
    c = pb.Context(0)
    for name, tree in (("spine", E.spine(400, 3, seed=21)), ("star1000", E.star(1000, 5, seed=22))):
        c.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
        for algo in (0, 1):
            codes, pc, ro, fr, lp = E.make_inputs(tree, algo, 0, ["none", "p70"][algo], "none", 0, 2049, 0.02, rng)
            for entry in ("codes", "async"):
                _options(c, reserve_sms=n_sms - 1, grid_pct=1, bwd_tail=bwd_tail, chunk_nodes=[0, 8][algo])
                _check(c, port, tree, algo, 0, codes, pc, ro, fr, lp, entry, (name, algo, bwd_tail))
    c.close()


# A context's epoch advances by 2 per pass (forward and backward) and the directory tag is its low 13 bits, so the tags of one
# directory wrap every 4096 passes, with one directory or with two used by alternate passes. A lane is a child context with its
# own epoch that runs every other pass: its tags wrap every 8192 passes. 9000 passes cross a wrap in all three set-ups.
WRAP_PASSES = 9000
B_PASSES = 6  # the first passes: both directories of the context and of its lane


@pytest.mark.parametrize("setup", ["sync_one_directory", "async_two_directories", "async_two_lanes"])
def test_directory_tag_wrap(port, setup):
    """One small tree in one column tile. Input B is noisy and leaves an entry in most (node, tile) slots of every directory
    (of the context and of its lane) in the first passes; input A is conserved, has a few records and runs every pass after.
    The entries B left are never rewritten, so each is read again by the A pass whose tag equals B's modulo the 13 bits,
    unless the directory was cleared before the wrap: such an entry, read as current, adds B's records to A's lists. A's lists
    are checked after every pass."""
    tree = random_tree(60, 31, "binary")
    rng = np.random.default_rng(32)
    width = 700
    base = rng.integers(0, 5, size=width).astype(np.uint8)
    a = np.repeat(base[None, :], tree.n_leaves, 0)
    a[3, 10] = (a[3, 10] + 1) % 5
    a[40, 500] = 9
    b = rng.integers(0, 16, size=(tree.n_leaves, width)).astype(np.uint8)
    want_a, _ = port.run(tree, 0, a, base, n_threads=2)
    want_b, _ = port.run(tree, 0, b, base, n_threads=2)
    assert 0 < want_a.node_offsets[-1] < 10
    assert (np.diff(want_b.node_offsets) > 0).mean() > 0.9
    a4, b4 = pb.pack_nibbles(a), pb.pack_nibbles(b)
    c = pb.Context(0)
    _options(c, overlap=int(setup != "sync_one_directory"), lanes=int(setup == "async_two_lanes"))
    c.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
    for i in range(WRAP_PASSES):
        if i in (0, B_PASSES):
            x4 = b4 if i == 0 else a4
            c.upload(width, tree.n_leaves, x4, x4.shape[1], base)
        if setup == "sync_one_directory":
            c.run_resident(pb.ALGO_FITCH)
        else:
            c.run_resident_async(pb.ALGO_FITCH)
        if i == B_PASSES - 1:
            assert _same(c.download(), want_b), setup
        elif i >= B_PASSES:
            assert _same(c.download(), want_a), (setup, i)
    c.close()
