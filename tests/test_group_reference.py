"""The column ranges and the case builders of tests/group_cases.py, without a GPU: pmb_group_column_range against the plain
restatement, the refusals of the range and create entries, every builder against what it claims, and the hand-shake
model: the schedules reach a wait that can never be met when the merge credits only the active ranks, and none when it
credits every rank."""
import ctypes as C

import numpy as np
import pytest

from oracle.oracle import random_tree
from tests import group_cases as GC

WORLDS = tuple(range(1, 65)) + (GC.MAX_WORLD,)


@pytest.fixture(scope="module")
def lib():
    import panman_b200 as pb

    pb.build_library()
    return pb.load_library()


def _range(lib, world, n_cols, rank):
    a, b = C.c_int64(), C.c_int64()
    rc = lib.pmb_group_column_range(world, n_cols, rank, C.byref(a), C.byref(b))
    return rc, a.value, b.value


def _widths(world):
    """0, and one below / on / above 1, world - 1, world, world + 1, 2 world + 1 tiles and tile counts up to 2^31 columns."""
    tiles = {1, 2, world - 1, world, world + 1, 2 * world + 1, 1000 * world + 3, 2 ** 21 - 1, 2 ** 21}
    out = {0, 2 ** 31 - 1, 2 ** 31}
    for t in tiles:
        for d in (-1, 0, 1):
            if t >= 1:
                out.add(t * GC.TILE + d)
    return sorted(x for x in out if 0 <= x <= 2 ** 31)


def test_column_range_matches_reference(lib):
    for world in WORLDS:
        for n_cols in _widths(world):
            ranges = []
            for rank in range(world):
                rc, a, b = _range(lib, world, n_cols, rank)
                assert rc == 0 and (a, b) == GC.range_reference(world, n_cols, rank), (world, n_cols, rank)
                ranges.append((a, b))
            # the properties the reference claims, checked on the library's answer
            assert ranges[0][0] == 0 and ranges[-1][1] == n_cols
            assert all(ranges[r][1] == ranges[r + 1][0] for r in range(world - 1)), (world, n_cols)
            assert all(a % GC.TILE == 0 or a == b == n_cols for a, b in ranges)
            tiles = [-(-(b - a) // GC.TILE) for a, b in ranges]
            assert max(tiles) - min(tiles) <= 1 and tiles == sorted(tiles, reverse=True)
            active = sum(b > a for a, b in ranges)
            assert active == GC.active_ranks(world, n_cols) == min(world, -(-n_cols // GC.TILE))
            assert all(b == a for a, b in ranges[active:]) and all(b > a for a, b in ranges[:active])


def test_range_and_create_refusals(lib):
    assert _range(lib, 0, 10, 0)[0] == -1
    assert _range(lib, -3, 10, 0)[0] == -1
    for world in (1, 4, GC.MAX_WORLD):
        assert _range(lib, world, 10, world)[0] == -1   # rank >= world
        assert _range(lib, world, 10, -1)[0] == -1
        assert _range(lib, world, -1, 0)[0] == -1       # negative n_cols
        assert _range(lib, world, -(2 ** 40), 0)[0] == -1
    a = C.c_int64()
    assert lib.pmb_group_column_range(2, 10, 0, None, C.byref(a)) == -1
    # create checks its arguments before it touches a device: these answers are the same with or without a GPU
    h = C.c_void_p()
    dev = (C.c_int * 1)(0)
    assert lib.pmb_group_create(C.byref(h), dev, 1, 0, 0) == -1 and not h.value                  # world 0
    assert lib.pmb_group_create(C.byref(h), dev, 1, 0, GC.MAX_WORLD + 1) == -1 and not h.value   # world 1025
    assert lib.pmb_group_create(C.byref(h), dev, 1, 3, 3) == -1 and not h.value                  # rank_base + n_local > world
    assert lib.pmb_group_create(C.byref(h), dev, 0, 0, 1) == -1 and not h.value


@pytest.mark.parametrize("world", range(1, 9))
def test_boundary_cases_place_their_features(port, world):
    """Every boundary case carries three different parent codes, root overrides and fwd_root_ref values at b - 1, b, b + 1,
    runs of 1 ... 13 that end at, start at and straddle b, and a record type that changes at b in the oracle's lists."""
    tree = random_tree(GC.FEATURE_ROWS + 10, 40 + world, "binary")
    widths = GC.boundary_widths(world)
    assert {GC.active_ranks(world, w) for w in widths} >= {1, max(1, world - 1), world}
    assert any(-(-w // GC.TILE) == world - 1 for w in widths) or world == 1
    for k, n_cols in enumerate(widths):
        algo, block = k % 2, (k // 2) % 2
        c = GC.boundary_case(tree.n_leaves, world, n_cols, algo, block, seed=k, presence=True, override=True,
                             fwd=algo == 0 and not block)
        assert c.codes.shape == (tree.n_leaves, n_cols) and list(c.bounds) == GC.boundaries(world, n_cols)
        assert len(c.bounds) == GC.active_ranks(world, n_cols) - 1
        nst = 3 if block else 16
        assert c.codes.max() < nst and c.parent_code.max() < nst
        for b in c.bounds:
            cols = np.arange(b - 1, min(n_cols, b + 2))
            for x in (c.parent_code, c.root_override, c.fwd_root_ref):
                if x is not None:
                    assert len(set(x[cols].tolist())) == len(cols) and x[cols].min() >= 0, (world, n_cols, b)
            slots = GC.run_slots(b, n_cols)
            for L in GC.RUN_LENGTHS:
                got = {lab: (lo, hi) for lab, LL, lo, hi in slots if LL == L}
                assert got["ends"][1] == b and got["starts"][0] == b
                if L >= 2 and b + L // 2 <= n_cols:
                    assert got["straddles"][0] < b < got["straddles"][1]
        assert c.leaf_present is not None and not c.leaf_present.all()
        assert c.leaf_present[:GC.FEATURE_ROWS].all() or not c.bounds
        if not c.bounds:
            continue
        want, _ = port.run(tree, algo, c.codes, c.parent_code, c.root_override, c.fwd_root_ref, c.leaf_present, block)
        node = np.repeat(np.arange(tree.n_nodes), np.diff(want.node_offsets))
        ty = want.type_code >> 4
        for b, rows in zip(c.bounds, c.type_rows):
            assert (c.codes[list(rows), b - 1] == 0).all() and (c.codes[list(rows), b] != 0).all()
            lineage = set()  # the rows' leaves and their ancestors
            for r in rows:
                v = int(np.flatnonzero(tree.leaf_row == r)[0])
                while v >= 0:
                    lineage.add(v)
                    v = int(tree.parent[v])
            before = set(node[(want.pos == b - 1) & (ty == 1)].tolist()) & lineage   # ND up to b - 1
            after = set(node[(want.pos == b) & (ty != 1)].tolist()) & lineage        # NS / NI from b on
            assert before and after, (world, n_cols, b, "the record type does not change at the boundary")


def test_padded_rows_and_odd_widths():
    rng = np.random.default_rng(3)
    for n_cols in (1, 2, 1023, 1024, 1025, 4097):
        codes = rng.integers(0, 16, size=(7, n_cols)).astype(np.uint8)
        for pad in (0, 5):
            buf, stride = GC.pack_padded(codes, pad, seed=n_cols)
            w = (n_cols + 1) // 2
            assert buf.shape == (7, stride) and stride == w + pad
            cols = np.arange(n_cols)
            assert np.array_equal((buf[:, cols // 2] >> (4 * (cols % 2))) & 15, codes)
            if n_cols % 2:
                assert (buf[:, w - 1] >> 4).min() > 0   # garbage where column n_cols would be
            assert (buf[:, w:] == 0xEE).all()


@pytest.mark.parametrize("world", [2, 3, 4, 5, 8, 16])
def test_schedules_reach_their_patterns(world):
    steps = GC.schedule(world, seed=world)
    acts = [s.active for s in steps]
    assert acts == GC.schedule_actives(world)
    assert all(GC.active_ranks(world, s.n_cols) == s.active for s in steps)
    for r in range(1, world):
        assert {1, 2, 3} <= set(GC.inactive_stretches(acts, r)), r
        # every rank but 0 is first active at a step > 2, when its wait for credit >= step - 2 is a real one
        assert acts.index(next(a for a in acts if a > r)) + 1 > 2
    grow = list(range(1, world + 1)) + list(range(world - 1, 0, -1))
    assert any(acts[i:i + len(grow)] == grow for i in range(len(acts)))
    kinds = [(s.algo, s.block) for s in steps]
    assert set(kinds) == set(GC.STEP_KINDS) and all(kinds[i] != kinds[i + 1] for i in range(len(kinds) - 1))


@pytest.mark.parametrize("world", list(range(2, 9)) + [16, 64])
def test_credit_rule_model(world):
    """Under the old rule (credit only to the active ranks) the schedule reaches a wait that is never met; crediting every
    rank meets all of them."""
    acts = GC.schedule_actives(world)
    stuck = GC.handshake_model(world, acts, "active")
    assert stuck, world
    assert {r for _, r in stuck} == set(range(1, world))  # every rank but 0 is caught by it somewhere
    assert GC.handshake_model(world, acts, "all") == []


def test_credit_rule_model_minimal_sequences():
    # 3000, 1000, 1000, 3000 columns on three ranks: ranks 1 and 2 sat out steps 2 and 3
    assert GC.handshake_model(3, [3, 1, 1, 3], "active") == [(4, 1), (4, 2)]
    assert GC.handshake_model(3, [3, 1, 3], "active") == []          # one step out is covered by the credit of step 1
    assert GC.handshake_model(3, [1, 1, 1, 3], "active") == [(4, 1), (4, 2)]  # first active since the reserve
    assert GC.handshake_model(3, [1, 1, 3], "active") == [(3, 1), (3, 2)]
    assert GC.handshake_model(3, [1, 3], "active") == []             # steps 1 and 2 wait for nothing
    for acts in ([3, 1, 1, 3], [1, 1, 1, 3], [1, 1, 3]):
        assert GC.handshake_model(3, acts, "all") == []
