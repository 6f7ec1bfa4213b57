"""Inputs for the column-sharded group (pmb_group_*; no GPU needed): the column ranges, the per-rank uploads and the
hand-shake between the ranks' streams and rank 0's merge stream. No tests here.

range_reference restates pmb_group_column_range. boundary_case builds an alignment whose features sit on every rank
boundary b: columns b - 1, b and b + 1 each carry their own parent_code, root_override and fwd_root_ref; runs of 1 ... 13
columns end at b, start at b and straddle b; and a clade turns from deleted to substituted exactly at b, so the record
type changes there. pack_padded lays rows out with a stride wider than the packed row and garbage in the unused high
nibble of an odd width. The widths put the group on and around its tile counts (one tile, world tiles, world - 1 tiles).

The schedules are widths for one group on one tree, step after step: each rank sits out 1, 2 and 3 consecutive steps
and comes back, the group grows from one active rank to all and shrinks back, and ranks become active for the first time
several steps after the mailbox was reserved. handshake_model replays the arrive / credit words of such a schedule under
a credit rule and lists the waits that could never be met."""
from dataclasses import dataclass

import numpy as np

TILE = 1024          # column granule of a range (pmb_group.cu GROUP_TILE)
RUN_LENGTHS = tuple(range(1, 14))
MAX_WORLD = 1024
FEATURE_ROWS = 120  # rows the features of one boundary take
STEP_KINDS = ((0, 0), (1, 0), (0, 1), (1, 1))  # (algo, block mode) in turn along a schedule


# ---------------------------------------------------------------------------------------------------------- ranges
def range_reference(world: int, n_cols: int, rank: int):
    """[begin, end) of `rank`: the ceil(n_cols / 1024) tiles are dealt out in contiguous blocks, the first tiles % world
    ranks one tile more than the rest, and the last tile is cut at n_cols. Ranks past the tile count own nothing."""
    assert 1 <= world and 0 <= rank < world and n_cols >= 0
    tiles = -(-n_cols // TILE)
    counts = [tiles // world + (1 if r < tiles % world else 0) for r in range(rank + 1)]
    first = sum(counts[:rank])
    return min(n_cols, first * TILE), min(n_cols, (first + counts[rank]) * TILE)


def active_ranks(world: int, n_cols: int) -> int:
    """The ranks with a non-empty range: always the first min(world, tiles) of them."""
    return min(world, -(-n_cols // TILE))


def boundaries(world: int, n_cols: int) -> list:
    """The first column of every active rank but rank 0."""
    return [range_reference(world, n_cols, r)[0] for r in range(1, active_ranks(world, n_cols))]


def width_for(world: int, active: int, rng) -> int:
    """A width at which exactly `active` ranks own columns; at active == world it may hold more tiles than ranks."""
    assert 1 <= active <= world
    if active < world:
        return (active - 1) * TILE + int(rng.integers(1, TILE + 1))
    return (world - 1) * TILE + int(rng.integers(1, 3 * TILE))


def boundary_widths(world: int) -> list:
    """1, 1023, 1024, 1025, world * 1024 - 1, world * 1024, world * 1024 + 1, (world + 1) * 1024 + 1 and a width of
    world - 1 tiles."""
    w = {1, 1023, 1024, 1025, world * TILE - 1, world * TILE, world * TILE + 1, (world + 1) * TILE + 1}
    if world >= 2:
        w.add((world - 1) * TILE - 517)
    return sorted(w)


# ---------------------------------------------------------------------------------------------------------- matrices
@dataclass
class Case:
    codes: np.ndarray        # uint8 (n_rows, n_cols), one code per byte
    parent_code: np.ndarray  # uint8 n_cols
    root_override: np.ndarray = None  # int8 n_cols or None
    fwd_root_ref: np.ndarray = None   # int8 n_cols or None
    leaf_present: np.ndarray = None   # uint8 n_rows or None
    algo: int = 0
    block: int = 0
    bounds: tuple = ()
    type_rows: tuple = ()    # the rows that turn from deleted to substituted at each boundary

    @property
    def flags(self) -> int:
        return 2 if self.block else 0  # PMB_FLAG_BLOCK_MODE

    def sliced(self, a: int, b: int):
        """parent_code, root_override, fwd_root_ref of columns [a, b)."""
        cut = lambda x: None if x is None else np.ascontiguousarray(x[a:b])
        return cut(self.parent_code), cut(self.root_override), cut(self.fwd_root_ref)


def run_slots(b: int, n_cols: int):
    """(label, run length, first column, end column) of every run placed at boundary b, clipped to the alignment."""
    out = []
    for L in RUN_LENGTHS:
        for label, a in (("ends", b - L), ("starts", b), ("straddles", b - (L + 1) // 2)):
            lo, hi = max(0, a), min(n_cols, a + L)
            if hi > lo:
                out.append((label, L, lo, hi))
    return out


def boundary_case(n_rows: int, world: int, n_cols: int, algo: int, block: int, seed: int, presence=False, override=False,
                  fwd=False, noise=0.01) -> Case:
    """A matrix for `world` ranks with its features on every boundary (see the module docstring). Each run goes to its own
    group of 1 ... 4 consecutive rows (a clade or neighbouring clades: rows follow pre-order); with n_rows >= FEATURE_ROWS
    the groups of one boundary do not overlap."""
    assert not (fwd and (algo == 1 or block)), "fwd_root_ref belongs to Fitch in nucleotide mode"
    rng = np.random.default_rng(seed)
    nst = 3 if block else 16
    base = rng.integers(1, min(nst, 5), size=n_cols)  # never a gap: a gap at a boundary is a feature
    codes = np.repeat(base[None, :], n_rows, 0)
    codes = np.where(rng.random(codes.shape) < noise, rng.integers(0, nst, size=codes.shape), codes).astype(np.uint8)
    pc = rng.integers(0, nst, size=n_cols).astype(np.uint8)
    ro = np.where(rng.random(n_cols) < 0.3, rng.integers(0, nst, size=n_cols), -1).astype(np.int8) if override else None
    fr = np.where(rng.random(n_cols) < 0.3, rng.integers(0, nst, size=n_cols), -1).astype(np.int8) if fwd else None
    bounds = boundaries(world, n_cols)
    next_row, type_rows = 0, []

    def rows(k):
        nonlocal next_row
        r0 = next_row % n_rows
        next_row += k
        return np.arange(r0, min(n_rows, r0 + k))

    for bi, b in enumerate(bounds):
        cols = np.arange(b - 1, min(n_cols, b + 2))
        pc[cols] = (np.arange(len(cols)) + bi) % nst  # three different parent codes
        if ro is not None:
            ro[cols] = (np.arange(len(cols)) + bi + 1) % nst
        if fr is not None:
            fr[cols] = (np.arange(len(cols)) + bi + 2) % nst
        next_row = 0  # the features of two boundaries are 1024 columns apart: they may share rows
        for k, (_, L, lo, hi) in enumerate(run_slots(b, n_cols)):
            r = rows(1 + (L + k) % 4)
            shift = 0 if block else k % 3  # never the base state, never a gap
            codes[np.ix_(r, np.arange(lo, hi))] = ((base[lo:hi] + shift) % (nst - 1) + 1)[None, :]
        r = rows(3)
        lo, hi = max(0, b - 6), min(n_cols, b + 6)
        codes[np.ix_(r, np.arange(lo, b))] = 0                       # deleted up to b - 1
        codes[np.ix_(r, np.arange(b, hi))] = (base[b:hi] % (nst - 1) + 1)[None, :]  # substituted from b on
        type_rows.append(tuple(int(x) for x in r))
        assert next_row <= FEATURE_ROWS
    lp = None
    if presence and n_rows > 1:
        lp = (rng.random(n_rows) < 0.75).astype(np.uint8)
        if bounds:  # the boundary features stay visible, and rows past them are omitted for sure
            lp[:FEATURE_ROWS] = 1
            lp[FEATURE_ROWS::2] = 0
        lp[0] = 1
    return Case(codes, pc, ro, fr, lp, algo, block, tuple(bounds), tuple(type_rows))


def pack_padded(codes: np.ndarray, pad: int, seed: int = 0):
    """(buffer, stride): rows of ceil(n_cols / 2) packed bytes followed by `pad` bytes of 0xEE, and for an odd width
    garbage in the high nibble of each row's last byte (column n_cols does not exist)."""
    import panman_b200 as pb

    c4 = pb.pack_nibbles(codes)
    n_rows, w = c4.shape
    out = np.full((n_rows, w + pad), 0xEE, np.uint8)
    out[:, :w] = c4
    if codes.shape[1] % 2:
        out[:, w - 1] |= (np.random.default_rng(seed).integers(1, 16, size=n_rows) << 4).astype(np.uint8)
    return out, w + pad


# ---------------------------------------------------------------------------------------------------------- schedules
@dataclass
class Step:
    active: int
    n_cols: int
    algo: int
    block: int


def schedule_actives(world: int) -> list:
    """Active-rank counts of consecutive steps right after a reserve: three steps on rank 0 alone (the other ranks then
    become active for the first time at a step > 2), growth to every rank and shrinking back to one, a step on all of them,
    then for every rank r >= 1 and d = 1, 2, 3 a stretch of d steps on ranks < r followed by a step on all of them."""
    if world == 1:
        return [1, 1, 1]
    acts = [1, 1, 1] + list(range(2, world + 1)) + list(range(world - 1, 0, -1)) + [world]
    for d in (1, 2, 3):
        for r in range(1, world):
            acts += [r] * d + [world]
    return acts


def schedule(world: int, seed: int) -> list:
    """schedule_actives with a width per step and (algo, block mode) alternating along it."""
    rng = np.random.default_rng(seed)
    return [Step(a, width_for(world, a, rng), *STEP_KINDS[i % len(STEP_KINDS)]) for i, a in enumerate(schedule_actives(world))]


def inactive_stretches(actives: list, rank: int) -> list:
    """Lengths of the maximal stretches of steps in which `rank` owns nothing and after which it is active again."""
    out, run = [], 0
    for a in actives:
        if rank >= a:
            run += 1
        else:
            if run:
                out.append(run)
            run = 0
    return out


def handshake_model(world: int, actives: list, rule: str) -> list:
    """The arrive / credit words of pmb_group.cu over steps 1, 2, ... (seq restarts at 0 on a reserve) with actives[s - 1]
    ranks active at step s. An active rank r waits for credit[r] >= s - 2 before it packs (s > 2); rank 0's merge stream
    waits for arrive[r] >= s of every active rank, merges and writes credit = s into the boxes of the ranks of `rule`:
    "active" (r < active) or "all" (r < world). The merge of step s cannot complete before rank r's wait at step s, so
    the credits that wait can see are those of steps 1 ... s - 1. Returns every (step, rank) whose wait could never be
    met, each evaluated as if the steps before it had completed."""
    assert rule in ("active", "all")
    credit = [0] * world
    stuck = []
    for s, act in enumerate(actives, 1):
        # every active rank that gets past its wait writes arrive[r] = s, which is all the merge of step s waits for
        stuck += [(s, r) for r in range(act) if s > 2 and credit[r] < s - 2]
        for r in range(act if rule == "active" else world):
            credit[r] = s
    return stuck
