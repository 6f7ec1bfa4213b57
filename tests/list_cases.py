"""Mutation lists for the list kernels behind the pass (no GPU needed): the shard pack and merge (pack_result_kernel,
merge_count/copy_kernel, scan_sums/apply_kernel) and the record-parallel run-merge (rm_*_kernel, compact_scan_kernel for
the piece counts). Each builder returns node-major lists, position-sorted within each node, with the type (0-3) in the
high nibble and the code (0-15) in the low one -- what a pass or a shard merge hands to pmb_merge_runs. The edges are
placed on purpose: runs around the six-record piece and the 2048-record block, one run longer than a 1024-block round of
the break max-scan, breaks at block edges, stretches of empty nodes, node counts around the 4096-node scan tile, positions
up to 2^31 - 2 and a list longer than one round of the piece-count scan. nucmut_reference is the plain reference of
pmb_merge_runs; pack_shard writes the packed shard layout of pmb_pack_result."""
from dataclasses import dataclass

import numpy as np

from oracle.oracle import wire_mut_info

RM_BLOCK = 2048                  # records per block of the run-merge kernels (pmb_kernels.cuh RM_BLOCK)
RM_ROUND = 1024 * RM_BLOCK       # records per 1024-block round of rm_scan_max_kernel
PIECE_ROUND = 8192 * RM_BLOCK    # records per round of compact_scan_kernel over the per-block piece counts
SCAN_TILE = 4096                 # nodes per block of the shard merge's offset scan
POS_LIMIT = 2 ** 31              # positions are int32
RUN_LENGTHS = (1, 5, 6, 7, 12, 13, 2047, 2048, 2049)


@dataclass
class Lists:
    off: np.ndarray  # int64, n_nodes + 1
    pos: np.ndarray  # int32
    tc: np.ndarray   # uint8, (type << 4) | code

    @property
    def n_nodes(self) -> int:
        return len(self.off) - 1

    @property
    def n(self) -> int:
        return int(self.off[-1])

    def node_of(self) -> np.ndarray:
        return np.repeat(np.arange(self.n_nodes, dtype=np.int64), np.diff(self.off))

    def same_as(self, o: "Lists") -> bool:
        return np.array_equal(self.off, o.off) and np.array_equal(self.pos, o.pos) and np.array_equal(self.tc, o.tc)


def _lists(counts, pos, tc) -> Lists:
    off = np.zeros(len(counts) + 1, np.int64)
    np.cumsum(counts, out=off[1:])
    assert off[-1] == len(pos) == len(tc)
    pos = np.asarray(pos, np.int64)
    assert len(pos) == 0 or (pos.min() >= 0 and pos.max() < POS_LIMIT - 1)
    return Lists(off, pos.astype(np.int32), np.asarray(tc, np.uint8))


def breaks(lists: Lists, col_break=None, col_base: int = 0) -> np.ndarray:
    """Records that start a run: a node's first record, a position that is not the previous + 1, a type change, or a
    column the caller marks as a break (col_break[position - col_base])."""
    n = lists.n
    p = lists.pos.astype(np.int64)
    ty = lists.tc >> 4
    brk = np.zeros(n, bool)
    a = lists.off[:-1]
    brk[a[a < lists.off[1:]]] = True
    if n:
        brk[0] = True
        brk[1:] |= (p[1:] != p[:-1] + 1) | (ty[1:] != ty[:-1])
    if col_break is not None and n:
        brk |= np.asarray(col_break, bool)[p - int(col_base)]
    return brk


def run_lengths(lists: Lists, col_break=None, col_base: int = 0) -> np.ndarray:
    s = np.flatnonzero(breaks(lists, col_break, col_base))
    return np.diff(np.append(s, lists.n))


def nucmut_reference(off, pos, tc, col_break=None, col_base: int = 0):
    """pmb_merge_runs in plain numpy (reference src/panman.cpp:1445-1466 + NucMut ctor src/panman.hpp:109-151): every
    maximal run is cut greedily into pieces of at most six records. Returns (node_offsets, nucPosition, mutInfo, nucs,
    wire form of mutInfo)."""
    L = Lists(np.asarray(off, np.int64), np.asarray(pos, np.int32), np.asarray(tc, np.uint8))
    n = L.n
    idx = np.arange(n, dtype=np.int64)
    start = np.maximum.accumulate(np.where(breaks(L, col_break, col_base), idx, 0)) if n else idx  # run start of each record
    piece = (idx - start) % 6 == 0
    first = np.flatnonzero(piece)
    length = np.diff(np.append(first, n))
    assert length.max(initial=1) <= 6
    code = (L.tc & 15).astype(np.uint32)
    nucs = np.zeros(len(first), np.uint32)
    for k in range(6):
        has = k < length
        nucs[has] += code[first[has] + k] << np.uint32(4 * (5 - k))
    mut_info = ((length << 4) + (L.tc[first] >> 4)).astype(np.uint8)
    before = np.zeros(n + 1, np.int64)
    np.cumsum(piece, out=before[1:])
    return (before[L.off], L.pos[first].copy(), mut_info, nucs, wire_mut_info(mut_info, nucs).astype(np.uint32))


# ---------------------------------------------------------------------------------------------------------- packing
def packed_layout(n_nodes: int, cap: int):
    """Byte offsets of the packed shard sections (pmb_kernels.cuh packed_pos_offset / packed_tc_offset / packed_bytes)."""
    pos_off = (16 + (n_nodes + 1) * 8 + 15) // 16 * 16
    tc_off = (pos_off + cap * 4 + 15) // 16 * 16
    return pos_off, tc_off, (tc_off + cap + 15) // 16 * 16


def pack_shard(off, pos, tc, n_nodes: int, capacity: int, n_override=None, nodes_override=None) -> np.ndarray:
    """{int64 n_mut, int64 n_nodes | int64 offsets[N+1] | int32 pos[cap] | uint8 type_code[cap]}, 16-byte aligned sections.
    n_override / nodes_override forge the header (a shard over capacity, flagged by its packer, or packed for another tree)."""
    n = int(off[-1])
    assert len(off) == n_nodes + 1 and n <= capacity
    pos_off, tc_off, total = packed_layout(n_nodes, capacity)
    out = np.zeros(total, np.uint8)
    out[:16].view(np.int64)[:] = (n if n_override is None else n_override, n_nodes if nodes_override is None else nodes_override)
    out[16:16 + 8 * (n_nodes + 1)].view(np.int64)[:] = off
    out[pos_off:pos_off + 4 * n].view(np.int32)[:] = np.asarray(pos, np.int32)[:n]
    out[tc_off:tc_off + n] = np.asarray(tc, np.uint8)[:n]
    return out


# ---------------------------------------------------------------------------------------------------------- shards
def split_columns(lists: Lists, cuts) -> list:
    """Column-range shards: shard s holds the records with cuts[s - 1] <= position < cuts[s] (cuts ascending, k - 1 of
    them for k shards). Runs that cross a cut straddle two shards; equal cuts leave a shard empty."""
    cuts = np.asarray(cuts, np.int64)
    assert np.all(np.diff(cuts) >= 0)
    shard = np.searchsorted(cuts, lists.pos.astype(np.int64), side="right")
    node = lists.node_of()
    out = []
    for s in range(len(cuts) + 1):
        m = shard == s
        out.append(_lists(np.bincount(node[m], minlength=lists.n_nodes), lists.pos[m], lists.tc[m]))
    return out


def concat_shards(shards) -> Lists:
    """What the shard merge must produce: each node's per-shard lists concatenated in shard order."""
    node = np.concatenate([s.node_of() for s in shards])
    sid = np.concatenate([np.full(s.n, k, np.int64) for k, s in enumerate(shards)])
    order = np.argsort(node * len(shards) + sid, kind="stable")
    pos = np.concatenate([s.pos for s in shards])[order]
    tc = np.concatenate([s.tc for s in shards])[order]
    return Lists(np.concatenate([[0], np.cumsum(sum(np.diff(s.off) for s in shards))]).astype(np.int64), pos, tc)


def cuts_for(rng, lists: Lists, k: int, empty=()) -> np.ndarray:
    """k - 1 cuts at positions of records (inside runs, so runs straddle shards); the shards listed in `empty` hold none."""
    cuts = np.sort(rng.choice(lists.pos.astype(np.int64), size=k - 1)) if lists.n else np.zeros(k - 1, np.int64)
    for s in sorted(empty):
        if s == 0:
            cuts[0] = -1
        elif s == k - 1:
            cuts[k - 2] = POS_LIMIT
        else:
            cuts[s] = cuts[s - 1]
    return cuts


def trim_to_residue(lists: Lists, r: int) -> Lists:
    """Drop the last 0-3 records so that the count is r mod 4 (merge_copy_kernel copies four records per thread)."""
    d = (lists.n - r) % 4 if lists.n >= 4 else 0
    n = lists.n - d
    return Lists(np.minimum(lists.off, n), lists.pos[:n].copy(), lists.tc[:n].copy())


# ---------------------------------------------------------------------------------------------------------- builders
def random_lists(rng, n_nodes: int, n_rec: int, p_jump=0.3, p_repeat=0.002, p_type=0.05, p_empty=0.2, max_base=1000) -> Lists:
    """Random records: runs of consecutive positions broken by jumps, repeated positions and type changes; a share of the
    nodes holds nothing."""
    w = rng.exponential(size=n_nodes) * (rng.random(n_nodes) >= p_empty)
    if not w.any():
        w[rng.integers(n_nodes)] = 1.0
    counts = rng.multinomial(n_rec, w / w.sum())
    u = rng.random(n_rec)
    step = np.where(u < p_jump, rng.integers(2, 9, size=n_rec), 1)
    step[u > 1 - p_repeat] = 0
    cs = np.cumsum(step)
    off = np.concatenate([[0], np.cumsum(counts)])
    node = np.repeat(np.arange(n_nodes), counts)
    pos = cs - cs[off[:-1][node]] + rng.integers(0, max_base + 1, size=n_nodes)[node]
    ty = np.cumsum(rng.random(n_rec) < p_type) % 4
    tc = (ty << 4) | rng.integers(0, 16, size=n_rec)
    return _lists(counts, pos, tc)


def _runs(rng, lengths, starts, types):
    """Records of consecutive runs: run j covers positions starts[j] .. starts[j] + lengths[j] - 1 with type types[j]."""
    lengths = np.asarray(lengths, np.int64)
    first = np.concatenate([[0], np.cumsum(lengths)[:-1]])
    i = np.arange(lengths.sum())
    pos = np.repeat(np.asarray(starts, np.int64), lengths) + i - np.repeat(first, lengths)
    tc = (np.repeat(np.asarray(types, np.int64), lengths) << 4) | rng.integers(0, 16, size=len(i))
    return pos, tc


def case_run_lengths(rng) -> Lists:
    """Runs of every length in RUN_LENGTHS (three of each, shuffled, so that the long ones meet block edges at several
    phases). Node 1 separates its runs by position gaps, node 3 by a type change at the next position (the runs are
    consecutive in position), node 4 repeats a position inside a run; nodes 0, 2 and 5 are empty."""
    lens = rng.permutation(np.repeat(RUN_LENGTHS, 3))
    gap_starts = np.cumsum(np.append(0, lens[:-1] + 2)) + 10
    p1, t1 = _runs(rng, lens, gap_starts, rng.integers(0, 4, size=len(lens)))
    lens3 = rng.permutation(lens)
    p3, t3 = _runs(rng, lens3, np.cumsum(np.append(0, lens3[:-1])) + 5, np.arange(len(lens3)) % 4)
    p4, t4 = _runs(rng, [13, 2049, 7], [100, 112, 3000], [1, 1, 2])  # position 112 twice: a run restarts there
    return _lists([0, len(p1), 0, len(p3), len(p4), 0], np.concatenate([p1, p3, p4]), np.concatenate([t1, t3, t4]))


LONG_RUN = 3_200_001


def case_long_run(rng) -> Lists:
    """One node holding one run of LONG_RUN consecutive positions. Random nodes before it end shortly before the first
    1024-block round of the break max-scan does, so the run covers the whole second round without a break and its start
    lies more than one round back from its last records."""
    head = random_lists(rng, 40, RM_ROUND - 5000)
    p, t = _runs(rng, [LONG_RUN], [1000], [2])
    tail = random_lists(rng, 3, 3000)
    counts = np.concatenate([np.diff(head.off), [0, LONG_RUN, 0], np.diff(tail.off)])
    return _lists(counts, np.concatenate([head.pos, p, tail.pos]), np.concatenate([head.tc, t, tail.tc]))


BLOCK_EDGE_KS = range(2, 30)


def case_block_edges(rng) -> Lists:
    """One node of consecutive positions (node 1; node 0 holds exactly one block of random records) whose runs break at
    list index k * 2048 - 1, k * 2048 and/or k * 2048 + 1 -- the subset cycles with k -- by a position jump or, for odd k,
    a type change."""
    head = random_lists(rng, 1, RM_BLOCK, p_empty=0.0)
    n1 = (BLOCK_EDGE_KS[-1] + 1) * RM_BLOCK
    gi = np.arange(RM_BLOCK, RM_BLOCK + n1)  # list index of node 1's records
    jump = np.zeros(n1, bool)
    tchg = np.zeros(n1, bool)
    for k in BLOCK_EDGE_KS:
        for d in (-1, 0, 1):
            if (k % 7 + 1) >> (d + 1) & 1:
                (tchg if k % 2 else jump)[k * RM_BLOCK + d - RM_BLOCK] = True
    assert not (jump[0] or tchg[0]) and gi[0] == RM_BLOCK
    pos = 50 + np.arange(n1) + np.cumsum(jump)
    ty = np.cumsum(tchg) % 4
    tc = (ty << 4) | rng.integers(0, 16, size=n1)
    return _lists([RM_BLOCK, n1, 0], np.concatenate([head.pos, pos]), np.concatenate([head.tc, tc]))


def block_edge_breaks():
    """The list indices at which case_block_edges places its breaks."""
    return sorted(k * RM_BLOCK + d for k in BLOCK_EDGE_KS for d in (-1, 0, 1) if (k % 7 + 1) >> (d + 1) & 1)


def case_empty_stretches(rng) -> Lists:
    """20 000 nodes: the first 3000 and the last 3000 empty, 7000 empty ones in the middle, and elsewhere nodes of 0-3
    records, so that four consecutive records often span two or more empty nodes."""
    N = 20_000
    counts = rng.choice([0, 0, 1, 1, 2, 3], size=N)
    counts[:3000] = 0
    counts[-3000:] = 0
    counts[8000:15000] = 0
    counts[3000] = max(counts[3000], 1)
    base = random_lists(rng, 1, int(counts.sum()), p_empty=0.0)
    node = np.repeat(np.arange(N), counts)
    off = np.concatenate([[0], np.cumsum(counts)])
    pos = base.pos.astype(np.int64) - base.pos[off[:-1][node]] + rng.integers(0, 100, size=N)[node]
    return _lists(counts, pos, base.tc)


NODE_COUNTS = (1, 255, 257, 4095, 4097, 299_999)


def case_nodes(rng, n_nodes: int) -> Lists:
    """Random lists over n_nodes nodes (around the 4096-node tile of the offset scan, and a tree of about 300 k nodes)."""
    return random_lists(rng, n_nodes, max(3 * n_nodes, 20_000))


def case_high_positions(rng) -> Lists:
    """Positions up to 2^31 - 2: a run that ends there, runs just below it, and one node near position 0."""
    top = POS_LIMIT - 2
    p1, t1 = _runs(rng, [7, 2049, 13], [top - 5000, top - 2060, top - 12], [0, 1, 1])
    p2, t2 = _runs(rng, [12, 6], [0, top - 5], [3, 3])
    p3, t3 = _runs(rng, [1, 5], [top - 100, top - 98], [2, 2])
    return _lists([0, len(p1), 0, len(p2), len(p3)], np.concatenate([p1, p2, p3]), np.concatenate([t1, t2, t3]))


HUGE_RECORDS = PIECE_ROUND + 500_000


def case_huge(rng) -> Lists:
    """More than 8192 blocks of records (17.3 M), so the piece-count scan carries its sum into a second round."""
    return random_lists(rng, 4097, HUGE_RECORDS, p_jump=0.5)


def cases():
    """name -> builder(rng) of every crafted list set."""
    c = {"run_lengths": case_run_lengths, "long_run": case_long_run, "block_edges": case_block_edges,
         "empty_stretches": case_empty_stretches, "high_positions": case_high_positions, "huge": case_huge}
    for n in NODE_COUNTS:
        c[f"nodes_{n}"] = lambda rng, n=n: case_nodes(rng, n)
    return c
