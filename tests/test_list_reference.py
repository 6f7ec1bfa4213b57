"""The numpy reference of the run-merge and the list builders of tests/list_cases.py, checked on the CPU before any GPU
test relies on them: nucmut_reference against the oracle port's greedy merge (pinned to the reference's own NucMut by
test_oracle.py), the packed layout against the library's pmb_packed_bytes, and every builder against what it claims."""
import numpy as np
import pytest

import panman_b200 as pb
from tests import list_cases as LC


def _per_node_port(port, L):
    off, P, M, U = [0], [], [], []
    for v in range(L.n_nodes):
        a, b = L.off[v], L.off[v + 1]
        p, mi, nu = port.merge_msa(L.pos[a:b], L.tc[a:b]) if b > a else (np.zeros(0, np.int32),) * 3
        P.append(p); M.append(mi); U.append(nu)
        off.append(off[-1] + len(p))
    return np.asarray(off, np.int64), np.concatenate(P), np.concatenate(M).astype(np.uint8), np.concatenate(U).astype(np.uint32)


def test_reference_matches_port_merge(port):
    rng = np.random.default_rng(2024)
    for trial in range(300):
        L = LC.random_lists(rng, int(rng.integers(1, 40)), int(rng.integers(0, 600)), p_jump=[0.02, 0.3, 0.8][trial % 3],
                            p_repeat=0.01, p_type=[0.0, 0.05, 0.3][trial // 3 % 3], p_empty=0.3)
        off, pos, mi, nu, wire = LC.nucmut_reference(L.off, L.pos, L.tc)
        woff, wpos, wmi, wnu = _per_node_port(port, L)
        assert np.array_equal(off, woff) and np.array_equal(pos, wpos), trial
        assert np.array_equal(mi, wmi) and np.array_equal(nu, wnu), trial
        from oracle.oracle import wire_mut_info
        assert np.array_equal(wire, wire_mut_info(wmi, wnu)), trial
    L = LC.case_run_lengths(rng)  # runs of 1 ... 2049 records
    got, want = LC.nucmut_reference(L.off, L.pos, L.tc), _per_node_port(port, L)
    assert all(np.array_equal(g, w) for g, w in zip(got, want))


def test_reference_with_breaks_matches_pangraph_merge(port):
    """Gap-slot columns (as test_emulation.py::test_run_merge_logic_matches_oracle sets them up): column c = (gap position
    j, slot k), and consecutive columns merge only inside one gap position -- the break is at every slot 0."""
    rng = np.random.default_rng(77)
    for trial in range(300):
        widths = rng.integers(1, 12, size=60)
        col_j = np.repeat(np.arange(len(widths)), widths)
        col_k = np.concatenate([np.arange(w) for w in widths])
        brk = (col_k == 0).astype(np.uint8)
        n = int(rng.integers(1, len(col_j)))
        cols = np.sort(rng.choice(len(col_j), size=n, replace=False))
        ty = np.cumsum(rng.random(n) < 0.1) % 3
        tc = ((ty << 4) | rng.integers(0, 16, size=n)).astype(np.uint8)
        base = int(rng.integers(0, 1 << 20))
        off, pos, mi, nu, _ = LC.nucmut_reference([0, n], cols + base, tc, brk, col_base=base)
        _, op_, og, wmi, wnu = port.merge_pangraph(1, np.zeros(n, np.int32), col_j[cols], col_k[cols], tc)
        c = pos - base
        assert off[-1] == len(op_) and np.array_equal(col_j[c], op_) and np.array_equal(col_k[c], og), trial
        assert np.array_equal(mi, wmi) and np.array_equal(nu, wnu), trial


def test_pack_shard_layout_matches_library():
    L = pb.load_library()  # pmb_packed_bytes is arithmetic: no device
    rng = np.random.default_rng(3)
    for n_nodes, cap in [(1, 0), (1, 1), (2, 3), (255, 1000), (257, 4097), (4095, 17), (4097, 1 << 20), (299_999, 12_345_679)]:
        assert LC.packed_layout(n_nodes, cap)[2] == L.pmb_packed_bytes(n_nodes, cap), (n_nodes, cap)
    lists = LC.random_lists(rng, 9, 50)
    buf = LC.pack_shard(lists.off, lists.pos, lists.tc, 9, 53)
    pos_off, tc_off, total = LC.packed_layout(9, 53)
    assert len(buf) == total == L.pmb_packed_bytes(9, 53) and pos_off % 16 == 0 and tc_off % 16 == 0
    assert tuple(buf[:16].view(np.int64)) == (50, 9) and np.array_equal(buf[16:16 + 80].view(np.int64), lists.off)
    assert np.array_equal(buf[pos_off:pos_off + 200].view(np.int32), lists.pos) and np.array_equal(buf[tc_off:tc_off + 50], lists.tc)
    bad = LC.pack_shard(lists.off, lists.pos, lists.tc, 9, 53, n_override=-1, nodes_override=10)
    assert tuple(bad[:16].view(np.int64)) == (-1, 10)


def _sorted_within_nodes(L):
    node = L.node_of()
    d = np.diff(L.pos.astype(np.int64))
    return bool(np.all((d >= 0) | (node[1:] != node[:-1])))


def test_builders_make_what_they_claim():
    rng = np.random.default_rng(5)
    built = {}
    for name, make in LC.cases().items():
        if name == "huge":
            continue
        L = make(rng)
        built[name] = L
        assert _sorted_within_nodes(L) and L.pos.min() >= 0 and int(L.pos.max()) <= LC.POS_LIMIT - 2, name
        assert (L.tc >> 4).max() <= 3, name
    # runs of every length around the piece and the block, split by a gap, a type change at the next position, a repeat
    rl = LC.run_lengths(built["run_lengths"])
    for k in LC.RUN_LENGTHS:
        assert (rl == k).sum() >= 6, k
    L = built["run_lengths"]
    assert [int(x) for x in np.diff(L.off)[[0, 2, 5]]] == [0, 0, 0]
    a, b = L.off[3], L.off[4]
    p, t = L.pos[a:b].astype(np.int64), L.tc[a:b] >> 4
    assert np.all(np.diff(p) == 1) and (np.diff(t.astype(int)) != 0).sum() == 3 * len(LC.RUN_LENGTHS) - 1
    a, b = L.off[4], L.off[5]
    assert (np.diff(L.pos[a:b].astype(np.int64)) == 0).sum() == 1
    # one run longer than a round of the break max-scan, covering the whole second round
    L = built["long_run"]
    br = np.flatnonzero(LC.breaks(L))
    s = br[np.argmax(np.diff(np.append(br, L.n)))]
    assert LC.run_lengths(L).max() == LC.LONG_RUN > 3_000_000
    assert s < LC.RM_ROUND and s + LC.LONG_RUN > 2 * LC.RM_ROUND
    # breaks at k * 2048 - 1, k * 2048, k * 2048 + 1: every placed one, and in node 1 no other
    L = built["block_edges"]
    want = LC.block_edge_breaks()
    br = np.flatnonzero(LC.breaks(L))
    assert np.array_equal(br[br > L.off[1]], np.asarray(want)) and L.off[1] == LC.RM_BLOCK
    assert {i % LC.RM_BLOCK for i in want} == {LC.RM_BLOCK - 1, 0, 1}
    # empty nodes first, last and in a long stretch
    c = np.diff(built["empty_stretches"].off)
    assert c[:3000].sum() == 0 and c[-3000:].sum() == 0 and c[8000:15000].sum() == 0 and c[3000] > 0
    for n in LC.NODE_COUNTS:
        assert built[f"nodes_{n}"].n_nodes == n
    assert int(built["high_positions"].pos.max()) == LC.POS_LIMIT - 2


def test_huge_case_and_reference_at_scale():
    """More than 8192 run-merge blocks; the reference handles it vectorised."""
    L = LC.case_huge(np.random.default_rng(8))
    assert L.n > LC.PIECE_ROUND and _sorted_within_nodes(L)
    off, pos, mi, nu, wire = LC.nucmut_reference(L.off, L.pos, L.tc)
    assert int(off[-1]) == len(pos) and int((mi >> 4).astype(np.int64).sum()) == L.n
    assert int(off[-1]) > LC.PIECE_ROUND // 2


def test_split_and_concat():
    rng = np.random.default_rng(9)
    L = LC.random_lists(rng, 300, 20_000)
    for k, empty in [(1, ()), (2, (0,)), (3, (1,)), (8, (0, 3, 7)), (17, (5, 6, 16)), (64, tuple(range(0, 64, 5)))]:
        cuts = LC.cuts_for(rng, L, k, empty)
        shards = LC.split_columns(L, cuts)
        assert len(shards) == k and all(shards[s].n == 0 for s in empty)
        assert LC.concat_shards(shards).same_as(L)
        if k >= 3:  # runs straddle the cuts, and some nodes hold records in some shards only
            nz = np.array([np.diff(s.off) > 0 for s in shards])
            assert ((nz.sum(0) > 0) & (nz.sum(0) < k - len(empty))).any()
        for r in (1, 2, 3):
            t = LC.trim_to_residue(shards[-1] if shards[-1].n else L, r)
            assert t.n % 4 == r and t.n_nodes == L.n_nodes


@pytest.mark.parametrize("col_base", [0, 1000])
def test_reference_break_indexing(col_base):
    """col_break is indexed by position - col_base: a break placed at a column splits the run there and nowhere else."""
    pos = np.arange(col_base + 10, col_base + 40, dtype=np.int32)
    tc = np.zeros(30, np.uint8)
    brk = np.zeros(50, np.uint8)
    brk[[13, 14, 30]] = 1
    off, p, mi, _, _ = LC.nucmut_reference([0, 30], pos, tc, brk, col_base)
    starts = [int(x) - col_base for x in p]
    assert starts == [10, 13, 14, 20, 26, 30, 36] and list(mi >> 4) == [3, 1, 6, 6, 4, 6, 4]
