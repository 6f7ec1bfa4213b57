"""The list kernels behind the pass on the device, at their block, scan and capacity edges (cases from tests/list_cases.py):
the shard pack and merge (pmb_pack_result, pmb_merge_packed) and the record-parallel run-merge (pmb_merge_runs) against
plain references -- concat_shards for the merged lists, nucmut_reference for the NucMut fields -- and the ordered
compaction of a pass against the oracle port where a (node, tile) directory entry holds its largest count. Also the
int32 range of positions: a batch whose columns pass 2^31 - 1 is refused."""
import numpy as np
import pytest

import panman_b200 as pb
from oracle.oracle import random_tree
from tests import list_cases as LC

pytestmark = pytest.mark.gpu

ERR_INVALID, ERR_CAPACITY = -1, -9


@pytest.fixture(scope="module")
def ctx():
    c = pb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def tree_of():
    """A tree of exactly n_nodes nodes (odd, >= 3): merging and run-merging need only the node count."""
    cache = {}

    def get(n_nodes):
        if n_nodes not in cache:
            L = (n_nodes + 1) // 2
            cache[n_nodes] = random_tree(L, 900 + L % 97, "binary" if L <= 5000 else "caterpillar")
            assert cache[n_nodes].n_nodes == n_nodes
        return cache[n_nodes]

    return get


def _set_tree(c, tree):
    c.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)


def _pad(lists, n_nodes):
    """The same records over n_nodes nodes: the added nodes are empty."""
    extra = n_nodes - lists.n_nodes
    return LC.Lists(np.concatenate([lists.off, np.full(extra, lists.off[-1], np.int64)]), lists.pos, lists.tc)


def _tree_size(n):
    return max(3, n | 1)


class _Arr:
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


def _device_lists(r, n_nodes):
    """The lists a pmb_result points to in device memory (pmb_merge_packed does not synchronise: the caller does)."""
    import torch

    torch.cuda.synchronize()
    off = torch.as_tensor(_Arr(r.node_offsets, n_nodes + 1, "<i8"), device="cuda").cpu().numpy()
    n = int(off[-1])
    pos = torch.as_tensor(_Arr(r.pos, max(n, 1), "<i4"), device="cuda")[:n].cpu().numpy()
    tc = torch.as_tensor(_Arr(r.type_code, max(n, 1), "|u1"), device="cuda")[:n].cpu().numpy()
    return LC.Lists(off, pos, tc)


def _packed(shards, cap, forge=None):
    """The shards packed back to back at `cap` records each, on the device; forge = (shard, pack_shard overrides)."""
    import torch

    bufs = []
    for k, s in enumerate(shards):
        kw = forge[1] if forge is not None and forge[0] == k else {}
        bufs.append(LC.pack_shard(s.off, s.pos, s.tc, s.n_nodes, cap, **kw))
    buf = torch.from_numpy(np.concatenate(bufs)).cuda()
    torch.cuda.synchronize()
    return buf


def _same_nucmut(got, want, what):
    names = ("node_offsets", "nucPosition", "mutInfo", "nucs", "wire")
    for g, w, nm in zip(got, want, names):
        assert np.array_equal(g, w), (what, nm)


def _merge_and_check(c, shards, cap, what, stream=None):
    want = LC.concat_shards(shards)
    buf = _packed(shards, cap)
    r = c.merge_packed(len(shards), buf, cap, stream)
    assert _device_lists(r, want.n_nodes).same_as(want), (what, "merged lists")
    _same_nucmut(c.merge_runs(source=1), LC.nucmut_reference(want.off, want.pos, want.tc), what)
    del buf


# ------------------------------------------------------------------------------------------------ run-merge, crafted lists
SHARDS = {"run_lengths": (3, (1,)), "long_run": (2, ()), "block_edges": (3, ()), "empty_stretches": (8, (0, 7)),
          "high_positions": (2, ()), "huge": (2, ()), "nodes_1": (1, ()), "nodes_255": (3, ()), "nodes_257": (3, (2,)),
          "nodes_4095": (8, (3,)), "nodes_4097": (17, (0, 9, 16)), "nodes_299999": (3, (1,))}


@pytest.mark.parametrize("name", list(SHARDS))
def test_run_merge_crafted(ctx, tree_of, name):
    """Crafted lists split into column-range shards (runs straddle the cuts), merged on the device, then run-merged:
    merged lists = the per-node concatenation in shard order, NucMut fields = the numpy reference."""
    rng = np.random.default_rng(sum(map(ord, name)))
    lists = LC.cases()[name](rng)
    lists = _pad(lists, _tree_size(lists.n_nodes))
    k, empty = SHARDS[name]
    shards = LC.split_columns(lists, LC.cuts_for(rng, lists, k, empty))
    assert LC.concat_shards(shards).same_as(lists)
    _set_tree(ctx, tree_of(lists.n_nodes))
    _merge_and_check(ctx, shards, max(s.n for s in shards) + 3, name)


# ------------------------------------------------------------------------------------------------ shard merge
@pytest.mark.parametrize("n_shards", [1, 2, 3, 8, 17, 64])
def test_shard_merge(ctx, tree_of, n_shards):
    """Many shards (blockIdx.y), empty shards, nodes present in some shards only, record counts = 1, 2, 3 (mod 4) and a
    shard holding exactly `capacity` records."""
    rng = np.random.default_rng(300 + n_shards)
    N = 4097 if n_shards % 2 else 8191
    lists = LC.random_lists(rng, N, 40_000 * n_shards, p_empty=0.3)
    empty = tuple(range(1, n_shards, 4)) if n_shards >= 3 else ()
    shards = LC.split_columns(lists, LC.cuts_for(rng, lists, n_shards, empty))
    nonempty = [k for k, s in enumerate(shards) if s.n]
    for i, k in enumerate(nonempty):
        shards[k] = LC.trim_to_residue(shards[k], 1 + i % 3)
    assert [shards[k].n % 4 for k in nonempty] == [1 + i % 3 for i in range(len(nonempty))]
    assert len(nonempty) == n_shards - len(empty)
    _set_tree(ctx, tree_of(N))
    _merge_and_check(ctx, shards, max(s.n for s in shards), f"{n_shards} shards at capacity")
    _merge_and_check(ctx, shards, max(s.n for s in shards) + 13, f"{n_shards} shards")


def _over_capacity(shards, cap, k):
    """Shard k packed at `cap` but claiming cap + 1 records (its offsets too): the record past the capacity would be read
    from the padding behind the positions."""
    import torch

    buf = _packed(shards, cap).cpu().numpy()
    sb = LC.packed_layout(shards[0].n_nodes, cap)[2]
    hdr = buf[k * sb:k * sb + 16].view(np.int64)
    off = buf[k * sb + 16:k * sb + 16 + 8 * (shards[0].n_nodes + 1)].view(np.int64)
    v = int(np.flatnonzero(np.diff(shards[k].off))[-1])
    hdr[0] = cap + 1
    off[v + 1:] += 1
    out = torch.from_numpy(buf).cuda()
    torch.cuda.synchronize()
    return out


def test_bad_headers_then_clean_merge(ctx, tree_of):
    """A shard over capacity, one flagged by its packer (PACK_HDR_BAD) and one packed for another tree are skipped and
    reported; the next clean merge on the same context is correct."""
    rng = np.random.default_rng(17)
    lists = LC.random_lists(rng, 257, 30_000)
    shards = LC.split_columns(lists, LC.cuts_for(rng, lists, 3))
    cap = max(s.n for s in shards)
    if cap % 16 == 0:  # one record less: the type codes of a full shard end before its last 16-byte line does
        shards = [LC.trim_to_residue(s, 3) if s.n == cap else s for s in shards]
        cap -= 1
    k_full = int(np.argmax([s.n for s in shards]))
    _set_tree(ctx, tree_of(257))
    forged = [("over capacity", _over_capacity(shards, cap, k_full), ERR_CAPACITY),
              ("flagged", _packed(shards, cap, (1, {"n_override": -1})), ERR_CAPACITY),
              ("another tree", _packed(shards, cap, (2, {"nodes_override": 259})), ERR_INVALID)]
    for i, (what, buf, code) in enumerate(forged):
        ctx.merge_packed(3, buf, cap)
        with pytest.raises(pb.PanmanError) as e:
            if i % 2:
                ctx.merge_status()
            else:
                ctx.merge_runs(source=1)
        assert e.value.code == code, what
        _merge_and_check(ctx, shards, cap, f"clean merge after {what}")


def test_merge_on_caller_stream_and_regrow(ctx, tree_of):
    """pmb_merge_packed on a caller's torch stream and pmb_merge_runs(source = 1) behind it; small and large merges in a
    row without a synchronisation, so the library regrows its buffers while the earlier merge is still queued."""
    import torch

    rng = np.random.default_rng(23)
    N = 4097
    _set_tree(ctx, tree_of(N))
    sizes = [2_000, 3_000_000, 5_000, 6_000_000]
    sets = []
    for n_rec in sizes:
        lists = LC.random_lists(rng, N, n_rec)
        shards = LC.split_columns(lists, LC.cuts_for(rng, lists, 3))
        cap = max(s.n for s in shards)
        sets.append((shards, cap, _packed(shards, cap)))
    s = torch.cuda.Stream()
    for i in range(0, len(sets), 2):
        for shards, cap, buf in sets[i:i + 2]:  # the second grows what the first still uses
            r = ctx.merge_packed(3, buf, cap, s.cuda_stream)
        want = LC.concat_shards(shards)
        assert _device_lists(r, N).same_as(want), i
        _same_nucmut(ctx.merge_runs(source=1), LC.nucmut_reference(want.off, want.pos, want.tc), f"stream, set {i + 1}")
    for shards, cap, buf in sets[::-1]:  # back on the context's own stream, large then small
        _merge_and_check(ctx, shards, cap, f"own stream, {cap}")
    s.synchronize()


def _noisy(rng, n_leaves, n_cols, p):
    base = rng.integers(0, 4, size=n_cols)
    codes = np.repeat(base[None, :], n_leaves, 0)
    codes = np.where(rng.random(codes.shape) < p, rng.integers(0, 16, size=codes.shape), codes).astype(np.uint8)
    return codes, base.astype(np.uint8)


def test_merge_runs_beside_async_passes(ctx, port):
    """merge_runs of merged shards and of the context's own pass, interleaved with asynchronous passes in flight."""
    rng = np.random.default_rng(29)
    tree = random_tree(200, 91, "binary")
    codes, pc = _noisy(rng, tree.n_leaves, 4000, 0.3)
    want, _ = port.run(tree, 0, codes, pc, n_threads=8)
    want_nm = LC.nucmut_reference(want.node_offsets, want.pos, want.type_code)
    lists = LC.random_lists(rng, tree.n_nodes, 200_000)
    shards = LC.split_columns(lists, LC.cuts_for(rng, lists, 3, (1,)))
    cap = max(s.n for s in shards)
    merged = LC.concat_shards(shards)
    want_sh = LC.nucmut_reference(merged.off, merged.pos, merged.tc)
    buf = _packed(shards, cap)
    _set_tree(ctx, tree)
    c4 = pb.pack_nibbles(codes)
    ctx.upload(4000, tree.n_leaves, c4, c4.shape[1], pc)
    for i in range(3):
        for _ in range(i + 1):
            ctx.run_resident_async(pb.ALGO_FITCH)
        ctx.merge_packed(3, buf, cap)
        _same_nucmut(ctx.merge_runs(source=1), want_sh, f"shards beside pass {i}")
        _same_nucmut(ctx.merge_runs(source=0), want_nm, f"own pass {i}")
        ctx.run_resident_async(pb.ALGO_FITCH)
        _same_nucmut(ctx.merge_runs(source=0), want_nm, f"own pass {i}, right behind it")
        _same_nucmut(ctx.merge_runs(source=1), want_sh, f"shards again {i}")
    ctx.wait()


# ------------------------------------------------------------------------------------------------ the pass at scale
@pytest.fixture(scope="module")
def big_pass(port):
    rng = np.random.default_rng(61)
    tree = random_tree(300, 62, "binary")
    codes, pc = _noisy(rng, tree.n_leaves, 10_000, 0.8)
    wants = {algo: port.run(tree, algo, codes, pc, n_threads=16)[0] for algo in (0, 1)}
    return tree, codes, pc, wants


@pytest.mark.parametrize("algo", [0, 1])
def test_pass_at_scale(ctx, big_pass, algo):
    """A pass of more than one round of the break max-scan (2 097 152 records): lists against the oracle port, run-merge
    against the reference, pack_result at capacity n_mut (accepted) and n_mut - 1 (refused, or flagged when the pass
    is still in flight)."""
    import torch

    tree, codes, pc, wants = big_pass
    want = wants[algo]
    n_mut = int(want.node_offsets[-1])
    assert n_mut > LC.RM_ROUND
    _set_tree(ctx, tree)
    res = ctx.run_codes(tree, algo, codes, pc)
    assert np.array_equal(res.node_offsets, want.node_offsets) and np.array_equal(res.pos, want.pos)
    assert np.array_equal(res.type_code, want.type_code)
    _same_nucmut(ctx.merge_runs(), LC.nucmut_reference(want.node_offsets, want.pos, want.type_code), "pass")
    buf = torch.empty(ctx.packed_bytes(n_mut), dtype=torch.uint8, device="cuda")
    ctx.pack_result(buf, n_mut)
    ctx.wait()
    r = ctx.merge_packed(1, buf, n_mut)
    assert _device_lists(r, tree.n_nodes).same_as(LC.Lists(want.node_offsets, want.pos, want.type_code))
    with pytest.raises(pb.PanmanError) as e:
        ctx.pack_result(buf, n_mut - 1)
    assert e.value.code == ERR_CAPACITY
    ctx.run_resident_async(algo)
    small = torch.empty(ctx.packed_bytes(n_mut - 1), dtype=torch.uint8, device="cuda")
    ctx.pack_result(small, n_mut - 1)
    ctx.wait()
    torch.cuda.synchronize()
    assert tuple(small[:16].cpu().numpy().view(np.int64)) == (-1, tree.n_nodes)  # PACK_HDR_BAD
    ctx.merge_packed(1, small, n_mut - 1)
    with pytest.raises(pb.PanmanError) as e:
        ctx.merge_status()
    assert e.value.code == ERR_CAPACITY


# ------------------------------------------------------------------------------------------------ full directory entries
def full_entry_input(rng):
    """One leaf, and separately the leaves of one internal clade, differ from the rest in every column of a tile (1 and
    4) and in the neighbouring 1023 + 1 columns: those (node, tile) entries hold 1024 records, their neighbours 1023 and 1."""
    tree = random_tree(64, 71, "binary")
    n_cols = 6 * 1024
    base = rng.integers(0, 4, size=n_cols)
    codes = np.repeat(base[None, :], tree.n_leaves, 0).astype(np.uint8)
    leaf = int(tree.leaves[5])
    codes[tree.leaf_row[leaf], 1:2049] = (base[1:2049] + 1) % 4
    below = {}
    for v in range(tree.n_nodes - 1, -1, -1):  # children have larger ids (pre-order)
        ch = tree.child_idx[tree.child_off[v]:tree.child_off[v + 1]]
        below[v] = [v] if len(ch) == 0 else sum((below[int(c)] for c in ch), [])
    clade = next(v for v in range(1, tree.n_nodes) if 4 <= len(below[v]) <= 8)
    rows = tree.leaf_row[below[clade]]
    codes[np.ix_(rows, np.arange(3073, 5121))] = ((base[3073:5121] + 2) % 4)[None, :]
    return tree, codes, base.astype(np.uint8), leaf, clade


def tile_counts(lists_off, pos, v, n_tiles):
    a, b = lists_off[v], lists_off[v + 1]
    return np.bincount(np.asarray(pos[a:b], np.int64) // 1024, minlength=n_tiles)


def test_full_directory_entries(ctx, port):
    rng = np.random.default_rng(73)
    tree, codes, pc, leaf, clade = full_entry_input(rng)
    _set_tree(ctx, tree)
    c4 = pb.pack_nibbles(codes)
    for algo in (0, 1):
        want, _ = port.run(tree, algo, codes, pc, n_threads=8)
        assert list(tile_counts(want.node_offsets, want.pos, leaf, 6)[:3]) == [1023, 1024, 1]
        assert list(tile_counts(want.node_offsets, want.pos, clade, 6)[3:]) == [1023, 1024, 1]
        res = ctx.run_codes(tree, algo, codes, pc)
        assert np.array_equal(res.node_offsets, want.node_offsets) and np.array_equal(res.pos, want.pos), algo
        assert np.array_equal(res.type_code, want.type_code), algo
        ctx.upload(codes.shape[1], tree.n_leaves, c4, c4.shape[1], pc)
        for _ in range(3):
            ctx.run_resident_async(algo)
        ctx.wait()
        res = ctx.download()
        assert np.array_equal(res.node_offsets, want.node_offsets) and np.array_equal(res.pos, want.pos), (algo, "async")
        assert np.array_equal(res.type_code, want.type_code), (algo, "async")


# ------------------------------------------------------------------------------------------------ column breaks, col_base
@pytest.mark.parametrize("col_base", [5, 2 ** 31 - 6000])
def test_column_breaks_with_col_base(ctx, port, col_base):
    """col_break is indexed by position - col_base; breaks sit at the columns of the records at list index k * 2048 - 1,
    k * 2048 and k * 2048 + 1 (the run-merge's block edges) and at random columns."""
    rng = np.random.default_rng(81)
    tree = random_tree(150, 82, "binary")
    n_cols = 6000
    codes, pc = _noisy(rng, tree.n_leaves, n_cols, 0.8)
    want, _ = port.run(tree, 0, codes, pc, n_threads=8)
    _set_tree(ctx, tree)
    res = ctx.run_codes(tree, 0, codes, pc, col_base=col_base)
    assert np.array_equal(res.node_offsets, want.node_offsets) and np.array_equal(res.type_code, want.type_code)
    assert np.array_equal(res.pos.astype(np.int64), want.pos.astype(np.int64) + col_base)
    n = res.n_mut
    idx = np.array([k * LC.RM_BLOCK + d for k in range(1, n // LC.RM_BLOCK) for d in (-1, 0, 1)])
    brk = np.zeros(n_cols, np.uint8)
    brk[res.pos[idx].astype(np.int64) - col_base] = 1
    brk[rng.choice(n_cols, 300, replace=False)] = 1
    ctx.set_column_breaks(brk)
    want_nm = LC.nucmut_reference(res.node_offsets, res.pos, res.type_code, brk, col_base)
    plain = LC.nucmut_reference(res.node_offsets, res.pos, res.type_code)
    assert len(plain[1]) != len(want_nm[1])  # the breaks matter
    _same_nucmut(ctx.merge_runs(), want_nm, f"breaks, col_base {col_base}")
    ctx.set_column_breaks(None)


# ------------------------------------------------------------------------------------------------ position range
def test_position_range(ctx, port):
    """Positions are int32: col_base = 2^31 - n_cols runs and emits 2^31 - 1; one column more, or col_base < 0, is refused
    by every upload entry (pmb_run_nuc, pmb_upload_nuc, pmb_upload_runs, pmb_run_runs), and the context stays usable."""
    rng = np.random.default_rng(91)
    tree = random_tree(40, 92, "binary")
    n_cols = 3000
    codes, pc = _noisy(rng, tree.n_leaves, n_cols, 0.05)
    codes[0, -6:] = (pc[-6:] + 1) % 4  # a run of six ending in the last column
    want, _ = port.run(tree, 0, codes, pc, n_threads=8)
    _set_tree(ctx, tree)
    hi = 2 ** 31 - n_cols
    res = ctx.run_codes(tree, 0, codes, pc, col_base=hi)
    assert int(res.pos.max()) == 2 ** 31 - 1
    assert np.array_equal(res.pos.astype(np.int64), want.pos.astype(np.int64) + hi)
    assert np.array_equal(res.node_offsets, want.node_offsets) and np.array_equal(res.type_code, want.type_code)
    _same_nucmut(ctx.merge_runs(), LC.nucmut_reference(res.node_offsets, res.pos, res.type_code), "top of the range")
    c4 = pb.pack_nibbles(codes)
    runs = pb.Runs.of_tree(tree, n_cols, c4, pc)
    try:
        for cb in (hi + 1, -1, 2 ** 32):
            calls = {"run_nuc": lambda: ctx.run_codes(tree, 0, codes, pc, col_base=cb),
                     "upload_nuc": lambda: ctx.upload(n_cols, tree.n_leaves, c4, c4.shape[1], pc, col_base=cb),
                     "upload_runs": lambda: ctx.upload_runs(runs, pc, col_base=cb),
                     "upload_runs_async": lambda: ctx.upload_runs(runs, pc, col_base=cb, sync=False),
                     "run_runs": lambda: ctx.run_runs(0, runs, pc, col_base=cb)}
            for name, call in calls.items():
                with pytest.raises(pb.PanmanError) as e:
                    call()
                assert e.value.code == ERR_INVALID and "2^31" in str(e.value), (cb, name)
        res = ctx.run_runs(0, runs, pc, col_base=hi)
        assert np.array_equal(res.pos.astype(np.int64), want.pos.astype(np.int64) + hi)
        res = ctx.run_codes(tree, 0, codes, pc)
        assert np.array_equal(res.pos, want.pos) and np.array_equal(res.node_offsets, want.node_offsets)
    finally:
        runs.close()


def test_group_uploads_refuse_past_int32(port):
    """A group batch of more than 2^31 columns is refused before anything is read (the buffers here are tiny); the group
    then runs a batch that fits."""
    rng = np.random.default_rng(95)
    tree = random_tree(20, 96, "binary")
    codes, pc = _noisy(rng, tree.n_leaves, 1500, 0.1)
    c4 = pb.pack_nibbles(codes)
    g = pb.Group([0])
    try:
        g.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
        big = 2 ** 31 + 1
        runs = pb.Runs.of_tree(tree, 1500, c4, pc)
        calls = {"upload_nuc": lambda: g.upload(big, tree.n_leaves, c4, (big + 1) // 2, pc),
                 "upload_shard": lambda: g.upload_shard(0, big, tree.n_leaves, c4, (big + 1) // 2, pc),
                 "upload_shard_runs": lambda: g.upload_shard_runs(0, big, runs, pc)}
        for name, call in calls.items():
            with pytest.raises(pb.PanmanError) as e:
                call()
            assert e.value.code == ERR_INVALID and "2^31" in str(e.value), name
        runs.close()
        want, _ = port.run(tree, 0, codes, pc, n_threads=4)
        res = g.run_nuc(0, 1500, tree.n_leaves, c4, c4.shape[1], pc)
        assert np.array_equal(res.pos, want.pos) and np.array_equal(res.node_offsets, want.node_offsets)
    finally:
        g.close()
