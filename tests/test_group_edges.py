"""The column-sharded group (pmb_group_*) at its edges, on the device. Every result is checked bit for bit on the whole
alignment against the oracle port (lists) and list_cases.nucmut_reference (NucMut fields), and against a single-context
pmb_run_nuc of the same batch.

The inputs come from tests/group_cases.py: features on every rank boundary, widths around the group's tile counts, rows
wider than the packed row, leaf_present, Fitch and Sankoff root overrides, fwd_root_ref and block mode, through every
entry (upload + several asynchronous steps, run_nuc, per-rank shards, the clade-run encoding whole and per rank).
Width schedules change the active ranks step after step on one group; a rank that sat out two or more steps waits for a
credit only the merge of the steps it sat out can give, so those runs go to a spawned child that is killed on a timeout:
a regression fails in bounded time and leaves no process behind. Also: a tree change mid-group (same node count, then
another), the mailbox at exactly the largest shard and one record short, the refusal of a stride too small for the whole
row and of a shard encoding of the wrong width, the -M flow over three builds of different widths on one group, and one
process per rank running a schedule that leaves rank 2 out for two steps."""
import multiprocessing as mp
import queue
import socket

import numpy as np
import pytest

import panman_b200 as pb
from oracle.oracle import random_tree
from tests import group_cases as GC
from tests.list_cases import nucmut_reference

pytestmark = pytest.mark.gpu

N_LEAVES = GC.FEATURE_ROWS + 40
ENTRIES = ("async", "run_nuc", "shard", "runs", "shard_runs")
# (algo, block mode, leaf_present, root_override, fwd_root_ref): fwd_root_ref only with Fitch in nucleotide mode
VARIANTS = ((0, 0, True, False, True), (0, 0, False, True, False), (1, 0, True, True, False), (0, 1, False, True, False),
            (1, 1, True, False, False), (0, 0, True, True, True))
SCHEDULE_TIMEOUT = 240


def _n_devices():
    import torch

    return torch.cuda.device_count()


def _same(res, want):
    return (np.array_equal(res.node_offsets, want.node_offsets) and np.array_equal(res.pos, want.pos)
            and np.array_equal(res.type_code, want.type_code))


def _same_nucmut(got, want):
    return all(np.array_equal(x, y) for x, y in zip(got, nucmut_reference(want.node_offsets, want.pos, want.type_code)))


def _oracle(port, tree, c):
    want, _ = port.run(tree, c.algo, c.codes, c.parent_code, c.root_override, c.fwd_root_ref, c.leaf_present, c.block, n_threads=4)
    return want


def _runs(tree, codes, pad, parent_code, seed):
    buf, stride = GC.pack_padded(codes, pad, seed)
    return pb.Runs(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row, codes.shape[1], buf, stride, parent_code)


def _run_entry(g, entry, tree, c, pad, steps=3):
    """One batch through one entry of the group; the merged lists of its last step."""
    n_rows, n_cols = c.codes.shape
    world = g.world
    buf, stride = GC.pack_padded(c.codes, pad, seed=n_cols)
    if entry == "run_nuc":
        return g.run_nuc(c.algo, n_cols, n_rows, buf, stride, c.parent_code, c.root_override, c.fwd_root_ref, c.leaf_present, c.flags)
    keep = []
    if entry == "async":
        g.upload(n_cols, n_rows, buf, stride, c.parent_code, c.root_override, c.fwd_root_ref, c.leaf_present)
    elif entry == "runs":
        keep.append(_runs(tree, c.codes, pad, c.parent_code, n_cols))
        g.upload_runs(keep[-1], c.parent_code, c.root_override, c.fwd_root_ref, c.leaf_present)
    else:
        for i in range(g.n_local):
            a, b = GC.range_reference(world, n_cols, i)
            if b == a:
                continue  # a rank past the tile count owns nothing and is given nothing
            pc, ro, fr = c.sliced(a, b)
            if entry == "shard":
                sbuf, sstride = GC.pack_padded(c.codes[:, a:b], pad, seed=i)
                g.upload_shard(i, n_cols, n_rows, sbuf, sstride, pc, ro, fr, c.leaf_present)
            else:
                keep.append(_runs(tree, c.codes[:, a:b], pad, pc, i))
                g.upload_shard_runs(i, n_cols, keep[-1], pc, ro, fr, c.leaf_present)
    for _ in range(steps):  # steps in flight on both mailbox parities
        g.run_async(c.algo, c.flags)
    g.wait()
    res = g.download()
    for r in keep:
        r.close()
    return res


def _boundaries(port, devices, seed):
    world = len(devices)
    tree = random_tree(N_LEAVES, seed, "binary")
    cases = []
    for k, n_cols in enumerate(GC.boundary_widths(world)):
        for v, (algo, block, lp, ro, fr) in enumerate(VARIANTS):
            c = GC.boundary_case(N_LEAVES, world, n_cols, algo, block, seed=seed * 1000 + 10 * k + v, presence=lp, override=ro, fwd=fr)
            cases.append((n_cols, v, c, _oracle(port, tree, c)))
    ctx = pb.Context(devices[0])
    ctx.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
    g = pb.Group(devices)
    g.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
    for n_cols, v, c, want in cases:
        if v == 0:
            # a new mailbox for every width, large enough for every shard of it: the set of active ranks never changes during
            # one mailbox's life, so this test runs in the pytest process without meeting a wait that only the credit of
            # inactive ranks can satisfy (the width schedules below do that, in a child process)
            g.reserve(max(int(w.node_offsets[-1]) for m, _, _, w in cases if m == n_cols) + 16)
        pad = 5 * ((n_cols + v) % 3)
        buf, stride = GC.pack_padded(c.codes, pad, seed=v)
        single = ctx.run_nuc(c.algo, n_cols, N_LEAVES, buf, stride, c.parent_code, c.root_override, c.fwd_root_ref, c.leaf_present, 0,
                             c.flags)
        assert _same(single, want), (world, n_cols, v, "single context vs oracle")
        for entry in ENTRIES:
            res = _run_entry(g, entry, tree, c, pad)
            assert _same(res, want), (world, n_cols, v, entry)
            assert _same_nucmut(g.merge_runs(), want), (world, n_cols, v, entry, "NucMut fields")
    g.close()
    ctx.close()


@pytest.mark.parametrize("world", range(1, 9))
def test_boundaries_on_one_device(port, world):
    _boundaries(port, [0] * world, seed=world)


def test_boundaries_over_all_devices(port):
    n = _n_devices()
    if n < 2:
        pytest.skip("one GPU visible: the multi-device mapping (peer access over NVLink) needs two")
    _boundaries(port, list(range(n)), seed=100 + n)


# ------------------------------------------------------------------------------------------------------- in a child
def _child(target, args, q):
    try:
        q.put(("ok", target(*args)))
    except BaseException as e:  # the parent reports it
        q.put(("error", repr(e)))


def _in_child(target, args, timeout):
    """target(*args) in a spawned process. Returns its value; fails the test on an error or when nothing came back in
    `timeout` seconds. The child is joined, or killed and joined, on every path."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    p = ctx.Process(target=_child, args=(target, args, q))
    p.start()
    got = None
    try:
        got = q.get(timeout=timeout)
    except queue.Empty:
        pass
    finally:
        p.join(timeout=60 if got else 0)
        if p.is_alive():
            p.kill()
            p.join()
    if got is None:
        pytest.fail(f"{target.__name__}{args}: no answer within {timeout} s (a wait of the hand-shake was never met)")
    kind, value = got
    assert kind == "ok", value
    return value


def _schedule_run(devices, seed):
    """The width schedule of group_cases on one group and one tree, right after a reserve; the lists and NucMut fields
    checked after every wait. Returns the failed steps."""
    from oracle.oracle import PortOracle

    port = PortOracle()
    world = len(devices)
    tree = random_tree(N_LEAVES, seed, "binary")
    steps = GC.schedule(world, seed)
    cases = [GC.boundary_case(N_LEAVES, world, s.n_cols, s.algo, s.block, seed=seed * 1000 + i, presence=i % 3 == 0,
                              override=i % 2 == 1, fwd=s.algo == 0 and not s.block and i % 8 == 0) for i, s in enumerate(steps)]
    wants = [_oracle(port, tree, c) for c in cases]
    g = pb.Group(devices)
    g.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
    g.reserve(max(int(w.node_offsets[-1]) for w in wants) + 16)
    bad = []
    for i, (s, c, want) in enumerate(zip(steps, cases, wants)):
        buf, stride = GC.pack_padded(c.codes, 3 * (i % 2), seed=i)
        g.upload(s.n_cols, N_LEAVES, buf, stride, c.parent_code, c.root_override, c.fwd_root_ref, c.leaf_present)
        g.run_async(c.algo, c.flags)
        g.wait()
        if not _same(g.download(), want):
            bad.append((i + 1, s.active, s.n_cols, "lists"))
        elif not _same_nucmut(g.merge_runs(), want):
            bad.append((i + 1, s.active, s.n_cols, "NucMut fields"))
    g.close()
    return bad


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_width_schedule_on_one_device(world):
    assert _in_child(_schedule_run, ([0] * world, 70 + world), SCHEDULE_TIMEOUT) == []


def test_width_schedule_over_all_devices():
    n = _n_devices()
    if n < 2:
        pytest.skip("one GPU visible")
    assert _in_child(_schedule_run, (list(range(n)), 90 + n), SCHEDULE_TIMEOUT) == []


def _msa_builds():
    """Three -M builds on one tree at 700, 900 and 3500 columns (one, one and three active ranks of Group([0, 0, 0])): the
    third step is the first one of ranks 1 and 2 since the group sized its mailbox. Returns the builds that differ from
    the context engine's."""
    from panman_b200.host import MsaBuild
    from tests.test_host import _fasta

    rng = np.random.default_rng(17)
    tree = random_tree(60, 17, "binary")
    names = [tree.names[v] for v in tree.leaves]
    alphabet = np.frombuffer(b"ACGTN-ACGTACGTRYKM", np.uint8)
    ctx, grp = pb.Context(0), pb.Group([0, 0, 0])
    bad = []
    for width, reference, low_mem in ((700, names[3], False), (900, names[11], True), (3500, names[29], False)):
        base = rng.choice(alphabet[:4], size=width)
        rows = np.repeat(base[None, :], len(names), 0)
        rows = np.where(rng.random(rows.shape) < 0.08, rng.choice(alphabet, size=rows.shape), rows).astype(np.uint8)
        rows[0] = base  # no all-gap column: every build keeps its width
        fasta = _fasta(names, rows)
        want = MsaBuild(ctx, fasta, tree.to_newick(), reference, low_mem)
        got = MsaBuild(grp, fasta, tree.to_newick(), reference, low_mem)
        same = (np.array_equal(got.tuple_offsets, want.tuple_offsets) and np.array_equal(got.tuple_pos, want.tuple_pos)
                and np.array_equal(got.tuple_type_code, want.tuple_type_code) and got.nucmut == want.nucmut and got.wire == want.wire)
        if not same or len(want.consensus) != width:
            bad.append(width)
        want.close()
        got.close()
    grp.close()
    ctx.close()
    return bad


def test_msa_builds_of_three_widths_on_one_group():
    assert _in_child(_msa_builds, (), SCHEDULE_TIMEOUT) == []


# ------------------------------------------------------------------------------------------------------- one process
def test_tree_changes_mid_group(port):
    """Another topology with the same node count keeps the mailbox (no reserve in between); another node count releases it
    and run_nuc sizes a new one. Every step keeps all three ranks active."""
    A = random_tree(N_LEAVES, 501, "binary")
    B = random_tree(N_LEAVES, 502, "caterpillar")
    Cx = random_tree(N_LEAVES + 37, 503, "polytomy", max_arity=4)
    assert A.n_nodes == B.n_nodes != Cx.n_nodes
    g = pb.Group([0, 0, 0])

    def check(tree, n_cols, entry, k):
        c = GC.boundary_case(tree.n_leaves, 3, n_cols, k % 2, 0, seed=600 + k, presence=k % 2 == 0, override=True, fwd=k % 2 == 0)
        want = _oracle(port, tree, c)
        assert _same(_run_entry(g, entry, tree, c, pad=k % 4), want), (k, n_cols, entry)
        assert _same_nucmut(g.merge_runs(), want), (k, "NucMut fields")

    g.set_tree(A.n_nodes, A.root, A.child_off, A.child_idx, A.leaf_row)
    check(A, 3 * 1024 + 5, "run_nuc", 0)  # sizes the mailbox
    check(A, 2500, "async", 1)
    g.set_tree(B.n_nodes, B.root, B.child_off, B.child_idx, B.leaf_row)
    check(B, 3100, "async", 2)  # no reserve: the mailbox of A's node count is still connected
    check(B, 2200, "shard", 3)
    check(B, 4000, "runs", 4)
    g.set_tree(Cx.n_nodes, Cx.root, Cx.child_off, Cx.child_idx, Cx.leaf_row)
    with pytest.raises(pb.PanmanError) as e:  # the mailbox was released with the old node count
        g.upload(2100, Cx.n_leaves, *GC.pack_padded(np.zeros((Cx.n_leaves, 2100), np.uint8), 0), np.zeros(2100, np.uint8))
        g.run_async(0)
    assert e.value.code == -5
    check(Cx, 3000, "run_nuc", 5)  # and run_nuc sizes a new one
    check(Cx, 2900, "async", 6)
    g.close()


def test_mailbox_capacity_exact_and_one_short(port):
    """Rank 1's shard is the largest: a mailbox of exactly its record count works, one record less fails the wait with
    PMB_ERR_CAPACITY, and a reserve brings the group back."""
    rng = np.random.default_rng(8)
    tree = random_tree(N_LEAVES, 8, "binary")
    n_cols = 3000
    c = GC.boundary_case(N_LEAVES, 3, n_cols, 0, 0, seed=8)
    noisy = rng.random((N_LEAVES, 1024)) < 0.3
    c.codes[:, 1024:2048] = np.where(noisy, rng.integers(0, 16, size=noisy.shape), c.codes[:, 1024:2048]).astype(np.uint8)
    want = _oracle(port, tree, c)
    shard_n = [int(((want.pos >= a) & (want.pos < b)).sum()) for a, b in (GC.range_reference(3, n_cols, r) for r in range(3))]
    assert int(np.argmax(shard_n)) == 1 and sorted(shard_n)[-2] < shard_n[1], shard_n
    cap = shard_n[1]
    g = pb.Group([0, 0, 0])
    g.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
    buf, stride = GC.pack_padded(c.codes, 0)
    g.reserve(cap)
    g.upload(n_cols, N_LEAVES, buf, stride, c.parent_code)
    for _ in range(3):
        g.run_async(0)
    g.wait()
    assert _same(g.download(), want) and _same_nucmut(g.merge_runs(), want)
    g.reserve(cap - 1)
    g.run_async(0)
    with pytest.raises(pb.PanmanError) as e:
        g.wait()
    assert e.value.code == -9
    g.reserve(cap)
    g.run_async(0)
    g.run_async(0)
    g.wait()
    assert _same(g.download(), want) and _same_nucmut(g.merge_runs(), want)
    g.close()


def test_stride_of_the_whole_row_and_shard_widths(port):
    """pmb_group_upload_nuc refuses a stride too small for the whole row even where every rank's range would fit in it
    (5000 columns on 5 ranks need 2500 bytes a row; each range needs at most 512). The host buffer holds exactly
    n_rows * 2500 bytes. An encoded shard of another width than the rank's range is refused too."""
    rng = np.random.default_rng(9)
    tree = random_tree(80, 9, "binary")
    n_cols, world = 5000, 5
    codes = np.where(rng.random((80, n_cols)) < 0.05, rng.integers(0, 16, size=(80, n_cols)), 2).astype(np.uint8)
    pc = np.full(n_cols, 2, np.uint8)
    c4 = pb.pack_nibbles(codes)
    assert c4.nbytes == 80 * 2500
    want, _ = port.run(tree, 0, codes, pc, n_threads=4)
    g = pb.Group([0] * world)
    g.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
    for stride in (600, 2499):
        with pytest.raises(pb.PanmanError) as e:
            g.upload(n_cols, 80, c4, stride, pc)
        assert e.value.code == -1 and "stride" in str(e.value)
        with pytest.raises(pb.PanmanError) as e:
            g.run_nuc(0, n_cols, 80, c4, stride, pc)
        assert e.value.code == -1
    assert _same(g.run_nuc(0, n_cols, 80, c4, 2500, pc), want)
    a, b = g.column_range(n_cols, 1)
    for wrong in (b - a - 1, b - a + 1, 2 * (b - a)):
        r = pb.Runs.of_tree(tree, wrong, pb.pack_nibbles(codes[:, a:a + wrong]), pc[a:a + wrong])
        with pytest.raises(pb.PanmanError) as e:
            g.upload_shard_runs(1, n_cols, r, pc[a:a + wrong])
        assert e.value.code == -1
        r.close()
    shards = []
    for i in range(world):
        a, b = g.column_range(n_cols, i)
        shards.append(pb.Runs.of_tree(tree, b - a, pb.pack_nibbles(codes[:, a:b]), pc[a:b]))
        g.upload_shard_runs(i, n_cols, shards[-1], pc[a:b])
    g.run_async(0)
    g.wait()
    assert _same(g.download(), want)
    for r in shards:
        r.close()
    g.close()


# ------------------------------------------------------------------------------------------------- one process per rank
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


RANK_WIDTHS = (3000, 1800, 1900, 3000, 2900, 1500, 3070)  # rank 2 owns nothing at steps 2 and 3 (and 6)


def _rank_schedule_main(rank, world, port_no, q):
    """One process per rank through torch.distributed (gloo) and CUDA IPC; every rank uploads its own range each step,
    an empty one when it owns none."""
    import os

    import torch
    import torch.distributed as dist

    from oracle.oracle import PortOracle
    from panman_b200.distributed import connect_group

    try:
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port_no)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        dev = rank % torch.cuda.device_count()
        torch.cuda.set_device(dev)
        port = PortOracle()
        tree = random_tree(N_LEAVES, 61, "binary")
        cases = [GC.boundary_case(N_LEAVES, world, w, i % 2, 0, seed=6100 + i, presence=i % 3 == 0, override=True, fwd=i % 2 == 0)
                 for i, w in enumerate(RANK_WIDTHS)]
        wants = [_oracle(port, tree, c) for c in cases]
        g = pb.Group([dev], rank_base=rank, world=world)
        g.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
        connect_group(g, dist, max(int(w.node_offsets[-1]) for w in wants) + 16)
        bad = []
        for i, (w, c, want) in enumerate(zip(RANK_WIDTHS, cases, wants)):
            a, b = pb.column_range(world, w, rank)
            if b > a:
                sbuf, sstride = GC.pack_padded(c.codes[:, a:b], 2, seed=i)
                pc, ro, fr = c.sliced(a, b)
                g.upload_shard(0, w, N_LEAVES, sbuf, sstride, pc, ro, fr, c.leaf_present)
            else:
                g.upload_shard(0, w, N_LEAVES, np.zeros((N_LEAVES, 1), np.uint8), 1, np.zeros(1, np.uint8))
            g.run_async(c.algo, c.flags)
            g.wait()
            res = g.download()
            if rank == 0:
                if not (_same(res, want) and _same_nucmut(g.merge_runs(), want)):
                    bad.append(i + 1)
            elif res.n_mut != 0:
                bad.append(i + 1)
        dist.barrier()
        g.close()
        dist.destroy_process_group()
        q.put((rank, bad))
    except BaseException as e:
        q.put((rank, repr(e)))


def test_one_process_per_rank_with_a_rank_out_for_two_steps():
    assert [GC.active_ranks(3, w) for w in RANK_WIDTHS] == [3, 2, 2, 3, 3, 2, 3]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port_no = _free_port()
    procs = [ctx.Process(target=_rank_schedule_main, args=(r, 3, port_no, q)) for r in range(3)]
    got = {}
    try:
        for p in procs:
            p.start()
        for _ in range(3):
            rank, value = q.get(timeout=300)
            got[rank] = value
    except queue.Empty:
        pass
    finally:
        for p in procs:
            p.join(timeout=60 if len(got) == 3 else 0)
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
    assert got == {0: [], 1: [], 2: []}, got
