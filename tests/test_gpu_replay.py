"""The device replay of a PanMAT's mutation lists (pmb_upload_replay) at the edges placed by tests/replay_cases.py, and at
full width against the dense upload.

* Cell by cell: the replay onto the tree the pieces were built on, then a Fitch pass with states. A leaf's state is its
  code, so the leaf rows of the states must equal replay_reference in every cell. Then the replay onto the rerooted tree
  with the tip: its lists must equal the oracle port's on the reference rows with the root forced to the tip's row.
* Full width (configs sars20k, ecoli4k and caterpillar100k, the nibble matrix made and kept on the device): the lists of a
  dense pass, run-merged, replayed onto the same tree must give bit-identical lists and NucMut fields (the replay
  property makes the planes identical), and replayed onto the rerooted tree they must give what a dense upload of the
  same matrix with the tip's row as the root override gives.
* One context through replays of every size, an empty piece list, clade-run and dense uploads in between, and
  asynchronous passes on two lanes borrowing the replayed planes."""
import numpy as np
import pytest

import panman_b200 as pb
from oracle.oracle import FlatTree
from tests import replay_cases as RC
from tests.test_msa_reroot import rerooted

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = pb.Context(0)
    yield c
    c.close()


def _set_tree(c, t):
    c.set_tree(t.n_nodes, t.root, t.child_off, t.child_idx, t.leaf_row)


def _same(a, b):
    return (np.array_equal(a.node_offsets, b.node_offsets) and np.array_equal(a.pos, b.pos)
            and np.array_equal(a.type_code, b.type_code))


def _replayed_rows(c, case, root_leaf_row=-1):
    """set_tree(old) -> upload_replay -> a Fitch pass with states -> the leaf rows of the states."""
    t = case.tree
    _set_tree(c, t)
    c.upload_replay(t, *case.pieces, case.n_cols, case.parent_code, root_leaf_row)
    c.run_resident(pb.ALGO_FITCH, pb.FLAG_WANT_STATES)
    st = c.download().states
    out = np.empty((t.n_leaves, case.n_cols), np.uint8)
    out[t.leaf_row[t.leaves]] = st[t.leaves]
    return out


def _check_rows(got, want, what):
    if not np.array_equal(got, want):
        r, col = np.argwhere(got != want)[0]
        n_bad = int((got != want).sum())
        pytest.fail(f"{what}: {n_bad} cells differ, first at row {r} column {col}: {got[r, col]} != {want[r, col]}")


@pytest.mark.parametrize("builder", list(RC.BUILDERS))
def test_cell_by_cell(ctx, port, builder):
    for case in RC.BUILDERS[builder]():
        want = case.reference()
        _check_rows(_replayed_rows(ctx, case), want, case.name)
        if case.tip_row < 0:
            continue
        tip = int(np.nonzero(case.tree.leaf_row == case.tip_row)[0][0])
        new = rerooted(case.tree, case.tree.names[tip])
        _set_tree(ctx, new)
        ctx.upload_replay(case.tree, *case.pieces, case.n_cols, case.parent_code, case.tip_row)
        ctx.run_resident(pb.ALGO_FITCH)
        res = ctx.download()
        w, _ = port.run(new, 0, want, case.parent_code, want[case.tip_row].astype(np.int8), None, None, n_threads=16)
        assert _same(res, w), (case.name, "rerooted lists")


def _nucmut_same(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("name", ["sars20k", "ecoli4k", "caterpillar100k"])
def test_full_width_against_dense_upload(name):
    import torch

    from panman_b200 import synth

    cfg = synth.CONFIGS[name]
    st = synth.make_tree(cfg["n_leaves"], cfg["seed"], cfg["kind"])
    width = cfg["n_cols"]
    codes4, pc = synth.simulate_msa(st, 0, width, synth.MsaSpec(cfg["seed"], cfg["p_sub"], cfg["f_gap"], cfg["p_N"]), device="cuda")
    pc = pc.cpu().numpy()
    old = FlatTree(st.names(), st.parent.astype(np.int32), st.child_off.astype(np.int32), st.child_idx.astype(np.int32), int(st.root),
                   st.leaf_row.astype(np.int32))
    c = pb.Context(0)
    try:
        _set_tree(c, old)
        c.upload(width, old.n_leaves, codes4, codes4.shape[1], pc)
        c.run_resident(pb.ALGO_FITCH)
        first = c.download()
        nm = c.merge_runs()
        assert first.n_mut > 0
        # (a) the same tree, no tip: a fixed point
        c.upload_replay(old, *nm[:4], width, pc, -1)
        c.run_resident(pb.ALGO_FITCH)
        assert _same(c.download(), first), (name, "replay onto the same tree: lists")
        assert _nucmut_same(c.merge_runs(), nm), (name, "replay onto the same tree: NucMut fields")
        # (b) the rerooted tree with the tip: the dense upload of the same matrix with the tip's row forced at the root
        tip = int(old.leaves[len(old.leaves) // 3])
        row = int(old.leaf_row[tip])
        new = rerooted(old, old.names[tip])
        _set_tree(c, new)
        c.upload_replay(old, *nm[:4], width, pc, row)
        c.run_resident(pb.ALGO_FITCH)
        rep, rep_nm = c.download(), c.merge_runs()
        override = synth.unpack_nibbles(codes4[row:row + 1], width)[0].to(torch.int8).contiguous()
        c.upload(width, old.n_leaves, codes4, codes4.shape[1], pc, override)
        c.run_resident(pb.ALGO_FITCH)
        dense = c.download()
        assert dense.n_mut > 0 and _same(rep, dense), (name, "rerooted: replay vs dense lists")
        assert _nucmut_same(rep_nm, c.merge_runs()), (name, "rerooted: replay vs dense NucMut fields")
    finally:
        c.close()
        del codes4
        torch.cuda.empty_cache()


def test_context_reuse(port):
    """One context: a large replay, a small one, no pieces, the large one again (buffers kept at their grown size with stale
    content); replay -> clade-run upload -> replay -> dense upload -> replay; asynchronous passes on two lanes on a replayed
    input. Every step against the reference."""
    large = RC.key_widths()[5]   # 2^20 + 1 records
    small = RC.piece_forms()[0]
    empty = RC.empty_and_one_sided()[0]
    assert large.n_records == 2 ** 20 + 1 and empty.n_records == 0
    c = pb.Context(0)
    for i, case in enumerate([large, small, empty, large, small]):
        _check_rows(_replayed_rows(c, case), case.reference(), f"sequence step {i}: {case.name}")

    case = RC.segment_edges()[0]
    t, want = case.tree, case.reference()
    rng = np.random.default_rng(89)
    other = want.copy()
    other[rng.random(other.shape) < 0.01] = 15
    runs = pb.Runs.of_tree(t, case.n_cols, pb.pack_nibbles(other), case.parent_code)
    _check_rows(_replayed_rows(c, case), want, "replay before a clade-run upload")
    c.upload_runs(runs, case.parent_code)
    c.run_resident(pb.ALGO_FITCH, pb.FLAG_WANT_STATES)
    st = c.download().states
    _check_rows(st[t.leaves][np.argsort(t.leaf_row[t.leaves])], other, "clade-run upload after a replay")
    _check_rows(_replayed_rows(c, case), want, "replay after a clade-run upload")
    runs.close()
    other4 = pb.pack_nibbles(other[:, ::-1])
    c.upload(case.n_cols, t.n_leaves, other4, other4.shape[1], case.parent_code[::-1].copy())
    c.run_resident(pb.ALGO_FITCH, pb.FLAG_WANT_STATES)
    st = c.download().states
    _check_rows(st[t.leaves][np.argsort(t.leaf_row[t.leaves])], other[:, ::-1], "dense upload after a replay")
    _check_rows(_replayed_rows(c, case), want, "replay after a dense upload")
    c.close()

    # asynchronous passes on two lanes read the replayed planes; then a replay of other pieces while they may still run
    c = pb.Context(0)
    c.set_option("overlap", 1)
    c.set_option("lanes", 1)
    case = RC.relabelled()[0]
    t, want = case.tree, case.reference()
    w, _ = port.run(t, 0, want, case.parent_code, n_threads=8)
    _set_tree(c, t)
    c.upload_replay(t, *case.pieces, case.n_cols, case.parent_code, -1)
    for _ in range(4):
        c.run_resident_async(pb.ALGO_FITCH)
    c.wait()
    assert _same(c.download(), w), "asynchronous passes on a replayed input"
    for _ in range(3):
        c.run_resident_async(pb.ALGO_FITCH)
    none = (np.zeros(t.n_nodes + 1, np.int64), np.zeros(0, np.int32), np.zeros(0, np.uint8), np.zeros(0, np.uint32))
    c.upload_replay(t, *none, case.n_cols, case.parent_code, -1)
    c.run_resident(pb.ALGO_FITCH, pb.FLAG_WANT_STATES)
    st = c.download().states
    _check_rows(st[t.leaves], np.broadcast_to(case.parent_code, (t.n_leaves, case.n_cols)), "replay behind asynchronous passes")
    c.upload_replay(t, *case.pieces, case.n_cols, case.parent_code, -1)
    c.run_resident_async(pb.ALGO_FITCH)
    c.wait()
    assert _same(c.download(), w), "asynchronous pass after the empty replay"
    c.close()
