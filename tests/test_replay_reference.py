"""The replay reference and the replay builders of tests/replay_cases.py, without a GPU: replay_reference against the
per-piece replay of tests/test_msa_reroot.py and the raw-record replay of tests/test_reroot.py, the replay property on the
oracle port's MSA run-merge, and every builder against what it claims to contain."""
import numpy as np
import pytest

from oracle.oracle import random_tree
from tests import replay_cases as RC
from tests.test_msa_reroot import evolve, hand_made_cases, pieces_of, replay_pieces
from tests.test_reroot import _replay


def _small(case):
    return case.tree.n_nodes < 10000 and case.n_cols <= 3000 and case.n_records < 100000


def test_reference_matches_piece_and_record_replays(port):
    """On lists of random Fitch and Sankoff builds (some leaves absent): the reference, the per-piece replay and the
    raw-record replay agree, and every present leaf gets its own row back (the replay property)."""
    rng = np.random.default_rng(88)
    kinds = ["binary", "polytomy", "caterpillar", "unary"]
    for trial in range(16):
        tree = random_tree(int(rng.integers(2, 300)), 8800 + trial, kinds[trial % 4], max_arity=5)
        rows, cons = evolve(tree, int(rng.integers(1, 2100)), rng, p_mut=[0.02, 0.2][trial % 2])
        present = (rng.random(tree.n_leaves) > 0.15).astype(np.uint8)
        present[0] = 1
        algo = trial % 2
        lists, _ = port.run(tree, algo, rows, cons, None, None, present)
        pieces = pieces_of(port, tree, lists)
        got = RC.replay_reference(tree, *pieces, cons)
        assert np.array_equal(got, replay_pieces(tree, *pieces, cons)), trial
        assert np.array_equal(got, _replay(tree, lists.node_offsets, lists.pos, lists.type_code, cons)), trial
        assert np.array_equal(got[present.astype(bool)], rows[present.astype(bool)]), trial


def test_reference_on_hand_made_cases():
    for t, pieces, pc, want in hand_made_cases():
        assert np.array_equal(RC.replay_reference(t, *pieces, pc), want)


@pytest.mark.parametrize("builder", list(RC.BUILDERS))
def test_builder_cases_match_piece_replay(builder):
    """Every case is well formed (what pmb_upload_replay accepts), and where it is small enough for the per-piece replay,
    the reference agrees with it."""
    for case in RC.BUILDERS[builder]():
        off, pos, info, nucs = case.pieces
        t = case.tree
        assert off[0] == 0 and off[-1] == len(pos) == len(info) == len(nucs) and (np.diff(off) >= 0).all(), case.name
        assert len(off) == t.n_nodes + 1
        ln, ty = info >> 4, info & 15
        assert ((ln >= 1) & (ln <= 6)).all() and (ty <= 2).all(), case.name
        assert (pos >= 0).all() and (pos.astype(np.int64) + ln <= case.n_cols).all(), case.name
        assert -1 <= case.tip_row < t.n_leaves
        assert sorted(t.leaf_row[t.leaves]) == list(range(t.n_leaves))
        if _small(case):
            assert np.array_equal(case.reference(), replay_pieces(t, *case.pieces, case.parent_code)), case.name


def test_segment_edges():
    (case,) = RC.segment_edges()
    c = case.claims
    n_seg, seg_rows = c["n_seg"], c["seg_rows"]
    assert (n_seg, seg_rows) == RC.segment_geometry(case.tree, case.n_cols)
    assert case.n_cols <= RC.TILE_COLS and case.tree.n_leaves >= 4000 and n_seg >= 24 and 60 <= seg_rows <= 70
    W = RC.walk(case.tree)
    has = np.diff(case.pieces[0]) > 0
    internal = np.diff(case.tree.child_off) > 0
    for key, on in (("x_on_start", W.x), ("y_on_start", W.y)):
        nodes = c[key]
        assert len(nodes) >= 40 and internal[nodes].sum() >= 30, key
        assert (on[nodes] % seg_rows == 0).all() and (on[nodes] > 0).all() and (on[nodes] < case.tree.n_leaves).all(), key
        assert has[nodes].all(), key
    sp = c["spans_two"]
    assert len(sp) >= 20 and has[sp].all()
    assert (W.y[sp] // seg_rows - (W.x[sp] + seg_rows - 1) // seg_rows >= 2).all()
    rows = case.reference()
    pc = case.parent_code
    assert len(c["restore_triples"]) >= 20
    for a, u, w in c["restore_triples"]:
        assert W.y[u] == W.x[w] and W.y[u] % seg_rows == 0 and W.y[u] - W.x[u] > 1
        assert int(case.tree.parent[u]) == a == int(case.tree.parent[w])
    # the restored column holds the consensus under u and differs from it under w and under a's other leaves
    for i, (a, u, w) in enumerate(c["restore_triples"]):
        col = case.n_cols - 100 + i
        under = lambda v: W.dfs_rows[W.x[v]:W.y[v]]
        assert (rows[under(u), col] == pc[col]).all() and (rows[under(w), col] != pc[col]).all()


def test_tip_positions():
    cases = RC.tip_positions()
    seg_rows, n_seg = cases[0].claims["seg_rows"], cases[0].claims["n_seg"]
    W = RC.walk(cases[0].tree)
    pos = {c.name: c.claims["tip_pos"] for c in cases}
    n = cases[0].tree.n_leaves
    assert pos["tip_first"] == 0 and pos["tip_last"] == n - 1 and pos["tip_none"] == -1
    assert pos["tip_segment_first"] % seg_rows == 0 and pos["tip_segment_last"] % seg_rows == seg_rows - 1
    assert 0 < pos["tip_segment_first"] // seg_rows == pos["tip_segment_last"] // seg_rows < n_seg - 1
    clade = cases[0].claims["clade"]
    assert pos["tip_clade_first"] == W.x[clade] and W.y[clade] - W.x[clade] >= 3
    node, col, _ = RC.records(cases[0].tree.n_nodes, *cases[0].pieces)
    assert set(col[node == clade].tolist()) == set(range(cases[0].n_cols))  # a record in every column
    for c in cases:
        assert c.tip_row == (int(W.dfs_rows[c.claims["tip_pos"]]) if c.claims["tip_pos"] >= 0 else -1), c.name


def test_nesting():
    cat, bal = RC.nesting()
    assert cat.tree.n_leaves >= 19000 and RC.stack_depth(cat.tree, cat.pieces, cat.claims["column"]) >= cat.claims["depth"] >= 19000
    node, col, code = RC.records(cat.tree.n_nodes, *cat.pieces)
    at = col == cat.claims["column"]
    spine = np.nonzero(np.diff(cat.tree.child_off) > 0)[0]
    assert np.array_equal(node[at], spine)  # one record at every spine node, none elsewhere
    of = dict(zip(node[at].tolist(), code[at].tolist()))
    assert all(of[int(v)] != of[int(cat.tree.parent[v])] for v in spine if v != cat.tree.root)  # every level changes the code
    rows = cat.reference()
    leaf_kids = [int(k) for k in cat.tree.child_idx if cat.tree.leaf_row[k] >= 0]
    assert all(rows[cat.tree.leaf_row[k], cat.claims["column"]] == of[int(cat.tree.parent[k])] for k in leaf_kids)
    assert bal.tree.n_leaves == 65536 and RC.stack_depth(bal.tree, bal.pieces, bal.claims["column"]) >= bal.claims["depth"] == 17
    node, col, code = RC.records(bal.tree.n_nodes, *bal.pieces)
    at = col == bal.claims["column"]
    assert np.array_equal(np.unique(node[at]), np.arange(bal.tree.n_nodes))
    # every node writes the column last among its pieces: a leaf's code there is its own record's
    rows = bal.reference()
    last = {int(v): int(k) for v, k in zip(node[at], code[at])}
    leaves = bal.tree.leaves
    assert np.array_equal(rows[bal.tree.leaf_row[leaves], bal.claims["column"]], [last[int(v)] for v in leaves])


def test_key_widths():
    cases = RC.key_widths()
    Rs = {c.claims["R"]: c for c in cases if "R" in c.claims}
    assert set(Rs) == {1, 2, 3} | {2 ** k + d for k in RC.KEY_WIDTH_K for d in (-1, 0, 1)}
    for R, c in Rs.items():
        assert c.n_records == R, c.name
        off = c.pieces[0]
        W = RC.walk(c.tree)
        last = int(W.pre[-1])
        assert off[last + 1] > off[last], c.name  # records are numbered pre-order-major: the highest is the last node's
        if R > 3:
            assert (np.diff(off) > 0).all(), c.name  # no node without pieces
    widths = {c.claims["n_cols"]: c for c in cases if "n_cols" in c.claims}
    assert set(widths) == {2 ** k + d for k in RC.COL_WIDTH_K for d in (-1, 0, 1)}
    for k in RC.COL_WIDTH_K:
        for n_cols in (2 ** k - 1, 2 ** k, 2 ** k + 1):
            c = widths[n_cols]
            assert c.n_cols == n_cols and c.claims["edge_cols"] == (0, 2 ** (k - 1), n_cols - 1)
            _, col, _ = RC.records(c.tree.n_nodes, *c.pieces)
            assert set(c.claims["edge_cols"]) <= set(col.tolist()), c.name


def test_piece_forms():
    (case,) = RC.piece_forms()
    off, pos, info, nucs = case.pieces
    ln, ty = (info >> 4).astype(np.int64), info & 15
    assert {(int(t), int(n)) for t, n in zip(ty, ln)} == {(t, n) for t in (0, 1, 2) for n in range(1, 7)}
    for t in (RC.NS, RC.NI):
        seen = set()
        for j in range(6):
            sel = (ty == t) & (ln > j)
            seen |= set(((nucs[sel].astype(np.int64) >> (4 * (5 - j))) & 15).tolist())
        assert seen == set(range(16)), t
    assert ((ty == RC.ND) & (nucs != 0)).sum() >= 6
    assert ((pos == 1020) & (ln == 6)).any()  # columns 1020 .. 1025 cross the first tile edge
    assert (pos.astype(np.int64) + ln == case.n_cols).sum() >= 3
    node = np.repeat(np.arange(case.tree.n_nodes), np.diff(off))
    o = case.claims["overlap"]
    mine = [(int(p), int(n)) for p, n in zip(pos[node == o], ln[node == o])]
    i = mine.index((5, 4))
    assert mine[i + 1] == (7, 3)
    rows = case.reference()
    for a, d, col in case.claims["same_code"]:
        assert int(case.tree.parent[d]) == a
        assert (rows[:, col] != case.parent_code[col]).any()


def test_empty_and_one_sided():
    none, none_tip, root, leaves = RC.empty_and_one_sided()
    assert none.pieces[0][-1] == 0 == none_tip.pieces[0][-1] and none.tip_row == -1 and none_tip.tip_row >= 0
    assert np.array_equal(none.reference(), np.broadcast_to(none.parent_code, (none.tree.n_leaves, none.n_cols)))
    r = root.tree.root
    assert root.pieces[0][r + 1] - root.pieces[0][r] == root.pieces[0][-1] > 0
    node = np.repeat(np.arange(leaves.tree.n_nodes), np.diff(leaves.pieces[0]))
    assert len(node) > 0 and (leaves.tree.leaf_row[node] >= 0).all()


def test_relabelled():
    base, rev, kids, perm = RC.relabelled()
    want = base.reference()
    Wb = RC.walk(base.tree)
    assert np.array_equal(Wb.pre, np.arange(base.tree.n_nodes))  # the base is in pre-order ...
    Wr = RC.walk(rev.tree)
    assert np.array_equal(Wr.pre, np.arange(rev.tree.n_nodes)[::-1])  # ... the first relabelling in reverse pre-order
    names = lambda c, W: [c.tree.names[v] for v in W.pre if c.tree.leaf_row[v] >= 0]
    Wk = RC.walk(kids.tree)
    assert names(kids, Wk) == names(base, Wb)[::-1]  # the depth-first order of the leaves is reversed
    Wp = RC.walk(perm.tree)
    assert names(perm, Wp) == names(base, Wb) and (Wp.dfs_rows != Wb.dfs_rows).mean() > 0.9
    for c in (rev, kids, perm):
        by_name = {c.tree.names[v]: int(c.tree.leaf_row[v]) for v in c.tree.leaves}
        assert all(by_name[base.tree.names[v]] == c.claims["rows_of"][base.tree.leaf_row[v]] for v in base.tree.leaves), c.name
        got = c.reference()
        assert np.array_equal(got[c.claims["rows_of"]], want), c.name
        assert c.tip_row == int(c.claims["rows_of"][base.tip_row])
