"""Tree::reroot of an MSA-built PanMAT (reference src/reroot.cpp:4-261): the mutation lists replayed into the leaf
sequences (getSequenceFromReference, src/reroot.cpp:19-35) on the device by pmb_upload_replay, then the forced-root Fitch
pass on the new tree (pmh_msa_reroot).

* CPU: a numpy replay of NucMut pieces against the raw-record replay of tests/test_reroot.py, and the replay property (every
  present leaf gets its own input back) on lists made by the port and its MSA run-merge;
* GPU: the device replay cell by cell (a present leaf's Fitch state is its code), pmh_msa_reroot end to end against the
  port driven as src/reroot.cpp drives the passes, the full-size configs through the C ABI, refusals and context state."""
import numpy as np
import pytest

from oracle.oracle import CODE_OF, FlatTree, block_mut_from_nuc, random_tree
from tests.test_reroot import _by_name, _flat, _py_transform, _replay

KINDS = ["binary", "polytomy", "caterpillar", "unary"]


def _preorder(tree):
    out, stack = [], [int(tree.root)]
    while stack:
        v = stack.pop()
        out.append(v)
        stack.extend(int(c) for c in tree.child_idx[tree.child_off[v]:tree.child_off[v + 1]][::-1])
    return out


def replay_pieces(tree, piece_off, pos, info, nucs, parent_code):
    """getSequenceFromReference on NucMut pieces: consensus, then root -> leaf every piece in stored order; NS / NI write
    their nucs nibble, ND writes '-' (0). Returns (n_leaves, n_cols) codes by leaf row."""
    pc = np.asarray(parent_code, np.uint8)
    rows = np.zeros((tree.n_leaves, len(pc)), np.uint8)
    cur = {}
    for v in _preorder(tree):
        base = pc.copy() if v == tree.root else cur[int(tree.parent[v])].copy()
        for k in range(piece_off[v], piece_off[v + 1]):
            n, t = int(info[k]) >> 4, int(info[k]) & 15
            for j in range(n):
                base[pos[k] + j] = 0 if t == 1 else (int(nucs[k]) >> (4 * (5 - j))) & 15
        cur[v] = base
        if tree.leaf_row[v] >= 0:
            rows[tree.leaf_row[v]] = base
    return rows


def pieces_of(port, tree, lists):
    """MSA run-merge of every node's raw lists (port.merge_msa) -> node-major piece arrays."""
    off, pos, info, nucs = [0], [], [], []
    for v in range(tree.n_nodes):
        p, tc = lists.of(v)
        wp, wmi, wnu = port.merge_msa(p, tc) if len(p) else ([], [], [])
        pos += list(wp)
        info += list(wmi)
        nucs += list(wnu)
        off.append(len(pos))
    return (np.asarray(off, np.int64), np.asarray(pos, np.int32), np.asarray(info, np.uint8), np.asarray(nucs, np.uint32))


def evolve(tree, n_cols, rng, p_mut=0.02):
    """Leaf codes evolved down the tree (clade-wide changes, gaps, N), the consensus = the root's sequence."""
    alphabet = np.asarray([1, 2, 4, 8, 0, 15, 5, 10], np.uint8)
    seq = {}
    root = rng.choice(alphabet[:4], size=n_cols).astype(np.uint8)
    for v in _preorder(tree):
        s = root.copy() if v == tree.root else seq[int(tree.parent[v])].copy()
        m = rng.random(n_cols) < p_mut
        s[m] = rng.choice(alphabet, size=int(m.sum()))
        seq[v] = s
    rows = np.zeros((tree.n_leaves, n_cols), np.uint8)
    for v in tree.leaves:
        rows[tree.leaf_row[v]] = seq[int(v)]
    return rows, root


def rerooted(old, tip_name):
    """pmh_tree_reroot of `old` with leaf rows carried by name (the rows of `old`)."""
    from panman_b200.host import reroot_newick

    t = reroot_newick(old.to_newick(), tip_name)
    row_of = {old.names[v]: int(old.leaf_row[v]) for v in old.leaves}
    lr = np.asarray([row_of[n] if t.leaf_row[v] >= 0 else -1 for v, n in enumerate(t.names)], np.int32)
    return FlatTree(list(t.names), t.parent.astype(np.int32), t.child_off.astype(np.int32), t.child_idx.astype(np.int32), int(t.root), lr)


def _case(rng, trial, n_leaves=None, width=None, kind=None, max_arity=5):
    kind = kind or KINDS[trial % 4]
    tree = random_tree(n_leaves or int(rng.integers(2, 120)), 6100 + trial, kind, max_arity=max_arity)
    rows, cons = evolve(tree, width or int(rng.integers(1, 1500)), rng)
    present = (rng.random(tree.n_leaves) > 0.15).astype(np.uint8)
    present[0] = 1
    return tree, rows, cons, present


# ------------------------------------------------------------------------------------------------------------------ CPU


def test_piece_replay_matches_record_replay(port):
    rng = np.random.default_rng(61)
    for trial in range(24):
        tree, rows, cons, present = _case(rng, trial)
        algo = trial % 2  # lists of a Fitch and of a --low-mem-mode (Sankoff) build
        fr = rows[0].astype(np.int8) if trial % 3 == 0 else None
        lists, _ = port.run(tree, algo, rows, cons, None if algo == 0 else fr, fr if algo == 0 else None, present)
        po, pos, info, nucs = pieces_of(port, tree, lists)
        got = replay_pieces(tree, po, pos, info, nucs, cons)
        assert np.array_equal(got, _replay(tree, lists.node_offsets, lists.pos, lists.type_code, cons)), trial
        assert np.array_equal(got[present.astype(bool)], rows[present.astype(bool)]), trial  # the replay property, SURVEY A.7


def hand_made_cases():
    """(tree, pieces, parent_code, expected rows): duplicate columns within a node, a unary chain, ND with non-zero nucs."""
    cases = []
    # ((a,b)n2,c)n1: node n2 (id 1) has two pieces over column 2; the later one wins
    t = FlatTree.from_children(["node_1", "node_2", "a", "b", "c"], [[1, 4], [2, 3], [], [], []])
    pc = np.asarray([1, 1, 1, 1], np.uint8)
    po = np.asarray([0, 0, 2, 2, 2, 2], np.int64)
    pos = np.asarray([1, 2], np.int32)
    info = np.asarray([(2 << 4) | 0, (1 << 4) | 2], np.uint8)
    nucs = np.asarray([(2 << 20) | (4 << 16), 8 << 20], np.uint32)
    cases.append((t, (po, pos, info, nucs), pc, np.asarray([[1, 2, 8, 1], [1, 2, 8, 1], [1, 1, 1, 1]], np.uint8)))
    # unary chain n1 -> n2 -> n3 -> (a, b); n2 and n3 both write column 0, n3 (deeper) wins; b overrides again
    t = FlatTree.from_children(["node_1", "node_2", "node_3", "a", "b"], [[1], [2], [3, 4], [], []])
    po = np.asarray([0, 0, 1, 2, 2, 3], np.int64)
    pos = np.asarray([0, 0, 0], np.int32)
    info = np.asarray([(1 << 4) | 0, (1 << 4) | 0, (1 << 4) | 1], np.uint8)
    nucs = np.asarray([2 << 20, 4 << 20, 0], np.uint32)
    cases.append((t, (po, pos, info, nucs), np.asarray([1, 1], np.uint8), np.asarray([[4, 1], [0, 1]], np.uint8)))
    # ND pieces whose nucs are not 0 still write '-'
    t = FlatTree.from_children(["node_1", "a", "b"], [[1, 2], [], []])
    po = np.asarray([0, 0, 1, 1], np.int64)
    pos = np.asarray([1], np.int32)
    info = np.asarray([(3 << 4) | 1], np.uint8)
    nucs = np.asarray([0xFFFFFF], np.uint32)
    cases.append((t, (po, pos, info, nucs), np.asarray([1, 2, 4, 8], np.uint8), np.asarray([[1, 0, 0, 0], [1, 2, 4, 8]], np.uint8)))
    return cases


def test_hand_made_replays():
    for t, (po, pos, info, nucs), pc, want in hand_made_cases():
        assert np.array_equal(replay_pieces(t, po, pos, info, nucs, pc), want)


# ------------------------------------------------------------------------------------------------------------------ GPU


def _replay_on_device(ctx, tree, pieces, pc, want_states=True):
    import panman_b200 as pb

    ctx.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
    ctx.upload_replay(tree, *pieces, len(pc), pc, -1)
    ctx.run_resident(pb.ALGO_FITCH, pb.FLAG_WANT_STATES if want_states else 0)
    return ctx.download()


def _leaf_states(tree, states):
    out = np.zeros((tree.n_leaves, states.shape[1]), np.uint8)
    out[tree.leaf_row[tree.leaves]] = states[tree.leaves]
    return out


@pytest.mark.gpu
def test_device_replay_cell_by_cell(port):
    """pmb_upload_replay with the old tree set and no root override, then a pass with states: a present leaf's Fitch state is
    its code, so the leaf rows of the states are the replayed sequences, checked in every cell; the lists of the pass are
    checked against the port on the numpy replay."""
    import panman_b200 as pb

    ctx = pb.Context(0)
    rng = np.random.default_rng(62)
    widths = [1, 1023, 1024, 1025, 3 * 1024 + 7]
    shapes = [("binary", 2, 2), ("binary", 2000, 2), ("polytomy", 900, 300), ("caterpillar", 700, 2), ("unary", 1500, 4),
              ("polytomy", 60, 5), ("caterpillar", 2000, 2)]
    for trial in range(12):
        kind, n, ar = shapes[trial % len(shapes)]
        tree, rows, cons, present = _case(rng, trial, n, widths[trial % len(widths)], kind, ar)
        lists, _ = port.run(tree, 0, rows, cons, None, None, present if trial % 2 else None)
        pieces = pieces_of(port, tree, lists)
        want = replay_pieces(tree, *pieces, cons)
        if trial == 0:  # on the port first: with every leaf present, a leaf's state is its code
            _, st = port.run(tree, 0, want, cons, want_states=True)
            assert np.array_equal(_leaf_states(tree, st), want)
        res = _replay_on_device(ctx, tree, pieces, cons)
        assert np.array_equal(_leaf_states(tree, res.states), want), (trial, kind, n)
        w, _ = port.run(tree, 0, want, cons, n_threads=4)
        assert np.array_equal(res.node_offsets, w.node_offsets) and np.array_equal(res.pos, w.pos) and np.array_equal(res.type_code, w.type_code)
    for t, pieces, pc, want in hand_made_cases():
        res = _replay_on_device(ctx, t, pieces, pc)
        assert np.array_equal(_leaf_states(t, res.states), want)
    ctx.close()


def _fasta(names, rows):
    from tests.test_host import _fasta as f

    return f(names, rows)


@pytest.mark.gpu
@pytest.mark.parametrize("low_mem", [False, True])
def test_msa_reroot_end_to_end(port, low_mem):
    """pmh_msa_reroot on random FASTA / Newick builds (Fitch and --low-mem-mode, with and without --reference, with leaves
    absent from the FASTA): the lists against the port run as src/reroot.cpp runs the pass, the NucMut fields against the MSA
    run-merge (and the reference's own NucMut where it is built), the root's block insertion against the block pass on the
    new tree; tips whose parent is the root, tips whose old root disappears, and a second reroot of the result."""
    import panman_b200 as pb
    from oracle.oracle import RefNucMut, have_ref_nucmut
    from panman_b200.host import MsaBuild
    from tests.golden_util import writer_layout

    refnm = RefNucMut() if have_ref_nucmut() else None
    ctx = pb.Context(0)
    rng = np.random.default_rng(63 + int(low_mem))
    chars = np.frombuffer(b"-ACMGRSVTWYHKDBN", np.uint8)
    for trial in range(6):
        tree = random_tree(int(rng.integers(4, 70)), 6300 + trial, ["binary", "polytomy", "caterpillar"][trial % 3], max_arity=4)
        codes, _ = evolve(tree, int(rng.integers(1, 2200)), rng, 0.05)
        codes[:, (codes == 0).all(0)] = 1  # no all-gap column: the -M branch would drop it
        names = [tree.names[v] for v in tree.leaves]
        keep = np.ones(len(names), bool)
        if trial % 2:
            keep[rng.choice(len(names), size=max(1, len(names) // 5), replace=False)] = False  # absent from the FASTA
            keep[0] = True
        kept_rows = tree.leaf_row[tree.leaves[keep]]
        codes[tree.leaf_row[tree.leaves[0]], (codes[kept_rows] == 0).all(0)] = 1  # --low-mem-mode refuses all-gap columns
        rows_txt = chars[codes[tree.leaf_row[tree.leaves]]]
        reference = names[0] if trial % 3 == 1 else ""
        build = MsaBuild(ctx, _fasta([n for n, k in zip(names, keep) if k], rows_txt[keep]), tree.to_newick(), reference, low_mem)
        pc = CODE_OF[np.frombuffer(build.consensus, np.uint8)]
        present = np.zeros(tree.n_leaves, bool)
        present[tree.leaf_row[tree.leaves[keep]]] = True
        cur = FlatTree(list(tree.names), tree.parent, tree.child_off, tree.child_idx, tree.root, tree.leaf_row)
        # tips: one under the root (topology unchanged, the pass still forced), one deeper (the old root may disappear)
        under_root = [int(v) for v in cur.leaves if cur.parent[v] == cur.root]
        deep = [int(v) for v in cur.leaves if cur.parent[v] != cur.root]
        picks = [cur.names[v] for v in (under_root[0] if under_root else int(cur.leaves[0]), deep[-1] if deep else int(cur.leaves[-1]))]
        for step, name in enumerate(picks):  # the second reroots the result of the first
            tip = cur.names.index(name)
            po, pos, info, nucs = _pieces_of_build(build)
            rows = replay_pieces(cur, po, pos, info, nucs, pc)
            if len(pc) == codes.shape[1]:  # no all-gap column was dropped: every present leaf gets its input back
                assert np.array_equal(rows[present], codes[present]), trial
            build.reroot(ctx, name)
            new = _flat(build.tree)
            assert _by_name(new) == _py_transform(cur, tip), (trial, step)
            assert {new.names[v]: int(new.leaf_row[v]) for v in new.leaves} == {cur.names[v]: int(cur.leaf_row[v]) for v in cur.leaves}
            row = int(cur.leaf_row[tip])
            want, _ = port.run(new, 0, rows, pc, rows[row].astype(np.int8), None, None, n_threads=2)
            assert np.array_equal(build.tuple_offsets, want.node_offsets), (trial, step)
            assert np.array_equal(build.tuple_pos, want.pos) and np.array_equal(build.tuple_type_code, want.type_code), (trial, step)
            blk, _ = port.run(new, 0, np.ones((new.n_leaves, 1), np.uint8), np.zeros(1, np.uint8), np.ones(1, np.int8), None, None, 1)
            for v in range(new.n_nodes):
                p, tc = want.of(v)
                wp, wmi, wnu = port.merge_msa(p, tc) if len(p) else ([], [], [])
                got = build.nucmut[v]
                assert [g[0] for g in got] == list(wp) and [g[4] for g in got] == list(wmi) and [g[5] for g in got] == list(wnu)
                assert all(g[1] == -1 and g[2] == 0 and g[3] == -1 for g in got)
                if refnm is not None and len(p):
                    rb, rsb, rp, rg, rinfo, rnucs = refnm.merge_pangraph(0, [0] * len(p), p, [-1] * len(p), tc >> 4, tc & 15)
                    assert got == [(int(rp[i]), int(rg[i]), int(rb[i]), int(rsb[i]), int(rinfo[i]), int(rnucs[i])) for i in range(len(rb))]
                bp, btc = blk.of(v)
                bt, inv = block_mut_from_nuc(btc >> 4, btc & 15)
                blockmut = [(int(bp[i]), -1, int(bt[i] == 1), int(inv[i])) for i in range(len(bp))]
                assert build.wire[v] == writer_layout(got, blockmut), (trial, step, v)
            assert build.wire[new.root][0][2] == 1  # the new root carries the block's insertion
            cur = new
        build.close()
    ctx.close()


def _pieces_of_build(build):
    off, pos, info, nucs = [0], [], [], []
    for v in range(build.tree.n_nodes):
        for g in build.nucmut[v]:
            pos.append(g[0])
            info.append(g[4])
            nucs.append(g[5])
        off.append(len(pos))
    return np.asarray(off, np.int64), np.asarray(pos, np.int32), np.asarray(info, np.uint8), np.asarray(nucs, np.uint32)


@pytest.mark.gpu
@pytest.mark.parametrize("name,c0,width", [("sars20k", 0, None), ("caterpillar100k", 14000, 2048), ("ecoli4k", 2_500_096, 16384)])
def test_full_size_configs(port, name, c0, width):
    """The configs through the C ABI: pass -> merge_runs -> pieces -> reroot_newick -> set_tree(new) -> upload_replay -> pass,
    against the port on the new tree. The slice's lists replay to the slice's own input (the replay property)."""
    import panman_b200 as pb
    from panman_b200 import synth

    cfg = synth.CONFIGS[name]
    st = synth.make_tree(cfg["n_leaves"], cfg["seed"], cfg["kind"])
    spec = synth.MsaSpec(cfg["seed"], cfg["p_sub"], cfg["f_gap"], cfg["p_N"])
    width = width or cfg["n_cols"]
    codes4, pc = synth.simulate_msa(st, c0, c0 + width, spec, device="cuda")
    codes = synth.unpack_nibbles(codes4, width).cpu().numpy()
    pc = pc.cpu().numpy()
    old = FlatTree(st.names(), st.parent.astype(np.int32), st.child_off.astype(np.int32), st.child_idx.astype(np.int32), int(st.root),
                   st.leaf_row.astype(np.int32))
    ctx = pb.Context(0)
    ctx.set_tree(old.n_nodes, old.root, old.child_off, old.child_idx, old.leaf_row)
    ctx.upload(width, old.n_leaves, codes4, codes4.shape[1], pc)
    ctx.run_resident(pb.ALGO_FITCH)
    po, pos, info, nucs, _ = ctx.merge_runs()
    tip = int(old.leaves[len(old.leaves) // 3])
    new = rerooted(old, old.names[tip])
    ctx.set_tree(new.n_nodes, new.root, new.child_off, new.child_idx, new.leaf_row)
    ctx.upload_replay(old, po, pos, info, nucs, width, pc, int(old.leaf_row[tip]))
    ctx.run_resident(pb.ALGO_FITCH)
    res = ctx.download()
    want, _ = port.run(new, 0, codes, pc, codes[old.leaf_row[tip]].astype(np.int8), None, None, n_threads=16)
    assert np.array_equal(res.node_offsets, want.node_offsets), name
    assert np.array_equal(res.pos, want.pos) and np.array_equal(res.type_code, want.type_code), name
    ctx.close()


@pytest.mark.gpu
def test_refusals_and_context_state(port):
    """Every refusal of pmb_upload_replay, each followed by a valid call; a replay issued while asynchronous passes run on two
    lanes; a dense upload after a replay on the same context."""
    import panman_b200 as pb

    rng = np.random.default_rng(64)
    tree, rows, cons, _ = _case(rng, 0, 300, 3000, "binary")
    lists, _ = port.run(tree, 0, rows, cons)
    po, pos, info, nucs = pieces_of(port, tree, lists)
    want_rows = replay_pieces(tree, po, pos, info, nucs, cons)
    tip = int(tree.leaves[7])
    new = rerooted(tree, tree.names[tip])
    want, _ = port.run(new, 0, want_rows, cons, want_rows[tree.leaf_row[tip]].astype(np.int8), None, None, n_threads=4)
    ctx = pb.Context(0)
    ctx.set_tree(new.n_nodes, new.root, new.child_off, new.child_idx, new.leaf_row)
    row = int(tree.leaf_row[tip])

    def good():
        ctx.upload_replay(tree, po, pos, info, nucs, len(cons), cons, row)
        ctx.run_resident(pb.ALGO_FITCH)
        r = ctx.download()
        assert np.array_equal(r.node_offsets, want.node_offsets) and np.array_equal(r.pos, want.pos)
        assert np.array_equal(r.type_code, want.type_code)

    def bad(**kw):
        a = dict(old_tree=tree, piece_offsets=po, nuc_position=pos, mut_info=info, nucs=nucs, n_cols=len(cons), parent_code=cons,
                 root_leaf_row=row)
        a.update(kw)
        with pytest.raises(pb.PanmanError) as e:
            ctx.upload_replay(**a)
        assert e.value.code == -1
        good()

    good()
    broken = FlatTree(tree.names, tree.parent, tree.child_off, tree.child_idx.copy(), tree.root, tree.leaf_row)
    broken.child_idx[3] = broken.child_idx[2]
    bad(old_tree=broken)  # malformed old tree
    other = random_tree(301, 5, "binary")
    bad(old_tree=other, piece_offsets=np.zeros(other.n_nodes + 1, np.int64))  # another leaf-row set
    bad(piece_offsets=po + 1)  # not starting at 0
    po2 = po.copy()
    k = int(np.argmax(np.diff(po) > 0))
    po2[k + 1], po2[k + 2] = po2[k + 2] + 1, po2[k + 1]
    bad(piece_offsets=po2)  # not monotone
    for i, bad_info in enumerate([(1 << 4) | 3, (1 << 4) | 4, 0 << 4, 7 << 4]):  # type above 2 (NSNP* forms), length 0 / 7
        inf = info.copy()
        inf[i] = bad_info
        bad(mut_info=inf)
    p2 = pos.copy()
    p2[-1] = len(cons) - (int(info[-1]) >> 4) + 1
    bad(nuc_position=p2)  # beyond n_cols
    bad(root_leaf_row=tree.n_leaves)
    bad(root_leaf_row=-2)
    # asynchronous passes on two lanes in flight, then a replay; then a dense upload on the same context
    codes4 = pb.pack_nibbles(want_rows)
    ctx.upload(len(cons), tree.n_leaves, codes4, codes4.shape[1], cons, want_rows[row].astype(np.int8))
    for _ in range(6):
        ctx.run_resident_async(pb.ALGO_FITCH)
    good()
    ctx.wait()
    w2, _ = port.run(new, 0, rows, cons, None, None, None, n_threads=4)
    r = ctx.run_codes(new, pb.ALGO_FITCH, rows, cons)
    assert np.array_equal(r.node_offsets, w2.node_offsets) and np.array_equal(r.pos, w2.pos) and np.array_equal(r.type_code, w2.type_code)
    good()
    ctx.close()


@pytest.mark.gpu
def test_msa_reroot_refusals():
    import ctypes as C

    import panman_b200 as pb
    from panman_b200.host import MsaBuild, load_host_library

    ctx = pb.Context(0)
    L = load_host_library()
    L.pmh_msa_prepare.restype = C.c_void_p
    L.pmh_msa_prepare.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_char_p, C.c_int, C.c_char_p, C.c_size_t]
    L.pmh_msa_reroot.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_char_p, C.c_size_t]
    err = C.create_string_buffer(256)
    fa = b">a\nACGT\n>b\nACGA\n>c\nTCGA\n"
    h = L.pmh_msa_prepare(fa, len(fa), b"((a,b),c);", b"", 0, err, 256)
    assert h and L.pmh_msa_reroot(ctx.h, h, b"a", err, 256) == -5 and b"pmh_msa_run" in err.value  # not built yet
    L.pmh_build_free(h)
    build = MsaBuild(ctx, b">a\nACGT\n>b\nACGA\n>c\nTCGA\n", "((a,b),c);")
    with pytest.raises(pb.PanmanError, match="not found"):
        build.reroot(ctx, "zzz")
    with pytest.raises(pb.PanmanError, match="not a tip"):
        build.reroot(ctx, "node_2")
    build.reroot(ctx, "a")
    assert build.tree.names[:2] == ["node_3", "a"]
    build.close()
    ctx.close()
