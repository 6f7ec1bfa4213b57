"""Inputs for the device replay of a PanMAT's mutation lists (pmb_upload_replay; no GPU needed): replay_piece_len_kernel,
the record sort on column << rec_bits | record number, replay_sweep_kernel (its stack of nested leaf intervals and the
restatement at every segment start), the event sort on item << 32 | event, replay_items_kernel and expand_runs_kernel.

replay_reference is the plain replay of NucMut pieces: consensus, then root -> leaf every piece in stored order (NS / NI
write their nucs nibbles, ND writes '-' = 0), vectorised so that it handles 65 536 leaves x 2 048 columns in seconds.

Each builder returns a list of Case: the tree the pieces were built on, the pieces (node-major over its node ids), the
consensus codes, the leaf row whose replayed codes become the root override (-1: none) and what the case claims to
contain. The edges are placed on purpose: leaf intervals starting, ending and spanning on segment starts (the geometry
is pb.Runs.info, computed by the same pmb::runs_segments the replay uses), the tip at the segment and clade edges, a
stack 20 000 deep and a column with a record at each of 131 071 nodes, record counts and widths at the key-width
boundaries, every piece type, length and nibble, pieces across a tile edge and at n_cols, no pieces at all, and the
same tree under three relabellings that are not in pre-order.

Not covered: segments of more than about 2^17 rows (the high bits of the 18-bit row field of an event) and
n_rows > RUNS_MAX_SEG_ROWS. runs_segments only makes segments that long with more than about 4 096 tiles of 262 k leaves,
a plane matrix no single B200 holds."""
from dataclasses import dataclass, field
from functools import lru_cache

import numpy as np

from oracle.oracle import FlatTree, random_tree

TILE_COLS = 1024
NS, ND, NI = 0, 1, 2
KEY_WIDTH_K = (17, 20)   # record counts 2^k - 1, 2^k, 2^k + 1
COL_WIDTH_K = (11, 16)   # n_cols 2^k - 1, 2^k, 2^k + 1


@dataclass
class Case:
    name: str
    tree: FlatTree
    pieces: tuple                 # (piece_off int64[n_nodes + 1], nuc_position int32, mut_info uint8, nucs uint32)
    parent_code: np.ndarray       # uint8, n_cols
    tip_row: int = -1
    claims: dict = field(default_factory=dict)

    @property
    def n_cols(self) -> int:
        return len(self.parent_code)

    @property
    def n_records(self) -> int:
        return int((self.pieces[2] >> 4).astype(np.int64).sum())

    def reference(self) -> np.ndarray:
        return replay_reference(self.tree, *self.pieces, self.parent_code)


# ------------------------------------------------------------------------------------------------------------ the tree


@dataclass
class Walk:
    pre: np.ndarray       # node ids in pre-order (children in stored order)
    depth: np.ndarray     # by node id, the root at 0
    x: np.ndarray         # by node id: [x, y) = its leaves in depth-first order
    y: np.ndarray
    dfs_rows: np.ndarray  # leaf rows in depth-first order


def walk(tree) -> Walk:
    n = tree.n_nodes
    co, ci = np.asarray(tree.child_off, np.int64), np.asarray(tree.child_idx, np.int64)
    pre = np.empty(n, np.int64)
    depth = np.zeros(n, np.int64)
    stack, k = [int(tree.root)], 0
    while stack:
        v = stack.pop()
        pre[k] = v
        k += 1
        kids = ci[co[v]:co[v + 1]]
        depth[kids] = depth[v] + 1
        stack.extend(kids[::-1].tolist())
    assert k == n
    is_leaf = np.diff(co) == 0
    par = np.full(n, -1, np.int64)
    par[ci] = np.repeat(np.arange(n), np.diff(co))
    n_leaf = is_leaf.astype(np.int64)
    for d in range(int(depth.max()), 0, -1):  # a level at a time, children before parents
        at = np.nonzero(depth == d)[0]
        np.add.at(n_leaf, par[at], n_leaf[at])
    x = np.zeros(n, np.int64)
    x[pre] = np.cumsum(is_leaf[pre]) - is_leaf[pre]
    return Walk(pre, depth, x, x + n_leaf, np.asarray(tree.leaf_row, np.int64)[pre[is_leaf[pre]]])


def segment_geometry(tree, n_cols):
    """(n_segments, seg_rows) of a replay of `tree` over n_cols columns, as pmb::runs_segments computes them."""
    import panman_b200 as pb

    codes4 = np.zeros((tree.n_leaves, (n_cols + 1) // 2), np.uint8)
    runs = pb.Runs.of_tree(tree, n_cols, codes4, np.zeros(n_cols, np.uint8))
    try:
        return int(runs.info.n_segments), int(runs.info.seg_rows)
    finally:
        runs.close()


def balanced_tree(n_leaves) -> FlatTree:
    """A complete binary tree of n_leaves (a power of two) leaves, ids in pre-order."""
    children, leaf = [], []
    stack = [(-1, n_leaves)]
    while stack:
        p, m = stack.pop()
        v = len(children)
        children.append([])
        leaf.append(m == 1)
        if p >= 0:
            children[p].append(v)
        if m > 1:
            stack += [(v, m // 2), (v, m // 2)]  # the left one is popped first and numbered in full before the right
    names = [f"B{v}" if leaf[v] else f"node_{v + 1}" for v in range(len(children))]
    return FlatTree.from_children(names, children)


def relabel(tree, new_id=None, reverse_children=False, row_perm=None) -> FlatTree:
    """The same tree under other node ids (new_id[v]), with every child list reversed, and/or leaf row r renamed
    row_perm[r]. Names travel with their nodes."""
    n = tree.n_nodes
    new_id = np.arange(n) if new_id is None else np.asarray(new_id)
    old_of = np.argsort(new_id)
    co, ci = np.asarray(tree.child_off), np.asarray(tree.child_idx)
    off, idx = [0], []
    for u in range(n):
        kids = [int(new_id[c]) for c in ci[co[old_of[u]]:co[old_of[u] + 1]]]
        idx += kids[::-1] if reverse_children else kids
        off.append(len(idx))
    parent = np.full(n, -1, np.int32)
    for u in range(n):
        parent[idx[off[u]:off[u + 1]]] = u
    lr = np.asarray(tree.leaf_row, np.int32)[old_of].copy()
    if row_perm is not None:
        lr[lr >= 0] = np.asarray(row_perm)[lr[lr >= 0]]
    return FlatTree([tree.names[v] for v in old_of], parent, np.asarray(off, np.int32), np.asarray(idx, np.int32),
                    int(new_id[tree.root]), lr)


# ---------------------------------------------------------------------------------------------------------- the pieces


def nucs_of(codes) -> int:
    """NucMut.nucs of a piece: code j in the nibble at bit 4 * (5 - j)."""
    return sum((int(c) & 15) << (4 * (5 - j)) for j, c in enumerate(codes))


class Pieces:
    """Pieces collected in any node order; pack() makes them node-major, in the order they were added within a node."""

    def __init__(self):
        self.parts = []

    def add(self, node, pos, typ, length, nucs):
        node, pos, typ, length, nucs = np.broadcast_arrays(*(np.asarray(a, np.int64) for a in (node, pos, typ, length, nucs)))
        self.parts.append((node.ravel(), pos.ravel(), typ.ravel(), length.ravel(), nucs.ravel()))
        return self

    def codes(self, node, pos, typ, codes):
        """One piece writing `codes` (1 .. 6 of them) from pos."""
        return self.add(node, pos, typ, len(codes), nucs_of(codes))

    def random(self, rng, nodes, n_cols, per_node=1.0, max_len=6, col0=0):
        """About per_node random pieces on each of `nodes` (Poisson) in columns col0 .. n_cols - 1, of every type, length
        and nibble."""
        nodes = np.asarray(nodes, np.int64)
        node = np.repeat(nodes, rng.poisson(per_node, size=len(nodes)))
        length = rng.integers(1, max_len + 1, size=len(node))
        return self.add(node, rng.integers(col0, n_cols - length + 1), rng.integers(0, 3, size=len(node)), length,
                        rng.integers(0, 1 << 24, size=len(node)))

    def pack(self, n_nodes):
        node, pos, typ, length, nucs = (np.concatenate([p[k] for p in self.parts]) if self.parts else np.zeros(0, np.int64)
                                        for k in range(5))
        order = np.argsort(node, kind="stable")
        off = np.zeros(n_nodes + 1, np.int64)
        np.cumsum(np.bincount(node, minlength=n_nodes), out=off[1:])
        assert ((length >= 1) & (length <= 6)).all() and ((typ >= 0) & (typ <= 2)).all()
        return (off, pos[order].astype(np.int32), ((length << 4) | typ)[order].astype(np.uint8),
                (nucs[order] & 0xFFFFFFFF).astype(np.uint32))


def relabel_pieces(pieces, new_id):
    """Node-major pieces over old ids -> node-major over new ids (each node keeps its own pieces in order)."""
    off, pos, info, nucs = pieces
    n = len(off) - 1
    node = np.asarray(new_id)[np.repeat(np.arange(n), np.diff(off))]
    order = np.argsort(node, kind="stable")
    new_off = np.zeros(n + 1, np.int64)
    np.cumsum(np.bincount(node, minlength=n), out=new_off[1:])
    return new_off, pos[order], info[order], nucs[order]


def records(n_nodes, piece_off, pos, info, nucs):
    """Pieces -> records (node, column, code) in stored order, the way replay_records_kernel expands them."""
    info = np.asarray(info, np.uint8)
    length = (info >> 4).astype(np.int64)
    piece = np.repeat(np.arange(len(info)), length)
    j = np.arange(len(piece)) - np.repeat(np.cumsum(length) - length, length)
    col = np.asarray(pos, np.int64)[piece] + j
    code = np.where((info[piece] & 15) == ND, 0, (np.asarray(nucs, np.int64)[piece] >> (4 * (5 - j))) & 15).astype(np.uint8)
    node = np.repeat(np.arange(n_nodes), np.diff(np.asarray(piece_off, np.int64)))[piece]
    return node, col, code


def replay_reference(tree, piece_off, pos, info, nucs, parent_code) -> np.ndarray:
    """getSequenceFromReference on NucMut pieces for every leaf: (n_leaves, n_cols) codes by leaf row. A depth-first walk
    keeps only the rows of the current root-to-node path; within a node the later of two records on one column wins (kept
    explicitly, not left to the order of a fancy assignment with repeated indices)."""
    pc = np.asarray(parent_code, np.uint8)
    n_cols, n = len(pc), tree.n_nodes
    node, col, code = records(n, piece_off, pos, info, nucs)
    key = node * n_cols + col
    _, last_rev = np.unique(key[::-1], return_index=True)
    keep = np.sort(len(key) - 1 - last_rev)  # the last record of every (node, column), in stored order
    node, col, code = node[keep], col[keep], code[keep]
    roff = np.searchsorted(node, np.arange(n + 1))
    W = walk(tree)
    lr = np.asarray(tree.leaf_row)
    rows = np.empty((tree.n_leaves, n_cols), np.uint8)
    path = [pc]  # path[d + 1]: the codes of the node at depth d on the current path
    for v in W.pre.tolist():
        d = int(W.depth[v])
        a, b = roff[v], roff[v + 1]
        if lr[v] >= 0:
            cur = rows[lr[v]]
            cur[:] = path[d]
        else:
            cur = path[d].copy()
            if len(path) == d + 1:
                path.append(cur)
            else:
                path[d + 1] = cur
        cur[col[a:b]] = code[a:b]
    return rows


def stack_depth(tree, pieces, column) -> int:
    """The most records of one column on a root-to-leaf path: the depth replay_sweep_kernel's stack reaches there."""
    node, col, _ = records(tree.n_nodes, *pieces)
    cnt = np.bincount(node[col == column], minlength=tree.n_nodes)
    W = walk(tree)
    par = np.full(tree.n_nodes, -1, np.int64)
    par[np.asarray(tree.child_idx)] = np.repeat(np.arange(tree.n_nodes), np.diff(tree.child_off))
    on_path = cnt.copy()
    for v in W.pre[1:]:  # parents before children
        on_path[v] += on_path[par[v]]
    return int(on_path.max())


# ------------------------------------------------------------------------------------------------------------ builders


def _consensus(rng, n_cols):
    return rng.choice(np.asarray([1, 2, 4, 8], np.uint8), size=n_cols)


@lru_cache(maxsize=None)
def segment_edges():
    """A tree of 4 100 leaves in one tile: 64 segments of 65 rows. Pieces on nodes whose leaf interval starts on a segment
    start, ends on one, or holds two or more whole segments; and siblings meeting on a segment start under a parent that
    writes column c, the first restoring the consensus in c, the second writing a third code."""
    rng = np.random.default_rng(81)
    tree = random_tree(4100, 8100, "binary")
    n_cols = 1000
    n_seg, seg_rows = segment_geometry(tree, n_cols)
    W = walk(tree)
    starts = np.arange(1, n_seg) * seg_rows
    internal = np.diff(tree.child_off) > 0
    x_on = np.nonzero(np.isin(W.x, starts))[0]
    y_on = np.nonzero(np.isin(W.y, starts))[0]
    spans = np.nonzero(W.y // seg_rows - (W.x + seg_rows - 1) // seg_rows >= 2)[0]
    spans = spans[spans != tree.root]
    pick = lambda a, k: rng.choice(a, size=min(k, len(a)), replace=False)
    x_on = np.concatenate([pick(x_on[internal[x_on]], 40), pick(x_on[~internal[x_on]], 20)])
    y_on = np.concatenate([pick(y_on[internal[y_on]], 40), pick(y_on[~internal[y_on]], 20)])
    spans = pick(spans, 40)
    pc = _consensus(rng, n_cols)
    P = Pieces().random(rng, np.arange(tree.n_nodes), n_cols - 100, per_node=0.3)
    for v in np.concatenate([x_on, y_on, spans]):
        P.random(rng, [v], n_cols - 100, per_node=3)
        P.codes(v, int(rng.integers(0, n_cols - 106)), NS, [int(k) for k in rng.integers(0, 16, size=6)])
    # siblings (u, w) with y[u] = x[w] on a segment start, under parent a: a writes c, u writes pc[c], w a third code
    triples = []
    for a in np.nonzero(internal)[0]:
        kids = tree.child_idx[tree.child_off[a]:tree.child_off[a + 1]]
        for u, w in zip(kids[:-1], kids[1:]):
            if W.y[u] in starts and W.y[u] - W.x[u] > 1 and len(triples) < 60:
                triples.append((int(a), int(u), int(w)))
    for i, (a, u, w) in enumerate(triples):
        c = n_cols - 100 + i
        other = [k for k in (1, 2, 4, 8) if k != pc[c]]
        P.codes(a, c, NS, [other[0]])
        P.codes(u, c, NS, [pc[c]])
        P.codes(w, c, NS, [other[1]])
    tip = int(W.dfs_rows[seg_rows * (n_seg // 3)])
    claims = dict(n_seg=n_seg, seg_rows=seg_rows, x_on_start=x_on, y_on_start=y_on, spans_two=spans, restore_triples=triples)
    return [Case("segment_edges", tree, P.pack(tree.n_nodes), pc, tip, claims)]


@lru_cache(maxsize=None)
def tip_positions():
    """The segment-edge tree and pieces, plus a clade with a record in every column; the tip at depth-first position 0, at
    the last one, at the first and last row of a middle segment, at the first leaf of that clade, and none."""
    base = segment_edges()[0]
    rng = np.random.default_rng(82)
    tree, n_cols = base.tree, base.n_cols
    n_seg, seg_rows = base.claims["n_seg"], base.claims["seg_rows"]
    W = walk(tree)
    sizes = W.y - W.x
    clade = int(rng.choice(np.nonzero((sizes >= 3) & (sizes <= 40) & (W.x > 0) & (W.x % seg_rows != 0))[0]))
    off, pos, info, nucs = base.pieces
    P = Pieces()
    node = np.repeat(np.arange(tree.n_nodes), np.diff(off))
    P.add(node, pos, info & 15, info >> 4, nucs)
    for c0 in range(0, n_cols, 6):
        ln = min(6, n_cols - c0)
        P.codes(clade, c0, NS, [int(k) for k in rng.choice([0, 1, 2, 4, 8, 15], size=ln)])
    pieces = P.pack(tree.n_nodes)
    mid = n_seg // 2
    where = dict(first=0, last=tree.n_leaves - 1, segment_first=mid * seg_rows, segment_last=(mid + 1) * seg_rows - 1,
                 clade_first=int(W.x[clade]))
    cases = [Case(f"tip_{k}", tree, pieces, base.parent_code, int(W.dfs_rows[p]), dict(tip_pos=p, clade=clade, **base.claims))
             for k, p in where.items()]
    cases.append(Case("tip_none", tree, pieces, base.parent_code, -1, dict(tip_pos=-1, clade=clade, **base.claims)))
    return cases


@lru_cache(maxsize=None)
def nesting():
    """A caterpillar of 20 000 leaves with a record at every spine node in column 17, the codes alternating so that every
    level changes the leaf code (a stack 19 999 deep); a complete binary tree of 65 536 leaves with a record at every node
    in column 1500 (131 071 records, a pop and a push between every two siblings)."""
    rng = np.random.default_rng(83)
    cat = random_tree(20000, 8300, "caterpillar")
    n_cols = 64
    pc = _consensus(rng, n_cols)
    pc[17] = 1
    W = walk(cat)
    spine = np.nonzero(np.diff(cat.child_off) > 0)[0]
    P = Pieces().random(rng, np.arange(cat.n_nodes), n_cols, per_node=0.05, col0=18)
    P.add(spine, 17, NS, 1, np.where(W.depth[spine] % 2 == 0, 2, 4) << 20)
    deepest = int(W.pre[np.argmax(np.where(np.diff(cat.child_off) == 0, W.depth, -1)[W.pre])])
    cases = [Case("caterpillar_stack", cat, P.pack(cat.n_nodes), pc, int(cat.leaf_row[deepest]), dict(column=17, depth=len(spine)))]
    bal = balanced_tree(65536)
    n_cols = 2048
    pc = _consensus(rng, n_cols)
    P = Pieces().random(rng, np.arange(bal.n_nodes), n_cols, per_node=0.3)
    P.add(np.arange(bal.n_nodes), 1500, NS, 1, rng.integers(0, 16, size=bal.n_nodes) << 20)
    cases.append(Case("balanced_every_node", bal, P.pack(bal.n_nodes), pc, -1, dict(column=1500, depth=17)))
    return cases


def _last_in_preorder(tree):
    return int(walk(tree).pre[-1])


def _exact_records(rng, tree, n_cols, R):
    """Pieces on every node, R records in all, the last of them on the node last in pre-order."""
    last = _last_in_preorder(tree)
    others = np.asarray([v for v in range(tree.n_nodes) if v != last])
    P = Pieces().add(others, rng.integers(0, n_cols, size=len(others)), NS, 1, rng.integers(0, 1 << 24, size=len(others)))  # none empty
    budget = R - R // 20 - len(others)  # the last node takes what is left
    length = rng.integers(1, 7, size=int(budget / 3))
    length = length[np.cumsum(length) <= budget]
    node = rng.choice(others, size=len(length))
    P.add(node, rng.integers(0, n_cols - length + 1), rng.integers(0, 3, size=len(node)), length, rng.integers(0, 1 << 24, size=len(node)))
    rest = R - sum(int(p[3].sum()) for p in P.parts)
    assert rest >= R // 20
    ln = np.full(rest // 6, 6)
    if rest % 6:
        ln = np.append(ln, rest % 6)
    P.add(last, rng.integers(0, n_cols - ln + 1), rng.integers(0, 3, size=len(ln)), ln, rng.integers(0, 1 << 24, size=len(ln)))
    return P.pack(tree.n_nodes)


@lru_cache(maxsize=None)
def key_widths():
    """Record counts R = 1, 2, 3 and 2^k - 1, 2^k, 2^k + 1 (k = 17, 20), the highest record number on the node last in
    pre-order; n_cols = 2^k - 1, 2^k, 2^k + 1 (k = 11, 16) with records in column 0, 2^(k - 1) and n_cols - 1."""
    rng = np.random.default_rng(84)
    cases = []
    tree = random_tree(2000, 8401, "binary")
    n_cols = 3000
    pc = _consensus(rng, n_cols)
    for k in KEY_WIDTH_K:
        for R in (2 ** k - 1, 2 ** k, 2 ** k + 1):
            tip = int(tree.leaf_row[_last_in_preorder(tree)]) if R % 2 else -1
            cases.append(Case(f"records_2^{k}{R - 2 ** k:+d}", tree, _exact_records(rng, tree, n_cols, R), pc, tip, dict(R=R)))
    small = random_tree(40, 8400, "polytomy", max_arity=4)
    n_cols = 100
    pc = _consensus(rng, n_cols)
    last, root = _last_in_preorder(small), int(small.root)
    mid = int(walk(small).pre[small.n_nodes // 2])
    for R, nodes in ((1, [last]), (2, [root, last]), (3, [root, mid, last])):
        P = Pieces()
        for v in nodes:
            P.codes(v, int(rng.integers(0, n_cols)), NS, [int(rng.choice([0, 2, 4, 15]))])
        cases.append(Case(f"records_{R}", small, P.pack(small.n_nodes), pc, int(small.leaf_row[last]), dict(R=R)))
    tree = random_tree(300, 8402, "binary")
    W = walk(tree)
    for k in COL_WIDTH_K:
        for n_cols in (2 ** k - 1, 2 ** k, 2 ** k + 1):
            pc = _consensus(rng, n_cols)
            P = Pieces().random(rng, np.arange(tree.n_nodes), n_cols, per_node=0.5)
            edge = (0, 2 ** (k - 1), n_cols - 1)
            for c in edge:
                for v in rng.choice(tree.n_nodes, size=12, replace=False):
                    P.codes(v, c, int(rng.integers(0, 3)), [int(rng.integers(0, 16))])
            P.codes(W.pre[-1], n_cols - 6, NS, [1, 2, 4, 8, 15, 0])
            tip = int(W.dfs_rows[-1]) if n_cols % 2 else -1
            cases.append(Case(f"cols_{n_cols}", tree, P.pack(tree.n_nodes), pc, tip, dict(n_cols=n_cols, edge_cols=edge)))
    return cases


@lru_cache(maxsize=None)
def piece_forms():
    """Every (type, length); every nibble 0 .. 15 in the nucs of NS and NI pieces, ND pieces with non-zero nucs; a length-6
    piece over columns 1020 .. 1025 (a tile edge) and pieces ending at n_cols; pieces overlapping within one node; an
    ancestor and a descendant writing the same code."""
    rng = np.random.default_rng(85)
    tree = random_tree(300, 8500, "polytomy", max_arity=5)
    n_cols = 2000
    pc = _consensus(rng, n_cols)
    n = tree.n_nodes
    W = walk(tree)
    P = Pieces().random(rng, np.arange(n), n_cols, per_node=0.5)
    for t in (NS, ND, NI):
        for ln in range(1, 7):
            P.codes(int(rng.integers(0, n)), int(rng.integers(0, n_cols - ln + 1)), t, [int(c) for c in rng.integers(0, 16, size=ln)])
    for t in (NS, NI):
        for j in range(6):  # nibble j of a length-6 piece takes every value
            for val in range(16):
                codes = [int(c) for c in rng.integers(0, 16, size=6)]
                codes[j] = val
                P.codes(int(rng.integers(0, n)), int(rng.integers(0, n_cols - 5)), t, codes)
    for ln in range(1, 7):
        P.add(int(rng.integers(0, n)), int(rng.integers(0, n_cols - ln + 1)), ND, ln, int(rng.integers(1, 1 << 24)))
    P.add(int(rng.integers(0, n)), 300, ND, 6, 0xFFFFFF)
    # unused low nibbles of a short piece hold garbage: only the top `length` nibbles are codes
    P.add(int(rng.integers(0, n)), 400, NS, 2, nucs_of([4, 8]) | 0xABCD)
    leaf = int(tree.leaves[5])
    P.codes(leaf, 1020, NS, [1, 2, 4, 8, 15, 0])
    P.codes(int(tree.root), 1020, NI, [3, 5, 6, 7, 9, 10])
    P.codes(leaf, n_cols - 6, NI, [11, 12, 13, 14, 3, 5])
    P.codes(int(tree.leaves[6]), n_cols - 1, NS, [0])
    P.codes(int(tree.root), n_cols - 3, ND, [9, 9, 9])
    over = int(tree.leaves[7])
    P.codes(over, 5, NS, [2, 2, 2, 2])
    P.codes(over, 7, NI, [8, 8, 8])
    P.codes(over, 6, ND, [4])
    inner = [v for v in W.pre[1:] if W.y[v] - W.x[v] >= 4][:5]
    same = []
    for i, a in enumerate(inner):  # the node and its first child write the same code: their events compose to nothing
        d = int(tree.child_idx[tree.child_off[a]])
        code = [k for k in (1, 2, 4, 8) if k != pc[600 + i]][0]
        P.codes(int(a), 600 + i, NS, [code])
        P.codes(d, 600 + i, NS, [code])
        same.append((int(a), d, 600 + i))
    claims = dict(tile_edge=(leaf, 1020), overlap=over, same_code=same)
    return [Case("piece_forms", tree, P.pack(n), pc, int(tree.leaf_row[leaf]), claims)]


@lru_cache(maxsize=None)
def empty_and_one_sided():
    """No piece at all, with and without a tip; pieces on the root only; pieces on leaves only."""
    rng = np.random.default_rng(86)
    tree = random_tree(500, 8600, "binary")
    n_cols = 1500
    pc = _consensus(rng, n_cols)
    none = Pieces().pack(tree.n_nodes)
    tip = int(tree.leaf_row[tree.leaves[250]])
    root = Pieces().random(rng, [tree.root], n_cols, per_node=300).pack(tree.n_nodes)
    leaves = Pieces().random(rng, tree.leaves, n_cols, per_node=3).pack(tree.n_nodes)
    return [Case("no_pieces", tree, none, pc, -1), Case("no_pieces_tip", tree, none, pc, tip),
            Case("root_only", tree, root, pc, tip), Case("leaves_only", tree, leaves, pc, tip)]


@lru_cache(maxsize=None)
def relabelled():
    """One tree and its pieces under node ids in reverse pre-order, with every child list reversed, and with leaf rows
    permuted against the depth-first order. Each case claims `rows_of`: the leaf-row map from the first case."""
    rng = np.random.default_rng(87)
    tree = random_tree(1500, 8700, "polytomy", max_arity=4)
    n_cols = 1100
    pc = _consensus(rng, n_cols)
    n = tree.n_nodes
    pieces = Pieces().random(rng, rng.choice(n, size=n // 2, replace=False), n_cols, per_node=2).pack(n)
    tip = int(tree.leaf_row[tree.leaves[100]])
    ident = np.arange(tree.n_leaves)
    cases = [Case("relabel_none", tree, pieces, pc, tip, dict(rows_of=ident))]
    rev = np.empty(n, np.int64)
    rev[walk(tree).pre] = np.arange(n)[::-1]
    cases.append(Case("relabel_reverse_preorder_ids", relabel(tree, rev), relabel_pieces(pieces, rev), pc, tip,
                      dict(rows_of=ident, new_id=rev)))
    cases.append(Case("relabel_reversed_children", relabel(tree, reverse_children=True), pieces, pc, tip, dict(rows_of=ident)))
    perm = rng.permutation(tree.n_leaves)
    cases.append(Case("relabel_permuted_rows", relabel(tree, row_perm=perm), pieces, pc, int(perm[tip]), dict(rows_of=perm)))
    return cases


BUILDERS = {"key_widths": key_widths, "segment_edges": segment_edges, "tip_positions": tip_positions, "nesting": nesting,
            "piece_forms": piece_forms, "empty_and_one_sided": empty_and_one_sided, "relabelled": relabelled}
