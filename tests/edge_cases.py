"""Case builders for the edge tests (test_emulation_edges.py on the CPU, test_gpu_edges.py on the device). No tests here.

The random suites derive every dimension from the trial index, so some combinations are never drawn. These builders place
the inputs on the boundaries where the kernels take their own code paths:
  * trees: stars of a given arity (the Sankoff counter width of an op is 2 / 4 / 8 / 20 bits for up to 3 / 15 / 255 / more
    references, tree_program.cpp), spines with leaf ribs (deep trees cut into chain segments), a tree holding one op of each
    width class under one wide op (per-op dispatch inside the 20-bit instantiation), and ops with 47 / 48 / 49 references
    or 31 / 32 / 33 leaf children (the shared-memory metadata windows of the pass kernels end at 48 references and 32 leaf
    entries);
  * inputs: presence masks (none, 70 %, one leaf, a run of rows omitted), root overrides, fwd_root_ref, block mode, noise,
    and on wide ops columns whose codes spread over every state, so that the per-state counters run near their top;
  * a small deterministic all-pairs generator over those dimensions and the schedule options.
Trees are numbered in pre-order, as the reference's Newick parser creates them."""
import itertools

import numpy as np

from oracle.oracle import FlatTree, random_tree

ARITIES = (2, 3, 4, 15, 16, 17, 31, 32, 33, 47, 48, 49, 255, 256, 257, 1000, 4096)
WIDTHS = (1, 31, 32, 33, 1023, 1024, 1025, 2049)
COL_BASE = 5  # a nonzero first column: positions come back shifted by it
PRESENCE = ("none", "p70", "one", "clade")
OVERRIDE = ("none", "some", "all")
NOISE = (0.0, 0.02, 0.5)


def pre_order(children, root=0) -> FlatTree:
    """A FlatTree of `children` (lists of node ids) renumbered in pre-order, children left to right."""
    order, stack = [], [root]
    while stack:
        v = stack.pop()
        order.append(v)
        stack.extend(reversed(children[v]))
    new = {v: i for i, v in enumerate(order)}
    return FlatTree.from_children([f"n{i}" for i in range(len(order))], [[new[c] for c in children[v]] for v in order], 0)


class _Builder:
    def __init__(self):
        self.children = [[]]  # node 0 is the root

    def add(self, kids=()):
        self.children.append(list(kids))
        return len(self.children) - 1

    def leaves(self, k):
        return [self.add() for _ in range(k)]

    def tree(self, root_kids):
        self.children[0] = list(root_kids)
        return pre_order(self.children, 0)


def star(a: int, n_cherries: int = 0, seed: int = 0) -> FlatTree:
    """A root with `a` children: `n_cherries` of them two-leaf internal nodes, the rest leaves, in a seeded order.
    The root's op has exactly `a` references."""
    rng = np.random.default_rng(seed)
    b = _Builder()
    kids = [b.add(b.leaves(2)) for _ in range(min(n_cherries, a))] + b.leaves(a - min(n_cherries, a))
    return b.tree([kids[i] for i in rng.permutation(len(kids))])


def spine(depth: int, rib_arity: int, seed: int = 0) -> FlatTree:
    """A backbone of `depth` internal nodes, each carrying `rib_arity` leaves beside the backbone child (on a seeded side):
    every backbone op has rib_arity + 1 references and rib_arity leaf children. The bottom node holds leaves only."""
    rng = np.random.default_rng(seed)
    b = _Builder()
    cur = b.add(b.leaves(rib_arity + 1))
    for _ in range(depth - 2):
        ribs = b.leaves(rib_arity)
        cur = b.add([cur] + ribs if rng.random() < 0.5 else ribs + [cur])
    ribs = b.leaves(rib_arity)
    return b.tree([cur] + ribs)


def mixed_classes(seed: int = 0) -> FlatTree:
    """One op of each counter width class under a single 300-reference op: children of 3 (2-bit), 15 (4-bit), 200 (8-bit) and
    260 (20-bit) leaves beside 296 leaves of the root itself. The kernel is instantiated for the widest class (MAXB = 20) and
    dispatches every op to its own width."""
    rng = np.random.default_rng(seed)
    b = _Builder()
    kids = [b.add(b.leaves(k)) for k in (3, 15, 200, 260)] + b.leaves(296)
    return b.tree([kids[i] for i in rng.permutation(len(kids))])


def op_arities(tree: FlatTree) -> np.ndarray:
    return np.diff(tree.child_off)


def shapes():
    """The named trees of the pairwise set: (name, builder) -- built lazily, each at most once per test module."""
    return {
        "star3": lambda: star(3, 1, seed=1),
        "star16": lambda: star(16, 2, seed=2),
        "star48": lambda: star(48, 3, seed=3),
        "star256": lambda: star(256, 5, seed=4),
        "star1000": lambda: star(1000, 5, seed=5),
        "spine_r1": lambda: spine(300, 1, seed=6),
        "spine_r3": lambda: spine(300, 3, seed=7),
        "spine_r20": lambda: spine(300, 20, seed=8),
        "caterpillar": lambda: random_tree(600, 9, "caterpillar"),
        "unary": lambda: random_tree(400, 10, "unary", max_arity=3),
        "mixed": lambda: mixed_classes(seed=11),
    }


DEEP_SHAPES = ("spine_r1", "spine_r3", "spine_r20", "caterpillar")


# ------------------------------------------------------------------------------------------------------------------ inputs
def presence(mode: str, n_leaves: int, rng) -> np.ndarray:
    """leaf_present per row: None (every leaf present), 70 % present, one leaf only, or a contiguous run of a third of the
    rows omitted (rows follow pre-order, so the run is a clade or a stretch of neighbouring clades)."""
    if mode == "none" or n_leaves < 2:
        return None
    if mode == "p70":
        lp = (rng.random(n_leaves) < 0.7).astype(np.uint8)
        lp[int(rng.integers(0, n_leaves))] = 1
        return lp
    if mode == "one":
        lp = np.zeros(n_leaves, np.uint8)
        lp[int(rng.integers(0, n_leaves))] = 1
        return lp
    assert mode == "clade"
    lp = np.ones(n_leaves, np.uint8)
    k = max(1, n_leaves // 3)
    a = int(rng.integers(0, n_leaves - k + 1))
    lp[a:a + k] = 0
    return lp


def make_inputs(tree: FlatTree, algo: int, block: int, presence_mode: str, override: str, fwd_ref: int, width: int, noise: float,
                rng, spread: bool = None):
    """(codes, parent_code, root_override, fwd_root_ref, leaf_present) for one case. Codes are a per-column base state with
    `noise` of the cells redrawn over every state of the mode (16 nucleotide codes, 3 block states). With `spread` (default:
    trees with an op of 16 or more references) every third column instead runs the codes through all states by row, and every
    fifth holds one state in all rows but one, so that per-state child counters reach their top and their top minus one."""
    nst = 3 if block else 16
    n = tree.n_leaves
    base = rng.integers(0, min(nst, 5), size=width)
    codes = np.repeat(base[None, :], n, 0)
    codes = np.where(rng.random(codes.shape) < noise, rng.integers(0, nst, size=codes.shape), codes)
    if spread is None:
        spread = int(op_arities(tree).max()) >= 16
    if spread:
        rows = np.arange(n)[:, None]
        cols = np.arange(width)
        s = cols[cols % 3 == 1]
        codes[:, s] = (rows + s[None, :]) % nst
        s = cols[cols % 5 == 2]
        codes[:, s] = base[s][None, :]
        codes[int(rng.integers(0, n)), s] = (base[s] + 1) % nst
    codes = codes.astype(np.uint8)
    pc = rng.integers(0, nst, size=width).astype(np.uint8)
    ro = None
    if override == "some":
        ro = np.where(rng.random(width) < 0.3, rng.integers(0, nst, size=width), -1).astype(np.int8)
    elif override == "all":
        ro = rng.integers(0, nst, size=width).astype(np.int8)
    fr = None
    if fwd_ref:
        assert algo == 0 and not block, "fwd_root_ref belongs to Fitch in nucleotide mode"
        fr = np.where(rng.random(width) < 0.3, rng.integers(0, nst, size=width), -1).astype(np.int8)
    return codes, pc, ro, fr, presence(presence_mode, n, rng)


# ---------------------------------------------------------------------------------------------------------------- all pairs
ENTRIES = ("codes", "resident", "async", "runs")
PAIRWISE_DIMS = {
    "shape": tuple(shapes()),
    "width": WIDTHS,
    "chunk_nodes": (0, 1, 2, 7, 64),
    "presence": PRESENCE,
    "entry": ENTRIES,
    "algo": (0, 1),
    "mode": ("nuc", "block"),
    "override": OVERRIDE,
    "noise": NOISE,
    "fwd_root_ref": (0, 1),
    "inline_nodes": (0, 3),
    "schedule": (0, 1),
}


def case_allowed(c: dict) -> bool:
    """The ABI's constraints on a (partial) case: fwd_root_ref only with Fitch in nucleotide mode."""
    if c.get("fwd_root_ref") == 1 and (c.get("algo") == 1 or c.get("mode") == "block"):
        return False
    return True


def all_pairs(dims: dict = None, allowed=case_allowed) -> list:
    """A deterministic covering array of strength 2: every allowed pair of values of two dimensions occurs in some case.
    Greedy: each case starts from the first pair not yet covered and takes, dimension by dimension, the value that covers the
    most open pairs with what is already chosen (ties: the value used least so far, then the first)."""
    dims = PAIRWISE_DIMS if dims is None else dims
    names = list(dims)
    open_pairs = set()
    for i, j in itertools.combinations(range(len(names)), 2):
        for a in dims[names[i]]:
            for b in dims[names[j]]:
                if allowed({names[i]: a, names[j]: b}):
                    open_pairs.add((i, a, j, b))
    used = {(i, v): 0 for i, n in enumerate(names) for v in dims[n]}
    cases = []
    while open_pairs:
        i0, a0, j0, b0 = min(open_pairs, key=lambda p: (p[0], p[2], dims[names[p[0]]].index(p[1]), dims[names[p[2]]].index(p[3])))
        chosen = {i0: a0, j0: b0}
        for k in range(len(names)):
            if k in chosen:
                continue
            best, best_key = None, None
            for v in dims[names[k]]:
                trial = {names[x]: y for x, y in chosen.items()}
                trial[names[k]] = v
                if not allowed(trial):
                    continue
                gain = sum(((min(k, x), v if k < x else y, max(k, x), y if k < x else v) in open_pairs) for x, y in chosen.items())
                key = (-gain, used[(k, v)])
                if best_key is None or key < best_key:
                    best, best_key = v, key
            chosen[k] = best
        for x, y in itertools.combinations(sorted(chosen), 2):
            open_pairs.discard((x, chosen[x], y, chosen[y]))
        for k, v in chosen.items():
            used[(k, v)] += 1
        cases.append({names[k]: chosen[k] for k in range(len(names))})
    return cases


def pairwise_cases() -> list:
    """The all-pairs set with a seed per case."""
    return [dict(c, seed=1000 + n) for n, c in enumerate(all_pairs())]


def case_inputs(tree: FlatTree, c: dict):
    rng = np.random.default_rng(c["seed"])
    return make_inputs(tree, c["algo"], int(c["mode"] == "block"), c["presence"], c["override"], c["fwd_root_ref"], c["width"],
                       c["noise"], rng)


def case_id(c: dict) -> str:
    return "-".join(str(c[k]) for k in ("shape", "algo", "mode", "entry", "width", "presence", "chunk_nodes"))
