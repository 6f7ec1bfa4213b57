"""ctypes mirror of include/panman_b200_host.h: the host-side adaptor (Newick, MSA flow, run-merge into NucMut)."""
import ctypes as C
import os

import numpy as np

from .lib import HERE, load_library

HOST_LIB_PATH = os.path.join(HERE, "libpanman_b200_host.so")


class pmh_nucmut(C.Structure):
    _fields_ = [("nucPosition", C.c_int32), ("nucGapPosition", C.c_int32), ("primaryBlockId", C.c_int32),
                ("secondaryBlockId", C.c_int32), ("mutInfo", C.c_uint8), ("nucs", C.c_uint32)]


class pmh_wire_nuc(C.Structure):
    _fields_ = [("nucPosition", C.c_int32), ("nucGapPosition", C.c_int32), ("nucGapExist", C.c_uint8), ("mutInfo", C.c_uint32)]


class pmh_wire_mutation(C.Structure):
    _fields_ = [("blockId", C.c_int64), ("blockGapExist", C.c_uint8), ("blockMutExist", C.c_uint8), ("blockMutInfo", C.c_uint8),
                ("blockInversion", C.c_uint8), ("nuc_begin", C.c_int64), ("nuc_end", C.c_int64)]


def _wire_of(fn, handle, node):
    """-> [(blockId, blockGapExist, blockMutExist, blockMutInfo, blockInversion, [(nucPosition, nucGapPosition, nucGapExist,
    mutInfo), ...]), ...] = the node's panman.capnp Mutation list as the reference's writer would fill it."""
    fn.restype = C.c_int64
    fn.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.POINTER(pmh_wire_mutation)), C.POINTER(C.POINTER(pmh_wire_nuc))]
    pm, pn = C.POINTER(pmh_wire_mutation)(), C.POINTER(pmh_wire_nuc)()
    k = fn(handle, node, C.byref(pm), C.byref(pn))
    if k < 0:
        raise RuntimeError("wire form unavailable for this node")
    out = []
    for i in range(k):
        m = pm[i]
        out.append((m.blockId, int(m.blockGapExist), int(m.blockMutExist), int(m.blockMutInfo), int(m.blockInversion),
                    [(pn[j].nucPosition, pn[j].nucGapPosition, int(pn[j].nucGapExist), pn[j].mutInfo) for j in range(m.nuc_begin, m.nuc_end)]))
    return out


class pmh_blockmut(C.Structure):
    _fields_ = [("primaryBlockId", C.c_int32), ("secondaryBlockId", C.c_int32), ("blockMutInfo", C.c_uint8), ("inversion", C.c_uint8)]


_hlib = None


def load_host_library():
    global _hlib
    if _hlib is not None:
        return _hlib
    load_library()  # the device library first (rpath $ORIGIN also finds it)
    if not os.path.exists(HOST_LIB_PATH):
        raise RuntimeError(f"{HOST_LIB_PATH} is missing: run __graft_entry__.build()")
    L = C.CDLL(HOST_LIB_PATH)
    vp = C.c_void_p
    L.pmh_tree_from_newick.restype = vp
    L.pmh_tree_from_newick.argtypes = [C.c_char_p, C.c_char_p, C.c_size_t]
    L.pmh_tree_free.argtypes = [vp]
    for f in ("pmh_tree_n_nodes", "pmh_tree_n_leaves", "pmh_tree_root", "pmh_tree_has_polytomy"):
        getattr(L, f).argtypes = [vp]
        getattr(L, f).restype = C.c_int32
    L.pmh_tree_name.argtypes = [vp, C.c_int32]
    L.pmh_tree_name.restype = C.c_char_p
    for f in ("pmh_tree_parent", "pmh_tree_child_offsets", "pmh_tree_child_index", "pmh_tree_leaf_row"):
        getattr(L, f).argtypes = [vp]
        getattr(L, f).restype = C.POINTER(C.c_int32)
    L.pmh_tree_reroot.restype = vp
    L.pmh_tree_reroot.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_size_t]
    L.pmh_build_from_msa.restype = vp
    L.pmh_build_from_msa.argtypes = [vp, C.c_char_p, C.c_size_t, C.c_char_p, C.c_char_p, C.c_int, C.c_char_p, C.c_size_t]
    L.pmh_build_free.argtypes = [vp]
    L.pmh_build_tree.argtypes = [vp]
    L.pmh_build_tree.restype = vp
    L.pmh_build_consensus.argtypes = [vp, C.POINTER(C.c_int64)]
    L.pmh_build_consensus.restype = C.POINTER(C.c_char)
    L.pmh_build_n_nucmut.argtypes = [vp, C.c_int32]
    L.pmh_build_n_nucmut.restype = C.c_int64
    L.pmh_build_nucmut.argtypes = [vp, C.c_int32]
    L.pmh_build_nucmut.restype = C.POINTER(pmh_nucmut)
    L.pmh_build_n_tuples.argtypes = [vp]
    L.pmh_build_n_tuples.restype = C.c_int64
    L.pmh_build_tuple_offsets.argtypes = [vp]
    L.pmh_build_tuple_offsets.restype = C.POINTER(C.c_int64)
    L.pmh_build_tuple_pos.argtypes = [vp]
    L.pmh_build_tuple_pos.restype = C.POINTER(C.c_int32)
    L.pmh_build_tuple_type_code.argtypes = [vp]
    L.pmh_build_tuple_type_code.restype = C.POINTER(C.c_uint8)
    L.pmh_build_seconds.argtypes = [vp]
    L.pmh_build_seconds.restype = C.POINTER(C.c_double)
    _hlib = L
    return L


class HostTree:
    """Result of the C++ Newick parser (reference src/panman.cpp:310-450 conventions)."""

    def __init__(self, handle, owned=True):
        self.L = load_host_library()
        self.h = handle
        self.owned = owned
        n = self.L.pmh_tree_n_nodes(handle)
        self.names = [self.L.pmh_tree_name(handle, v).decode() for v in range(n)]
        self.parent = np.ctypeslib.as_array(self.L.pmh_tree_parent(handle), (n,)).copy()
        self.child_off = np.ctypeslib.as_array(self.L.pmh_tree_child_offsets(handle), (n + 1,)).copy()
        self.child_idx = np.ctypeslib.as_array(self.L.pmh_tree_child_index(handle), (max(n - 1, 1),))[:n - 1].copy()
        self.leaf_row = np.ctypeslib.as_array(self.L.pmh_tree_leaf_row(handle), (n,)).copy()
        self.root = int(self.L.pmh_tree_root(handle))
        self.n_nodes = n
        self.n_leaves = int(self.L.pmh_tree_n_leaves(handle))
        self.polytomy = bool(self.L.pmh_tree_has_polytomy(handle))
        if owned:
            self.L.pmh_tree_free(handle)
            self.h = None


def parse_newick(newick: str, keep: bool = False) -> HostTree:
    L = load_host_library()
    err = C.create_string_buffer(256)
    h = L.pmh_tree_from_newick(newick.encode(), err, 256)
    if not h:
        raise ValueError(err.value.decode())
    return HostTree(h, owned=not keep)


def reroot_newick(newick: str, leaf_name: str) -> HostTree:
    """pmh_tree_reroot (reference Tree::transform, src/panman.cpp:5831-5906) on the tree of `newick`."""
    L = load_host_library()
    err = C.create_string_buffer(256)
    h = L.pmh_tree_from_newick(newick.encode(), err, 256)
    if not h:
        raise ValueError(err.value.decode())
    h2 = L.pmh_tree_reroot(h, leaf_name.encode(), err, 256)
    L.pmh_tree_free(h)
    if not h2:
        raise ValueError(err.value.decode())
    return HostTree(h2)


class MsaBuild:
    """panmanUtils -M msa.fa -N tree.nwk [--reference id] [--low-mem-mode] through libpanman_b200. The build keeps its handle
    until close(): reroot() works on it."""

    def __init__(self, ctx, fasta: bytes, newick: str, reference: str = "", low_mem_mode: bool = False):
        """ctx: a Context (one GPU) or a single-process Group (pmh_msa_run_group: column ranges over the GPUs of the box)."""
        from .api import Group

        L = load_host_library()
        self.L = L
        err = C.create_string_buffer(512)
        if isinstance(ctx, Group):
            vp = C.c_void_p
            L.pmh_msa_prepare.restype = vp
            L.pmh_msa_prepare.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_char_p, C.c_int, C.c_char_p, C.c_size_t]
            L.pmh_msa_run_group.argtypes = [vp, vp, C.c_char_p, C.c_size_t]
            h = L.pmh_msa_prepare(fasta, len(fasta), newick.encode(), reference.encode(), int(low_mem_mode), err, 512)
            if h and L.pmh_msa_run_group(ctx.h, h, err, 512) != 0:
                L.pmh_build_free(h)
                h = None
        else:
            h = L.pmh_build_from_msa(ctx.h, fasta, len(fasta), newick.encode(), reference.encode(), int(low_mem_mode), err, 512)
        if not h:
            raise RuntimeError(err.value.decode())
        self.h = h
        n = C.c_int64()
        p = L.pmh_build_consensus(h, C.byref(n))
        self.consensus = C.string_at(p, n.value)
        self._refresh()

    def _refresh(self):
        """tree, nucmut, wire, tuple arrays and seconds from the handle (after the build and after every reroot)."""
        L, h = self.L, self.h
        self.tree = HostTree(L.pmh_build_tree(h), owned=False)
        self.nucmut = []
        for v in range(self.tree.n_nodes):
            k = L.pmh_build_n_nucmut(h, v)
            arr = L.pmh_build_nucmut(h, v)
            self.nucmut.append([(arr[i].nucPosition, arr[i].nucGapPosition, arr[i].primaryBlockId, arr[i].secondaryBlockId,
                                 arr[i].mutInfo, arr[i].nucs) for i in range(k)])
        self.wire = [_wire_of(L.pmh_build_wire, h, v) for v in range(self.tree.n_nodes)]
        nt = L.pmh_build_n_tuples(h)
        N = self.tree.n_nodes
        self.tuple_offsets = np.ctypeslib.as_array(L.pmh_build_tuple_offsets(h), (N + 1,)).copy()
        self.tuple_pos = np.ctypeslib.as_array(L.pmh_build_tuple_pos(h), (max(nt, 1),))[:nt].copy()
        self.tuple_type_code = np.ctypeslib.as_array(L.pmh_build_tuple_type_code(h), (max(nt, 1),))[:nt].copy()
        self.seconds = list(np.ctypeslib.as_array(L.pmh_build_seconds(h), (4,)))

    def reroot(self, ctx, leaf_name: str):
        """Tree::reroot (reference src/reroot.cpp) on the built PanMAT (pmh_msa_reroot), on one GPU: the mutation lists are
        replayed into the leaf sequences on the device and every column is inferred again on the re-rooted tree. The
        attributes then describe the re-rooted tree."""
        from .api import Context, PanmanError

        if not isinstance(ctx, Context):
            raise TypeError("reroot runs on one GPU: pass a Context")
        if not self.h:
            raise RuntimeError("the build was closed")
        self.L.pmh_msa_reroot.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_char_p, C.c_size_t]
        err = C.create_string_buffer(512)
        rc = self.L.pmh_msa_reroot(ctx.h, self.h, leaf_name.encode(), err, 512)
        if rc:
            raise PanmanError(rc, err.value.decode())
        self._refresh()

    def close(self):
        if getattr(self, "h", None):
            self.L.pmh_build_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MsaPrepared:
    """pmh_msa_prepare: the host-only half of the -M flow (reader, consensus, all-gap column removal, packing)."""

    def __init__(self, fasta: bytes, newick: str, reference: str = "", low_mem_mode: bool = False):
        L = load_host_library()
        vp = C.c_void_p
        L.pmh_msa_prepare.restype = vp
        L.pmh_msa_prepare.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_char_p, C.c_int, C.c_char_p, C.c_size_t]
        L.pmh_build_n_cols.argtypes = [vp]
        L.pmh_build_n_cols.restype = C.c_int64
        L.pmh_build_codes4.argtypes = [vp, C.POINTER(C.c_int64)]
        L.pmh_build_codes4.restype = C.POINTER(C.c_uint8)
        for f, t in (("present", C.c_uint8), ("parent_code", C.c_uint8), ("root_override", C.c_int8), ("fwd_root_ref", C.c_int8)):
            getattr(L, "pmh_build_" + f).argtypes = [vp]
            getattr(L, "pmh_build_" + f).restype = C.POINTER(t)
        err = C.create_string_buffer(512)
        h = L.pmh_msa_prepare(fasta, len(fasta), newick.encode(), reference.encode(), int(low_mem_mode), err, 512)
        if not h:
            raise RuntimeError(err.value.decode())
        self.tree = HostTree(L.pmh_build_tree(h), owned=False)
        n = C.c_int64()
        p = L.pmh_build_consensus(h, C.byref(n))
        self.consensus = C.string_at(p, n.value)
        self.n_cols = int(L.pmh_build_n_cols(h))
        nl, nc = self.tree.n_leaves, self.n_cols
        stride = C.c_int64()
        cp = L.pmh_build_codes4(h, C.byref(stride))
        if nc and cp:
            c4 = np.ctypeslib.as_array(cp, (nl, stride.value)).copy()
            codes = np.empty((nl, 2 * stride.value), np.uint8)
            codes[:, 0::2] = c4 & 15
            codes[:, 1::2] = c4 >> 4
            self.codes = codes[:, :nc]
        else:
            self.codes = np.zeros((nl, 0), np.uint8)

        def arr(name, count):
            q = getattr(L, "pmh_build_" + name)(h)
            return np.ctypeslib.as_array(q, (count,)).copy() if q and count else None

        self.present = arr("present", nl)
        self.parent_code = arr("parent_code", nc)
        self.root_override = arr("root_override", nc)
        self.fwd_root_ref = arr("fwd_root_ref", nc)
        L.pmh_build_free(h)


class PanGraphBuild:
    """panmanUtils -P pangraph.json -N tree.nwk [--reference id] through libpanman_b200 (include/panman_b200_host.h):
    load() builds the per-block column batches on the host, run() executes the block-level pass and one pass per block."""

    def __init__(self, json_text: bytes, newick: str, reference: str = ""):
        L = load_host_library()
        vp = C.c_void_p
        L.pmh_pangraph_load.restype = vp
        L.pmh_pangraph_load.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_char_p, C.c_char_p, C.c_size_t]
        L.pmh_pangraph_free.argtypes = [vp]
        L.pmh_pangraph_tree.argtypes = [vp]
        L.pmh_pangraph_tree.restype = vp
        L.pmh_pangraph_n_blocks.argtypes = [vp]
        L.pmh_pangraph_n_blocks.restype = C.c_int32
        L.pmh_pangraph_block_id.argtypes = [vp, C.c_int32]
        L.pmh_pangraph_block_id.restype = C.c_char_p
        L.pmh_pangraph_block_states.argtypes = [vp]
        L.pmh_pangraph_block_states.restype = C.POINTER(C.c_uint8)
        L.pmh_pangraph_n_cols.argtypes = [vp, C.c_int32]
        L.pmh_pangraph_n_cols.restype = C.c_int64
        L.pmh_pangraph_codes4.argtypes = [vp, C.c_int32, C.POINTER(C.c_int64)]
        L.pmh_pangraph_codes4.restype = C.POINTER(C.c_uint8)
        for f, t in (("present", C.c_uint8), ("parent_code", C.c_uint8), ("root_override", C.c_int8), ("col_pos", C.c_int32),
                     ("col_gap", C.c_int32)):
            getattr(L, "pmh_pangraph_" + f).argtypes = [vp, C.c_int32]
            getattr(L, "pmh_pangraph_" + f).restype = C.POINTER(t)
        L.pmh_pangraph_run.argtypes = [vp, vp, C.c_int, C.c_char_p, C.c_size_t]
        L.pmh_pangraph_result.argtypes = [vp, C.c_int32, C.POINTER(C.POINTER(C.c_int64)), C.POINTER(C.POINTER(C.c_int32)),
                                          C.POINTER(C.POINTER(C.c_uint8))]
        L.pmh_pangraph_result.restype = C.c_int64
        self.L = L
        err = C.create_string_buffer(512)
        self.h = L.pmh_pangraph_load(json_text, len(json_text), newick.encode(), reference.encode(), err, 512)
        if not self.h:
            raise ValueError(err.value.decode())
        self.tree = HostTree(L.pmh_pangraph_tree(self.h), owned=False)
        self.n_blocks = int(L.pmh_pangraph_n_blocks(self.h))
        n_leaves = self.tree.n_leaves
        self.block_ids = [L.pmh_pangraph_block_id(self.h, b).decode() for b in range(self.n_blocks)]
        self.block_states = np.ctypeslib.as_array(L.pmh_pangraph_block_states(self.h), (n_leaves, max(self.n_blocks, 1)))[:, :self.n_blocks].copy()
        L.pmh_pangraph_rotation_index.argtypes = [vp]
        L.pmh_pangraph_rotation_index.restype = C.POINTER(C.c_int32)
        self.rotation_index = np.ctypeslib.as_array(L.pmh_pangraph_rotation_index(self.h), (max(n_leaves, 1),))[:n_leaves].copy()
        L.pmh_pangraph_block_override.argtypes = [vp]
        L.pmh_pangraph_block_override.restype = C.POINTER(C.c_int8)
        bo = L.pmh_pangraph_block_override(self.h)
        self.block_override = np.ctypeslib.as_array(bo, (self.n_blocks,)).copy() if bo and self.n_blocks else None
        self.batches = []
        for b in range(self.n_blocks):
            n = int(L.pmh_pangraph_n_cols(self.h, b))
            stride = C.c_int64()
            p = L.pmh_pangraph_codes4(self.h, b, C.byref(stride))
            c4 = np.ctypeslib.as_array(p, (n_leaves, stride.value)).copy()
            codes = np.empty((n_leaves, 2 * stride.value), np.uint8)
            codes[:, 0::2] = c4 & 15
            codes[:, 1::2] = c4 >> 4

            def arr(name, count):
                return np.ctypeslib.as_array(getattr(L, "pmh_pangraph_" + name)(self.h, b), (count,)).copy()

            self.batches.append(dict(id=self.block_ids[b], codes=codes[:, :n], present=arr("present", n_leaves), parent_code=arr("parent_code", n),
                                     root_override=arr("root_override", n), col_j=arr("col_pos", n), col_k=arr("col_gap", n)))

    def run(self, ctx, algo: int):
        """Returns [MutLists-like (node_offsets, pos, type_code)] for the block-level pass followed by every block."""
        err = C.create_string_buffer(512)
        rc = self.L.pmh_pangraph_run(ctx.h, self.h, int(algo), err, 512)
        if rc:
            raise RuntimeError(err.value.decode())
        N = self.tree.n_nodes
        out = []
        for b in range(-1, self.n_blocks):
            po, pp, pt = C.POINTER(C.c_int64)(), C.POINTER(C.c_int32)(), C.POINTER(C.c_uint8)()
            n = int(self.L.pmh_pangraph_result(self.h, b, C.byref(po), C.byref(pp), C.byref(pt)))
            off = np.ctypeslib.as_array(po, (N + 1,)).copy()
            pos = np.ctypeslib.as_array(pp, (max(n, 1),))[:n].copy()
            tc = np.ctypeslib.as_array(pt, (max(n, 1),))[:n].copy()
            out.append((off, pos, tc))
        return out

    def _results(self):
        N = self.tree.n_nodes
        out = []
        for b in range(-1, self.n_blocks):
            po, pp, pt = C.POINTER(C.c_int64)(), C.POINTER(C.c_int32)(), C.POINTER(C.c_uint8)()
            n = int(self.L.pmh_pangraph_result(self.h, b, C.byref(po), C.byref(pp), C.byref(pt)))
            off = np.ctypeslib.as_array(po, (N + 1,)).copy()
            pos = np.ctypeslib.as_array(pp, (max(n, 1),))[:n].copy()
            tc = np.ctypeslib.as_array(pt, (max(n, 1),))[:n].copy()
            out.append((off, pos, tc))
        return out

    def reroot(self, ctx, leaf_name: str):
        """Tree::reroot (reference src/reroot.cpp) on the built graph; self.tree becomes the re-rooted tree. Returns the lists
        of the block-level pass followed by every block, as run() does."""
        self.L.pmh_pangraph_reroot.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_char_p, C.c_size_t]
        err = C.create_string_buffer(512)
        rc = self.L.pmh_pangraph_reroot(ctx.h, self.h, leaf_name.encode(), err, 512)
        if rc:
            raise RuntimeError(err.value.decode())
        self.tree = HostTree(self.L.pmh_pangraph_tree(self.h), owned=False)
        return self._results()

    def wire(self):
        """Per node, the Mutation list the reference's writer would store (pmh_pangraph_wire)."""
        return [_wire_of(self.L.pmh_pangraph_wire, self.h, v) for v in range(self.tree.n_nodes)]

    def blockmut(self):
        """Node::blockMutation per node: lists of (primaryBlockId, secondaryBlockId, blockMutInfo, inversion)."""
        self.L.pmh_pangraph_n_blockmut.argtypes = [C.c_void_p, C.c_int32]
        self.L.pmh_pangraph_n_blockmut.restype = C.c_int64
        self.L.pmh_pangraph_blockmut.argtypes = [C.c_void_p, C.c_int32]
        self.L.pmh_pangraph_blockmut.restype = C.POINTER(pmh_blockmut)
        out = []
        for v in range(self.tree.n_nodes):
            k = self.L.pmh_pangraph_n_blockmut(self.h, v)
            arr = self.L.pmh_pangraph_blockmut(self.h, v)
            out.append([(arr[i].primaryBlockId, arr[i].secondaryBlockId, int(arr[i].blockMutInfo), int(arr[i].inversion)) for i in range(k)])
        return out

    def nucmut(self):
        """Node::nucMutation per node after run(): lists of (nucPosition, nucGapPosition, primaryBlockId, secondaryBlockId,
        mutInfo, nucs)."""
        self.L.pmh_pangraph_n_nucmut.argtypes = [C.c_void_p, C.c_int32]
        self.L.pmh_pangraph_n_nucmut.restype = C.c_int64
        self.L.pmh_pangraph_nucmut.argtypes = [C.c_void_p, C.c_int32]
        self.L.pmh_pangraph_nucmut.restype = C.POINTER(pmh_nucmut)
        out = []
        for v in range(self.tree.n_nodes):
            k = self.L.pmh_pangraph_n_nucmut(self.h, v)
            arr = self.L.pmh_pangraph_nucmut(self.h, v)
            out.append([(arr[i].nucPosition, arr[i].nucGapPosition, arr[i].primaryBlockId, arr[i].secondaryBlockId, arr[i].mutInfo,
                         arr[i].nucs) for i in range(k)])
        return out

    def close(self):
        if self.h:
            self.L.pmh_pangraph_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
