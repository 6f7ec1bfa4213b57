"""ctypes mirror of include/panman_b200.h (same names, argument meaning and error behaviour)."""
import ctypes as C
from dataclasses import dataclass

import numpy as np

from .lib import GROUP_HANDLE_BYTES, load_library, pmb_nucmut_result, pmb_result, pmb_runs_info, pmb_timings

ALGO_FITCH, ALGO_SANKOFF = 0, 1
FLAG_WANT_STATES, FLAG_BLOCK_MODE = 1, 2


class PanmanError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libpanman_b200 error {code}: {msg}")
        self.code = code


@dataclass
class Result:
    node_offsets: np.ndarray  # int64 n_nodes+1
    pos: np.ndarray  # int32
    type_code: np.ndarray  # uint8 (type<<4)|code
    states: np.ndarray = None  # uint8 n_nodes x n_cols, 0xFF = none

    @property
    def n_mut(self):
        return int(self.node_offsets[-1]) if len(self.node_offsets) else 0


@dataclass
class Timings:
    forward_ms: float
    backward_ms: float
    compact_ms: float
    total_ms: float
    n_launches: int
    n_levels: int


def pack_nibbles(codes: np.ndarray) -> np.ndarray:
    """(n_rows, n_cols) uint8 codes -> (n_rows, ceil(n_cols/2)) bytes; column c is the low nibble of byte c//2 when c is
    even, the high nibble when odd (the pmb_run_nuc convention)."""
    codes = np.ascontiguousarray(codes, np.uint8)
    n_rows, n_cols = codes.shape
    if n_cols % 2:
        codes = np.concatenate([codes, np.zeros((n_rows, 1), np.uint8)], 1)
    return np.ascontiguousarray((codes[:, 0::2] & 15) | ((codes[:, 1::2] & 15) << 4))


def _ptr(x):
    """numpy array / torch tensor (host or device) / int / None -> raw address."""
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if isinstance(x, np.ndarray):
        assert x.flags["C_CONTIGUOUS"]
        return x.ctypes.data
    return x.data_ptr()  # torch tensor


def _nucmut_arrays(r: pmb_nucmut_result):
    n, N = int(r.n), int(r.n_nodes)

    def view(addr, ctype, count, dtype):
        if count == 0 or not addr:
            return np.zeros(0, dtype)
        return np.ctypeslib.as_array(C.cast(addr, C.POINTER(ctype)), (count,)).astype(dtype, copy=True)

    return (view(r.node_offsets, C.c_int64, N + 1, np.int64), view(r.nuc_position, C.c_int32, n, np.int32),
            view(r.mut_info, C.c_uint8, n, np.uint8), view(r.nucs, C.c_uint32, n, np.uint32),
            view(r.mut_info_wire, C.c_uint32, n, np.uint32))


def column_range(world: int, n_cols: int, rank: int):
    """pmb_group_column_range: the contiguous, 1024-aligned column range of `rank` (needs no device)."""
    a, b = C.c_int64(), C.c_int64()
    rc = load_library().pmb_group_column_range(int(world), int(n_cols), int(rank), C.byref(a), C.byref(b))
    if rc != 0:
        raise PanmanError(rc, "pmb_group_column_range: bad arguments")
    return int(a.value), int(b.value)


class Runs:
    """pmb_runs: the clade-run encoding of a HOST nibble matrix for one tree (pmb_runs_encode). Needs no device."""

    def __init__(self, n_nodes, root, child_off, child_idx, leaf_row, n_cols, codes4, row_stride, parent_code, n_threads: int = 0):
        self.L = load_library()
        co = np.ascontiguousarray(child_off, np.int32)
        ci = np.ascontiguousarray(child_idx, np.int32)
        lr = np.ascontiguousarray(leaf_row, np.int32)
        n_rows = int((lr >= 0).sum())
        self.h = C.c_void_p()
        rc = self.L.pmb_runs_encode(int(n_nodes), int(root), _ptr(co), _ptr(ci), _ptr(lr), int(n_cols), n_rows, _ptr(codes4), int(row_stride),
                                    _ptr(parent_code), int(n_threads), C.byref(self.h))
        if rc != 0:
            self.h = None
            raise PanmanError(rc, "pmb_runs_encode: bad arguments" if rc == -1 else "pmb_runs_encode failed")
        self.info = pmb_runs_info()
        self.L.pmb_runs_describe(self.h, C.byref(self.info))
        self._tree = (int(n_nodes), int(root), co, ci, lr)

    @classmethod
    def of_tree(cls, tree, n_cols, codes4, parent_code, n_threads: int = 0):
        return cls(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row, n_cols, codes4, codes4.shape[1], parent_code,
                   n_threads)

    n_cols = property(lambda self: int(self.info.n_cols))
    n_rows = property(lambda self: int(self.info.n_rows))
    n_events = property(lambda self: int(self.info.n_events))
    nbytes = property(lambda self: int(self.info.bytes))

    def events(self):
        n = self.n_events
        return np.ctypeslib.as_array(C.cast(self.info.events, C.POINTER(C.c_uint32)), (max(n, 1),))[:n]

    def item_offsets(self):
        n = self.info.n_tiles * self.info.n_segments + 1
        return np.ctypeslib.as_array(C.cast(self.info.item_offsets, C.POINTER(C.c_int64)), (n,))

    def dfs_rows(self):
        """The caller's leaf rows in depth-first order of the tree (children in Newick order): the order of the encoding."""
        _, root, co, ci, lr = self._tree
        out, stack = [], [root]
        while stack:
            v = stack.pop()
            a, z = int(co[v]), int(co[v + 1])
            if a == z:
                out.append(int(lr[v]))
            else:
                stack.extend(int(c) for c in ci[a:z][::-1])
        return np.asarray(out, np.int64)

    def decode(self, parent_code) -> np.ndarray:
        """The (n_rows, n_cols) code matrix back from the events, the way expand_runs_kernel rebuilds it (test helper)."""
        I = self.info
        ev, off, order = self.events(), self.item_offsets(), self.dfs_rows()
        pc = np.zeros(I.n_tiles * 1024, np.uint8)
        pc[:I.n_cols] = np.asarray(parent_code, np.uint8)[:I.n_cols] & 15
        out = np.zeros((I.n_rows, I.n_tiles * 1024), np.uint8)
        for t in range(I.n_tiles):
            base = pc[t * 1024:(t + 1) * 1024]
            for sg in range(I.n_segments):
                e = ev[off[t * I.n_segments + sg]:off[t * I.n_segments + sg + 1]]
                r0 = sg * I.seg_rows
                nr = min(I.seg_rows, I.n_rows - r0)
                rows, cols, x = (e >> 14).astype(np.int64), ((e >> 4) & 1023).astype(np.int64), (e & 15).astype(np.uint8)
                assert bool((np.diff(rows) >= 0).all()) and (len(rows) == 0 or rows[-1] < nr)
                delta = np.zeros((nr, 1024), np.uint8)
                np.bitwise_xor.at(delta, (rows, cols), x)
                out[order[r0:r0 + nr], t * 1024:(t + 1) * 1024] = np.bitwise_xor.accumulate(delta, 0) ^ base[None, :]
        return out[:, :I.n_cols]

    def close(self):
        if getattr(self, "h", None):
            self.L.pmb_runs_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Context:
    """One context per CUDA device / rank (pmb_ctx). Not thread-safe."""

    def __init__(self, device: int = 0, _borrowed=None):
        self.L = load_library()
        self._keep = []
        self._owned = _borrowed is None
        if _borrowed is not None:  # a context owned by a Group
            self.h = C.c_void_p(_borrowed)
            return
        self.h = C.c_void_p()
        rc = self.L.pmb_create(C.byref(self.h), device)
        if rc != 0:
            msg = self.L.pmb_last_error(self.h).decode() if self.h else "pmb_create failed"
            if self.h:
                self.L.pmb_destroy(self.h)
                self.h = None
            raise PanmanError(rc, msg)
        self._keep = []

    def close(self):
        if getattr(self, "h", None):
            if self._owned:
                self.L.pmb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise PanmanError(rc, self.L.pmb_last_error(self.h).decode())

    def set_option(self, key: str, value: int):
        self._check(self.L.pmb_set_option(self.h, key.encode(), int(value)))

    def set_tree(self, n_nodes, root, child_off, child_idx, leaf_row):
        co = np.ascontiguousarray(child_off, np.int32)
        ci = np.ascontiguousarray(child_idx, np.int32)
        lr = np.ascontiguousarray(leaf_row, np.int32)
        self.n_nodes = int(n_nodes)
        self._check(self.L.pmb_set_tree(self.h, int(n_nodes), int(root), _ptr(co), _ptr(ci), _ptr(lr)))

    def upload(self, n_cols, n_rows, codes4, row_stride, parent_code, root_override=None, fwd_root_ref=None, leaf_present=None,
               col_base=0):
        self._check(self.L.pmb_upload_nuc(self.h, int(n_cols), int(n_rows), _ptr(codes4), int(row_stride), _ptr(leaf_present),
                                          _ptr(parent_code), _ptr(root_override), _ptr(fwd_root_ref), int(col_base)))

    def upload_replay(self, old_tree, piece_offsets, nuc_position, mut_info, nucs, n_cols, parent_code, root_leaf_row=-1):
        """pmb_upload_replay: the leaf codes of the context's tree rebuilt on the device from a PanMAT's NucMut pieces, built on
        `old_tree` (n_nodes, root, child_off, child_idx, leaf_row attributes), node-major over its node ids. root_leaf_row >= 0
        forces the root to that leaf's replayed codes."""
        co = np.ascontiguousarray(old_tree.child_off, np.int32)
        ci = np.ascontiguousarray(old_tree.child_idx, np.int32)
        lr = np.ascontiguousarray(old_tree.leaf_row, np.int32)
        po = np.ascontiguousarray(piece_offsets, np.int64)
        pos = np.ascontiguousarray(nuc_position, np.int32)
        info = np.ascontiguousarray(mut_info, np.uint8)
        nu = np.ascontiguousarray(nucs, np.uint32)
        pc = np.ascontiguousarray(parent_code, np.uint8)
        self._check(self.L.pmb_upload_replay(self.h, int(old_tree.n_nodes), int(old_tree.root), _ptr(co), _ptr(ci), _ptr(lr), _ptr(po),
                                             _ptr(pos), _ptr(info), _ptr(nu), int(n_cols), _ptr(pc), int(root_leaf_row)))

    def run_resident(self, algo=ALGO_FITCH, flags=0) -> Timings:
        self._check(self.L.pmb_run_resident(self.h, int(algo), int(flags)))
        return self.timings()

    def run_resident_async(self, algo=ALGO_FITCH, flags=0):
        self._check(self.L.pmb_run_resident_async(self.h, int(algo), int(flags)))

    def join(self):
        """pmb_join: pmb_stream now follows every pass enqueued so far (an event recorded on it marks their end)."""
        self._check(self.L.pmb_join(self.h))

    def wait(self) -> Timings:
        self._check(self.L.pmb_wait(self.h))
        return self.timings()

    def timings(self) -> Timings:
        t = pmb_timings()
        self._check(self.L.pmb_last_timings(self.h, C.byref(t)))
        return Timings(t.forward_ms, t.backward_ms, t.compact_ms, t.total_ms, t.n_launches, t.n_levels)

    def algorithmic_bytes(self, algo=ALGO_FITCH) -> int:
        return int(self.L.pmb_algorithmic_bytes(self.h, int(algo)))

    def _result(self, r: pmb_result, copy=True) -> Result:
        n, N = int(r.n_mut), int(r.n_nodes)

        def view(addr, ctype, count, dtype):
            if count == 0 or not addr:
                return np.empty(0, dtype)
            a = np.ctypeslib.as_array(C.cast(addr, C.POINTER(ctype)), (count,))
            return a.copy() if copy else a

        off = view(r.node_offsets, C.c_int64, N + 1, np.int64)
        pos = view(r.pos, C.c_int32, n, np.int32)
        tc = view(r.type_code, C.c_uint8, n, np.uint8)
        states = None
        if r.states:
            states = view(r.states, C.c_uint8, N * int(r.n_cols), np.uint8).reshape(N, int(r.n_cols))
        return Result(off, pos, tc, states)

    def download(self, copy=True) -> Result:
        r = pmb_result()
        self._check(self.L.pmb_download(self.h, C.byref(r)))
        return self._result(r, copy)

    def result_device(self) -> pmb_result:
        r = pmb_result()
        self._check(self.L.pmb_result_device(self.h, C.byref(r)))
        return r

    # column-range shards (multi-GPU): pack -> one collective by the caller -> merge on the receiving rank
    def stream_handle(self) -> int:
        return int(self.L.pmb_stream(self.h) or 0)

    def result_stream_handle(self) -> int:
        return int(self.L.pmb_result_stream(self.h) or 0)

    def packed_bytes(self, capacity: int) -> int:
        return int(self.L.pmb_packed_bytes(self.n_nodes, int(capacity)))

    def pack_result(self, d_packed, capacity: int, stream=None):
        self._check(self.L.pmb_pack_result(self.h, _ptr(d_packed), int(capacity), stream))

    def merge_packed(self, n_shards: int, d_packed, capacity: int, stream=None) -> pmb_result:
        r = pmb_result()
        self._check(self.L.pmb_merge_packed(self.h, int(n_shards), _ptr(d_packed), int(capacity), stream, C.byref(r)))
        return r

    def merge_status(self):
        self._check(self.L.pmb_merge_status(self.h))

    def set_column_breaks(self, col_break):
        """pmb_set_column_breaks: n_cols bytes (host or device), 1 = a run never continues INTO this column; None clears."""
        self._check(self.L.pmb_set_column_breaks(self.h, _ptr(col_break)))

    def merge_runs(self, source: int = 0):
        """Greedy <= 6 run-merge of the per-node lists into NucMut fields on the device (pmb_merge_runs); returns host arrays
        (node_offsets int64[N+1], nuc_position int32, mut_info uint8, nucs uint32, mut_info_wire uint32 = the capnp writer's
        form, src/panman.cpp:2876). source 1 = the last merge_packed."""
        r = pmb_nucmut_result()
        self._check(self.L.pmb_merge_runs(self.h, int(source), 1, C.byref(r)))
        return _nucmut_arrays(r)

    def run_nuc(self, algo, n_cols, n_rows, codes4, row_stride, parent_code, root_override=None, fwd_root_ref=None,
                leaf_present=None, col_base=0, flags=0, copy=True) -> Result:
        r = pmb_result()
        self._check(self.L.pmb_run_nuc(self.h, int(algo), int(n_cols), int(n_rows), _ptr(codes4), int(row_stride),
                                       _ptr(leaf_present), _ptr(parent_code), _ptr(root_override), _ptr(fwd_root_ref),
                                       int(col_base), int(flags), C.byref(r)))
        return self._result(r, copy)

    def upload_runs(self, runs: Runs, parent_code, root_override=None, fwd_root_ref=None, leaf_present=None, col_begin=0, n_cols=None,
                    col_base=0, sync=True):
        n = runs.n_cols - int(col_begin) if n_cols is None else int(n_cols)
        f = self.L.pmb_upload_runs if sync else self.L.pmb_upload_runs_async
        self._check(f(self.h, runs.h, int(col_begin), n, _ptr(leaf_present), _ptr(parent_code), _ptr(root_override), _ptr(fwd_root_ref),
                      int(col_base)))

    def run_runs(self, algo, runs: Runs, parent_code, root_override=None, fwd_root_ref=None, leaf_present=None, col_base=0, flags=0,
                 copy=True) -> Result:
        r = pmb_result()
        self._check(self.L.pmb_run_runs(self.h, int(algo), runs.h, _ptr(leaf_present), _ptr(parent_code), _ptr(root_override),
                                        _ptr(fwd_root_ref), int(col_base), int(flags), C.byref(r)))
        return self._result(r, copy)

    # convenience for tests: unpacked codes, numpy everywhere
    def run_codes(self, tree, algo, codes, parent_code, root_override=None, fwd_root_ref=None, leaf_present=None, block_mode=0,
                  want_states=False, col_base=0) -> Result:
        codes4 = pack_nibbles(codes)
        n_rows, n_cols = codes.shape
        pc = np.ascontiguousarray(parent_code, np.uint8)
        ro = None if root_override is None else np.ascontiguousarray(root_override, np.int8)
        fr = None if fwd_root_ref is None else np.ascontiguousarray(fwd_root_ref, np.int8)
        lp = None if leaf_present is None else np.ascontiguousarray(leaf_present, np.uint8)
        flags = (FLAG_WANT_STATES if want_states else 0) | (FLAG_BLOCK_MODE if block_mode else 0)
        return self.run_nuc(algo, n_cols, n_rows, codes4, codes4.shape[1], pc, ro, fr, lp, col_base, flags)


class Group:
    """pmb_group: one column-sharded pass over several GPUs. Single process: Group([0, 1, ...]). One process per GPU
    (torchrun): Group([local_device], rank_base=rank, world=world), then reserve(), export() -> all-gather -> connect()
    (panman_b200.distributed.connect_group does the exchange over torch.distributed)."""

    def __init__(self, devices, rank_base: int = 0, world: int = None):
        self.L = load_library()
        devices = [int(d) for d in devices]
        self.n_local = len(devices)
        self.rank_base = int(rank_base)
        self.world = int(world) if world is not None else self.n_local
        self.h = C.c_void_p()
        arr = (C.c_int * self.n_local)(*devices)
        rc = self.L.pmb_group_create(C.byref(self.h), arr, self.n_local, self.rank_base, self.world)
        if rc != 0:
            msg = self.L.pmb_group_last_error(self.h).decode() if self.h else "pmb_group_create: bad arguments"
            if self.h:
                self.L.pmb_group_destroy(self.h)
                self.h = None
            raise PanmanError(rc, msg)
        self.n_nodes = 0

    def close(self):
        if getattr(self, "h", None):
            self.L.pmb_group_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise PanmanError(rc, self.L.pmb_group_last_error(self.h).decode())

    def ctx(self, local_index: int = 0) -> Context:
        return Context(_borrowed=self.L.pmb_group_ctx(self.h, int(local_index)))

    def column_range(self, n_cols: int, rank: int):
        return column_range(self.world, n_cols, rank)

    def set_tree(self, n_nodes, root, child_off, child_idx, leaf_row):
        co = np.ascontiguousarray(child_off, np.int32)
        ci = np.ascontiguousarray(child_idx, np.int32)
        lr = np.ascontiguousarray(leaf_row, np.int32)
        self.n_nodes = int(n_nodes)
        self._check(self.L.pmb_group_set_tree(self.h, int(n_nodes), int(root), _ptr(co), _ptr(ci), _ptr(lr)))

    def reserve(self, capacity: int):
        self._check(self.L.pmb_group_reserve(self.h, int(capacity)))

    def export(self) -> bytes:
        buf = C.create_string_buffer(self.n_local * GROUP_HANDLE_BYTES)
        self._check(self.L.pmb_group_export(self.h, buf))
        return buf.raw

    def connect(self, all_handles: bytes):
        assert len(all_handles) == self.world * GROUP_HANDLE_BYTES
        self._check(self.L.pmb_group_connect(self.h, C.create_string_buffer(all_handles, len(all_handles))))

    def upload(self, n_cols, n_rows, codes4, row_stride, parent_code, root_override=None, fwd_root_ref=None, leaf_present=None):
        self._check(self.L.pmb_group_upload_nuc(self.h, int(n_cols), int(n_rows), _ptr(codes4), int(row_stride), _ptr(leaf_present),
                                                _ptr(parent_code), _ptr(root_override), _ptr(fwd_root_ref)))

    def upload_shard(self, local_index, n_cols_total, n_rows, codes4, row_stride, parent_code, root_override=None, fwd_root_ref=None,
                     leaf_present=None):
        self._check(self.L.pmb_group_upload_shard(self.h, int(local_index), int(n_cols_total), int(n_rows), _ptr(codes4),
                                                  int(row_stride), _ptr(leaf_present), _ptr(parent_code), _ptr(root_override),
                                                  _ptr(fwd_root_ref)))

    def upload_runs(self, runs: Runs, parent_code, root_override=None, fwd_root_ref=None, leaf_present=None):
        self._check(self.L.pmb_group_upload_runs(self.h, runs.h, _ptr(leaf_present), _ptr(parent_code), _ptr(root_override),
                                                 _ptr(fwd_root_ref)))

    def upload_shard_runs(self, local_index, n_cols_total, runs: Runs, parent_code, root_override=None, fwd_root_ref=None,
                          leaf_present=None):
        self._check(self.L.pmb_group_upload_shard_runs(self.h, int(local_index), int(n_cols_total), runs.h, _ptr(leaf_present),
                                                       _ptr(parent_code), _ptr(root_override), _ptr(fwd_root_ref)))

    def run_runs(self, algo, runs: Runs, parent_code, root_override=None, fwd_root_ref=None, leaf_present=None, flags=0, copy=True) -> Result:
        r = pmb_result()
        self._check(self.L.pmb_group_run_runs(self.h, int(algo), runs.h, _ptr(leaf_present), _ptr(parent_code), _ptr(root_override),
                                              _ptr(fwd_root_ref), int(flags), C.byref(r)))
        return Context._result(None, r, copy)

    def run_async(self, algo=ALGO_FITCH, flags=0):
        self._check(self.L.pmb_group_run_async(self.h, int(algo), int(flags)))

    def wait(self):
        self._check(self.L.pmb_group_wait(self.h))

    def result_device(self) -> pmb_result:
        r = pmb_result()
        self._check(self.L.pmb_group_result_device(self.h, C.byref(r)))
        return r

    def download(self, copy=True) -> Result:
        r = pmb_result()
        self._check(self.L.pmb_group_download(self.h, C.byref(r)))
        return Context._result(None, r, copy)

    def merge_runs(self, to_host: bool = True):
        """pmb_group_merge_runs. to_host=False leaves the NucMut fields on the device (returns the raw pmb_nucmut_result)."""
        r = pmb_nucmut_result()
        self._check(self.L.pmb_group_merge_runs(self.h, 1 if to_host else 0, C.byref(r)))
        return _nucmut_arrays(r) if to_host else r

    def run_nuc(self, algo, n_cols, n_rows, codes4, row_stride, parent_code, root_override=None, fwd_root_ref=None,
                leaf_present=None, flags=0, copy=True) -> Result:
        r = pmb_result()
        self._check(self.L.pmb_group_run_nuc(self.h, int(algo), int(n_cols), int(n_rows), _ptr(codes4), int(row_stride),
                                             _ptr(leaf_present), _ptr(parent_code), _ptr(root_override), _ptr(fwd_root_ref),
                                             int(flags), C.byref(r)))
        return Context._result(None, r, copy)
