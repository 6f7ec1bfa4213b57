"""Loader for libpanman_b200.so. Fails loudly: a missing or unloadable extension is an error, never a fallback."""
import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PANMAN_B200_LIB", os.path.join(HERE, "libpanman_b200.so"))  # override: tuning variants only

# every symbol include/panman_b200.h declares
EXPORTS = ["pmb_create", "pmb_destroy", "pmb_last_error", "pmb_set_option", "pmb_set_tree", "pmb_run_nuc", "pmb_upload_nuc",
           "pmb_run_resident", "pmb_download", "pmb_result_device", "pmb_last_timings", "pmb_algorithmic_bytes", "pmb_version",
           "pmb_packed_bytes", "pmb_pack_result", "pmb_merge_packed", "pmb_stream", "pmb_run_resident_async", "pmb_wait",
           "pmb_host_alloc", "pmb_host_free", "pmb_merge_runs", "pmb_set_column_breaks", "pmb_run_block",
           "pmb_upload_nuc_async", "pmb_merge_status", "pmb_result_stream",
           "pmb_group_create", "pmb_group_destroy", "pmb_group_last_error", "pmb_group_world", "pmb_group_ctx",
           "pmb_group_column_range", "pmb_group_set_tree", "pmb_group_reserve", "pmb_group_export", "pmb_group_connect",
           "pmb_group_upload_nuc", "pmb_group_upload_shard", "pmb_group_run_async", "pmb_group_wait",
           "pmb_group_result_device", "pmb_group_download", "pmb_group_merge_runs", "pmb_group_run_nuc",
           "pmb_runs_encode", "pmb_runs_free", "pmb_runs_describe", "pmb_upload_runs", "pmb_upload_runs_async", "pmb_run_runs",
           "pmb_group_upload_runs", "pmb_group_upload_shard_runs", "pmb_group_run_runs", "pmb_join", "pmb_upload_replay"]
GROUP_HANDLE_BYTES = 128


class pmb_result(C.Structure):
    _fields_ = [("n_mut", C.c_int64), ("n_nodes", C.c_int32), ("reserved", C.c_int32), ("node_offsets", C.c_void_p),
                ("pos", C.c_void_p), ("type_code", C.c_void_p), ("states", C.c_void_p), ("n_cols", C.c_int64)]


class pmb_nucmut_result(C.Structure):
    _fields_ = [("n", C.c_int64), ("n_nodes", C.c_int32), ("reserved", C.c_int32), ("node_offsets", C.c_void_p),
                ("nuc_position", C.c_void_p), ("mut_info", C.c_void_p), ("nucs", C.c_void_p), ("mut_info_wire", C.c_void_p)]


class pmb_runs_info(C.Structure):
    _fields_ = [("n_cols", C.c_int64), ("n_rows", C.c_int32), ("n_tiles", C.c_int32), ("n_segments", C.c_int32), ("seg_rows", C.c_int32),
                ("n_events", C.c_int64), ("bytes", C.c_int64), ("events", C.c_void_p), ("item_offsets", C.c_void_p)]


class pmb_timings(C.Structure):
    _fields_ = [("forward_ms", C.c_float), ("backward_ms", C.c_float), ("compact_ms", C.c_float), ("total_ms", C.c_float),
                ("n_launches", C.c_int32), ("n_levels", C.c_int32)]


def build_library(verbose: bool = False) -> str:
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> panman_b200/libpanman_b200.so (cross-compiles without a GPU)."""
    out = None if verbose else subprocess.DEVNULL
    subprocess.check_call(["make", "-C", os.path.join(HERE, "csrc")], stdout=out)
    return LIB_PATH


_lib = None


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    for name in EXPORTS:
        if not hasattr(L, name):
            raise RuntimeError(f"{LIB_PATH} does not export {name}")
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.pmb_create.argtypes = [C.POINTER(vp), C.c_int]
    L.pmb_destroy.argtypes = [vp]
    L.pmb_destroy.restype = None
    L.pmb_last_error.argtypes = [vp]
    L.pmb_last_error.restype = C.c_char_p
    L.pmb_set_option.argtypes = [vp, C.c_char_p, i64]
    L.pmb_set_tree.argtypes = [vp, i32, i32, vp, vp, vp]
    L.pmb_run_nuc.argtypes = [vp, C.c_int, i64, i32, vp, i64, vp, vp, vp, vp, i64, C.c_int, C.POINTER(pmb_result)]
    L.pmb_upload_nuc.argtypes = [vp, i64, i32, vp, i64, vp, vp, vp, vp, i64]
    L.pmb_upload_replay.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, i64, vp, i32]
    L.pmb_run_resident.argtypes = [vp, C.c_int, C.c_int]
    L.pmb_run_resident_async.argtypes = [vp, C.c_int, C.c_int]
    L.pmb_wait.argtypes = [vp]
    L.pmb_join.argtypes = [vp]
    L.pmb_download.argtypes = [vp, C.POINTER(pmb_result)]
    L.pmb_result_device.argtypes = [vp, C.POINTER(pmb_result)]
    L.pmb_last_timings.argtypes = [vp, C.POINTER(pmb_timings)]
    L.pmb_algorithmic_bytes.argtypes = [vp, C.c_int]
    L.pmb_algorithmic_bytes.restype = i64
    L.pmb_version.restype = C.c_char_p
    L.pmb_stream.argtypes = [vp]
    L.pmb_stream.restype = vp
    L.pmb_result_stream.argtypes = [vp]
    L.pmb_result_stream.restype = vp
    L.pmb_packed_bytes.argtypes = [i32, i64]
    L.pmb_packed_bytes.restype = i64
    L.pmb_host_alloc.argtypes = [C.c_size_t]
    L.pmb_host_alloc.restype = vp
    L.pmb_host_free.argtypes = [vp]
    L.pmb_host_free.restype = None
    L.pmb_merge_runs.argtypes = [vp, C.c_int, C.c_int, C.POINTER(pmb_nucmut_result)]
    L.pmb_set_column_breaks.argtypes = [vp, vp]
    L.pmb_run_block.argtypes = [vp, C.c_int, i64, i32, vp, vp, C.POINTER(pmb_result)]
    L.pmb_pack_result.argtypes = [vp, vp, i64, vp]
    L.pmb_merge_packed.argtypes = [vp, i32, vp, i64, vp, C.POINTER(pmb_result)]
    L.pmb_upload_nuc_async.argtypes = [vp, i64, i32, vp, i64, vp, vp, vp, vp, i64]
    L.pmb_merge_status.argtypes = [vp]
    L.pmb_group_create.argtypes = [C.POINTER(vp), C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int]
    L.pmb_group_destroy.argtypes = [vp]
    L.pmb_group_destroy.restype = None
    L.pmb_group_last_error.argtypes = [vp]
    L.pmb_group_last_error.restype = C.c_char_p
    L.pmb_group_world.argtypes = [vp]
    L.pmb_group_ctx.argtypes = [vp, C.c_int]
    L.pmb_group_ctx.restype = vp
    L.pmb_group_column_range.argtypes = [C.c_int, i64, C.c_int, C.POINTER(i64), C.POINTER(i64)]
    L.pmb_group_set_tree.argtypes = [vp, i32, i32, vp, vp, vp]
    L.pmb_group_reserve.argtypes = [vp, i64]
    L.pmb_group_export.argtypes = [vp, vp]
    L.pmb_group_connect.argtypes = [vp, vp]
    L.pmb_group_upload_nuc.argtypes = [vp, i64, i32, vp, i64, vp, vp, vp, vp]
    L.pmb_group_upload_shard.argtypes = [vp, C.c_int, i64, i32, vp, i64, vp, vp, vp, vp]
    L.pmb_group_run_async.argtypes = [vp, C.c_int, C.c_int]
    L.pmb_group_wait.argtypes = [vp]
    L.pmb_group_result_device.argtypes = [vp, C.POINTER(pmb_result)]
    L.pmb_group_download.argtypes = [vp, C.POINTER(pmb_result)]
    L.pmb_group_merge_runs.argtypes = [vp, C.c_int, C.POINTER(pmb_nucmut_result)]
    L.pmb_group_run_nuc.argtypes = [vp, C.c_int, i64, i32, vp, i64, vp, vp, vp, vp, C.c_int, C.POINTER(pmb_result)]
    L.pmb_runs_encode.argtypes = [i32, i32, vp, vp, vp, i64, i32, vp, i64, vp, C.c_int, C.POINTER(vp)]
    L.pmb_runs_free.argtypes = [vp]
    L.pmb_runs_free.restype = None
    L.pmb_runs_describe.argtypes = [vp, C.POINTER(pmb_runs_info)]
    L.pmb_upload_runs.argtypes = [vp, vp, i64, i64, vp, vp, vp, vp, i64]
    L.pmb_upload_runs_async.argtypes = [vp, vp, i64, i64, vp, vp, vp, vp, i64]
    L.pmb_run_runs.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, i64, C.c_int, C.POINTER(pmb_result)]
    L.pmb_group_upload_runs.argtypes = [vp, vp, vp, vp, vp, vp]
    L.pmb_group_upload_shard_runs.argtypes = [vp, C.c_int, i64, vp, vp, vp, vp, vp]
    L.pmb_group_run_runs.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, C.c_int, C.POINTER(pmb_result)]
    _lib = L
    return L
