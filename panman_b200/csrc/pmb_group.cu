// Column-sharded passes over the GPUs of one box (pmb_group_* of include/panman_b200.h).
//
// The reference parallelises its column loop over the threads of one process (tbb::parallel_for, src/panman.cpp:1568) and
// sorts + run-merges per node after all columns (:1445-1466, :1625-1646); it has no collective of any kind. Here the
// column ranges go to the GPUs, and the one exchange -- every rank's per-node lists to rank 0 -- is done by the packing
// kernel's own stores into rank 0's memory over NVLink (peer access inside a process, CUDA IPC between processes).
// Hand-shakes are stream memory operations (cuStreamWriteValue32 / cuStreamWaitValue32) on words in device memory:
//   arrive[r]  (rank 0's mailbox)  = last step whose shard rank r has finished writing     (written by rank r's stream)
//   credit     (every rank's box)   = last step whose shards rank 0 has finished merging    (written by rank 0's merge stream)
// so neither an SM nor a host thread is involved between "pass enqueued" and "merged lists ready" (a polling warp in place
// of the merge stream's waits was tried: it cost rank 0 2 % of its pass time and gained nothing once the merge itself was
// fast). Mailbox slots are double-buffered by step parity, so the gather + merge of step i overlap pass i + 1.
#include <cuda.h>
#include <cuda_runtime.h>
#include <unistd.h>

#include <time.h>

#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/panman_b200.h"

namespace {

constexpr int64_t GROUP_TILE = 1024;      // column granule of a range = the kernels' tile width
constexpr size_t BOX_ARRIVE = 0;          // u32 arrive[world]
constexpr size_t BOX_CREDIT = 8192;       // u32 credit
constexpr size_t BOX_SLOTS = 16384;       // mailbox slots (rank 0 only)
constexpr int MAX_WORLD = 1024;

struct Handle {  // PMB_GROUP_HANDLE_BYTES
    cudaIpcMemHandle_t mem;  // 64 bytes
    int64_t box_bytes;
    int64_t capacity;
    int32_t rank, device, pid, n_nodes;
    uint64_t magic;
    char pad[PMB_GROUP_HANDLE_BYTES - 64 - 16 - 16 - 8];
};
static_assert(sizeof(Handle) == PMB_GROUP_HANDLE_BYTES, "handle size");
constexpr uint64_t HANDLE_MAGIC = 0x706d625f67727031ull;

typedef CUresult (*WriteValue32Fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
typedef CUresult (*WaitValue32Fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);

struct Pinned {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMallocHost(&p, bytes ? bytes : 1);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

struct Local {
    int device = 0;
    pmb_ctx* ctx = nullptr;
    char* box = nullptr;  // own allocation: flags (+ slots on rank 0)
    size_t box_bytes = 0;
    char* root_box = nullptr;  // rank 0's box as this rank addresses it
    bool root_box_ipc = false;
    bool active = false;       // owns a non-empty column range of the resident alignment
};

}  // namespace

struct pmb_group {
    int n_local = 0, rank_base = 0, world = 1;
    std::vector<Local> local;
    std::string err;
    bool have_tree = false, connected = false, have_input = false;
    int32_t n_nodes = 0;
    int64_t capacity = 0;
    size_t shard_bytes = 0;
    int active = 0;  // ranks with a non-empty range: the first `active` ones
    int64_t n_cols_total = 0;
    uint32_t seq = 0;
    // process holding rank 0
    cudaStream_t merge_stream = nullptr;
    std::vector<char*> peer_box;  // every rank's box as rank 0 addresses it
    std::vector<char> peer_ipc;
    pmb_result merged{};
    bool have_merged = false;
    Pinned h_off, h_pos, h_tc;
    WriteValue32Fn write32 = nullptr;
    WaitValue32Fn wait32 = nullptr;
    bool has_root() const { return rank_base == 0; }
};

namespace {

int gfail(pmb_group* g, int code, const std::string& msg) {
    if (g) g->err = msg;
    return code;
}

int gcuda(pmb_group* g, cudaError_t e, const char* what) {
    std::string m = std::string(what) + ": " + cudaGetErrorString(e);
    cudaGetLastError();
    return gfail(g, e == cudaErrorMemoryAllocation ? PMB_ERR_OOM : PMB_ERR_CUDA, m);
}

int gctx(pmb_group* g, int rc, const Local& l) {  // an error of a local context becomes the group's
    if (rc) g->err = std::string("rank ") + std::to_string(g->rank_base + int(&l - g->local.data())) + ": " + pmb_last_error(l.ctx);
    return rc;
}

#define G_CUDA(call)                                         \
    do {                                                     \
        cudaError_t e__ = (call);                            \
        if (e__ != cudaSuccess) return gcuda(g, e__, #call); \
    } while (0)

#define G_CU(call)                                                                     \
    do {                                                                               \
        CUresult r__ = (call);                                                         \
        if (r__ != CUDA_SUCCESS) return gfail(g, PMB_ERR_CUDA, std::string(#call) + " failed with CUresult " + std::to_string(int(r__))); \
    } while (0)

void range_of(int world, int64_t n_cols, int rank, int64_t* b, int64_t* e) {
    const int64_t tiles = (n_cols + GROUP_TILE - 1) / GROUP_TILE;
    const int64_t base = tiles / world, rem = tiles % world;
    const int64_t t0 = base * rank + std::min<int64_t>(rank, rem), t1 = t0 + base + (rank < rem ? 1 : 0);
    *b = std::min(n_cols, t0 * GROUP_TILE);
    *e = std::min(n_cols, t1 * GROUP_TILE);
}

void release_boxes(pmb_group* g) {
    for (auto& l : g->local) {
        cudaSetDevice(l.device);
        if (l.root_box && l.root_box_ipc) cudaIpcCloseMemHandle(l.root_box);
        l.root_box = nullptr;
        l.root_box_ipc = false;
    }
    if (!g->local.empty()) cudaSetDevice(g->local[0].device);
    for (size_t r = 0; r < g->peer_box.size(); r++)
        if (g->peer_box[r] && g->peer_ipc[r]) cudaIpcCloseMemHandle(g->peer_box[r]);
    g->peer_box.clear();
    g->peer_ipc.clear();
    for (auto& l : g->local) {
        cudaSetDevice(l.device);
        if (l.box) cudaFree(l.box);
        l.box = nullptr;
        l.box_bytes = 0;
    }
    cudaGetLastError();
    g->connected = false;
}

int enable_peer(pmb_group* g, int from_device, int to_device) {
    if (from_device == to_device) return PMB_OK;
    int can = 0;
    G_CUDA(cudaDeviceCanAccessPeer(&can, from_device, to_device));
    if (!can) return gfail(g, PMB_ERR_CUDA, "devices " + std::to_string(from_device) + " and " + std::to_string(to_device) +
                                                " have no peer access: the column-range gather needs NVLink / PCIe peer mapping");
    G_CUDA(cudaSetDevice(from_device));
    cudaError_t e = cudaDeviceEnablePeerAccess(to_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();
        e = cudaSuccess;
    }
    if (e != cudaSuccess) return gcuda(g, e, "cudaDeviceEnablePeerAccess");
    return PMB_OK;
}

// single-process group: all pointers are local, mapping = peer access between rank 0's device and the others
int connect_single(pmb_group* g) {
    const int d0 = g->local[0].device;
    g->peer_box.assign(size_t(g->world), nullptr);
    g->peer_ipc.assign(size_t(g->world), 0);
    for (int i = 0; i < g->n_local; i++) {
        Local& l = g->local[i];
        int rc;
        if ((rc = enable_peer(g, l.device, d0))) return rc;
        if ((rc = enable_peer(g, d0, l.device))) return rc;
        l.root_box = g->local[0].box;
        l.root_box_ipc = false;
        g->peer_box[size_t(i)] = l.box;
    }
    g->connected = true;
    return PMB_OK;
}

int signal_ready(pmb_group* g) {
    if (g->write32 && g->wait32) return PMB_OK;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuStreamWriteValue32", &fn, cudaEnableDefault, &qr) != cudaSuccess || !fn) {
        cudaGetLastError();
        return gfail(g, PMB_ERR_CUDA, "cuStreamWriteValue32 is not available from this driver: the group hand-shake needs stream memory operations");
    }
    g->write32 = reinterpret_cast<WriteValue32Fn>(fn);
    fn = nullptr;
    if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &fn, cudaEnableDefault, &qr) != cudaSuccess || !fn) {
        cudaGetLastError();
        return gfail(g, PMB_ERR_CUDA, "cuStreamWaitValue32 is not available from this driver: the group hand-shake needs stream memory operations");
    }
    g->wait32 = reinterpret_cast<WaitValue32Fn>(fn);
    return PMB_OK;
}

int enqueue_step(pmb_group* g, int algo, int flags, uint32_t s) {
    const size_t buf = size_t(s & 1u) * size_t(g->world) * g->shard_bytes;
    for (int i = 0; i < g->n_local; i++) {
        Local& l = g->local[size_t(i)];
        const int r = g->rank_base + i;
        if (!l.active) continue;
        int rc = pmb_run_resident_async(l.ctx, algo, flags);
        if (rc) return gctx(g, rc, l);
        G_CUDA(cudaSetDevice(l.device));
        // the pass ends on its result stream (the compaction's): packing and the hand-shake go there, and the main stream is
        // free to start the next forward kernel
        CUstream st = static_cast<CUstream>(pmb_result_stream(l.ctx));
        // the slot of this parity is free again once rank 0 has merged step s - 2
        if (s > 2) G_CU(g->wait32(st, CUdeviceptr(l.box + BOX_CREDIT), s - 2, CU_STREAM_WAIT_VALUE_GEQ));
        rc = pmb_pack_result(l.ctx, l.root_box + BOX_SLOTS + buf + size_t(r) * g->shard_bytes, g->capacity, nullptr);
        if (rc) return gctx(g, rc, l);
        // default flags: the write is ordered after the packing kernel's stores (memory barrier before the write)
        G_CU(g->write32(st, CUdeviceptr(l.root_box + BOX_ARRIVE + 4 * size_t(r)), s, CU_STREAM_WRITE_VALUE_DEFAULT));
    }
    if (g->has_root()) {
        Local& l0 = g->local[0];
        G_CUDA(cudaSetDevice(l0.device));
        CUstream ms = static_cast<CUstream>(g->merge_stream);
        for (int r = 0; r < g->active; r++) G_CU(g->wait32(ms, CUdeviceptr(l0.box + BOX_ARRIVE + 4 * size_t(r)), s, CU_STREAM_WAIT_VALUE_GEQ));
        int rc = pmb_merge_packed(l0.ctx, g->active, l0.box + BOX_SLOTS + buf, g->capacity, g->merge_stream, &g->merged);
        if (rc) return gctx(g, rc, l0);
        for (int r = 0; r < g->active; r++) G_CU(g->write32(ms, CUdeviceptr(g->peer_box[size_t(r)] + BOX_CREDIT), s, CU_STREAM_WRITE_VALUE_DEFAULT));
        g->have_merged = true;
    }
    return PMB_OK;
}

void unblock_step(pmb_group* g, uint32_t s) {
    for (int i = 0; i < g->n_local; i++) {
        Local& l = g->local[size_t(i)];
        if (!l.active || !l.root_box) continue;
        if (cudaSetDevice(l.device) != cudaSuccess) continue;
        cudaStream_t aux = nullptr;
        if (cudaStreamCreateWithFlags(&aux, cudaStreamNonBlocking) != cudaSuccess) continue;
        g->write32(static_cast<CUstream>(aux), CUdeviceptr(l.root_box + BOX_ARRIVE + 4 * size_t(g->rank_base + i)), s, CU_STREAM_WRITE_VALUE_DEFAULT);
        if (g->has_root())
            for (int r = 0; r < g->active && r < int(g->peer_box.size()); r++)
                if (g->peer_box[size_t(r)]) g->write32(static_cast<CUstream>(aux), CUdeviceptr(g->peer_box[size_t(r)] + BOX_CREDIT), s, CU_STREAM_WRITE_VALUE_DEFAULT);
        cudaStreamSynchronize(aux);
        cudaStreamDestroy(aux);
    }
    cudaGetLastError();
}

}  // namespace

extern "C" {

int pmb_group_column_range(int world, int64_t n_cols, int rank, int64_t* col_begin, int64_t* col_end) {
    if (world < 1 || rank < 0 || rank >= world || n_cols < 0 || !col_begin || !col_end) return PMB_ERR_INVALID;
    range_of(world, n_cols, rank, col_begin, col_end);
    return PMB_OK;
}

int pmb_group_create(pmb_group** out, const int* devices, int n_local, int rank_base, int world) {
    if (!out) return PMB_ERR_INVALID;
    *out = nullptr;
    if (!devices || n_local < 1 || world < n_local || world > MAX_WORLD || rank_base < 0 || rank_base + n_local > world) return PMB_ERR_INVALID;
    pmb_group* g = new (std::nothrow) pmb_group();
    if (!g) return PMB_ERR_OOM;
    g->n_local = n_local;
    g->rank_base = rank_base;
    g->world = world;
    g->local.resize(size_t(n_local));
    *out = g;
    for (int i = 0; i < n_local; i++) {
        g->local[i].device = devices[i];
        int rc = pmb_create(&g->local[i].ctx, devices[i]);
        if (rc) return gctx(g, rc, g->local[i]);  // the group stays alive so that pmb_group_last_error can say why
        pmb_set_option(g->local[i].ctx, "lanes", 0);  // a rank's steps are ordered by the mailbox hand-shake: one pipeline each
    }
    if (g->has_root() && world > 1) {
        G_CUDA(cudaSetDevice(g->local[0].device));
        int lo = 0, hi = 0;
        G_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        // the merge fills the SMs the persistent pass kernels of the next step leave idle while they drain: lowest priority
        G_CUDA(cudaStreamCreateWithPriority(&g->merge_stream, cudaStreamNonBlocking, lo));
    }
    return PMB_OK;
}

void pmb_group_destroy(pmb_group* g) {
    if (!g) return;
    for (auto& l : g->local)
        if (l.ctx) {
            cudaSetDevice(l.device);
            cudaDeviceSynchronize();
        }
    cudaGetLastError();
    release_boxes(g);
    if (g->merge_stream) {
        cudaSetDevice(g->local[0].device);
        cudaStreamDestroy(g->merge_stream);
    }
    g->h_off.release();
    g->h_pos.release();
    g->h_tc.release();
    for (auto& l : g->local)
        if (l.ctx) pmb_destroy(l.ctx);
    delete g;
}

const char* pmb_group_last_error(const pmb_group* g) { return g ? g->err.c_str() : "null group"; }

int pmb_group_world(const pmb_group* g) { return g ? g->world : 0; }

pmb_ctx* pmb_group_ctx(pmb_group* g, int local_index) {
    if (!g || local_index < 0 || local_index >= g->n_local) return nullptr;
    return g->local[size_t(local_index)].ctx;
}

int pmb_group_set_tree(pmb_group* g, int32_t n_nodes, int32_t root, const int32_t* child_offsets, const int32_t* child_index,
                       const int32_t* leaf_row) {
    if (!g) return PMB_ERR_INVALID;
    for (auto& l : g->local) {
        int rc = pmb_set_tree(l.ctx, n_nodes, root, child_offsets, child_index, leaf_row);
        if (rc) return gctx(g, rc, l);
    }
    if (g->have_tree && n_nodes != g->n_nodes && g->capacity > 0) {  // the mailbox slots were sized for another tree
        release_boxes(g);
        g->capacity = 0;
    }
    g->n_nodes = n_nodes;
    g->have_tree = true;
    g->have_input = false;
    g->have_merged = false;
    return PMB_OK;
}

int pmb_group_reserve(pmb_group* g, int64_t capacity) {
    if (!g || capacity < 0) return PMB_ERR_INVALID;
    if (!g->have_tree) return gfail(g, PMB_ERR_NO_TREE, "pmb_group_set_tree has not been called");
    if (g->world == 1) return PMB_OK;  // nothing to exchange
    int rc = signal_ready(g);
    if (rc) return rc;
    for (auto& l : g->local) {  // nothing may still be using the old boxes
        G_CUDA(cudaSetDevice(l.device));
        G_CUDA(cudaDeviceSynchronize());
    }
    release_boxes(g);
    g->capacity = capacity;
    g->shard_bytes = size_t(pmb_packed_bytes(g->n_nodes, capacity));  // a multiple of 16; the stride pmb_merge_packed expects
    g->seq = 0;
    g->have_merged = false;
    for (int i = 0; i < g->n_local; i++) {
        Local& l = g->local[size_t(i)];
        const bool is_root = g->rank_base + i == 0;
        // at least 2 MB: a whole allocation granule of its own, so that the IPC mapping exposes nothing else
        l.box_bytes = std::max<size_t>(size_t(2) << 20, BOX_SLOTS + (is_root ? 2 * size_t(g->world) * g->shard_bytes : 0));
        G_CUDA(cudaSetDevice(l.device));
        G_CUDA(cudaMalloc(reinterpret_cast<void**>(&l.box), l.box_bytes));
        G_CUDA(cudaMemset(l.box, 0, BOX_SLOTS));
        G_CUDA(cudaDeviceSynchronize());
    }
    if (g->n_local == g->world) return connect_single(g);
    return PMB_OK;
}

int pmb_group_export(pmb_group* g, void* handles_out) {
    if (!g || !handles_out) return PMB_ERR_INVALID;
    if (g->world > 1 && !g->local[0].box) return gfail(g, PMB_ERR_NO_INPUT, "pmb_group_reserve has not been called");
    Handle* h = static_cast<Handle*>(handles_out);
    for (int i = 0; i < g->n_local; i++) {
        Local& l = g->local[size_t(i)];
        std::memset(&h[i], 0, sizeof(Handle));
        h[i].magic = HANDLE_MAGIC;
        h[i].rank = g->rank_base + i;
        h[i].device = l.device;
        h[i].pid = int32_t(getpid());
        h[i].n_nodes = g->n_nodes;
        h[i].capacity = g->capacity;
        h[i].box_bytes = int64_t(l.box_bytes);
        if (g->world > 1) {
            G_CUDA(cudaSetDevice(l.device));
            G_CUDA(cudaIpcGetMemHandle(&h[i].mem, l.box));
        }
    }
    return PMB_OK;
}

int pmb_group_connect(pmb_group* g, const void* all_handles) {
    if (!g || !all_handles) return PMB_ERR_INVALID;
    if (g->world == 1) return PMB_OK;
    if (!g->local[0].box) return gfail(g, PMB_ERR_NO_INPUT, "pmb_group_reserve has not been called");
    if (g->n_local == g->world) return PMB_OK;  // connected by pmb_group_reserve
    const Handle* h = static_cast<const Handle*>(all_handles);
    const int32_t pid = int32_t(getpid());
    for (int r = 0; r < g->world; r++) {
        if (h[r].magic != HANDLE_MAGIC || h[r].rank != r) return gfail(g, PMB_ERR_INVALID, "pmb_group_connect: handle " + std::to_string(r) + " is not rank " + std::to_string(r) + "'s");
        if (h[r].n_nodes != g->n_nodes || h[r].capacity != g->capacity)
            return gfail(g, PMB_ERR_INVALID, "pmb_group_connect: rank " + std::to_string(r) + " was set up with another tree or mailbox capacity");
    }
    // every local rank addresses rank 0's box
    char* mapped_root = nullptr;
    for (int i = 0; i < g->n_local; i++) {
        Local& l = g->local[size_t(i)];
        G_CUDA(cudaSetDevice(l.device));
        if (h[0].pid == pid) {  // rank 0 lives in this process
            int rc = enable_peer(g, l.device, g->local[0].device);
            if (rc) return rc;
            l.root_box = g->local[0].box;
            l.root_box_ipc = false;
        } else if (!mapped_root) {
            G_CUDA(cudaIpcOpenMemHandle(reinterpret_cast<void**>(&mapped_root), h[0].mem, cudaIpcMemLazyEnablePeerAccess));
            l.root_box = mapped_root;
            l.root_box_ipc = true;
        } else {  // one mapping per process; further local devices reach it through peer access to rank 0's device
            int rc = enable_peer(g, l.device, h[0].device);
            if (rc) return rc;
            l.root_box = mapped_root;
            l.root_box_ipc = false;
        }
    }
    if (g->has_root()) {
        g->peer_box.assign(size_t(g->world), nullptr);
        g->peer_ipc.assign(size_t(g->world), 0);
        G_CUDA(cudaSetDevice(g->local[0].device));
        for (int r = 0; r < g->world; r++) {
            if (h[r].pid == pid) {
                const int i = r - g->rank_base;
                if (i < 0 || i >= g->n_local) return gfail(g, PMB_ERR_INVALID, "pmb_group_connect: inconsistent handles");
                int rc = enable_peer(g, g->local[0].device, g->local[size_t(i)].device);
                if (rc) return rc;
                G_CUDA(cudaSetDevice(g->local[0].device));
                g->peer_box[size_t(r)] = g->local[size_t(i)].box;
            } else {
                char* p = nullptr;
                G_CUDA(cudaIpcOpenMemHandle(reinterpret_cast<void**>(&p), h[r].mem, cudaIpcMemLazyEnablePeerAccess));
                g->peer_box[size_t(r)] = p;
                g->peer_ipc[size_t(r)] = 1;
            }
        }
    }
    g->connected = true;
    return PMB_OK;
}

// positions are int32: a column past 2^31 - 1 could not be emitted on any rank
constexpr int64_t MAX_COLS_TOTAL = int64_t(1) << 31;

// one local rank's range, from a nibble matrix of the range (shard_codes_4bit) or from an encoded batch (runs: the range's
// columns start at runs_col_begin of it)
static int upload_shard_impl(pmb_group* g, int local_index, int64_t n_cols_total, int32_t n_rows, const uint8_t* shard_codes_4bit,
                             int64_t row_stride_bytes, const uint8_t* leaf_present, const uint8_t* shard_parent_code,
                             const int8_t* shard_root_override, const int8_t* shard_fwd_root_ref, const pmb_runs* runs,
                             int64_t runs_col_begin) {
    if (!g || local_index < 0 || local_index >= g->n_local || n_cols_total <= 0) return PMB_ERR_INVALID;
    if (!g->have_tree) return gfail(g, PMB_ERR_NO_TREE, "pmb_group_set_tree has not been called");
    if (n_cols_total > MAX_COLS_TOTAL) return gfail(g, PMB_ERR_INVALID, "n_cols_total exceeds 2^31: positions are int32");
    if (g->have_input && g->n_cols_total != n_cols_total) {  // a new alignment: every local rank must be given its range again
        for (auto& l : g->local) l.active = false;
        g->have_input = false;
    }
    Local& l = g->local[size_t(local_index)];
    int64_t b, e;
    range_of(g->world, n_cols_total, g->rank_base + local_index, &b, &e);
    g->n_cols_total = n_cols_total;
    g->active = int(std::min<int64_t>(g->world, (n_cols_total + GROUP_TILE - 1) / GROUP_TILE));
    g->have_merged = false;
    l.active = e > b;
    if (l.active) {
        int rc = runs ? pmb_upload_runs_async(l.ctx, runs, runs_col_begin, e - b, leaf_present, shard_parent_code, shard_root_override,
                                              shard_fwd_root_ref, b)
                      : pmb_upload_nuc_async(l.ctx, e - b, n_rows, shard_codes_4bit, row_stride_bytes, leaf_present, shard_parent_code,
                                             shard_root_override, shard_fwd_root_ref, b);
        if (rc) return gctx(g, rc, l);
    }
    g->have_input = true;
    return PMB_OK;
}

int pmb_group_upload_shard(pmb_group* g, int local_index, int64_t n_cols_total, int32_t n_rows, const uint8_t* shard_codes_4bit,
                           int64_t row_stride_bytes, const uint8_t* leaf_present, const uint8_t* shard_parent_code,
                           const int8_t* shard_root_override, const int8_t* shard_fwd_root_ref) {
    return upload_shard_impl(g, local_index, n_cols_total, n_rows, shard_codes_4bit, row_stride_bytes, leaf_present, shard_parent_code,
                             shard_root_override, shard_fwd_root_ref, nullptr, 0);
}

int pmb_group_upload_shard_runs(pmb_group* g, int local_index, int64_t n_cols_total, const pmb_runs* shard_runs, const uint8_t* leaf_present,
                                const uint8_t* shard_parent_code, const int8_t* shard_root_override, const int8_t* shard_fwd_root_ref) {
    if (!g || !shard_runs) return g ? gfail(g, PMB_ERR_INVALID, "null runs") : PMB_ERR_INVALID;
    if (n_cols_total > MAX_COLS_TOTAL) return gfail(g, PMB_ERR_INVALID, "n_cols_total exceeds 2^31: positions are int32");
    pmb_runs_info info{};
    pmb_runs_describe(shard_runs, &info);
    int64_t b, e;
    if (local_index >= 0 && local_index < g->n_local) {
        range_of(g->world, n_cols_total, g->rank_base + local_index, &b, &e);
        if (e > b && info.n_cols != e - b) return gfail(g, PMB_ERR_INVALID, "the encoded shard does not cover the rank's column range");
    }
    return upload_shard_impl(g, local_index, n_cols_total, info.n_rows, nullptr, 0, leaf_present, shard_parent_code, shard_root_override,
                             shard_fwd_root_ref, shard_runs, 0);
}

int pmb_group_upload_runs(pmb_group* g, const pmb_runs* runs, const uint8_t* leaf_present, const uint8_t* parent_code,
                          const int8_t* root_override, const int8_t* fwd_root_ref) {
    if (!g || !runs || !parent_code) return g ? gfail(g, PMB_ERR_INVALID, "bad input arguments") : PMB_ERR_INVALID;
    pmb_runs_info info{};
    pmb_runs_describe(runs, &info);
    for (int i = 0; i < g->n_local; i++) {
        int64_t b, e;
        range_of(g->world, info.n_cols, g->rank_base + i, &b, &e);
        int rc = upload_shard_impl(g, i, info.n_cols, info.n_rows, nullptr, 0, leaf_present, parent_code + b, root_override ? root_override + b : nullptr,
                                   fwd_root_ref ? fwd_root_ref + b : nullptr, runs, b);
        if (rc) return rc;
    }
    return PMB_OK;
}

int pmb_group_upload_nuc(pmb_group* g, int64_t n_cols, int32_t n_rows, const uint8_t* leaf_codes_4bit, int64_t row_stride_bytes,
                         const uint8_t* leaf_present, const uint8_t* parent_code, const int8_t* root_override,
                         const int8_t* fwd_root_ref) {
    if (!g || n_cols <= 0 || !leaf_codes_4bit || !parent_code) return g ? gfail(g, PMB_ERR_INVALID, "bad input arguments") : PMB_ERR_INVALID;
    for (int i = 0; i < g->n_local; i++) {
        int64_t b, e;
        range_of(g->world, n_cols, g->rank_base + i, &b, &e);  // b is a multiple of 1024: a whole byte of every row
        int rc = pmb_group_upload_shard(g, i, n_cols, n_rows, leaf_codes_4bit + b / 2, row_stride_bytes, leaf_present, parent_code + b,
                                        root_override ? root_override + b : nullptr, fwd_root_ref ? fwd_root_ref + b : nullptr);
        if (rc) return rc;
    }
    return PMB_OK;
}

int pmb_group_run_async(pmb_group* g, int algo, int flags) {
    if (!g) return PMB_ERR_INVALID;
    if (!g->have_input) return gfail(g, PMB_ERR_NO_INPUT, "no resident input: call pmb_group_upload_nuc / pmb_group_upload_shard first");
    if (flags & PMB_FLAG_WANT_STATES) return gfail(g, PMB_ERR_INVALID, "PMB_FLAG_WANT_STATES is per context: run the ranks' contexts (pmb_group_ctx) for state matrices");
    if (g->world == 1) {
        int rc = pmb_run_resident_async(g->local[0].ctx, algo, flags);
        return rc ? gctx(g, rc, g->local[0]) : PMB_OK;
    }
    if (!g->connected) return gfail(g, PMB_ERR_NO_INPUT, "the group is not connected: pmb_group_reserve (+ pmb_group_export / pmb_group_connect across processes)");
    const uint32_t s = ++g->seq;
    int rc = enqueue_step(g, algo, flags, s);
    if (rc) {
        // part of the step may be enqueued already: streams of this or of other processes would wait for ever for the
        // words this process did not get to write. Write them from a stream of their own (the shards of such a step are
        // garbage; the caller sees the error and the group must be re-reserved before it is used again).
        std::string keep = g->err;
        unblock_step(g, s);
        g->err = keep;
        g->connected = false;
    }
    return rc;
}

int pmb_group_wait(pmb_group* g) {
    if (!g) return PMB_ERR_INVALID;
    int first = PMB_OK;
    static const bool debug = getenv("PMB_GROUP_DEBUG") != nullptr;
    timespec t0{}, t1{}, t2{};
    if (debug) clock_gettime(CLOCK_MONOTONIC, &t0);
    for (auto& l : g->local) {
        int rc = pmb_wait(l.ctx);
        if (rc && !first) first = gctx(g, rc, l);
    }
    if (debug) clock_gettime(CLOCK_MONOTONIC, &t1);
    if (g->world > 1 && g->has_root() && g->have_merged) {
        int rc = pmb_merge_status(g->local[0].ctx);
        if (rc && !first) first = gctx(g, rc, g->local[0]);
    }
    if (debug) {
        clock_gettime(CLOCK_MONOTONIC, &t2);
        auto ms = [](const timespec& a, const timespec& b) { return (b.tv_sec - a.tv_sec) * 1e3 + (b.tv_nsec - a.tv_nsec) * 1e-6; };
        fprintf(stderr, "[pmb_group_wait rank %d] contexts %.3f ms, merge %.3f ms\n", g->rank_base, ms(t0, t1), ms(t1, t2));
    }
    return first;
}

int pmb_group_result_device(pmb_group* g, pmb_result* out) {
    if (!g || !out) return PMB_ERR_INVALID;
    std::memset(out, 0, sizeof *out);
    if (!g->has_root()) return PMB_OK;
    if (g->world == 1) {
        int rc = pmb_result_device(g->local[0].ctx, out);
        return rc ? gctx(g, rc, g->local[0]) : PMB_OK;
    }
    if (!g->have_merged) return gfail(g, PMB_ERR_NO_INPUT, "no merged result: call pmb_group_run_async first");
    *out = g->merged;
    out->n_cols = g->n_cols_total;
    return PMB_OK;
}

int pmb_group_download(pmb_group* g, pmb_result* out) {
    if (!g || !out) return PMB_ERR_INVALID;
    std::memset(out, 0, sizeof *out);
    int rc = pmb_group_wait(g);
    if (rc) return rc;
    if (!g->has_root()) return PMB_OK;
    if (g->world == 1) {
        rc = pmb_download(g->local[0].ctx, out);
        return rc ? gctx(g, rc, g->local[0]) : PMB_OK;
    }
    if (!g->have_merged) return gfail(g, PMB_ERR_NO_INPUT, "no merged result: call pmb_group_run_async first");
    const size_t N = size_t(g->n_nodes);
    G_CUDA(cudaSetDevice(g->local[0].device));
    G_CUDA(g->h_off.ensure((N + 1) * sizeof(int64_t)));
    G_CUDA(cudaMemcpyAsync(g->h_off.p, g->merged.node_offsets, (N + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, g->merge_stream));
    G_CUDA(cudaStreamSynchronize(g->merge_stream));
    const size_t n = size_t(static_cast<const int64_t*>(g->h_off.p)[N]);
    G_CUDA(g->h_pos.ensure(std::max<size_t>(1, n) * sizeof(int32_t)));
    G_CUDA(g->h_tc.ensure(std::max<size_t>(1, n)));
    if (n) {
        G_CUDA(cudaMemcpyAsync(g->h_pos.p, g->merged.pos, n * sizeof(int32_t), cudaMemcpyDeviceToHost, g->merge_stream));
        G_CUDA(cudaMemcpyAsync(g->h_tc.p, g->merged.type_code, n, cudaMemcpyDeviceToHost, g->merge_stream));
        G_CUDA(cudaStreamSynchronize(g->merge_stream));
    }
    out->n_mut = int64_t(n);
    out->n_nodes = g->n_nodes;
    out->node_offsets = static_cast<const int64_t*>(g->h_off.p);
    out->pos = static_cast<const int32_t*>(g->h_pos.p);
    out->type_code = static_cast<const uint8_t*>(g->h_tc.p);
    out->states = nullptr;
    out->n_cols = g->n_cols_total;
    return PMB_OK;
}

int pmb_group_merge_runs(pmb_group* g, int to_host, pmb_nucmut_result* out) {
    if (!g || !out) return PMB_ERR_INVALID;
    std::memset(out, 0, sizeof *out);
    if (!g->has_root()) return PMB_OK;
    if (g->world > 1 && !g->have_merged) return gfail(g, PMB_ERR_NO_INPUT, "no merged result: call pmb_group_run_async first");
    int rc = pmb_merge_runs(g->local[0].ctx, g->world == 1 ? 0 : 1, to_host, out);
    return rc ? gctx(g, rc, g->local[0]) : PMB_OK;
}

static int step_after_upload(pmb_group* g, int algo, int flags, pmb_result* out);

int pmb_group_run_nuc(pmb_group* g, int algo, int64_t n_cols, int32_t n_rows, const uint8_t* leaf_codes_4bit, int64_t row_stride_bytes,
                      const uint8_t* leaf_present, const uint8_t* parent_code, const int8_t* root_override, const int8_t* fwd_root_ref,
                      int flags, pmb_result* out) {
    if (!g || !out) return PMB_ERR_INVALID;
    int rc = pmb_group_upload_nuc(g, n_cols, n_rows, leaf_codes_4bit, row_stride_bytes, leaf_present, parent_code, root_override,
                                  fwd_root_ref);
    if (rc) return rc;
    return step_after_upload(g, algo, flags, out);
}

int pmb_group_run_runs(pmb_group* g, int algo, const pmb_runs* runs, const uint8_t* leaf_present, const uint8_t* parent_code,
                       const int8_t* root_override, const int8_t* fwd_root_ref, int flags, pmb_result* out) {
    if (!g || !out) return PMB_ERR_INVALID;
    int rc = pmb_group_upload_runs(g, runs, leaf_present, parent_code, root_override, fwd_root_ref);
    if (rc) return rc;
    return step_after_upload(g, algo, flags, out);
}

// one step on the resident input + download, sizing the mailbox on the way where the group can do that by itself
static int step_after_upload(pmb_group* g, int algo, int flags, pmb_result* out) {
    int rc;
    if (g->world > 1 && g->capacity == 0) {
        // no mailbox yet: only a single-process group can size one by itself (a first pass, then the largest shard + 25 %)
        if (g->n_local != g->world) return gfail(g, PMB_ERR_NO_INPUT, "pmb_group_reserve / export / connect must precede the first step of a multi-process group");
        int64_t need = 0;
        for (auto& l : g->local) {
            if (!l.active) continue;
            if ((rc = pmb_run_resident(l.ctx, algo, flags))) return gctx(g, rc, l);
            pmb_result r{};
            if ((rc = pmb_result_device(l.ctx, &r))) return gctx(g, rc, l);
            need = std::max(need, r.n_mut);
        }
        if ((rc = pmb_group_reserve(g, need + need / 4 + 4096))) return rc;
    }
    for (int attempt = 0;; attempt++) {
        if ((rc = pmb_group_run_async(g, algo, flags))) return rc;
        rc = pmb_group_download(g, out);
        if (rc == PMB_ERR_STAGING && attempt < 4) continue;  // the pool has been grown
        if (rc == PMB_ERR_CAPACITY && attempt < 4 && g->n_local == g->world) {
            int64_t need = 0;
            for (auto& l : g->local) {
                if (!l.active) continue;
                pmb_result r{};
                if (pmb_result_device(l.ctx, &r) == PMB_OK) need = std::max(need, r.n_mut);
            }
            if ((rc = pmb_group_reserve(g, std::max(need + need / 4 + 4096, 2 * g->capacity)))) return rc;
            continue;
        }
        return rc;
    }
}

}  // extern "C"
