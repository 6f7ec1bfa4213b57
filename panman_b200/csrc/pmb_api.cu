// C-ABI implementation of libpanman_b200 (see include/panman_b200.h).
// Host side: context, device buffers, the level schedule of kernel launches, result download.
// There is deliberately no CPU compute path here: without a device every compute call fails.
#include <cuda_runtime.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/panman_b200.h"
#include "pmb_kernels.cuh"
#include "pmb_runs.h"
#include "tree_program.h"

using namespace pmb;

namespace {

// PMB_DEBUG_CANARY=1 (environment, read once): every device buffer gets 256 guard bytes on either side filled with 0xC5 and
// a body poisoned with 0xAB instead of whatever the allocator returns; pmb_debug_check_canaries() counts guard bytes that
// changed. compute-sanitizer is not available on every pool: this is the library's own out-of-bounds-write / uninitialised-
// read check (tools/sanitize_small.py runs every kernel path under it and compares the results with the oracle).
struct DevBuf;
static bool g_canary = getenv("PMB_DEBUG_CANARY") != nullptr && getenv("PMB_DEBUG_CANARY")[0] == '1';
static std::vector<DevBuf*> g_canary_bufs;
constexpr size_t CANARY = 256;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    void* raw = nullptr;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        release();
        if (!g_canary) {
            cudaError_t e = cudaMalloc(&p, bytes);
            if (e == cudaSuccess) cap = bytes;
            return e;
        }
        const size_t body = (bytes + 255) / 256 * 256;
        cudaError_t e = cudaMalloc(&raw, body + 2 * CANARY);
        if (e != cudaSuccess) return e;
        cudaMemset(raw, 0xC5, CANARY);
        cudaMemset(static_cast<char*>(raw) + CANARY, 0xAB, body);
        cudaMemset(static_cast<char*>(raw) + CANARY + body, 0xC5, CANARY);
        cudaDeviceSynchronize();
        p = static_cast<char*>(raw) + CANARY;
        cap = bytes;
        g_canary_bufs.push_back(this);
        return cudaSuccess;
    }
    void release() {
        if (raw) {
            cudaFree(raw);
            g_canary_bufs.erase(std::remove(g_canary_bufs.begin(), g_canary_bufs.end(), this), g_canary_bufs.end());
        } else if (p) {
            cudaFree(p);
        }
        p = raw = nullptr;
        cap = 0;
    }
    long long bad_guard_bytes() const {
        if (!raw) return 0;
        const size_t body = (cap + 255) / 256 * 256;
        std::vector<unsigned char> g(2 * CANARY);
        cudaMemcpy(g.data(), raw, CANARY, cudaMemcpyDeviceToHost);
        cudaMemcpy(g.data() + CANARY, static_cast<char*>(raw) + CANARY + body, CANARY, cudaMemcpyDeviceToHost);
        long long bad = 0;
        for (unsigned char c : g) bad += c != 0xC5;
        return bad;
    }
    template <class T> T* as() const { return static_cast<T*>(p); }
};

struct HostBuf {  // pinned
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
    template <class T> T* as() const { return static_cast<T*>(p); }
};

}  // namespace

struct pmb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    std::string err;

    // options
    int64_t opt_chunk_nodes = 0;      // 0 = choose from the tile count
    int64_t opt_staging_records = 0;  // 0 = choose from the problem size
    int64_t opt_inline_nodes = 3;     // light subtrees up to this size are evaluated inside the parent's chunk
    int64_t opt_schedule = 1;         // 1 = persistent kernels with dependency flags, 0 = one launch per level
    int64_t opt_trace = 0;            // debug: record a per-item timeline (pmb_debug_trace)
    DevBuf d_trace;
    std::vector<unsigned long long> h_trace;
    DevBuf d_scan_state;              // compaction: group prefixes (u64) followed by group totals (u32)
    int64_t opt_target_items = 0;     // (chunk, tile) work items aimed for when the chunk size is chosen (0 = default)
    int64_t opt_reserve_sms = 0;      // SMs the persistent kernels leave free (room for a concurrent NCCL kernel)
    int64_t opt_bwd_tail = 20;        // tenths of a machine-full of warps whose items form the backward pass' sorted tail
    int64_t opt_col_groups = 0;       // column-tile groups run on separate streams (0 = chosen from the tile count)
    static constexpr int MAX_GROUPS = 16;
    cudaStream_t gstream[MAX_GROUPS] = {};
    cudaEvent_t gev_fwd[MAX_GROUPS] = {}, gev_done[MAX_GROUPS] = {}, ev_fork = nullptr;
    cudaEvent_t ev_slab_copied[2] = {nullptr, nullptr}, ev_slab_packed[2] = {nullptr, nullptr};
    int n_sms = 0;
    size_t total_mem = 0;
    struct Occupancy { const void* kernel; size_t smem; int per_sm; };
    std::vector<Occupancy> occupancy;
    unsigned int epoch = 0;
    unsigned int dir_clean_epoch = 0;  // epoch at which the staging directory was last cleared (0 = never)
    unsigned int dir2_clean_epoch = 0; // the same for the second directory (double-buffered staging, see run_impl)
    bool sticky_dirty = false;         // a synchronous run left a status bit in the sticky words that pmb_wait must not see
    bool state_dirty = true;           // per-run device state (counters, tickets, node counts, directory) must be re-initialised
    unsigned int pack_seq = 0;
    bool async_pending = false;
    bool upload_pending = false;       // pmb_upload_nuc_async: borrowed input buffers are still being read
    // Compaction runs on a stream of its own: the pass after it starts its forward kernel at once and the compaction
    // kernels fill the SMs that kernel leaves idle while it drains through the top of the tree; only the NEXT backward
    // kernel (which refills the staging pool and the directory) waits for them.
    cudaStream_t cstream = nullptr;
    // The backward kernel has a stream of its own as well: with a second set matrix (small problems only, opt_overlap) the
    // forward kernel of pass i + 1 runs beside the backward kernel of pass i and fills the SMs that one leaves idle while it
    // drains. Order: fwd(i) -> bwd(i) -> compact(i); bwd(i) also after compact(i - 1) (staging pool, directory); fwd(i)
    // after compact(i - 2) (same set matrix and ticket set), or after bwd(i - 1) when there is only one set matrix.
    cudaStream_t bstream = nullptr;
    cudaEvent_t ev_fwd_done = nullptr, ev_bwd_done = nullptr, ev_compact_done[2] = {nullptr, nullptr};
    DevBuf d_sets2, d_dir2, d_staging2;
    int64_t opt_grid_pct = 0;             // persistent kernels take at most this share of the resident block slots (0 = auto)
    int cur_grid_pct = 100;
    int64_t opt_overlap = 1;              // 1 = double-buffer the set matrix when it is small enough (see run_impl)
    unsigned int run_seq = 0;             // parity selects the ticket set of a run
    cudaStream_t merge_stream = nullptr;  // stream of the last pmb_merge_packed (never owned)
    cudaEvent_t ev_merge = nullptr, ev_rm = nullptr;
    cudaStream_t rm_stream = nullptr;     // stream of the last pmb_merge_runs
    DevBuf d_merge_err, d_mblock_sums, d_mrel;
    bool async_phase_events = true;
    int async_groups = 1;

    // tree
    bool have_tree = false;
    int32_t n_nodes = 0, root = -1;
    std::vector<int32_t> child_off, child_idx, leaf_row;
    TreeProgram prog;
    int32_t prog_chunk_nodes = -1, prog_inline_nodes = -1, prog_tail = -1;
    // Programs built for other tile counts of the SAME tree (chunk size and backward tail follow the tile count): a PanGraph
    // build issues one batch per block, each of another width; without the cache every batch would rebuild and re-upload
    // the program (O(N log N) on the host + nine copies). A handful of entries, least recently used goes first.
    struct ProgramSlot {
        int32_t k = -1, inl = -1, tail = -1;
        unsigned long long used = 0;
        TreeProgram prog;
        DevBuf bufs[9];
    };
    std::vector<ProgramSlot> prog_cache;
    unsigned long long prog_clock = 0;
    static constexpr size_t PROG_CACHE_SLOTS = 6;
    DevBuf d_fwd_ops, d_refs, d_bwd_ops, d_bwd_leaves, d_chunks, d_bwd_order, d_level_order, d_row_slot, d_deps;

    // resident input
    bool have_input = false;
    int64_t n_cols = 0, col_base = 0;
    int32_t T = 0;
    bool have_present = false;
    DevBuf d_leaf_planes, d_present, d_colparams, d_tmp_codes, d_tmp_cols;
    // Second pass lane. A small problem's pass is a chain of dependent hops, not a stream of bytes: two INDEPENDENT pipelines
    // side by side fill the machine where one cannot (measured with two contexts, tools/lanes_probe.py: 10k leaves x 15 tiles
    // 0.185 -> 0.149 ms per pass, 20k x 30 tiles 0.534 -> 0.503). `lane` is a child context that owns everything a pass writes
    // (set matrices, flags, staging, lists, streams) and borrows what a pass only reads (program, leaf planes, column
    // parameters) from this one; asynchronous passes alternate between the two, results are read from the one that ran last.
    pmb_ctx* lane = nullptr;
    bool is_lane = false;
    int64_t opt_lanes = 1;                 // 0: never use the second lane
    unsigned lane_seq = 0;                 // asynchronous passes dispatched while lanes were in use
    pmb_ctx* last = nullptr;               // context holding the result of the pass enqueued last (nullptr = this one)
    unsigned long long input_gen = 1, lane_mirror_gen = 0;  // what this context holds / what the lane mirrors of it
    cudaEvent_t ev_input_ready = nullptr;  // end of the last upload on `stream`: a lane pass waits for it
    // clade-run encoded input (pmb_upload_runs): the tree's leaves in depth-first order, the events of the resident range
    std::vector<int32_t> dfs_rows, h_dfs_slot;
    uint64_t dfs_hash = 0;
    DevBuf d_run_events, d_run_off, d_dfs_slot;
    // mutation lists replayed into leaf planes (pmb_upload_replay): pieces, records (keys sorted through two buffers, the spare one
    // then holds the sweep's stacks; code and node per record), events per column, events per (tile, segment) item, CUB scratch
    DevBuf d_rp_pos, d_rp_info, d_rp_nucs, d_rp_poff, d_rp_pre, d_rp_span, d_rp_nbase, d_rp_roff, d_rp_keys[2], d_rp_code, d_rp_rpre,
        d_rp_cnt, d_rp_ev[2], d_rp_tmp;

    // work + result
    DevBuf d_done, d_fdone, d_ticket, d_block_sums;
    DevBuf d_mcounts, d_moff, d_mpos, d_mtc;  // merged shards
    DevBuf d_rm_counts, d_rm_off, d_rm_pos, d_rm_info, d_rm_nucs, d_rm_wire, d_rm_flags, d_rm_oidx;  // run-merge (pmb_merge_runs)
    DevBuf d_col_break;
    bool have_col_break = false;
    HostBuf h_rm_off, h_rm_pos, h_rm_info, h_rm_nucs, h_rm_wire;
    HostBuf h_pack_header;
    DevBuf d_sets, d_fstore, d_states_planes, d_dir, d_staging, d_counters, d_offsets, d_pos, d_tc,
        d_states_u8;
    unsigned long long staging_cap = 0;
    bool staging_floor_dirty = false;
    bool have_result = false;
    int last_algo = 0, last_flags = 0;
    int64_t n_mut = 0;
    pmb_timings timings{};
    HostBuf h_offsets, h_pos, h_tc, h_states, h_counters;
};

namespace {

int fail(pmb_ctx* c, int code, const std::string& msg) {
    if (c) c->err = msg;
    return code;
}

int cuda_fail(pmb_ctx* c, cudaError_t e, const char* what) {
    std::string m = std::string(what) + ": " + cudaGetErrorString(e);
    cudaGetLastError();
    return fail(c, e == cudaErrorMemoryAllocation ? PMB_ERR_OOM : PMB_ERR_CUDA, m);
}

#define PMB_CUDA(call)                                         \
    do {                                                       \
        cudaError_t e__ = (call);                              \
        if (e__ != cudaSuccess) return cuda_fail(c, e__, #call); \
    } while (0)

template <class T>
int upload_vec(pmb_ctx* c, DevBuf& buf, const std::vector<T>& v) {
    size_t bytes = std::max<size_t>(v.size() * sizeof(T), 16);
    PMB_CUDA(buf.ensure(bytes));
    if (!v.empty()) PMB_CUDA(cudaMemcpyAsync(buf.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, c->stream));
    return PMB_OK;
}

// The chunk size trades tree-level parallelism against per-chunk scheduling overhead: aim for enough
// (chunk x tile) warps to fill 148 SMs several times over at the widest level.
int32_t pick_chunk_nodes(const pmb_ctx* c) {
    if (c->opt_chunk_nodes > 0) return int32_t(std::min<int64_t>(c->opt_chunk_nodes, 1 << 30));
    const int64_t target_warps = c->opt_target_items > 0 ? c->opt_target_items : 148LL * 32;  // measured: tools/sweep.py
    int64_t want_chunks = std::max<int64_t>(1, (target_warps + c->T - 1) / std::max(1, c->T));
    int64_t n_internal = 0;
    for (int32_t v = 0; v < c->n_nodes; v++) n_internal += c->child_off[v + 1] > c->child_off[v];
    // Few column tiles: more than ~160 chunks only deepen the chunk tree -- every level is a dependent hop between warps --
    // and consecutive passes of such small problems overlap anyway (second set matrix), so the items they would add are
    // not missed (measured, tools/sweep.py: 10k leaves x 15 tiles 0.201 -> 0.187 ms per pipelined pass at 62 instead of 31
    // ops per chunk; 20k leaves x 30 tiles unchanged at ~126)
    if (c->opt_target_items <= 0 && c->opt_overlap > 0 && size_t(n_internal) * size_t(c->T) * 4096 <= (size_t(4) << 30))
        want_chunks = std::min<int64_t>(want_chunks, 160);
    int64_t k = n_internal / want_chunks;
    // never beyond 512: with thousands of column tiles there are items enough, and a warp walking thousands of ops in
    // one item overflows its parent-state stack into global memory (config 4: 18.8 ms with one 4 000-op chunk, 16.1 ms
    // with chunks of 250 .. 1 000 ops)
    return int32_t(std::max<int64_t>(8, std::min<int64_t>(k, 512)));
}

int ensure_program(pmb_ctx* c) {
    int32_t k = pick_chunk_nodes(c);
    int32_t inl = int32_t(std::max<int64_t>(0, std::min<int64_t>(c->opt_inline_nodes, 1 << 20)));
    // backward tail: enough short items to cover opt_bwd_tail / 10 times the warps the GPU holds at once
    const int64_t resident_warps = int64_t(c->n_sms) * 5 * WARPS_PER_BLOCK;
    const int32_t tail = int32_t(std::min<int64_t>(1 << 30, std::max<int64_t>(0, c->opt_bwd_tail) * resident_warps / 10 / std::max(1, c->T)));
    if (k == c->prog_chunk_nodes && inl == c->prog_inline_nodes && tail == c->prog_tail) return PMB_OK;
    {   // park the current program, look for one built earlier for these parameters
        DevBuf* cur[9] = {&c->d_fwd_ops, &c->d_refs, &c->d_bwd_ops, &c->d_bwd_leaves, &c->d_chunks, &c->d_bwd_order, &c->d_level_order,
                          &c->d_row_slot, &c->d_deps};
        auto swap_with = [&](pmb_ctx::ProgramSlot& s) {
            std::swap(s.prog, c->prog);
            for (int i = 0; i < 9; i++) std::swap(s.bufs[i], *cur[i]);
            std::swap(s.k, c->prog_chunk_nodes);
            std::swap(s.inl, c->prog_inline_nodes);
            std::swap(s.tail, c->prog_tail);
            s.used = ++c->prog_clock;
        };
        if (c->prog_chunk_nodes >= 0) {
            if (c->prog_cache.size() < pmb_ctx::PROG_CACHE_SLOTS) {
                c->prog_cache.emplace_back();
                swap_with(c->prog_cache.back());
            } else {
                size_t lru = 0;
                for (size_t i = 1; i < c->prog_cache.size(); i++)
                    if (c->prog_cache[i].used < c->prog_cache[lru].used) lru = i;
                swap_with(c->prog_cache[lru]);  // the evicted program is now "current" and is overwritten below
                c->prog_chunk_nodes = -1;
            }
        }
        for (size_t i = 0; i < c->prog_cache.size(); i++) {
            pmb_ctx::ProgramSlot& s = c->prog_cache[i];
            if (s.k == k && s.inl == inl && s.tail == tail) {
                swap_with(s);
                if (s.k < 0) {  // what came back is not a program: drop the slot (its buffers are idle: the stream was ordered
                                // behind every earlier pass before the upload got here)
                    for (DevBuf& b : s.bufs) b.release();
                    c->prog_cache.erase(c->prog_cache.begin() + long(i));
                }
                return PMB_OK;
            }
        }
        c->prog_chunk_nodes = -1;
    }
    std::string e = build_tree_program(c->n_nodes, c->root, c->child_off.data(), c->child_idx.data(), c->leaf_row.data(), k,
                                       inl, &c->prog, tail);
    if (e.empty() && c->opt_chunk_nodes <= 0 && c->prog.n_chain_segments > 0 && k > 128) {
        // a deep tree: its chain segments run independently of each other (speculative evaluation), so shorter
        // segments cost nothing in dependencies and balance better (measured: caterpillar 100k x 30k)
        e = build_tree_program(c->n_nodes, c->root, c->child_off.data(), c->child_idx.data(), c->leaf_row.data(), 128, inl, &c->prog,
                               tail);
    }
    if (!e.empty()) return fail(c, PMB_ERR_INVALID, e);
    int rc;
    if ((rc = upload_vec(c, c->d_fwd_ops, c->prog.fwd_ops))) return rc;
    if ((rc = upload_vec(c, c->d_refs, c->prog.refs))) return rc;
    if ((rc = upload_vec(c, c->d_bwd_ops, c->prog.bwd_ops))) return rc;
    if ((rc = upload_vec(c, c->d_bwd_leaves, c->prog.bwd_leaves))) return rc;
    if ((rc = upload_vec(c, c->d_chunks, c->prog.chunks))) return rc;
    if ((rc = upload_vec(c, c->d_bwd_order, c->prog.bwd_order))) return rc;
    if ((rc = upload_vec(c, c->d_level_order, c->prog.level_order))) return rc;
    if ((rc = upload_vec(c, c->d_row_slot, c->prog.row_slot))) return rc;
    if ((rc = upload_vec(c, c->d_deps, c->prog.deps))) return rc;
    PMB_CUDA(cudaStreamSynchronize(c->stream));  // the vectors above may be rebuilt before the copies ran
    c->prog_chunk_nodes = k;
    c->prog_inline_nodes = inl;
    c->prog_tail = tail;
    return PMB_OK;
}

// zero-filled on growth: flag words hold the epoch of the run that published them, epochs start at 1
int ensure_flags(pmb_ctx* c, DevBuf& buf, size_t words) {
    size_t bytes = std::max<size_t>(16, words * sizeof(unsigned int));
    if (bytes <= buf.cap) return PMB_OK;
    PMB_CUDA(buf.ensure(bytes));
    PMB_CUDA(cudaMemsetAsync(buf.p, 0, buf.cap, c->stream));
    return PMB_OK;
}

template <class K>
int launch_kernel(pmb_ctx* c, cudaStream_t stream, K kernel, size_t smem, const RunParams& rp_in, int chunk_begin, int n_chunks,
                  int* n_launches) {
    RunParams rp = rp_in;
    dim3 block(WARPS_PER_BLOCK * 32);
    long long warps = (long long)n_chunks * rp.tile_count;
    if (warps <= 0) return PMB_OK;
    unsigned blocks;
    if (rp.ticket) {
        int per_sm = -1;  // the occupancy query is a driver call: once per (kernel, shared memory size)
        const void* key = reinterpret_cast<const void*>(kernel);
        for (const auto& e : c->occupancy)
            if (e.kernel == key && e.smem == smem) per_sm = e.per_sm;
        if (per_sm < 0) {
            PMB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, WARPS_PER_BLOCK * 32, smem));
            c->occupancy.push_back({key, smem, per_sm});
        }
        const long long sms = std::max<long long>(1, c->n_sms - std::max<int64_t>(0, std::min<int64_t>(c->opt_reserve_sms, c->n_sms - 1)));
        long long resident = (long long)std::max(1, per_sm) * sms;
        resident = std::max<long long>(sms, resident * std::max(1, std::min(100, c->cur_grid_pct)) / 100);
        blocks = unsigned(std::min<long long>(resident, (warps + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK));
        // the ticket is zero: compact_copy_kernel of the previous run (or the initial clearing) left it so
    } else {
        blocks = unsigned((warps + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK);
    }
    kernel<<<blocks, block, smem, stream>>>(rp, chunk_begin, n_chunks);
    (*n_launches)++;
    return PMB_OK;
}

template <class K>
int launch_schedule(pmb_ctx* c, cudaStream_t stream, int ticket_slot, K kernel, size_t smem, RunParams rp, bool forward,
                    int* n_launches) {
    const TreeProgram& P = c->prog;
    int rc;
    if (smem > 48 * 1024) PMB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    if (c->opt_schedule == 1) {
        // persistent: tickets follow chunks[] (forward) or bwd_order (backward), both topological for their pass
        rp.ticket = c->d_ticket.as<unsigned long long>() + ticket_slot;
        rp.order = forward ? nullptr : c->d_bwd_order.as<int>();
        rp.stage_block = 512;
        if ((rc = launch_kernel(c, stream, kernel, smem, rp, 0, int(P.chunks.size()), n_launches))) return rc;
    } else {
        rp.ticket = nullptr;
        rp.order = c->d_level_order.as<int>();
        rp.stage_block = 32;
        const int L = P.n_levels();
        for (int i = 0; i < L; i++) {
            int l = forward ? i : L - 1 - i;
            int cb = P.level_chunk_begin[l], nc = P.level_chunk_begin[l + 1] - cb;
            if ((rc = launch_kernel(c, stream, kernel, smem, rp, cb, nc, n_launches))) return rc;
        }
    }
    PMB_CUDA(cudaGetLastError());
    return PMB_OK;
}

int launch_pass(pmb_ctx* c, cudaStream_t stream, int ticket_slot, const RunParams& rp, int algo, bool forward, int* n_launches) {
    const TreeProgram& P = c->prog;
    const size_t fwd_smem = size_t(WARPS_PER_BLOCK) * (FWD_DEPTH * (2 + 4) * 32 + FWD_META_U4) * sizeof(uint4);
    const size_t fwd_smem_s = size_t(WARPS_PER_BLOCK) * (FWD_DEPTH * (2 + 5) * 32 + FWD_META_U4) * sizeof(uint4);
    const size_t bwd_smem_f = size_t(WARPS_PER_BLOCK) * FITCH_BWD_PER_WARP * sizeof(uint4);  // + the mbarriers of the bulk variant
    const size_t bwd_smem_s = size_t(WARPS_PER_BLOCK) * (BWD_DEPTH * (8 + 2) * 32 + BWD_META_U4 + BWD_STACK_U4) * sizeof(uint4);
    if (algo == PMB_ALGO_FITCH) {
        if (P.n_chain_segments > 0)
            return forward ? launch_schedule(c, stream, ticket_slot, fitch_forward_kernel<true>, fwd_smem, rp, true, n_launches)
                           : launch_schedule(c, stream, ticket_slot, fitch_backward_kernel<true>, bwd_smem_f, rp, false, n_launches);
        return forward ? launch_schedule(c, stream, ticket_slot, fitch_forward_kernel<false>, fwd_smem, rp, true, n_launches)
                       : launch_schedule(c, stream, ticket_slot, fitch_backward_kernel<false>, bwd_smem_f, rp, false, n_launches);
    }
    const bool chains = P.n_chain_segments > 0;
    if (!forward)
        return chains ? launch_schedule(c, stream, ticket_slot, sankoff_backward_kernel<true>, bwd_smem_s, rp, false, n_launches)
                      : launch_schedule(c, stream, ticket_slot, sankoff_backward_kernel<false>, bwd_smem_s, rp, false, n_launches);
#define PMB_SANKOFF_FWD(B)                                                                                                    \
    return chains ? launch_schedule(c, stream, ticket_slot, sankoff_forward_kernel<B, true>, fwd_smem_s, rp, true, n_launches) \
                  : launch_schedule(c, stream, ticket_slot, sankoff_forward_kernel<B, false>, fwd_smem_s, rp, true, n_launches)
    if (P.max_arity <= 3) PMB_SANKOFF_FWD(2);
    if (P.max_arity <= 15) PMB_SANKOFF_FWD(4);
    if (P.max_arity <= 255) PMB_SANKOFF_FWD(8);
    PMB_SANKOFF_FWD(20);
#undef PMB_SANKOFF_FWD
}

// Column tiles are split into groups that run forward -> backward on their own streams: a group's low-parallelism
// phases (the top of the tree at the end of its forward pass and at the start of its backward pass) overlap another
// group's bulk work, and a group's set rows are re-read by its backward pass soon after they were written.
int pick_groups(const pmb_ctx* c) {
    int64_t g = c->opt_col_groups;
    if (g <= 0) g = 1;  // measured (tools/sweep.py): with the critical-path ticket orders one group is as good or better
    g = std::min<int64_t>(g, std::min<int64_t>(c->T, pmb_ctx::MAX_GROUPS));
    return int(std::max<int64_t>(1, g));
}

}  // namespace

extern "C" {

const char* pmb_version(void) { return "panman_b200 0.1 (sm_100a)"; }

int pmb_create(pmb_ctx** out, int device) {
    if (!out) return PMB_ERR_INVALID;
    *out = nullptr;
    pmb_ctx* c = new pmb_ctx();
    c->device = device;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    for (int i = 0; i < 4 && e == cudaSuccess; i++) e = cudaEventCreate(&c->ev[i]);
    if (e != cudaSuccess) {
        // keep the context so that pmb_last_error can say why; every compute call will refuse to run
        c->err = std::string("no usable CUDA device: ") + cudaGetErrorString(e);
        cudaGetLastError();
        c->stream = nullptr;
        *out = c;
        return PMB_ERR_CUDA;
    }
    for (int g = 0; g < pmb_ctx::MAX_GROUPS && e == cudaSuccess; g++) {
        e = cudaStreamCreateWithFlags(&c->gstream[g], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->gev_fwd[g], cudaEventDefault);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->gev_done[g], cudaEventDefault);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_merge, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_fwd_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_bwd_done, cudaEventDisableTiming);
    for (int k = 0; k < 2 && e == cudaSuccess; k++) e = cudaEventCreateWithFlags(&c->ev_compact_done[k], cudaEventDisableTiming);
    if (e == cudaSuccess) {
        int lo = 0, hi = 0;
        e = cudaDeviceGetStreamPriorityRange(&lo, &hi);
        // highest priority: its small kernels take the first SM slots that come free beside a draining pass kernel; the
        // backward kernel (older work) goes before the next pass' forward kernel on the default-priority main stream
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&c->cstream, cudaStreamNonBlocking, hi);
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&c->bstream, cudaStreamNonBlocking, hi < lo ? hi + 1 : hi);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_rm, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_input_ready, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        c->err = std::string("stream/event creation failed: ") + cudaGetErrorString(e);
        cudaGetLastError();
        c->stream = nullptr;
        *out = c;
        return PMB_ERR_CUDA;
    }
    cudaDeviceGetAttribute(&c->n_sms, cudaDevAttrMultiProcessorCount, device);
    if (c->n_sms <= 0) c->n_sms = 148;
    {
        size_t free_b = 0;
        if (cudaMemGetInfo(&free_b, &c->total_mem) != cudaSuccess) {
            cudaGetLastError();
            c->total_mem = size_t(64) << 30;
        }
    }
    *out = c;
    return PMB_OK;
}

// what a lane borrows from its parent (never freed through the lane)
static void lane_borrowed(pmb_ctx* L, DevBuf** out) {
    DevBuf* b[13] = {&L->d_fwd_ops, &L->d_refs, &L->d_bwd_ops, &L->d_bwd_leaves, &L->d_chunks, &L->d_bwd_order, &L->d_level_order,
                     &L->d_row_slot, &L->d_deps, &L->d_leaf_planes, &L->d_present, &L->d_colparams, &L->d_col_break};
    for (int i = 0; i < 13; i++) out[i] = b[i];
}

static void drop_lane(pmb_ctx* c);
void pmb_destroy(pmb_ctx* c) {
    if (!c) return;
    drop_lane(c);
    if (c->stream) {
        cudaSetDevice(c->device);
        cudaStreamSynchronize(c->stream);
        for (DevBuf* b : {&c->d_fwd_ops, &c->d_refs, &c->d_bwd_ops, &c->d_bwd_leaves, &c->d_chunks, &c->d_bwd_order,
                          &c->d_level_order, &c->d_row_slot, &c->d_deps, &c->d_block_sums, &c->d_leaf_planes,
                          &c->d_present, &c->d_colparams, &c->d_tmp_codes, &c->d_tmp_cols, &c->d_sets, &c->d_sets2, &c->d_fstore,
                          &c->d_states_planes, &c->d_dir, &c->d_staging, &c->d_counters, &c->d_offsets,
                          &c->d_pos, &c->d_tc, &c->d_states_u8, &c->d_done, &c->d_fdone, &c->d_ticket, &c->d_mcounts, &c->d_moff,
                          &c->d_mpos, &c->d_mtc, &c->d_scan_state, &c->d_trace, &c->d_rm_counts, &c->d_rm_off, &c->d_rm_pos,
                          &c->d_rm_info, &c->d_rm_nucs, &c->d_rm_wire, &c->d_rm_flags, &c->d_rm_oidx, &c->d_col_break, &c->d_merge_err, &c->d_mblock_sums, &c->d_mrel,
                          &c->d_run_events, &c->d_run_off, &c->d_dfs_slot, &c->d_dir2, &c->d_staging2, &c->d_rp_pos, &c->d_rp_info,
                          &c->d_rp_nucs, &c->d_rp_poff, &c->d_rp_pre, &c->d_rp_span, &c->d_rp_roff, &c->d_rp_keys[0], &c->d_rp_keys[1],
                          &c->d_rp_nbase, &c->d_rp_code, &c->d_rp_rpre, &c->d_rp_cnt, &c->d_rp_ev[0], &c->d_rp_ev[1], &c->d_rp_tmp})
            b->release();
        for (auto& s : c->prog_cache)
            for (DevBuf& b : s.bufs) b.release();
        for (HostBuf* b : {&c->h_offsets, &c->h_pos, &c->h_tc, &c->h_states, &c->h_counters, &c->h_pack_header, &c->h_rm_off, &c->h_rm_pos,
                           &c->h_rm_info, &c->h_rm_nucs, &c->h_rm_wire}) b->release();
        for (int i = 0; i < 4; i++)
            if (c->ev[i]) cudaEventDestroy(c->ev[i]);
        for (int g = 0; g < pmb_ctx::MAX_GROUPS; g++) {
            if (c->gev_fwd[g]) cudaEventDestroy(c->gev_fwd[g]);
            if (c->gev_done[g]) cudaEventDestroy(c->gev_done[g]);
            if (c->gstream[g]) cudaStreamDestroy(c->gstream[g]);
        }
        if (c->ev_fork) cudaEventDestroy(c->ev_fork);
        if (c->ev_merge) cudaEventDestroy(c->ev_merge);
        if (c->bstream) cudaStreamSynchronize(c->bstream);
        if (c->cstream) cudaStreamSynchronize(c->cstream);
        if (c->ev_fwd_done) cudaEventDestroy(c->ev_fwd_done);
        if (c->ev_bwd_done) cudaEventDestroy(c->ev_bwd_done);
        for (int k = 0; k < 2; k++)
            if (c->ev_compact_done[k]) cudaEventDestroy(c->ev_compact_done[k]);
        if (c->cstream) cudaStreamDestroy(c->cstream);
        if (c->bstream) cudaStreamDestroy(c->bstream);
        if (c->ev_rm) cudaEventDestroy(c->ev_rm);
        if (c->ev_input_ready) cudaEventDestroy(c->ev_input_ready);
        for (int k = 0; k < 2; k++) {
            if (c->ev_slab_copied[k]) cudaEventDestroy(c->ev_slab_copied[k]);
            if (c->ev_slab_packed[k]) cudaEventDestroy(c->ev_slab_packed[k]);
        }
        cudaStreamDestroy(c->stream);
    }
    delete c;
}

const char* pmb_last_error(const pmb_ctx* c) { return c ? c->err.c_str() : "null context"; }

void* pmb_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

void pmb_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

int pmb_set_option(pmb_ctx* c, const char* key, int64_t value) {
    if (!c || !key) return PMB_ERR_INVALID;
    std::string k(key);
    if (k == "chunk_nodes") c->opt_chunk_nodes = value;
    else if (k == "staging_records") {
        c->opt_staging_records = value;
        c->staging_cap = 0;  // takes effect at the next run
    }
    else if (k == "inline_nodes") c->opt_inline_nodes = value;
    else if (k == "schedule") c->opt_schedule = value;
    else if (k == "col_groups") c->opt_col_groups = value;
    else if (k == "bwd_tail") c->opt_bwd_tail = value;
    else if (k == "reserve_sms") c->opt_reserve_sms = value;
    else if (k == "target_items") c->opt_target_items = value;
    else if (k == "trace") c->opt_trace = value;
    else if (k == "overlap") c->opt_overlap = value;
    else if (k == "grid_pct") c->opt_grid_pct = value;
    else if (k == "lanes") c->opt_lanes = value;
    else return fail(c, PMB_ERR_INVALID, "unknown option " + k);
    return PMB_OK;
}

static int set_tree_impl(pmb_ctx* c, int32_t n_nodes, int32_t root, const int32_t* child_offsets, const int32_t* child_index,
                         const int32_t* leaf_row) {
    if (!c) return PMB_ERR_INVALID;
    if (!c->stream) return fail(c, PMB_ERR_CUDA, "no usable CUDA device (pmb_create failed); there is no CPU fallback");
    if (n_nodes < 2 || !child_offsets || !child_index || !leaf_row) return fail(c, PMB_ERR_INVALID, "bad tree arguments");
    // validate with a throw-away build (chunk size does not matter for validity)
    TreeProgram probe;
    std::string e = build_tree_program(n_nodes, root, child_offsets, child_index, leaf_row, 64, 3, &probe);
    if (!e.empty()) return fail(c, PMB_ERR_INVALID, e);
    c->n_nodes = n_nodes;
    c->root = root;
    c->child_off.assign(child_offsets, child_offsets + n_nodes + 1);
    c->child_idx.assign(child_index, child_index + child_offsets[n_nodes]);
    c->leaf_row.assign(leaf_row, leaf_row + n_nodes);
    c->dfs_rows = dfs_leaf_rows(n_nodes, root, child_offsets, child_index, leaf_row);
    c->dfs_hash = leaf_order_hash(c->dfs_rows);
    c->prog = std::move(probe);
    c->prog_chunk_nodes = -1;  // (re)built for the tile count at upload time
    if (!c->prog_cache.empty()) {  // programs of the previous tree
        cudaDeviceSynchronize();
        for (auto& s : c->prog_cache)
            for (DevBuf& b : s.bufs) b.release();
        c->prog_cache.clear();
    }
    c->have_tree = true;
    c->have_input = false;
    c->have_result = false;
    c->last = nullptr;
    c->input_gen++;
    if (c->lane && c->lane->stream) {  // its passes belong to the previous tree
        cudaStreamSynchronize(c->lane->stream);
        cudaStreamSynchronize(c->lane->bstream);
        cudaStreamSynchronize(c->lane->cstream);
        c->lane->have_input = false;
        c->lane->have_result = false;
    }
    return PMB_OK;
}

// The C ABI never lets an exception out: host allocations (tree program, staging vectors) that fail come back as codes.
#define PMB_GUARDED(c, expr)                                                       \
    try {                                                                          \
        return (expr);                                                             \
    } catch (const std::bad_alloc&) {                                              \
        return fail((c), PMB_ERR_OOM, "out of host memory");                       \
    } catch (const std::exception& ex) {                                           \
        return fail((c), PMB_ERR_INVALID, std::string("internal: ") + ex.what()); \
    }

int pmb_set_tree(pmb_ctx* c, int32_t n_nodes, int32_t root, const int32_t* child_offsets, const int32_t* child_index,
                 const int32_t* leaf_row) {
    PMB_GUARDED(c, set_tree_impl(c, n_nodes, root, child_offsets, child_index, leaf_row))
}

// pmb_upload_replay's input (host memory) and what its host-side check derives from it
struct ReplayInput {
    int32_t n_nodes, root;
    const int32_t *child_off, *child_idx, *leaf_row;
    const int64_t* piece_off;
    const int32_t* pos;
    const uint8_t* info;
    const uint32_t* nucs;
    int32_t root_leaf_row;
};
struct ReplayPlan {
    std::vector<int32_t> pre_of, dfs_rows;  // node -> pre-order index; leaf rows in depth-first order
    std::vector<int2> span;                 // pre-order index -> [first, end) of its leaves in depth-first order
    std::vector<int64_t> node_base;         // node -> number of its first record, records numbered pre-order-major
    int32_t tip_pos = -1;                   // depth-first position of root_leaf_row
    int64_t n_pieces = 0, n_rec = 0;
};

// Everything pmb_upload_replay refuses is found here, before anything is enqueued. Returns "" or the reason.
static std::string replay_check(const ReplayInput& in, int32_t n_rows, int64_t n_cols, ReplayPlan* P) {
    const int32_t n = in.n_nodes;
    if (n < 2 || in.root < 0 || in.root >= n || !in.child_off || !in.child_idx || !in.leaf_row || !in.piece_off)
        return "bad old tree arguments";
    if (in.child_off[0] != 0 || in.child_off[n] != n - 1) return "old tree: child_offsets must start at 0 and hold n_nodes - 1 children";
    {
        std::vector<char> seen(size_t(n), 0);
        for (int32_t v = 0; v < n; v++) {
            if (in.child_off[v + 1] < in.child_off[v]) return "old tree: child_offsets not monotone";
            for (int32_t e = in.child_off[v]; e < in.child_off[v + 1]; e++) {
                const int32_t ch = in.child_idx[e];
                if (ch < 0 || ch >= n || ch == in.root || seen[size_t(ch)]) return "old tree: child_index is not a tree";
                seen[size_t(ch)] = 1;
            }
        }
    }
    // depth-first walk from the root (children in stored order): pre-order index and leaf interval of every node
    P->pre_of.assign(size_t(n), -1);
    P->span.assign(size_t(n), make_int2(0, 0));
    P->dfs_rows.clear();
    std::vector<char> row_seen(size_t(n_rows), 0);
    std::vector<std::pair<int32_t, int32_t>> st;  // (node, next child edge)
    int32_t n_pre = 0;
    auto enter = [&](int32_t v) -> bool {
        const int32_t pre = n_pre++;
        P->pre_of[size_t(v)] = pre;
        P->span[size_t(pre)].x = int32_t(P->dfs_rows.size());
        if (in.child_off[v] == in.child_off[v + 1]) {
            const int32_t r = in.leaf_row[v];
            if (r < 0 || r >= n_rows || row_seen[size_t(r)]) return false;
            row_seen[size_t(r)] = 1;
            P->dfs_rows.push_back(r);
            P->span[size_t(pre)].y = int32_t(P->dfs_rows.size());
        } else {
            if (in.leaf_row[v] != -1) return false;
            st.emplace_back(v, in.child_off[v]);
        }
        return true;
    };
    if (in.child_off[in.root] == in.child_off[in.root + 1]) return "old tree: the root must be an internal node";
    enter(in.root);
    while (!st.empty()) {
        auto& f = st.back();
        if (f.second < in.child_off[f.first + 1]) {
            if (!enter(in.child_idx[f.second++])) return "old tree: its leaf rows are not the rows of the tree set on the context";
        } else {
            P->span[size_t(P->pre_of[size_t(f.first)])].y = int32_t(P->dfs_rows.size());
            st.pop_back();
        }
    }
    if (n_pre != n) return "old tree: not connected";
    if (int32_t(P->dfs_rows.size()) != n_rows) return "old tree: its leaf rows are not the rows of the tree set on the context";
    if (in.root_leaf_row < -1 || in.root_leaf_row >= n_rows) return "root_leaf_row is not a row of the tree";
    P->tip_pos = -1;
    for (int32_t i = 0; i < n_rows && in.root_leaf_row >= 0; i++)
        if (P->dfs_rows[size_t(i)] == in.root_leaf_row) P->tip_pos = i;
    // pieces: NucMut fields, node-major
    if (in.piece_off[0] != 0) return "piece_offsets must start at 0";
    for (int32_t v = 0; v < n; v++)
        if (in.piece_off[v + 1] < in.piece_off[v]) return "piece_offsets not monotone";
    P->n_pieces = in.piece_off[n];
    if (P->n_pieces > 0 && (!in.pos || !in.info || !in.nucs)) return "null piece arrays";
    std::vector<int64_t> by_pre(size_t(n), 0);  // records per node, at its pre-order index
    for (int32_t v = 0; v < n; v++)
        for (int64_t k = in.piece_off[v]; k < in.piece_off[v + 1]; k++) {
            const int type = in.info[k] & 15, len = in.info[k] >> 4;
            if (type > 2) return "piece " + std::to_string(k) + ": type " + std::to_string(type) + " (only NS 0, ND 1, NI 2)";
            if (len < 1 || len > 6) return "piece " + std::to_string(k) + ": length " + std::to_string(len) + " (1 .. 6)";
            if (in.pos[k] < 0 || int64_t(in.pos[k]) + len > n_cols) return "piece " + std::to_string(k) + ": positions beyond n_cols";
            by_pre[size_t(P->pre_of[size_t(v)])] += len;
        }
    P->n_rec = 0;
    for (int64_t& x : by_pre) {
        const int64_t cnt = x;
        x = P->n_rec;
        P->n_rec += cnt;
    }
    if (P->n_rec >= (int64_t(1) << 32)) return "more than 2^32 piece positions";
    P->node_base.resize(size_t(n));
    for (int32_t v = 0; v < n; v++) P->node_base[size_t(v)] = by_pre[size_t(P->pre_of[size_t(v)])];
    return "";
}

extern "C++" {
template <class F>
static int with_cub_scratch(pmb_ctx* c, F f) {  // f(temp, bytes): a CUB device call, sized first
    size_t bytes = 0;
    PMB_CUDA(f(nullptr, bytes));
    PMB_CUDA(c->d_rp_tmp.ensure(std::max<size_t>(bytes, 16)));
    PMB_CUDA(f(c->d_rp_tmp.p, bytes));
    return PMB_OK;
}
}

static unsigned blocks_for(long long n) { return unsigned(std::max<long long>(1, (n + 255) / 256)); }

// Replay kernels on c->stream: pieces -> sorted records -> per-column sweep (counted, then written) -> events sorted into
// (tile, segment) items in c->d_run_events / c->d_run_off, the layout expand_runs_kernel reads. d_parent: the parent codes on
// the device; d_tip (or NULL): receives the code of the leaf at P.tip_pos in every column.
static int replay_events(pmb_ctx* c, const ReplayInput& in, const ReplayPlan& P, int64_t n_cols, int32_t n_rows, int32_t n_seg,
                         int32_t seg_rows, const uint8_t* d_parent, int8_t* d_tip) {
    cudaStream_t s = c->stream;
    const int32_t n = in.n_nodes;
    const long long NP = P.n_pieces, R = P.n_rec;
    int rec_bits = 1, col_bits = 1;
    while ((1LL << rec_bits) < R) rec_bits++;
    while ((1LL << col_bits) <= n_cols) col_bits++;  // column + 1 <= n_cols < 2^31: rec_bits + col_bits <= 64
    PMB_CUDA(c->d_rp_poff.ensure(size_t(n + 1) * sizeof(long long)));
    PMB_CUDA(c->d_rp_pre.ensure(size_t(n) * sizeof(int)));
    PMB_CUDA(c->d_rp_span.ensure(size_t(n) * sizeof(int2)));
    PMB_CUDA(c->d_rp_nbase.ensure(size_t(n) * sizeof(long long)));
    PMB_CUDA(cudaMemcpyAsync(c->d_rp_poff.p, in.piece_off, size_t(n + 1) * sizeof(long long), cudaMemcpyHostToDevice, s));
    PMB_CUDA(cudaMemcpyAsync(c->d_rp_pre.p, P.pre_of.data(), size_t(n) * sizeof(int), cudaMemcpyHostToDevice, s));
    PMB_CUDA(cudaMemcpyAsync(c->d_rp_span.p, P.span.data(), size_t(n) * sizeof(int2), cudaMemcpyHostToDevice, s));
    PMB_CUDA(cudaMemcpyAsync(c->d_rp_nbase.p, P.node_base.data(), size_t(n) * sizeof(long long), cudaMemcpyHostToDevice, s));
    PMB_CUDA(c->d_rp_cnt.ensure(size_t(std::max<long long>(NP, n_cols + 1)) * sizeof(long long)));
    PMB_CUDA(c->d_rp_roff.ensure(size_t(std::max<long long>(NP, n_cols + 1)) * sizeof(long long)));
    for (int k = 0; k < 2; k++) PMB_CUDA(c->d_rp_keys[k].ensure(size_t(std::max<long long>(R, 2)) * sizeof(unsigned long long)));
    PMB_CUDA(c->d_rp_code.ensure(size_t(std::max<long long>(R, 16))));
    PMB_CUDA(c->d_rp_rpre.ensure(size_t(std::max<long long>(R, 4)) * sizeof(int)));
    cub::DoubleBuffer<unsigned long long> keys(c->d_rp_keys[0].as<unsigned long long>(), c->d_rp_keys[1].as<unsigned long long>());
    int rc;
    if (NP > 0) {
        PMB_CUDA(c->d_rp_pos.ensure(size_t(NP) * sizeof(int32_t)));
        PMB_CUDA(c->d_rp_info.ensure(size_t(NP)));
        PMB_CUDA(c->d_rp_nucs.ensure(size_t(NP) * sizeof(uint32_t)));
        PMB_CUDA(cudaMemcpyAsync(c->d_rp_pos.p, in.pos, size_t(NP) * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        PMB_CUDA(cudaMemcpyAsync(c->d_rp_info.p, in.info, size_t(NP), cudaMemcpyHostToDevice, s));
        PMB_CUDA(cudaMemcpyAsync(c->d_rp_nucs.p, in.nucs, size_t(NP) * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
        long long* len = c->d_rp_cnt.as<long long>();
        long long* roff = c->d_rp_roff.as<long long>();
        replay_piece_len_kernel<<<blocks_for(NP), 256, 0, s>>>(c->d_rp_info.as<uint8_t>(), NP, len);
        if ((rc = with_cub_scratch(c, [&](void* t, size_t& b) { return cub::DeviceScan::ExclusiveSum(t, b, len, roff, NP, s); }))) return rc;
        replay_records_kernel<<<blocks_for(NP), 256, 0, s>>>(c->d_rp_poff.as<long long>(), n, c->d_rp_nbase.as<long long>(), c->d_rp_pre.as<int>(),
                                                             c->d_rp_pos.as<int32_t>(), c->d_rp_info.as<uint8_t>(), c->d_rp_nucs.as<uint32_t>(), NP,
                                                             roff, rec_bits, keys.Current(), c->d_rp_code.as<uint8_t>(), c->d_rp_rpre.as<int>());
        PMB_CUDA(cudaGetLastError());
        if ((rc = with_cub_scratch(c, [&](void* t, size_t& b) {
                 return cub::DeviceRadixSort::SortKeys(t, b, keys, R, 0, rec_bits + col_bits, s);
             })))
            return rc;
    }
    // count the events of every column, offsets by an exclusive scan over n_cols + 1 counts (the last one 0: the total)
    long long* cnt = c->d_rp_cnt.as<long long>();
    long long* ev_off = c->d_rp_roff.as<long long>();
    PMB_CUDA(cudaMemsetAsync(cnt + n_cols, 0, sizeof(long long), s));
    replay_sweep_kernel<false><<<blocks_for(n_cols), 256, 0, s>>>(keys.Current(), c->d_rp_code.as<uint8_t>(), c->d_rp_rpre.as<int>(), R, rec_bits, c->d_rp_span.as<int2>(), d_parent,
                                                                  n_cols, n_rows, n_seg, seg_rows, P.tip_pos, keys.Alternate(), cnt,
                                                                  nullptr, nullptr, nullptr);
    PMB_CUDA(cudaGetLastError());
    if ((rc = with_cub_scratch(c, [&](void* t, size_t& b) { return cub::DeviceScan::ExclusiveSum(t, b, cnt, ev_off, n_cols + 1, s); })))
        return rc;
    long long E = 0;
    PMB_CUDA(cudaMemcpyAsync(&E, ev_off + n_cols, sizeof(long long), cudaMemcpyDeviceToHost, s));
    PMB_CUDA(cudaStreamSynchronize(s));
    for (int k = 0; k < 2; k++) PMB_CUDA(c->d_rp_ev[k].ensure(size_t(std::max<long long>(E, 2)) * sizeof(unsigned long long)));
    cub::DoubleBuffer<unsigned long long> ev(c->d_rp_ev[0].as<unsigned long long>(), c->d_rp_ev[1].as<unsigned long long>());
    replay_sweep_kernel<true><<<blocks_for(n_cols), 256, 0, s>>>(keys.Current(), c->d_rp_code.as<uint8_t>(), c->d_rp_rpre.as<int>(), R, rec_bits, c->d_rp_span.as<int2>(), d_parent,
                                                                 n_cols, n_rows, n_seg, seg_rows, P.tip_pos, keys.Alternate(), nullptr, ev_off,
                                                                 ev.Current(), d_tip);
    PMB_CUDA(cudaGetLastError());
    const long long n_items = (long long)c->T * n_seg;
    int item_bits = 1;
    while ((1LL << item_bits) <= n_items) item_bits++;
    if (E > 0 && (rc = with_cub_scratch(c, [&](void* t, size_t& b) { return cub::DeviceRadixSort::SortKeys(t, b, ev, E, 0, 32 + item_bits, s); })))
        return rc;
    PMB_CUDA(c->d_run_events.ensure(size_t(std::max<long long>(E, 4)) * sizeof(uint32_t)));
    PMB_CUDA(c->d_run_off.ensure(size_t(n_items + 1) * sizeof(long long)));
    replay_items_kernel<<<blocks_for(std::max(E, n_items + 1)), 256, 0, s>>>(ev.Current(), E, n_items, c->d_run_events.as<uint32_t>(),
                                                                            c->d_run_off.as<long long>());
    PMB_CUDA(cudaGetLastError());
    return PMB_OK;
}

// The leaf codes come either as a nibble matrix (leaf_codes_4bit), clade-run encoded (runs, columns from runs_col_begin on) or
// as the mutation lists of a PanMAT replayed over parent_code (replay).
static int upload_impl(pmb_ctx* c, int64_t n_cols, int32_t n_rows, const uint8_t* leaf_codes_4bit, int64_t row_stride_bytes,
                       const uint8_t* leaf_present, const uint8_t* parent_code, const int8_t* root_override,
                       const int8_t* fwd_root_ref, int64_t col_base, bool sync, const pmb_runs* runs = nullptr,
                       int64_t runs_col_begin = 0, const ReplayInput* replay = nullptr) {
    if (!c) return PMB_ERR_INVALID;
    if (!c->stream) return fail(c, PMB_ERR_CUDA, "no usable CUDA device; there is no CPU fallback");
    if (!c->have_tree) return fail(c, PMB_ERR_NO_TREE, "pmb_set_tree has not been called");
    if (n_cols <= 0 || (!leaf_codes_4bit && !runs && !replay) || !parent_code) return fail(c, PMB_ERR_INVALID, "bad input arguments");
    if (n_rows != c->prog.n_rows) return fail(c, PMB_ERR_INVALID, "n_rows does not match the tree's leaf count");
    if (!runs && !replay && row_stride_bytes < (n_cols + 1) / 2) return fail(c, PMB_ERR_INVALID, "row_stride_bytes too small");
    if (runs) {
        if (runs->order_hash != c->dfs_hash || runs->n_rows != n_rows)
            return fail(c, PMB_ERR_INVALID, "the batch was encoded for another tree (leaf order differs)");
        if (runs_col_begin < 0 || runs_col_begin % TILE_COLS != 0 || runs_col_begin + n_cols > runs->n_cols ||
            (runs_col_begin + n_cols != runs->n_cols && n_cols % TILE_COLS != 0))
            return fail(c, PMB_ERR_INVALID, "a column range of an encoded batch starts on a multiple of 1024 and ends on one or with the batch");
    }
    if (n_cols > (int64_t(1) << 40)) return fail(c, PMB_ERR_INVALID, "n_cols too large");
    // positions are int32 (NucMut.nucPosition): every column col_base .. col_base + n_cols - 1 must be one
    if (col_base < 0 || col_base > (int64_t(1) << 31) - n_cols)
        return fail(c, PMB_ERR_INVALID, "col_base + n_cols exceeds 2^31 (or col_base < 0): positions are int32");
    ReplayPlan plan;
    if (replay) {
        const std::string e = replay_check(*replay, n_rows, n_cols, &plan);
        if (!e.empty()) return fail(c, PMB_ERR_INVALID, e);
    }
    PMB_CUDA(cudaSetDevice(c->device));
    // passes still in flight on the backward / compaction streams read what is overwritten here
    PMB_CUDA(cudaStreamWaitEvent(c->stream, c->ev_bwd_done, 0));
    for (int k = 0; k < 2; k++) PMB_CUDA(cudaStreamWaitEvent(c->stream, c->ev_compact_done[k], 0));
    if (c->lane && c->lane->stream) {  // the lane's passes read the same leaf planes and column parameters
        PMB_CUDA(cudaStreamWaitEvent(c->stream, c->lane->ev_bwd_done, 0));
        for (int k = 0; k < 2; k++) PMB_CUDA(cudaStreamWaitEvent(c->stream, c->lane->ev_compact_done[k], 0));
    }
    c->last = nullptr;
    c->input_gen++;
    c->have_input = false;
    c->have_result = false;
    c->have_col_break = false;
    c->staging_floor_dirty = true;  // the pool keeps what it has grown to; the default for the new size is a lower bound
    c->n_cols = n_cols;
    c->col_base = col_base;
    c->T = int32_t((n_cols + TILE_COLS - 1) / TILE_COLS);
    int rc = ensure_program(c);
    if (rc) return rc;
    const size_t plane_bytes = size_t(n_rows) * c->T * 32 * sizeof(uint4);
    PMB_CUDA(c->d_leaf_planes.ensure(plane_bytes));
    PMB_CUDA(c->d_tmp_cols.ensure(size_t(n_cols) * 3));
    uint8_t* t = c->d_tmp_cols.as<uint8_t>();
    PMB_CUDA(cudaMemcpyAsync(t, parent_code, size_t(n_cols), cudaMemcpyDefault, c->stream));
    if (root_override) PMB_CUDA(cudaMemcpyAsync(t + n_cols, root_override, size_t(n_cols), cudaMemcpyDefault, c->stream));
    if (fwd_root_ref) PMB_CUDA(cudaMemcpyAsync(t + 2 * n_cols, fwd_root_ref, size_t(n_cols), cudaMemcpyDefault, c->stream));
    int32_t rp_seg = 0, rp_seg_rows = 0;
    if (replay) {  // the tip's replayed codes become the root override
        runs_segments(n_rows, c->T, &rp_seg, &rp_seg_rows);
        const bool tip = replay->root_leaf_row >= 0;
        if ((rc = replay_events(c, *replay, plan, n_cols, n_rows, rp_seg, rp_seg_rows, t, tip ? reinterpret_cast<int8_t*>(t + n_cols) : nullptr)))
            return rc;
        if (tip) root_override = reinterpret_cast<const int8_t*>(t + n_cols);
    }
    PMB_CUDA(c->d_colparams.ensure(size_t(c->T) * 128 * sizeof(uint4)));
    {
        long long threads = (long long)c->T * 32 * 32;
        unsigned blocks = unsigned((threads + 255) / 256);
        pack_colparams_kernel<<<blocks, 256, 0, c->stream>>>(t, root_override ? reinterpret_cast<const int8_t*>(t + n_cols) : nullptr,
                                                             fwd_root_ref ? reinterpret_cast<const int8_t*>(t + 2 * n_cols) : nullptr,
                                                             n_cols, c->T, c->d_colparams.as<uint4>());
    }
    PMB_CUDA(cudaGetLastError());
    // Where does the nibble matrix live? Device memory and pinned (or registered) host memory are read by the packing
    // kernel in place -- for pinned memory that fuses the host-to-device transfer with the transposition, one pass at
    // PCIe speed and no staging buffer. Pageable host memory is staged through a bounded device buffer.
    // Device memory is read by the packing kernel in place. Host memory is staged through two slabs of device memory:
    // the copy engine fills one (on a side stream) while the kernel transposes the other, so the upload runs at the
    // speed of the PCIe copy alone (measured on B200: the kernel reading pinned memory in place reaches 47 GB/s, the copy
    // engine 54 GB/s; tools/e2e_breakdown.py). Pageable memory takes the same path at the driver's staging speed.
    bool on_device = false;
    if (!runs && !replay) {
        cudaPointerAttributes attr{};
        if (cudaPointerGetAttributes(&attr, leaf_codes_4bit) == cudaSuccess)
            on_device = attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged;
        else
            cudaGetLastError();
    }
    auto pack = [&](const uint8_t* src, int64_t src_stride, int32_t r0, int32_t nr) {
        long long total = (long long)nr * c->T * 32;
        unsigned blocks = unsigned((total + 255) / 256);
        pack_leaves_kernel<<<blocks, 256, 0, c->stream>>>(src, src_stride, r0, nr, n_rows, n_cols, c->T, c->d_row_slot.as<int>(),
                                                          c->d_leaf_planes.as<uint4>());
    };
    if (runs) {
        // events of the range's tiles -> device, then one kernel rebuilds the planes the dense path would have packed
        const long long n_items = (long long)c->T * runs->n_seg, item0 = (runs_col_begin / TILE_COLS) * runs->n_seg;
        const long long ev_base = runs->item_off[item0], n_ev = runs->item_off[item0 + n_items] - ev_base;
        PMB_CUDA(c->d_run_events.ensure(size_t(std::max<long long>(n_ev, 4)) * sizeof(uint32_t)));
        PMB_CUDA(c->d_run_off.ensure(size_t(n_items + 1) * sizeof(long long)));
        PMB_CUDA(c->d_dfs_slot.ensure(size_t(n_rows) * sizeof(int)));
        c->h_dfs_slot.resize(size_t(n_rows));
        for (int32_t i = 0; i < n_rows; i++) c->h_dfs_slot[size_t(i)] = c->prog.row_slot[size_t(c->dfs_rows[size_t(i)])];
        PMB_CUDA(cudaMemcpyAsync(c->d_run_off.p, runs->item_off + item0, size_t(n_items + 1) * sizeof(long long), cudaMemcpyHostToDevice, c->stream));
        PMB_CUDA(cudaMemcpyAsync(c->d_dfs_slot.p, c->h_dfs_slot.data(), size_t(n_rows) * sizeof(int), cudaMemcpyHostToDevice, c->stream));
        // the events cross the link in a few slabs of whole tiles on the copy stream, each expanded as soon as it is there
        const int n_slabs = int(std::max<long long>(1, std::min<long long>(std::min<long long>(8, c->T), n_ev * 4 / (4 << 20))));
        cudaStream_t copy = c->gstream[0];
        for (int k = 0; k < 2; k++)
            if (!c->ev_slab_copied[k]) PMB_CUDA(cudaEventCreateWithFlags(&c->ev_slab_copied[k], cudaEventDisableTiming));
        PMB_CUDA(cudaEventRecord(c->ev_fork, c->stream));  // the event buffer may still be read by an earlier expansion
        PMB_CUDA(cudaStreamWaitEvent(copy, c->ev_fork, 0));
        for (int sl = 0; sl < n_slabs; sl++) {
            const long long ia = (long long)c->T * sl / n_slabs * runs->n_seg, ib = (long long)c->T * (sl + 1) / n_slabs * runs->n_seg;
            const long long ea = runs->item_off[item0 + ia] - ev_base, eb = runs->item_off[item0 + ib] - ev_base;
            if (eb > ea) {
                PMB_CUDA(cudaMemcpyAsync(c->d_run_events.as<uint32_t>() + ea, runs->events + ev_base + ea, size_t(eb - ea) * sizeof(uint32_t),
                                         cudaMemcpyHostToDevice, copy));
                PMB_CUDA(cudaEventRecord(c->ev_slab_copied[sl & 1], copy));
                PMB_CUDA(cudaStreamWaitEvent(c->stream, c->ev_slab_copied[sl & 1], 0));
            }
            if (ib > ia) {
                const unsigned blocks = unsigned(((ib - ia) * 32 + 255) / 256);
                expand_runs_kernel<<<blocks, 256, 0, c->stream>>>(c->d_run_events.as<uint32_t>(), c->d_run_off.as<long long>(), ev_base, ia, ib,
                                                                  runs->n_seg, runs->seg_rows, n_rows, c->d_dfs_slot.as<int>(),
                                                                  c->d_colparams.as<uint4>(), c->d_leaf_planes.as<uint4>());
            }
        }
        PMB_CUDA(cudaEventRecord(c->ev_fork, copy));  // a later upload's copies into these buffers are ordered behind c->stream anyway;
        PMB_CUDA(cudaStreamWaitEvent(c->stream, c->ev_fork, 0));  // this joins the copy stream so that a wait on c->stream covers it
    } else if (replay) {
        PMB_CUDA(c->d_dfs_slot.ensure(size_t(n_rows) * sizeof(int)));
        c->h_dfs_slot.resize(size_t(n_rows));
        for (int32_t i = 0; i < n_rows; i++) c->h_dfs_slot[size_t(i)] = c->prog.row_slot[size_t(plan.dfs_rows[size_t(i)])];
        PMB_CUDA(cudaMemcpyAsync(c->d_dfs_slot.p, c->h_dfs_slot.data(), size_t(n_rows) * sizeof(int), cudaMemcpyHostToDevice, c->stream));
        const long long n_items = (long long)c->T * rp_seg;
        expand_runs_kernel<<<blocks_for(n_items * 32), 256, 0, c->stream>>>(c->d_run_events.as<uint32_t>(), c->d_run_off.as<long long>(), 0, 0, n_items,
                                                                            rp_seg, rp_seg_rows, n_rows, c->d_dfs_slot.as<int>(),
                                                                            c->d_colparams.as<uint4>(), c->d_leaf_planes.as<uint4>());
    } else if (on_device) {
        pack(leaf_codes_4bit, row_stride_bytes, 0, n_rows);
    } else {
        // Only the batch's own columns cross the link: a slab holds rows of (n_cols + 1) / 2 bytes at a 16-byte pitch, whatever
        // the caller's row stride is -- a column range of a wider matrix (pmb_group_upload_nuc) is copied as a 2-D region,
        // not with the other ranges' bytes in between (and nothing behind the last row's range is touched).
        const size_t row_bytes = size_t((n_cols + 1) / 2), pitch = (row_bytes + 15) / 16 * 16;
        const size_t slab_budget = size_t(32) << 20;
        const int32_t slab_rows = int32_t(std::max<size_t>(1, std::min<size_t>(size_t(n_rows), slab_budget / pitch)));
        const size_t slab_bytes = size_t(slab_rows) * pitch;
        PMB_CUDA(c->d_tmp_codes.ensure(2 * slab_bytes));
        cudaStream_t copy = c->gstream[0];
        for (int k = 0; k < 2; k++) {
            if (!c->ev_slab_copied[k]) PMB_CUDA(cudaEventCreateWithFlags(&c->ev_slab_copied[k], cudaEventDisableTiming));
            if (!c->ev_slab_packed[k]) PMB_CUDA(cudaEventCreateWithFlags(&c->ev_slab_packed[k], cudaEventDisableTiming));
        }
        PMB_CUDA(cudaEventRecord(c->ev_fork, c->stream));  // the staging buffer may still be in use by earlier work
        PMB_CUDA(cudaStreamWaitEvent(copy, c->ev_fork, 0));
        const bool tight = size_t(row_stride_bytes) == pitch;  // rows already lie back to back at the slab's pitch: one flat copy
        int slab = 0;
        for (int32_t r0 = 0; r0 < n_rows; r0 += slab_rows, slab++) {
            const int k = slab & 1;
            const int32_t nr = std::min(slab_rows, n_rows - r0);
            uint8_t* buf = c->d_tmp_codes.as<uint8_t>() + size_t(k) * slab_bytes;
            if (slab >= 2) PMB_CUDA(cudaStreamWaitEvent(copy, c->ev_slab_packed[k], 0));
            const uint8_t* src = leaf_codes_4bit + size_t(r0) * size_t(row_stride_bytes);
            if (tight)
                PMB_CUDA(cudaMemcpyAsync(buf, src, size_t(nr - 1) * pitch + row_bytes, cudaMemcpyHostToDevice, copy));
            else
                PMB_CUDA(cudaMemcpy2DAsync(buf, pitch, src, size_t(row_stride_bytes), row_bytes, size_t(nr), cudaMemcpyHostToDevice, copy));
            PMB_CUDA(cudaEventRecord(c->ev_slab_copied[k], copy));
            PMB_CUDA(cudaStreamWaitEvent(c->stream, c->ev_slab_copied[k], 0));
            pack(buf, int64_t(pitch), r0, nr);
            PMB_CUDA(cudaEventRecord(c->ev_slab_packed[k], c->stream));
        }
    }
    PMB_CUDA(cudaGetLastError());
    c->have_present = leaf_present != nullptr;
    if (leaf_present) {  // kernels index presence by leaf slot
        std::vector<uint8_t> tmp(static_cast<size_t>(n_rows)), by_slot(static_cast<size_t>(n_rows));
        PMB_CUDA(cudaMemcpy(tmp.data(), leaf_present, size_t(n_rows), cudaMemcpyDefault));
        for (int32_t r = 0; r < n_rows; r++) by_slot[c->prog.row_slot[r]] = tmp[r];
        PMB_CUDA(c->d_present.ensure(size_t(n_rows)));
        PMB_CUDA(cudaMemcpy(c->d_present.p, by_slot.data(), size_t(n_rows), cudaMemcpyHostToDevice));
    }
    PMB_CUDA(cudaEventRecord(c->ev_input_ready, c->stream));
    if (sync) PMB_CUDA(cudaStreamSynchronize(c->stream));  // inputs were borrowed: they may be released on return
    c->upload_pending = !sync;
    c->have_input = true;
    return PMB_OK;
}

int pmb_upload_nuc(pmb_ctx* c, int64_t n_cols, int32_t n_rows, const uint8_t* leaf_codes_4bit, int64_t row_stride_bytes,
                   const uint8_t* leaf_present, const uint8_t* parent_code, const int8_t* root_override,
                   const int8_t* fwd_root_ref, int64_t col_base) {
    PMB_GUARDED(c, upload_impl(c, n_cols, n_rows, leaf_codes_4bit, row_stride_bytes, leaf_present, parent_code, root_override,
                               fwd_root_ref, col_base, true))
}

int pmb_upload_nuc_async(pmb_ctx* c, int64_t n_cols, int32_t n_rows, const uint8_t* leaf_codes_4bit, int64_t row_stride_bytes,
                         const uint8_t* leaf_present, const uint8_t* parent_code, const int8_t* root_override,
                         const int8_t* fwd_root_ref, int64_t col_base) {
    PMB_GUARDED(c, upload_impl(c, n_cols, n_rows, leaf_codes_4bit, row_stride_bytes, leaf_present, parent_code, root_override,
                               fwd_root_ref, col_base, false))
}

int pmb_upload_replay(pmb_ctx* c, int32_t old_n_nodes, int32_t old_root, const int32_t* old_child_offsets, const int32_t* old_child_index,
                      const int32_t* old_leaf_row, const int64_t* piece_offsets, const int32_t* nuc_position, const uint8_t* mut_info,
                      const uint32_t* nucs, int64_t n_cols, const uint8_t* parent_code, int32_t root_leaf_row) {
    if (!c) return PMB_ERR_INVALID;
    const ReplayInput in{old_n_nodes, old_root, old_child_offsets, old_child_index, old_leaf_row, piece_offsets, nuc_position, mut_info, nucs,
                         root_leaf_row};
    PMB_GUARDED(c, upload_impl(c, n_cols, c->have_tree ? c->prog.n_rows : 0, nullptr, 0, nullptr, parent_code, nullptr, nullptr, 0, true,
                               nullptr, 0, &in))
}

static int run_impl(pmb_ctx* c, int algo, int flags, bool async) {
    if (!c) return PMB_ERR_INVALID;
    if (!c->stream) return fail(c, PMB_ERR_CUDA, "no usable CUDA device; there is no CPU fallback");
    if (!c->have_tree) return fail(c, PMB_ERR_NO_TREE, "pmb_set_tree has not been called");
    if (!c->have_input) return fail(c, PMB_ERR_NO_INPUT, "pmb_upload_nuc has not been called");
    if (algo != PMB_ALGO_FITCH && algo != PMB_ALGO_SANKOFF) return fail(c, PMB_ERR_INVALID, "unknown algo");
    PMB_CUDA(cudaSetDevice(c->device));
    c->have_result = false;
    const TreeProgram& P = c->prog;
    const size_t T = size_t(c->T);
    const size_t set_bytes_per = (algo == PMB_ALGO_FITCH ? 128 : 256) * sizeof(uint4);
    const size_t set_bytes = size_t(P.n_internal) * T * set_bytes_per;
    // a second set matrix lets consecutive passes overlap (see bstream): up to 48 GB and a quarter of the device's memory --
    // BASELINE.json's config 4 whole on one B200 (40 GB; measured on its halves: 0.973 of the roofline overlapping, 0.948
    // without) -- and a large one only where the device clearly has the room for it beside everything else of the pass
    bool overlap = c->opt_overlap > 0 && c->opt_schedule == 1 && pick_groups(c) == 1 && set_bytes <= std::min(size_t(48) << 30, c->total_mem / 4);
    if (overlap && set_bytes > c->d_sets2.cap && set_bytes > (size_t(8) << 30)) {
        size_t free_b = 0, total_b = 0;
        const size_t need = set_bytes + (set_bytes > c->d_sets.cap ? set_bytes - c->d_sets.cap : 0) + (size_t(16) << 30);
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) {
            cudaGetLastError();
            overlap = false;
        } else if (free_b + c->d_sets2.cap < need) {
            overlap = false;
        }
    }
    if (set_bytes > c->d_sets.cap || (overlap && set_bytes > c->d_sets2.cap)) {  // cudaFree of a matrix a running pass uses
        PMB_CUDA(cudaStreamSynchronize(c->bstream));
        PMB_CUDA(cudaStreamSynchronize(c->cstream));
    }
    PMB_CUDA(c->d_sets.ensure(set_bytes));
    if (overlap) PMB_CUDA(c->d_sets2.ensure(set_bytes));
    PMB_CUDA(c->d_fstore.ensure(std::max<size_t>(16, size_t(P.n_fslots) * T * FSLOT_WORDS * sizeof(uint32_t))));
    const bool want_states = flags & PMB_FLAG_WANT_STATES;
    if (want_states) PMB_CUDA(c->d_states_planes.ensure(size_t(P.n_nodes) * T * 64 * sizeof(uint4)));
    const size_t dir_bytes = size_t(P.n_nodes) * T * sizeof(unsigned long long);
    if (dir_bytes > c->d_dir.cap) c->dir_clean_epoch = 0;
    PMB_CUDA(c->d_dir.ensure(dir_bytes));
    // With overlapping passes the staging pool, its directory and the run words are double-buffered too: the backward kernel
    // of pass i then only follows the backward kernel of pass i - 1, not its compaction (a small problem's pass is a chain of
    // dependent hops, and backward -> compaction -> backward was the longest chain through consecutive passes)
    const bool dbl = overlap;
    if (dbl) {
        if (dir_bytes > c->d_dir2.cap) c->dir2_clean_epoch = 0;
        PMB_CUDA(c->d_dir2.ensure(dir_bytes));
    }
    if (!c->d_counters.p) {
        PMB_CUDA(c->d_counters.ensure(128));
        c->state_dirty = true;
    }
    PMB_CUDA(c->h_counters.ensure(128));
    if (!c->d_ticket.p) c->state_dirty = true;
    PMB_CUDA(c->d_ticket.ensure(128 * sizeof(unsigned long long)));  // two sets: consecutive runs overlap (see cstream)
    {
        int rcf;
        if ((rcf = ensure_flags(c, c->d_done, size_t(P.n_internal) * T))) return rcf;
        if ((rcf = ensure_flags(c, c->d_fdone, size_t(std::max(1, P.n_fslots)) * T))) return rcf;
    }
    PMB_CUDA(c->d_offsets.ensure(size_t(P.n_nodes + 1) * sizeof(long long)));
    if (c->staging_cap == 0 || c->staging_floor_dirty) {
        unsigned long long cells = (unsigned long long)P.n_nodes * (unsigned long long)c->n_cols;
        // default: one record per 32 cells, plus the part of a reserved block every resident warp may leave unused. A pool that
        // earlier batches have grown stays grown (an asynchronous pass cannot regrow it on the fly: the next batch of a
        // dense alignment would overflow again after every upload).
        unsigned long long cap = c->opt_staging_records > 0 ? (unsigned long long)c->opt_staging_records
                                                            : std::max<unsigned long long>(1ull << 20, cells / 32) +
                                                                  (unsigned long long)c->n_sms * 8 * WARPS_PER_BLOCK * 512ull;
        c->staging_cap = c->opt_staging_records > 0 && c->staging_cap == 0 ? cap : std::max(c->staging_cap, cap);
        c->staging_floor_dirty = false;
    }

    RunParams rp{};
    rp.fwd_ops = c->d_fwd_ops.as<FwdOp>();
    rp.refs = c->d_refs.as<uint32_t>();
    rp.bwd_ops = c->d_bwd_ops.as<BwdOp>();
    rp.bwd_leaves = c->d_bwd_leaves.as<BwdLeaf>();
    rp.chunks = c->d_chunks.as<Chunk>();
    rp.deps = c->d_deps.as<int>();
    rp.leaf_planes = c->d_leaf_planes.as<uint4>();
    rp.leaf_present = c->have_present ? c->d_present.as<uint8_t>() : nullptr;
    const int parity = int(c->run_seq & 1u);
    const bool second = dbl && parity;  // this pass works on the second staging pool / directory / run words
    rp.sets = (overlap && parity) ? c->d_sets2.as<uint4>() : c->d_sets.as<uint4>();
    rp.fstore = c->d_fstore.as<uint32_t>();
    rp.order = nullptr;
    rp.stage_block = 512;
    rp.colparams = c->d_colparams.as<uint4>();
    rp.states = want_states ? c->d_states_planes.as<uint4>() : nullptr;
    rp.dir = second ? c->d_dir2.as<unsigned long long>() : c->d_dir.as<unsigned long long>();
    unsigned long long* const run_words = c->d_counters.as<unsigned long long>() + (second ? 8 : 0);
    rp.pool_count = run_words;
    rp.error = reinterpret_cast<unsigned int*>(run_words + 1);
    rp.done = c->d_done.as<unsigned int>();
    rp.fdone = c->d_fdone.as<unsigned int>();
    rp.ticket = nullptr;
    rp.T = c->T;
    rp.n_ops = P.n_internal;
    rp.n_rows = P.n_rows;
    rp.n_fslots = std::max(1, P.n_fslots);
    rp.n_refs_total = int(P.refs.size());
    rp.flags = ((flags & PMB_FLAG_BLOCK_MODE) ? RUN_BLOCK_MODE : 0) | (want_states ? RUN_WANT_STATES : 0);

    int n_launches = 0;
    int rc = 0;
    const size_t trace_items = size_t(P.chunks.size()) * T;
    rp.trace = nullptr;
    if (c->opt_trace) {
        PMB_CUDA(c->d_trace.ensure(trace_items * 2 * 4 * sizeof(unsigned long long)));
        PMB_CUDA(cudaMemsetAsync(c->d_trace.p, 0, trace_items * 2 * 4 * sizeof(unsigned long long), c->stream));
        rp.trace = c->d_trace.as<unsigned long long>();
    }
    const int G = pick_groups(c);
    auto group_range = [&](int g, int* tb, int* tc) {
        *tb = int((long long)c->T * g / G);
        *tc = int((long long)c->T * (g + 1) / G) - *tb;
    };
    // Per-run device state is left clean by the run before (compact_copy_kernel's last block resets the counters and
    // tickets; directory entries carry a run tag): nothing is cleared on the stream in steady state.
    if (c->state_dirty) {
        PMB_CUDA(cudaStreamSynchronize(c->bstream));  // kernels of an abandoned run may still be using what is reset here
        PMB_CUDA(cudaStreamSynchronize(c->cstream));
        PMB_CUDA(cudaMemsetAsync(c->d_ticket.p, 0, 128 * sizeof(unsigned long long), c->stream));
        PMB_CUDA(cudaMemsetAsync(c->d_counters.p, 0, 128, c->stream));
        unsigned int* init = c->h_counters.as<unsigned int>() + 16;  // pinned
        init[0] = 0xFFFFFFFFu;
        PMB_CUDA(cudaMemcpyAsync(c->d_counters.as<char>() + 12, init, 4, cudaMemcpyHostToDevice, c->stream));
        PMB_CUDA(cudaMemcpyAsync(c->d_counters.as<char>() + 20, init, 4, cudaMemcpyHostToDevice, c->stream));
        PMB_CUDA(cudaMemcpyAsync(c->d_counters.as<char>() + 64 + 12, init, 4, cudaMemcpyHostToDevice, c->stream));
        c->dir_clean_epoch = 0;
        c->dir2_clean_epoch = 0;
    }
    if (c->sticky_dirty && !c->async_pending) {  // synchronous runs report their own status; only asynchronous ones use the sticky words
        unsigned int* init = c->h_counters.as<unsigned int>() + 18;  // pinned
        init[0] = 0u;
        init[1] = 0xFFFFFFFFu;
        PMB_CUDA(cudaMemcpyAsync(c->d_counters.as<char>() + 16, init, 8, cudaMemcpyHostToDevice, c->stream));
        c->sticky_dirty = false;
    }
    c->state_dirty = true;  // until everything below has been enqueued
    // forward kernel: after the pass two back has left this set matrix and ticket set, or -- one set matrix -- after the
    // previous backward kernel
    PMB_CUDA(cudaStreamWaitEvent(c->stream, c->ev_compact_done[parity], 0));
    if (!overlap) PMB_CUDA(cudaStreamWaitEvent(c->stream, c->ev_bwd_done, 0));
    PMB_CUDA(cudaEventRecord(c->ev[0], c->stream));
    rp.epoch = ++c->epoch;
    const unsigned int fwd_epoch = rp.epoch;
    const int ticket_set = 64 * parity;  // the compaction of the run before resets the other set
    c->run_seq++;
    cudaStream_t const bwd_stream = G == 1 ? c->bstream : c->stream;
    // Overlapping passes share the machine: each persistent kernel then takes 80 % of the block slots it could hold, so
    // that the blocks of the pass behind it find room before it has drained completely (measured, tools/sweep.py: 20k x 30k
    // 0.544 -> 0.538 ms, 10k x 15k 0.201 -> 0.191 ms, 4k x 625k 2.048 -> 2.012 ms per pipelined pass; alone, a kernel is
    // 3-4 % slower at 80 %). Deep trees keep the full grid: their chain segments need every slot to run side by side
    // (100k-leaf caterpillar x 30k: 2.569 ms at 100 %, 2.591 ms at 80 %).
    // Problems of very few column tiles are latency-bound throughout and gain from a little more room still (10k leaves x
    // 15 tiles: 0.189 ms at 80 %, 0.184 ms at 70 %).
    c->cur_grid_pct = c->opt_grid_pct > 0 ? int(c->opt_grid_pct)
                                          : (async && overlap && P.n_chain_segments == 0 ? (c->T < 24 ? 70 : 80) : 100);
    unsigned int* const run_error = rp.error;
    // the forward kernel may run beside the previous run's compaction, whose last block snapshots and resets the per-run
    // error words: its only status, the watchdog bit, goes straight to the sticky word
    unsigned int* const fwd_error = reinterpret_cast<unsigned int*>(c->d_counters.as<unsigned long long>() + 2);
    for (int attempt = 0;; attempt++) {
        PMB_CUDA(c->d_staging.ensure(size_t(c->staging_cap) * sizeof(uint16_t)));
        if (dbl) PMB_CUDA(c->d_staging2.ensure(size_t(c->staging_cap) * sizeof(uint16_t)));
        PMB_CUDA(c->d_pos.ensure(size_t(c->staging_cap) * sizeof(int32_t)));
        PMB_CUDA(c->d_tc.ensure(size_t(c->staging_cap)));
        rp.staging = second ? c->d_staging2.as<uint16_t>() : c->d_staging.as<uint16_t>();
        rp.staging_cap = c->staging_cap;
        const unsigned int bwd_epoch = ++c->epoch;
        rp.dir_tag = bwd_epoch & DIR_TAG_MASK;
        // per-phase events only where somebody reads them: an asynchronous pass on one stream is timed as a whole, and
        // every record between two kernels costs the stream a microsecond or two
        const bool phase_events = !async || G > 1;
        if (G > 1) PMB_CUDA(cudaEventRecord(c->ev_fork, c->stream));
        for (int g = 0; g < G; g++) {
            cudaStream_t st = G == 1 ? c->stream : c->gstream[g];
            if (G > 1) PMB_CUDA(cudaStreamWaitEvent(st, c->ev_fork, 0));
            group_range(g, &rp.tile_begin, &rp.tile_count);
            // debug trace slots: forward items of the group, then (second half) its backward items
            rp.trace_base = (unsigned long long)P.chunks.size() * rp.tile_begin;
            if (attempt == 0) {  // the forward result stays valid across a staging-pool retry
                rp.epoch = fwd_epoch;
                rp.error = fwd_error;
                if ((rc = launch_pass(c, st, ticket_set + 2 * g, rp, algo, true, &n_launches))) return rc;
                rp.error = run_error;
            }
            if (phase_events) PMB_CUDA(cudaEventRecord(c->gev_fwd[g], st));
            if (G == 1) {  // the backward kernel continues on its own stream
                PMB_CUDA(cudaEventRecord(c->ev_fwd_done, st));
                st = bwd_stream;
                PMB_CUDA(cudaStreamWaitEvent(st, c->ev_fwd_done, 0));
            }
            // the backward kernel refills a staging pool and a directory: the compaction that read them last must be through
            // (the previous pass' when there is one of each, the pass before that when they are double-buffered)
            for (int k = 0; k < 2; k++)
                if (!dbl || k == parity) PMB_CUDA(cudaStreamWaitEvent(st, c->ev_compact_done[k], 0));
            unsigned int& clean_epoch = second ? c->dir2_clean_epoch : c->dir_clean_epoch;
            if (g == 0 && (clean_epoch == 0 || bwd_epoch - clean_epoch >= DIR_TAG_MASK - 8u)) {  // new buffer, or the tag would wrap
                DevBuf& dirbuf = second ? c->d_dir2 : c->d_dir;
                PMB_CUDA(cudaMemsetAsync(dirbuf.p, 0, dirbuf.cap, st));
                clean_epoch = bwd_epoch;
                if (G > 1) {  // the other groups' backward kernels write the directory too
                    PMB_CUDA(cudaEventRecord(c->ev_fork, st));
                    for (int g2 = 1; g2 < G; g2++) PMB_CUDA(cudaStreamWaitEvent(c->gstream[g2], c->ev_fork, 0));
                }
            }
            rp.epoch = bwd_epoch;
            rp.trace_base = trace_items + (unsigned long long)P.chunks.size() * rp.tile_begin;
            if ((rc = launch_pass(c, st, ticket_set + 2 * g + 1 + 32 * (attempt & 1), rp, algo, false, &n_launches))) return rc;
            if (phase_events) PMB_CUDA(cudaEventRecord(c->gev_done[g], st));
            if (G > 1) PMB_CUDA(cudaStreamWaitEvent(c->stream, c->gev_done[g], 0));
        }
        if (phase_events) PMB_CUDA(cudaEventRecord(c->ev[2], bwd_stream));
        c->async_phase_events = phase_events;
        PMB_CUDA(cudaEventRecord(c->ev_bwd_done, bwd_stream));
        PMB_CUDA(cudaStreamWaitEvent(c->cstream, c->ev_bwd_done, 0));
        {
            const unsigned long long n_entries = (unsigned long long)P.n_nodes * (unsigned long long)c->T;
            const unsigned groups = unsigned((n_entries + CPT_GROUP - 1) / CPT_GROUP);
            if (size_t(groups) * 12 + 16 > c->d_scan_state.cap) PMB_CUDA(cudaStreamSynchronize(c->cstream));
            PMB_CUDA(c->d_scan_state.ensure(size_t(groups) * 12 + 16));
            unsigned long long* gprefix = c->d_scan_state.as<unsigned long long>();
            unsigned int* gtotals = reinterpret_cast<unsigned int*>(gprefix + groups);
            compact_count_kernel<<<(groups + 7) / 8, 256, 0, c->cstream>>>(n_entries, rp.dir, rp.dir_tag, gtotals, groups);
            compact_scan_kernel<<<1, 1024, 0, c->cstream>>>(gtotals, int(groups), gprefix, c->d_offsets.as<long long>() + P.n_nodes);
            compact_copy_kernel<<<groups, CPT_GROUP, 0, c->cstream>>>(
                P.n_nodes, c->T, gprefix, c->d_offsets.as<long long>(), rp.dir, rp.dir_tag, rp.staging, c->col_base,
                c->d_pos.as<int32_t>(), c->d_tc.as<uint8_t>(), c->d_counters.as<unsigned long long>(), run_words, rp.staging_cap,
                c->d_ticket.as<unsigned long long>() + ticket_set, 64);
            n_launches += 2;
            n_launches += 1;
        }
        PMB_CUDA(cudaGetLastError());
        PMB_CUDA(cudaEventRecord(c->ev[3], c->cstream));
        PMB_CUDA(cudaEventRecord(c->ev_compact_done[parity], c->cstream));
        c->state_dirty = false;
        if (async) {  // status, overflow handling and timings wait for pmb_wait
            c->async_pending = true;
            c->async_groups = G;
            c->timings.n_launches = n_launches;
            c->timings.n_levels = P.n_levels();
            c->last_algo = algo;
            c->last_flags = flags;
            c->n_mut = -1;
            c->have_result = true;
            return PMB_OK;
        }
        PMB_CUDA(cudaMemcpyAsync(c->h_counters.p, c->d_counters.as<char>() + 32, 16, cudaMemcpyDeviceToHost, c->cstream));  // snapshot
        PMB_CUDA(cudaMemcpyAsync(c->h_counters.as<char>() + 16, c->d_offsets.as<long long>() + P.n_nodes, 8, cudaMemcpyDeviceToHost,
                                 c->cstream));
        PMB_CUDA(cudaMemcpyAsync(c->h_counters.as<char>() + 24, c->d_counters.as<char>() + 16, 4, cudaMemcpyDeviceToHost, c->cstream));  // sticky
        PMB_CUDA(cudaStreamSynchronize(c->cstream));  // ordered behind the backward kernels of the main stream
        PMB_CUDA(cudaStreamSynchronize(c->stream));
        c->upload_pending = false;
        unsigned long long total = *c->h_counters.as<unsigned long long>();
        unsigned int eflags = c->h_counters.as<unsigned int>()[2], ecol = c->h_counters.as<unsigned int>()[3];
        eflags |= c->h_counters.as<unsigned int>()[6] & 2u;  // the forward kernel's watchdog bit
        if (eflags || total > c->staging_cap) c->sticky_dirty = true;
        if (eflags & 2u) return fail(c, PMB_ERR_INTERNAL, "scheduler watchdog fired: a dependency flag never arrived");
        if (eflags & 1u) {
            char buf[160];
            snprintf(buf, sizeof buf, "Sankoff root has no finite cost at column %lld and no root override was given",
                     (long long)ecol + (long long)c->col_base);
            return fail(c, PMB_ERR_SANKOFF_ROOT, buf);
        }
        if (total > c->staging_cap) {  // denser than provisioned: resize and redo the backward pass
            if (attempt >= 4) return fail(c, PMB_ERR_INTERNAL, "staging pool overflow persisted");
            // `total` includes the unused part of the blocks the warps reserved, and which warp reserves how much differs
            // from run to run: leave room for one more block per resident warp
            c->staging_cap = total + total / 8 + (unsigned long long)c->n_sms * 8 * WARPS_PER_BLOCK * 512ull;
            continue;
        }
        c->n_mut = *reinterpret_cast<long long*>(c->h_counters.as<char>() + 16);  // offsets[n_nodes]; the pool also holds slack
        break;
    }
    // groups overlap: "forward" = until the last group's forward pass ended, "backward" = the rest up to compaction
    float to_bwd_end = 0.f;
    c->timings.forward_ms = 0.f;
    for (int g = 0; g < G; g++) {
        float f = 0.f;
        PMB_CUDA(cudaEventElapsedTime(&f, c->ev[0], c->gev_fwd[g]));
        c->timings.forward_ms = std::max(c->timings.forward_ms, f);
    }
    PMB_CUDA(cudaEventElapsedTime(&to_bwd_end, c->ev[0], c->ev[2]));
    c->timings.backward_ms = to_bwd_end - c->timings.forward_ms;
    PMB_CUDA(cudaEventElapsedTime(&c->timings.compact_ms, c->ev[2], c->ev[3]));
    PMB_CUDA(cudaEventElapsedTime(&c->timings.total_ms, c->ev[0], c->ev[3]));
    if (c->opt_trace) {
        c->h_trace.resize(trace_items * 2 * 4);
        PMB_CUDA(cudaMemcpy(c->h_trace.data(), c->d_trace.p, c->h_trace.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    }
    c->timings.n_launches = n_launches;
    c->timings.n_levels = P.n_levels();
    c->last_algo = algo;
    c->last_flags = flags;
    c->have_result = true;
    return PMB_OK;
}

static pmb_ctx* result_ctx(pmb_ctx* c) { return c && c->last ? c->last : c; }
static const pmb_ctx* result_cctx(const pmb_ctx* c) { return c && c->last ? c->last : c; }
static bool lane_pending(const pmb_ctx* c) { return c && c->lane && (c->lane->async_pending || c->lane->upload_pending); }

int pmb_run_resident(pmb_ctx* c, int algo, int flags) {
    if (c && (c->async_pending || lane_pending(c))) {
        int rc = pmb_wait(c);
        if (rc) return rc;
    }
    if (c) c->last = nullptr;
    return run_impl(c, algo, flags, false);
}

// Is this pass one for the two lanes? Asynchronous passes of problems small enough to be latency-bound (set matrix up to
// 4 GB; the lane holds a second pair), persistent schedule, no chain segments (a deep tree's segments want every block slot
// for themselves), no state output (kept to one context), and not a rank of a group (its steps are ordered by the mailbox).
static bool lanes_apply(const pmb_ctx* c, int algo, int flags) {
    if (!c || !c->stream || c->is_lane || c->opt_lanes <= 0 || !c->have_tree || !c->have_input) return false;
    if (c->opt_schedule != 1 || c->opt_overlap <= 0 || c->opt_trace || (flags & PMB_FLAG_WANT_STATES)) return false;
    if (algo != PMB_ALGO_FITCH && algo != PMB_ALGO_SANKOFF) return false;
    if (c->prog.n_chain_segments > 0 || pick_groups(c) != 1) return false;
    const size_t set_bytes = size_t(c->prog.n_internal) * size_t(c->T) * (algo == PMB_ALGO_FITCH ? 128 : 256) * sizeof(uint4);
    return set_bytes <= std::min(size_t(4) << 30, c->total_mem / 16);
}

static int run_on_lane(pmb_ctx* c, int algo, int flags) {
    if (!c->lane) {
        pmb_ctx* L = nullptr;
        int rc = pmb_create(&L, c->device);
        if (rc) {
            c->err = std::string("second pass lane: ") + (L ? L->err : std::string("out of memory"));
            if (L) pmb_destroy(L);
            return rc;
        }
        L->is_lane = true;
        L->opt_lanes = 0;
        c->lane = L;
    }
    pmb_ctx* L = c->lane;
    PMB_CUDA(cudaSetDevice(c->device));
    L->opt_chunk_nodes = c->opt_chunk_nodes;
    L->opt_staging_records = c->opt_staging_records;
    L->opt_inline_nodes = c->opt_inline_nodes;
    L->opt_schedule = c->opt_schedule;
    L->opt_target_items = c->opt_target_items;
    L->opt_reserve_sms = c->opt_reserve_sms;
    L->opt_bwd_tail = c->opt_bwd_tail;
    L->opt_col_groups = c->opt_col_groups;
    L->opt_grid_pct = c->opt_grid_pct;
    L->opt_overlap = c->opt_overlap;
    if (L->lane_mirror_gen != c->input_gen) {  // another tree, program or batch since the lane last looked
        L->n_nodes = c->n_nodes;
        L->root = c->root;
        L->prog = c->prog;
        L->have_tree = true;
        L->n_cols = c->n_cols;
        L->col_base = c->col_base;
        L->T = c->T;
        L->have_present = c->have_present;
        L->have_input = true;
        L->staging_floor_dirty = true;
        DevBuf* dst[13];
        lane_borrowed(L, dst);
        DevBuf* src[13];
        lane_borrowed(c, src);
        for (int i = 0; i < 13; i++) {
            dst[i]->p = src[i]->p;
            dst[i]->cap = src[i]->cap;
            dst[i]->raw = nullptr;
        }
        L->have_col_break = c->have_col_break;
        L->lane_mirror_gen = c->input_gen;
    }
    L->staging_cap = std::max(L->staging_cap, c->staging_cap);  // what this context's pool has grown to, the lane's starts from
    PMB_CUDA(cudaStreamWaitEvent(L->stream, c->ev_input_ready, 0));  // what the main stream uploaded, not the passes behind it
    int rc = run_impl(L, algo, flags, true);
    if (rc) {
        c->err = L->err;
        return rc;
    }
    c->last = L;
    c->have_result = true;
    c->last_algo = algo;
    c->last_flags = flags;
    return PMB_OK;
}

static void drop_lane(pmb_ctx* c) {
    if (!c->lane) return;
    pmb_ctx* L = c->lane;
    if (L->stream) {
        cudaSetDevice(c->device);
        cudaStreamSynchronize(L->stream);
        cudaStreamSynchronize(L->bstream);
        cudaStreamSynchronize(L->cstream);
    }
    DevBuf* b[13];
    lane_borrowed(L, b);
    for (DevBuf* x : b) { x->p = nullptr; x->raw = nullptr; x->cap = 0; }
    if (c->last == L) c->last = nullptr;
    c->lane = nullptr;
    pmb_destroy(L);
}

int pmb_run_resident_async(pmb_ctx* c, int algo, int flags) {
    if (lanes_apply(c, algo, flags)) {
        if (c->lane_seq++ & 1u) {
            int rc;
            try {
                rc = run_on_lane(c, algo, flags);
            } catch (const std::bad_alloc&) {
                rc = PMB_ERR_OOM;
            } catch (const std::exception& ex) {
                return fail(c, PMB_ERR_INVALID, std::string("internal: ") + ex.what());
            }
            if (rc != PMB_ERR_OOM) return rc;
            // no room for a second set of pass buffers: one pipeline it is (nothing of the lane's pass has been enqueued)
            drop_lane(c);
            c->opt_lanes = 0;
            c->err.clear();
        }
    } else if (c) {
        c->lane_seq = 0;
    }
    if (c) c->last = nullptr;
    return run_impl(c, algo, flags, true);
}

static int wait_one(pmb_ctx* c);

int pmb_wait(pmb_ctx* c) {
    if (!c) return PMB_ERR_INVALID;
    int rc = wait_one(c);
    if (c->lane && c->lane->stream) {
        const int rc2 = wait_one(c->lane);
        if (rc2 && !rc) {
            c->err = c->lane->err;
            rc = rc2;
        }
    }
    return rc;
}

// Orders the context's main stream (pmb_stream) behind every pass enqueued so far, on either lane: an event recorded on
// pmb_stream after this call marks the end of all of them.
int pmb_join(pmb_ctx* c) {
    if (!c) return PMB_ERR_INVALID;
    if (!c->stream) return fail(c, PMB_ERR_CUDA, "no usable CUDA device; there is no CPU fallback");
    PMB_CUDA(cudaSetDevice(c->device));
    PMB_CUDA(cudaStreamWaitEvent(c->stream, c->ev[3], 0));
    if (c->lane && c->lane->stream) PMB_CUDA(cudaStreamWaitEvent(c->stream, c->lane->ev[3], 0));
    return PMB_OK;
}

static int wait_one(pmb_ctx* c) {
    if (!c) return PMB_ERR_INVALID;
    if (!c->stream) return fail(c, PMB_ERR_CUDA, "no usable CUDA device; there is no CPU fallback");
    if (!c->async_pending) {
        if (c->upload_pending) {
            PMB_CUDA(cudaSetDevice(c->device));
            PMB_CUDA(cudaStreamSynchronize(c->stream));
            c->upload_pending = false;
        }
        return PMB_OK;
    }
    PMB_CUDA(cudaSetDevice(c->device));
    c->upload_pending = false;
    const int N = c->prog.n_nodes;
    // [0,8) snapshot of the last run's staging reservation, [16,24) sticky status of all runs since the last wait
    PMB_CUDA(cudaStreamSynchronize(c->stream));
    PMB_CUDA(cudaMemcpyAsync(c->h_counters.p, c->d_counters.as<char>() + 32, 8, cudaMemcpyDeviceToHost, c->cstream));
    PMB_CUDA(cudaMemcpyAsync(c->h_counters.as<char>() + 16, c->d_counters.as<char>() + 16, 8, cudaMemcpyDeviceToHost, c->cstream));
    PMB_CUDA(cudaMemcpyAsync(c->h_counters.as<char>() + 32, c->d_offsets.as<long long>() + N, 8, cudaMemcpyDeviceToHost, c->cstream));
    PMB_CUDA(cudaStreamSynchronize(c->cstream));
    c->async_pending = false;
    const unsigned int sticky = c->h_counters.as<unsigned int>()[4], scol = c->h_counters.as<unsigned int>()[5];
    unsigned int sticky_init[2] = {0u, 0xFFFFFFFFu};
    PMB_CUDA(cudaMemcpy(c->d_counters.as<char>() + 16, sticky_init, 8, cudaMemcpyHostToDevice));
    if (sticky & 2u) { c->have_result = false; return fail(c, PMB_ERR_INTERNAL, "scheduler watchdog fired: a dependency flag never arrived"); }
    if (sticky & 1u) {
        char buf[160];
        snprintf(buf, sizeof buf, "Sankoff root has no finite cost at column %lld and no root override was given",
                 (long long)scol + (long long)c->col_base);
        c->have_result = false;
        return fail(c, PMB_ERR_SANKOFF_ROOT, buf);
    }
    if (sticky & 4u) {
        c->have_result = false;
        // as in the synchronous retry: what the pass reserved, plus room for one more block per resident warp (which warp
        // reserves how much differs from run to run)
        const unsigned long long total = *c->h_counters.as<unsigned long long>();
        c->staging_cap = std::max<unsigned long long>(c->staging_cap * 4, total + total / 8 + (unsigned long long)c->n_sms * 8 * WARPS_PER_BLOCK * 512ull);
        return fail(c, PMB_ERR_STAGING, "the mutation staging pool overflowed during an asynchronous run; rerun (the pool was grown)");
    }
    c->n_mut = *reinterpret_cast<long long*>(c->h_counters.as<char>() + 32);
    PMB_CUDA(cudaEventElapsedTime(&c->timings.total_ms, c->ev[0], c->ev[3]));
    c->timings.forward_ms = c->timings.backward_ms = c->timings.compact_ms = 0.f;
    if (!c->async_phase_events) return PMB_OK;  // timed as a whole
    PMB_CUDA(cudaEventElapsedTime(&c->timings.compact_ms, c->ev[2], c->ev[3]));
    float to_bwd_end = 0.f;
    for (int g = 0; g < c->async_groups; g++) {
        float f = 0.f;
        PMB_CUDA(cudaEventElapsedTime(&f, c->ev[0], c->gev_fwd[g]));
        c->timings.forward_ms = std::max(c->timings.forward_ms, f);
    }
    PMB_CUDA(cudaEventElapsedTime(&to_bwd_end, c->ev[0], c->ev[2]));
    c->timings.backward_ms = to_bwd_end - c->timings.forward_ms;
    return PMB_OK;
}

static int result_device_one(pmb_ctx* c, pmb_result* out);
int pmb_result_device(pmb_ctx* c, pmb_result* out) {
    pmb_ctx* r = result_ctx(c);
    const int rc = result_device_one(r, out);
    if (rc && r != c) c->err = r->err;
    return rc;
}
static int result_device_one(pmb_ctx* c, pmb_result* out) {
    if (!c || !out) return PMB_ERR_INVALID;
    if (!c->have_result) return fail(c, PMB_ERR_NO_INPUT, "no result: call pmb_run_resident first");
    out->n_mut = c->n_mut;
    out->n_nodes = c->prog.n_nodes;
    out->reserved = 0;
    out->node_offsets = reinterpret_cast<const int64_t*>(c->d_offsets.p);
    out->pos = c->d_pos.as<int32_t>();
    out->type_code = c->d_tc.as<uint8_t>();
    out->states = nullptr;
    out->n_cols = c->n_cols;
    return PMB_OK;
}

static int download_one(pmb_ctx* c, pmb_result* out);
int pmb_download(pmb_ctx* c, pmb_result* out) {
    if (!c || !out) return PMB_ERR_INVALID;
    if (c->stream && c->have_result && (c->async_pending || lane_pending(c))) {
        int rcw = pmb_wait(c);
        if (rcw) return rcw;
    }
    pmb_ctx* r = result_ctx(c);
    const int rc = download_one(r, out);
    if (rc && r != c) c->err = r->err;
    return rc;
}
static int download_one(pmb_ctx* c, pmb_result* out) {
    if (!c || !out) return PMB_ERR_INVALID;
    if (!c->stream) return fail(c, PMB_ERR_CUDA, "no usable CUDA device; there is no CPU fallback");
    if (!c->have_result) return fail(c, PMB_ERR_NO_INPUT, "no result: call pmb_run_resident first");
    if (c->async_pending) {
        int rcw = wait_one(c);
        if (rcw) return rcw;
    }
    PMB_CUDA(cudaSetDevice(c->device));
    const size_t n = size_t(c->n_mut), N = size_t(c->prog.n_nodes);
    PMB_CUDA(c->h_offsets.ensure((N + 1) * sizeof(int64_t)));
    PMB_CUDA(c->h_pos.ensure(std::max<size_t>(n, 1) * sizeof(int32_t)));
    PMB_CUDA(c->h_tc.ensure(std::max<size_t>(n, 1)));
    PMB_CUDA(cudaMemcpyAsync(c->h_offsets.p, c->d_offsets.p, (N + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, c->cstream));
    if (n) {
        PMB_CUDA(cudaMemcpyAsync(c->h_pos.p, c->d_pos.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, c->cstream));
        PMB_CUDA(cudaMemcpyAsync(c->h_tc.p, c->d_tc.p, n, cudaMemcpyDeviceToHost, c->cstream));
    }
    out->states = nullptr;
    if (c->last_flags & PMB_FLAG_WANT_STATES) {
        const size_t cells = N * size_t(c->n_cols);
        PMB_CUDA(c->d_states_u8.ensure(cells));
        PMB_CUDA(c->h_states.ensure(cells));
        unsigned blocks = unsigned((cells + 255) / 256);
        unpack_states_kernel<<<blocks, 256, 0, c->cstream>>>(c->d_states_planes.as<uint4>(), c->prog.n_nodes, c->n_cols, c->T,
                                                            c->d_states_u8.as<uint8_t>());
        PMB_CUDA(cudaGetLastError());
        PMB_CUDA(cudaMemcpyAsync(c->h_states.p, c->d_states_u8.p, cells, cudaMemcpyDeviceToHost, c->cstream));
        out->states = c->h_states.as<uint8_t>();
    }
    PMB_CUDA(cudaStreamSynchronize(c->cstream));
    out->n_mut = c->n_mut;
    out->n_nodes = c->prog.n_nodes;
    out->reserved = 0;
    out->node_offsets = c->h_offsets.as<int64_t>();
    out->pos = c->h_pos.as<int32_t>();
    out->type_code = c->h_tc.as<uint8_t>();
    out->n_cols = c->n_cols;
    return PMB_OK;
}

int pmb_run_nuc(pmb_ctx* c, int algo, int64_t n_cols, int32_t n_rows, const uint8_t* leaf_codes_4bit, int64_t row_stride_bytes,
                const uint8_t* leaf_present, const uint8_t* parent_code, const int8_t* root_override,
                const int8_t* fwd_root_ref, int64_t col_base, int flags, pmb_result* out) {
    int rc = pmb_upload_nuc(c, n_cols, n_rows, leaf_codes_4bit, row_stride_bytes, leaf_present, parent_code, root_override,
                            fwd_root_ref, col_base);
    if (rc) return rc;
    if ((rc = pmb_run_resident(c, algo, flags))) return rc;
    return pmb_download(c, out);
}

int pmb_upload_runs(pmb_ctx* c, const pmb_runs* runs, int64_t col_begin, int64_t n_cols, const uint8_t* leaf_present,
                    const uint8_t* parent_code, const int8_t* root_override, const int8_t* fwd_root_ref, int64_t col_base) {
    if (!runs) return c ? fail(c, PMB_ERR_INVALID, "null runs") : PMB_ERR_INVALID;
    PMB_GUARDED(c, upload_impl(c, n_cols, runs->n_rows, nullptr, 0, leaf_present, parent_code, root_override, fwd_root_ref, col_base, true,
                               runs, col_begin))
}

int pmb_upload_runs_async(pmb_ctx* c, const pmb_runs* runs, int64_t col_begin, int64_t n_cols, const uint8_t* leaf_present,
                          const uint8_t* parent_code, const int8_t* root_override, const int8_t* fwd_root_ref, int64_t col_base) {
    if (!runs) return c ? fail(c, PMB_ERR_INVALID, "null runs") : PMB_ERR_INVALID;
    PMB_GUARDED(c, upload_impl(c, n_cols, runs->n_rows, nullptr, 0, leaf_present, parent_code, root_override, fwd_root_ref, col_base, false,
                               runs, col_begin))
}

int pmb_run_runs(pmb_ctx* c, int algo, const pmb_runs* runs, const uint8_t* leaf_present, const uint8_t* parent_code,
                 const int8_t* root_override, const int8_t* fwd_root_ref, int64_t col_base, int flags, pmb_result* out) {
    if (!runs) return c ? fail(c, PMB_ERR_INVALID, "null runs") : PMB_ERR_INVALID;
    int rc = pmb_upload_runs(c, runs, 0, runs->n_cols, leaf_present, parent_code, root_override, fwd_root_ref, col_base);
    if (rc) return rc;
    if ((rc = pmb_run_resident(c, algo, flags))) return rc;
    return pmb_download(c, out);
}

static int run_block_impl(pmb_ctx* c, int algo, int64_t n_blocks, int32_t n_rows, const uint8_t* leaf_block_state,
                          const int8_t* root_override, pmb_result* out) {
    if (!c || !leaf_block_state || !out || n_blocks <= 0 || n_rows <= 0) return c ? fail(c, PMB_ERR_INVALID, "bad block arguments") : PMB_ERR_INVALID;
    const int64_t stride = (n_blocks + 1) / 2;
    std::vector<uint8_t> codes4(size_t(n_rows) * size_t(stride), 0), parent(size_t(n_blocks), 0);  // parent state: absent
    for (int32_t r = 0; r < n_rows; r++)
        for (int64_t b = 0; b < n_blocks; b++) {
            const uint8_t st = leaf_block_state[size_t(r) * size_t(n_blocks) + size_t(b)];
            if (st > 2) return fail(c, PMB_ERR_INVALID, "block states are 0 (absent), 1 (forward) or 2 (reverse)");
            codes4[size_t(r) * size_t(stride) + size_t(b >> 1)] |= uint8_t(st << (4 * (b & 1)));
        }
    return pmb_run_nuc(c, algo, n_blocks, n_rows, codes4.data(), stride, nullptr, parent.data(), root_override, nullptr, 0,
                       PMB_FLAG_BLOCK_MODE, out);
}

int pmb_run_block(pmb_ctx* c, int algo, int64_t n_blocks, int32_t n_rows, const uint8_t* leaf_block_state, const int8_t* root_override,
                  pmb_result* out) {
    PMB_GUARDED(c, run_block_impl(c, algo, n_blocks, n_rows, leaf_block_state, root_override, out))
}

// Debug only (not part of include/panman_b200.h): the per-item timeline of the last run made with option "trace".
// Layout: 2 * n_items records of 4 x uint64 {start ns, end ns, (chunk << 32) | tile, (sm << 32) | ns spent waiting};
// the first n_items are forward items, the rest backward items. Returns the number of uint64 copied.
long long pmb_debug_trace(const pmb_ctx* c, unsigned long long* out, long long max_words) {
    if (!c || !out) return 0;
    long long n = std::min<long long>(max_words, (long long)c->h_trace.size());
    std::memcpy(out, c->h_trace.data(), size_t(n) * sizeof(unsigned long long));
    return n;
}

// Debug only (not part of include/panman_b200.h): with PMB_DEBUG_CANARY=1, the number of guard bytes around ALL live device
// buffers of the process that no longer hold their fill value (0 = no kernel wrote outside its buffers); -1 without canaries.
long long pmb_debug_check_canaries(void) {
    if (!g_canary) return -1;
    cudaDeviceSynchronize();
    long long bad = 0;
    for (const DevBuf* b : g_canary_bufs) bad += b->bad_guard_bytes();
    return bad;
}

void* pmb_stream(pmb_ctx* c) { return c ? static_cast<void*>(c->stream) : nullptr; }
void* pmb_result_stream(pmb_ctx* c) { return c ? static_cast<void*>(result_ctx(c)->cstream) : nullptr; }

int64_t pmb_packed_bytes(int32_t n_nodes, int64_t capacity) { return int64_t(packed_bytes(n_nodes, capacity)); }

static int pack_result_one(pmb_ctx* c, void* d_packed, int64_t capacity, void* stream_v);
int pmb_pack_result(pmb_ctx* c, void* d_packed, int64_t capacity, void* stream_v) {
    pmb_ctx* r = result_ctx(c);
    const int rc = pack_result_one(r, d_packed, capacity, stream_v);
    if (rc && r != c) c->err = r->err;
    return rc;
}
static int pack_result_one(pmb_ctx* c, void* d_packed, int64_t capacity, void* stream_v) {
    if (!c || !d_packed) return PMB_ERR_INVALID;
    if (!c->stream) return fail(c, PMB_ERR_CUDA, "no usable CUDA device; there is no CPU fallback");
    if (!c->have_result) return fail(c, PMB_ERR_NO_INPUT, "no result: call pmb_run_resident first");
    if (capacity < 0 || (reinterpret_cast<uintptr_t>(d_packed) & 15u)) return fail(c, PMB_ERR_INVALID, "pmb_pack_result: buffer must be 16-byte aligned");
    if (c->n_mut >= 0 && capacity < c->n_mut) return fail(c, PMB_ERR_CAPACITY, "pmb_pack_result: capacity below the record count");
    PMB_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = stream_v ? static_cast<cudaStream_t>(stream_v) : c->cstream;  // the lists are produced on the compaction stream
    if (st != c->cstream) PMB_CUDA(cudaStreamWaitEvent(st, c->ev[3], 0));  // ev[3]: end of the pass enqueued last
    const long long N = c->prog.n_nodes;
    unsigned char* out = static_cast<unsigned char*>(d_packed);
    // everything is read on the device (n_mut = offsets[N] and the overflow status included), so nothing here needs the
    // host to know the result of a still running asynchronous pass
    pack_result_kernel<<<c->n_sms * 2, 512, 0, st>>>(c->d_offsets.as<long long>(), c->d_pos.as<int32_t>(), c->d_tc.as<uint8_t>(), N,
                                                    capacity, (long long)c->staging_cap, c->d_counters.as<unsigned long long>(), out);
    PMB_CUDA(cudaGetLastError());
    if (st != c->cstream) {  // the next pass' compaction overwrites the lists: it must wait for this copy
        PMB_CUDA(cudaEventRecord(c->ev_fork, st));
        PMB_CUDA(cudaStreamWaitEvent(c->cstream, c->ev_fork, 0));
    }
    return PMB_OK;
}

int pmb_merge_packed(pmb_ctx* c, int32_t n_shards, const void* d_packed_shards, int64_t capacity, void* stream_v,
                     pmb_result* out) {
    if (!c || !d_packed_shards || !out || n_shards < 1 || capacity < 0) return PMB_ERR_INVALID;
    if (!c->stream) return fail(c, PMB_ERR_CUDA, "no usable CUDA device; there is no CPU fallback");
    if (!c->have_tree) return fail(c, PMB_ERR_NO_TREE, "pmb_set_tree has not been called");
    PMB_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = stream_v ? static_cast<cudaStream_t>(stream_v) : c->cstream;
    const int N = c->prog.n_nodes;
    const size_t shard_bytes = packed_bytes(N, capacity);
    const size_t total_cap = size_t(n_shards) * size_t(capacity);
    // a pmb_merge_runs(source = 1) still reading the merged lists on another stream must finish first
    if (c->rm_stream && c->rm_stream != st) PMB_CUDA(cudaStreamWaitEvent(st, c->ev_rm, 0));
    if (c->merge_stream && c->merge_stream != st) PMB_CUDA(cudaStreamWaitEvent(st, c->ev_merge, 0));
    const bool grow = size_t(N) * sizeof(unsigned int) > c->d_mcounts.cap || size_t(N + 1) * sizeof(long long) > c->d_moff.cap ||
                      size_t(n_shards) * size_t(N) * sizeof(unsigned int) > c->d_mrel.cap ||
                      std::max<size_t>(1, total_cap) * sizeof(int32_t) > c->d_mpos.cap || std::max<size_t>(1, total_cap) > c->d_mtc.cap;
    if (grow && c->merge_stream) PMB_CUDA(cudaStreamSynchronize(c->merge_stream));  // cudaFree of a buffer in use
    PMB_CUDA(c->d_mcounts.ensure(size_t(N) * sizeof(unsigned int)));
    PMB_CUDA(c->d_mrel.ensure(size_t(n_shards) * size_t(N) * sizeof(unsigned int)));
    PMB_CUDA(c->d_moff.ensure(size_t(N + 1) * sizeof(long long)));
    PMB_CUDA(c->d_mpos.ensure(std::max<size_t>(1, total_cap) * sizeof(int32_t)));
    PMB_CUDA(c->d_mtc.ensure(std::max<size_t>(1, total_cap)));
    const int scan_blocks = (N + SCAN_TILE - 1) / SCAN_TILE;
    PMB_CUDA(c->d_mblock_sums.ensure(size_t(scan_blocks) * sizeof(unsigned long long)));
    if (!c->d_merge_err.p) {
        PMB_CUDA(c->d_merge_err.ensure(16));
        PMB_CUDA(cudaMemsetAsync(c->d_merge_err.p, 0, 16, st));
    }
    const unsigned char* packed = static_cast<const unsigned char*>(d_packed_shards);
    merge_count_kernel<<<(N + 255) / 256, 256, 0, st>>>(packed, shard_bytes, n_shards, N, capacity, c->d_mcounts.as<unsigned int>(),
                                                        c->d_mrel.as<unsigned int>(), c->d_merge_err.as<unsigned int>());
    scan_sums_kernel<<<scan_blocks, SCAN_BLOCK, 0, st>>>(c->d_mcounts.as<unsigned int>(), N, c->d_mblock_sums.as<unsigned long long>());
    scan_apply_kernel<<<scan_blocks, SCAN_BLOCK, 0, st>>>(c->d_mcounts.as<unsigned int>(), N, c->d_mblock_sums.as<unsigned long long>(),
                                                           c->d_moff.as<long long>());
    merge_copy_kernel<<<dim3(unsigned(c->n_sms * 2), unsigned(n_shards)), 256, 0, st>>>(packed, shard_bytes, N, capacity,
                                                                                          c->d_moff.as<long long>(), c->d_mrel.as<unsigned int>(),
                                                                                          c->d_mpos.as<int32_t>(), c->d_mtc.as<uint8_t>());
    PMB_CUDA(cudaGetLastError());
    PMB_CUDA(cudaEventRecord(c->ev_merge, st));
    c->merge_stream = st;
    out->n_mut = -1;  // on the device: node_offsets[n_nodes]; the call does not synchronise
    out->n_nodes = N;
    out->reserved = 0;
    out->node_offsets = reinterpret_cast<const int64_t*>(c->d_moff.p);
    out->pos = c->d_mpos.as<int32_t>();
    out->type_code = c->d_mtc.as<uint8_t>();
    out->states = nullptr;
    out->n_cols = 0;
    return PMB_OK;
}

int pmb_merge_status(pmb_ctx* c) {
    if (!c) return PMB_ERR_INVALID;
    if (!c->stream) return fail(c, PMB_ERR_CUDA, "no usable CUDA device; there is no CPU fallback");
    if (!c->merge_stream || !c->d_merge_err.p) return PMB_OK;
    PMB_CUDA(cudaSetDevice(c->device));
    unsigned int flags = 0;
    PMB_CUDA(cudaMemcpyAsync(&flags, c->d_merge_err.p, 4, cudaMemcpyDeviceToHost, c->merge_stream));
    PMB_CUDA(cudaStreamSynchronize(c->merge_stream));
    if (!flags) return PMB_OK;
    PMB_CUDA(cudaMemsetAsync(c->d_merge_err.p, 0, 16, c->merge_stream));
    if (flags & 2u) return fail(c, PMB_ERR_INVALID, "a merged shard was packed for a different tree (node count mismatch)");
    return fail(c, PMB_ERR_CAPACITY, "a column-range shard held more records than the capacity it was packed with (or its pass "
                                     "overflowed the staging pool): it was skipped; reserve more and repeat the step");
}

int pmb_set_column_breaks(pmb_ctx* c, const uint8_t* col_break) {
    if (!c) return PMB_ERR_INVALID;
    if (!c->stream) return fail(c, PMB_ERR_CUDA, "no usable CUDA device; there is no CPU fallback");
    if (!c->have_input) return fail(c, PMB_ERR_NO_INPUT, "pmb_upload_nuc has not been called");
    PMB_CUDA(cudaSetDevice(c->device));
    c->have_col_break = false;
    if (!col_break) return PMB_OK;
    PMB_CUDA(c->d_col_break.ensure(size_t(c->n_cols)));
    PMB_CUDA(cudaMemcpyAsync(c->d_col_break.p, col_break, size_t(c->n_cols), cudaMemcpyDefault, c->stream));
    PMB_CUDA(cudaStreamSynchronize(c->stream));  // the caller's buffer is borrowed
    c->have_col_break = true;
    c->input_gen++;
    return PMB_OK;
}

static int merge_runs_one(pmb_ctx* c, int source, int to_host, pmb_nucmut_result* out);
int pmb_merge_runs(pmb_ctx* c, int source, int to_host, pmb_nucmut_result* out) {
    pmb_ctx* r = source == 0 ? result_ctx(c) : c;
    if (r != c) {  // the lists of the last pass are the lane's; the column breaks are this context's
        if (c->async_pending || lane_pending(c)) {
            int rcw = pmb_wait(c);
            if (rcw) return rcw;
        }
        r->have_col_break = c->have_col_break;
        r->d_col_break.p = c->d_col_break.p;
        r->d_col_break.cap = c->d_col_break.cap;
        r->d_col_break.raw = nullptr;
    }
    const int rc = merge_runs_one(r, source, to_host, out);
    if (rc && r != c) c->err = r->err;
    return rc;
}
static int merge_runs_one(pmb_ctx* c, int source, int to_host, pmb_nucmut_result* out) {
    if (!c || !out || (source != 0 && source != 1)) return PMB_ERR_INVALID;
    if (!c->stream) return fail(c, PMB_ERR_CUDA, "no usable CUDA device; there is no CPU fallback");
    if (!c->have_tree) return fail(c, PMB_ERR_NO_TREE, "pmb_set_tree has not been called");
    if (source == 0 && !c->have_result) return fail(c, PMB_ERR_NO_INPUT, "no result: call pmb_run_resident first");
    if (source == 1 && (!c->d_moff.p || !c->merge_stream)) return fail(c, PMB_ERR_NO_INPUT, "no merged shards: call pmb_merge_packed first");
    PMB_CUDA(cudaSetDevice(c->device));
    if (source == 0 && c->async_pending) {
        int rcw = wait_one(c);
        if (rcw) return rcw;
    }
    // source 0 runs on the stream the lists are produced on, source 1 on the stream of the pmb_merge_packed that produced
    // them; the output buffers are shared, so a call on the other stream waits for the one before it
    cudaStream_t st = source == 0 ? c->cstream : c->merge_stream;
    if (c->rm_stream && c->rm_stream != st) PMB_CUDA(cudaStreamWaitEvent(st, c->ev_rm, 0));
    const int N = c->prog.n_nodes;
    const long long* off = source == 0 ? c->d_offsets.as<long long>() : c->d_moff.as<long long>();
    const int32_t* pos = source == 0 ? c->d_pos.as<int32_t>() : c->d_mpos.as<int32_t>();
    const uint8_t* tc = source == 0 ? c->d_tc.as<uint8_t>() : c->d_mtc.as<uint8_t>();
    // pieces <= records; the record count of merged shards is only known on the device, their capacity on the host
    const size_t cap = std::max<size_t>(1, source == 0 ? size_t(c->n_mut) : c->d_mtc.cap);
    const size_t n_blocks = (cap + RM_BLOCK - 1) / RM_BLOCK;  // cap >= the record count (known on the device for merged shards)
    const size_t scratch_bytes = n_blocks * (8 + 8 + 8 + 4) + 64;
    const bool grow = size_t(N + 1) * sizeof(long long) > c->d_rm_off.cap || cap * sizeof(int32_t) > c->d_rm_pos.cap ||
                      cap > c->d_rm_info.cap || cap * sizeof(uint32_t) > c->d_rm_nucs.cap || cap * sizeof(uint32_t) > c->d_rm_wire.cap ||
                      cap > c->d_rm_flags.cap || cap * sizeof(long long) > c->d_rm_oidx.cap || scratch_bytes > c->d_rm_counts.cap;
    if (grow && c->rm_stream) PMB_CUDA(cudaStreamSynchronize(c->rm_stream));
    PMB_CUDA(c->d_rm_off.ensure(size_t(N + 1) * sizeof(long long)));
    PMB_CUDA(c->d_rm_pos.ensure(cap * sizeof(int32_t)));
    PMB_CUDA(c->d_rm_info.ensure(cap));
    PMB_CUDA(c->d_rm_nucs.ensure(cap * sizeof(uint32_t)));
    PMB_CUDA(c->d_rm_wire.ensure(cap * sizeof(uint32_t)));
    PMB_CUDA(c->d_rm_flags.ensure(cap));
    PMB_CUDA(c->d_rm_oidx.ensure(cap * sizeof(long long)));
    PMB_CUDA(c->d_rm_counts.ensure(scratch_bytes));
    long long* last = c->d_rm_counts.as<long long>();
    long long* carry = last + n_blocks;
    unsigned long long* base = reinterpret_cast<unsigned long long*>(carry + n_blocks);
    unsigned int* counts = reinterpret_cast<unsigned int*>(base + n_blocks);
    uint8_t* flags = c->d_rm_flags.as<uint8_t>();
    const uint8_t* brk = (source == 0 && c->have_col_break) ? c->d_col_break.as<uint8_t>() : nullptr;
    PMB_CUDA(cudaMemsetAsync(flags, 0, cap, st));
    rm_mark_starts_kernel<<<(N + 255) / 256, 256, 0, st>>>(off, N, flags);
    rm_block_last_kernel<<<unsigned(n_blocks), RM_THREADS, 0, st>>>(off, N, pos, tc, flags, brk, c->col_base, last);
    rm_scan_max_kernel<<<1, 1024, 0, st>>>(last, int(n_blocks), carry);
    rm_flags_kernel<<<unsigned(n_blocks), RM_THREADS, 0, st>>>(off, N, pos, tc, flags, brk, c->col_base, carry, counts);
    compact_scan_kernel<<<1, 1024, 0, st>>>(counts, int(n_blocks), base, c->d_rm_off.as<long long>() + N);
    rm_fill_kernel<<<unsigned(n_blocks), RM_THREADS, 0, st>>>(off, N, pos, tc, flags, base, c->d_rm_oidx.as<long long>(),
                                                             c->d_rm_pos.as<int32_t>(), c->d_rm_info.as<uint8_t>(), c->d_rm_nucs.as<uint32_t>(),
                                                             c->d_rm_wire.as<uint32_t>());
    rm_node_offsets_kernel<<<(N + 255) / 256, 256, 0, st>>>(off, N, c->d_rm_oidx.as<long long>(), c->d_rm_off.as<long long>());
    PMB_CUDA(cudaGetLastError());
    PMB_CUDA(cudaEventRecord(c->ev_rm, st));
    c->rm_stream = st;
    out->n_nodes = N;
    out->reserved = 0;
    if (!to_host) {
        out->n = -1;
        out->node_offsets = reinterpret_cast<const int64_t*>(c->d_rm_off.p);
        out->nuc_position = c->d_rm_pos.as<int32_t>();
        out->mut_info = c->d_rm_info.as<uint8_t>();
        out->nucs = c->d_rm_nucs.as<uint32_t>();
        out->mut_info_wire = c->d_rm_wire.as<uint32_t>();
        return PMB_OK;
    }
    if (source == 1) {
        int rcm = pmb_merge_status(c);
        if (rcm) return rcm;
    }
    PMB_CUDA(c->h_rm_off.ensure(size_t(N + 1) * sizeof(int64_t)));
    PMB_CUDA(cudaMemcpyAsync(c->h_rm_off.p, c->d_rm_off.p, size_t(N + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    PMB_CUDA(cudaStreamSynchronize(st));
    const size_t m = size_t(c->h_rm_off.as<int64_t>()[N]);
    PMB_CUDA(c->h_rm_pos.ensure(std::max<size_t>(m, 1) * sizeof(int32_t)));
    PMB_CUDA(c->h_rm_info.ensure(std::max<size_t>(m, 1)));
    PMB_CUDA(c->h_rm_nucs.ensure(std::max<size_t>(m, 1) * sizeof(uint32_t)));
    PMB_CUDA(c->h_rm_wire.ensure(std::max<size_t>(m, 1) * sizeof(uint32_t)));
    if (m) {
        PMB_CUDA(cudaMemcpyAsync(c->h_rm_pos.p, c->d_rm_pos.p, m * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        PMB_CUDA(cudaMemcpyAsync(c->h_rm_info.p, c->d_rm_info.p, m, cudaMemcpyDeviceToHost, st));
        PMB_CUDA(cudaMemcpyAsync(c->h_rm_nucs.p, c->d_rm_nucs.p, m * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        PMB_CUDA(cudaMemcpyAsync(c->h_rm_wire.p, c->d_rm_wire.p, m * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        PMB_CUDA(cudaStreamSynchronize(st));
    }
    out->n = int64_t(m);
    out->node_offsets = c->h_rm_off.as<int64_t>();
    out->nuc_position = c->h_rm_pos.as<int32_t>();
    out->mut_info = c->h_rm_info.as<uint8_t>();
    out->nucs = c->h_rm_nucs.as<uint32_t>();
    out->mut_info_wire = c->h_rm_wire.as<uint32_t>();
    return PMB_OK;
}

int pmb_last_timings(const pmb_ctx* c, pmb_timings* out) {
    if (!c || !out) return PMB_ERR_INVALID;
    *out = result_cctx(c)->timings;
    return PMB_OK;
}

int64_t pmb_algorithmic_bytes(const pmb_ctx* c, int algo) {
    if (!c || !c->have_tree || !c->have_input) return 0;
    const int64_t L = c->prog.n_rows, I = c->prog.n_internal;
    const int64_t per_col = L + (algo == PMB_ALGO_SANKOFF ? 8 : 4) * I;  // SURVEY.md 8(d)
    const pmb_ctx* r = result_cctx(c);
    return c->n_cols * per_col + 8 * (r->have_result ? std::max<int64_t>(0, r->n_mut) : 0);
}

}  // extern "C"
