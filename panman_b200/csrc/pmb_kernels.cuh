// sm_100a kernels of libpanman_b200: persistent Fitch / Sankoff passes over bit-plane matrices (chain segments of deep
// trees evaluated speculatively but exactly), mutation staging with warp-ballot + prefix-sum compaction, ordered
// compaction by directory entry, the greedy run-merge into NucMut fields, shard merging, and the ingest packers.
//
// Work decomposition: one WARP owns (chunk of the tree) x (tile of 1024 columns). Lane l holds, for every
// node it touches, one 32-bit word per bit-plane = columns [tile*1024 + l*32, +32). All HBM traffic is
// 128-bit per lane, 512 contiguous bytes per warp instruction; every matrix is TILE-major, so a warp streams
// through contiguous memory in program order:
//   leaf matrix   uint4 [tile][leaf slot][lane]      4 code planes            (0.5 B / column)
//   set matrix    uint4 [tile][op][J][lane]          J=4 Fitch (16 planes),   (2 B / column)
//                                                    J=8 Sankoff (G,H planes) (4 B / column)
// Reference semantics implemented here: src/fitchSankoff.cpp:30-171 (nuc Fitch), :224-308 (block Fitch),
// :359-531 + :676-703 (nuc Sankoff), :707-818 (block Sankoff); see plane_math.h for the per-op logic.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "plane_math.h"
#include "tree_program.h"

namespace pmb {

constexpr int TILE_COLS = 1024;
constexpr int WARPS_PER_BLOCK = 4;
constexpr unsigned FULL = 0xFFFFFFFFu;
constexpr int FSLOT_WORDS = 160;   // parked assigned state of one (node, tile): 4 code planes + visited plane per lane

enum : int { RUN_BLOCK_MODE = 1, RUN_WANT_STATES = 2 };

struct RunParams {
    const FwdOp* fwd_ops;
    const uint32_t* refs;
    const BwdOp* bwd_ops;
    const BwdLeaf* bwd_leaves;
    const Chunk* chunks;
    const int* deps;              // forward dependency lists of the chunks
    const uint4* leaf_planes;
    const uint8_t* leaf_present;  // device, n_rows bytes, or nullptr = all present
    uint4* sets;
    uint32_t* fstore;             // [fslot][tile][FSLOT_WORDS]: 32 x uint4 code planes, then 32 visited words
    const uint4* colparams;       // [tile][4][lane]: parent code, override code, fwd ref code, {ov_valid, ref_valid, col_valid, 0}
    uint4* states;                // [node][tile][2][lane] or nullptr
    unsigned long long* dir;      // [node][tile]: (staging base << 11) | count
    uint16_t* staging;
    unsigned long long* pool_count;
    unsigned long long staging_cap;
    unsigned int* error;          // [0] flags (1 Sankoff root undefined, 2 scheduler watchdog), [1] first offending column
    unsigned int* done;           // [op][tile]   forward: set matrix row published (value = epoch)
    unsigned int* fdone;          // [fslot][tile] backward: assigned-state slot published
    unsigned long long* ticket;   // persistent launch: work-item counter; nullptr = one static item per warp
    const int* order;             // item i works on chunk order[i / T]; nullptr = identity
    unsigned int epoch;
    unsigned int dir_tag;         // backward: tag of this run's directory entries (entries with another tag are stale = empty)
    int T;
    int n_ops, n_rows, n_fslots;  // matrices are TILE-major: [tile][op], [tile][leaf slot], [tile][fslot]
    int n_refs_total;
    int flags;
    int stage_block;              // staging records a warp reserves per atomic
    int tile_begin, tile_count;   // this launch covers tiles [tile_begin, tile_begin + tile_count) (column group)
    unsigned long long* trace;    // debug: per item {start ns, end ns, (chunk << 32) | tile, (sm << 32) | waited ns}; or nullptr
    unsigned long long trace_base;
};

struct TraceItem {  // debug timeline of one work item (option "trace")
    unsigned long long t0 = 0, w = 0;
    unsigned waited = 0;
};
__device__ __forceinline__ unsigned smid() {
    unsigned r;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(r));
    return r;
}

// Tile-major addressing: for one tile the rows of consecutive ops (and the leaf rows in the order the program
// consumes them) are contiguous, so a warp streams through memory instead of hopping between far-apart rows.
__device__ __forceinline__ size_t set_index(const RunParams& p, unsigned op, int tile) { return (size_t)tile * p.n_ops + op; }
__device__ __forceinline__ size_t leaf_index(const RunParams& p, unsigned slot, int tile) { return (size_t)tile * p.n_rows + slot; }
__device__ __forceinline__ size_t fslot_index(const RunParams& p, unsigned f, int tile) { return (size_t)tile * p.n_fslots + f; }

__device__ __forceinline__ uint4 ld_stream(const uint4* p) { return __ldcs(p); }
__device__ __forceinline__ uint4 ld_l2(const uint4* p) { return __ldcg(p); }

__device__ __forceinline__ void load_planes16(const uint4* base, int lane, uint32_t S[16]) {
#pragma unroll
    for (int j = 0; j < 4; j++) {
        uint4 v = ld_l2(base + j * 32 + lane);
        S[4 * j + 0] = v.x; S[4 * j + 1] = v.y; S[4 * j + 2] = v.z; S[4 * j + 3] = v.w;
    }
}
__device__ __forceinline__ void store_planes16(uint4* base, int lane, const uint32_t S[16]) {
#pragma unroll
    for (int j = 0; j < 4; j++) base[j * 32 + lane] = make_uint4(S[4 * j], S[4 * j + 1], S[4 * j + 2], S[4 * j + 3]);
}
__device__ __forceinline__ void unpack16(const uint4 v[4], uint32_t S[16]) {
#pragma unroll
    for (int j = 0; j < 4; j++) { S[4 * j] = v[j].x; S[4 * j + 1] = v[j].y; S[4 * j + 2] = v[j].z; S[4 * j + 3] = v[j].w; }
}

// ------------------------------------------------------------------ work items and dependencies
// A work item is (chunk, tile). Level launches give every warp one static item; the persistent launch hands
// items out through an atomic ticket in the program's topological chunk order (reverse for the backward pass).
// An item may only wait for data of items with SMALLER tickets, and every ticket holder is a resident, running
// warp, so the lowest unfinished ticket always makes progress: no deadlock, no co-residency requirement.
__device__ __forceinline__ unsigned long long global_ns();
struct ItemIter {
    bool taken = false;
};
__device__ __forceinline__ bool next_item(const RunParams& p, ItemIter& it, int chunk_begin, int n_chunks, int& chunk,
                                          int& tile, int lane, TraceItem& tr) {
    unsigned long long w;
    if (p.ticket) {
        if (lane == 0) w = atomicAdd(p.ticket, 1ull);
        w = __shfl_sync(FULL, w, 0);
    } else {
        if (it.taken) return false;
        it.taken = true;
        w = (unsigned long long)blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
    }
    if (w >= (unsigned long long)n_chunks * (unsigned long long)p.tile_count) return false;
    int c = chunk_begin + int(w / (unsigned)p.tile_count);
    chunk = p.order ? __ldg(p.order + c) : c;
    tile = p.tile_begin + int(w % (unsigned)p.tile_count);
    if (p.trace) {
        tr.t0 = global_ns();
        tr.w = w;
        tr.waited = 0;
    }
    return true;
}
__device__ __forceinline__ void trace_end(const RunParams& p, const TraceItem& tr, int chunk, int tile, int lane) {
    if (p.trace && lane == 0) {
        unsigned long long* q = p.trace + (p.trace_base + tr.w) * 4;
        q[0] = tr.t0;
        q[1] = global_ns();
        q[2] = ((unsigned long long)(unsigned)chunk << 32) | (unsigned)tile;
        q[3] = ((unsigned long long)smid() << 32) | tr.waited;
    }
}

__device__ __forceinline__ unsigned ld_acquire(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(unsigned* p, unsigned v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Warp-collective wait until *flag == epoch. Lane 0 polls with back-off; a watchdog (wall clock) turns a
// scheduling bug into error bit 2 instead of a hung GPU. Returns false if the run must be abandoned.
__device__ __noinline__ bool wait_flag_slow(const unsigned* flag, unsigned epoch, unsigned* error, int lane, unsigned* waited) {
    unsigned ok = 1;
    if (lane == 0) {
        unsigned long long t0 = global_ns();
        unsigned spins = 0;
        while (ld_acquire(flag) != epoch) {
            __nanosleep(64);
            if ((++spins & 255u) == 0) {
                if ((*reinterpret_cast<volatile unsigned*>(error) & 2u) || global_ns() - t0 > 20000000000ull) {
                    atomicOr(error, 2u);
                    ok = 0;
                    break;
                }
            }
        }
        *waited += unsigned(global_ns() - t0);
    }
    ok = __shfl_sync(FULL, ok, 0);
    __syncwarp();  // the other lanes' reads of the published rows are ordered behind lane 0's acquire
    return ok != 0;
}
__device__ __forceinline__ bool wait_flag(const unsigned* flag, unsigned epoch, unsigned* error, int lane, TraceItem& tr) {
    unsigned v = 0;
    if (lane == 0) v = ld_acquire(flag);
    v = __shfl_sync(FULL, v, 0);
    if (v == epoch) {
        __syncwarp();  // a shuffle is no memory ordering: the barrier is what puts every lane's reads behind the acquire
        return true;
    }
    return wait_flag_slow(flag, epoch, error, lane, &tr.waited);
}
// Forward dependencies: a chunk lists the external rows it reads in consumption order (Chunk::dep_*), and an
// external ref names its ordinal k in that list. The warp keeps `upto` = number of leading dependencies known to be
// published; when ref k is not covered yet, all 32 lanes poll the next 32 flags at once, so one L2 round trip (one
// acquire) usually verifies the dependencies of many upcoming ops -- the per-op acquire of the earlier version was
// what made the top-of-tree chain slow (profiles/r01_v5). Consumption stays progressive: an item starts working
// before its later inputs exist.
struct DepCursor {
    int upto = 0;
};
__device__ __forceinline__ bool wait_dep(const RunParams& p, const Chunk& ck, const unsigned* done_tile, DepCursor& dc, int k,
                                         int lane, TraceItem& tr) {
    if (k < dc.upto) return true;
    unsigned long long t0 = 0;
    unsigned spins = 0;
    for (;;) {
        const int i = dc.upto + lane;
        bool ok = false;
        if (i < ck.dep_count) ok = ld_acquire(done_tile + __ldg(p.deps + ck.dep_begin + i)) == p.epoch;
        const unsigned b = __ballot_sync(FULL, ok);
        dc.upto += (b == FULL) ? 32 : (__ffs(~b) - 1);
        if (k < dc.upto) break;
        if (spins == 0) t0 = global_ns();
        __nanosleep(64);
        if ((++spins & 255u) == 0) {
            bool dead = (*reinterpret_cast<volatile unsigned*>(p.error) & 2u) || global_ns() - t0 > 20000000000ull;
            if (__any_sync(FULL, dead)) {
                atomicOr(p.error, 2u);
                return false;
            }
        }
    }
    if (spins) tr.waited += unsigned(global_ns() - t0);
    __syncwarp();  // each flag was acquired by ONE lane; all lanes read the rows
    return true;
}
// row of a set reference: direct, or through the dependency list for an external ref
__device__ __forceinline__ uint32_t ref_row(const RunParams& p, const Chunk& ck, uint32_t ref) {
    const uint32_t v = ref & REF_IDX_MASK;
    return (ref & REF_EXT) ? (uint32_t)__ldg(p.deps + ck.dep_begin + v) : v;
}

// Publish: every lane's earlier stores happen-before the release store of lane 0 (warp barrier + release).
__device__ __forceinline__ void signal_flag(unsigned* flag, unsigned epoch, int lane) {
    __syncwarp();
    if (lane == 0) st_release(flag, epoch);
}

__device__ __forceinline__ uint32_t leaf_present_mask(const RunParams& p, int row) {
    if (p.leaf_present == nullptr) return FULL;
    return __ldg(p.leaf_present + row) ? FULL : 0u;
}

// ------------------------------------------------------------------ mutation staging
// Appends the records of one (node, tile) in ascending column order: warp ballot to skip the common empty
// case, shuffle prefix sum over per-lane popcounts. Staging space is reserved per warp in blocks of
// p.stage_block records (one atomic per block, not per append: the round trip of a per-append atomic was 46 % of
// the backward pass' stall samples in profiles/r01_v2). The (node, tile) directory remembers where each
// segment went; compact_copy_kernel later lays the segments out node-major in column order.
// Record: column-in-tile (10 bits) | code << 10 | type << 14.
// Directory entry: tag (13 bits) | staging base (40 bits) | count (11 bits). The tag names the run that wrote the entry,
// so the directory needs no clearing between runs (the host clears it when the tag is about to wrap).
constexpr int DIR_TAG_SHIFT = 51;
constexpr unsigned DIR_TAG_MASK = 0x1FFFu;
struct StageCursor {
    unsigned long long base = 0;
    int left = 0;
};
__device__ __forceinline__ void emit(const RunParams& p, StageCursor& sc, int node, int tile, int lane, uint32_t mut,
                                     const uint32_t P[4], const uint32_t F[4]) {
    if (__ballot_sync(FULL, mut != 0) == 0) return;
    int cnt = __popc(mut);
    int incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int t = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += t;
    }
    const int total = __shfl_sync(FULL, incl, 31);
    if (total > sc.left) {
        const int take = max(total, p.stage_block);
        unsigned long long b = 0;
        if (lane == 0) b = atomicAdd(p.pool_count, (unsigned long long)take);
        sc.base = __shfl_sync(FULL, b, 0);
        sc.left = take;
    }
    const unsigned long long base = sc.base;
    sc.base += total;
    sc.left -= total;
    if (lane == 0)
        p.dir[(size_t)node * p.T + tile] = ((unsigned long long)p.dir_tag << DIR_TAG_SHIFT) | (base << 11) | (unsigned long long)total;
    if (base + (unsigned long long)total > p.staging_cap) return;  // host grows the pool and reruns the pass
    uint32_t t0, t1;
    mutation_type(P, F, t0, t1);
    uint16_t* dst = p.staging + base + (incl - cnt);
    uint32_t m = mut;
    while (m) {
        int b = __ffs(m) - 1;
        m &= m - 1;
        uint32_t code = ((F[0] >> b) & 1u) | (((F[1] >> b) & 1u) << 1) | (((F[2] >> b) & 1u) << 2) | (((F[3] >> b) & 1u) << 3);
        uint32_t type = ((t0 >> b) & 1u) | (((t1 >> b) & 1u) << 1);
        *dst++ = uint16_t((lane * 32 + b) | (code << 10) | (type << 14));
    }
}

__device__ __forceinline__ void store_state(const RunParams& p, int node, int tile, int lane, const uint32_t F[4], uint32_t vis) {
    uint4* s = p.states + ((size_t)node * p.T + tile) * 64;
    s[lane] = make_uint4(F[0], F[1], F[2], F[3]);
    s[32 + lane] = make_uint4(vis, 0, 0, 0);
}

// ------------------------------------------------------------------ asynchronous input ring (cp.async)
// Every warp keeps a ring of DEPTH "stages" in shared memory, one stage per upcoming op, filled with LDGSTS
// (cp.async.cg, 16 B per lane = 512 B per warp instruction) DEPTH ops ahead of use. Only IMMUTABLE inputs go
// through the ring -- leaf rows, and in the backward pass the set rows written by the finished forward pass --
// so no ordering against this kernel's own stores is ever needed. Each lane copies and later reads its own
// 16 bytes: completion is tracked per thread with cp.async.wait_group, no barrier involved.
__device__ __forceinline__ void cp_async16(uint4* smem_dst, const uint4* gsrc) {
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_pending(int n) {  // at most n groups still in flight
    switch (n) {
    case 0: asm volatile("cp.async.wait_group 0;" ::: "memory"); break;
    case 1: asm volatile("cp.async.wait_group 1;" ::: "memory"); break;
    case 2: asm volatile("cp.async.wait_group 2;" ::: "memory"); break;
    case 3: asm volatile("cp.async.wait_group 3;" ::: "memory"); break;
    case 4: asm volatile("cp.async.wait_group 4;" ::: "memory"); break;
    case 5: asm volatile("cp.async.wait_group 5;" ::: "memory"); break;
    case 6: asm volatile("cp.async.wait_group 6;" ::: "memory"); break;
    default: asm volatile("cp.async.wait_group 7;" ::: "memory"); break;
    }
}

// ------------------------------------------------------------------ bulk-copy ring (experiment, -DPMB_BULK=1)
// The same ring filled by the bulk asynchronous copy unit instead of per-lane LDGSTS: ONE elected lane issues one
// cp.async.bulk per row (a set row is 2 KB contiguous in the tile-major layout, a leaf row 512 B) and the bytes are
// counted on an mbarrier per stage; all lanes wait on the barrier's phase. Fewer instructions per op (1 + rows instead of
// 32 x rows + commit + wait), at the price of a warp barrier before a stage is refilled (the per-lane ring needs none:
// every lane copies and reads only its own 16 bytes). Built with `make VARIANT=_bulk EXTRA=-DPMB_BULK=1`; result in
// profiles/r02_summary.md.
#ifndef PMB_BULK
#define PMB_BULK 0
#endif
__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_copy(void* smem_dst, const void* gsrc, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_addr(bar)),
        "r"(parity)
        : "memory");
}

// Measured on B200 (tools/sweep.py, profiles/r01_v8_summary.md): shallower rings and smaller windows win because shared
// memory is what limits residency (forward 4 -> 5 blocks per SM, backward 4 -> 6), and more resident warps hide latency
// better than a deeper per-warp ring does.
#ifndef PMB_BWD_DEPTH
#define PMB_BWD_DEPTH 2
#endif
#ifndef PMB_FWD_DEPTH
#define PMB_FWD_DEPTH 3
#endif
#ifndef PMB_META_OPS
#define PMB_META_OPS 16
#endif
constexpr int FWD_DEPTH = PMB_FWD_DEPTH;  // forward: stage = 2 leaf rows + one child set row (3 KB Fitch / 3.5 KB Sankoff)
constexpr int BWD_DEPTH = PMB_BWD_DEPTH;  // backward: stage = set row + 2 leaf rows           (3 KB Fitch / 5 KB Sankoff)

template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
// steady state: DEPTH - 1 younger groups may stay in flight; near the end of a chunk simply drain
template <int DEPTH>
__device__ __forceinline__ void cp_async_wait_stage(int ops_left_after) {
    if (ops_left_after >= DEPTH - 1) cp_async_wait<DEPTH - 1>();
    else cp_async_wait<0>();
}

// ------------------------------------------------------------------ program metadata windows
// Op records and child references are tiny but sat on the critical path of every op as dependent L2 loads
// (profiles/r01_v3: the top stall in both passes). Each warp therefore keeps a window of its chunk's metadata in
// shared memory, refilled with a few coalesced loads every META_OPS - depth ops. Records are 32 bytes and carry
// their first two references inline, so the bifurcating common case is straight-line code.
constexpr int META_OPS = PMB_META_OPS, META_REFS = 3 * PMB_META_OPS, META_LEAVES = 2 * PMB_META_OPS;
constexpr int FWD_META_U4 = 2 * META_OPS + META_REFS / 4;
constexpr int BWD_META_U4 = 2 * META_OPS + META_LEAVES / 2;
constexpr int BWD_STACK_U4 = BWD_STACK_DEPTH * FSLOT_WORDS / 4;  // per-warp stack of parked assigned states

struct FwdMeta {
    int4* ops;
    uint32_t* refs;
    int wb;       // first op of the window
    unsigned rb;  // first ref of the window
};
__device__ __forceinline__ void fwd_meta_load(const RunParams& p, FwdMeta& m, int wb, int op_end, int lane) {
    __syncwarp();  // all lanes are done with the previous window
    m.wb = wb;
    int4 h0 = make_int4(0, 0, 0, 0), h1 = h0;
    if (lane < META_OPS && wb + lane < op_end) {
        h0 = __ldg(reinterpret_cast<const int4*>(p.fwd_ops + wb + lane));
        h1 = __ldg(reinterpret_cast<const int4*>(p.fwd_ops + wb + lane) + 1);
    }
    if (lane < META_OPS) {
        m.ops[2 * lane] = h0;
        m.ops[2 * lane + 1] = h1;
    }
    m.rb = (unsigned)__shfl_sync(FULL, h0.x, 0);
#pragma unroll
    for (int d = lane; d < META_REFS; d += 32) {
        const unsigned i = m.rb + d;
        m.refs[d] = i < (unsigned)p.n_refs_total ? __ldg(p.refs + i) : 0u;
    }
    __syncwarp();
}
__device__ __forceinline__ uint32_t fwd_ref(const RunParams& p, const FwdMeta& m, unsigned i) {
    const unsigned d = i - m.rb;
    return d < (unsigned)META_REFS ? m.refs[d] : __ldg(p.refs + i);
}

struct BwdMeta {
    int4* ops;
    int2* leaves;
    int lo;       // lowest op of the window (ops run downwards)
    unsigned lb;  // first leaf entry of the window
};
__device__ __forceinline__ void bwd_meta_load(const RunParams& p, BwdMeta& m, int top, int op_begin, int lane) {
    __syncwarp();
    m.lo = max(op_begin, top - (META_OPS - 1));
    int4 h0 = make_int4(0, 0, 0, 0), h1 = h0;
    if (lane < META_OPS && m.lo + lane <= top) {
        h0 = __ldg(reinterpret_cast<const int4*>(p.bwd_ops + m.lo + lane));
        h1 = __ldg(reinterpret_cast<const int4*>(p.bwd_ops + m.lo + lane) + 1);
    }
    if (lane < META_OPS) {
        m.ops[2 * lane] = h0;
        m.ops[2 * lane + 1] = h1;
    }
    m.lb = (unsigned)__shfl_sync(FULL, h0.w, 0);
#pragma unroll
    for (int d = lane; d < META_LEAVES; d += 32) {
        const unsigned i = m.lb + d;
        m.leaves[d] = i < (unsigned)p.n_rows ? __ldg(reinterpret_cast<const int2*>(p.bwd_leaves + i)) : make_int2(0, 0);
    }
    __syncwarp();
}
struct BwdHead {
    int4 b0;  // node, parent_ref, fslot_out, leaf_begin
    int4 b1;  // n_leaves, flags, leaf0 slot, leaf1 slot
};
__device__ __forceinline__ int2 bwd_leaf(const RunParams& p, const BwdMeta& m, unsigned i) {
    const unsigned d = i - m.lb;
    return d < (unsigned)META_LEAVES ? m.leaves[d] : __ldg(reinterpret_cast<const int2*>(p.bwd_leaves + i));
}

// per-item base pointers (tile-major layouts), already offset by the lane
struct TileCtx {
    const uint4* leaf;  // + slot * 32
    uint4* sets;        // + op * JROW * 32
    unsigned* done;     // + op
};
template <int JROW>
__device__ __forceinline__ TileCtx tile_ctx(const RunParams& p, int tile, int lane) {
    TileCtx t;
    t.leaf = p.leaf_planes + (size_t)tile * p.n_rows * 32 + lane;
    t.sets = p.sets + (size_t)tile * p.n_ops * (JROW * 32) + lane;
    t.done = p.done + (size_t)tile * p.n_ops;
    return t;
}

// A set row other than the register accumulator can be prefetched when it is already final at issue time:
// written by another chunk (after its done flag) or by this warp at least FWD_DEPTH ops before the consumer.
__device__ __forceinline__ bool fwd_set_prefetched(uint32_t ref, int op) {
    return (ref & REF_EXT) || int(ref & REF_IDX_MASK) + FWD_DEPTH <= op;
}
template <int JS, int JROW>
__device__ __forceinline__ bool fwd_issue_set(const RunParams& p, const Chunk& ck, const TileCtx& tc, DepCursor& dc, uint4* st,
                                              uint32_t ref, uint32_t row_idx, int op, int lane, TraceItem& tr) {
    if (!fwd_set_prefetched(ref, op)) return true;
    if (ref & REF_EXT) {
        if (!wait_dep(p, ck, tc.done, dc, int(ref & REF_IDX_MASK), lane, tr)) return false;
    }
    const uint4* row = tc.sets + (size_t)row_idx * (JROW * 32);
#pragma unroll
    for (int j = 0; j < JS; j++) cp_async16(st + (2 + j) * 32, row + j * 32);
    return true;
}
// forward: queue the inputs of `op` into stage `st` (lane-offset pointer) and commit one group: the first two leaf
// rows and, when prefetchable, the first set row. JS = vectors of a set row the consumer needs, JROW = row length.
template <int JS, int JROW>
__device__ __forceinline__ bool fwd_issue(const RunParams& p, const Chunk& ck, const FwdMeta& m, const TileCtx& tc, DepCursor& dc,
                                          uint4* st, int op, int lane, TraceItem& tr) {
    const int4 w0 = m.ops[2 * (op - m.wb)], w1 = m.ops[2 * (op - m.wb) + 1];
    const uint32_t r0 = (uint32_t)w1.x, r1 = (uint32_t)w1.y;
    bool ok = true;
    switch ((w0.z >> OPF_TYPE_SHIFT) & 15) {
    case FT_LEAF_LEAF:
        cp_async16(st, tc.leaf + (size_t)(r0 & REF_IDX_MASK) * 32);
        cp_async16(st + 32, tc.leaf + (size_t)(r1 & REF_IDX_MASK) * 32);
        break;
    case FT_LEAF_ACC:
        cp_async16(st, tc.leaf + (size_t)(r0 & REF_IDX_MASK) * 32);
        break;
    case FT_LEAF_INT:
        cp_async16(st, tc.leaf + (size_t)(r0 & REF_IDX_MASK) * 32);
        ok = fwd_issue_set<JS, JROW>(p, ck, tc, dc, st, r1, (uint32_t)w1.w, op, lane, tr);
        break;
    case FT_INT_ACC:
        ok = fwd_issue_set<JS, JROW>(p, ck, tc, dc, st, r0, (uint32_t)w1.z, op, lane, tr);
        break;
    default: {
        int nl = 0, ni = 0;
        for (int r = 0; r < w0.y && (nl < 2 || ni < 1); r++) {
            const uint32_t ref = fwd_ref(p, m, w0.x + r);
            const uint32_t kind = ref >> 30;
            if (kind == REF_LEAF) {
                if (nl < 2) cp_async16(st + nl * 32, tc.leaf + (size_t)(ref & REF_IDX_MASK) * 32);
                nl++;
            } else if (kind == REF_INT) {
                if (ni == 0) ok = fwd_issue_set<JS, JROW>(p, ck, tc, dc, st, ref, ref_row(p, ck, ref), op, lane, tr) && ok;
                ni++;
            }
        }
    }
    }
    cp_async_commit();
    return ok;
}
__device__ __forceinline__ void stage_set16(const uint4* st, uint32_t X[16]) {
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const uint4 v = st[(2 + j) * 32];
        X[4 * j] = v.x; X[4 * j + 1] = v.y; X[4 * j + 2] = v.z; X[4 * j + 3] = v.w;
    }
}
__device__ __forceinline__ void row_set16(const uint4* row, uint32_t X[16]) {
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const uint4 v = ld_l2(row + j * 32);
        X[4 * j] = v.x; X[4 * j + 1] = v.y; X[4 * j + 2] = v.z; X[4 * j + 3] = v.w;
    }
}

// ------------------------------------------------------------------ chain segments (speculative evaluation)
// See tree_program.h. `head` is the latest op seen on the segment's heavy path (-1 before the first one): an op is on
// the path iff it holds the REF_CHAIN child or consumes `head`.
__device__ __forceinline__ bool fwd_on_path(const RunParams& p, const int4 w0, int op, int head) {
    for (int r = 0; r < w0.y; r++) {
        const uint32_t ref = __ldg(p.refs + w0.x + r), kind = ref >> 30;
        if (kind == REF_CHAIN) return true;
        if (head < 0) continue;
        if (kind == REF_ACC && head == op - 1) return true;
        if (kind == REF_INT && !(ref & REF_EXT) && int(ref & REF_IDX_MASK) == head) return true;
    }
    return false;
}
// Folds the KNOWN children of `op` (all but the one on the path) into fold.A / fold.O. Every leaf is present here
// (speculation is only used without a presence mask). ACC_REGS: the previous op's result is still in `acc`.
template <bool ACC_REGS>
__device__ __forceinline__ bool fitch_fold_known(const RunParams& p, const Chunk& ck, const TileCtx& tc, DepCursor& dc, const int4 w0,
                                                 int op, int head, const uint32_t acc[16], int lane, FitchFold& fold, TraceItem& tr) {
    fold.reset();
    for (int r = 0; r < w0.y; r++) {
        const uint32_t ref = __ldg(p.refs + w0.x + r), kind = ref >> 30, idx = ref & REF_IDX_MASK;
        if (kind == REF_CHAIN) continue;
        if (kind == REF_LEAF) {
            const uint4 c = ld_stream(tc.leaf + (size_t)idx * 32);
            const uint32_t cc[4] = {c.x, c.y, c.z, c.w};
            fold.add_leaf(cc, FULL);
        } else if (kind == REF_ACC) {
            if (head >= 0 && head == op - 1) continue;
            if (ACC_REGS) {
                fold.add_set(acc);
            } else {
                uint32_t S[16];
                row_set16(tc.sets + (size_t)(op - 1) * 128, S);
                fold.add_set(S);
            }
        } else {
            if (!(ref & REF_EXT) && head >= 0 && int(idx) == head) continue;
            if (ref & REF_EXT) {
                if (!wait_dep(p, ck, tc.done, dc, int(idx), lane, tr)) return false;
            }
            uint32_t S[16];
            row_set16(tc.sets + (size_t)ref_row(p, ck, ref) * 128, S);
            fold.add_set(S);
        }
    }
    return true;
}
// refState: the root's forward value is replaced where a reference state is given (fitchSankoff.cpp:45-47)
__device__ __forceinline__ void fitch_root_ref(const RunParams& p, int tile, int lane, uint32_t S[16]) {
    const uint4* cp = p.colparams + (size_t)tile * 128;
    uint4 rc = __ldg(cp + 64 + lane);
    uint32_t rv = __ldg(cp + 96 + lane).y;
    uint32_t r4[4] = {rc.x, rc.y, rc.z, rc.w}, d[16];
    decode16(r4, d);
#pragma unroll
    for (int k = 0; k < 16; k++) S[k] = (rv & d[k]) | (~rv & S[k]);
}
__device__ __forceinline__ void store_set16(uint4* out, const uint32_t S[16]) {
#pragma unroll
    for (int j = 0; j < 4; j++) out[j * 32] = make_uint4(S[4 * j], S[4 * j + 1], S[4 * j + 2], S[4 * j + 3]);
}

// ------------------------------------------------------------------ Fitch forward
// SPEC = the program has chain segments (tree_program.h); trees without them run the leaner instantiation
constexpr int FITCH_FWD_STAGE = (2 + 4) * 32, FITCH_FWD_PER_WARP = FWD_DEPTH * FITCH_FWD_STAGE + FWD_META_U4;
// one work item: the chunk's ops for one column tile. `ring` = the warp's shared memory; false = abandon the run
template <bool SPEC>
__device__ __forceinline__ bool fitch_forward_item(const RunParams& p, uint4* ring, int chunk, int tile, int lane, TraceItem& tr) {
    constexpr int JS = 4, STAGE = FITCH_FWD_STAGE;
    FwdMeta m;
    m.ops = reinterpret_cast<int4*>(ring + FWD_DEPTH * STAGE);
    m.refs = reinterpret_cast<uint32_t*>(m.ops + 2 * META_OPS);
    uint4* const ring_l = ring + lane;
    {
        const Chunk ck = p.chunks[chunk];
        const TileCtx tc = tile_ctx<4>(p, tile, lane);
        DepCursor dc;
        uint32_t acc[16];
#pragma unroll
        for (int k = 0; k < 16; k++) acc[k] = 0;
        // Chain segment: the value entering from the segment below is not waited for. Bounds on it are carried up the
        // path until no column depends on it any more (op `resolved`); the plain loop continues from there and the
        // few ops before it are redone at the end, once the segment below has published.
        const bool spec = SPEC && ck.chain_op >= 0 && p.leaf_present == nullptr;
        int first = ck.op_begin, resolved = -1;
        if (spec) {
            FitchInterval iv;
            iv.reset();
            int head = -1;
            first = ck.op_end;
            for (int op = ck.op_begin; op < ck.op_end; op++) {
                const int4 w0 = __ldg(reinterpret_cast<const int4*>(p.fwd_ops + op));
                const bool on_path = fwd_on_path(p, w0, op, head);
                FitchFold fold;
                if (!fitch_fold_known<true>(p, ck, tc, dc, w0, op, head, acc, lane, fold, tr)) return false;
                if (!on_path) {  // a light subtree evaluated inside the segment: exact
                    fold.finish(acc);
                    store_set16(tc.sets + (size_t)op * 128, acc);
                    continue;
                }
                iv.step(fold.A, fold.O);
                if ((w0.z & OPF_ROOT) && !(p.flags & RUN_BLOCK_MODE)) {
                    fitch_root_ref(p, tile, lane, iv.lo);
                    fitch_root_ref(p, tile, lane, iv.hi);
                }
                head = op;
                if (!__any_sync(FULL, iv.open() != 0)) {
#pragma unroll
                    for (int k = 0; k < 16; k++) acc[k] = iv.lo[k];
                    store_set16(tc.sets + (size_t)op * 128, acc);
                    if (w0.z & OPF_SIGNAL) signal_flag(tc.done + op, p.epoch, lane);
                    resolved = op;
                    first = op + 1;
                    break;
                }
            }
        }
        if (first < ck.op_end) fwd_meta_load(p, m, first, ck.op_end, lane);
        for (int i = 0; i < FWD_DEPTH && first + i < ck.op_end; i++) {
            if (!fwd_issue<JS, 4>(p, ck, m, tc, dc, ring_l + i * STAGE, first + i, lane, tr)) return false;
        }
        int stage = 0;
        for (int op = first; op < ck.op_end; op++) {
            if (op + FWD_DEPTH >= m.wb + META_OPS && m.wb + META_OPS < ck.op_end) fwd_meta_load(p, m, op, ck.op_end, lane);
            const int4 w0 = m.ops[2 * (op - m.wb)], w1 = m.ops[2 * (op - m.wb) + 1];  // {ref_begin, n_refs, flags, bits}, {ref0, ref1}
            cp_async_wait_stage<FWD_DEPTH>(ck.op_end - 1 - op);
            uint4* st = ring_l + stage * STAGE;
            const int type = p.leaf_present ? FT_GENERIC : ((w0.z >> OPF_TYPE_SHIFT) & 15);
            if (type == FT_LEAF_LEAF) {
                const uint4 l0 = st[0], l1 = st[32];
                const uint32_t c0[4] = {l0.x, l0.y, l0.z, l0.w}, c1[4] = {l1.x, l1.y, l1.z, l1.w};
                fitch_leaf_leaf(c0, c1, acc);
            } else if (type == FT_LEAF_ACC) {
                const uint4 l0 = st[0];
                const uint32_t c0[4] = {l0.x, l0.y, l0.z, l0.w};
                uint32_t X[16];
#pragma unroll
                for (int k = 0; k < 16; k++) X[k] = acc[k];
                fitch_leaf_set(c0, X, acc);
            } else if (type == FT_LEAF_INT || type == FT_INT_ACC) {
                const uint32_t ref = (uint32_t)(type == FT_LEAF_INT ? w1.y : w1.x);
                uint32_t X[16];
                if (fwd_set_prefetched(ref, op)) stage_set16(st, X);
                else row_set16(tc.sets + (size_t)(ref & REF_IDX_MASK) * 128, X);
                if (type == FT_LEAF_INT) {
                    const uint4 l0 = st[0];
                    const uint32_t c0[4] = {l0.x, l0.y, l0.z, l0.w};
                    fitch_leaf_set(c0, X, acc);
                } else {
                    uint32_t Y[16];
#pragma unroll
                    for (int k = 0; k < 16; k++) Y[k] = acc[k];
                    fitch_set_set(X, Y, acc);
                }
            } else {
                FitchFold fold;
                fold.reset();
                int nl = 0, ni = 0;
                for (int r = 0; r < w0.y; r++) {
                    const uint32_t ref = fwd_ref(p, m, w0.x + r);
                    const uint32_t kind = ref >> 30, idx = ref & REF_IDX_MASK;
                    if (kind == REF_LEAF) {
                        uint4 c;
                        if (nl < 2) c = st[nl * 32];
                        else c = ld_stream(tc.leaf + (size_t)idx * 32);
                        nl++;
                        uint32_t cc[4] = {c.x, c.y, c.z, c.w};
                        fold.add_leaf(cc, leaf_present_mask(p, idx));
                    } else if (kind == REF_ACC) {
                        fold.add_set(acc);
                    } else if (SPEC && kind == REF_CHAIN) {  // not speculating (presence mask): wait for the segment below
                        if (!wait_flag(tc.done + idx, p.epoch, p.error, lane, tr)) return false;
                        uint32_t S[16];
                        row_set16(tc.sets + (size_t)idx * 128, S);
                        fold.add_set(S);
                    } else {
                        uint32_t S[16];
                        if (ni == 0 && fwd_set_prefetched(ref, op)) {
                            stage_set16(st, S);
                        } else {
                            if (ref & REF_EXT) {
                                if (!wait_dep(p, ck, tc.done, dc, int(idx), lane, tr)) return false;
                            }
                            row_set16(tc.sets + (size_t)ref_row(p, ck, ref) * 128, S);
                        }
                        ni++;
                        fold.add_set(S);
                    }
                }
                fold.finish(acc);
            }
            if ((w0.z & OPF_ROOT) && !(p.flags & RUN_BLOCK_MODE)) fitch_root_ref(p, tile, lane, acc);
            store_set16(tc.sets + (size_t)op * 128, acc);
            if (w0.z & OPF_SIGNAL) signal_flag(tc.done + op, p.epoch, lane);
            // the stage of this op is consumed and its result stored: refill the stage for the op FWD_DEPTH ahead
            if (op + FWD_DEPTH < ck.op_end) {
                if (!fwd_issue<JS, 4>(p, ck, m, tc, dc, st, op + FWD_DEPTH, lane, tr)) return false;
            }
            stage = (stage + 1 == FWD_DEPTH) ? 0 : stage + 1;
        }
        if (spec) {  // the value from below is needed now: redo the path ops that depended on it
            if (!wait_flag(tc.done + ck.chain_row, p.epoch, p.error, lane, tr)) return false;
            uint32_t S[16];
            row_set16(tc.sets + (size_t)ck.chain_row * 128, S);
            const int end = resolved >= 0 ? resolved : ck.op_end;
            int head = -1;
            for (int op = ck.chain_op; op < end; op++) {
                const int4 w0 = __ldg(reinterpret_cast<const int4*>(p.fwd_ops + op));
                if (!fwd_on_path(p, w0, op, head)) continue;
                FitchFold fold;
                if (!fitch_fold_known<false>(p, ck, tc, dc, w0, op, head, acc, lane, fold, tr)) return false;
                fold.add_set(S);
                fold.finish(S);
                if ((w0.z & OPF_ROOT) && !(p.flags & RUN_BLOCK_MODE)) fitch_root_ref(p, tile, lane, S);
                store_set16(tc.sets + (size_t)op * 128, S);
                if (w0.z & OPF_SIGNAL) signal_flag(tc.done + op, p.epoch, lane);
                head = op;
            }
        }
        trace_end(p, tr, chunk, tile, lane);
    }
    return true;
}

template <bool SPEC>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32, SPEC ? 4 : 5) fitch_forward_kernel(RunParams p, int chunk_begin, int n_chunks) {
    extern __shared__ uint4 smem[];
    const int lane = threadIdx.x & 31;
    uint4* ring = smem + (size_t)(threadIdx.x >> 5) * FITCH_FWD_PER_WARP;
    ItemIter it;
    TraceItem tr;
    int chunk, tile;
    while (next_item(p, it, chunk_begin, n_chunks, chunk, tile, lane, tr))
        if (!fitch_forward_item<SPEC>(p, ring, chunk, tile, lane, tr)) return;
}

// ------------------------------------------------------------------ backward: shared pieces
// stage layout: [J set-row vectors][2 leaf rows], each 32 lanes wide; J = 4 (Fitch) or 8 (Sankoff)
template <int J>
__device__ __forceinline__ void bwd_issue(const BwdMeta& m, const TileCtx& tc, uint4* st, int op) {
    const uint4* srow = tc.sets + (size_t)op * (J * 32);
#pragma unroll
    for (int j = 0; j < J; j++) cp_async16(st + j * 32, srow + j * 32);
    const int4 b1 = m.ops[2 * (op - m.lo) + 1];  // n_leaves, flags, leaf0 slot, leaf1 slot
    if (b1.x > 0) cp_async16(st + J * 32, tc.leaf + (size_t)b1.z * 32);
    if (b1.x > 1) cp_async16(st + (J + 1) * 32, tc.leaf + (size_t)b1.w * 32);
    cp_async_commit();
}

// bulk variant: `stage_base` / `sets_base` / `leaf_base` carry NO lane offset; the elected lane issues the rows of one op
template <int J>
__device__ __forceinline__ void bwd_issue_bulk(const BwdMeta& m, const uint4* sets_base, const uint4* leaf_base, uint4* stage_base,
                                               unsigned long long* bar, int op, int lane) {
    __syncwarp();  // every lane has consumed what this stage held
    if (lane == 0) {
        const int4 b1 = m.ops[2 * (op - m.lo) + 1];  // n_leaves, flags, leaf0 slot, leaf1 slot
        const int nl = min(b1.x, 2);
        mbar_expect_tx(bar, unsigned(J * 512 + nl * 512));
        bulk_copy(stage_base, sets_base + (size_t)op * (J * 32), J * 512, bar);
        if (nl > 0) bulk_copy(stage_base + J * 32, leaf_base + (size_t)b1.z * 32, 512, bar);
        if (nl > 1) bulk_copy(stage_base + (J + 1) * 32, leaf_base + (size_t)b1.w * 32, 512, bar);
    }
}

// parent's assigned state from its parked slot (possibly written by another chunk)
__device__ __forceinline__ bool bwd_parent_slot(const RunParams& p, const BwdHead& h, int tile, int lane, uint32_t P[4],
                                                uint32_t& pvis, TraceItem& tr) {
    const size_t fi = fslot_index(p, h.b0.y, tile);
    if (h.b1.y & OPF_PARENT_EXT) {
        if (!wait_flag(p.fdone + fi, p.epoch, p.error, lane, tr)) return false;
    }
    const uint32_t* fs = p.fstore + fi * FSLOT_WORDS;
    uint4 a = ld_l2(reinterpret_cast<const uint4*>(fs) + lane);
    pvis = __ldcg(fs + 128 + lane);
    P[0] = a.x; P[1] = a.y; P[2] = a.z; P[3] = a.w;
    return true;
}

// what follows the assignment of an internal node, shared by Fitch and Sankoff: its own record, the parked
// state for later children, and its leaf children (a present leaf is always assigned its own code).
// The common case (every leaf present, no state dump) is straight-line for the first two leaves: one ballot each,
// and the leaf's node id is only fetched when it really has a record.
__device__ __forceinline__ void bwd_finish_op(const RunParams& p, const BwdMeta& m, const TileCtx& tc, StageCursor& sc,
                                              const BwdHead& h, const uint4* leaf_stage, uint32_t* stack, int tile, int lane,
                                              const uint32_t P[4], const uint32_t F[4], uint32_t vis, bool sankoff_block,
                                              bool own_record = true) {
    if (own_record) emit(p, sc, h.b0.x, tile, lane, vis & differs4(F, P), P, F);
    if (h.b1.y & OPF_PUSH) {  // a later op of this chunk needs this state: park it in the warp's shared-memory stack
        uint32_t* e = stack + ((h.b1.y >> OPF_PUSH_SHIFT) & 15) * FSLOT_WORDS;
        reinterpret_cast<uint4*>(e)[lane] = make_uint4(F[0], F[1], F[2], F[3]);
        e[128 + lane] = vis;
    }
    if (h.b0.z >= 0) {
        const size_t fi = fslot_index(p, h.b0.z, tile);
        uint32_t* fs = p.fstore + fi * FSLOT_WORDS;
        reinterpret_cast<uint4*>(fs)[lane] = make_uint4(F[0], F[1], F[2], F[3]);
        fs[128 + lane] = vis;
        if (h.b1.y & OPF_SIGNAL_F) signal_flag(p.fdone + fi, p.epoch, lane);
    }
    const bool plain = p.states == nullptr && p.leaf_present == nullptr;
    if (p.states) store_state(p, h.b0.x, tile, lane, F, vis);
    int l0 = 0;
    if (plain) {
        const int nfast = min(h.b1.x, 2);
        for (; l0 < nfast; l0++) {
            const uint4 c = leaf_stage[l0 * 32];
            const uint32_t cc[4] = {c.x, c.y, c.z, c.w};
            const uint32_t mut = vis & differs4(cc, F);
            if (__ballot_sync(FULL, mut != 0)) emit(p, sc, bwd_leaf(p, m, h.b0.w + l0).y, tile, lane, mut, F, cc);
        }
    }
    for (int l = l0; l < h.b1.x; l++) {
        const int2 lf = bwd_leaf(p, m, h.b0.w + l);  // slot, node
        uint4 c;
        if (l < 2) c = leaf_stage[l * 32];
        else c = ld_stream(tc.leaf + (size_t)lf.x * 32);
        uint32_t cc[4] = {c.x, c.y, c.z, c.w};
        uint32_t present = leaf_present_mask(p, lf.x);
        if (sankoff_block && !present) {  // omitted block leaf = "absent" state (fitchSankoff.cpp:711-714)
            cc[0] = cc[1] = cc[2] = cc[3] = 0;
            present = FULL;
        }
        const uint32_t lvis = vis & present;
        emit(p, sc, lf.y, tile, lane, lvis & differs4(cc, F), F, cc);
        if (p.states) {
            uint32_t m4[4] = {cc[0] & lvis, cc[1] & lvis, cc[2] & lvis, cc[3] & lvis};
            store_state(p, lf.y, tile, lane, m4, lvis);
        }
    }
}

// ------------------------------------------------------------------ Fitch backward + mutation detection
constexpr int FITCH_BWD_STAGE = (4 + 2) * 32,
              FITCH_BWD_PER_WARP = BWD_DEPTH * FITCH_BWD_STAGE + BWD_META_U4 + BWD_STACK_U4 + (PMB_BULK ? (BWD_DEPTH * 8 + 15) / 16 : 0);
// `phases`: bit s = the parity the next wait on stage s's mbarrier expects (bulk variant; lives across items)
template <bool SPEC>
__device__ __forceinline__ bool fitch_backward_item(const RunParams& p, uint4* ring, StageCursor& sc, int chunk, int tile, int lane,
                                                    TraceItem& tr, unsigned& phases) {
    constexpr int J = 4, STAGE = FITCH_BWD_STAGE;
    BwdMeta m;
    m.ops = reinterpret_cast<int4*>(ring + BWD_DEPTH * STAGE);
    m.leaves = reinterpret_cast<int2*>(m.ops + 2 * META_OPS);
    uint32_t* stack = reinterpret_cast<uint32_t*>(ring + BWD_DEPTH * STAGE + BWD_META_U4);
    uint4* const ring_l = ring + lane;
#if PMB_BULK
    unsigned long long* const bars = reinterpret_cast<unsigned long long*>(ring + BWD_DEPTH * STAGE + BWD_META_U4 + BWD_STACK_U4);
    const uint4* const sets_base = p.sets + (size_t)tile * p.n_ops * (J * 32);
    const uint4* const leaf_base = p.leaf_planes + (size_t)tile * p.n_rows * 32;
#endif
    {
        const Chunk ck = p.chunks[chunk];
        const TileCtx tc = tile_ctx<J>(p, tile, lane);
        const int last = ck.op_end - 1;
        uint32_t accF[4] = {0, 0, 0, 0}, accVis = 0;
        // Chain segment: the state handed down by the segment above is not waited for. The states it may be are
        // narrowed down the segment's heavy path until one is left in every column (op `resolved`); that op's subtree
        // is processed first, then -- once the segment above has published -- the ops above it, and its own record.
        int resolved = -1;
        uint32_t specF[4] = {0, 0, 0, 0}, specVis = 0;
        if (SPEC && p.leaf_present == nullptr && (ck.flags & CHUNK_CHAIN_TOP)) {
            uint32_t Q[16];
#pragma unroll
            for (int k = 0; k < 16; k++) Q[k] = FULL;
            for (int op = last; op >= ck.op_begin; op--) {
                if (op != last && !(__ldg(&p.bwd_ops[op].flags) & OPF_HEAVY)) continue;
                uint32_t S[16];
                row_set16(tc.sets + (size_t)op * 128, S);
                fitch_candidates_step(Q, S);
                if (!__any_sync(FULL, candidates_open(Q) != 0)) {
                    resolved = op;
                    encode16(Q, specF);
                    specVis = __ldg(p.colparams + (size_t)tile * 128 + 96 + lane).z;  // every set is non-empty: visited = valid column
#pragma unroll
                    for (int k = 0; k < 4; k++) specF[k] &= specVis;
                    break;
                }
            }
        }
        for (int range = (resolved >= 0 ? 0 : 1); range < 2; range++) {
        // range 0: the resolved op (state known, own record postponed) and everything below it;
        // range 1: the ops above it in full, then the resolved op's own record -- or, without speculation, the whole chunk
        const int hi = range == 0 ? resolved : last;
        const int lo = (range == 1 && resolved >= 0) ? resolved : ck.op_begin;
        bwd_meta_load(p, m, hi, lo, lane);
#if PMB_BULK
        for (int i = 0; i < BWD_DEPTH && hi - i >= lo; i++) bwd_issue_bulk<J>(m, sets_base, leaf_base, ring + i * STAGE, bars + i, hi - i, lane);
#else
        for (int i = 0; i < BWD_DEPTH && hi - i >= lo; i++) bwd_issue<J>(m, tc, ring_l + i * STAGE, hi - i);
#endif
        int stage = 0;
        for (int op = hi; op >= lo; op--) {
            if (op - BWD_DEPTH < m.lo && m.lo > lo) bwd_meta_load(p, m, op, lo, lane);
            BwdHead h;
            h.b0 = m.ops[2 * (op - m.lo)];
            h.b1 = m.ops[2 * (op - m.lo) + 1];
            const bool given = range == 0 && op == resolved, own_only = range == 1 && op == resolved;
            uint32_t P[4] = {0, 0, 0, 0}, pvis = 0, F[4], vis;
            if (given) {
            } else if (h.b0.y == PARENT_ACC) {
                P[0] = accF[0]; P[1] = accF[1]; P[2] = accF[2]; P[3] = accF[3];
                pvis = accVis;
            } else if (h.b0.y <= PARENT_STACK0) {
                const uint32_t* e = stack + (PARENT_STACK0 - h.b0.y) * FSLOT_WORDS;
                const uint4 a = reinterpret_cast<const uint4*>(e)[lane];
                pvis = e[128 + lane];
                P[0] = a.x; P[1] = a.y; P[2] = a.z; P[3] = a.w;
            } else if (h.b0.y >= 0) {
                if (!bwd_parent_slot(p, h, tile, lane, P, pvis, tr)) return false;
            }
#if PMB_BULK
            mbar_wait(bars + stage, (phases >> stage) & 1u);
            phases ^= 1u << stage;
#else
            cp_async_wait_stage<BWD_DEPTH>(op - lo);
#endif
            uint4* st = ring_l + stage * STAGE;
            uint32_t S[16];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const uint4 v = st[j * 32];
                S[4 * j] = v.x; S[4 * j + 1] = v.y; S[4 * j + 2] = v.z; S[4 * j + 3] = v.w;
            }
            if (given) {
                F[0] = specF[0]; F[1] = specF[1]; F[2] = specF[2]; F[3] = specF[3];
                vis = specVis;
            } else if (h.b0.y == PARENT_ROOT) {
                const uint4* cp = p.colparams + (size_t)tile * 128;
                uint4 pc = __ldg(cp + lane), ov = __ldg(cp + 32 + lane), fl = __ldg(cp + 96 + lane);
                P[0] = pc.x; P[1] = pc.y; P[2] = pc.z; P[3] = pc.w;
                uint32_t o4[4] = {ov.x, ov.y, ov.z, ov.w};
                const uint32_t ov_valid = fl.x & fl.z, colmask = fl.z;
                if (p.flags & RUN_BLOCK_MODE) {
                    // blockFitchBackwardPassNew: the root is treated like any node with parentState (:249-263)
                    uint32_t v0;
                    fitch_assign(S, P, colmask, F, v0);
                    vis = (v0 | ov_valid) & colmask;
#pragma unroll
                    for (int k = 0; k < 4; k++) F[k] = ((ov_valid & o4[k]) | (~ov_valid & F[k])) & vis;
                } else {
                    fitch_assign_root(S, o4, ov_valid, colmask, F, vis);
                }
            } else {
                fitch_assign(S, P, pvis, F, vis);
            }
            if (own_only) emit(p, sc, h.b0.x, tile, lane, vis & differs4(F, P), P, F);
            else bwd_finish_op(p, m, tc, sc, h, st + J * 32, stack, tile, lane, P, F, vis, false, !given);
            // this stage has been consumed by this lane: refill it for the op BWD_DEPTH further down
#if PMB_BULK
            if (op - BWD_DEPTH >= lo) bwd_issue_bulk<J>(m, sets_base, leaf_base, ring + stage * STAGE, bars + stage, op - BWD_DEPTH, lane);
#else
            if (op - BWD_DEPTH >= lo) bwd_issue<J>(m, tc, st, op - BWD_DEPTH);
#endif
            stage = (stage + 1 == BWD_DEPTH) ? 0 : stage + 1;
            accF[0] = F[0]; accF[1] = F[1]; accF[2] = F[2]; accF[3] = F[3];
            accVis = vis;
        }
        }
        trace_end(p, tr, chunk, tile, lane);
    }
    return true;
}

template <bool SPEC>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32) fitch_backward_kernel(RunParams p, int chunk_begin, int n_chunks) {
    extern __shared__ uint4 smem[];
    const int lane = threadIdx.x & 31;
    uint4* ring = smem + (size_t)(threadIdx.x >> 5) * FITCH_BWD_PER_WARP;
    unsigned phases = 0;
#if PMB_BULK
    {
        unsigned long long* bars = reinterpret_cast<unsigned long long*>(ring + BWD_DEPTH * FITCH_BWD_STAGE + BWD_META_U4 + BWD_STACK_U4);
        if (lane == 0) {
            for (int s = 0; s < BWD_DEPTH; s++) mbar_init(bars + s, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
    }
#endif
    ItemIter it;
    TraceItem tr;
    StageCursor sc;
    int chunk, tile;
    while (next_item(p, it, chunk_begin, n_chunks, chunk, tile, lane, tr))
        if (!fitch_backward_item<SPEC>(p, ring, sc, chunk, tile, lane, tr, phases)) return;
}

// ------------------------------------------------------------------ Sankoff forward
// first non-accumulator set row either comes prefetched from the stage (G planes + first H vector) or is loaded here
template <int B>
__device__ __forceinline__ bool sankoff_forward_op(const RunParams& p, const Chunk& ck, DepCursor& dc, const FwdMeta& m,
                                                   const TileCtx& tc, const int4 w0, int op, const uint4* st, int lane,
                                                   uint32_t accG[16], uint32_t accH[16], TraceItem& tr) {
    SankoffFold<B> fold;
    fold.reset();
    int nl = 0, ni = 0;
    for (int r = 0; r < w0.y; r++) {
        const uint32_t ref = fwd_ref(p, m, w0.x + r);
        const uint32_t kind = ref >> 30, idx = ref & REF_IDX_MASK;
        if (kind == REF_LEAF) {
            uint4 c;
            if (nl < 2) c = st[nl * 32];
            else c = ld_stream(tc.leaf + (size_t)idx * 32);
            nl++;
            uint32_t present = leaf_present_mask(p, idx);
            uint32_t cc[4] = {c.x, c.y, c.z, c.w};
            if ((p.flags & RUN_BLOCK_MODE) && !present) {  // omitted block leaf = "absent" state (:711-714)
                cc[0] = cc[1] = cc[2] = cc[3] = 0;
                present = FULL;
            }
            fold.add_leaf(cc, present);
        } else if (kind == REF_ACC) {
            fold.add_set(accG, sankoff_none(accG, accH));
        } else if (kind == REF_CHAIN) {  // a chain segment that is not evaluated speculatively waits for the segment below
            if (!wait_flag(tc.done + idx, p.epoch, p.error, lane, tr)) return false;
            const uint4* row = tc.sets + (size_t)idx * 256;
            uint32_t G[16];
            row_set16(row, G);
            const uint32_t h0 = ld_l2(row + 128).x;
            fold.add_set(G, h0 & ~G[0]);
        } else {
            uint32_t G[16], h0;
            if (ni == 0 && fwd_set_prefetched(ref, op)) {
                stage_set16(st, G);
                h0 = st[(2 + 4) * 32].x;
            } else {
                if (ref & REF_EXT) {
                    if (!wait_dep(p, ck, tc.done, dc, int(idx), lane, tr)) return false;
                }
                const uint4* row = tc.sets + (size_t)ref_row(p, ck, ref) * 256;
                row_set16(row, G);
                h0 = ld_l2(row + 128).x;
            }
            ni++;
            fold.add_set(G, h0 & ~G[0]);
        }
    }
    fold.finish(accG, accH);
    return true;
}

// ---- chain segments, Sankoff (plane_math.h): helpers with direct loads, only used without a presence mask, so no
// vector is ever NONE. Speculation covers segments whose path ops are binary and whose inlined light subtrees have at
// most three children per node (everything a bifurcating tree produces); any other segment simply waits.
__device__ __forceinline__ void store_gh(uint4* out, const uint32_t G[16], const uint32_t H[16]) {
#pragma unroll
    for (int j = 0; j < 4; j++) {
        out[j * 32] = make_uint4(G[4 * j], G[4 * j + 1], G[4 * j + 2], G[4 * j + 3]);
        out[(4 + j) * 32] = make_uint4(H[4 * j], H[4 * j + 1], H[4 * j + 2], H[4 * j + 3]);
    }
}
// exact evaluation of an op with at most 3 children, all known; acc = previous op's result in, this op's result out
__device__ __forceinline__ bool sankoff_eval_small(const RunParams& p, const Chunk& ck, const TileCtx& tc, DepCursor& dc, const int4 w0,
                                                   uint32_t accG[16], uint32_t accH[16], int lane, TraceItem& tr) {
    SankoffFold<2> fold;
    fold.reset();
    for (int r = 0; r < w0.y; r++) {
        const uint32_t ref = __ldg(p.refs + w0.x + r), kind = ref >> 30, idx = ref & REF_IDX_MASK;
        if (kind == REF_LEAF) {
            const uint4 c = ld_stream(tc.leaf + (size_t)idx * 32);
            const uint32_t cc[4] = {c.x, c.y, c.z, c.w};
            fold.add_leaf(cc, FULL);
        } else if (kind == REF_ACC) {
            fold.add_set(accG, 0u);
        } else {
            if (ref & REF_EXT) {
                if (!wait_dep(p, ck, tc.done, dc, int(idx), lane, tr)) return false;
            }
            uint32_t G[16];
            row_set16(tc.sets + (size_t)ref_row(p, ck, ref) * 256, G);
            fold.add_set(G, 0u);
        }
    }
    fold.finish(accG, accH);
    return true;
}
// G planes of the KNOWN child of a binary op on the path (the ref that is not the path's)
template <bool ACC_REGS>
__device__ __forceinline__ bool sankoff_known_child(const RunParams& p, const Chunk& ck, const TileCtx& tc, DepCursor& dc, const int4 w0,
                                                    int op, int head, const uint32_t accG[16], int lane, uint32_t g[16], TraceItem& tr) {
    for (int r = 0; r < w0.y; r++) {
        const uint32_t ref = __ldg(p.refs + w0.x + r), kind = ref >> 30, idx = ref & REF_IDX_MASK;
        if (kind == REF_CHAIN) continue;
        if (kind == REF_LEAF) {
            const uint4 c = ld_stream(tc.leaf + (size_t)idx * 32);
            const uint32_t cc[4] = {c.x, c.y, c.z, c.w};
            sankoff_leaf_g(cc, FULL, g);
        } else if (kind == REF_ACC) {
            if (head >= 0 && head == op - 1) continue;
            if (ACC_REGS) {
#pragma unroll
                for (int k = 0; k < 16; k++) g[k] = accG[k];
            } else {
                row_set16(tc.sets + (size_t)(op - 1) * 256, g);
            }
        } else {
            if (!(ref & REF_EXT) && head >= 0 && int(idx) == head) continue;
            if (ref & REF_EXT) {
                if (!wait_dep(p, ck, tc.done, dc, int(idx), lane, tr)) return false;
            }
            row_set16(tc.sets + (size_t)ref_row(p, ck, ref) * 256, g);
        }
    }
    return true;
}

// Sankoff rows are [G: 4 vectors][H: 4 vectors]; the forward pass only needs G and the first H vector (NONE marker)
// of a child, which are contiguous: JS = 5 of JROW = 8.
// MAXB = widest child counter any op of this tree needs (2: up to 3 children, 4: 15, 8: 255, 20: more), so
// that binary trees do not pay registers for polytomy paths. SPEC = the program has chain segments.
template <int MAXB, bool SPEC>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32) sankoff_forward_kernel(RunParams p, int chunk_begin, int n_chunks) {
    extern __shared__ uint4 smem[];
    constexpr int JS = 5, STAGE = (2 + JS) * 32, PER_WARP = FWD_DEPTH * STAGE + FWD_META_U4;
    const int lane = threadIdx.x & 31;
    uint4* ring = smem + (size_t)(threadIdx.x >> 5) * PER_WARP;
    FwdMeta m;
    m.ops = reinterpret_cast<int4*>(ring + FWD_DEPTH * STAGE);
    m.refs = reinterpret_cast<uint32_t*>(m.ops + 2 * META_OPS);
    uint4* const ring_l = ring + lane;
    ItemIter it;
    TraceItem tr;
    int chunk, tile;
    while (next_item(p, it, chunk_begin, n_chunks, chunk, tile, lane, tr)) {
        const Chunk ck = p.chunks[chunk];
        const TileCtx tc = tile_ctx<8>(p, tile, lane);
        DepCursor dc;
        uint32_t accG[16], accH[16];
#pragma unroll
        for (int k = 0; k < 16; k++) { accG[k] = 0; accH[k] = 0; }
        // Chain segment (see fitch_forward_kernel): bounds on the zero-excess set entering from the segment below until
        // no column depends on it; G of the op where they meet is exact, its H is redone at the end with the ops before.
        bool spec = SPEC && ck.chain_op >= 0 && p.leaf_present == nullptr;
        int first = ck.op_begin, resolved = -1;
        if (spec) {
            FitchInterval iv;
            iv.reset();
            int head = -1;
            first = ck.op_end;
            for (int op = ck.op_begin; op < ck.op_end; op++) {
                const int4 w0 = __ldg(reinterpret_cast<const int4*>(p.fwd_ops + op));
                const bool on_path = fwd_on_path(p, w0, op, head);
                if ((on_path && w0.y != 2) || (!on_path && w0.w != 2)) {  // not covered: fall back to waiting
                    spec = false;
                    break;
                }
                if (!on_path) {  // a light subtree evaluated inside the segment: exact
                    if (!sankoff_eval_small(p, ck, tc, dc, w0, accG, accH, lane, tr)) return;
                    store_gh(tc.sets + (size_t)op * 256, accG, accH);
                    continue;
                }
                uint32_t g[16];
                if (!sankoff_known_child<true>(p, ck, tc, dc, w0, op, head, accG, lane, g, tr)) return;
#pragma unroll
                for (int k = 0; k < 16; k++) g[k] = ~g[k];  // zero-excess set of the known child
                iv.step(g, g);
                head = op;
                if (!__any_sync(FULL, iv.open() != 0)) {
#pragma unroll
                    for (int k = 0; k < 16; k++) { accG[k] = ~iv.lo[k]; accH[k] = 0; }
                    store_gh(tc.sets + (size_t)op * 256, accG, accH);  // G exact, H provisional (readers ahead only use G)
                    if (w0.z & OPF_SIGNAL) signal_flag(tc.done + op, p.epoch, lane);
                    resolved = op;
                    first = op + 1;
                    break;
                }
            }
            if (!spec) {
                first = ck.op_begin;
#pragma unroll
                for (int k = 0; k < 16; k++) { accG[k] = 0; accH[k] = 0; }
            }
        }
        if (first < ck.op_end) fwd_meta_load(p, m, first, ck.op_end, lane);
        for (int i = 0; i < FWD_DEPTH && first + i < ck.op_end; i++) {
            if (!fwd_issue<JS, 8>(p, ck, m, tc, dc, ring_l + i * STAGE, first + i, lane, tr)) return;
        }
        int stage = 0;
        for (int op = first; op < ck.op_end; op++) {
            if (op + FWD_DEPTH >= m.wb + META_OPS && m.wb + META_OPS < ck.op_end) fwd_meta_load(p, m, op, ck.op_end, lane);
            const int4 w0 = m.ops[2 * (op - m.wb)];
            cp_async_wait_stage<FWD_DEPTH>(ck.op_end - 1 - op);
            uint4* st = ring_l + stage * STAGE;
            bool ok = true;
            const int type = (w0.z >> OPF_TYPE_SHIFT) & 15;
            if (type != FT_GENERIC) {
                // two children: closed form (plane_math.h sankoff_pair)
                const int4 w1 = m.ops[2 * (op - m.wb) + 1];
                uint32_t g1[16], g2[16], n1, n2;
                auto leaf_child = [&](int slot_k, uint32_t ref, uint32_t g[16], uint32_t& none) {
                    const uint4 c = st[slot_k * 32];
                    uint32_t cc[4] = {c.x, c.y, c.z, c.w};
                    uint32_t present = leaf_present_mask(p, ref & REF_IDX_MASK);
                    if ((p.flags & RUN_BLOCK_MODE) && !present) {  // omitted block leaf = "absent" state (:711-714)
                        cc[0] = cc[1] = cc[2] = cc[3] = 0;
                        present = FULL;
                    }
                    sankoff_leaf_g(cc, present, g);
                    none = ~present;
                };
                auto set_child = [&](uint32_t ref, uint32_t g[16], uint32_t& none) {
                    uint32_t h0;
                    if (fwd_set_prefetched(ref, op)) {
                        stage_set16(st, g);
                        h0 = st[(2 + 4) * 32].x;
                    } else {
                        const uint4* row = tc.sets + (size_t)(ref & REF_IDX_MASK) * 256;
                        row_set16(row, g);
                        h0 = ld_l2(row + 128).x;
                    }
                    none = h0 & ~g[0];
                };
                auto acc_child = [&](uint32_t g[16], uint32_t& none) {
#pragma unroll
                    for (int k = 0; k < 16; k++) g[k] = accG[k];
                    none = sankoff_none(accG, accH);
                };
                if (type == FT_LEAF_LEAF) {
                    leaf_child(0, (uint32_t)w1.x, g1, n1);
                    leaf_child(1, (uint32_t)w1.y, g2, n2);
                } else if (type == FT_LEAF_ACC) {
                    leaf_child(0, (uint32_t)w1.x, g1, n1);
                    acc_child(g2, n2);
                } else if (type == FT_LEAF_INT) {
                    leaf_child(0, (uint32_t)w1.x, g1, n1);
                    set_child((uint32_t)w1.y, g2, n2);
                } else {
                    set_child((uint32_t)w1.x, g1, n1);
                    acc_child(g2, n2);
                }
                sankoff_pair(g1, n1, g2, n2, accG, accH);
            } else if (MAXB == 2 || w0.w == 2) ok = sankoff_forward_op<2>(p, ck, dc, m, tc, w0, op, st, lane, accG, accH, tr);
            else if (MAXB == 4 || w0.w == 4) ok = sankoff_forward_op<4>(p, ck, dc, m, tc, w0, op, st, lane, accG, accH, tr);
            else if (MAXB == 8 || w0.w == 8) ok = sankoff_forward_op<8>(p, ck, dc, m, tc, w0, op, st, lane, accG, accH, tr);
            else ok = sankoff_forward_op<20>(p, ck, dc, m, tc, w0, op, st, lane, accG, accH, tr);
            if (!ok) return;
            uint4* out = tc.sets + (size_t)op * 256;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                out[j * 32] = make_uint4(accG[4 * j], accG[4 * j + 1], accG[4 * j + 2], accG[4 * j + 3]);
                out[(4 + j) * 32] = make_uint4(accH[4 * j], accH[4 * j + 1], accH[4 * j + 2], accH[4 * j + 3]);
            }
            if (w0.z & OPF_SIGNAL) signal_flag(tc.done + op, p.epoch, lane);
            if (op + FWD_DEPTH < ck.op_end) {
                if (!fwd_issue<JS, 8>(p, ck, m, tc, dc, st, op + FWD_DEPTH, lane, tr)) return;
            }
            stage = (stage + 1 == FWD_DEPTH) ? 0 : stage + 1;
        }
        if (spec) {  // the vector from below is needed now: redo the path ops up to and including the resolved one
            if (!wait_flag(tc.done + ck.chain_row, p.epoch, p.error, lane, tr)) return;
            uint32_t Gc[16];
            row_set16(tc.sets + (size_t)ck.chain_row * 256, Gc);
            const int end = resolved >= 0 ? resolved + 1 : ck.op_end;
            int head = -1;
            for (int op = ck.chain_op; op < end; op++) {
                const int4 w0 = __ldg(reinterpret_cast<const int4*>(p.fwd_ops + op));
                if (!fwd_on_path(p, w0, op, head)) continue;
                uint32_t g[16], G[16], H[16];
                if (!sankoff_known_child<false>(p, ck, tc, dc, w0, op, head, accG, lane, g, tr)) return;
                sankoff_pair(g, 0u, Gc, 0u, G, H);
                store_gh(tc.sets + (size_t)op * 256, G, H);
                if (w0.z & OPF_SIGNAL) signal_flag(tc.done + op, p.epoch, lane);
#pragma unroll
                for (int k = 0; k < 16; k++) Gc[k] = G[k];
                head = op;
            }
        }
        trace_end(p, tr, chunk, tile, lane);
    }
}

// ------------------------------------------------------------------ Sankoff backward + mutation detection
template <bool SPEC>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32) sankoff_backward_kernel(RunParams p, int chunk_begin, int n_chunks) {
    extern __shared__ uint4 smem[];
    constexpr int J = 8, STAGE = (J + 2) * 32, PER_WARP = BWD_DEPTH * STAGE + BWD_META_U4 + BWD_STACK_U4;
    const int lane = threadIdx.x & 31;
    uint4* ring = smem + (size_t)(threadIdx.x >> 5) * PER_WARP;
    BwdMeta m;
    m.ops = reinterpret_cast<int4*>(ring + BWD_DEPTH * STAGE);
    m.leaves = reinterpret_cast<int2*>(m.ops + 2 * META_OPS);
    uint32_t* stack = reinterpret_cast<uint32_t*>(ring + BWD_DEPTH * STAGE + BWD_META_U4);
    uint4* const ring_l = ring + lane;
    ItemIter it;
    TraceItem tr;
    StageCursor sc;
    int chunk, tile;
    while (next_item(p, it, chunk_begin, n_chunks, chunk, tile, lane, tr)) {
        const Chunk ck = p.chunks[chunk];
        const TileCtx tc = tile_ctx<J>(p, tile, lane);
        const int last = ck.op_end - 1;
        uint32_t accF[4] = {0, 0, 0, 0}, accVis = 0;
        // Chain segment (see fitch_backward_kernel): candidate states of the parent above are narrowed down the heavy
        // path until one is left in every column.
        int resolved = -1;
        uint32_t specF[4] = {0, 0, 0, 0}, specVis = 0;
        if (SPEC && p.leaf_present == nullptr && (ck.flags & CHUNK_CHAIN_TOP)) {
            uint32_t Q[16];
#pragma unroll
            for (int k = 0; k < 16; k++) Q[k] = FULL;
            for (int op = last; op >= ck.op_begin; op--) {
                if (op != last && !(__ldg(&p.bwd_ops[op].flags) & OPF_HEAVY)) continue;
                uint32_t G[16], H[16];
                row_set16(tc.sets + (size_t)op * 256, G);
                row_set16(tc.sets + (size_t)op * 256 + 128, H);
                sankoff_candidates_step(Q, G, H);
                if (!__any_sync(FULL, candidates_open(Q) != 0)) {
                    resolved = op;
                    encode16(Q, specF);
                    specVis = __ldg(p.colparams + (size_t)tile * 128 + 96 + lane).z;  // no vector is NONE: visited = valid column
#pragma unroll
                    for (int k = 0; k < 4; k++) specF[k] &= specVis;
                    break;
                }
            }
        }
        for (int range = (resolved >= 0 ? 0 : 1); range < 2; range++) {
        const int hi = range == 0 ? resolved : last;
        const int lo = (range == 1 && resolved >= 0) ? resolved : ck.op_begin;
        bwd_meta_load(p, m, hi, lo, lane);
        for (int i = 0; i < BWD_DEPTH && hi - i >= lo; i++) bwd_issue<J>(m, tc, ring_l + i * STAGE, hi - i);
        int stage = 0;
        for (int op = hi; op >= lo; op--) {
            if (op - BWD_DEPTH < m.lo && m.lo > lo) bwd_meta_load(p, m, op, lo, lane);
            BwdHead h;
            h.b0 = m.ops[2 * (op - m.lo)];
            h.b1 = m.ops[2 * (op - m.lo) + 1];
            const bool given = range == 0 && op == resolved, own_only = range == 1 && op == resolved;
            uint32_t P[4] = {0, 0, 0, 0}, pvis = 0, F[4], vis;
            if (given) {
            } else if (h.b0.y == PARENT_ACC) {
                P[0] = accF[0]; P[1] = accF[1]; P[2] = accF[2]; P[3] = accF[3];
                pvis = accVis;
            } else if (h.b0.y <= PARENT_STACK0) {
                const uint32_t* e = stack + (PARENT_STACK0 - h.b0.y) * FSLOT_WORDS;
                const uint4 a = reinterpret_cast<const uint4*>(e)[lane];
                pvis = e[128 + lane];
                P[0] = a.x; P[1] = a.y; P[2] = a.z; P[3] = a.w;
            } else if (h.b0.y >= 0) {
                if (!bwd_parent_slot(p, h, tile, lane, P, pvis, tr)) return;
            }
            cp_async_wait_stage<BWD_DEPTH>(op - lo);
            uint4* st = ring_l + stage * STAGE;
            uint32_t G[16], H[16];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const uint4 v = st[j * 32], w = st[(4 + j) * 32];
                G[4 * j] = v.x; G[4 * j + 1] = v.y; G[4 * j + 2] = v.z; G[4 * j + 3] = v.w;
                H[4 * j] = w.x; H[4 * j + 1] = w.y; H[4 * j + 2] = w.z; H[4 * j + 3] = w.w;
            }
            if (given) {
                F[0] = specF[0]; F[1] = specF[1]; F[2] = specF[2]; F[3] = specF[3];
                vis = specVis;
            } else if (h.b0.y == PARENT_ROOT) {
                const uint4* cp = p.colparams + (size_t)tile * 128;
                uint4 pc = __ldg(cp + lane), ov = __ldg(cp + 32 + lane), fl = __ldg(cp + 96 + lane);
                P[0] = pc.x; P[1] = pc.y; P[2] = pc.z; P[3] = pc.w;
                uint32_t o4[4] = {ov.x, ov.y, ov.z, ov.w}, undefined;
                sankoff_assign_root(G, H, o4, fl.x & fl.z, fl.z, F, vis, undefined);
                if (undefined) {  // reference: assert(minPtr != -1), fitchSankoff.cpp:505 (block variant returns, :754-757)
                    if (!(p.flags & RUN_BLOCK_MODE)) {
                        atomicOr(p.error, 1u);
                        atomicMin(p.error + 1, (unsigned)(tile * TILE_COLS + lane * 32 + (__ffs(undefined) - 1)));
                    }
                }
            } else {
                sankoff_assign(G, H, P, pvis, F, vis);
            }
            // leaf vector is 0 at its code and INF elsewhere: the parent's argmin always lands on that code
            if (own_only) emit(p, sc, h.b0.x, tile, lane, vis & differs4(F, P), P, F);
            else bwd_finish_op(p, m, tc, sc, h, st + J * 32, stack, tile, lane, P, F, vis, (p.flags & RUN_BLOCK_MODE) != 0, !given);
            if (op - BWD_DEPTH >= lo) bwd_issue<J>(m, tc, st, op - BWD_DEPTH);
            stage = (stage + 1 == BWD_DEPTH) ? 0 : stage + 1;
            accF[0] = F[0]; accF[1] = F[1]; accF[2] = F[2]; accF[3] = F[3];
            accVis = vis;
        }
        }
        trace_end(p, tr, chunk, tile, lane);
    }
}

// ------------------------------------------------------------------ scan over per-node counts (shard merging)
// Exclusive scan over per-node counts in two fully parallel kernels (block sums, then block-local scan + prefix of the
// block sums): used when column-range shards are merged. A pass itself compacts with the kernels below.
constexpr int SCAN_BLOCK = 1024, SCAN_ITEMS = 4, SCAN_TILE = SCAN_BLOCK * SCAN_ITEMS;

__device__ __forceinline__ unsigned long long block_reduce_sum(unsigned long long v, unsigned long long* sh) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(FULL, v, d);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    unsigned long long t = (threadIdx.x < 32) ? sh[threadIdx.x] : 0ull;  // SCAN_BLOCK / 32 == 32 warps
    if (threadIdx.x < 32) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) t += __shfl_down_sync(FULL, t, d);
        if (threadIdx.x == 0) sh[32] = t;
    }
    __syncthreads();
    unsigned long long r = sh[32];
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(SCAN_BLOCK) scan_sums_kernel(const unsigned int* counts, int n, unsigned long long* block_sums) {
    __shared__ unsigned long long sh[33];
    const int base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    unsigned long long s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++)
        if (base + k < n) s += counts[base + k];
    s = block_reduce_sum(s, sh);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = s;
}

__global__ void __launch_bounds__(SCAN_BLOCK) scan_apply_kernel(const unsigned int* counts, int n, const unsigned long long* block_sums,
                                                                long long* offsets) {
    __shared__ unsigned long long sh[33];
    __shared__ unsigned long long warp_tot[32];
    // prefix of the sums of the blocks before this one
    unsigned long long before = 0;
    for (int b = threadIdx.x; b < (int)blockIdx.x; b += SCAN_BLOCK) before += block_sums[b];
    before = block_reduce_sum(before, sh);
    const int base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    unsigned long long v[SCAN_ITEMS], s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        v[k] = (base + k < n) ? counts[base + k] : 0u;
        s += v[k];
    }
    // inclusive scan of the per-thread sums: warp shuffle scan, then the warp totals
    unsigned long long incl = s;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        unsigned long long t = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        unsigned long long w = warp_tot[lane], wi = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long t = __shfl_up_sync(FULL, wi, d);
            if (lane >= d) wi += t;
        }
        warp_tot[lane] = wi - w;  // exclusive
    }
    __syncthreads();
    unsigned long long run = before + warp_tot[warp] + (incl - s);
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        if (base + k < n) offsets[base + k] = (long long)run;
        run += v[k];
        if (base + k == n - 1) offsets[n] = (long long)run;
    }
}

// ------------------------------------------------------------------ ordered compaction
// An exclusive scan over the record counts of ALL directory entries, in (node, tile) order, is the final position of
// every staged segment, and the value at (node, 0) is the node's offset. Three small launches without any spinning:
// totals per group of CPT_GROUP entries, scan of the group totals (one block), then one thread per entry: rescan inside
// the group, copy the entry's (short) segment, and the end-of-run bookkeeping. Work is spread over all entries instead
// of one warp walking a node's tiles: the earlier per-node gather was latency-bound at 13 us (config 2) to 1 ms
// (config 4) per pass, and a thread copying several entries' records in a row is no better (61 us on config 3).
constexpr int CPT_GROUP = 256;  // entries per group = threads per block of compact_copy_kernel

__device__ __forceinline__ unsigned long long dir_valid(unsigned long long d, unsigned dir_tag) {
    if (unsigned(d >> DIR_TAG_SHIFT) != dir_tag) return 0ull;  // written by an earlier run: empty
    return d & ((1ull << DIR_TAG_SHIFT) - 1ull);
}

// one warp per group: lane l sums entries [8 l, 8 l + 8) of the group (dir is 16-byte aligned, groups are 2 KB)
__global__ void __launch_bounds__(256) compact_count_kernel(unsigned long long n_entries, const unsigned long long* dir, unsigned dir_tag,
                                                           unsigned int* group_totals, unsigned n_groups) {
    const unsigned g = (blockIdx.x * 256u + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (g >= n_groups) return;
    const unsigned long long e0 = (unsigned long long)g * CPT_GROUP + lane * 8u;
    unsigned sum = 0;
    if (e0 + 8 <= n_entries) {
#pragma unroll
        for (int k = 0; k < 8; k += 2) {
            const uint4 v = __ldcg(reinterpret_cast<const uint4*>(dir + e0 + k));
            sum += unsigned(dir_valid((unsigned long long)v.x | ((unsigned long long)v.y << 32), dir_tag) & 0x7FFull);
            sum += unsigned(dir_valid((unsigned long long)v.z | ((unsigned long long)v.w << 32), dir_tag) & 0x7FFull);
        }
    } else {
        for (int k = 0; k < 8; k++)
            if (e0 + k < n_entries) sum += unsigned(dir_valid(__ldcg(dir + e0 + k), dir_tag) & 0x7FFull);
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) sum += __shfl_down_sync(FULL, sum, s);
    if (lane == 0) group_totals[g] = sum;
}

// exclusive scan of the group totals by ONE block (a few thousand to a few hundred thousand groups): every thread owns
// SCAN1_ITEMS consecutive totals per round
constexpr int SCAN1_ITEMS = 8;
__global__ void __launch_bounds__(1024) compact_scan_kernel(const unsigned int* block_totals, int n_blocks, unsigned long long* block_prefix,
                                                            long long* offsets_end) {
    __shared__ unsigned long long s_w[32];
    __shared__ unsigned long long s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int b0 = 0; b0 < n_blocks; b0 += 1024 * SCAN1_ITEMS) {
        const int b = b0 + tid * SCAN1_ITEMS;
        unsigned v[SCAN1_ITEMS];
        unsigned long long sum = 0;
#pragma unroll
        for (int k = 0; k < SCAN1_ITEMS; k++) {
            v[k] = b + k < n_blocks ? block_totals[b + k] : 0u;
            sum += v[k];
        }
        unsigned long long incl = sum;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            unsigned long long t = __shfl_up_sync(FULL, incl, s);
            if (lane >= s) incl += t;
        }
        if (lane == 31) s_w[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            unsigned long long w = s_w[lane], wi = w;
#pragma unroll
            for (int s = 1; s < 32; s <<= 1) {
                unsigned long long t = __shfl_up_sync(FULL, wi, s);
                if (lane >= s) wi += t;
            }
            s_w[lane] = wi - w;  // exclusive
        }
        __syncthreads();
        const unsigned long long carry = s_carry;
        unsigned long long run = carry + s_w[warp] + incl - sum;
#pragma unroll
        for (int k = 0; k < SCAN1_ITEMS; k++) {
            if (b + k < n_blocks) block_prefix[b + k] = run;
            run += v[k];
        }
        __syncthreads();
        if (tid == 1023) s_carry = run;
        __syncthreads();
    }
    if (tid == 0) *offsets_end = (long long)s_carry;
}

// counters (128 bytes): layout below; [24,28) finished-block count of this kernel
__global__ void __launch_bounds__(CPT_GROUP) compact_copy_kernel(int n_nodes, int T, const unsigned long long* group_prefix,
                                                                long long* offsets, const unsigned long long* dir, unsigned dir_tag,
                                                                const uint16_t* staging, long long col_base, int32_t* pos,
                                                                uint8_t* type_code, unsigned long long* counters,
                                                                unsigned long long* run_words, unsigned long long staging_cap,
                                                                unsigned long long* tickets, int n_tickets) {
    __shared__ unsigned s_w[CPT_GROUP / 32];
    __shared__ unsigned s_last;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned long long n_entries = (unsigned long long)n_nodes * (unsigned long long)T;
    const unsigned long long e = (unsigned long long)blockIdx.x * CPT_GROUP + tid;
    const unsigned long long d = e < n_entries ? dir_valid(__ldcg(dir + e), dir_tag) : 0ull;
    const unsigned cnt = unsigned(d & 0x7FFull);
    unsigned incl = cnt;
#pragma unroll
    for (int s = 1; s < 32; s <<= 1) {
        unsigned t = __shfl_up_sync(FULL, incl, s);
        if (lane >= s) incl += t;
    }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    unsigned before = 0;
#pragma unroll
    for (int w = 0; w < CPT_GROUP / 32; w++)
        if (w < warp) before += s_w[w];
    if (e < n_entries) {
        const unsigned long long at = group_prefix[blockIdx.x] + before + (incl - cnt);
        unsigned long long node, tile;
        if (n_entries <= 0xFFFFFFFFull) {
            node = unsigned(e) / unsigned(T);
            tile = unsigned(e) - unsigned(node) * unsigned(T);
        } else {
            node = e / (unsigned long long)T;
            tile = e - node * (unsigned long long)T;
        }
        if (tile == 0) offsets[node] = (long long)at;
        // after a pool overflow nothing is copied: the host grows the pool and reruns the backward pass
        if (cnt && run_words[0] <= staging_cap) {
            const uint16_t* src = staging + (d >> 11);
            const long long cb = col_base + (long long)tile * TILE_COLS;
            for (unsigned q0 = 0; q0 < cnt; q0 += 4) {  // four independent loads in flight
                uint32_t r[4];
#pragma unroll
                for (int i = 0; i < 4; i++) r[i] = q0 + i < cnt ? src[q0 + i] : 0u;
#pragma unroll
                for (int i = 0; i < 4; i++)
                    if (q0 + i < cnt) {
                        pos[at + q0 + i] = int32_t(cb + (r[i] & 1023u));
                        type_code[at + q0 + i] = uint8_t(((r[i] >> 14) << 4) | ((r[i] >> 10) & 15u));
                    }
            }
        }
    }
    // ---- the last block to finish does the end-of-run bookkeeping
    __syncthreads();
    unsigned int* done_blocks = reinterpret_cast<unsigned int*>(counters + 3);
    if (tid == 0) {
        __threadfence();
        s_last = atomicAdd(done_blocks, 1u) == gridDim.x - 1 ? 1u : 0u;
    }
    __syncthreads();
    if (s_last) {
        if (tid == 0) {
            unsigned int* error = reinterpret_cast<unsigned int*>(run_words + 1);
            unsigned int* sticky = reinterpret_cast<unsigned int*>(counters + 2);
            const unsigned long long pool = run_words[0];
            const unsigned int er0 = error[0], er1 = error[1];
            const unsigned int st = er0 | (pool > staging_cap ? 4u : 0u);
            if (st) sticky[0] |= st;
            if ((er0 & 1u) && er1 < sticky[1]) sticky[1] = er1;
            counters[4] = pool;
            reinterpret_cast<unsigned int*>(counters + 5)[0] = er0;
            reinterpret_cast<unsigned int*>(counters + 5)[1] = er1;
            run_words[0] = 0ull;
            error[0] = 0u;
            error[1] = 0xFFFFFFFFu;
            done_blocks[0] = 0u;
        }
        for (int i = tid; i < n_tickets; i += CPT_GROUP) tickets[i] = 0ull;
    }
}

// counters (128 bytes): [0,8) staging records reserved, [8,12) error flags, [12,16) first bad column -- the "run words" of
// a pass; passes of odd parity use [64,80) instead where the staging pool and the directory are double-buffered, so that a
// backward kernel may run beside the compaction of the pass before it -- [16,20) sticky status, [20,24) sticky first bad
// column, [24,28) compact_copy_kernel's finished-block count, [32,48) snapshot of the run words for the host.
// compact_copy_kernel's last block folds the status into the sticky words (they survive until pmb_wait), snapshots the
// run words and resets them and the work tickets.

// ------------------------------------------------------------------ merging column-range shards (multi-GPU)
// A packed shard = {int64 n_mut, int64 n_nodes | int64 offsets[N+1] | int32 pos[cap] | uint8 type_code[cap]} (16-byte
// aligned sections). Shards are column ranges in ascending order, so a node's merged list is the concatenation of its
// per-shard lists in shard order.
__host__ __device__ inline size_t packed_pos_offset(long long n_nodes) { return (16 + size_t(n_nodes + 1) * 8 + 15) / 16 * 16; }
__host__ __device__ inline size_t packed_tc_offset(long long n_nodes, long long cap) {
    return (packed_pos_offset(n_nodes) + size_t(cap) * 4 + 15) / 16 * 16;
}
__host__ __device__ inline size_t packed_bytes(long long n_nodes, long long cap) {
    return (packed_tc_offset(n_nodes, cap) + size_t(cap) + 15) / 16 * 16;
}

// one launch instead of five copies: header, offsets, and the n = offsets[n_nodes] records actually present. `out` may be
// peer memory (the gathering rank's mailbox mapped over NVLink): the column-range gather is then this kernel's stores.
// A result that does not fit (`cap`), or whose offsets are not to be trusted because the pass overflowed its staging pool
// (`src_cap` = records the source arrays hold), is flagged in the header and NO record is copied: the merge skips it.
constexpr long long PACK_HDR_BAD = -1;
__global__ void pack_result_kernel(const long long* offsets, const int32_t* pos, const uint8_t* type_code, long long n_nodes,
                                   long long cap, long long src_cap, const unsigned long long* counters, unsigned char* out) {
    const long long total = offsets[n_nodes];
    // counters[4]: staging records the last pass reserved (snapshot by compact_copy_kernel); beyond src_cap nothing was copied
    const bool ok = total >= 0 && total <= cap && total <= src_cap && counters[4] <= (unsigned long long)src_cap;
    const long long n = ok ? total : 0;
    long long* hdr = reinterpret_cast<long long*>(out);
    long long* off_out = hdr + 2;
    int32_t* pos_out = reinterpret_cast<int32_t*>(out + packed_pos_offset(n_nodes));
    uint8_t* tc_out = out + packed_tc_offset(n_nodes, cap);
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i0 == 0) {
        hdr[0] = ok ? total : PACK_HDR_BAD;
        hdr[1] = n_nodes;
    }
    if (!ok) return;
    for (long long i = i0; i <= n_nodes; i += stride) off_out[i] = offsets[i];
    // records: 16 bytes per thread and step while both arrays are aligned (they are: cudaMalloc + 16-byte sections)
    const long long n4 = n / 4;
    const int4* pos4 = reinterpret_cast<const int4*>(pos);
    int4* pos_out4 = reinterpret_cast<int4*>(pos_out);
    for (long long i = i0; i < n4; i += stride) pos_out4[i] = pos4[i];
    const long long n16 = n / 16;
    const uint4* tc16 = reinterpret_cast<const uint4*>(type_code);
    uint4* tc_out16 = reinterpret_cast<uint4*>(tc_out);
    for (long long i = i0; i < n16; i += stride) tc_out16[i] = tc16[i];
    for (long long i = n4 * 4 + i0; i < n; i += stride) pos_out[i] = pos[i];
    for (long long i = n16 * 16 + i0; i < n; i += stride) tc_out[i] = type_code[i];
}

// a shard is merged only if its header is sane: packed for this tree, not flagged, within the capacity
__device__ __forceinline__ bool shard_ok(const unsigned char* shard, int n_nodes, long long cap) {
    const long long* hdr = reinterpret_cast<const long long*>(shard);
    return hdr[1] == n_nodes && hdr[0] >= 0 && hdr[0] <= cap;
}

// merge_err: bit 0 = a shard over capacity / flagged by its packer, bit 1 = a shard packed for another tree.
// rel[k * n_nodes + v] = records of node v in the shards before k = where shard k's segment starts inside the node's list
__global__ void merge_count_kernel(const unsigned char* packed, size_t shard_bytes, int n_shards, int n_nodes, long long cap,
                                   unsigned int* counts, unsigned int* rel, unsigned int* merge_err) {
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_nodes) return;
    unsigned int c = 0;
    for (int k = 0; k < n_shards; k++) {
        const unsigned char* sh = packed + k * shard_bytes;
        rel[(size_t)k * n_nodes + v] = c;
        if (!shard_ok(sh, n_nodes, cap)) {
            if (v == 0) atomicOr(merge_err, reinterpret_cast<const long long*>(sh)[1] == n_nodes ? 1u : 2u);
            continue;
        }
        const long long* off = reinterpret_cast<const long long*>(sh + 16);
        c += (unsigned int)(off[v + 1] - off[v]);
    }
    counts[v] = c;
}

// Source-parallel copy: blockIdx.y = shard, a thread takes four consecutive records of that shard (grid stride). The node of
// the first one by binary search in the shard's own offsets, the following ones by walking on; destination = node's merged
// offset + the shard's place inside the node (rel) + the record's place inside the segment. Per-node lists are very uneven
// -- the nodes next to the root of a gappy alignment hold tens of thousands of records, most nodes a few dozen -- and the
// round-1 warp-per-node copy spent a millisecond in the few long ones (2 shards x 0.66 M records: 1.2 ms, so that rank 0's
// merge no longer hid behind a 2 ms pass); a first record-parallel version searched the merged offsets and then walked the
// shards per OUTPUT record (8 shards, 5.3 M records: 95 us).
__global__ void merge_copy_kernel(const unsigned char* packed, size_t shard_bytes, int n_nodes, long long cap, const long long* merged_off,
                                  const unsigned int* rel, int32_t* pos, uint8_t* type_code) {
    const int k = blockIdx.y;
    const unsigned char* sh = packed + (size_t)k * shard_bytes;
    if (!shard_ok(sh, n_nodes, cap)) return;
    const long long n = reinterpret_cast<const long long*>(sh)[0];
    const long long* off = reinterpret_cast<const long long*>(sh + 16);
    const int32_t* spos = reinterpret_cast<const int32_t*>(sh + packed_pos_offset(n_nodes));
    const uint8_t* stc = sh + packed_tc_offset(n_nodes, cap);
    const unsigned int* relk = rel + (size_t)k * n_nodes;
    const long long stride = (long long)gridDim.x * blockDim.x * 4;
    for (long long j0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; j0 < n; j0 += stride) {
        int lo = 0, hi = n_nodes;  // the node v with off[v] <= j0 < off[v + 1]
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(off + mid) <= j0) lo = mid;
            else hi = mid;
        }
        int v = lo;
        long long end = __ldg(off + v + 1);
        long long dst = __ldg(merged_off + v) + __ldg(relk + v) - __ldg(off + v);  // + j = destination of record j of node v
        const long long j1 = min(n, j0 + 4);
        for (long long j = j0; j < j1; j++) {
            while (j >= end) {  // next non-empty node
                v++;
                end = __ldg(off + v + 1);
                dst = __ldg(merged_off + v) + __ldg(relk + v) - __ldg(off + v);
            }
            pos[dst + j] = spos[j];
            type_code[dst + j] = stc[j];
        }
    }
}

// ------------------------------------------------------------------ run-merge into NucMut fields (MSA form)
// reference src/panman.cpp:1445-1466 + NucMut ctor src/panman.hpp:109-151: a node's position-sorted records are cut where
// the position is not the previous + 1 or the type changes, and every such maximal run greedily into pieces of at most
// six; a piece becomes one NucMut {nucPosition = first position, mutInfo = (length << 4) + type, nucs = code_k <<
// 4 (5 - k)}, plus the wire form of mutInfo (src/panman.cpp:2876: ((nucs >> (24 - 4 length)) << 8) + mutInfo).
// col_break (optional, indexed by position - col_base): 1 = the column never continues the run of the column before it
// (PanGraph batches: the first gap slot of every position, src/panman.cpp:1242, 1261).
//
// Record-parallel over the WHOLE node-major list (round 1 walked each node with one warp: the few nodes with tens of
// thousands of records -- next to the root of a gappy alignment -- took 7.8 ms on 5.3 M records, 99 % of it in a dozen
// warps). A record starts a piece iff (index - start of its run) % 6 == 0, and the start of its run is the latest "break"
// at or before it: a max-scan. Breaks include the first record of every node, so runs never cross nodes and the pieces
// of all nodes, numbered by a prefix sum over the piece flags, come out node-major in order; a node's offset is the
// piece number of its first record. Blocks of RM_BLOCK records; two tiny one-block scans carry the latest break and
// the piece counts across blocks. flags[i]: bit 0 = first record of a node, bit 1 = starts a piece.
constexpr int RM_THREADS = 256, RM_ITEMS = 8, RM_BLOCK = RM_THREADS * RM_ITEMS;

__global__ void rm_mark_starts_kernel(const long long* off, int n_nodes, uint8_t* flags) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < n_nodes && off[v] < off[v + 1]) flags[off[v]] = 1;
}
__device__ __forceinline__ bool rm_is_break(long long i, const int32_t* pos, const uint8_t* tc, const uint8_t* flags,
                                            const uint8_t* col_break, long long col_base) {
    if (flags[i] & 1) return true;  // includes record 0
    const int32_t p = pos[i];
    return p != pos[i - 1] + 1 || (tc[i] >> 4) != (tc[i - 1] >> 4) || (col_break && col_break[p - col_base]);
}
// last[b] = index of the latest break inside block b, or -1
__global__ void __launch_bounds__(RM_THREADS) rm_block_last_kernel(const long long* off, int n_nodes, const int32_t* pos, const uint8_t* tc,
                                                                   const uint8_t* flags, const uint8_t* col_break, long long col_base,
                                                                   long long* last) {
    __shared__ long long s_w[RM_THREADS / 32];
    const long long n = off[n_nodes], i0 = ((long long)blockIdx.x * RM_THREADS + threadIdx.x) * RM_ITEMS;
    long long m = -1;
    for (int k = 0; k < RM_ITEMS; k++)
        if (i0 + k < n && rm_is_break(i0 + k, pos, tc, flags, col_break, col_base)) m = i0 + k;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) m = max(m, __shfl_down_sync(FULL, m, d));
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < RM_THREADS / 32; w++) m = max(m, s_w[w]);
        last[blockIdx.x] = m;
    }
}
// carry[b] = latest break in any block before b (exclusive max-scan), one block
__global__ void __launch_bounds__(1024) rm_scan_max_kernel(const long long* last, int n_blocks, long long* carry) {
    __shared__ long long s_w[32];
    __shared__ long long s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry = -1;
    __syncthreads();
    for (int b0 = 0; b0 < n_blocks; b0 += 1024) {
        const int b = b0 + tid;
        const long long v = b < n_blocks ? last[b] : -1;
        long long incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const long long t = __shfl_up_sync(FULL, incl, d);
            if (lane >= d) incl = max(incl, t);
        }
        if (lane == 31) s_w[warp] = incl;
        __syncthreads();
        long long before = s_carry;
        for (int w = 0; w < warp; w++) before = max(before, s_w[w]);
        long long excl = __shfl_up_sync(FULL, incl, 1);
        if (lane == 0) excl = -1;
        if (b < n_blocks) carry[b] = max(before, excl);
        __syncthreads();
        if (tid == 1023) s_carry = max(before, incl);
        __syncthreads();
    }
}
// piece flags (bit 1) and the number of pieces per block
__global__ void __launch_bounds__(RM_THREADS) rm_flags_kernel(const long long* off, int n_nodes, const int32_t* pos, const uint8_t* tc,
                                                              uint8_t* flags, const uint8_t* col_break, long long col_base,
                                                              const long long* carry, unsigned int* counts) {
    __shared__ long long s_w[RM_THREADS / 32];
    __shared__ unsigned s_c[RM_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long n = off[n_nodes], i0 = ((long long)blockIdx.x * RM_THREADS + tid) * RM_ITEMS;
    long long rs[RM_ITEMS], m = -1;
#pragma unroll
    for (int k = 0; k < RM_ITEMS; k++) {
        if (i0 + k < n && rm_is_break(i0 + k, pos, tc, flags, col_break, col_base)) m = i0 + k;
        rs[k] = m;  // latest break at or before the record, within this thread's records
    }
    long long incl = m;  // latest break in the threads up to and including this one
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const long long t = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl = max(incl, t);
    }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    long long before = carry[blockIdx.x];
    for (int w = 0; w < warp; w++) before = max(before, s_w[w]);
    long long excl = __shfl_up_sync(FULL, incl, 1);
    if (lane == 0) excl = -1;
    before = max(before, excl);
    unsigned cnt = 0;
#pragma unroll
    for (int k = 0; k < RM_ITEMS; k++) {
        const long long i = i0 + k;
        if (i >= n) break;
        const long long start = max(rs[k], before);  // >= 0: record 0 is a break
        const bool piece = (i - start) % 6 == 0;
        flags[i] = uint8_t((flags[i] & 1) | (piece ? 2 : 0));
        cnt += piece;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) cnt += __shfl_down_sync(FULL, cnt, d);
    if (lane == 0) s_c[warp] = cnt;
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < RM_THREADS / 32; w++) cnt += s_c[w];
        counts[blockIdx.x] = cnt;
    }
}
// the pieces: output index = pieces of earlier blocks + pieces before the record in this block
__global__ void __launch_bounds__(RM_THREADS) rm_fill_kernel(const long long* off, int n_nodes, const int32_t* pos, const uint8_t* tc,
                                                             const uint8_t* flags, const unsigned long long* base, long long* oidx,
                                                             int32_t* nuc_position, uint8_t* mut_info, uint32_t* nucs, uint32_t* wire) {
    __shared__ unsigned s_c[RM_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long n = off[n_nodes], i0 = ((long long)blockIdx.x * RM_THREADS + tid) * RM_ITEMS;
    unsigned mine = 0;
#pragma unroll
    for (int k = 0; k < RM_ITEMS; k++)
        if (i0 + k < n && (flags[i0 + k] & 2)) mine++;
    unsigned incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned t = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) s_c[warp] = incl;
    __syncthreads();
    unsigned long long o = base[blockIdx.x] + (incl - mine);
    for (int w = 0; w < warp; w++) o += s_c[w];
    for (int k = 0; k < RM_ITEMS; k++) {
        const long long i = i0 + k;
        if (i >= n) break;
        const uint8_t f = flags[i];
        if (!(f & 2)) continue;
        if (f & 1) oidx[i] = (long long)o;  // a node's first record: its piece number is the node's offset
        const uint32_t t = uint32_t(tc[i]) >> 4;
        uint32_t packed = (uint32_t(tc[i]) & 15u) << 20;
        int len = 1;
        for (; len < 6 && i + len < n && !(flags[i + len] & 2); len++) packed += (uint32_t(tc[i + len]) & 15u) << (4 * (5 - len));
        nuc_position[o] = pos[i];
        mut_info[o] = uint8_t((len << 4) + int(t));
        nucs[o] = packed;
        wire[o] = ((packed >> (24 - 4 * len)) << 8) + uint32_t((len << 4) + int(t));
        o++;
    }
}
// out_off[v] = piece number of the node's first record; a node without records takes the next node's (off[v] is then the
// first record of the next non-empty node, or the end). out_off[n_nodes] has been written by the scan of the block counts.
__global__ void rm_node_offsets_kernel(const long long* off, int n_nodes, const long long* oidx, long long* out_off) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_nodes) return;
    const long long a = off[v];
    out_off[v] = a < off[n_nodes] ? oidx[a] : out_off[n_nodes];
}

// ------------------------------------------------------------------ ingest
// nibble-packed rows -> code planes. One thread per (row, 32-column group).
__global__ void pack_leaves_kernel(const uint8_t* codes, long long row_stride, int row_begin, int n_rows_slab, int n_rows_total,
                                   long long n_cols, int T, const int* row_slot, uint4* planes) {
    const long long groups = (long long)T * 32;  // 32-column groups per row, padded to whole tiles
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= groups * n_rows_slab) return;
    const long long row = idx / groups, g = idx % groups;
    uint32_t pl[4] = {0, 0, 0, 0};
    const uint8_t* src = codes + (size_t)row * row_stride;
    long long c0 = g * 32;
    // whole groups are fetched with the widest load the address allows (the source may be pinned HOST memory read
    // across PCIe, where byte loads would waste the link); the ragged last group of a row goes byte by byte
    uint32_t xw[4] = {0, 0, 0, 0};
    const bool whole = c0 + 32 <= n_cols;
    if (whole) {
        const uint8_t* a = src + (c0 >> 1);
        const unsigned long long addr = (unsigned long long)a;
        if ((addr & 15) == 0) {
            const uint4 v = *reinterpret_cast<const uint4*>(a);
            xw[0] = v.x; xw[1] = v.y; xw[2] = v.z; xw[3] = v.w;
        } else if ((addr & 7) == 0) {
            const uint2 v0 = *reinterpret_cast<const uint2*>(a), v1 = *reinterpret_cast<const uint2*>(a + 8);
            xw[0] = v0.x; xw[1] = v0.y; xw[2] = v1.x; xw[3] = v1.y;
        } else if ((addr & 3) == 0) {
#pragma unroll
            for (int w = 0; w < 4; w++) xw[w] = *reinterpret_cast<const uint32_t*>(a + 4 * w);
        } else {
#pragma unroll
            for (int w = 0; w < 4; w++)
                xw[w] = uint32_t(a[4 * w]) | (uint32_t(a[4 * w + 1]) << 8) | (uint32_t(a[4 * w + 2]) << 16) | (uint32_t(a[4 * w + 3]) << 24);
        }
    }
    for (int w = 0; w < 4; w++) {  // 8 columns = 4 bytes per step
        uint32_t x = xw[w];
        long long cb = c0 + w * 8;
        if (!whole && cb < n_cols) {
            long long byte = cb >> 1;
            long long ncol = min(n_cols, cb + 8) - cb;
            long long nbytes = (ncol + 1) >> 1;
            for (int k = 0; k < nbytes; k++) x |= uint32_t(src[byte + k]) << (8 * k);
            if (ncol < 8) x &= (1u << (4 * ncol)) - 1u;
        }
#pragma unroll
        for (int b = 0; b < 4; b++) {
            uint32_t y = (x >> b) & 0x11111111u;       // bit b of each of the 8 nibbles, at stride 4
            y = (y | (y >> 3)) & 0x03030303u;
            y = (y | (y >> 6)) & 0x000F000Fu;
            y = (y | (y >> 12)) & 0xFFu;
            pl[b] |= y << (8 * w);
        }
    }
    // tile-major, rows in the order the forward program consumes them
    const int slot = row_slot[row_begin + row];
    const long long tile = g >> 5, lane = g & 31;
    planes[((size_t)tile * n_rows_total + slot) * 32 + lane] = make_uint4(pl[0], pl[1], pl[2], pl[3]);
}

// clade-run encoded leaves (pmb_runs.h) -> the same code planes. One warp per (tile, segment of leaves in depth-first
// order): lane l keeps the running (code ^ parent code) of its 32 columns in four plane words, applies the toggle events
// of each leaf as it comes to it (the events of an item are sorted by leaf) and stores parent planes ^ running planes as
// that leaf's row: every row is one coalesced 512-byte store, the kernel is bound by writing the plane matrix.
__global__ void __launch_bounds__(256, 8)
expand_runs_kernel(const uint32_t* events, const long long* item_off, long long ev_base, long long item_begin, long long item_end,
                   int n_seg, int seg_rows, int n_rows, const int* dfs_slot, const uint4* colparams, uint4* planes) {
    const int lane = threadIdx.x & 31;
    const long long item = item_begin + (((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (item >= item_end) return;
    const long long tile = item / n_seg;
    const int seg = int(item % n_seg);
    const int r0 = seg * seg_rows, nr = min(seg_rows, n_rows - r0);
    uint4 cur = colparams[(size_t)tile * 128 + lane];  // parent code planes of the tile (pack_colparams_kernel) ^ running xor
    long long k = item_off[item] - ev_base;
    const long long k_end = item_off[item + 1] - ev_base;
    uint32_t ev = (k + lane < k_end) ? events[k + lane] : 0xFFFFFFFFu;  // the all-ones row never comes up: the list's end
    int j = 0;
    uint32_t next_row = __shfl_sync(FULL, ev, 0) >> 14;  // row of the first event not yet applied (warp-uniform)
    uint4* out = planes + (size_t)tile * n_rows * 32 + lane;
    for (int rb = 0; rb < nr; rb += 32) {
        const int my_slot = (rb + lane < nr) ? dfs_slot[r0 + rb + lane] : 0;
        const int lim = min(32, nr - rb);
        for (int i = 0; i < lim; i++) {
            while (next_row == uint32_t(rb + i)) {  // a few per column in all, so on most rows not taken
                const uint32_t e = __shfl_sync(FULL, ev, j);
                if (lane == int((e >> 9) & 31u)) {  // column in tile = bits 4..13; its lane = the upper five of them
                    const uint32_t bit = 1u << ((e >> 4) & 31u);
                    cur.x ^= (e & 1u) ? bit : 0u;
                    cur.y ^= (e & 2u) ? bit : 0u;
                    cur.z ^= (e & 4u) ? bit : 0u;
                    cur.w ^= (e & 8u) ? bit : 0u;
                }
                if (++j == 32) {
                    k += 32;
                    ev = (k + lane < k_end) ? events[k + lane] : 0xFFFFFFFFu;
                    j = 0;
                }
                next_row = __shfl_sync(FULL, ev, j) >> 14;
            }
            const int slot = __shfl_sync(FULL, my_slot, i);
            out[(size_t)slot * 32] = cur;
        }
    }
}

// ---- a PanMAT's mutation lists -> the clade-run events expand_runs_kernel turns into leaf planes (pmb_upload_replay) ----
// Every piece position becomes a record. Records are numbered by the pre-order index of their node in the tree the lists were
// built on, then in stored order within the node, and sorted by column << rec_bits | record number: per column, the nodes of
// the records are then nested intervals of that tree's depth-first leaf order, and a leaf's code is the code of the last
// record whose interval holds it (the deepest node wins, and within a node the later piece).

__device__ __forceinline__ long long lower_bound_u64(const unsigned long long* a, long long n, unsigned long long key) {
    long long lo = 0, hi = n;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

__global__ void replay_piece_len_kernel(const uint8_t* mut_info, long long n_pieces, long long* len) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_pieces) len[i] = mut_info[i] >> 4;
}

// one thread per piece. rec_off: exclusive scan of the piece lengths (node-major); node_base[v]: number of node v's first record
// (pre-order-major). A deletion writes '-' whatever its nucs hold.
__global__ void replay_records_kernel(const long long* piece_off, int n_nodes, const long long* node_base, const int* pre_of,
                                      const int32_t* nuc_position, const uint8_t* mut_info, const uint32_t* nucs, long long n_pieces,
                                      const long long* rec_off, int rec_bits, unsigned long long* keys, uint8_t* rec_code, int* rec_pre) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pieces) return;
    int lo = 0, hi = n_nodes - 1;  // the node owning piece i: the last v with piece_off[v] <= i
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (piece_off[mid] <= i) lo = mid;
        else hi = mid - 1;
    }
    const int len = mut_info[i] >> 4, type = mut_info[i] & 15, pre = pre_of[lo];
    const unsigned long long col = (unsigned long long)nuc_position[i];
    const uint32_t nu = nucs[i];
    const long long r = node_base[lo] + rec_off[i] - rec_off[piece_off[lo]];
    for (int j = 0; j < len; j++) {
        keys[r + j] = ((col + j) << rec_bits) | (unsigned long long)(r + j);
        rec_code[r + j] = type == 1 ? uint8_t(0) : uint8_t((nu >> (4 * (5 - j))) & 15u);
        rec_pre[r + j] = pre;
    }
}

// One thread per column sweeps its sorted records with a stack of open intervals (kept in stack_mem at the column's own
// record range, so it can never overflow) and emits an event wherever the code seen by expand_runs_kernel changes along the
// leaf order: at a change of the leaf code, and at the first leaf of every segment whose code is not the parent code (each
// (tile, segment) item restarts from the parent planes). Events of one (leaf, column) compose by XOR. EMIT = false only
// counts them; EMIT = true writes item << 32 | event (pmb_runs.h layout) and the code of the leaf at tip_pos.
template <bool EMIT>
__global__ void replay_sweep_kernel(const unsigned long long* keys, const uint8_t* rec_code, const int* rec_pre, long long n_rec, int rec_bits, const int2* span,
                                    const uint8_t* parent_code, long long n_cols, int n_rows, int n_seg, int seg_rows, int tip_pos,
                                    unsigned long long* stack_mem, long long* counts, const long long* ev_off, unsigned long long* ev_out,
                                    int8_t* tip_code) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cols) return;
    const long long a = lower_bound_u64(keys, n_rec, (unsigned long long)c << rec_bits);
    const long long b = lower_bound_u64(keys, n_rec, (unsigned long long)(c + 1) << rec_bits);
    const unsigned long long rec_mask = (1ull << rec_bits) - 1;
    const int pc = parent_code[c] & 15;
    const unsigned long long item0 = (unsigned long long)(c / TILE_COLS) * n_seg;
    const uint32_t col_field = uint32_t(c % TILE_COLS) << 4;
    unsigned long long* out = EMIT ? ev_out + ev_off[c] : nullptr;
    long long n_ev = 0, next_seg = seg_rows;
    int val = pc, tipv = pc;  // val: the code expand_runs_kernel holds at the current leaf
    auto emit = [&](long long p, int x) {
        if (EMIT) {
            const long long seg = p / seg_rows;
            out[n_ev] = ((item0 + seg) << 32) | (uint32_t(p - seg * seg_rows) << 14) | col_field | uint32_t(x);
        }
        n_ev++;
    };
    auto change = [&](long long p, int nv) {  // from leaf p on, the code is nv (p never decreases)
        if (p >= n_rows) return;
        for (; next_seg <= p; next_seg += seg_rows) {
            if (next_seg < p) {
                if (val != pc) emit(next_seg, val ^ pc);
            } else {
                val = pc;
            }
        }
        if (nv != val) {
            emit(p, nv ^ val);
            val = nv;
        }
        if (p <= tip_pos) tipv = nv;
    };
    unsigned long long* st = stack_mem + a;  // (interval end << 4) | code
    long long sp = 0;
    for (long long r = a; r < b; r++) {
        const long long k = (long long)(keys[r] & rec_mask);
        const int2 s = span[rec_pre[k]];
        const int code = rec_code[k];
        while (sp > 0 && (long long)(st[sp - 1] >> 4) <= s.x) {
            const long long end = (long long)(st[--sp] >> 4);
            change(end, sp ? int(st[sp - 1] & 15) : pc);
        }
        change(s.x, code);
        st[sp++] = ((unsigned long long)s.y << 4) | (unsigned long long)code;
    }
    while (sp > 0) {
        const long long end = (long long)(st[--sp] >> 4);
        change(end, sp ? int(st[sp - 1] & 15) : pc);
    }
    for (; next_seg < n_rows; next_seg += seg_rows)
        if (val != pc) emit(next_seg, val ^ pc);
    if (!EMIT) counts[c] = n_ev;
    else if (tip_code) tip_code[c] = int8_t(tipv);
}

// sorted item << 32 | event keys -> the events and item offsets expand_runs_kernel reads
__global__ void replay_items_kernel(const unsigned long long* ev, long long n_ev, long long n_items, uint32_t* ev32, long long* item_off) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_ev) ev32[i] = uint32_t(ev[i]);
    if (i <= n_items) item_off[i] = lower_bound_u64(ev, n_ev, (unsigned long long)i << 32);
}

// per-column parameters -> planes; one warp per 32-column group (ballot builds the planes)
__global__ void pack_colparams_kernel(const uint8_t* parent_code, const int8_t* root_override, const int8_t* fwd_root_ref,
                                      long long n_cols, int T, uint4* colparams) {
    long long g = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int l = threadIdx.x & 31;
    if (g >= (long long)T * 32) return;
    long long c = g * 32 + l;
    bool valid = c < n_cols;
    int pc = valid ? parent_code[c] & 15 : 0;
    int ov = (valid && root_override) ? root_override[c] : -1;
    int fr = (valid && fwd_root_ref) ? fwd_root_ref[c] : -1;
    uint32_t pcp[4], ovp[4], frp[4];
#pragma unroll
    for (int b = 0; b < 4; b++) {
        pcp[b] = __ballot_sync(FULL, (pc >> b) & 1);
        ovp[b] = __ballot_sync(FULL, ov >= 0 && ((ov >> b) & 1));
        frp[b] = __ballot_sync(FULL, fr >= 0 && ((fr >> b) & 1));
    }
    uint32_t ovv = __ballot_sync(FULL, ov >= 0), frv = __ballot_sync(FULL, fr >= 0), cv = __ballot_sync(FULL, valid);
    if (l == 0) {
        int tile = int(g >> 5), lane = int(g & 31);
        uint4* cp = colparams + (size_t)tile * 128;
        cp[lane] = make_uint4(pcp[0], pcp[1], pcp[2], pcp[3]);
        cp[32 + lane] = make_uint4(ovp[0], ovp[1], ovp[2], ovp[3]);
        cp[64 + lane] = make_uint4(frp[0], frp[1], frp[2], frp[3]);
        cp[96 + lane] = make_uint4(ovv, frv, cv, 0);
    }
}

// assigned-state planes -> one byte per node x column (0xFF = not assigned)
__global__ void unpack_states_kernel(const uint4* states, int n_nodes, long long n_cols, int T, uint8_t* out) {
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)n_nodes * n_cols) return;
    const long long node = idx / n_cols, c = idx % n_cols;
    int tile = int(c / TILE_COLS), lane = int((c % TILE_COLS) >> 5), bit = int(c & 31);
    const uint4* s = states + ((size_t)node * T + tile) * 64;
    uint4 f = s[lane];
    uint32_t vis = s[32 + lane].x;
    uint32_t code = ((f.x >> bit) & 1u) | (((f.y >> bit) & 1u) << 1) | (((f.z >> bit) & 1u) << 2) | (((f.w >> bit) & 1u) << 3);
    out[idx] = ((vis >> bit) & 1u) ? uint8_t(code) : uint8_t(0xFF);
}

}  // namespace pmb
