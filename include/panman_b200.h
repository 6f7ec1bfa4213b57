/* libpanman_b200 -- C ABI of the B200-native Fitch/Sankoff construction pass of PanMAN.
 *
 * This is the drop-in boundary for the per-column loops of the reference's Tree constructor
 * (reference src/panman.cpp:873-963, 1004-1233, 1381-1435, 1568-1613; later src/reroot.cpp:54-224).
 * The reference has no plugin/FFI layer: its hot path is 19 member functions of panmanUtils::Tree
 * (declared src/panman.hpp:846-902, defined src/fitchSankoff.cpp:5-818) called once per alignment
 * column with std::unordered_map<std::string,...> state maps. This library replaces a whole BATCH of
 * those per-column call triples by one call:
 *
 *   nucFitchForwardPass / nucFitchBackwardPass / nucFitchAssignMutations      (fitchSankoff.cpp:30-171)
 *   nucSankoffForwardPass / nucSankoffBackwardPass / nucSankoffAssignMutations (fitchSankoff.cpp:359-531, 676-703)
 *   blockFitch*New / blockSankoff*                                              (fitchSankoff.cpp:224-308, 707-818)
 *
 * Everything before (parsing, consensus, block order) and after (run-merge into NucMut, the capnp
 * writer) stays host code; see INTEGRATION.md for the binding a maintainer adds to panman.cpp.
 *
 * Conventions
 *   - plain pointers and sizes only; no allocation crosses the boundary. Inputs are borrowed for the
 *     duration of the call; outputs are owned by the context and stay valid until the next
 *     pmb_run_* / pmb_upload_* / pmb_destroy on that context.
 *   - every call returns PMB_OK (0) or a negative code; text via pmb_last_error. The library never
 *     exits or throws (the reference exit()s / asserts, e.g. fitchSankoff.cpp:505).
 *   - a context is bound to ONE CUDA device and is not thread-safe; use one per host thread / rank.
 *   - codes are the 4-bit IUPAC codes of reference src/panman.hpp:27-44 ('-' = 0, A1 C2 M3 G4 R5 S6 V7
 *     T8 W9 Y10 H11 K12 D13 B14 N15); a Fitch leaf set is 1 << code (src/panman.cpp:1409-1417), a
 *     Sankoff leaf vector is 0 at its code and SANKOFF_INF elsewhere (src/panman.cpp:1574-1582).
 *   - record types: NS=0 (substitution), ND=1 (deletion), NI=2 (insertion)  (src/panman.hpp:46-61).
 *   - there is NO CPU fallback: without a CUDA device every compute entry returns PMB_ERR_CUDA.
 */
#ifndef PANMAN_B200_H
#define PANMAN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pmb_ctx pmb_ctx;

enum {
    PMB_OK = 0,
    PMB_ERR_INVALID = -1,      /* bad argument / malformed tree */
    PMB_ERR_CUDA = -2,         /* CUDA runtime failure or no device */
    PMB_ERR_NO_TREE = -3,      /* pmb_set_tree not called */
    PMB_ERR_SANKOFF_ROOT = -4, /* a column's root has no finite cost and no override: the reference
                                  would fail assert(minPtr != -1), src/fitchSankoff.cpp:505 */
    PMB_ERR_NO_INPUT = -5,     /* pmb_run_resident without pmb_upload_nuc */
    PMB_ERR_OOM = -6,          /* device memory */
    PMB_ERR_INTERNAL = -7,     /* scheduler watchdog fired; never expected */
    PMB_ERR_STAGING = -8,      /* an asynchronous pass emitted more records than the staging pool held: the pool has been
                                  grown, run the pass again (a synchronous pass regrows and retries by itself) */
    PMB_ERR_CAPACITY = -9      /* a packed column-range shard holds more records than the capacity it was packed /
                                  merged with: reserve more and repeat the step */
};

enum { PMB_ALGO_FITCH = 0, PMB_ALGO_SANKOFF = 1 };

enum {
    PMB_FLAG_WANT_STATES = 1, /* also return the assigned state of every node x column */
    PMB_FLAG_BLOCK_MODE = 2   /* 3-state block columns (0 absent, 1 forward, 2 reverse strand):
                                 Fitch root gets no take-lowest-bit special case (fitchSankoff.cpp:247-270),
                                 Sankoff treats an omitted leaf as "absent" not "unknown" (:711-714).
                                 Records come back nuc-style: NI = block insertion (code 2 => inverted),
                                 ND = block deletion, NS = inversion (:272-308, :788-818). */
};

/* Result of one batch: per-node mutation lists, node-major, each list in ascending column order
 * (what the reference obtains by std::sort of its per-node tuples, src/panman.cpp:1447). */
typedef struct pmb_result {
    int64_t n_mut;               /* total records */
    int32_t n_nodes;
    int32_t reserved;
    const int64_t* node_offsets; /* n_nodes + 1; node v owns [node_offsets[v], node_offsets[v+1]) */
    const int32_t* pos;          /* column index (col_base + local column) */
    const uint8_t* type_code;    /* (type << 4) | code */
    const uint8_t* states;       /* PMB_FLAG_WANT_STATES: n_nodes x n_cols codes, 0xFF = not assigned; else NULL */
    int64_t n_cols;
} pmb_result;

/* Device-time breakdown of the last pmb_run_resident, CUDA events on the library's stream. After an asynchronous pass
 * (pmb_run_resident_async + pmb_wait) only total_ms is filled: the pass is timed as a whole. */
typedef struct pmb_timings {
    float forward_ms;   /* post-order pass (all levels) */
    float backward_ms;  /* pre-order pass + mutation detection + staging append (all levels) */
    float compact_ms;   /* directory scan + ordered gather into the final lists */
    float total_ms;     /* first kernel start to last kernel end */
    int32_t n_launches; /* kernels launched by the last run */
    int32_t n_levels;   /* dependency levels of the tree schedule */
} pmb_timings;

/* ---- lifecycle ---- */
int pmb_create(pmb_ctx** ctx, int device);
void pmb_destroy(pmb_ctx* ctx);
const char* pmb_last_error(const pmb_ctx* ctx);
/* Tuning knobs (all optional): "chunk_nodes" (largest bottom subtree evaluated by one warp; 0 = chosen from the
 * column count), "inline_nodes" (light subtrees up to this size stay in their parent's chunk), "schedule"
 * (1 = persistent kernels with dependency flags [default], 0 = one launch per dependency level),
 * "staging_records" (initial capacity of the mutation staging pool; 0 = chosen from the problem size),
 * "bwd_tail" (tenths of a machine-full of warps whose items form the sorted tail of the backward tickets; default 20),
 * "reserve_sms" (SMs the persistent kernels leave free, e.g. for an NCCL kernel running beside them; default 0),
 * "col_groups" (column-tile groups run on separate streams; default 1), "overlap" (1 [default]: set matrices up to 48 GB
 * and a quarter of the device's memory are double-buffered -- with the staging pool and its directory -- so that the forward
 * kernel of an asynchronous pass runs beside the backward kernel of the pass before it; 0: one set matrix, passes strictly
 * one after the other), "grid_pct" (share of the resident block slots a
 * persistent kernel takes; 0 = automatic: 80 for overlapping asynchronous passes, 100 otherwise), "lanes" (1 [default]:
 * asynchronous passes of small problems -- set matrix up to 4 GB, no chain segments, no state output -- alternate between two
 * independent pipelines inside the context, each with its own set matrices, flags, staging and lists, both reading the same
 * resident input; 0: one pipeline), "trace" (debug timeline). */
int pmb_set_option(pmb_ctx* ctx, const char* key, int64_t value);

/* Page-locked host memory for the caller's input buffers. pmb_run_nuc / pmb_upload_nuc accept any host pointer, but
 * only page-locked memory moves at PCIe speed (measured on B200: 50-54 GB/s against 11 GB/s from pageable memory).
 * Returns NULL when there is no usable device or the allocation fails. */
void* pmb_host_alloc(size_t bytes);
void pmb_host_free(void* p);

/* ---- tree: replaces the Node* tree walked by every reference call ----
 * CSR children in Newick order (reference src/panman.cpp:223-229 appends children in that order).
 * leaf_row[v] = row of leaf v in the code matrix, -1 for internal nodes. Unary nodes and polytomies are legal.
 * The library flattens this into a level-ordered chunk schedule replicated on the device. */
int pmb_set_tree(pmb_ctx* ctx, int32_t n_nodes, int32_t root, const int32_t* child_offsets,
                 const int32_t* child_index, const int32_t* leaf_row);

/* ---- one batch of columns, host or device buffers in, host lists out (the end-to-end entry) ----
 * leaf_codes_4bit : n_rows x row_stride_bytes, row-major; column c of a row is the low nibble of byte c/2 when
 *                   c is even, the high nibble when odd. May be host or device memory (UVA decides).
 * leaf_present    : n_rows bytes or NULL; 0 => the leaf is omitted from the state map for every column of
 *                   this call (reference: sequences lacking a block, src/panman.cpp:1027-1030).
 * parent_code     : n_cols; code of the consensus character = parentState handed to the root
 *                   (src/panman.cpp:1424-1425, 1600-1606).
 * root_override   : n_cols or NULL; -1 none, else the code the root is forced to (defaultState,
 *                   src/panman.cpp:1057-1079, 1583-1604; src/reroot.cpp:189-190).
 * fwd_root_ref    : n_cols or NULL; -1 none, else the forward-pass root reference code (refState,
 *                   src/panman.cpp:1419-1420). Fitch only.
 * col_base        : added to every emitted position (column-range sharding across GPUs). Positions are int32 (the
 *                   reference's NucMut.nucPosition): 0 <= col_base and col_base + n_cols <= 2^31, else PMB_ERR_INVALID
 *                   (the same for every upload entry; the group uploads refuse n_cols_total > 2^31). */
int pmb_run_nuc(pmb_ctx* ctx, int algo, int64_t n_cols, int32_t n_rows, const uint8_t* leaf_codes_4bit,
                int64_t row_stride_bytes, const uint8_t* leaf_present, const uint8_t* parent_code,
                const int8_t* root_override, const int8_t* fwd_root_ref, int64_t col_base, int flags,
                pmb_result* out);

/* ---- the block-level pass of a PanGraph build: one 3-state column per block ----
 * Replaces blockFitchForwardPassNew / BackwardPassNew / AssignMutationsNew and blockSankoff* as driven by
 * src/panman.cpp:873-963 (and src/reroot.cpp:54-122). leaf_block_state: n_rows x n_blocks bytes in HOST memory, row-major,
 * 0 = the sequence lacks the block, 1 = forward strand, 2 = reverse strand (the reference's 1 / 2 / 4 and its 3-vector
 * {absent, forward, reverse}); root_override: n_blocks or NULL, -1 none else the state the root is forced to
 * (defaultState, :886-897). The parent state handed to the root is "absent", as in the reference. Records use the
 * nucleotide form (see oracle.block_mut_from_nuc for the reference pair): type 2 = block insertion (code = strand state,
 * 2 = inverted), type 1 = block deletion, type 0 = inversion of a present block. Same as pmb_run_nuc with
 * PMB_FLAG_BLOCK_MODE on nibble-packed states. */
int pmb_run_block(pmb_ctx* ctx, int algo, int64_t n_blocks, int32_t n_rows, const uint8_t* leaf_block_state,
                  const int8_t* root_override, pmb_result* out);

/* ---- the same, split so that the pass can be timed with inputs resident in HBM ----
 * pmb_upload_nuc copies + bit-plane-packs the inputs into device memory (the "packed leaf matrix resident in
 * HBM"); pmb_run_resident runs forward + backward + compaction on it, leaving the lists in device memory;
 * pmb_download copies them to host memory owned by the context. pmb_run_nuc = the three in a row. */
int pmb_upload_nuc(pmb_ctx* ctx, int64_t n_cols, int32_t n_rows, const uint8_t* leaf_codes_4bit,
                   int64_t row_stride_bytes, const uint8_t* leaf_present, const uint8_t* parent_code,
                   const int8_t* root_override, const int8_t* fwd_root_ref, int64_t col_base);
/* The same without the final synchronisation: returns once the copies are enqueued; the input buffers must stay valid
 * until the next pmb_wait / pmb_run_resident / pmb_download on the context (several devices can then upload at once). */
int pmb_upload_nuc_async(pmb_ctx* ctx, int64_t n_cols, int32_t n_rows, const uint8_t* leaf_codes_4bit, int64_t row_stride_bytes,
                         const uint8_t* leaf_present, const uint8_t* parent_code, const int8_t* root_override,
                         const int8_t* fwd_root_ref, int64_t col_base);
/* Leaf codes rebuilt from a PanMAT's mutation lists instead of a code matrix: the upload entry of Tree::reroot (reference
 * src/reroot.cpp:19-35, getSequenceFromReference). The context's tree (pmb_set_tree) is the tree the pass will run on;
 * old_* describe the tree the lists were built on, with the same set of leaf rows. Pieces are NucMut fields in HOST memory,
 * node-major over old node ids: piece_offsets[old_n_nodes + 1], nuc_position, mut_info ((length << 4) + type, type 0..2,
 * length 1..6), nucs. Positions lie in [0, n_cols). A leaf's code in column c is parent_code[c] overwritten, walking old
 * root -> leaf, by every piece that covers c, in stored order (NS / NI write their nucs nibble, ND writes '-'): the deepest
 * node wins, and within a node the later piece. A leaf without pieces of its own gets its nearest ancestor's codes, and every
 * leaf takes part in the pass (no leaf_present). root_leaf_row >= 0: root_override = that leaf's replayed code in every
 * column; -1: none. No fwd_root_ref, col_base 0. The replay runs on the device (only the pieces cross the link); afterwards
 * as pmb_upload_nuc. PMB_ERR_INVALID, before anything is enqueued, for a malformed old tree, leaf rows that differ from the
 * context's tree, piece_offsets not starting at 0 or not monotone, a type above 2, a length of 0 or above 6, a piece beyond
 * n_cols, or a root_leaf_row that is not a row. Synchronous: the inputs may be released on return. */
int pmb_upload_replay(pmb_ctx* ctx, int32_t old_n_nodes, int32_t old_root, const int32_t* old_child_offsets,
                      const int32_t* old_child_index, const int32_t* old_leaf_row, const int64_t* piece_offsets,
                      const int32_t* nuc_position, const uint8_t* mut_info, const uint32_t* nucs, int64_t n_cols,
                      const uint8_t* parent_code, int32_t root_leaf_row);
int pmb_run_resident(pmb_ctx* ctx, int algo, int flags);
/* Asynchronous form: enqueues the pass on the context's stream and returns; several passes (and the caller's own
 * stream work ordered with pmb_stream) can be in flight. pmb_wait blocks until the stream drains and reports the
 * status of everything since the last wait (the first error wins). The mutation staging pool is not regrown on
 * the fly in this mode: an overflow is reported by pmb_wait (and the pool grown for the next attempt). */
int pmb_run_resident_async(pmb_ctx* ctx, int algo, int flags);
int pmb_wait(pmb_ctx* ctx);
/* Orders pmb_stream(ctx) behind every pass enqueued so far (consecutive asynchronous passes run on several streams, small
 * problems on two lanes): an event recorded on pmb_stream after pmb_join marks the end of all of them. Does not block. */
int pmb_join(pmb_ctx* ctx);
int pmb_download(pmb_ctx* ctx, pmb_result* out);

/* ---- post-processing: greedy <= 6 run-merge of the per-node lists into NucMut fields, on the device ----
 * Replaces the sort + merge loop of the MSA branches (src/panman.cpp:1445-1466, 1625-1646; NucMut ctor
 * src/panman.hpp:109-151): the lists are already position-sorted per node. source = 0: the lists of the last run;
 * source = 1: the lists of the last pmb_merge_packed (column-range shards must be merged FIRST: a run may straddle a
 * shard boundary). to_host != 0 copies the result to host memory owned by the context, else pointers are device memory
 * and n is -1 (it is node_offsets[n_nodes], on the device). Entry k of node v = k-th NucMut the reference would append
 * to Node::nucMutation: nucPosition, mutInfo = (length << 4) + type, nucs = code_j << (4 * (5 - j)); the other fields
 * are constants for an MSA build (nucGapPosition -1, primaryBlockId 0, secondaryBlockId -1). */
typedef struct pmb_nucmut_result {
    int64_t n;
    int32_t n_nodes;
    int32_t reserved;
    const int64_t* node_offsets; /* n_nodes + 1 */
    const int32_t* nuc_position;
    const uint8_t* mut_info;
    const uint32_t* nucs;
    const uint32_t* mut_info_wire; /* the same piece as the reference's capnp writer stores it (src/panman.cpp:2876):
                                      ((nucs >> (24 - 4 * length)) << 8) + mutInfo; pieces of one node are already in the
                                      writer's order (nucMutation order inside the single block group of an MSA build) */
} pmb_nucmut_result;
int pmb_merge_runs(pmb_ctx* ctx, int source, int to_host, pmb_nucmut_result* out);
/* Optional, for the batch uploaded last (cleared by the next upload): col_break[c] != 0 means column c never continues a
 * run of column c - 1 even at a consecutive position. A PanGraph block batch lays its main positions first and the gap
 * slots (pos, k) after them, so the first gap slot of every position is a break (src/panman.cpp:1242, 1261: non-gap
 * records merge on pos + 1, gap records on equal pos and gapPos + 1). n_cols bytes, host or device; NULL clears. */
int pmb_set_column_breaks(pmb_ctx* ctx, const uint8_t* col_break);

/* Device-side view of the last result (for an NCCL gather straight from HBM). Pointers are device memory. */
int pmb_result_device(pmb_ctx* ctx, pmb_result* out);

/* ---- column-range shards (one context / GPU / rank per contiguous column range) ----
 * A rank packs its last result into ONE device buffer (header, node offsets, positions, type|code bytes) so that a
 * single collective (e.g. an NCCL gather issued by the host program) moves it; the receiving rank merges the packed
 * shards, given in ascending column-range order, into node-major lists: per node the shard lists are concatenated in
 * shard order (each is already in ascending position), nothing is sorted. The reference's <=6 run-merge
 * (src/panman.cpp:1445-1466) must run on the merged lists, never per shard. `capacity` = records the buffer can hold
 * (>= n_mut of every shard); `stream` = CUDA stream (cudaStream_t) to enqueue on, NULL = pmb_result_stream. */
void* pmb_stream(pmb_ctx* ctx); /* the cudaStream_t the forward and backward kernels are enqueued on */
/* The cudaStream_t on which a pass ENDS: the ordered compaction runs on a stream of its own (behind the backward kernel), so
 * that the next pass' forward kernel starts at once and the compaction fills the SMs that kernel leaves idle while it
 * drains; only the next backward kernel waits for it. Work that consumes the lists (pmb_pack_result, pmb_merge_runs with
 * source 0, pmb_download) is enqueued here; order caller work after a pass on THIS stream. */
void* pmb_result_stream(pmb_ctx* ctx);
int64_t pmb_packed_bytes(int32_t n_nodes, int64_t capacity);
/* Stream rules. `stream` = NULL means pmb_result_stream. pmb_pack_result on another stream first makes that stream wait for
 * the pass enqueued last (an event), so it may be called right behind pmb_run_resident_async. pmb_merge_packed remembers its stream:
 * pmb_merge_runs(source = 1) and pmb_merge_status run on / wait for that stream. The destination of pmb_pack_result may be
 * peer memory (another GPU's buffer mapped into this process): the shard is then written over NVLink by the packing
 * kernel itself. A shard that holds more than `capacity` records is packed truncated and flagged in its header; merging
 * skips such a shard and pmb_merge_status / pmb_merge_runs(source = 1) return PMB_ERR_CAPACITY. */
int pmb_pack_result(pmb_ctx* ctx, void* d_packed, int64_t capacity, void* stream);
int pmb_merge_packed(pmb_ctx* ctx, int32_t n_shards, const void* d_packed_shards, int64_t capacity, void* stream,
                     pmb_result* out_device);
/* Blocks until the last pmb_merge_packed has finished; PMB_OK, or PMB_ERR_CAPACITY / PMB_ERR_INVALID when a shard was
 * skipped (over capacity / packed for another tree). */
int pmb_merge_status(pmb_ctx* ctx);

/* ---- column-sharded passes over several GPUs (BASELINE.json north_star: "alignment column ranges are partitioned across
 * the 8 GPUs of one box with the tree replicated on each; per-GPU mutation lists are merged by a column-range gather") ----
 * The reference runs its column loop on the threads of one process (tbb::parallel_for over columns, src/panman.cpp:1568;
 * per-node sort + merge AFTER all columns, :1445-1466 / :1625-1646). A pmb_group is the same loop over the GPUs of one
 * box: rank r of `world` owns the r-th contiguous, 1024-column-aligned range of the alignment (pmb_group_column_range),
 * every rank runs the whole pass on its range, packs its per-node lists straight into rank 0's mailbox over NVLink (the
 * packing kernel's own stores into peer memory -- no copy through the host, no extra kernel), and rank 0 concatenates
 * the shards per node in rank order (positions are already ascending: nothing is sorted). The <= 6 run-merge follows the
 * gather, never a shard (a run may straddle a range boundary).
 *
 * Two ways to form a group, one implementation:
 *   - ONE process driving several GPUs (what panmanUtils is: a single process): n_local == world, rank_base = 0.
 *     Everything is set up by pmb_group_create.
 *   - one process per GPU (torchrun / mpirun): n_local = 1, rank_base = the process' rank. Each process then calls
 *     pmb_group_export, the caller all-gathers the PMB_GROUP_HANDLE_BYTES-byte handles of all ranks in rank order with
 *     whatever transport it has (torch.distributed / MPI: the same role as ncclGetUniqueId + broadcast), and every
 *     process calls pmb_group_connect with the `world` handles. Rank 0's mailbox is mapped into the other processes
 *     with CUDA IPC.
 * "shard arrived" / "mailbox slot free again" are 32-bit sequence numbers written and awaited by the streams themselves
 * (stream memory operations): no SM is taken from the persistent pass kernels and no host thread waits in between, so
 * the gather + merge of step i overlap the pass of step i + 1 (two mailbox slots per rank).
 * A group is not thread-safe. All entries return PMB_OK or a negative code (text: pmb_group_last_error). */
typedef struct pmb_group pmb_group;
#define PMB_GROUP_HANDLE_BYTES 128
int pmb_group_create(pmb_group** group, const int* devices, int n_local, int rank_base, int world);
void pmb_group_destroy(pmb_group* group);
const char* pmb_group_last_error(const pmb_group* group);
int pmb_group_world(const pmb_group* group);
pmb_ctx* pmb_group_ctx(pmb_group* group, int local_index); /* the context of a local rank: options, timings, stream */
/* Column range [*col_begin, *col_end) of `rank` for an alignment of n_cols columns split over `world` ranks: contiguous,
 * ascending with the rank, boundaries on multiples of 1024 columns; empty for the last ranks of a very short alignment. */
int pmb_group_column_range(int world, int64_t n_cols, int rank, int64_t* col_begin, int64_t* col_end);
int pmb_group_set_tree(pmb_group* group, int32_t n_nodes, int32_t root, const int32_t* child_offsets, const int32_t* child_index,
                       const int32_t* leaf_row);
/* Mailbox capacity, in records per shard (rank 0 holds 2 x world slots of pmb_packed_bytes(n_nodes, capacity)). Must be
 * called after pmb_group_set_tree, with the same value on every rank, before export / connect; a single-process group
 * (n_local == world) may call it again later to grow. */
int pmb_group_reserve(pmb_group* group, int64_t shard_capacity_records);
int pmb_group_export(pmb_group* group, void* handles_out /* n_local x PMB_GROUP_HANDLE_BYTES */);
int pmb_group_connect(pmb_group* group, const void* all_handles /* world x PMB_GROUP_HANDLE_BYTES, rank order */);
/* Inputs. pmb_group_upload_nuc takes the WHOLE alignment (arguments as pmb_upload_nuc, positions count from column 0):
 * every local rank copies its own column range out of it. pmb_group_upload_shard takes one local rank's range only (the
 * caller sliced or generated it): column col_begin of the range is the low nibble of byte 0 of every row, parent_code /
 * root_override / fwd_root_ref start at col_begin too. Uploads of the local ranks run concurrently. */
int pmb_group_upload_nuc(pmb_group* group, int64_t n_cols, int32_t n_rows, const uint8_t* leaf_codes_4bit, int64_t row_stride_bytes,
                         const uint8_t* leaf_present, const uint8_t* parent_code, const int8_t* root_override,
                         const int8_t* fwd_root_ref);
int pmb_group_upload_shard(pmb_group* group, int local_index, int64_t n_cols_total, int32_t n_rows, const uint8_t* shard_codes_4bit,
                           int64_t row_stride_bytes, const uint8_t* leaf_present, const uint8_t* shard_parent_code,
                           const int8_t* shard_root_override, const int8_t* shard_fwd_root_ref);
/* One step, enqueued on every local rank and returning at once: pass -> pack into rank 0's mailbox -> signal; on the
 * process holding rank 0 also: wait for all `world` signals -> merge -> release the slots. Steps may be issued back to
 * back; pmb_group_wait drains everything and reports the first error of any local rank or of the merge. */
int pmb_group_run_async(pmb_group* group, int algo, int flags);
int pmb_group_wait(pmb_group* group);
/* Results, on the process holding rank 0 (elsewhere: n_mut = 0, NULL pointers). Device view / host copy of the merged
 * lists of the last step, and their run-merge (as pmb_merge_runs). */
int pmb_group_result_device(pmb_group* group, pmb_result* out);
int pmb_group_download(pmb_group* group, pmb_result* out);
int pmb_group_merge_runs(pmb_group* group, int to_host, pmb_nucmut_result* out);
/* Host buffers in, merged host lists out: upload + one step + wait + download (the end-to-end entry over several GPUs). */
int pmb_group_run_nuc(pmb_group* group, int algo, int64_t n_cols, int32_t n_rows, const uint8_t* leaf_codes_4bit,
                      int64_t row_stride_bytes, const uint8_t* leaf_present, const uint8_t* parent_code, const int8_t* root_override,
                      const int8_t* fwd_root_ref, int flags, pmb_result* out);

/* ---- a denser form of the same input at the boundary: the clade-run encoding ("pmb_runs") ----
 * The nibble matrix above is what crosses PCIe in pmb_run_nuc: 0.5 byte per leaf and column, the end-to-end limit of a
 * pass that itself runs at the HBM roofline. A phylogenetic alignment is far more regular than that: with the leaves in
 * depth-first order of the tree a clade is a run of consecutive rows, and inside a column a leaf almost always carries
 * the code of the leaf before it. pmb_runs_encode walks the rows of a HOST nibble matrix in that order and keeps, per
 * tile of 1024 columns, only the places where (code XOR parent_code) changes from one leaf to the next -- a few events
 * per column (in the order of the column's parsimony score) instead of one nibble per leaf. The device rebuilds exactly
 * the bit-planes pmb_upload_nuc would have produced (expand_runs_kernel), so every result is bit-identical; only the
 * bytes that cross the link differ. Pure host-side data preparation, like the nibble packing it stands in for: it needs no
 * device (the buffers are page-locked when there is one) and takes the tree by value, not a context.
 * The reference has no counterpart (its columns are read out of std::string sequences, src/panman.cpp:1396-1418). */
typedef struct pmb_runs pmb_runs;
typedef struct pmb_runs_info {
    int64_t n_cols;
    int32_t n_rows, n_tiles, n_segments, seg_rows; /* events are grouped per (tile, segment of seg_rows leaves) */
    int64_t n_events;
    int64_t bytes;                /* what an upload of the whole batch moves: events + item offsets */
    const uint32_t* events;       /* row in segment << 14 | column in tile << 4 | xor nibble */
    const int64_t* item_offsets;  /* n_tiles * n_segments + 1 */
} pmb_runs_info;
/* Tree arguments as pmb_set_tree, matrix arguments as pmb_run_nuc (host memory). n_threads <= 0: all cores. */
int pmb_runs_encode(int32_t n_nodes, int32_t root, const int32_t* child_offsets, const int32_t* child_index, const int32_t* leaf_row,
                    int64_t n_cols, int32_t n_rows, const uint8_t* leaf_codes_4bit, int64_t row_stride_bytes, const uint8_t* parent_code,
                    int n_threads, pmb_runs** out);
void pmb_runs_free(pmb_runs* runs);
int pmb_runs_describe(const pmb_runs* runs, pmb_runs_info* out);
/* As pmb_upload_nuc / pmb_upload_nuc_async / pmb_run_nuc with the leaf codes taken from `runs`: columns
 * [col_begin, col_begin + n_cols) of the encoded batch (col_begin a multiple of 1024; the range ends on a multiple of 1024 or
 * with the batch). parent_code / root_override / fwd_root_ref point at the RANGE's first column; parent_code must be the
 * one the batch was encoded against. The context's tree must be the tree of the encoding (PMB_ERR_INVALID otherwise). */
int pmb_upload_runs(pmb_ctx* ctx, const pmb_runs* runs, int64_t col_begin, int64_t n_cols, const uint8_t* leaf_present,
                    const uint8_t* parent_code, const int8_t* root_override, const int8_t* fwd_root_ref, int64_t col_base);
int pmb_upload_runs_async(pmb_ctx* ctx, const pmb_runs* runs, int64_t col_begin, int64_t n_cols, const uint8_t* leaf_present,
                          const uint8_t* parent_code, const int8_t* root_override, const int8_t* fwd_root_ref, int64_t col_base);
int pmb_run_runs(pmb_ctx* ctx, int algo, const pmb_runs* runs, const uint8_t* leaf_present, const uint8_t* parent_code,
                 const int8_t* root_override, const int8_t* fwd_root_ref, int64_t col_base, int flags, pmb_result* out);
/* Over a group. pmb_group_upload_runs: `runs` encodes the WHOLE alignment, every local rank takes the tiles of its own
 * column range (only those events cross its link). pmb_group_upload_shard_runs: `shard_runs` encodes one local rank's
 * range only (one process per GPU: every rank encodes and uploads its own). pmb_group_run_runs = upload + step + download. */
int pmb_group_upload_runs(pmb_group* group, const pmb_runs* runs, const uint8_t* leaf_present, const uint8_t* parent_code,
                          const int8_t* root_override, const int8_t* fwd_root_ref);
int pmb_group_upload_shard_runs(pmb_group* group, int local_index, int64_t n_cols_total, const pmb_runs* shard_runs,
                                const uint8_t* leaf_present, const uint8_t* shard_parent_code, const int8_t* shard_root_override,
                                const int8_t* shard_fwd_root_ref);
int pmb_group_run_runs(pmb_group* group, int algo, const pmb_runs* runs, const uint8_t* leaf_present, const uint8_t* parent_code,
                       const int8_t* root_override, const int8_t* fwd_root_ref, int flags, pmb_result* out);

/* ---- introspection ---- */
int pmb_last_timings(const pmb_ctx* ctx, pmb_timings* out);
/* Bytes the roofline is computed on, for the resident input and `algo` (SURVEY.md 8d):
 * Fitch n_cols*(1.0*L + 4*I), Sankoff n_cols*(1.0*L + 8*I), plus 8 bytes per emitted record. */
int64_t pmb_algorithmic_bytes(const pmb_ctx* ctx, int algo);
const char* pmb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PANMAN_B200_H */
