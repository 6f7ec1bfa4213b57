/* libpanman_b200_host -- host-side adaptor above libpanman_b200 (C++ inside, C ABI outside).
 *
 * It restates the parts of the reference's Tree constructor that surround the per-column passes, so that the
 * -M / -N construction flow can be exercised end to end without the reference's TBB/Boost/capnp dependencies:
 *   - Newick -> tree with the reference's node ids and child order   (reference src/panman.cpp:310-450)
 *   - FASTA/MSA reader, consensus rule, all-gap column removal        (reference src/panman.cpp:1288-1362, 1479-1557)
 *   - per-column inputs -> pmb_run_nuc                                 (replaces the loops at :1381-1435 and :1568-1613)
 *   - per-node sort order + greedy <=6 run-merge into NucMut fields    (reference src/panman.cpp:1445-1466, 1625-1646;
 *                                                                        NucMut ctor src/panman.hpp:109-151)
 * The outputs are exactly the fields the reference stores in Node::nucMutation / Node::blockMutation, in the order
 * it stores them; the capnp writer (src/panman.cpp:2854-2929) stays the reference's own.
 */
#ifndef PANMAN_B200_HOST_H
#define PANMAN_B200_HOST_H

#include <stddef.h>
#include <stdint.h>

#include "panman_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pmh_tree pmh_tree;
typedef struct pmh_build pmh_build;

/* One NucMut as the reference holds it (src/panman.hpp:75-81). */
typedef struct pmh_nucmut {
    int32_t nucPosition;
    int32_t nucGapPosition;   /* -1 for MSA builds */
    int32_t primaryBlockId;   /* 0 for MSA builds */
    int32_t secondaryBlockId; /* -1 */
    uint8_t mutInfo;          /* (length << 4) + type */
    uint32_t nucs;            /* code_k << (4 * (5 - k)) */
} pmh_nucmut;

/* One BlockMut as the reference holds it (src/panman.hpp:429-440; ctor :467-484). */
typedef struct pmh_blockmut {
    int32_t primaryBlockId;
    int32_t secondaryBlockId; /* -1 */
    uint8_t blockMutInfo;     /* 1 = insertion; 0 = deletion, or an inversion when `inversion` is set */
    uint8_t inversion;        /* insertion: the block is inserted inverted; else: the present block is inverted */
} pmh_blockmut;

/* One node's mutations as the reference's writer lays them out (Tree::getNodesPreorder, src/panman.cpp:2854-2929; schema
 * panman.capnp Mutation / NucMut): the node's NucMut grouped by block in std::map order, every piece with mutInfo in its wire
 * form ((nucs >> (24 - 4 * length)) << 8) + mutInfo, every group with the node's block mutation of that block if any. This
 * is the content of the capnp message; the byte encoding itself needs Cap'n Proto and stays the reference's. Nodes are
 * written in pre-order, which is the node id order of pmh_tree. */
typedef struct pmh_wire_nuc {
    int32_t nucPosition;
    int32_t nucGapPosition; /* 0 when nucGapExist is 0 */
    uint8_t nucGapExist;
    uint32_t mutInfo;
} pmh_wire_nuc;
typedef struct pmh_wire_mutation {
    int64_t blockId;        /* (primaryBlockId << 32) + secondaryBlockId, the latter only when blockGapExist */
    uint8_t blockGapExist;
    uint8_t blockMutExist;  /* the node has a block mutation for this block */
    uint8_t blockMutInfo;   /* insertion (1) / deletion or inversion (0); 1 when blockMutExist is 0 (the writer's default) */
    uint8_t blockInversion; /* 1 when blockMutExist is 0 (the writer's default) */
    int64_t nuc_begin, nuc_end; /* this group's pieces: [nuc_begin, nuc_end) of the node's pmh_wire_nuc array */
} pmh_wire_mutation;

/* ---- Newick ---- */
pmh_tree* pmh_tree_from_newick(const char* newick, char* err, size_t err_len); /* NULL on malformed input */
void pmh_tree_free(pmh_tree* t);
int32_t pmh_tree_n_nodes(const pmh_tree* t);
int32_t pmh_tree_n_leaves(const pmh_tree* t);
int32_t pmh_tree_root(const pmh_tree* t);
const char* pmh_tree_name(const pmh_tree* t, int32_t node);
const int32_t* pmh_tree_parent(const pmh_tree* t);
const int32_t* pmh_tree_child_offsets(const pmh_tree* t);
const int32_t* pmh_tree_child_index(const pmh_tree* t);
const int32_t* pmh_tree_leaf_row(const pmh_tree* t);
int pmh_tree_has_polytomy(const pmh_tree* t); /* reference src/panman.cpp:621-631 */
/* Tree::transform (reference src/panman.cpp:5831-5906, called by Tree::reroot src/reroot.cpp:38): a NEW tree in which the
 * tip `leaf_name` is the first child of a new root "node_<k+1>" and its former ancestors hang below it upside down (each
 * receives its old parent as its last child; an old root left with one child disappears). A tip that is the root's child
 * changes nothing. Node ids of the result are a pre-order walk; names and leaf rows travel with the nodes. NULL + err when
 * the name is unknown or not a tip (src/reroot.cpp:5-13). */
pmh_tree* pmh_tree_reroot(const pmh_tree* t, const char* leaf_name, char* err, size_t err_len);

/* ---- MSA construction: panmanUtils -M msa.fa -N tree.nwk [--reference id] [--low-mem-mode] ----
 * fasta / newick are the file contents. low_mem_mode = 0: Fitch (reference FILE_TYPE::MSA, src/panman.cpp:1274-1466);
 * 1: Sankoff (FILE_TYPE::MSA_OPTIMIZE, :1467-1649). Returns NULL and fills err on failure. */
pmh_build* pmh_build_from_msa(pmb_ctx* ctx, const char* fasta, size_t fasta_len, const char* newick, const char* reference,
                              int low_mem_mode, char* err, size_t err_len);
/* The same in two steps. pmh_msa_prepare is host-only (reader, consensus, all-gap column removal, packing: no device
 * needed) and leaves the column batch in the build object; pmh_msa_run uploads it, runs the pass and the run-merge. */
pmh_build* pmh_msa_prepare(const char* fasta, size_t fasta_len, const char* newick, const char* reference, int low_mem_mode,
                           char* err, size_t err_len);
int pmh_msa_run(pmb_ctx* ctx, pmh_build* b, char* err, size_t err_len);
/* The same over the GPUs of a box: `group` = a single-process pmb_group (pmb_group_create with all its devices); the columns
 * of the batch are split into contiguous ranges, one per GPU, and the lists come back merged (include/panman_b200.h). */
int pmh_msa_run_group(pmb_group* group, pmh_build* b, char* err, size_t err_len);
/* Tree::reroot (reference src/reroot.cpp:4-261) of a built MSA PanMAT, with the tip `leaf_name` as the new root: the tree is
 * transformed (pmh_tree_reroot); every leaf's sequence is what the build's Node::nucMutation yields for it
 * (getSequenceFromReference, src/reroot.cpp:19-35), rebuilt on the device by pmb_upload_replay; every column is inferred
 * again by Fitch (also for a --low-mem-mode build) with the root forced to the tip's own code, and the lists are run-merged
 * (src/reroot.cpp:134-261). Afterwards pmh_build_tree / _nucmut / _wire / the tuple arrays describe the re-rooted tree (new
 * node ids); it may be rerooted again. PMB_ERR_INVALID with "Sequence with name ... not found!" for an unknown name, or for a
 * node that is not a tip (its message from pmh_tree_reroot); PMB_ERR_NO_INPUT before pmh_msa_run / pmh_build_from_msa. */
int pmh_msa_reroot(pmb_ctx* ctx, pmh_build* b, const char* leaf_name, char* err, size_t err_len);
int64_t pmh_build_n_cols(const pmh_build* b);
const uint8_t* pmh_build_codes4(const pmh_build* b, int64_t* row_stride); /* n_leaves rows; NULL once pmh_msa_run consumed it */
const uint8_t* pmh_build_present(const pmh_build* b);                      /* n_leaves */
const uint8_t* pmh_build_parent_code(const pmh_build* b);                  /* n_cols */
const int8_t* pmh_build_root_override(const pmh_build* b);                 /* n_cols or NULL */
const int8_t* pmh_build_fwd_root_ref(const pmh_build* b);                  /* n_cols or NULL */
void pmh_build_free(pmh_build* b);
/* Tuning: FASTA texts of at least this many bytes are cut at header lines and parsed by several threads (default 8 MiB;
 * 0 = always). The records are stored in file order either way, so the result does not depend on it. */
void pmh_set_reader_parallel_bytes(int64_t bytes);
const pmh_tree* pmh_build_tree(const pmh_build* b);
const char* pmh_build_consensus(const pmh_build* b, int64_t* len); /* blocks[0] consensus (src/panman.cpp:1439) */
int64_t pmh_build_n_nucmut(const pmh_build* b, int32_t node);
const pmh_nucmut* pmh_build_nucmut(const pmh_build* b, int32_t node); /* Node::nucMutation, in stored order */
/* the node's Mutation list as the writer would store it (see pmh_wire_mutation); the root carries the block insertion of
 * the single block (src/panman.cpp:1439-1440). Returns the number of groups. */
int64_t pmh_build_wire(const pmh_build* b, int32_t node, const pmh_wire_mutation** mutations, const pmh_wire_nuc** nucs);
/* raw per-node tuples (pos, type, code) before the merge, node-major (debugging / parity) */
int64_t pmh_build_n_tuples(const pmh_build* b);
const int64_t* pmh_build_tuple_offsets(const pmh_build* b);
const int32_t* pmh_build_tuple_pos(const pmh_build* b);
const uint8_t* pmh_build_tuple_type_code(const pmh_build* b);
/* seconds spent: [0] parse+consensus, [1] pack, [2] pmb_run_nuc, [3] run-merge */
const double* pmh_build_seconds(const pmh_build* b);

/* ---- PanGraph construction: panmanUtils -P pangraph.json -N tree.nwk [--reference id] ----
 * pmh_pangraph_load parses the PanGraph JSON (reference src/panman.cpp:6200-6258) and builds, per block, the column batch
 * the nucleotide passes run on: one column per consensus position 0..len ("main", the last one '-') and one per gap slot
 * (pos, k); a sequence contributes its aligned character (consensus + substitutions / insertions / deletions,
 * src/panman.cpp:1006-1045), sequences whose path lacks the block are omitted (leaf_present). Block columns ("blocks" below)
 * follow the reference's own ordering: the consensus order chain_align builds over the paths (src/chaining.cpp:153-310,
 * driven by src/panman.cpp:6347-6425), one column per occurrence of a duplicated block with the mutations recorded for
 * that occurrence ("number"), circular paths rotated against the first path (src/rotation.cpp:14-110); a path entry that
 * the two-pointer alignment to that order cannot place is dropped as in the reference (src/panman.cpp:6427-6465). The
 * root override follows the rules stated in panman_b200/host/pangraph.cpp. pmh_pangraph_run runs the block-level pass (3 states, PMB_FLAG_BLOCK_MODE,
 * src/panman.cpp:873-963) and one pmb_run_nuc per block (src/panman.cpp:1048-1232); algo = PMB_ALGO_FITCH for a bifurcating
 * tree, PMB_ALGO_SANKOFF for the reference's polytomy branch. Results are the per-node (position-sorted) lists of every
 * batch; column c of block b is (pmh_pangraph_col_pos[c], pmh_pangraph_col_gap[c]), gap = -1 for main columns. */
typedef struct pmh_pangraph pmh_pangraph;
pmh_pangraph* pmh_pangraph_load(const char* json, size_t json_len, const char* newick, const char* reference, char* err,
                                size_t err_len);
void pmh_pangraph_free(pmh_pangraph* g);
const pmh_tree* pmh_pangraph_tree(const pmh_pangraph* g);
int32_t pmh_pangraph_n_blocks(const pmh_pangraph* g);
const char* pmh_pangraph_block_id(const pmh_pangraph* g, int32_t block);
const uint8_t* pmh_pangraph_block_states(const pmh_pangraph* g); /* n_leaves x n_blocks: 0 absent, 1 forward, 2 reverse */
/* n_leaves: by how many blocks a circular path was rotated to line up with the first path (what the reference keeps as
 * Tree::rotationIndexes, src/panman.cpp:835-837, src/rotation.cpp:96); 0 for linear paths */
const int32_t* pmh_pangraph_rotation_index(const pmh_pangraph* g);
/* n_blocks or NULL (no --reference): the state the block-level pass forces the root to (defaultState, src/panman.cpp:881-897),
 * -1 where no sequence matches */
const int8_t* pmh_pangraph_block_override(const pmh_pangraph* g);
int64_t pmh_pangraph_n_cols(const pmh_pangraph* g, int32_t block);
const uint8_t* pmh_pangraph_codes4(const pmh_pangraph* g, int32_t block, int64_t* row_stride);
const uint8_t* pmh_pangraph_present(const pmh_pangraph* g, int32_t block);
const uint8_t* pmh_pangraph_parent_code(const pmh_pangraph* g, int32_t block);
const int8_t* pmh_pangraph_root_override(const pmh_pangraph* g, int32_t block);
const int32_t* pmh_pangraph_col_pos(const pmh_pangraph* g, int32_t block);
const int32_t* pmh_pangraph_col_gap(const pmh_pangraph* g, int32_t block);
int pmh_pangraph_run(pmb_ctx* ctx, pmh_pangraph* g, int algo, char* err, size_t err_len);
/* Node::nucMutation after pmh_pangraph_run (greedy <= 6 run-merge on the device, src/panman.cpp:1236-1272; 6-tuple NucMut
 * ctor src/panman.hpp:154-189): the non-gap pieces of all blocks, then the gap pieces; primaryBlockId = block index. */
int64_t pmh_pangraph_n_nucmut(const pmh_pangraph* g, int32_t node);
const pmh_nucmut* pmh_pangraph_nucmut(const pmh_pangraph* g, int32_t node);
/* Node::blockMutation after pmh_pangraph_run / pmh_pangraph_reroot: BlockMut(blockId, (type, inversion)) of
 * src/panman.hpp:467-484 as applied at src/panman.cpp:971-980, in ascending block id. */
int64_t pmh_pangraph_n_blockmut(const pmh_pangraph* g, int32_t node);
const pmh_blockmut* pmh_pangraph_blockmut(const pmh_pangraph* g, int32_t node);
/* the node's Mutation list as the writer would store it (see pmh_wire_mutation), after pmh_pangraph_run / _reroot.
 * Returns the number of groups. */
int64_t pmh_pangraph_wire(const pmh_pangraph* g, int32_t node, const pmh_wire_mutation** mutations, const pmh_wire_nuc** nucs);
/* Tree::reroot (reference src/reroot.cpp:4-261) on the loaded graph, with `leaf_name` as the new root: the tree is
 * transformed (pmh_tree_reroot), then every block column (src/reroot.cpp:54-122) and every nucleotide column (:134-224) is
 * inferred again by Fitch with the root forced to the new root's own state (root override on EVERY column), every leaf
 * taking part with the characters the built PanMAT yields for it (getSequenceFromReference, src/reroot.cpp:19-35: the
 * mutations of the last pmh_pangraph_run replayed from the root over the consensus -- call that first), and the lists are
 * run-merged (:226-261).
 * Afterwards pmh_pangraph_tree / _nucmut / _blockmut / _result describe the re-rooted tree (new node ids). */
int pmh_pangraph_reroot(pmb_ctx* ctx, pmh_pangraph* g, const char* leaf_name, char* err, size_t err_len);
/* lists of one batch after pmh_pangraph_run; block = -1: the block-level pass. Returns the record count. */
int64_t pmh_pangraph_result(const pmh_pangraph* g, int32_t block, const int64_t** node_offsets, const int32_t** pos,
                            const uint8_t** type_code);

#ifdef __cplusplus
}
#endif
#endif
