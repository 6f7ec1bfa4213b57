// Clade-run encoded leaf matrix (pmb_runs, include/panman_b200.h): internal layout shared by the host encoder
// (pmb_runs.cpp) and the upload path (pmb_api.cu, expand_runs_kernel).
#pragma once
#include <cstdint>
#include <vector>

// Leaves are numbered in depth-first order of the tree (children in Newick order), so a clade is one contiguous run of
// rows. Per column tile (1024 columns) and per segment of `seg_rows` consecutive leaves, walking the leaves in that order:
// whenever the leaf's 4-bit code XOR the column's parent code differs from the previous leaf's (0 at the start of a
// segment), one event says which nibble toggles by what:
//     event = row-in-segment << 14 | column-in-tile << 4 | xor of the two (code ^ parent_code) nibbles
// Events of an item (tile * n_seg + segment) are consecutive, ascending by row, then by column; item_off indexes them.
struct pmb_runs {
    int64_t n_cols = 0;
    int32_t n_rows = 0;
    int32_t T = 0;         // column tiles
    int32_t n_seg = 0;     // segments of leaves per tile
    int32_t seg_rows = 0;  // leaves per segment (< 2^18 - 1: the all-ones row is the end marker on the device)
    uint64_t order_hash = 0;  // of the depth-first leaf order the rows were walked in (a batch only fits its own tree)
    int64_t n_events = 0;
    uint32_t* events = nullptr;   // page-locked when a device is usable, else plain
    int64_t* item_off = nullptr;  // T * n_seg + 1
    bool pinned_events = false, pinned_off = false;
};

namespace pmb {
constexpr int RUNS_ROW_SHIFT = 14;
constexpr uint32_t RUNS_MAX_SEG_ROWS = (1u << 18) - 2;

// caller's leaf rows in depth-first order of the tree; empty on a malformed tree
std::vector<int32_t> dfs_leaf_rows(int32_t n_nodes, int32_t root, const int32_t* child_off, const int32_t* child_idx,
                                   const int32_t* leaf_row);
uint64_t leaf_order_hash(const std::vector<int32_t>& rows);
// leaves per (tile, segment) item for n_rows leaves and T column tiles (pmb_runs_encode, pmb_upload_replay)
void runs_segments(int64_t n_rows, int64_t T, int32_t* n_seg, int32_t* seg_rows);
}  // namespace pmb
