// Host-side encoder of the clade-run form of a leaf matrix (pmb_runs_encode, include/panman_b200.h). Data preparation
// only -- like the nibble packing it replaces at the boundary -- no part of the Fitch / Sankoff computation happens here.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <new>
#include <thread>

#include "../../include/panman_b200.h"
#include "pmb_runs.h"

namespace pmb {

std::vector<int32_t> dfs_leaf_rows(int32_t n_nodes, int32_t root, const int32_t* child_off, const int32_t* child_idx,
                                   const int32_t* leaf_row) {
    std::vector<int32_t> rows;
    if (n_nodes < 1 || root < 0 || root >= n_nodes) return rows;
    std::vector<int32_t> stack{root};
    int64_t visited = 0;
    while (!stack.empty()) {
        const int32_t v = stack.back();
        stack.pop_back();
        if (++visited > n_nodes) return {};  // a cycle
        const int32_t a = child_off[v], z = child_off[v + 1];
        if (a == z) {
            rows.push_back(leaf_row[v]);
            continue;
        }
        for (int32_t e = z - 1; e >= a; e--) {  // first child on top
            const int32_t c = child_idx[e];
            if (c < 0 || c >= n_nodes) return {};
            stack.push_back(c);
        }
    }
    return rows;
}

uint64_t leaf_order_hash(const std::vector<int32_t>& rows) {
    uint64_t h = 1469598103934665603ull;  // FNV-1a over the row numbers
    for (int32_t r : rows) {
        h ^= uint64_t(uint32_t(r));
        h *= 1099511628211ull;
    }
    return h ^ (uint64_t(rows.size()) << 32);
}

// enough (tile, segment) items to give every resident warp of the device one, never fewer than 64 leaves per segment (every
// segment start re-states its first leaf in full), never more than the row field holds
void runs_segments(int64_t n_rows, int64_t T, int32_t* n_seg_out, int32_t* seg_rows_out) {
    int64_t n_seg = std::max<int64_t>(1, (8192 + T - 1) / T);
    n_seg = std::min<int64_t>(n_seg, std::max<int64_t>(1, n_rows / 64));
    n_seg = std::max<int64_t>(n_seg, (n_rows + RUNS_MAX_SEG_ROWS - 1) / RUNS_MAX_SEG_ROWS);
    const int64_t seg_rows = (n_rows + n_seg - 1) / n_seg;
    *n_seg_out = int32_t((n_rows + seg_rows - 1) / seg_rows);
    *seg_rows_out = int32_t(seg_rows);
}

}  // namespace pmb

namespace {

constexpr int TILE_BYTES = 512;  // 1024 columns of one row, nibble-packed
constexpr int TILE_WORDS = 64;
constexpr int GROUP = 8;         // tiles walked side by side: one row contributes 4 KB of consecutive bytes

void* alloc_host(size_t bytes, bool* pinned) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) == cudaSuccess) {
        *pinned = true;
        return p;
    }
    cudaGetLastError();  // no usable device: the encoder itself needs none
    *pinned = false;
    return std::malloc(bytes ? bytes : 1);
}

void free_host(void* p, bool pinned) {
    if (!p) return;
    if (pinned) cudaFreeHost(p);
    else std::free(p);
}

// 512 bytes of row `src` starting at byte `b0`, zero beyond the row's `row_bytes`; the unused high nibble of an odd
// column count is cleared (pack_leaves_kernel does the same)
inline void load_block(const uint8_t* src, int64_t b0, int64_t row_bytes, bool odd, uint64_t* dst) {
    const int64_t have = std::min<int64_t>(TILE_BYTES, row_bytes - b0);
    if (have == TILE_BYTES && !(odd && b0 + TILE_BYTES == row_bytes)) {
        std::memcpy(dst, src + b0, TILE_BYTES);
        return;
    }
    std::memset(dst, 0, TILE_BYTES);
    if (have <= 0) return;
    std::memcpy(dst, src + b0, size_t(have));
    if (odd && b0 + have == row_bytes) reinterpret_cast<uint8_t*>(dst)[have - 1] &= 0x0F;
}

}  // namespace

extern "C" {

int pmb_runs_encode(int32_t n_nodes, int32_t root, const int32_t* child_offsets, const int32_t* child_index, const int32_t* leaf_row,
                    int64_t n_cols, int32_t n_rows, const uint8_t* leaf_codes_4bit, int64_t row_stride_bytes, const uint8_t* parent_code,
                    int n_threads, pmb_runs** out) {
    if (!out) return PMB_ERR_INVALID;
    *out = nullptr;
    if (!child_offsets || !child_index || !leaf_row || !leaf_codes_4bit || !parent_code || n_cols <= 0 || n_rows <= 0 ||
        row_stride_bytes < (n_cols + 1) / 2 || n_cols > (int64_t(1) << 40))
        return PMB_ERR_INVALID;
    pmb_runs* R = nullptr;
    try {
        const std::vector<int32_t> order = pmb::dfs_leaf_rows(n_nodes, root, child_offsets, child_index, leaf_row);
        if (int64_t(order.size()) != n_rows) return PMB_ERR_INVALID;
        {
            std::vector<char> seen(size_t(n_rows), 0);
            for (int32_t r : order) {
                if (r < 0 || r >= n_rows || seen[size_t(r)]) return PMB_ERR_INVALID;
                seen[size_t(r)] = 1;
            }
        }
        const int64_t T = (n_cols + 1023) / 1024;
        if (T > (int64_t(1) << 30)) return PMB_ERR_INVALID;
        int32_t n_seg32 = 0, seg_rows32 = 0;
        pmb::runs_segments(n_rows, T, &n_seg32, &seg_rows32);
        const int64_t n_seg = n_seg32, seg_rows = seg_rows32;

        R = new pmb_runs();
        R->n_cols = n_cols;
        R->n_rows = n_rows;
        R->T = int32_t(T);
        R->n_seg = int32_t(n_seg);
        R->seg_rows = int32_t(seg_rows);
        R->order_hash = pmb::leaf_order_hash(order);
        const int64_t n_items = T * n_seg;
        R->item_off = static_cast<int64_t*>(alloc_host(size_t(n_items + 1) * sizeof(int64_t), &R->pinned_off));
        if (!R->item_off) throw std::bad_alloc();

        const int64_t row_bytes = (n_cols + 1) / 2;
        const bool odd = n_cols & 1;
        std::vector<std::vector<uint32_t>> tile_events(static_cast<size_t>(T));
        std::vector<int64_t> item_count(size_t(n_items), 0);
        const int64_t n_groups = (T + GROUP - 1) / GROUP;
        std::atomic<int64_t> next{0};
        std::atomic<bool> oom{false};
        auto worker = [&]() {
            try {
                std::vector<uint64_t> cons(size_t(GROUP) * TILE_WORDS), prev(size_t(GROUP) * TILE_WORDS), cur(TILE_WORDS);
                for (;;) {
                    const int64_t g = next.fetch_add(1);
                    if (g >= n_groups || oom.load()) break;
                    const int64_t t0 = g * GROUP, nt = std::min<int64_t>(GROUP, T - t0);
                    for (int64_t k = 0; k < nt; k++) {  // the parent codes of the tile, packed like a row
                        uint8_t* cb = reinterpret_cast<uint8_t*>(&cons[size_t(k) * TILE_WORDS]);
                        std::memset(cb, 0, TILE_BYTES);
                        const int64_t c0 = (t0 + k) * 1024, c1 = std::min<int64_t>(n_cols, c0 + 1024);
                        for (int64_t c = c0; c < c1; c++) cb[(c - c0) >> 1] |= uint8_t((parent_code[c] & 15) << (4 * ((c - c0) & 1)));
                    }
                    for (int64_t seg = 0; seg < n_seg; seg++) {
                        std::fill(prev.begin(), prev.end(), 0);
                        const int64_t r_begin = seg * seg_rows, r_end = std::min<int64_t>(n_rows, r_begin + seg_rows);
                        for (int64_t r = r_begin; r < r_end; r++) {
                            const uint8_t* src = leaf_codes_4bit + size_t(order[size_t(r)]) * size_t(row_stride_bytes);
                            const uint32_t row_field = uint32_t(r - r_begin) << pmb::RUNS_ROW_SHIFT;
                            for (int64_t k = 0; k < nt; k++) {
                                load_block(src, (t0 + k) * TILE_BYTES, row_bytes, odd, cur.data());
                                const uint64_t* cw = &cons[size_t(k) * TILE_WORDS];
                                uint64_t* pw = &prev[size_t(k) * TILE_WORDS];
                                uint64_t any = 0;
                                for (int w = 0; w < TILE_WORDS; w++) {
                                    cur[size_t(w)] ^= cw[w];
                                    any |= cur[size_t(w)] ^ pw[w];
                                }
                                if (!any) continue;
                                std::vector<uint32_t>& ev = tile_events[size_t(t0 + k)];
                                for (int w = 0; w < TILE_WORDS; w++) {
                                    uint64_t d = cur[size_t(w)] ^ pw[w];
                                    pw[w] = cur[size_t(w)];
                                    while (d) {
                                        const int nib = __builtin_ctzll(d) >> 2;
                                        const uint32_t x = uint32_t(d >> (4 * nib)) & 15u;
                                        ev.push_back(row_field | uint32_t(w * 16 + nib) << 4 | x);
                                        item_count[size_t((t0 + k) * n_seg + seg)]++;
                                        d &= ~(uint64_t(15) << (4 * nib));
                                    }
                                }
                            }
                        }
                    }
                }
            } catch (const std::bad_alloc&) {
                oom.store(true);
            }
        };
        int nth = n_threads > 0 ? n_threads : int(std::thread::hardware_concurrency());
        nth = int(std::max<int64_t>(1, std::min<int64_t>(std::min(nth, 256), n_groups)));
        {
            std::vector<std::thread> pool;
            for (int i = 1; i < nth; i++) pool.emplace_back(worker);
            worker();
            for (auto& t : pool) t.join();
        }
        if (oom.load()) throw std::bad_alloc();
        R->item_off[0] = 0;
        for (int64_t i = 0; i < n_items; i++) R->item_off[i + 1] = R->item_off[i] + item_count[size_t(i)];
        R->n_events = R->item_off[n_items];
        R->events = static_cast<uint32_t*>(alloc_host(size_t(std::max<int64_t>(1, R->n_events)) * sizeof(uint32_t), &R->pinned_events));
        if (!R->events) throw std::bad_alloc();
        {   // a tile's events are already in item order (segment-major, rows ascending): one copy per tile
            std::atomic<int64_t> nt{0};
            auto copier = [&]() {
                for (;;) {
                    const int64_t t = nt.fetch_add(1);
                    if (t >= T) break;
                    const std::vector<uint32_t>& ev = tile_events[size_t(t)];
                    if (!ev.empty()) std::memcpy(R->events + R->item_off[t * n_seg], ev.data(), ev.size() * sizeof(uint32_t));
                }
            };
            std::vector<std::thread> pool;
            for (int i = 1; i < std::min(nth, 8); i++) pool.emplace_back(copier);
            copier();
            for (auto& t : pool) t.join();
        }
        *out = R;
        return PMB_OK;
    } catch (const std::bad_alloc&) {
        pmb_runs_free(R);
        return PMB_ERR_OOM;
    } catch (const std::exception&) {
        pmb_runs_free(R);
        return PMB_ERR_INVALID;
    }
}

void pmb_runs_free(pmb_runs* r) {
    if (!r) return;
    free_host(r->events, r->pinned_events);
    free_host(r->item_off, r->pinned_off);
    delete r;
}

int pmb_runs_describe(const pmb_runs* r, pmb_runs_info* out) {
    if (!r || !out) return PMB_ERR_INVALID;
    out->n_cols = r->n_cols;
    out->n_rows = r->n_rows;
    out->n_tiles = r->T;
    out->n_segments = r->n_seg;
    out->seg_rows = r->seg_rows;
    out->n_events = r->n_events;
    out->bytes = r->n_events * int64_t(sizeof(uint32_t)) + (int64_t(r->T) * r->n_seg + 1) * int64_t(sizeof(int64_t));
    out->events = r->events;
    out->item_offsets = r->item_off;
    return PMB_OK;
}

}  // extern "C"
