// Host adaptor for `panmanUtils -M msa.fa -N tree.nwk [--reference id] [--low-mem-mode]` on top of the C ABI of
// libpanman_b200. Restates what surrounds the per-column passes in the reference's Tree constructor
// (src/panman.cpp:1274-1466 for FILE_TYPE::MSA, :1467-1649 for FILE_TYPE::MSA_OPTIMIZE); the passes themselves
// (the loops at :1381-1435 and :1568-1613) become ONE pmb_run_nuc call.
#include <algorithm>
#include <chrono>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <sstream>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/panman_b200_host.h"
#include "host_tree.hpp"

struct pmh_build {
    pmh_tree tree;
    std::string consensus;
    // the column batch (pmh_msa_prepare): nibble-packed leaf rows, presence, per-column parameters
    int low_mem_mode = 0;
    int64_t n_cols = 0, stride = 0;
    uint8_t* codes4 = nullptr;  // page-locked where the device library can provide it
    bool codes_cached = false;  // codes4 is the process-wide cached buffer (returned, not freed)
    std::vector<uint8_t> codes_pageable, present, parent_code;
    std::vector<int8_t> per_col;  // root_override (low-memory branch) or fwd_root_ref (MSA branch); empty = none
    ~pmh_build();
    std::vector<std::vector<pmh_nucmut>> nuc;
    mutable std::vector<pmh_wire_mutation> wire_muts;  // scratch of pmh_build_wire (one node at a time)
    mutable std::vector<pmh_wire_nuc> wire_nucs;
    std::vector<int64_t> tuple_off;
    std::vector<int32_t> tuple_pos;
    std::vector<uint8_t> tuple_tc;
    bool ran = false;  // the lists above describe `tree` (pmh_msa_run / pmh_msa_reroot succeeded)
    double seconds[4] = {0, 0, 0, 0};
};

namespace {

using Clock = std::chrono::steady_clock;
double since(Clock::time_point t0) { return std::chrono::duration<double>(Clock::now() - t0).count(); }

void set_err(char* err, size_t n, const std::string& m) {
    if (err && n) {
        std::strncpy(err, m.c_str(), n - 1);
        err[n - 1] = 0;
    }
}

// Page-locking costs about as much as one pageable upload of the same bytes, so one buffer is kept for the following
// builds of the process (PanGraph blocks, --low-mem-mode batches); a build that finds it taken pins its own.
struct PinCache {
    std::mutex m;
    uint8_t* buf = nullptr;
    size_t cap = 0;
    bool in_use = false;
} g_pin;

uint8_t* pin_acquire(size_t bytes, bool* cached) {
    std::lock_guard<std::mutex> lock(g_pin.m);
    if (!g_pin.in_use) {
        if (bytes > g_pin.cap) {
            pmb_host_free(g_pin.buf);
            g_pin.cap = 0;
            g_pin.buf = static_cast<uint8_t*>(pmb_host_alloc(bytes + bytes / 4));
            if (g_pin.buf) g_pin.cap = bytes + bytes / 4;
        }
        if (g_pin.buf) {
            g_pin.in_use = true;
            *cached = true;
            return g_pin.buf;
        }
    }
    *cached = false;
    return static_cast<uint8_t*>(pmb_host_alloc(bytes));  // may be NULL (no device): the caller falls back to pageable memory
}

void pin_release(uint8_t* p, bool cached) {
    if (!p) return;
    if (cached) {
        std::lock_guard<std::mutex> lock(g_pin.m);
        g_pin.in_use = false;
    } else {
        pmb_host_free(p);
    }
}

// reference src/panman.cpp:78-113 (getCodeFromNucleotide) as a table: unlisted characters (incl. '-') -> 0
struct CodeTable {
    uint8_t t[256];
    CodeTable() {
        std::memset(t, 0, sizeof t);
        const char* sym = "ACMGRSVTWYHKDBN";  // codes 1..15, src/panman.hpp:27-44
        for (int i = 0; i < 15; i++) t[(unsigned char)sym[i]] = uint8_t(i + 1);
    }
};
const CodeTable kCode;

// FASTA reader of the MSA branch (src/panman.cpp:1288-1325). `strip_cr`: the MSA branch cuts lines and ids at '\r',
// the low-memory branch (:1479-1501, readFastaInBatch :677-724) does not.
std::string first_piece(const std::string& s, char delim) {
    std::vector<std::string> w;
    pmh::split_quote_aware(s, delim, w);
    return w.empty() ? std::string() : w[0];
}

struct FastaRecord {
    std::string id;   // as the header gives it (text after '>' up to the first blank), before any '\r' cut
    std::string seq;  // the record's sequence lines joined
};

// One contiguous piece of the file, line by line, exactly like the reference's reader. A piece either starts at a header
// line or at the very beginning of the file (where sequence lines without a header belong to the id "").
// One copy per sequence byte: a line without '\r' is appended straight from the input (splitting at an absent delimiter
// returns the whole line).
void parse_fasta_piece(const char* text, size_t begin, size_t end, bool strip_cr, size_t reserve_hint, std::vector<FastaRecord>* out) {
    FastaRecord cur;
    bool open = false;  // a record (or the headerless start of the file) is being collected
    size_t p = begin;
    while (p < end) {
        const char* nl = static_cast<const char*>(std::memchr(text + p, '\n', end - p));
        size_t e = nl ? size_t(nl - text) : end;
        const char* lp = text + p;
        const size_t ln = e - p;
        p = e + 1;
        if (ln == 0) continue;
        if (lp[0] == '>') {
            if (open) out->push_back(std::move(cur));
            cur = FastaRecord();
            cur.id = first_piece(std::string(lp, ln), ' ').substr(1);
            cur.seq.reserve(reserve_hint);
            open = true;
        } else {
            open = true;
            if (strip_cr && std::memchr(lp, '\r', ln)) cur.seq += first_piece(std::string(lp, ln), '\r');
            else cur.seq.append(lp, ln);
        }
    }
    if (open) out->push_back(std::move(cur));
}

size_t g_reader_parallel_bytes = size_t(8) << 20;  // files at least this large are parsed by several threads

// FASTA reader of the MSA branch (src/panman.cpp:1288-1325). `strip_cr`: the MSA branch cuts lines and ids at '\r',
// the low-memory branch (:1479-1501, readFastaInBatch :677-724) does not. The reference's rules, kept record by record:
// a record without sequence is dropped; the first stored record fixes the length every other one must have; every
// record but the LAST is stored under its id cut at '\r' (MSA branch), the last keeps its id as is (:1316-1325); a
// later record with the same id replaces the earlier one. Large files are cut at header lines and the pieces parsed in
// parallel; the records are then stored in file order, so the result does not depend on the number of threads.
std::string read_msa(const char* text, size_t len, bool strip_cr, std::map<std::string, std::string>* seqs, size_t* line_length) {
    std::vector<std::vector<FastaRecord>> pieces;
    const unsigned hw = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    if (len < g_reader_parallel_bytes || hw == 1) {
        pieces.resize(1);
        parse_fasta_piece(text, 0, len, strip_cr, 0, &pieces[0]);
    } else {
        // header lines: '>' at the start of the file or right after a newline
        std::vector<std::vector<size_t>> found(hw);
        {
            std::vector<std::thread> th;
            for (unsigned k = 0; k < hw; k++)
                th.emplace_back([&, k]() {
                    const size_t a = len * k / hw, b = len * (k + 1) / hw;
                    for (size_t i = a; i < b;) {
                        const char* q = static_cast<const char*>(std::memchr(text + i, '>', b - i));
                        if (!q) break;
                        const size_t at = size_t(q - text);
                        if (at == 0 || text[at - 1] == '\n') found[k].push_back(at);
                        i = at + 1;
                    }
                });
            for (auto& t : th) t.join();
        }
        std::vector<size_t> headers;
        for (auto& f : found) headers.insert(headers.end(), f.begin(), f.end());
        // cut points: piece k starts at the first header at or after len * k / hw (piece 0 at the start of the file)
        std::vector<size_t> cuts{0};
        for (unsigned k = 1; k < hw; k++) {
            auto it = std::lower_bound(headers.begin(), headers.end(), len * k / hw);
            if (it != headers.end() && *it > cuts.back()) cuts.push_back(*it);
        }
        cuts.push_back(len);
        const size_t hint = headers.size() > 1 ? (len / headers.size()) : 0;
        pieces.resize(cuts.size() - 1);
        std::vector<std::thread> th;
        for (size_t k = 0; k + 1 < cuts.size(); k++)
            th.emplace_back([&, k]() { parse_fasta_piece(text, cuts[k], cuts[k + 1], strip_cr, hint, &pieces[k]); });
        for (auto& t : th) t.join();
    }
    // the last record of the file, if it has a sequence, is the one the reference stores after its loop
    FastaRecord* last = nullptr;
    for (auto it = pieces.rbegin(); it != pieces.rend() && !last; ++it)
        if (!it->empty()) last = &it->back();
    size_t ll = 0;
    for (auto& piece : pieces)
        for (FastaRecord& r : piece) {
            if (r.seq.empty()) continue;
            if (ll == 0) ll = r.seq.size();
            else if (ll != r.seq.size()) return "sequence lengths don't match: " + r.id;
            const bool is_last = &r == last;
            (*seqs)[(strip_cr && !is_last) ? first_piece(r.id, '\r') : r.id] = std::move(r.seq);
        }
    *line_length = ll;
    return "";
}

}  // namespace

pmh_build::~pmh_build() { pin_release(codes4, codes_cached); }

namespace {
// the lists of the pass just run on b->tree (pmb_result) and their run-merge (pmb_merge_runs) -> the build's NucMut fields
void store_lists(pmh_build* b, const pmb_result& res, const pmb_nucmut_result& mr) {
    const int32_t N = b->tree.t.n_nodes();
    b->tuple_off.assign(res.node_offsets, res.node_offsets + N + 1);
    b->tuple_pos.assign(res.pos, res.pos + res.n_mut);
    b->tuple_tc.assign(res.type_code, res.type_code + res.n_mut);
    b->nuc.assign(size_t(N), {});
    for (int32_t v = 0; v < N; v++) {
        const int64_t a = mr.node_offsets[v], z = mr.node_offsets[v + 1];
        b->nuc[v].resize(size_t(z - a));
        for (int64_t k = a; k < z; k++) {
            pmh_nucmut& m = b->nuc[v][size_t(k - a)];
            m.nucPosition = mr.nuc_position[k];
            m.nucGapPosition = -1;
            m.primaryBlockId = 0;
            m.secondaryBlockId = -1;
            m.mutInfo = mr.mut_info[k];
            m.nucs = mr.nucs[k];
        }
    }
}
}  // namespace

extern "C" {

static pmh_tree* tree_from_newick_impl(const char* newick, char* err, size_t err_len) {
    if (!newick) { set_err(err, err_len, "null newick"); return nullptr; }
    pmh_tree* t = new pmh_tree();
    std::string e = pmh::parse_newick(newick, &t->t);
    if (!e.empty()) {
        set_err(err, err_len, e);
        delete t;
        return nullptr;
    }
    return t;
}
void pmh_tree_free(pmh_tree* t) { delete t; }
int32_t pmh_tree_n_nodes(const pmh_tree* t) { return t->t.n_nodes(); }
int32_t pmh_tree_n_leaves(const pmh_tree* t) { return t->t.n_leaves; }
int32_t pmh_tree_root(const pmh_tree* t) { return t->t.root; }
const char* pmh_tree_name(const pmh_tree* t, int32_t v) { return t->t.names[v].c_str(); }
const int32_t* pmh_tree_parent(const pmh_tree* t) { return t->t.parent.data(); }
const int32_t* pmh_tree_child_offsets(const pmh_tree* t) { return t->t.child_off.data(); }
const int32_t* pmh_tree_child_index(const pmh_tree* t) { return t->t.child_idx.data(); }
const int32_t* pmh_tree_leaf_row(const pmh_tree* t) { return t->t.leaf_row.data(); }
int pmh_tree_has_polytomy(const pmh_tree* t) { return t->t.has_polytomy() ? 1 : 0; }

static pmh_build* msa_prepare_impl(const char* fasta, size_t fasta_len, const char* newick, const char* reference_c, int low_mem_mode,
                           char* err, size_t err_len) {
    if (!fasta || !newick) { set_err(err, err_len, "null argument"); return nullptr; }
    const std::string reference = reference_c ? reference_c : "";
    pmh_build* b = new pmh_build();
    auto fail = [&](const std::string& m) -> pmh_build* {
        set_err(err, err_len, m);
        delete b;
        return nullptr;
    };
    auto t0 = Clock::now();
    {   // std::getline(secondFin, newickString) : first line only (src/panman.cpp:1277, 1470)
        std::string nw(newick);
        size_t nl = nw.find('\n');
        if (nl != std::string::npos) nw.resize(nl);
        std::string e = pmh::parse_newick(nw, &b->tree.t);
        if (!e.empty()) return fail(e);
    }
    const pmh::HostTree& T = b->tree.t;
    std::map<std::string, std::string> seqs;  // std::map: id order decides the consensus (src/panman.cpp:1280)
    size_t line_length = 0;
    std::string e = read_msa(fasta, fasta_len, /*strip_cr=*/!low_mem_mode, &seqs, &line_length);
    if (!e.empty()) return fail(e);
    std::vector<const std::string*> ordered;
    for (auto& u : seqs) ordered.push_back(&u.second);

    std::string& cons = b->consensus;
    const std::string* ref_seq = nullptr;
    if (!reference.empty()) {
        auto it = seqs.find(reference);
        if (it != seqs.end()) ref_seq = &it->second;
    }
    if (!low_mem_mode) {
        if (!reference.empty()) {
            // consensusSeq = sequenceIdsToSequences[reference] (:1333-1334); an unknown id yields an empty consensus
            cons = ref_seq ? *ref_seq : std::string();
        } else {
            // first non-gap character in map order; all-gap columns are removed from every sequence (:1336-1361)
            cons.assign(line_length, 0);
            std::vector<char> keep(line_length, 0);
            for (size_t i = 0; i < line_length; i++)
                for (const std::string* s : ordered)
                    if ((*s)[i] != '-') { cons[i] = (*s)[i]; keep[i] = 1; break; }
            size_t kept = size_t(std::count(keep.begin(), keep.end(), 1));
            if (kept != line_length) {
                for (auto& u : seqs) {
                    std::string f;
                    f.reserve(kept);
                    for (size_t i = 0; i < u.second.size(); i++)
                        if (keep[i]) f += u.second[i];
                    u.second.swap(f);
                }
                // the reference keeps consensusSeq at full length with '\0' at the dropped positions but then iterates
                // i < consensusSeq.size() over the SHORTENED sequences; positions line up only when nothing was dropped.
                // We follow the intent that also matches every later use (blocks[0] = consensus of kept columns).
                std::string f;
                for (size_t i = 0; i < line_length; i++)
                    if (keep[i]) f += cons[i];
                cons.swap(f);
            }
        }
    } else {
        // low-memory branch: consensus per batch (:1527-1557); batches only bound memory, columns are independent
        cons.assign(line_length, 0);
        if (!reference.empty() && !ref_seq) return fail("Reference not found in the sequence");  // exit(0) at :1592-1595
        for (size_t i = 0; i < line_length; i++) {
            if (ref_seq && (*ref_seq)[i] != '-') { cons[i] = (*ref_seq)[i]; continue; }
            bool found = false;
            for (const std::string* s : ordered)
                if ((*s)[i] != '-') { cons[i] = (*s)[i]; found = true; break; }
            if (!found && !ref_seq) return fail("all-gap column without --reference (the reference exits here)");  // :1548-1551
        }
    }
    const int64_t n_cols = int64_t(cons.size());
    b->low_mem_mode = low_mem_mode;
    b->n_cols = n_cols;
    b->seconds[0] = since(t0);
    b->nuc.assign(T.n_nodes(), {});
    b->tuple_off.assign(T.n_nodes() + 1, 0);
    if (n_cols == 0) return b;

    // ---- pack: leaf rows (4-bit codes, two columns per byte) in tree leaf order; leaves without a sequence are absent
    t0 = Clock::now();
    const int64_t stride = ((n_cols + 1) / 2 + 15) / 16 * 16;
    const size_t codes_bytes = size_t(T.n_leaves) * size_t(stride);
    b->stride = stride;
    b->codes4 = pin_acquire(codes_bytes, &b->codes_cached);
    if (!b->codes4) b->codes_pageable.resize(codes_bytes);
    uint8_t* const codes4 = b->codes4 ? b->codes4 : b->codes_pageable.data();  // rows of absent leaves are never read (presence mask)
    std::vector<uint8_t>& present = b->present;
    present.assign(T.n_leaves, 0);
    std::vector<std::pair<int32_t, const std::string*>> rows;
    for (int32_t v = 0; v < T.n_nodes(); v++) {
        if (T.leaf_row[v] < 0) continue;
        auto it = seqs.find(T.names[v]);
        if (it == seqs.end()) continue;
        present[T.leaf_row[v]] = 1;
        rows.emplace_back(T.leaf_row[v], &it->second);
    }
    {
        unsigned nt = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
        std::vector<std::thread> th;
        for (unsigned k = 0; k < nt; k++)
            th.emplace_back([&, k]() {
                for (size_t r = k; r < rows.size(); r += nt) {
                    const unsigned char* s = reinterpret_cast<const unsigned char*>(rows[r].second->data());
                    uint8_t* d = codes4 + size_t(rows[r].first) * size_t(stride);
                    int64_t c = 0;
                    for (; c + 1 < n_cols; c += 2) d[c >> 1] = uint8_t(kCode.t[s[c]] | (kCode.t[s[c + 1]] << 4));
                    if (c < n_cols) d[c >> 1] = kCode.t[s[c]];
                }
            });
        for (auto& x : th) x.join();
    }
    std::vector<uint8_t>& parent_code = b->parent_code;
    parent_code.resize(n_cols);
    for (int64_t i = 0; i < n_cols; i++) parent_code[i] = kCode.t[(unsigned char)cons[i]];
    if (ref_seq) {  // defaultState of the low-memory branch (:1583-1604) / refState of the MSA branch (:1419-1420)
        b->per_col.resize(n_cols);
        for (int64_t i = 0; i < n_cols; i++) b->per_col[i] = int8_t(kCode.t[(unsigned char)(*ref_seq)[i]]);
    }
    b->seconds[1] = since(t0);
    return b;
}

// one device (ctx) or the GPUs of a box (grp): the same flow on either engine
static int msa_run_impl(pmb_ctx* ctx, pmb_group* grp, pmh_build* b, char* err, size_t err_len) {
    if ((!ctx && !grp) || !b) { set_err(err, err_len, "null argument"); return PMB_ERR_INVALID; }
    auto engine_error = [&]() { return std::string(grp ? pmb_group_last_error(grp) : pmb_last_error(ctx)); };
    auto fail = [&](const std::string& m) -> int {
        set_err(err, err_len, m);
        return PMB_ERR_INVALID;
    };
    const pmh::HostTree& T = b->tree.t;
    const int64_t n_cols = b->n_cols, stride = b->stride;
    if (n_cols == 0) {
        b->ran = true;
        return PMB_OK;
    }
    const uint8_t* codes4 = b->codes4 ? b->codes4 : b->codes_pageable.data();
    if (!codes4 || b->present.empty()) return fail("the batch was already consumed by an earlier pmh_msa_run");
    const std::vector<uint8_t>& present = b->present;
    const std::vector<uint8_t>& parent_code = b->parent_code;
    const int low_mem_mode = b->low_mem_mode;
    const int8_t* root_override = (!b->per_col.empty() && low_mem_mode) ? b->per_col.data() : nullptr;
    const int8_t* fwd_root_ref = (!b->per_col.empty() && !low_mem_mode) ? b->per_col.data() : nullptr;

    // ---- the passes
    auto t0 = Clock::now();
    int rc = grp ? pmb_group_set_tree(grp, T.n_nodes(), T.root, T.child_off.data(), T.child_idx.data(), T.leaf_row.data())
                 : pmb_set_tree(ctx, T.n_nodes(), T.root, T.child_off.data(), T.child_idx.data(), T.leaf_row.data());
    if (rc) return fail(std::string("pmb_set_tree: ") + engine_error());
    bool all_present = std::all_of(present.begin(), present.end(), [](uint8_t x) { return x != 0; });
    pmb_result res;
    const int algo = low_mem_mode ? PMB_ALGO_SANKOFF : PMB_ALGO_FITCH;
    rc = grp ? pmb_group_run_nuc(grp, algo, n_cols, T.n_leaves, codes4, stride, all_present ? nullptr : present.data(), parent_code.data(),
                                 root_override, fwd_root_ref, 0, &res)
             : pmb_run_nuc(ctx, algo, n_cols, T.n_leaves, codes4, stride, all_present ? nullptr : present.data(), parent_code.data(),
                           root_override, fwd_root_ref, 0, 0, &res);
    if (rc) return fail(std::string("pmb_run_nuc: ") + engine_error());
    b->seconds[2] = since(t0);
    pin_release(b->codes4, b->codes_cached);  // uploaded: the page-locked buffer can serve the next build
    b->codes4 = nullptr;
    b->codes_pageable = std::vector<uint8_t>();

    // ---- lists are already per node in ascending position (= std::sort of the tuples, :1447); merge runs
    t0 = Clock::now();
    // greedy <= 6 run-merge on the device (pmb_merge_runs; src/panman.cpp:1445-1466, NucMut ctor src/panman.hpp:109-151)
    pmb_nucmut_result mr;
    rc = grp ? pmb_group_merge_runs(grp, /*to_host*/1, &mr) : pmb_merge_runs(ctx, /*source*/0, /*to_host*/1, &mr);
    if (rc) return fail(std::string("pmb_merge_runs: ") + engine_error());
    store_lists(b, res, mr);
    b->ran = true;
    b->seconds[3] = since(t0);
    return PMB_OK;
}

// Tree::reroot (reference src/reroot.cpp:4-261) of an MSA-built PanMAT: the tree is transformed (pmh::reroot_tree), every
// leaf's sequence is rebuilt on the device from the build's Node::nucMutation (pmb_upload_replay: only the pieces cross the
// link), and every column is inferred again by Fitch on the new tree with the root forced to the tip's own code
// (src/reroot.cpp:134-224; also for a --low-mem-mode build), then run-merged (:226-261, the MSA form for one block).
static int msa_reroot_impl(pmb_ctx* ctx, pmh_build* b, const char* leaf_name, char* err, size_t err_len) {
    if (!ctx || !b || !leaf_name) { set_err(err, err_len, "null argument"); return PMB_ERR_INVALID; }
    auto fail = [&](int rc, const std::string& m) -> int {
        set_err(err, err_len, m);
        return rc;
    };
    const pmh::HostTree& OT = b->tree.t;  // the tree the lists were built on
    const int32_t tip = pmh::find_node(OT, leaf_name);
    if (tip < 0) return fail(PMB_ERR_INVALID, std::string("Sequence with name ") + leaf_name + " not found!");  // src/reroot.cpp:5-8
    if (!b->ran) return fail(PMB_ERR_NO_INPUT, "reroot works on a built PanMAT: call pmh_msa_run first");
    pmh::HostTree nt;
    const std::string e = pmh::reroot_tree(OT, tip, &nt);
    if (!e.empty()) return fail(PMB_ERR_INVALID, e);
    if (b->n_cols == 0) {
        b->tree.t = std::move(nt);
        b->nuc.assign(size_t(b->tree.t.n_nodes()), {});
        b->tuple_off.assign(size_t(b->tree.t.n_nodes()) + 1, 0);
        return PMB_OK;
    }
    auto t0 = Clock::now();
    const int32_t N = OT.n_nodes();
    std::vector<int64_t> piece_off(size_t(N) + 1, 0);
    for (int32_t v = 0; v < N; v++) piece_off[size_t(v) + 1] = piece_off[size_t(v)] + int64_t(b->nuc[size_t(v)].size());
    std::vector<int32_t> pos(static_cast<size_t>(piece_off[size_t(N)]));
    std::vector<uint8_t> info(pos.size());
    std::vector<uint32_t> nucs(pos.size());
    for (int32_t v = 0; v < N; v++)
        for (size_t k = 0; k < b->nuc[size_t(v)].size(); k++) {
            const pmh_nucmut& m = b->nuc[size_t(v)][k];
            const size_t i = size_t(piece_off[size_t(v)]) + k;
            pos[i] = m.nucPosition;
            info[i] = m.mutInfo;
            nucs[i] = m.nucs;
        }
    int rc = pmb_set_tree(ctx, nt.n_nodes(), nt.root, nt.child_off.data(), nt.child_idx.data(), nt.leaf_row.data());
    if (rc) return fail(rc, std::string("pmb_set_tree: ") + pmb_last_error(ctx));
    rc = pmb_upload_replay(ctx, N, OT.root, OT.child_off.data(), OT.child_idx.data(), OT.leaf_row.data(), piece_off.data(), pos.data(),
                           info.data(), nucs.data(), b->n_cols, b->parent_code.data(), OT.leaf_row[tip]);
    if (rc) return fail(rc, std::string("pmb_upload_replay: ") + pmb_last_error(ctx));
    rc = pmb_run_resident(ctx, PMB_ALGO_FITCH, 0);
    pmb_result res;
    if (!rc) rc = pmb_download(ctx, &res);
    if (rc) return fail(rc, std::string("pmb_run_resident: ") + pmb_last_error(ctx));
    b->seconds[2] = since(t0);
    t0 = Clock::now();
    pmb_nucmut_result mr;
    rc = pmb_merge_runs(ctx, /*source*/0, /*to_host*/1, &mr);
    if (rc) return fail(rc, std::string("pmb_merge_runs: ") + pmb_last_error(ctx));
    b->tree.t = std::move(nt);
    store_lists(b, res, mr);
    b->seconds[3] = since(t0);
    return PMB_OK;
}

pmh_build* pmh_build_from_msa(pmb_ctx* ctx, const char* fasta, size_t fasta_len, const char* newick, const char* reference,
                              int low_mem_mode, char* err, size_t err_len) {
    if (!ctx) { set_err(err, err_len, "null argument"); return nullptr; }
    pmh_build* b = pmh_msa_prepare(fasta, fasta_len, newick, reference, low_mem_mode, err, err_len);
    if (!b) return nullptr;
    if (pmh_msa_run(ctx, b, err, err_len) != PMB_OK) {
        delete b;
        return nullptr;
    }
    return b;
}

// The C ABI never lets an exception out (a bad input file must come back as an error, not abort the host process).
pmh_tree* pmh_tree_from_newick(const char* newick, char* err, size_t err_len) {
    try {
        return tree_from_newick_impl(newick, err, err_len);
    } catch (const std::exception& ex) {
        set_err(err, err_len, std::string("Newick: ") + ex.what());
        return nullptr;
    }
}
pmh_build* pmh_msa_prepare(const char* fasta, size_t fasta_len, const char* newick, const char* reference, int low_mem_mode, char* err,
                           size_t err_len) {
    try {
        return msa_prepare_impl(fasta, fasta_len, newick, reference, low_mem_mode, err, err_len);
    } catch (const std::exception& ex) {
        set_err(err, err_len, std::string("MSA input: ") + ex.what());
        return nullptr;
    }
}
int pmh_msa_run_group(pmb_group* group, pmh_build* b, char* err, size_t err_len) {
    try {
        return msa_run_impl(nullptr, group, b, err, err_len);
    } catch (const std::bad_alloc&) {
        set_err(err, err_len, "out of host memory");
        return PMB_ERR_OOM;
    } catch (const std::exception& ex) {
        set_err(err, err_len, std::string("pmh_msa_run_group: ") + ex.what());
        return PMB_ERR_INVALID;
    }
}
int pmh_msa_run(pmb_ctx* ctx, pmh_build* b, char* err, size_t err_len) {
    try {
        return msa_run_impl(ctx, nullptr, b, err, err_len);
    } catch (const std::bad_alloc&) {
        set_err(err, err_len, "out of host memory");
        return PMB_ERR_OOM;
    } catch (const std::exception& ex) {
        set_err(err, err_len, std::string("pmh_msa_run: ") + ex.what());
        return PMB_ERR_INVALID;
    }
}
int pmh_msa_reroot(pmb_ctx* ctx, pmh_build* b, const char* leaf_name, char* err, size_t err_len) {
    try {
        return msa_reroot_impl(ctx, b, leaf_name, err, err_len);
    } catch (const std::bad_alloc&) {
        set_err(err, err_len, "out of host memory");
        return PMB_ERR_OOM;
    } catch (const std::exception& ex) {
        set_err(err, err_len, std::string("pmh_msa_reroot: ") + ex.what());
        return PMB_ERR_INVALID;
    }
}
void pmh_build_free(pmh_build* b) { delete b; }
void pmh_set_reader_parallel_bytes(int64_t bytes) { g_reader_parallel_bytes = bytes < 0 ? 0 : size_t(bytes); }
int64_t pmh_build_n_cols(const pmh_build* b) { return b->n_cols; }
const uint8_t* pmh_build_codes4(const pmh_build* b, int64_t* row_stride) {
    if (row_stride) *row_stride = b->stride;
    return b->codes4 ? b->codes4 : (b->codes_pageable.empty() ? nullptr : b->codes_pageable.data());
}
const uint8_t* pmh_build_present(const pmh_build* b) { return b->present.data(); }
const uint8_t* pmh_build_parent_code(const pmh_build* b) { return b->parent_code.data(); }
const int8_t* pmh_build_root_override(const pmh_build* b) { return (!b->per_col.empty() && b->low_mem_mode) ? b->per_col.data() : nullptr; }
const int8_t* pmh_build_fwd_root_ref(const pmh_build* b) { return (!b->per_col.empty() && !b->low_mem_mode) ? b->per_col.data() : nullptr; }
const pmh_tree* pmh_build_tree(const pmh_build* b) { return &b->tree; }
const char* pmh_build_consensus(const pmh_build* b, int64_t* len) {
    if (len) *len = int64_t(b->consensus.size());
    return b->consensus.data();
}
int64_t pmh_build_n_nucmut(const pmh_build* b, int32_t v) { return int64_t(b->nuc[v].size()); }
const pmh_nucmut* pmh_build_nucmut(const pmh_build* b, int32_t v) { return b->nuc[v].data(); }
int64_t pmh_build_wire(const pmh_build* b, int32_t node, const pmh_wire_mutation** mutations, const pmh_wire_nuc** nucs) {
    if (!b || node < 0 || node >= int32_t(b->nuc.size())) return -1;
    try {
        std::vector<pmh_blockmut> blk;
        if (node == b->tree.t.root) blk.push_back(pmh_blockmut{0, -1, 1, 0});  // root->blockMutation.emplace_back(0, (BI, false)), :1439-1440
        pmh::build_wire(b->nuc[size_t(node)], blk, &b->wire_muts, &b->wire_nucs);
    } catch (const std::exception&) {
        return -1;
    }
    if (mutations) *mutations = b->wire_muts.data();
    if (nucs) *nucs = b->wire_nucs.data();
    return int64_t(b->wire_muts.size());
}
int64_t pmh_build_n_tuples(const pmh_build* b) { return int64_t(b->tuple_pos.size()); }
const int64_t* pmh_build_tuple_offsets(const pmh_build* b) { return b->tuple_off.data(); }
const int32_t* pmh_build_tuple_pos(const pmh_build* b) { return b->tuple_pos.data(); }
const uint8_t* pmh_build_tuple_type_code(const pmh_build* b) { return b->tuple_tc.data(); }
const double* pmh_build_seconds(const pmh_build* b) { return b->seconds; }

}  // extern "C"
