// psb_internal.h -- declarations shared by the host side of libparasail_b200.so.
#pragma once
#include <cstdint>
#include <map>
#include <functional>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/parasail_b200.h"

namespace psb {

// ---- function-name grammar [REF src/aligner/mod.rs:289-331] --------------------------------
struct FnConfig {
    int mode = 0;  // 0 nw, 1 sg, 2 sw (kern_gotoh32.cuh MODE_*)
    int s1_beg = 0, s1_end = 0, s2_beg = 0, s2_end = 0;
    bool trace = false, stats = false, table = false, rowcol = false;
    int strategy = 0;  // 0 striped, 1 scan, 2 diag: echoed in the result flags only
    bool profile = false;
    int width = 0;  // 8, 16, 32, 64, or 0 for "sat"
    int band = 0;   // parasail_nw_banded only: half-width of the diagonal band (0 = full table)
    int flag() const;
};
// true iff `name` (with or without "parasail_") is a function upstream parasail defines
bool parse_fn_name(const char *name, FnConfig *cfg);
int encode_fn(const FnConfig &c);       // dense id for the thunk tables
FnConfig decode_fn(int id);
int fn_id_count();

void set_error(const std::string &msg);

// ---- matrices ------------------------------------------------------------------------------
// value-type snapshot of a parasail_matrix_t, safe to keep after the caller frees the original
struct HostMatrix {
    std::vector<int> table;   // length x size
    uint8_t mapper[256];
    int size = 0, length = 0, type = 0, max = 0, min = 0;
    std::vector<uint8_t> query;  // pssm: the query it was converted from (may be empty)
    explicit HostMatrix(const parasail_matrix_t *m);
    HostMatrix() = default;
};

// ---- results -------------------------------------------------------------------------------
// The flag-byte / table block of one pair traced with K rows per lane (gotoh32_kernel) is [strip][step][lane][K]:
// strips of 32 * K rows, rlen + 31 steps of a strip (lane l reaches column j at step j + l), one byte (or int) per
// row of a lane.  The byte index of cell (i, j):
inline size_t trace_cell_index(int K, int rlen, int i, int j) {
    const int strip = i / (32 * K), rem = i % (32 * K), lane = rem / K, k = rem % K;
    return (((size_t)strip * (rlen + 31) + (j + lane)) * 32 + lane) * K + k;
}
// and its size in cells (not rounded)
inline long long trace_block_cells(int K, long long qlen, long long rlen) {
    return ((qlen + 32 * K - 1) / (32 * K)) * (rlen + 31) * 32 * K;
}
// The flag-byte block of one pair on the band kernel (band32_kernel, band of W offsets starting at diagonal lo =
// j - i of offset 0) is [row][offset]: the byte index of cell (i, j) of the band
inline size_t band_cell_index(int W, int lo, int i, int j) { return (size_t)i * W + (size_t)(j - i - lo); }
// and the block's size in cells
inline long long band_block_cells(long long qlen, int W) { return qlen * W; }
}  // namespace psb

struct psb_result_extra {
    int matches = 0, similar = 0, length = 0;
    int qlen = 0, rlen = 0;
    std::vector<int> score_table, matches_table, similar_table, length_table;
    std::vector<int> score_row, matches_row, similar_row, length_row;
    std::vector<int> score_col, matches_col, similar_col, length_col;
    std::vector<int8_t> trace;  // row-major TraceFlags bytes (qlen x rlen): built on the first parasail_result_get_trace_table
    // the device's trace block as it came back, [strip][step][lane][K] (gotoh32_kernel): every traced single-pair
    // call fetches it, only a caller that asks for the table pays for the row-major copy
    std::vector<uint8_t> trace_blob;
    int trace_K = 0;
    // a long pair's traced call runs on the whole-GPU wavefront kernel, whose records serve the walk (CIGAR,
    // traceback strings) but are not flag bytes: the block is then fetched by this closure -- the pair once
    // more, on the one-warp flag-byte kernel -- only when a caller asks for the table
    std::function<void(psb_result_extra *)> trace_lazy;
    std::once_flag trace_once;
    const int8_t *trace_table() {
        std::call_once(trace_once, [this]() {
            if (trace_blob.empty() && trace_lazy) { trace_lazy(this); trace_lazy = nullptr; }
            if (trace_blob.empty() || trace_K <= 0) return;
            const int K = trace_K, rows = 32 * K;
            trace.resize((size_t)qlen * rlen);
            // a row reads the block with a stride of one step record (32 * K bytes, psb::trace_cell_index).  Column
            // blocks of kBlock keep the ~kBlock + 31 records a strip's rows share in cache (a 20 kb x 20 kb table:
            // 400 MB through this loop)
            constexpr int kBlock = 64;
            for (int i0 = 0; i0 < qlen; i0 += rows)
                for (int j0 = 0; j0 < rlen; j0 += kBlock) {
                    const int j1 = j0 + kBlock < rlen ? j0 + kBlock : rlen, i1 = i0 + rows < qlen ? i0 + rows : qlen;
                    for (int i = i0; i < i1; ++i) {
                        const uint8_t *src = trace_blob.data() + psb::trace_cell_index(K, rlen, i, 0);
                        int8_t *dst = trace.data() + (size_t)i * rlen;
                        for (int j = j0; j < j1; ++j) dst[j] = (int8_t)src[(size_t)j * rows];
                    }
                }
            std::vector<uint8_t>().swap(trace_blob);
        });
        return trace.empty() ? nullptr : trace.data();
    }
    // _trace: the CIGAR the device walk produced (len<<4|op, forward order) and where it starts
    std::vector<uint32_t> cigar_ops;
    int beg_query = 0, beg_ref = 0;
};

struct parasail_profile {
    std::vector<uint8_t> query;  // raw residues (deep copy, SURVEY Appendix D Q2)
    psb::HostMatrix matrix;      // deep copy
    bool stats = false;
    int width = 0;
    // device-resident state, created on first use per device and then immutable
    mutable std::mutex mu;
    mutable std::map<int, void *> resident;
};

namespace psb {

// ---- engine (pairs.cu, ctx.cu, scan.cu) -------------------------------------------------------
struct PairsRequest {
    FnConfig cfg;
    const HostMatrix *matrix = nullptr;
    int open = 0, gap = 0;
    const uint8_t *q_cat = nullptr;
    const int64_t *q_off = nullptr;   // n+1 entries; shared_query: 2 entries
    bool shared_query = false;
    const uint8_t *r_cat = nullptr;
    const int64_t *r_off = nullptr;
    int64_t n = 0;
    // references out of a resident database instead of r_cat (psb_db_align): pair i's reference is subject r_ids[i]
    // (caller order), gathered from the packed store on the device; r_off still holds their offsets (from host_len).
    // The database's inverse permutation must exist before run_pairs is called.
    const psb_db_t *r_db = nullptr;
    const int *r_ids = nullptr;
    // single-pair API extras (n == 1): full tables / last row+col / row-major trace bytes
    psb_result_extra *extra = nullptr;
    // single-pair API, `_trace`: the flag-byte block itself is wanted (the lazy trace-table export), so even a long
    // pair stays on the one-warp kernel that writes it
    bool want_flag_bytes = false;
};
int run_pairs(const PairsRequest &req, psb_batch_t **out);
void free_batch(psb_batch_t *b);
void release_profile_resident(parasail_profile *p);

// SURVEY A.8: true when an explicit _8/_16 request cannot hold this pair's values; the one rule every
// entry point (single pair, psb_align_pairs, psb_scan, psb_scan_host) applies
bool saturates(const FnConfig &cfg, const HostMatrix &m, int score, int qlen, int rlen, int open, int gap);

// one pair through the batch path, wrapped as a parasail_result_t (never NULL)
parasail_result_t *align_one(const FnConfig &cfg, const HostMatrix &m, const uint8_t *q, int qlen, const uint8_t *r,
                             int rlen, int open, int gap);

}  // namespace psb
