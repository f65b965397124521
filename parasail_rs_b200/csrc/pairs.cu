// pairs.cu -- the pairs pass behind psb_align_pairs and psb_align_pairs_banded (SURVEY configs C1/C3/C4), the
// single-pair API and psb_db_align: a batch cut into passes, each pass planned, uploaded and launched in named stages
// over the packed 16-bit, 32-bit, wavefront and band kernels.  The kernels of kern_band32.cuh and kern_util.cuh are
// instantiated here; the launchers at the end serve the other files that use kern_util.cuh's kernels.
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <future>
#include <limits>
#include <mutex>
#include <string>
#include <vector>

#include "engine.h"
#include "kern_band32.cuh"
#include "kern_util.cuh"
#include "pairs16_host.h"

namespace psb {

struct PairChunk {
    int64_t lo, hi;  // pair range of the caller's batch handled by this pass
};

// what a pass hands back besides the slices of the batch's arrays it fills: the passes of a batch may run on two
// host threads at once (run_pairs_lanes), so nothing that depends on the other passes is written by a pass itself
struct PassOut {
    double cells = 0;
    DevMem d_csr;                     // device: this pass's CIGAR words (forward order, pairs lo..hi-1 back to back);
                                      // run_pairs copies every pass's words straight into the batch's one array
    std::vector<long long> csr_off;   // n+1 word offsets into d_csr
    float ms = 0.f;                   // timed region of the pass
    int launches = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // (multi-lane only) begin / end of the pass on the device
};

// ---- banded nw (kern_band32.cuh) ----------------------------------------------------------------------
// A pair of a banded request goes to the band kernel unless its band covers the whole table, boundary row and column
// included: then nothing is masked and the pair is an ordinary nw pair (packed 16-bit, general or wavefront kernels).
static bool band_covers(const BandGeom &b, int lq, int lr) { return b.lo <= -lq && b.hi >= lr; }
static bool band_kernel_pair(const FnConfig &cfg, int lq, int lr) {
    return cfg.band > 0 && cfg.mode == MODE_NW && !band_covers(band_geom(lq, lr, cfg.band), lq, lr);
}
// band-kernel variants: R = 2, 4, 8, 16 offsets per lane in registers, then the shared-memory form
static constexpr int kBandGroups = 5;
static int band_group(int W) {
    for (int g = 0; g < 4; ++g) if (W <= 64 << g) return g;
    return 4;
}
template <int R, bool SMEM> static const void *band32_fn_r(bool stats, bool trace) {
    if (trace) return (const void *)band32_kernel<R, SMEM, false, true>;
    if (stats) return (const void *)band32_kernel<R, SMEM, true, false>;
    return (const void *)band32_kernel<R, SMEM, false, false>;
}
static const void *band32_fn(int group, bool stats, bool trace) {
    switch (group) {
        case 0: return band32_fn_r<2, false>(stats, trace);
        case 1: return band32_fn_r<4, false>(stats, trace);
        case 2: return band32_fn_r<8, false>(stats, trace);
        case 3: return band32_fn_r<16, false>(stats, trace);
        case 4: return band32_fn_r<2, true>(stats, trace);
    }
    return nullptr;
}
// cells of the table inside the band: the whole table less the two triangles beyond the band's edges
static double band_cells(int lq, int lr, const BandGeom &b) {
    // sum over x = 0 .. n-1 of max(0, m - x)
    auto tri = [](long long m, long long n) -> double {
        if (m <= 0) return 0;
        if (m <= n) return (double)m * (m + 1) / 2;
        return (double)n * m - (double)n * (n - 1) / 2;
    };
    return (double)lq * lr - tri((long long)lr - b.hi - 1, lq) - tri((long long)lq + b.lo - 1, lr);
}

// hands out the passes of a batch in order, cutting each one when it is asked for (thread-safe: the lanes ask)
struct PassCutter {
    const PairsRequest &req;
    const bool mem_cut, p16_scheme;
    const int64_t budget, pass_res;
    std::mutex mu;
    int64_t lo = 0;
    std::deque<PairChunk> chunks;   // deques: the lanes hold pointers into them while later passes are appended
    std::deque<PassOut> pouts;
    PassCutter(const PairsRequest &r, bool mc, bool p16, int64_t bud, int64_t pr) : req(r), mem_cut(mc), p16_scheme(p16), budget(bud), pass_res(pr) {}
    int64_t res_upto(int64_t i) const { return (req.shared_query ? 0 : req.q_off[i] - req.q_off[0]) + (req.r_off[i] - req.r_off[0]); }
    bool next(PairChunk *ch, PassOut **po) {
        std::lock_guard<std::mutex> lk(mu);
        if (lo >= req.n) return false;
        int64_t hi;
        if (mem_cut) {
            int64_t bytes = 0;
            const int64_t res_lo = res_upto(lo);
            hi = lo;
            while (hi < req.n) {
                const int64_t lq = req.shared_query ? req.q_off[1] - req.q_off[0] : req.q_off[hi + 1] - req.q_off[hi];
                const int64_t lr = req.r_off[hi + 1] - req.r_off[hi];
                int64_t need;
                if (band_kernel_pair(req.cfg, (int)lq, (int)lr))   // one flag byte per offset and row
                    need = req.cfg.trace ? band_block_cells(lq, band_geom((int)lq, (int)lr, req.cfg.band).W) + 8 * (lq + lr) : 0;
                else if (p16_scheme && lq <= 512) need = (lr + 32) * (lq + 96) * 5 / 4 + 8 * (lq + lr);   // one byte of H per cell of the padded frame
                else if (req.cfg.trace) need = trace_block_cells(16, lq, lr) + 8 * (lq + lr);   // (16: the most rows per lane of any class)
                else need = 0;
                if (hi > lo && (bytes + need > budget || res_upto(hi + 1) - res_lo > pass_res)) break;
                bytes += need; ++hi;
            }
        } else if (pass_res == std::numeric_limits<int64_t>::max()) {
            hi = req.n;
        } else {
            // the last pair index whose residues still fit the pass (res_upto is monotone)
            int64_t a = lo + 1, z = req.n;
            while (a < z) { const int64_t mid = (a + z + 1) / 2; if (res_upto(mid) - res_upto(lo) <= pass_res) a = mid; else z = mid - 1; }
            hi = a;
            if (req.n - hi < (hi - lo) / 4) hi = req.n;   // no runt at the end
        }
        chunks.push_back({lo, hi});
        pouts.emplace_back();
        *ch = chunks.back();
        *po = &pouts.back();
        lo = hi;
        return true;
    }
};

// offset of pair i's CIGAR scratch (lq + lr + 2 words per pair, pair order) from the offset arrays on the device
__global__ void rev_off_kernel(const long long *q_off, const long long *r_off, int q_shared, long long qlen, long long q_base, long long r_base,
                               long long n, long long *out) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        out[i] = (q_shared ? i * qlen : q_off[i] - q_base) + (r_off[i] - r_base) + 2 * i;
}

// the packed 16-bit path (kern_pairs16.cuh) may take this request's scoring scheme: not switched off (PSB_NO_P16),
// within the static 16-bit bound, and no explicit 32/64-bit width asked for.  Each caller adds its own conditions.
static bool p16_allowed(const PairsRequest &req) {
    const HostMatrix &m = *req.matrix;
    return !std::getenv("PSB_NO_P16") && pairs16_scheme_ok(m.size, m.min, m.max, req.open, req.gap, m.type == PARASAIL_MATRIX_TYPE_PSSM) &&
           req.cfg.width != 32 && req.cfg.width != 64;
}

// which kernel each pair of a pass goes to (pair ids count from the pass's first pair)
struct PassPlan {
    const PairsRequest *req = nullptr;
    int64_t lo = 0, hi = 0, n = 0;
    int64_t q_lo = 0, q_hi = 0, r_lo = 0, r_hi = 0;   // the pass's residues in the caller's arrays
    bool pssm = false, q_two = false;                 // q_two: one query for every pair (offsets {0, qbytes})
    size_t qbytes = 0;
    bool want_table = false, banded = false, fine = false;
    ClassTable ct{};
    bool p16_on = false, p16_walk = false;
    std::vector<int> c16_of;                  // query length -> packed class (-1: none)
    std::vector<std::vector<int>> p16_ids;    // pairs of each packed 16-bit class
    long long n_p16 = 0;
    std::vector<std::vector<int>> cls;        // pairs of each 32-bit class
    std::vector<int> wave_ids;                // long pairs: spread over the whole GPU one at a time
    int band_k = 0;                           // banded nw: the band's half-width (0: no band kernel in this pass)
    std::vector<int> band_ids[kBandGroups];   // pairs of each band-kernel variant (band_group)
    int band_maxW[kBandGroups] = {};
    bool uniform = true;                      // every pair of the same lengths and class: no ordering needed
    int first_cls = -1;
    int max_lr_multistrip = 0;
    bool wide_stats = false;                  // the strip-boundary scratch carries the wide statistics word
    double cells = 0;
    int lq(int64_t i) const {
        return pssm ? req->matrix->length : (int)(req->shared_query ? q_hi - q_lo : req->q_off[lo + i + 1] - req->q_off[lo + i]);
    }
    int lr(int64_t i) const { return (int)(req->r_off[lo + i + 1] - req->r_off[lo + i]); }
    // longest reference first: a dynamic queue then ends on short pairs, and the pairs of a packed word (and the words
    // of a warp) are of similar size
    void longest_first(std::vector<int> &ids) const {
        std::stable_sort(ids.begin(), ids.end(), [this](int a, int b) { return lr(a) > lr(b); });
    }
};

static int plan_pass(const PairsRequest &req, int64_t lo, int64_t hi, PassPlan *plan) {
    PassPlan &P = *plan;
    const FnConfig &cfg = req.cfg;
    const HostMatrix &m = *req.matrix;
    P.req = &req; P.lo = lo; P.hi = hi; P.n = hi - lo;
    P.pssm = m.type == PARASAIL_MATRIX_TYPE_PSSM;
    P.q_lo = req.shared_query ? req.q_off[0] : req.q_off[lo];
    P.q_hi = req.shared_query ? req.q_off[1] : req.q_off[hi];
    P.r_lo = req.r_off[lo]; P.r_hi = req.r_off[hi];
    P.q_two = req.shared_query || P.pssm;
    P.qbytes = P.pssm ? (size_t)m.length : (size_t)(P.q_hi - P.q_lo);
    P.want_table = req.extra && (cfg.table || cfg.rowcol);
    // banded nw: every pair whose band does not cover the table goes to the band kernel.  The single-pair API
    // (parasail_nw_banded) keeps the masked general kernel for a band wider than kBandMaxW, and for every band under
    // PSB_NO_BAND_KERNEL (A/B tests)
    P.band_k = cfg.band > 0 && cfg.mode == MODE_NW ? cfg.band : 0;
    if (P.band_k && req.extra && P.n == 1) {
        const int lq0 = P.lq(0), lr0 = P.lr(0);
        const BandGeom b = band_geom(lq0, lr0, P.band_k);
        P.banded = (std::getenv("PSB_NO_BAND_KERNEL") || (!band_covers(b, lq0, lr0) && b.W > kBandMaxW)) && !cfg.stats && !cfg.trace &&
                   !P.want_table;
        if (P.banded) P.band_k = 0;
    }
    P.fine = gotoh32_profile_ok(m.size, m.min, m.max, req.open, P.pssm) && !P.want_table && !P.banded;
    P.ct = class_table(P.fine);
    P.cls.resize(kNumClass);
    // packed 16-bit path: pairs whose scoring scheme and lengths pass the static 16-bit bound; `_stats` results come
    // from the trace walk there.  Explicit 32/64-bit requests, table outputs and the single-pair trace-table export
    // stay on the 32-bit kernels.
    P.p16_walk = cfg.trace || cfg.stats;
    P.p16_on = p16_allowed(req) && !P.want_table && !P.banded && !(req.extra && cfg.trace) &&
               (!P.p16_walk || pairs16_trace_ok(m.min, m.max, req.open));
    P.p16_ids.resize(P.p16_on ? p16_num_classes() : 0);
    // Wide (32-lane) groups halve the profile bytes per warp: taken when the narrow class would leave fewer than 8
    // warps per SM (protein alphabets, queries beyond ~200 residues)
    P.c16_of.assign(513, -1);
    if (P.p16_on) {
        const char *ev = std::getenv("PSB_P16_WIDE");
        for (int lq = 1; lq <= 512; ++lq) {
            const int narrow = p16_pick_class(lq, false);
            bool wide = narrow >= 0 && 227 * 1024 / pairs16_warp_smem(p16_class(narrow).K, m.size + 1, cfg.mode == MODE_SW) < 8;
            if (ev) wide = std::atoi(ev) != 0;
            P.c16_of[lq] = p16_pick_class(lq, wide);
        }
    }
    size_t wave_avail = ~(size_t)0;   // device memory a traced wavefront launch may use (queried on the first long pair)
    int max_sum = 0, max_min = 0;
    long long first_cells = -1;
    int first_lq = -1, first_lr = -1;
    for (int64_t i = 0; i < P.n; ++i) {
        const int lq = P.lq(i), lr = P.lr(i);
        if (lq <= 0 || lr <= 0) { set_error("empty sequence in batch (pair " + std::to_string(lo + i) + ")"); return PSB_EINVAL; }
        if (first_lq < 0) { first_lq = lq; first_lr = lr; }
        else if (lq != first_lq || lr != first_lr) P.uniform = false;
        if (P.band_k) {
            const BandGeom b = band_geom(lq, lr, P.band_k);
            if (!band_covers(b, lq, lr)) {
                if (b.W > kBandMaxW) {
                    set_error("band of " + std::to_string(b.W) + " diagonals (pair " + std::to_string(lo + i) + ") is wider than the band kernel's " +
                              std::to_string(kBandMaxW));
                    return PSB_EUNSUPPORTED;
                }
                if (cfg.stats && (std::min(lq, lr) >= (1 << 21) || lq + lr >= (1 << 22))) {
                    set_error("pair " + std::to_string(lo + i) + " too long for the band kernel's statistics word");
                    return PSB_EUNSUPPORTED;
                }
                const int g = band_group(b.W);
                P.band_ids[g].push_back((int)i);
                P.band_maxW[g] = std::max(P.band_maxW[g], b.W);
                P.cells += band_cells(lq, lr, b);
                continue;
            }
        }
        if (P.p16_on && lq <= 512) {
            const int c16 = P.c16_of[lq];
            if (c16 >= 0 && pairs16_fits(p16_class(c16).G * p16_class(c16).K, lq, lr, m.max, m.min, req.open, req.gap, cfg.mode == MODE_SW)) {
                P.p16_ids[c16].push_back((int)i);
                ++P.n_p16;
                P.cells += (double)lq * lr;
                continue;
            }
        }
        const int cl = class_of_len(P.ct, lq);
        bool wave = lq >= kWaveMinLq && lr >= 64 && !P.pssm && !(req.extra && (cfg.table || cfg.rowcol || (cfg.trace && req.want_flag_bytes))) && !P.banded;
        if (wave && (cfg.stats || cfg.trace)) {
            // with traceback / statistics: the traced wavefront launch + walk32_kernel when its preconditions hold
            // and its 1.25 bytes per cell fit (the single-pair API's trace-table export needs the flag bytes of the
            // one-warp kernel: align_one fetches them with a second, want_flag_bytes call when the table is asked for)
            if (wave_avail == ~(size_t)0) wave_avail = device_mem_available();
            wave = wave_walk_ok(m, req.open, req.gap, cfg.mode == MODE_SW, lq, lr, wave_avail);
        }
        if (wave) { P.wave_ids.push_back((int)i); P.uniform = false; }
        else P.cls[cl].push_back((int)i);
        if (!wave && lq > 32 * P.ct.k[cl]) P.max_lr_multistrip = std::max(P.max_lr_multistrip, lr);
        max_sum = std::max(max_sum, lq + lr);
        max_min = std::max(max_min, std::min(lq, lr));
        const long long cells = (long long)lq * lr;
        if (P.first_cls < 0) { P.first_cls = cl; first_cells = cells; }
        else if (cl != P.first_cls || cells != first_cells) P.uniform = false;
        P.cells += (double)cells;
    }
    // the coarse family carries only the wide statistics word: the strip-boundary scratch is sized for it
    P.wide_stats = !(max_min < 1024 && max_sum < 4096) || !P.fine;
    return PSB_OK;
}

// the buffers of a pass that outlive a stage.  The driver owns them: device buffers go back to the pool on the stream
// when the pass returns (after its last synchronise), and the host vectors are the sources of queued copies.
struct PassBufs {
    DevMem d_q, d_r, d_qoff, d_roff, d_matrix, d_rids;
    DevMem d_out[6], d_counter, d_bnd;
    DevMem d_traceoff, d_tab[4], d_revoff, d_nops, d_beg[2];
    KeptMem d_trace{0}, d_rev{1};
    std::vector<long long> trace_off;   // pairs on the 32-bit kernels: offset of the pair's trace / table block
    long long trace_total = 0;
    Gotoh32Params p;                    // the pass's device pointers, shared by every launch
    DevMem d_items, d_toff16, d_slot16, d_ids16, d_mat8, d_cnt16;
    KeptMem d_trace16{2};
    std::vector<int> h_items, h_slot16, h_ids16;
    std::vector<long long> h_toff16;
    std::vector<int8_t> h_mat8 = std::vector<int8_t>(33 * 32);
    std::vector<int> cls_item0, cls_id0;   // first item / pair of each packed class in d_items / d_ids16
    std::vector<DevMem> d_orders = std::vector<DevMem>(kNumClass);
    DevMem d_csroff, d_scan_tmp;
    std::vector<DevMem> d_band_orders = std::vector<DevMem>(kBandGroups);
    DevMem d_band_cnt;
};

// upload residues + offsets (relative to this range) and the matrix; references out of a resident database: their ids
static int upload_pass(const PairsRequest &req, const PassPlan &P, PassBufs &B) {
    Ctx &c = g_ctx;
    const HostMatrix &m = *req.matrix;
    const int64_t n = P.n, lo = P.lo;
    PSB_TRY(B.d_q.alloc(P.qbytes, c.stream));
    PSB_TRY(B.d_r.alloc((size_t)(P.r_hi - P.r_lo), c.stream));
    // the offsets go up as the caller gave them (absolute): the device pointers are biased by the range's first
    // byte instead, so that base + off[pair] lands inside this pass's upload (no per-pair pass to make them relative)
    static_assert(sizeof(int64_t) == sizeof(long long), "offset arrays are uploaded as they are");
    const long long qoff2[2] = {0, (long long)P.qbytes};
    PSB_TRY(B.d_qoff.alloc((P.q_two ? 2 : (size_t)n + 1) * sizeof(long long), c.stream));
    PSB_TRY(B.d_roff.alloc(((size_t)n + 1) * sizeof(long long), c.stream));
    PSB_TRY(B.d_matrix.alloc(m.table.size() * sizeof(int), c.stream));
    if (P.pssm && m.query.size() == (size_t)m.length)
        PSB_CUDA(cudaMemcpyAsync(B.d_q.p, m.query.data(), P.qbytes, cudaMemcpyHostToDevice, c.stream));
    else if (P.pssm)
        PSB_CUDA(cudaMemsetAsync(B.d_q.p, 0xff, P.qbytes, c.stream));  // no query residues: nothing "matches"
    else
        PSB_CUDA(upload_h2d(B.d_q.p, req.q_cat + P.q_lo, P.qbytes, c.stream));
    if (req.r_db) {
        PSB_TRY(B.d_rids.alloc((size_t)n * sizeof(int), c.stream));
        PSB_CUDA(upload_h2d(B.d_rids.p, req.r_ids + lo, (size_t)n * sizeof(int), c.stream));
    } else {
        PSB_CUDA(upload_h2d(B.d_r.p, req.r_cat + P.r_lo, (size_t)(P.r_hi - P.r_lo), c.stream));
    }
    if (P.q_two) PSB_CUDA(cudaMemcpyAsync(B.d_qoff.p, qoff2, sizeof(qoff2), cudaMemcpyHostToDevice, c.stream));
    else PSB_CUDA(upload_h2d(B.d_qoff.p, req.q_off + lo, ((size_t)n + 1) * sizeof(long long), c.stream));
    PSB_CUDA(upload_h2d(B.d_roff.p, req.r_off + lo, ((size_t)n + 1) * sizeof(long long), c.stream));
    PSB_CUDA(cudaMemcpyAsync(B.d_matrix.p, m.table.data(), m.table.size() * sizeof(int), cudaMemcpyHostToDevice, c.stream));
    return PSB_OK;
}

// outputs, strip-boundary scratch, the trace / table blocks of the pairs on the 32-bit kernels and the CIGAR scratch
// of the device-side walks; fills the pass's Gotoh32Params
static int alloc_pass(const PairsRequest &req, const PassPlan &P, PassBufs &B) {
    Ctx &c = g_ctx;
    const FnConfig &cfg = req.cfg;
    const HostMatrix &m = *req.matrix;
    const int64_t n = P.n;
    const int nout = cfg.stats || P.want_table ? 6 : 3;
    for (int k = 0; k < nout; ++k) PSB_TRY(B.d_out[k].alloc((size_t)n * sizeof(int), c.stream));
    PSB_TRY(B.d_counter.alloc(sizeof(int) * (kNumClass + 1), c.stream));
    PSB_CUDA(cudaMemsetAsync(B.d_counter.p, 0, sizeof(int) * (kNumClass + 1), c.stream));
    const bool stats_kernel = cfg.stats || P.want_table;
    const int bnd_words_per_col = 2 + (stats_kernel ? 2 * ((P.wide_stats || P.want_table) ? 2 : 1) : 0);
    const long long bnd_stride = (long long)P.max_lr_multistrip * bnd_words_per_col;
    if (bnd_stride > 0) PSB_TRY(B.d_bnd.alloc((size_t)(bnd_stride * max_grid_warps(n)) * sizeof(int), c.stream));

    // CIGAR scratch: pair i owns lq + lr + 2 words, in pair order, so its offset has a closed form that the device
    // computes from the offset arrays it already holds (rev_off_kernel); only the trace blocks of pairs on the
    // 32-bit kernels (none in a typical batch) need a host pass
    const long long rev_total = (P.q_two ? (long long)n * (long long)P.qbytes : (long long)(P.q_hi - P.q_lo)) + (long long)(P.r_hi - P.r_lo) + 2 * (long long)n;
    bool any32 = false;
    for (int cl = 0; cl < kNumClass; ++cl) any32 = any32 || !P.cls[cl].empty();
    for (int g = 0; g < kBandGroups; ++g) any32 = any32 || !P.band_ids[g].empty();
    if ((cfg.trace || P.want_table) && any32) {
        B.trace_off.assign(n, 0);
        for (int cl = 0; cl < kNumClass; ++cl)
            for (int id : P.cls[cl]) {
                B.trace_off[id] = B.trace_total;
                B.trace_total += ((trace_block_cells(P.ct.k[cl], P.lq(id), P.lr(id)) + 15) / 16) * 16;
            }
        for (int g = 0; g < kBandGroups; ++g)
            for (int id : P.band_ids[g]) {
                B.trace_off[id] = B.trace_total;
                B.trace_total += ((band_block_cells(P.lq(id), band_geom(P.lq(id), P.lr(id), P.band_k).W) + 15) / 16) * 16;
            }
        PSB_TRY(B.d_traceoff.alloc((size_t)n * sizeof(long long), c.stream));
        PSB_CUDA(cudaMemcpyAsync(B.d_traceoff.p, B.trace_off.data(), (size_t)n * sizeof(long long), cudaMemcpyHostToDevice, c.stream));
        if (cfg.trace) PSB_TRY(B.d_trace.alloc((size_t)B.trace_total, c.stream));
        if (P.want_table) for (int k = 0; k < 4; ++k) PSB_TRY(B.d_tab[k].alloc((size_t)B.trace_total * sizeof(int), c.stream));
    }

    Gotoh32Params &p = B.p;
    std::memset(&p, 0, sizeof(p));
    p.q = B.d_q.as<uint8_t>() - (P.q_two ? 0 : P.q_lo); p.q_off = B.d_qoff.as<long long>();
    p.r = B.d_r.as<uint8_t>() - P.r_lo; p.r_off = B.d_roff.as<long long>();
    p.shared_query = P.q_two ? 1 : 0;
    p.matrix = B.d_matrix.as<int>(); p.size = m.size; p.is_pssm = P.pssm ? 1 : 0;
    p.open = req.open; p.gap = req.gap;
    p.mode = cfg.mode; p.s1_beg = cfg.s1_beg; p.s1_end = cfg.s1_end; p.s2_beg = cfg.s2_beg; p.s2_end = cfg.s2_end;
    p.score = B.d_out[0].as<int>(); p.end_query = B.d_out[1].as<int>(); p.end_ref = B.d_out[2].as<int>();
    p.matches = B.d_out[3].as<int>(); p.similar = B.d_out[4].as<int>(); p.length = B.d_out[5].as<int>();
    p.bnd = B.d_bnd.as<int>(); p.bnd_stride = bnd_stride;
    p.trace = B.d_trace.as<uint8_t>(); p.trace_off = B.d_traceoff.as<long long>();
    p.tabH = B.d_tab[0].as<int>(); p.tabM = B.d_tab[1].as<int>(); p.tabS = B.d_tab[2].as<int>(); p.tabL = B.d_tab[3].as<int>();
    p.tab_off = B.d_traceoff.as<long long>();
    if (P.banded) {
        // [REF src/aligner/mod.rs:457-489] band of half-width k around the main diagonal, widened by the
        // length difference so that the corner (Lq-1, Lr-1) stays inside
        const int d = P.lr(0) - P.lq(0);
        p.banded = 1; p.band_lo = -cfg.band + (d < 0 ? d : 0); p.band_hi = cfg.band + (d > 0 ? d : 0);
    }

    // CIGAR scratch of the device-side walks (every kernel family writes the same reversed run lists)
    if (cfg.trace) {
        PSB_TRY(B.d_rev.alloc((size_t)rev_total * sizeof(unsigned), c.stream));
        PSB_TRY(B.d_revoff.alloc((size_t)n * sizeof(long long), c.stream));
        rev_off_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)c.sms * 8), 256, 0, c.stream>>>(
            B.d_qoff.as<long long>(), B.d_roff.as<long long>(), P.q_two ? 1 : 0, (long long)P.qbytes, (long long)P.q_lo, (long long)P.r_lo,
            (long long)n, B.d_revoff.as<long long>());
        c.launches++;
        PSB_TRY(B.d_nops.alloc(((size_t)n + 1) * sizeof(int), c.stream));
        PSB_CUDA(cudaMemsetAsync(B.d_nops.p, 0, ((size_t)n + 1) * sizeof(int), c.stream));
        PSB_TRY(B.d_beg[0].alloc((size_t)n * sizeof(int), c.stream));
        PSB_TRY(B.d_beg[1].alloc((size_t)n * sizeof(int), c.stream));
    }
    return PSB_OK;
}

// packed 16-bit classes: two pairs per register, sorted by reference length so that the pairs of a word (and the
// words of a warp) are of similar size.  Builds and queues the items, their trace offsets and the byte matrix.
static int queue_items16(const PairsRequest &req, PassPlan &P, PassBufs &B) {
    Ctx &c = g_ctx;
    const HostMatrix &m = *req.matrix;
    const size_t nc16 = P.p16_ids.size();
    const bool top_free = free_ends(req.cfg).top;
    B.cls_item0.assign(nc16 + 1, 0);
    B.cls_id0.assign(nc16 + 1, 0);
    if (P.n_p16 == 0) return PSB_OK;
    B.h_items.reserve((size_t)P.n_p16 + 2 * nc16);
    B.h_ids16.reserve((size_t)P.n_p16);
    if (P.p16_walk) B.h_slot16.assign((size_t)P.n, 0);
    B.h_toff16.push_back(0);
    for (size_t c16 = 0; c16 < nc16; ++c16) {
        std::vector<int> &ids = P.p16_ids[c16];
        B.cls_item0[c16] = (int)(B.h_items.size() / 2);
        B.cls_id0[c16] = (int)B.h_ids16.size();
        if (ids.empty()) continue;
        const P16Class pc = p16_class((int)c16);
        if (!P.uniform) P.longest_first(ids);
        for (size_t t = 0; t < ids.size(); t += 2) {
            const int a = ids[t], bb = t + 1 < ids.size() ? ids[t + 1] : -1;
            const int item = (int)(B.h_items.size() / 2);
            B.h_items.push_back(a); B.h_items.push_back(bb);
            if (P.p16_walk) {
                const int lrb = bb >= 0 ? P.lr(bb) : 0;
                B.h_toff16.push_back(B.h_toff16.back() + pairs16_item_trace_words(pc.G, pc.K, std::max(P.lr(a), lrb)));
                B.h_slot16[a] = 2 * item;
                if (bb >= 0) B.h_slot16[bb] = 2 * item + 1;
            }
        }
        B.h_ids16.insert(B.h_ids16.end(), ids.begin(), ids.end());
    }
    B.cls_item0[nc16] = (int)(B.h_items.size() / 2);
    B.cls_id0[nc16] = (int)B.h_ids16.size();
    pairs16_build_mat8(m.table.data(), m.size, req.open, top_free, B.h_mat8.data());
    PSB_TRY(B.d_items.alloc(B.h_items.size() * sizeof(int), c.stream));
    PSB_TRY(B.d_mat8.alloc(B.h_mat8.size(), c.stream));
    PSB_TRY(B.d_cnt16.alloc(sizeof(int) * (nc16 + 1), c.stream));
    PSB_CUDA(cudaMemcpyAsync(B.d_items.p, B.h_items.data(), B.h_items.size() * sizeof(int), cudaMemcpyHostToDevice, c.stream));
    PSB_CUDA(cudaMemcpyAsync(B.d_mat8.p, B.h_mat8.data(), B.h_mat8.size(), cudaMemcpyHostToDevice, c.stream));
    PSB_CUDA(cudaMemsetAsync(B.d_cnt16.p, 0, sizeof(int) * (nc16 + 1), c.stream));
    if (P.p16_walk) {
        PSB_TRY(B.d_toff16.alloc(B.h_toff16.size() * sizeof(long long), c.stream));
        PSB_TRY(B.d_slot16.alloc(B.h_slot16.size() * sizeof(int), c.stream));
        PSB_TRY(B.d_ids16.alloc(B.h_ids16.size() * sizeof(int), c.stream));
        PSB_TRY(B.d_trace16.alloc((size_t)B.h_toff16.back() * sizeof(unsigned) + 64, c.stream));
        PSB_CUDA(cudaMemcpyAsync(B.d_toff16.p, B.h_toff16.data(), B.h_toff16.size() * sizeof(long long), cudaMemcpyHostToDevice, c.stream));
        PSB_CUDA(cudaMemcpyAsync(B.d_slot16.p, B.h_slot16.data(), B.h_slot16.size() * sizeof(int), cudaMemcpyHostToDevice, c.stream));
        PSB_CUDA(cudaMemcpyAsync(B.d_ids16.p, B.h_ids16.data(), B.h_ids16.size() * sizeof(int), cudaMemcpyHostToDevice, c.stream));
    }
    return PSB_OK;
}

// residues to matrix columns on the device; references out of a resident database are gathered from its packed
// store instead (already matrix codes, written at the same biased offsets an upload would have put them)
static void launch_map(const PairsRequest &req, const PassPlan &P, PassBufs &B) {
    Ctx &c = g_ctx;
    const HostMatrix &m = *req.matrix;
    MapParams mp;
    fill_lut(mp.lut, m.mapper);
    const int blocks = c.sms * 8;
    if (!(P.pssm && m.query.size() != (size_t)m.length)) {
        mp.data = B.d_q.as<uint8_t>(); mp.n = (long long)P.qbytes;
        map_residues_kernel<<<blocks, 256, 0, c.stream>>>(mp);
        c.launches++;
    }
    if (req.r_db) {
        UnpackParams u;
        u.words = req.r_db->d_words; u.word_off = req.r_db->d_word_off; u.ids = B.d_rids.as<int>(); u.inv_perm = req.r_db->d_inv_perm;
        u.out_off = B.d_roff.as<long long>(); u.out = B.d_r.as<uint8_t>() - P.r_lo; u.n = P.n; u.bits = req.r_db->bits;
        unpack_db_kernel<<<(unsigned)std::min<int64_t>((P.n + 7) / 8, blocks), 256, 0, c.stream>>>(u);
    } else {
        mp.data = B.d_r.as<uint8_t>(); mp.n = (long long)(P.r_hi - P.r_lo);
        map_residues_kernel<<<blocks, 256, 0, c.stream>>>(mp);
    }
    c.launches++;
}

// the packed classes' fill kernels, each followed by its walk when the request wants traceback or statistics
static int launch_pairs16(const PairsRequest &req, const PassPlan &P, PassBufs &B, PassTimeline &tl) {
    Ctx &c = g_ctx;
    const FnConfig &cfg = req.cfg;
    const HostMatrix &m = *req.matrix;
    const Gotoh32Params &p = B.p;
    const bool sw = cfg.mode == MODE_SW;
    if (P.n_p16 == 0) return PSB_OK;
    std::string err;
    for (int c16 = 0; c16 < (int)P.p16_ids.size(); ++c16) {
        const int nitems = B.cls_item0[c16 + 1] - B.cls_item0[c16];
        if (nitems == 0) continue;
        Pairs16Params pp;
        std::memset(&pp, 0, sizeof(pp));
        pp.q = p.q; pp.q_off = p.q_off; pp.r = p.r; pp.r_off = p.r_off; pp.shared_query = p.shared_query;
        pp.items = B.d_items.as<int>() + 2 * (size_t)B.cls_item0[c16]; pp.nitems = nitems;
        pp.mat8 = B.d_mat8.as<int8_t>(); pp.size = m.size; pp.open = req.open; pp.gap = req.gap;
        pp.mode = cfg.mode; pp.s1_beg = cfg.s1_beg; pp.s1_end = cfg.s1_end; pp.s2_beg = cfg.s2_beg; pp.s2_end = cfg.s2_end;
        pp.score = p.score; pp.end_query = p.end_query; pp.end_ref = p.end_ref;
        pp.trace = B.d_trace16.as<unsigned>(); pp.trace_off = P.p16_walk ? B.d_toff16.as<long long>() + B.cls_item0[c16] : nullptr;
        pp.counter = B.d_cnt16.as<int>() + c16;
        int wps = 0;
        tl.begin("pairs16 fill G" + std::to_string(p16_class(c16).G) + " K" + std::to_string(p16_class(c16).K) + " items " + std::to_string(nitems));
        const int rc16 = p16_launch(c16, sw, P.p16_walk, pp, c.sms, c.stream, &err, &wps);
        tl.end();
        if (tl.on) tl.marks.back().what += " warps/SM " + std::to_string(wps);
        if (rc16 != PSB_OK) { set_error(err); return rc16; }
        c.launches++;
        if (P.p16_walk) {
            Walk16Params w;
            std::memset(&w, 0, sizeof(w));
            w.q = p.q; w.q_off = p.q_off; w.r = p.r; w.r_off = p.r_off; w.shared_query = p.shared_query;
            w.pair_ids = B.d_ids16.as<int>() + B.cls_id0[c16]; w.pair_slot = B.d_slot16.as<int>(); w.n = B.cls_id0[c16 + 1] - B.cls_id0[c16];
            w.G = p16_class(c16).G; w.K = p16_class(c16).K;
            w.trace = B.d_trace16.as<unsigned>(); w.trace_off = B.d_toff16.as<long long>();
            w.matrix = p.matrix; w.size = m.size; w.open = req.open; w.gap = req.gap; w.is_sw = sw ? 1 : 0;
            const FreeEnds fe = free_ends(cfg);
            w.top_free = fe.top ? 1 : 0; w.left_free = fe.left ? 1 : 0;
            w.score = p.score; w.end_query = p.end_query; w.end_ref = p.end_ref;
            w.rev_ops = B.d_rev.as<unsigned>(); w.rev_off = B.d_revoff.as<long long>();
            w.nops = B.d_nops.as<int>(); w.beg_query = B.d_beg[0].as<int>(); w.beg_ref = B.d_beg[1].as<int>();
            w.matches = p.matches; w.similar = p.similar; w.length = p.length;
            tl.begin("walk16");
            const int rcw = p16_launch_walk(w, !cfg.trace, c.stream, &err);
            tl.end();
            if (rcw != PSB_OK) { set_error(err); return rcw; }
            c.launches++;
        }
    }
    return PSB_OK;
}

// one launch of the one-warp-per-pair kernel per 32-bit class, longest pairs first unless every pair is alike
static int launch_classes(const PairsRequest &req, PassPlan &P, PassBufs &B) {
    Ctx &c = g_ctx;
    const FnConfig &cfg = req.cfg;
    Gotoh32Params &p = B.p;
    for (int cl = 0; cl < kNumClass; ++cl) {
        std::vector<int> &ids = P.cls[cl];
        if (ids.empty()) continue;
        p.order = nullptr;
        if (!P.uniform) {
            P.longest_first(ids);
            PSB_TRY(B.d_orders[cl].alloc(ids.size() * sizeof(int), c.stream));
            PSB_CUDA(cudaMemcpyAsync(B.d_orders[cl].p, ids.data(), ids.size() * sizeof(int), cudaMemcpyHostToDevice, c.stream));
            p.order = B.d_orders[cl].as<int>();
        }
        p.n = (int)ids.size();
        p.counter = B.d_counter.as<int>() + cl;
        const Variant v = P.want_table ? V_TABLE : (cfg.trace ? V_TRACE : (cfg.stats ? (P.wide_stats ? V_STATS64 : V_STATS32) : V_SCORE));
        PSB_TRY(launch_gotoh32(P.ct.k[cl], v, p, p.n, P.fine));
    }
    return PSB_OK;
}

// the long pairs, one at a time over the whole GPU
static int launch_waves(const PairsRequest &req, const PassPlan &P, PassBufs &B, PassTimeline &tl) {
    const FnConfig &cfg = req.cfg;
    for (int id : P.wave_ids) {
        // (byte offsets relative to the biased p.q / p.r)
        const long long qb = req.shared_query ? 0 : req.q_off[P.lo + id], rb = req.r_off[P.lo + id];
        WaveWalk ww;
        ww.stats = !cfg.trace;
        ww.rev_ops = B.d_rev.as<unsigned>(); ww.rev_off = B.d_revoff.as<long long>();
        ww.nops = B.d_nops.as<int>(); ww.beg_query = B.d_beg[0].as<int>(); ww.beg_ref = B.d_beg[1].as<int>();
        PSB_TRY(launch_wave32(B.p, *req.matrix, qb, P.lq(id), rb, P.lr(id), id, (cfg.stats || cfg.trace) ? &ww : nullptr, tl));
    }
    return PSB_OK;
}

// the pairs of a banded request on the band kernel: one launch per variant, longest reference first
static int launch_band(const PairsRequest &req, PassPlan &P, PassBufs &B) {
    Ctx &c = g_ctx;
    const FnConfig &cfg = req.cfg;
    const Gotoh32Params &g = B.p;
    bool any = false;
    for (int gi = 0; gi < kBandGroups; ++gi) any = any || !P.band_ids[gi].empty();
    if (!any) return PSB_OK;
    PSB_TRY(B.d_band_cnt.alloc(sizeof(int) * kBandGroups, c.stream));
    PSB_CUDA(cudaMemsetAsync(B.d_band_cnt.p, 0, sizeof(int) * kBandGroups, c.stream));
    for (int gi = 0; gi < kBandGroups; ++gi) {
        std::vector<int> &ids = P.band_ids[gi];
        if (ids.empty()) continue;
        P.longest_first(ids);
        PSB_TRY(B.d_band_orders[gi].alloc(ids.size() * sizeof(int), c.stream));
        PSB_CUDA(cudaMemcpyAsync(B.d_band_orders[gi].p, ids.data(), ids.size() * sizeof(int), cudaMemcpyHostToDevice, c.stream));
        Band32Params p;
        std::memset(&p, 0, sizeof(p));
        p.q = g.q; p.q_off = g.q_off; p.r = g.r; p.r_off = g.r_off; p.shared_query = g.shared_query;
        p.order = B.d_band_orders[gi].as<int>(); p.n = (int)ids.size();
        p.matrix = g.matrix; p.size = g.size; p.is_pssm = g.is_pssm; p.open = g.open; p.gap = g.gap; p.k = P.band_k;
        p.score = g.score; p.end_query = g.end_query; p.end_ref = g.end_ref;
        p.matches = g.matches; p.similar = g.similar; p.length = g.length;
        p.trace = g.trace; p.trace_off = g.trace_off;
        p.counter = B.d_band_cnt.as<int>() + gi;
        const bool smem_form = gi == kBandGroups - 1;
        p.rr = smem_form ? 2 * ((P.band_maxW[gi] + 63) / 64) : 0;
        const void *fn = band32_fn(gi, cfg.stats, cfg.trace);
        // the shared-memory form: as many warps per CTA (up to kWarpsPerBlock) as the band state of each leaves room for
        const size_t mat = band32_smem_bytes(g.is_pssm ? 0 : g.size, 1, false, 0, false);
        int wpb = kWarpsPerBlock;
        if (smem_form)
            while (wpb > 1 && mat + (size_t)wpb * band32_warp_smem(p.rr, cfg.stats) > (size_t)200 * 1024) --wpb;
        const size_t smem = band32_smem_bytes(g.is_pssm ? 0 : g.size, wpb, smem_form, p.rr, cfg.stats);
        if (smem > (size_t)227 * 1024) { set_error("band state and substitution matrix too large for shared memory"); return PSB_EUNSUPPORTED; }
        int per_sm = 0;
        PSB_CUDA(occupancy_per_sm(fn, wpb, smem, &per_sm));
        PSB_CUDA(launch_persistent(fn, &p, p.n, wpb, smem, per_sm, c.sms, c.stream));
        c.launches++;
    }
    return PSB_OK;
}

// traceback: the walks of the pairs on the 32-bit kernels, then the CIGAR CSR offsets (exclusive scan of the run counts)
static int launch_walks(const PairsRequest &req, const PassPlan &P, PassBufs &B) {
    Ctx &c = g_ctx;
    const Gotoh32Params &p = B.p;
    const int64_t n = P.n;
    if (!req.cfg.trace) return PSB_OK;
    for (int cl = 0; cl < kNumClass; ++cl) {
        if (P.cls[cl].empty()) continue;
        if (!B.d_orders[cl].p) {
            PSB_TRY(B.d_orders[cl].alloc(P.cls[cl].size() * sizeof(int), c.stream));
            PSB_CUDA(cudaMemcpyAsync(B.d_orders[cl].p, P.cls[cl].data(), P.cls[cl].size() * sizeof(int), cudaMemcpyHostToDevice, c.stream));
        }
        WalkParams w;
        w.q = p.q; w.q_off = p.q_off; w.r = p.r; w.r_off = p.r_off; w.shared_query = p.shared_query;
        w.ids = B.d_orders[cl].as<int>(); w.n = (int)P.cls[cl].size(); w.K = P.ct.k[cl];
        w.trace = p.trace; w.trace_off = p.trace_off; w.end_query = p.end_query; w.end_ref = p.end_ref;
        w.rev_ops = B.d_rev.as<unsigned>(); w.rev_off = B.d_revoff.as<long long>();
        w.nops = B.d_nops.as<int>(); w.beg_query = B.d_beg[0].as<int>(); w.beg_ref = B.d_beg[1].as<int>();
        walk_trace_kernel<<<(w.n + 127) / 128, 128, 0, c.stream>>>(w);
        c.launches++;
    }
    for (int gi = 0; gi < kBandGroups; ++gi) {
        if (P.band_ids[gi].empty()) continue;
        WalkParams w;
        std::memset(&w, 0, sizeof(w));
        w.q = p.q; w.q_off = p.q_off; w.r = p.r; w.r_off = p.r_off; w.shared_query = p.shared_query;
        w.ids = B.d_band_orders[gi].as<int>(); w.n = (int)P.band_ids[gi].size();
        w.trace = p.trace; w.trace_off = p.trace_off; w.end_query = p.end_query; w.end_ref = p.end_ref;
        w.rev_ops = B.d_rev.as<unsigned>(); w.rev_off = B.d_revoff.as<long long>();
        w.nops = B.d_nops.as<int>(); w.beg_query = B.d_beg[0].as<int>(); w.beg_ref = B.d_beg[1].as<int>();
        walk_band_kernel<<<(w.n + 127) / 128, 128, 0, c.stream>>>(w, P.band_k);
        c.launches++;
    }
    // exclusive scan of nops[0..n] -> csr offsets (n+1)
    PSB_TRY(B.d_csroff.alloc(((size_t)n + 1) * sizeof(long long), c.stream));
    PSB_TRY(exclusive_sum(B.d_nops.as<int>(), B.d_csroff.as<long long>(), (int)(n + 1), B.d_scan_tmp, c.stream));
    c.launches++;
    return PSB_OK;
}

// results back to the batch's pinned arrays; with traceback, the walks' run lists compacted into the pass's CIGAR words
static int copy_results(const PairsRequest &req, const PassPlan &P, PassBufs &B, psb_batch_t *b, PassOut *po, PassTimeline &tl) {
    Ctx &c = g_ctx;
    const int64_t n = P.n, lo = P.lo;
    const std::array<int *, 6> outs = batch_outputs(b);
    const int ncopy = req.cfg.stats ? 6 : 3;
    for (int k = 0; k < ncopy; ++k)
        PSB_CUDA(cudaMemcpyAsync(outs[k] + lo, B.d_out[k].p, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    if (!req.cfg.trace) return PSB_OK;
    std::vector<long long> csr_off(n + 1);
    PSB_CUDA(cudaMemcpyAsync(csr_off.data(), B.d_csroff.p, ((size_t)n + 1) * sizeof(long long), cudaMemcpyDeviceToHost, c.stream));
    PSB_CUDA(cudaStreamSynchronize(c.stream));
    tl.phase("wait-kernels");
    const long long total = csr_off[n];
    PSB_TRY(po->d_csr.alloc((size_t)total * sizeof(unsigned), c.stream));
    CompactParams cp;
    cp.rev_ops = B.d_rev.as<unsigned>(); cp.rev_off = B.d_revoff.as<long long>();
    cp.csr_off = B.d_csroff.as<long long>(); cp.csr_ops = po->d_csr.as<unsigned>(); cp.n = (int)n;
    compact_cigar_kernel<<<c.sms * 8, 256, 0, c.stream>>>(cp);
    c.launches++;
    PSB_CUDA(cudaMemcpyAsync(b->beg_query + lo, B.d_beg[0].p, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    PSB_CUDA(cudaMemcpyAsync(b->beg_ref + lo, B.d_beg[1].p, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    po->csr_off.swap(csr_off);
    return PSB_OK;
}

// single-pair extras: the trace block as it is (psb_result_extra::trace_table() makes it row-major for the caller that
// asks), tables, last row / column
static int copy_extras(const PairsRequest &req, const PassPlan &P, PassBufs &B) {
    Ctx &c = g_ctx;
    const FnConfig &cfg = req.cfg;
    if (!(req.extra && P.n == 1 && (cfg.trace || P.want_table))) return PSB_OK;
    psb_result_extra *x = req.extra;
    const int K = P.first_cls >= 0 ? P.ct.k[P.first_cls] : 1;
    const int lq = x->qlen, lr = x->rlen;
    if (cfg.trace && P.first_cls >= 0 && B.trace_total > 0) {   // (a pair on the wavefront kernel has no flag bytes)
        // (the copy is synchronised with the results)
        x->trace_blob.resize((size_t)B.trace_total);
        x->trace_K = K;
        PSB_CUDA(cudaMemcpyAsync(x->trace_blob.data(), B.d_trace.p, x->trace_blob.size(), cudaMemcpyDeviceToHost, c.stream));
    }
    if (!P.want_table) return PSB_OK;
    std::vector<int> planes[4];
    const int np = cfg.stats ? 4 : 1;
    for (int k = 0; k < np; ++k) {
        planes[k].resize((size_t)B.trace_total);
        PSB_CUDA(cudaMemcpyAsync(planes[k].data(), B.d_tab[k].p, planes[k].size() * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    }
    PSB_CUDA(cudaStreamSynchronize(c.stream));
    std::vector<int> *tabs[4] = {&x->score_table, &x->matches_table, &x->similar_table, &x->length_table};
    std::vector<int> *rows[4] = {&x->score_row, &x->matches_row, &x->similar_row, &x->length_row};
    std::vector<int> *cols[4] = {&x->score_col, &x->matches_col, &x->similar_col, &x->length_col};
    for (int k = 0; k < np; ++k) {
        if (cfg.table) {
            tabs[k]->resize((size_t)lq * lr);
            for (int i = 0; i < lq; ++i)
                for (int j = 0; j < lr; ++j) (*tabs[k])[(size_t)i * lr + j] = planes[k][trace_cell_index(K, lr, i, j)];
        } else {
            rows[k]->resize(lr); cols[k]->resize(lq);
            for (int j = 0; j < lr; ++j) (*rows[k])[j] = planes[k][trace_cell_index(K, lr, lq - 1, j)];
            for (int i = 0; i < lq; ++i) (*cols[k])[i] = planes[k][trace_cell_index(K, lr, i, lr - 1)];
        }
    }
    return PSB_OK;
}

// One pass: pairs lo..hi-1 of the batch.  Their results land in the batch's slices lo..hi-1 and in *po.
static int run_pairs_range(const PairsRequest &req, int64_t lo, int64_t hi, psb_batch_t *b, PassOut *po) {
    Ctx &c = g_ctx;
    const int launches_at_entry = c.launches;
    PassTimeline tl;
    PassPlan plan;
    PSB_TRY(plan_pass(req, lo, hi, &plan));
    po->cells = plan.cells;
    tl.phase("classify");
    PassBufs bufs;
    PSB_TRY(upload_pass(req, plan, bufs));
    tl.phase("uploads");
    PSB_TRY(alloc_pass(req, plan, bufs));
    tl.phase("trace-offsets");
    PSB_TRY(queue_items16(req, plan, bufs));
    tl.phase("items");
    // every host->device copy of this pass is queued: the timed region (psb_last_kernel_ms) starts here
    PSB_CUDA(cudaEventRecord(c.ev0, c.stream));
    launch_map(req, plan, bufs);
    PSB_TRY(launch_pairs16(req, plan, bufs, tl));
    PSB_TRY(launch_classes(req, plan, bufs));
    PSB_TRY(launch_waves(req, plan, bufs, tl));
    PSB_TRY(launch_band(req, plan, bufs));
    PSB_TRY(launch_walks(req, plan, bufs));
    PSB_CUDA(cudaEventRecord(c.ev1, c.stream));
    tl.phase("launches");
    PSB_TRY(copy_results(req, plan, bufs, b, po, tl));
    PSB_TRY(copy_extras(req, plan, bufs));
    tl.phase("results-queued");
    PSB_CUDA(cudaStreamSynchronize(c.stream));
    tl.phase("wait");
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c.ev0, c.ev1) == cudaSuccess) { c.last_ms += ms; po->ms = ms; }
    po->launches = c.launches - launches_at_entry;
    tl.report(lo, hi, ms);
    return PSB_OK;
}

// ---- lanes for the passes of a large psb_align_pairs batch ------------------------------------------------
// Each lane is a resident host thread bound to the caller's device, with its own context (streams, events): the
// passes are handed out in order, so that while one lane's pass is in its kernels the other lane uploads and
// prepares the next one.  The passes write disjoint slices of the batch; what is not a slice comes back in PassOut.
static int run_pairs_lanes(const PairsRequest &req, PassCutter &cutter, const PairChunk &first, PassOut *first_out, psb_batch_t *b, int lanes) {
    Ctx &c = g_ctx;
    const int kLanes = std::max(1, std::min(kPairLanes, lanes));
    std::atomic<int> first_rc{PSB_OK};
    std::string errs[kPairLanes];
    std::promise<void> done[kPairLanes];
    const auto t0 = std::chrono::steady_clock::now();
    for (int t = 0; t < kLanes; ++t) {
        pair_lane(c.device, t)->submit([&, t] {
            int rc = ensure_ctx();
            PairChunk ch = first;
            PassOut *po = first_out;
            bool have = t == 0;   // lane 0 starts with the pass the caller has already cut
            while (rc == PSB_OK && first_rc.load() == PSB_OK) {
                if (!have && !cutter.next(&ch, &po)) break;
                have = false;
                rc = run_pairs_range(req, ch.lo, ch.hi, b, po);
            }
            if (rc != PSB_OK) {
                errs[t] = psb_last_error();
                int expected = PSB_OK;
                first_rc.compare_exchange_strong(expected, rc);
                cudaStreamSynchronize(g_ctx.stream);
                release_kept();
            }
            // (no release_kept() on success: a lane keeps its decision buffers from batch to batch -- giving 2 x 16 GB
            // back to the pool and taking them again at the start of every batch is what made one call in three
            // take 130-180 ms instead of 50; psb_trim() releases them)
            done[t].set_value();
        });
    }
    for (int t = 0; t < kLanes; ++t) done[t].get_future().wait();
    // the passes' timed regions overlap, so their sum says nothing: the figure reported for a pipelined batch is
    // the wall time of the pipelined section (PSB_PAIRS_LANES=1 gives the serial per-pass kernel times instead)
    c.last_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    for (const PassOut &po : cutter.pouts) c.launches += po.launches;
    const int rc = first_rc.load();
    if (rc != PSB_OK) for (int t = 0; t < kLanes; ++t) if (!errs[t].empty()) { set_error(errs[t]); break; }
    return rc;
}

int run_pairs(const PairsRequest &req, psb_batch_t **out) {
    if (out) *out = nullptr;
    if (!out || !req.matrix || !(req.r_cat || (req.r_db && req.r_ids)) || !req.r_off || req.n <= 0 || (!req.q_cat && req.matrix->type != PARASAIL_MATRIX_TYPE_PSSM)) {
        set_error("psb: NULL argument or empty batch");
        return PSB_EINVAL;
    }
    if (req.n > 0x7fffffff) { set_error("psb: more than 2^31-1 pairs in one batch"); return PSB_EUNSUPPORTED; }
    if (req.matrix->size > 96 && req.matrix->type != PARASAIL_MATRIX_TYPE_PSSM) { set_error("psb: alphabets above 96 letters are not supported"); return PSB_EUNSUPPORTED; }
    if ((req.cfg.table || req.cfg.rowcol) && !(req.extra && req.n == 1)) {
        set_error("psb: _table/_rowcol outputs exist only on the single-pair API");
        return PSB_EUNSUPPORTED;
    }
    PSB_TRY(ensure_ctx());
    Ctx &c = g_ctx;
    c.last_ms = 0.0; c.launches = 0;
    psb_batch_t *b = new_batch(req.n, req.cfg);
    if (!b) { set_error("pinned host allocation failed"); return PSB_ENOMEM; }
    // batches that keep per-cell decisions (trace, and `_stats` on the packed path, whose statistics come from
    // the walk) are cut so that a pass's decision bits + scratch stay within a budget of device memory
    int64_t budget = (int64_t)64 << 30;
    if (req.n > 4096 && (req.cfg.trace || req.cfg.stats)) {   // (a driver query: kept off the single-pair path)
        if (const size_t avail = device_mem_available()) budget = std::min<int64_t>(budget, (int64_t)(avail / 2));   // (0: unknown)
        budget = std::max<int64_t>(budget, (int64_t)1 << 30);
        budget = budget >> 30 << 30;   // whole gigabytes: small changes of the free figure do not move the cuts
    }
    const HostMatrix &hm0 = *req.matrix;
    const bool p16_scheme = p16_allowed(req) && pairs16_trace_ok(hm0.min, hm0.max, req.open) && !req.extra;
    // ---- passes.  A large batch is cut into passes twice over: by device memory (above) and by residues, so that
    // two host threads ("lanes", each with its own streams) can work on alternate passes: the uploads and the host
    // preparation of one pass run under the kernels of the other.  Small batches stay one pass on the calling thread.
    auto res_upto = [&](int64_t i) { return (req.shared_query ? 0 : req.q_off[i] - req.q_off[0]) + (req.r_off[i] - req.r_off[0]); };
    const int64_t total_res = res_upto(req.n);
    int lanes = kPairLanes;
    if (const char *ev = std::getenv("PSB_PAIRS_LANES")) lanes = std::max(1, std::min(kPairLanes, std::atoi(ev)));
    int64_t pass_res = std::numeric_limits<int64_t>::max();
    if (lanes > 1 && !req.extra && req.n >= 4096 && total_res >= ((int64_t)64 << 20))
        pass_res = std::min<int64_t>((int64_t)256 << 20, std::max<int64_t>((int64_t)16 << 20, total_res / (4 * lanes)));
    if (const char *ev = std::getenv("PSB_PAIRS_PASS_MB")) pass_res = std::max<int64_t>(1, std::atoll(ev)) << 20;
    const bool mem_cut = req.cfg.trace || (req.cfg.stats && p16_scheme);
    if (mem_cut && pass_res != std::numeric_limits<int64_t>::max()) budget /= lanes;   // one pass per lane is in flight
    // the passes are cut on demand (a pass's cut reads every pair's lengths when device memory bounds it: 10^7
    // pairs are 0.1 s of that, which the lanes do for themselves, pass by pass, instead of the caller up front)
    PassCutter cutter(req, mem_cut, p16_scheme, budget, pass_res);
    bool has_long = false;   // pairs for the whole-GPU wavefront kernel: those passes are not run side by side
    PairChunk first;
    PassOut *first_out = nullptr;
    cutter.next(&first, &first_out);
    const bool single = first.hi >= req.n;
    if (!single && lanes > 1 && hm0.type != PARASAIL_MATRIX_TYPE_PSSM && !req.cfg.stats && !req.cfg.trace) {
        if (req.shared_query) has_long = req.q_off[1] - req.q_off[0] >= kWaveMinLq;
        else for (int64_t i = 0; i < req.n && !has_long; ++i) has_long = req.q_off[i + 1] - req.q_off[i] >= kWaveMinLq;
    }
    int rc = PSB_OK;
    const bool host_dbg = debug_timing();
    const auto t_run = std::chrono::steady_clock::now();
    if (single || lanes == 1 || has_long) {
        PairChunk ch = first;
        PassOut *po = first_out;
        do rc = run_pairs_range(req, ch.lo, ch.hi, b, po); while (rc == PSB_OK && cutter.next(&ch, &po));
        if (rc != PSB_OK) cudaStreamSynchronize(c.stream);
    } else {
        rc = run_pairs_lanes(req, cutter, first, first_out, b, lanes);
    }
    std::deque<PairChunk> &chunks = cutter.chunks;
    std::deque<PassOut> &pouts = cutter.pouts;
    const auto t_join = std::chrono::steady_clock::now();
    if (rc == PSB_OK && req.cfg.trace) {
        // the passes' CIGAR words are still on the device: one pinned array for the batch, one copy per pass into it
        long long total = 0;
        for (const PassOut &po : pouts) total += po.csr_off.empty() ? 0 : po.csr_off.back();
        BatchImpl *impl = (BatchImpl *)b->impl;
        b->cigar_ops = (uint32_t *)impl->take((size_t)(total + 1) * sizeof(uint32_t));
        if (!b->cigar_ops) { set_error("pinned allocation failed"); rc = PSB_ENOMEM; }
        long long used = 0;
        for (size_t k = 0; k < pouts.size() && rc == PSB_OK; ++k) {
            const PassOut &po = pouts[k];
            const int64_t n = chunks[k].hi - chunks[k].lo;
            if ((int64_t)po.csr_off.size() != n + 1) { set_error("psb: a pass returned no CIGAR offsets"); rc = PSB_ECUDA; break; }
            if (po.csr_off[n] > 0 &&
                cudaMemcpyAsync(b->cigar_ops + used, po.d_csr.p, (size_t)po.csr_off[n] * sizeof(uint32_t), cudaMemcpyDeviceToHost, c.stream) != cudaSuccess) {
                set_error(std::string("psb: CIGAR copy: ") + cudaGetErrorString(cudaGetLastError())); rc = PSB_ECUDA; break;
            }
            for (int64_t i = 0; i <= n; ++i) b->cigar_off[chunks[k].lo + i] = used + po.csr_off[i];
            used += po.csr_off[n];
        }
        if (cudaStreamSynchronize(c.stream) != cudaSuccess && rc == PSB_OK) { set_error("psb: CIGAR copy failed"); rc = PSB_ECUDA; }
    }
    for (PassOut &po : pouts) {
        b->cells += po.cells;
        po.d_csr.release();
    }
    release_kept();
    if (host_dbg)
        std::fprintf(stderr, "[psb] run_pairs: %zu passes, passes %.3f ms, join %.3f ms\n", chunks.size(),
                     std::chrono::duration<double, std::milli>(t_join - t_run).count(),
                     std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_join).count());
    if (rc != PSB_OK) { free_batch(b); return rc; }
    *out = b;
    return PSB_OK;
}

// psb_align_pairs / psb_align_pairs_banded once the name is parsed: the pairs pass, then, for explicit narrow widths,
// the pairs whose values do not fit flagged (SURVEY A.8), the same rule as align_one
static int align_pairs(const FnConfig &cfg, const HostMatrix &hm, int open, int gap, const uint8_t *q_cat, const int64_t *q_off,
                       const uint8_t *r_cat, const int64_t *r_off, int64_t n, psb_batch_t **out) {
    PairsRequest req;
    req.cfg = cfg; req.matrix = &hm; req.open = open; req.gap = gap;
    req.q_cat = q_cat; req.q_off = q_off; req.r_cat = r_cat; req.r_off = r_off; req.n = n;
    const int rc = run_pairs(req, out);
    const bool pssm = hm.type == PARASAIL_MATRIX_TYPE_PSSM;
    if (rc == PSB_OK)
        flag_saturated(cfg, hm, open, gap, *out, [&](int64_t i) { return std::make_pair(pssm ? hm.length : span(q_off, i), span(r_off, i)); });
    return rc;
}

// launchers of kern_util.cuh's kernels for the files that do not include it (a second copy of its non-template kernels
// would define their host stubs twice)
void launch_unpack_db(const psb_db *db, const int *ids, const int *inv_perm, const long long *out_off, uint8_t *out, long long n, unsigned grid,
                      unsigned block, cudaStream_t stream) {
    UnpackParams u;
    u.words = db->d_words; u.word_off = db->d_word_off; u.ids = ids; u.inv_perm = inv_perm;
    u.out_off = out_off; u.out = out; u.n = n; u.bits = db->bits;
    unpack_db_kernel<<<grid, block, 0, stream>>>(u);
}
void launch_pack_db(const DbBuild &B, unsigned grid, unsigned block, size_t smem, cudaStream_t stream) {
    const psb_db *db = B.db;
    PackParams pp;
    pp.raw = B.raw(); pp.raw_off = B.offs(); pp.raw_base = B.raw_base; pp.perm = db->d_perm;
    pp.word_off = db->d_word_off; pp.words = db->d_words; pp.n = db->n; pp.bits = db->bits;
    std::memcpy(pp.lut, B.lut, sizeof(pp.lut));
    pack_db_kernel<<<grid, block, smem, stream>>>(pp);
}
void launch_invert_perm(const int *perm, long long n, int *inv, unsigned grid, unsigned block, cudaStream_t stream) {
    invert_perm_kernel<<<grid, block, 0, stream>>>(perm, n, inv);
}

}  // namespace psb

using namespace psb;

extern "C" {

int psb_align_pairs(const char *fn_name, const parasail_matrix_t *matrix, int open, int gap, const uint8_t *q_cat,
                    const int64_t *q_off, const uint8_t *r_cat, const int64_t *r_off, int64_t n, psb_batch_t **out) {
    FnConfig cfg;
    if (!parse_fn_name(fn_name, &cfg) || cfg.profile) { set_error(std::string("psb_align_pairs: unknown function name: ") + (fn_name ? fn_name : "(null)")); return PSB_EINVAL; }
    if (!matrix) { set_error("psb_align_pairs: NULL matrix"); return PSB_EINVAL; }
    HostMatrix hm(matrix);
    return align_pairs(cfg, hm, open, gap, q_cat, q_off, r_cat, r_off, n, out);
}

int psb_align_pairs_banded(const char *fn_name, const parasail_matrix_t *matrix, int open, int gap, int k, const uint8_t *q_cat,
                           const int64_t *q_off, const uint8_t *r_cat, const int64_t *r_off, int64_t n, psb_batch_t **out) {
    if (out) *out = nullptr;
    FnConfig cfg;
    if (!parse_fn_name(fn_name, &cfg) || cfg.profile) { set_error(std::string("psb_align_pairs_banded: unknown function name: ") + (fn_name ? fn_name : "(null)")); return PSB_EINVAL; }
    if (cfg.mode != MODE_NW) { set_error(std::string("psb_align_pairs_banded: banded alignment is global only (nw): ") + fn_name); return PSB_EINVAL; }
    if (cfg.table || cfg.rowcol) { set_error("psb_align_pairs_banded: _table/_rowcol outputs exist only on the single-pair API"); return PSB_EUNSUPPORTED; }
    if (k <= 0) { set_error("psb_align_pairs_banded: band half-width " + std::to_string(k) + " is not positive"); return PSB_EINVAL; }
    if (!matrix || !q_off || !r_cat || !r_off || !out || n <= 0 || (!q_cat && matrix->type != PARASAIL_MATRIX_TYPE_PSSM)) {
        set_error("psb_align_pairs_banded: NULL argument or empty batch");
        return PSB_EINVAL;
    }
    HostMatrix hm(matrix);
    const bool pssm = hm.type == PARASAIL_MATRIX_TYPE_PSSM;
    for (int64_t i = 0; i < n; ++i) {
        const int lq = pssm ? hm.length : (int)(q_off[i + 1] - q_off[i]), lr = (int)(r_off[i + 1] - r_off[i]);
        if (lq <= 0 || lr <= 0) { set_error("psb_align_pairs_banded: empty sequence in batch (pair " + std::to_string(i) + ")"); return PSB_EINVAL; }
        const BandGeom b = band_geom(lq, lr, k);
        if (!band_covers(b, lq, lr) && b.W > kBandMaxW) {
            set_error("psb_align_pairs_banded: pair " + std::to_string(i) + " (" + std::to_string(lq) + " x " + std::to_string(lr) + ") has a band of W = " +
                      std::to_string(b.W) + " diagonals; the band kernel takes at most " + std::to_string(kBandMaxW));
            return PSB_EUNSUPPORTED;
        }
    }
    cfg.band = k;
    const int rc = align_pairs(cfg, hm, open, gap, q_cat, q_off, r_cat, r_off, n, out);
    if (rc == PSB_OK) (*out)->flag |= PARASAIL_FLAG_BANDED;
    return rc;
}

}  // extern "C"
