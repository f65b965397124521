// search.cu -- many query profiles against a resident database in one call (psb_db_search).  Per query, the score-only
// scan of scan.cu and then, on the device and behind it in the same stream, the selection of its kk best subjects
// (kern_topk.cuh): only kk rows per query ever reach the host, in one copy at the end.  The hits of every query then
// go through one pairs pass (or one per group of queries that share a matrix) for _trace / _stats names.
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cstring>
#include <memory>
#include <numeric>
#include <string>
#include <vector>

#include "engine.h"
#include "kern_topk.cuh"

namespace psb {

static constexpr int kTopkThreads = 256;
static constexpr int kTopkIdsPerWarp = 2048;

// the selection's launch shape and the device buffers every query of a call reuses, one query after another
struct TopkBufs {
    unsigned hist_blocks = 1;
    int nwarps = 1;
    long long chunk = 32;
    DevMem st, counts, offs, tmp, sat;
};

static int topk_prepare(int64_t n, bool saturation, TopkBufs &B) {
    Ctx &c = g_ctx;
    B.hist_blocks = (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + kTopkThreads - 1) / kTopkThreads, (int64_t)c.sms * 4));
    B.nwarps = (int)std::max<int64_t>(1, std::min<int64_t>((n + kTopkIdsPerWarp - 1) / kTopkIdsPerWarp, (int64_t)c.sms * 16));
    B.chunk = topk_chunk(n, B.nwarps);
    PSB_TRY(B.st.alloc(sizeof(TopkState), c.stream));
    PSB_TRY(B.counts.alloc(2 * (size_t)B.nwarps * sizeof(int), c.stream));
    PSB_TRY(B.offs.alloc(2 * (size_t)B.nwarps * sizeof(long long), c.stream));
    if (saturation) PSB_TRY(B.sat.alloc((size_t)n * sizeof(int), c.stream));
    return PSB_OK;
}

// the rule of saturates() (result.cpp) for one query of `qlen` residues, as thresholds on the score and on the longer
// of the two sequences
static TopkSat topk_sat(const FnConfig &cfg, const HostMatrix &m, int qlen, int open, int gap, const psb_db *db) {
    const long long hi = cfg.width == 8 ? 127 : 32767, lo = -hi - 1;
    TopkSat s;
    s.score_hi = (int)(hi - std::max(m.max, 0));
    s.score_lo = INT_MIN;
    s.len_hi = INT_MAX;
    s.qlen = qlen;
    s.len_sorted = db->d_len; s.inv_perm = db->d_inv_perm;
    if (cfg.mode != MODE_SW) {
        s.score_lo = (int)(lo - std::min(m.min, 0));
        // -open - (L - 1) * gap + min(m.min, 0) < lo  <=>  (L - 1) * gap > x
        const long long x = -(long long)open + std::min(m.min, 0) - lo;
        if (cfg.mode == MODE_NW || !cfg.s1_beg || !cfg.s2_beg)
            s.len_hi = x < 0 ? 0 : (gap > 0 ? (int)std::min<long long>(INT_MAX, x / gap + 1) : INT_MAX);
    }
    return s;
}

// the kk best subjects of one scan (job.d_out, caller order) into the rows rows[plane * nrows + row0 ...]; `sat`:
// explicit widths, applied first
static int launch_topk(ScanJob &job, int64_t n, int kk, const TopkSat *sat, TopkBufs &B, int *rows, int64_t nrows, int64_t row0) {
    Ctx &c = g_ctx;
    TopkParams p;
    std::memset(&p, 0, sizeof(p));
    p.score = job.d_out[0].as<int>(); p.end_query = job.d_out[1].as<int>(); p.end_ref = job.d_out[2].as<int>();
    p.n = n; p.kk = kk; p.st = B.st.as<TopkState>();
    p.chunk = B.chunk; p.nwarps = B.nwarps; p.counts = B.counts.as<int>(); p.offs = B.offs.as<long long>();
    p.sat = sat ? B.sat.as<int>() : nullptr;
    int *planes[5];
    for (int k = 0; k < 5; ++k) planes[k] = rows + (size_t)k * nrows + row0;
    p.out_id = planes[0]; p.out_score = planes[1]; p.out_end_query = planes[2]; p.out_end_ref = planes[3]; p.out_sat = planes[4];
    PSB_CUDA(cudaMemsetAsync(B.st.p, 0, sizeof(TopkState), c.stream));
    if (sat) { topk_saturate_kernel<<<B.hist_blocks, kTopkThreads, 0, c.stream>>>(p, *sat); c.launches++; }
    for (int shift = 24; shift >= 0; shift -= 8) {
        p.shift = shift;
        topk_hist_kernel<<<B.hist_blocks, kTopkThreads, kTopkBins * sizeof(int), c.stream>>>(p);
        topk_pick_kernel<<<1, 32, 0, c.stream>>>(p);
        c.launches += 2;
    }
    const unsigned take_blocks = (unsigned)((B.nwarps + kTopkThreads / 32 - 1) / (kTopkThreads / 32));
    topk_take_kernel<false><<<take_blocks, kTopkThreads, 0, c.stream>>>(p);
    PSB_CUDA(cudaGetLastError());
    PSB_TRY(exclusive_sum(B.counts.as<int>(), B.offs.as<long long>(), 2 * B.nwarps, B.tmp, c.stream));
    topk_take_kernel<true><<<take_blocks, kTopkThreads, 0, c.stream>>>(p);
    c.launches += 4;   // the two compaction launches and cub's two (init, scan)
    PSB_CUDA(cudaGetLastError());
    return PSB_OK;
}

// queries whose hits can share a pairs pass: equal matrices (type, size, values, mapper).  A PSSM profile gets a pass
// of its own.
static bool same_matrix(const HostMatrix &a, const HostMatrix &b) {
    return a.type == b.type && a.size == b.size && a.length == b.length && a.table == b.table && std::memcmp(a.mapper, b.mapper, 256) == 0;
}

// the alignments of the rows `rows` (one group: equal matrices), in that order: one pairs pass.  Rows of one query are
// psb_db_align's request exactly; rows of several carry each row's query bytes.
static int align_group(const FnConfig &cfg, const parasail_profile_t *const *profiles, const std::vector<int64_t> &rows, const int64_t *row_q,
                       const int64_t *row_id, int open, int gap, psb_db *db, psb_batch_t **out) {
    const int64_t n = (int64_t)rows.size();
    std::vector<int> rid((size_t)n);
    std::vector<int64_t> r_off((size_t)n + 1), q_off;
    std::vector<uint8_t> q_cat;
    r_off[0] = 0;
    bool one_query = true;
    for (int64_t i = 0; i < n; ++i) {
        const int64_t id = row_id[rows[(size_t)i]];
        rid[(size_t)i] = (int)id;
        r_off[(size_t)i + 1] = r_off[(size_t)i] + db->host_len[(size_t)id];
        one_query = one_query && row_q[rows[(size_t)i]] == row_q[rows[0]];
    }
    const parasail_profile_t *p0 = profiles[row_q[rows[0]]];
    PairsRequest req;
    req.cfg = cfg;
    req.matrix = &p0->matrix; req.open = open; req.gap = gap;
    if (one_query) {
        q_off = {0, (int64_t)p0->query.size()};
        req.q_cat = p0->query.data(); req.shared_query = true;
    } else {
        q_off.assign((size_t)n + 1, 0);
        for (int64_t i = 0; i < n; ++i) {
            const std::vector<uint8_t> &q = profiles[row_q[rows[(size_t)i]]]->query;
            q_cat.insert(q_cat.end(), q.begin(), q.end());
            q_off[(size_t)i + 1] = (int64_t)q_cat.size();
        }
        req.q_cat = q_cat.data(); req.shared_query = false;
    }
    req.q_off = q_off.data();
    req.r_off = r_off.data(); req.n = n; req.r_db = db; req.r_ids = rid.data();
    PSB_TRY(run_pairs(req, out));
    flag_saturated(cfg, p0->matrix, open, gap, *out, [&](int64_t i) {
        return std::make_pair((int)profiles[row_q[rows[(size_t)i]]]->query.size(), span(r_off.data(), i));
    });
    return PSB_OK;
}

int gather_rows(const FnConfig &cfg, const std::vector<psb_batch_t *> &gb, const std::vector<std::pair<int, int64_t>> &src, psb_batch_t **out) {
    const int64_t n = (int64_t)src.size();
    psb_batch_t *b = new_batch(n, cfg);
    if (!b) { set_error("pinned host allocation failed"); return PSB_ENOMEM; }
    long long nops = 0;
    for (int64_t i = 0; i < n; ++i) {
        const psb_batch_t *s = gb[(size_t)src[(size_t)i].first];
        const int64_t j = src[(size_t)i].second;
        b->score[i] = s->score[j]; b->end_query[i] = s->end_query[j]; b->end_ref[i] = s->end_ref[j]; b->saturated[i] = s->saturated[j];
        if (cfg.stats) { b->matches[i] = s->matches[j]; b->similar[i] = s->similar[j]; b->length[i] = s->length[j]; }
        if (cfg.trace) {
            b->beg_query[i] = s->beg_query[j]; b->beg_ref[i] = s->beg_ref[j];
            nops += s->cigar_off[j + 1] - s->cigar_off[j];
            b->cigar_off[i + 1] = nops;
        }
    }
    if (cfg.trace) {
        b->cigar_ops = (uint32_t *)((BatchImpl *)b->impl)->take((size_t)(nops + 1) * sizeof(uint32_t));
        if (!b->cigar_ops) { free_batch(b); set_error("pinned host allocation failed"); return PSB_ENOMEM; }
        for (int64_t i = 0; i < n; ++i) {
            const psb_batch_t *s = gb[(size_t)src[(size_t)i].first];
            const int64_t j = src[(size_t)i].second;
            std::memcpy(b->cigar_ops + b->cigar_off[i], s->cigar_ops + s->cigar_off[j], (size_t)(s->cigar_off[j + 1] - s->cigar_off[j]) * sizeof(uint32_t));
        }
    }
    for (const psb_batch_t *s : gb) b->cells += s->cells;
    *out = b;
    return PSB_OK;
}

int align_rows(const FnConfig &cfg, const parasail_profile_t *const *profiles, int64_t nq, const int64_t *row_q, const int64_t *row_id,
               int64_t n, int open, int gap, psb_db *db, psb_batch_t **out) {
    // the groups in order of their first row; a PSSM profile gets a group of its own
    std::vector<int> group_of((size_t)nq, -1);
    std::vector<std::vector<int64_t>> groups;
    for (int64_t i = 0; i < n; ++i) {
        const int64_t q = row_q[i];
        if (group_of[(size_t)q] < 0) {
            const HostMatrix &m = profiles[q]->matrix;
            auto it = std::find_if(groups.begin(), groups.end(), [&](const std::vector<int64_t> &g) {
                const HostMatrix &g0 = profiles[row_q[g[0]]]->matrix;
                return m.type != PARASAIL_MATRIX_TYPE_PSSM && g0.type != PARASAIL_MATRIX_TYPE_PSSM && same_matrix(m, g0);
            });
            group_of[(size_t)q] = (int)(it - groups.begin());
            if (it == groups.end()) groups.emplace_back();
        }
        groups[(size_t)group_of[(size_t)q]].push_back(i);
    }
    int first_use = 0;
    PSB_TRY(db_inv_perm(db, &first_use));
    Ctx &c = g_ctx;
    double ms = c.last_ms;
    int launches = c.launches + first_use;
    std::vector<psb_batch_t *> gb;
    std::vector<std::pair<int, int64_t>> src((size_t)n);
    int rc = PSB_OK;
    for (size_t g = 0; g < groups.size() && rc == PSB_OK; ++g) {
        psb_batch_t *b = nullptr;
        rc = align_group(cfg, profiles, groups[g], row_q, row_id, open, gap, db, &b);   // (run_pairs restarts the counters)
        ms += c.last_ms; launches += c.launches;
        if (rc != PSB_OK) break;
        gb.push_back(b);
        for (size_t t = 0; t < groups[g].size(); ++t) src[(size_t)groups[g][t]] = {(int)g, (int64_t)t};
    }
    c.last_ms = ms; c.launches = launches;
    if (rc == PSB_OK && gb.size() == 1) { *out = gb[0]; return PSB_OK; }   // one group holds every row in row order
    if (rc == PSB_OK) rc = gather_rows(cfg, gb, src, out);
    for (psb_batch_t *b : gb) free_batch(b);
    return rc;
}

int search_select(const FnConfig &cfg, const parasail_profile_t *const *profiles, int64_t nq, int open, int gap, psb_db *db, int64_t kk,
                  SearchHits *hits) {
    const int64_t R = nq * kk;
    Ctx &c = g_ctx;
    c.last_ms = 0.0; c.launches = 0;
    // the scans run under the name without _trace / _stats, the rule of Aligner.search
    FnConfig scfg = cfg;
    scfg.trace = false; scfg.stats = false;
    const bool saturation = cfg.width == 8 || cfg.width == 16;
    if (saturation) {
        int first_use = 0;
        PSB_TRY(db_inv_perm(db, &first_use));
        c.launches += first_use;
    }
    // every profile's device copy and packed form first: a first use waits for its upload, which would otherwise
    // stall the stream between two scans
    for (int64_t q = 0; q < nq; ++q) PSB_TRY(prepare_query(scfg, profiles[q], open, gap));
    TopkBufs B;
    DevMem d_rows;
    PSB_TRY(topk_prepare(db->n, saturation, B));
    PSB_TRY(d_rows.alloc((size_t)R * 5 * sizeof(int), c.stream));
    std::vector<std::unique_ptr<ScanJob>> jobs;
    int rc = PSB_OK;
    for (int64_t q = 0; q < nq && rc == PSB_OK; ++q) {
        jobs.emplace_back(new ScanJob());
        ScanJob &job = *jobs.back();
        rc = scan_enqueue(job, scfg, profiles[q], open, gap, db, nullptr, 0);
        TopkSat sat;
        if (saturation) sat = topk_sat(cfg, profiles[q]->matrix, (int)profiles[q]->query.size(), open, gap, db);
        if (rc == PSB_OK) rc = launch_topk(job, db->n, (int)kk, saturation ? &sat : nullptr, B, d_rows.as<int>(), R, q * kk);
        for (DevMem &d : job.d_out) d.release();   // in stream order: one query's n-sized results are live at a time
    }
    int *rows = rc == PSB_OK ? (int *)pinned_alloc((size_t)R * 5 * sizeof(int)) : nullptr;
    if (rc == PSB_OK && !rows) { set_error("pinned host allocation failed"); rc = PSB_ENOMEM; }
    if (rc == PSB_OK && cudaEventRecord(c.ev1, c.stream) != cudaSuccess) { set_error("psb_db_search: cudaEventRecord failed"); rc = PSB_ECUDA; }
    if (rc == PSB_OK && cudaMemcpyAsync(rows, d_rows.p, (size_t)R * 5 * sizeof(int), cudaMemcpyDeviceToHost, c.stream) != cudaSuccess) {
        set_error("psb_db_search: row copy failed"); rc = PSB_ECUDA;
    }
    if (rc == PSB_OK && cudaStreamSynchronize(c.stream) != cudaSuccess) {
        set_error(std::string("psb_db_search: ") + cudaGetErrorString(cudaGetLastError())); rc = PSB_ECUDA;
    }
    for (auto &j : jobs) {
        if (rc == PSB_OK) rc = scan_finish(*j);
        hits->retried += j->retried;
    }
    if (rc != PSB_OK) {
        cudaStreamSynchronize(c.stream);
        if (rows) pinned_free(rows, (size_t)R * 5 * sizeof(int));
        return rc;
    }
    // the device time of the scans and selections, back to back on the stream (replaces scan_finish's sum of scans)
    float sel_ms = 0.f;
    if (cudaEventElapsedTime(&sel_ms, jobs[0]->ev0, c.ev1) == cudaSuccess) c.last_ms = sel_ms;
    jobs.clear();
    // each query's rows in the order of psb_batch_topk
    const int *r_id = rows, *r_score = rows + R;
    std::vector<int64_t> order((size_t)R);
    for (int64_t q = 0; q < nq; ++q) {
        int64_t *o = order.data() + q * kk;
        std::iota(o, o + kk, q * kk);
        std::sort(o, o + kk, [&](int64_t a, int64_t b) { return r_score[a] != r_score[b] ? r_score[a] > r_score[b] : r_id[a] < r_id[b]; });
    }
    std::vector<int> *planes[5] = {&hits->id, &hits->score, &hits->end_query, &hits->end_ref, &hits->saturated};
    for (int k = 0; k < 5; ++k) {
        planes[k]->resize((size_t)R);
        const int *src = rows + (size_t)k * R;
        for (int64_t i = 0; i < R; ++i) (*planes[k])[(size_t)i] = src[order[(size_t)i]];
    }
    pinned_free(rows, (size_t)R * 5 * sizeof(int));
    return PSB_OK;
}

}  // namespace psb

using namespace psb;

extern "C" {

int psb_db_search(const char *fn_name, const parasail_profile_t *const *profiles, int64_t nq, int open, int gap, const psb_db_t *db_c, int k,
                  int64_t *ids_out, psb_batch_t **out) {
    if (out) *out = nullptr;
    FnConfig cfg;
    if (!parse_fn_name(fn_name, &cfg) || !cfg.profile) {
        set_error(std::string("psb_db_search: not a profile function name: ") + (fn_name ? fn_name : "(null)"));
        return PSB_EINVAL;
    }
    if (cfg.table || cfg.rowcol) { set_error("psb_db_search: _table/_rowcol outputs exist only on the single-pair API"); return PSB_EUNSUPPORTED; }
    if (!profiles || !db_c || !ids_out || !out) { set_error("psb_db_search: NULL argument"); return PSB_EINVAL; }
    if (nq <= 0 || k <= 0) { set_error("psb_db_search: " + std::to_string(nq) + " queries, k = " + std::to_string(k)); return PSB_EINVAL; }
    psb_db *db = const_cast<psb_db *>(db_c);
    PSB_TRY(db_check("psb_db_search", db));
    const int64_t kk = std::min<int64_t>(k, db->n);
    if (nq > INT_MAX / kk) {
        set_error("psb_db_search: " + std::to_string(nq) + " queries x " + std::to_string(kk) + " hits is more than 2^31-1 rows");
        return PSB_EUNSUPPORTED;
    }
    for (int64_t q = 0; q < nq; ++q) {
        const std::string who = "psb_db_search: profiles[" + std::to_string(q) + "]";
        if (!profiles[q]) { set_error(who + " is NULL"); return PSB_EINVAL; }
        PSB_TRY(profile_db_check(who.c_str(), profiles[q], db));
    }
    const int64_t R = nq * kk;
    SearchHits h;
    PSB_TRY(search_select(cfg, profiles, nq, open, gap, db, kk, &h));
    for (int64_t i = 0; i < R; ++i) ids_out[i] = h.id[(size_t)i];
    double scan_cells = 0;
    for (int64_t q = 0; q < nq; ++q) scan_cells += (double)profiles[q]->query.size() * (double)db->residues;
    psb_batch_t *b = nullptr;
    if (cfg.trace || cfg.stats) {
        std::vector<int64_t> row_q((size_t)R);
        for (int64_t i = 0; i < R; ++i) row_q[(size_t)i] = i / kk;
        PSB_TRY(align_rows(cfg, profiles, nq, row_q.data(), ids_out, R, open, gap, db, &b));
    } else {
        b = new_batch(R, cfg);
        if (!b) { set_error("pinned host allocation failed"); return PSB_ENOMEM; }
        for (int64_t i = 0; i < R; ++i) {
            b->score[i] = h.score[(size_t)i]; b->end_query[i] = h.end_query[(size_t)i]; b->end_ref[i] = h.end_ref[(size_t)i];
            b->saturated[i] = (uint8_t)h.saturated[(size_t)i];
        }
    }
    b->cells += scan_cells;
    b->n_retried = h.retried;
    *out = b;
    return PSB_OK;
}

}  // extern "C"
