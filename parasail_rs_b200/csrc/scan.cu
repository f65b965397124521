// scan.cu -- a resident query profile against a resident packed database: psb_scan (SURVEY config C2) and
// psb_db_align.  The packed 16-bit scan (kern_sw16.cuh) is planned, then launched in named stages beside the
// wavefront launch of the longest subjects and the 32-bit re-run of those that leave the 16-bit range.  The
// one-warp-per-pair 32-bit kernels are instantiated and launched here too.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "engine.h"
#include "kern_gotoh32.cuh"
#include "kern_sw16.cuh"
#include "pairs16_host.h"

namespace psb {

// ---- the one-warp-per-pair 32-bit kernels (kern_gotoh32.cuh): the pairs pass and the scan's general path and re-run
// launch them through launch_gotoh32.  They are instantiated beside the packed scan kernel: compiled in a module of
// their own, ptxas gives nine of them one to four registers more or less.
// Two kernel families.  "fine": per-warp int8 profile, mode-specialised, 13 row-per-lane classes
// (the many-pairs fast path).  "coarse": substitution matrix read directly (values that do not fit
// a byte, PSSMs, table outputs), mode read at run time, 3 classes.
static const int kFineK[] = {1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 12, 14, 16};
static const int kCoarseK[] = {4, 8, 16};
ClassTable class_table(bool fine) { return fine ? ClassTable{kFineK, 13} : ClassTable{kCoarseK, 3}; }
int class_of_len(const ClassTable &t, int lq) {
    for (int c = 0; c < t.n; ++c) if (lq <= 32 * t.k[c]) return c;
    return t.n - 1;
}

template <int K, int MS> static const void *gotoh32_fine_km(Variant v) {
    switch (v) {
        case V_SCORE: return (const void *)gotoh32_kernel<K, false, false, false, unsigned, true, MS>;
        case V_STATS32: return (const void *)gotoh32_kernel<K, true, false, false, unsigned, true, MS>;
        case V_STATS64: return (const void *)gotoh32_kernel<K, true, false, false, unsigned long long, true, MS>;
        case V_TRACE: return (const void *)gotoh32_kernel<K, false, true, false, unsigned, true, MS>;
        default: return nullptr;
    }
}
template <int K> static const void *gotoh32_fine_k(Variant v, bool sw) { return sw ? gotoh32_fine_km<K, 1>(v) : gotoh32_fine_km<K, 2>(v); }
template <int K> static const void *gotoh32_coarse_k(Variant v) {
    switch (v) {
        case V_SCORE: return (const void *)gotoh32_kernel<K, false, false, false, unsigned>;
        case V_STATS32:
        case V_STATS64: return (const void *)gotoh32_kernel<K, true, false, false, unsigned long long>;
        case V_TRACE: return (const void *)gotoh32_kernel<K, false, true, false, unsigned>;
        case V_TABLE: return (const void *)gotoh32_kernel<K, true, false, true, unsigned long long>;
    }
    return nullptr;
}
static const void *gotoh32_fn(int K, Variant v, bool fine, bool sw) {
    if (!fine) {
        switch (K) {
            case 4: return gotoh32_coarse_k<4>(v);
            case 8: return gotoh32_coarse_k<8>(v);
            case 16: return gotoh32_coarse_k<16>(v);
        }
        return nullptr;
    }
    switch (K) {
        case 1: return gotoh32_fine_k<1>(v, sw);
        case 2: return gotoh32_fine_k<2>(v, sw);
        case 3: return gotoh32_fine_k<3>(v, sw);
        case 4: return gotoh32_fine_k<4>(v, sw);
        case 5: return gotoh32_fine_k<5>(v, sw);
        case 6: return gotoh32_fine_k<6>(v, sw);
        case 7: return gotoh32_fine_k<7>(v, sw);
        case 8: return gotoh32_fine_k<8>(v, sw);
        case 9: return gotoh32_fine_k<9>(v, sw);
        case 10: return gotoh32_fine_k<10>(v, sw);
        case 12: return gotoh32_fine_k<12>(v, sw);
        case 14: return gotoh32_fine_k<14>(v, sw);
        case 16: return gotoh32_fine_k<16>(v, sw);
    }
    return nullptr;
}

int launch_gotoh32(int K, Variant v, Gotoh32Params &p, int nwork, bool prof, long long *grid_warps_out) {
    Ctx &c = g_ctx;
    if (!prof && v == V_STATS32) v = V_STATS64;   // the coarse family carries only the wide statistics word
    const void *fn = gotoh32_fn(K, v, prof, p.mode == MODE_SW);
    if (!fn) { set_error("internal: no kernel for this class"); return PSB_EUNSUPPORTED; }
    const bool stats = v == V_STATS32 || v == V_STATS64 || v == V_TABLE;
    const int statw = v == V_STATS32 ? 4 : 8;
    const size_t smem = gotoh32_smem_bytes(p.is_pssm ? 0 : p.size, kWarpsPerBlock, stats, statw, prof);
    if (smem > 200 * 1024) { set_error("substitution matrix too large for shared memory"); return PSB_EUNSUPPORTED; }
    int per_sm = 0;
    long long blocks = 0;
    PSB_CUDA(occupancy_per_sm(fn, kWarpsPerBlock, smem, &per_sm));
    PSB_CUDA(launch_persistent(fn, &p, nwork, kWarpsPerBlock, smem, per_sm, c.sms, c.stream, &blocks));
    if (grid_warps_out) *grid_warps_out = blocks * kWarpsPerBlock;
    c.launches++;
    return PSB_OK;
}

// upper bound on the warps any launch of `nwork` items can have resident (scratch lines are per warp)
long long max_grid_warps(long long nwork) {
    const long long cap = (long long)g_ctx.sms * 16 * kWarpsPerBlock;
    const long long need = ((nwork + kWarpsPerBlock - 1) / kWarpsPerBlock) * kWarpsPerBlock;
    return std::max<long long>(kWarpsPerBlock, std::min(cap, need));
}

// ---- the scan --------------------------------------------------------------------------------------
struct DevProfile {
    uint8_t *d_query = nullptr;     // mapped residues
    long long *d_qoff = nullptr;    // {0, Lq}
    int *d_matrix = nullptr;
    cudaStream_t stream = nullptr;  // allocation stream (stream-ordered pool)
    std::vector<uint8_t> mapped;    // host copy of the mapped query
    // packed profiles (+open) of the 16-bit scan kernel, one per gap-open value ever used with this
    // profile on this device: built under the profile's mutex, immutable afterwards and freed only in
    // release_profile_resident, so concurrent scans with different penalties never see a buffer replaced
    std::map<int, std::vector<Sw16Profile>> sw16;   // one entry per strip of the query (queries <= 400 aa: one)
};

void release_profile_resident(parasail_profile *p) {
    std::lock_guard<std::mutex> lk(p->mu);
    for (auto &kv : p->resident) {
        DevProfile *d = (DevProfile *)kv.second;
        int cur = 0;
        cudaGetDevice(&cur);
        cudaSetDevice(kv.first);
        void *ptrs[] = {d->d_query, d->d_qoff, d->d_matrix};
        for (void *q : ptrs) if (q) cudaFreeAsync(q, d->stream);
        for (auto &sv : d->sw16) for (auto &sp : sv.second) if (sp.prof) cudaFreeAsync(sp.prof, d->stream);
        cudaSetDevice(cur);
        delete d;
    }
    p->resident.clear();
}

static int get_dev_profile(const parasail_profile *prof, DevProfile **out) {
    Ctx &c = g_ctx;
    std::lock_guard<std::mutex> lk(prof->mu);
    auto it = prof->resident.find(c.device);
    if (it != prof->resident.end()) { *out = (DevProfile *)it->second; return PSB_OK; }
    DevProfile *d = new DevProfile();
    const HostMatrix &m = prof->matrix;
    const size_t lq = prof->query.size();
    std::vector<uint8_t> mapped(lq);
    for (size_t i = 0; i < lq; ++i) mapped[i] = m.mapper[prof->query[i]];
    long long qoff[2] = {0, (long long)lq};
    d->stream = c.stream;
    PSB_CUDA(cudaMallocAsync(&d->d_query, std::max<size_t>(lq, 16), c.stream));
    PSB_CUDA(cudaMallocAsync(&d->d_qoff, sizeof(qoff), c.stream));
    PSB_CUDA(cudaMallocAsync(&d->d_matrix, m.table.size() * sizeof(int), c.stream));
    PSB_CUDA(cudaMemcpyAsync(d->d_query, mapped.data(), lq, cudaMemcpyHostToDevice, c.stream));
    PSB_CUDA(cudaMemcpyAsync(d->d_qoff, qoff, sizeof(qoff), cudaMemcpyHostToDevice, c.stream));
    PSB_CUDA(cudaMemcpyAsync(d->d_matrix, m.table.data(), m.table.size() * sizeof(int), cudaMemcpyHostToDevice, c.stream));
    d->mapped = mapped;
    PSB_CUDA(cudaStreamSynchronize(c.stream));
    prof->resident[c.device] = d;
    *out = d;
    return PSB_OK;
}

// general 32-bit path over (a subset of) the resident database, reading the subjects straight from
// the bit-packed store; results land in caller order.  With `d_count` the number of subset entries is
// read on the device (the 16-bit scan's re-run list), so no host synchronisation is needed to launch.
static int scan_general(const FnConfig &cfg, const parasail_profile *prof, DevProfile *dp, int open, int gap, psb_db *db,
                        const int *d_subset, int nsubset, const int *d_count, int *const d_out[6]) {
    Ctx &c = g_ctx;
    const HostMatrix &m = prof->matrix;
    const int lq = (int)prof->query.size();
    const bool pssm = m.type == PARASAIL_MATRIX_TYPE_PSSM;
    const bool fine = gotoh32_profile_ok(m.size, m.min, m.max, open, pssm);
    const ClassTable ct = class_table(fine);
    const int K = ct.k[class_of_len(ct, lq)];
    DevMem d_counter, d_bnd;
    PSB_TRY(d_counter.alloc(sizeof(int), c.stream));
    PSB_CUDA(cudaMemsetAsync(d_counter.p, 0, sizeof(int), c.stream));
    const bool wide = !(std::min(lq, db->maxlen) < 1024 && lq + db->maxlen < 4096) || !fine;
    // a re-run list is almost always empty or tiny: a small persistent grid serves any count
    const int nwork = d_count ? (int)std::min<int64_t>(nsubset, (int64_t)g_ctx.sms * 2 * kWarpsPerBlock) : (d_subset ? nsubset : (int)db->n);
    long long bnd_stride = 0;
    if (lq > 32 * K) {
        bnd_stride = (long long)db->maxlen * (2 + (cfg.stats ? (wide ? 4 : 2) : 0));
        PSB_TRY(d_bnd.alloc((size_t)(bnd_stride * max_grid_warps(nwork)) * sizeof(int), c.stream));
    }
    Gotoh32Params p;
    std::memset(&p, 0, sizeof(p));
    p.q = dp->d_query; p.q_off = dp->d_qoff;
    p.r_words = db->d_words; p.r_word_off = db->d_word_off; p.r_len = db->d_len; p.r_bits = db->bits;
    p.order = d_subset; p.n = d_subset ? nsubset : (int)db->n; p.n_dev = d_count; p.shared_query = 1;
    p.matrix = dp->d_matrix; p.size = m.size; p.is_pssm = pssm ? 1 : 0;
    p.open = open; p.gap = gap;
    p.mode = cfg.mode; p.s1_beg = cfg.s1_beg; p.s1_end = cfg.s1_end; p.s2_beg = cfg.s2_beg; p.s2_end = cfg.s2_end;
    p.score = d_out[0]; p.end_query = d_out[1]; p.end_ref = d_out[2];
    p.matches = d_out[3]; p.similar = d_out[4]; p.length = d_out[5];
    p.bnd = d_bnd.as<int>(); p.bnd_stride = bnd_stride;
    p.counter = d_counter.as<int>();
    p.out_map = db->d_perm;
    const Variant v = cfg.stats ? (wide ? V_STATS64 : V_STATS32) : V_SCORE;
    PSB_TRY(launch_gotoh32(K, v, p, nwork, fine));
    return PSB_OK;
}

// the packed 16-bit profile(s) for this gap-open penalty: built once per (device, open) and then shared
// read-only by every thread that scans with this profile (Profile: Send + Sync upstream).  Queries of more
// than 400 residues are cut into strips of equal height (at most 25 rows per lane each), one profile per
// strip: the scan then sweeps the database once per strip, handing the bottom row over through HBM.
static constexpr int kSw16StripRows = 400, kSw16MaxStrips = 16;
static bool sw16_prepare(const parasail_profile *prof, DevProfile *dp, int open, int gap, std::vector<Sw16Profile> *out) {
    Ctx &c = g_ctx;
    const HostMatrix &m = prof->matrix;
    if (m.type != PARASAIL_MATRIX_TYPE_SQUARE) return false;
    std::lock_guard<std::mutex> lk(prof->mu);
    auto it = dp->sw16.find(open);
    if (it != dp->sw16.end()) {
        *out = it->second;
        return !it->second.empty() && sw16_supported(it->second[0], open, gap);
    }
    const int lq = (int)dp->mapped.size();
    const int nstrips = (lq + kSw16StripRows - 1) / kSw16StripRows;
    std::vector<Sw16Profile> built;
    bool ok = nstrips >= 1 && nstrips <= kSw16MaxStrips;
    // every strip but the last is exactly 16*K rows high (its bottom row, the one handed over, must be a real
    // query row): the smallest of the strip classes whose nstrips strips cover the query
    int rows = lq;
    if (ok && nstrips > 1) {
        rows = 0;
        for (int k : {12, 16, 20, 25}) if (!rows && SW16_G * k * nstrips >= lq) rows = SW16_G * k;
        ok = rows > 0;
    }
    for (int st = 0; ok && st < nstrips; ++st) {
        const int r0 = st * rows, nr = std::min(rows, lq - r0);
        Sw16Profile np_;
        std::vector<int8_t> host;
        ok = nr > 0 && sw16_build_profile(dp->mapped.data() + r0, nr, m.table.data(), m.size, open, &np_, &host);
        if (!ok) break;
        np_.row0 = r0;
        if (cudaMallocAsync(&np_.prof, host.size(), c.stream) != cudaSuccess) { cudaGetLastError(); ok = false; break; }
        built.push_back(np_);
        if (cudaMemcpyAsync(np_.prof, host.data(), host.size(), cudaMemcpyHostToDevice, c.stream) != cudaSuccess) { ok = false; break; }
        cudaStreamSynchronize(c.stream);  // `host` goes out of scope; other streams may use the buffer from here on
    }
    if (!ok) {
        for (auto &sp : built) if (sp.prof) cudaFreeAsync(sp.prof, c.stream);
        built.clear();   // remembered: this penalty / query has no packed form
    }
    dp->sw16[open] = built;
    *out = built;
    return ok && sw16_supported(built[0], open, gap);
}

template <int K> static const void *sw16_fn_k() { return (const void *)sw16_scan_kernel<K>; }
template <int K> static const void *sw16_strip_fn_k() { return (const void *)sw16_scan_kernel<K, true>; }
static const void *sw16_fn(int K, bool strip = false) {
    if (strip) {
        switch (K) {
            case 4: return sw16_strip_fn_k<4>();
            case 8: return sw16_strip_fn_k<8>();
            case 12: return sw16_strip_fn_k<12>();
            case 16: return sw16_strip_fn_k<16>();
            case 20: return sw16_strip_fn_k<20>();
            case 25: return sw16_strip_fn_k<25>();
        }
        return nullptr;
    }
    switch (K) {
        case 4: return sw16_fn_k<4>();
        case 8: return sw16_fn_k<8>();
        case 12: return sw16_fn_k<12>();
        case 16: return sw16_fn_k<16>();
        case 20: return sw16_fn_k<20>();
        case 25: return sw16_fn_k<25>();
        case 28: return sw16_fn_k<28>();
        case 32: return sw16_fn_k<32>();
    }
    return nullptr;
}

static constexpr int kSw16WarpsPerBlock = SW16_WARPS_PER_BLOCK;

// measured scan rate (cell updates per second) per rows-per-lane class, exponentially averaged over the
// single-strip scan jobs of this process that were large enough to be meaningful
static std::atomic<double> g_sw16_rate[33];
static double sw16_rate_get(int K) {
    const double r = g_sw16_rate[K & 31].load(std::memory_order_relaxed);
    return r > 1e11 ? r : 4.9e12;
}
static void sw16_rate_update(int K, double cells, double ms) {
    if (cells < 2e9 || ms <= 0.05) return;
    const double now = cells / (ms * 1e-3), old = g_sw16_rate[K & 31].load(std::memory_order_relaxed);
    g_sw16_rate[K & 31].store(old > 1e11 ? 0.7 * old + 0.3 * now : now, std::memory_order_relaxed);
}

// packed 16-bit local scan of the whole database.  Subjects that leave the 16-bit range are
// re-run by the 32-bit per-pair kernel; subjects too long for 16-bit column indices go to the
// multi-pair wavefront kernel.  The sweep of one subject is serial in its length, and on an SM
// shared by sixteen ALU-bound warps a step takes ~0.6 us, so the longest subjects of a shard
// (7 000 aa in the UniProt-like distribution) bound the kernel at ~4 ms however small the shard
// is -- what limits strong scaling at 8 GPUs.  Those few subjects ("head") are therefore swept by
// a separate small launch of the same kernel, one warp per SM sub-partition on SMs it owns
// outright, beside the main launch.
//
// What one scan launches, decided before the first launch.  The database is sorted by decreasing length: the first
// nroute subjects go to the wavefront kernel, the next nhead to the head launch, the rest to the main launch.
struct ScanPlan {
    double rate = 0, est_ms = 0, long_len = 0;
    int64_t nroute = 0, nhead = 0;
    int64_t nshort = 0;     // subjects on the packed kernel (head included)
    bool multi = false;     // the query has several strips: one sweep of every subject per strip, no head
    bool general = false;   // more over-long subjects than the route takes: the whole job goes to scan_general
};
static ScanPlan plan_scan(const std::vector<Sw16Profile> &strips, int lq, const psb_db *db) {
    ScanPlan P;
    const int K = strips[0].K;
    P.multi = strips.size() > 1;
    // Keep a subject's serial sweep under ~40 % of the time the whole shard needs.  Both figures follow from
    // ONE quantity, the scan rate of this kernel class on this device, which is measured, not assumed: every
    // finished scan job updates it (scan_finish); 4.9 TCUPS is only the value before the first measurement.
    // A group step advances 64*K cells of one of the SM's 16 resident warps: step = 64*K*16*SMs / rate.
    P.rate = sw16_rate_get(K);
    P.est_ms = (double)lq * (double)db->residues / P.rate * 1e3;
    const double step_ms = 64.0 * K * 16.0 * g_ctx.sms / P.rate * 1e3;
    P.long_len = std::max(1024.0, 0.4 * P.est_ms / step_ms);
    while (P.nroute < (int64_t)db->top_len.size() && db->top_len[P.nroute] > 65535) ++P.nroute;
    int64_t nhead = P.nroute;
    while (nhead < (int64_t)db->top_len.size() && db->top_len[nhead] > P.long_len) ++nhead;
    P.nhead = std::min<int64_t>(((nhead - P.nroute + 3) / 4) * 4, std::max<int64_t>(0, (db->n - P.nroute) / 8 / 4 * 4));
    if (P.multi) P.nhead = 0;
    P.nshort = db->n - P.nroute;
    P.general = db->nlong > P.nroute;
    if (!P.general && debug_timing())
        std::fprintf(stderr, "[psb] sw16: n %lld residues %lld est %.2f ms long_len %.0f nroute %lld nhead %lld top %d\n", (long long)db->n,
                     (long long)db->residues, P.est_ms, P.long_len, (long long)P.nroute, (long long)P.nhead, db->top_len.empty() ? 0 : db->top_len[0]);
    return P;
}

// device buffers the launches of one scan share; freed in stream order when the scan returns
struct ScanBufs {
    DevMem retry, cnt;                     // the re-run list; counters: re-runs, main launch, head launch
    DevMem lbytes, loff, bnd, ctl, cand;   // routed subjects: their bytes, offsets and wavefront state
    DevMem bndA, bndB;                     // strip by strip: the bottom rows handed to the strip below
};

// what every packed launch of a scan fills alike: the profile (strip), penalties, database, outputs and re-run list
static Sw16Params sw16_base_params(const Sw16Profile &sp, int open, int gap, const psb_db *db, int *const d_out[6], ScanBufs &B) {
    Sw16Params p;
    std::memset(&p, 0, sizeof(p));
    p.prof = sp.prof; p.nletters = sp.nletters; p.lq = sp.lq; p.open = open; p.gap = gap; p.max_score = sp.max_score;
    p.words = db->d_words; p.bits = db->bits;
    p.score = d_out[0]; p.end_query = d_out[1]; p.end_ref = d_out[2];
    p.retry = B.retry.as<int>(); p.retry_count = B.cnt.as<int>();
    p.mul_one = 1u; p.mul_64k = 65536u;
    return p;
}
// the launch's subjects: sorted positions first .. first + n - 1
static void sw16_subjects(Sw16Params &p, const psb_db *db, int64_t first, int64_t n) {
    p.word_off = db->d_word_off + first; p.len = db->d_len + first; p.n = n; p.out_map = db->d_perm + first;
    p.sid_base = (int)first;
}

// CTA size of a packed launch: two CTAs of 8 warps when their profile copies fit an SM together, else one of 16
// (long queries with a protein alphabet: one 50 KB profile copy instead of two).  The kernel's shared-memory limit
// is first raised to the largest of both shapes and `other_smem`, the request of another launch of the kernel.
struct Sw16Shape { int wpb, per_sm; size_t smem; };
static int sw16_cta_shape(const void *fn, const Sw16Profile &sp, bool strip, size_t other_smem, Sw16Shape *out) {
    int wpb = kSw16WarpsPerBlock, per_sm = 0;
    size_t smem = sw16_smem_bytes(sp.nletters, sp.K, wpb, strip);
    const size_t smem16 = sw16_smem_bytes(sp.nletters, sp.K, 16, strip);
    PSB_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max(std::max(smem, other_smem), smem16)));
    PSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, wpb * 32, smem));
    if (per_sm * wpb < 16) {
        int per_sm16 = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm16, fn, 16 * 32, smem16) == cudaSuccess && per_sm16 * 16 > per_sm * wpb) {
            wpb = 16; per_sm = per_sm16; smem = smem16;
        } else cudaGetLastError();
    }
    *out = {wpb, std::max(per_sm, 1), smem};
    return PSB_OK;
}

// the subjects too long for the packed kernel's 16-bit column indices: unpacked to bytes and swept by the multi-pair
// wavefront kernel, then reduced into the results
static int launch_route(const FnConfig &cfg, const parasail_profile *prof, DevProfile *dp, int open, int gap, const psb_db *db,
                        const ScanPlan &P, int *const d_out[6], ScanBufs &B) {
    if (P.nroute == 0) return PSB_OK;
    Ctx &c = g_ctx;
    const HostMatrix &m = prof->matrix;
    const int lq = (int)prof->query.size();
    const int64_t nroute = P.nroute;
    std::vector<long long> loff(nroute + 1);
    loff[0] = 0;
    for (int64_t i = 0; i < nroute; ++i) loff[i + 1] = loff[i] + db->top_len[i];
    const int K = lq <= 64 ? 1 : 2;
    const int nstrips = (lq + 32 * K - 1) / (32 * K);
    PSB_TRY(B.lbytes.alloc((size_t)loff[nroute], c.stream));
    PSB_TRY(B.loff.alloc((size_t)(nroute + 1) * sizeof(long long), c.stream));
    PSB_TRY(B.bnd.alloc((size_t)nstrips * 2 * (size_t)loff[nroute] * sizeof(int), c.stream));
    PSB_TRY(B.ctl.alloc(((size_t)nroute * nstrips + 2) * sizeof(int), c.stream));
    PSB_TRY(B.cand.alloc((size_t)nroute * nstrips * 8 * sizeof(int), c.stream));
    PSB_CUDA(cudaMemcpyAsync(B.loff.p, loff.data(), (size_t)(nroute + 1) * sizeof(long long), cudaMemcpyHostToDevice, c.stream));
    PSB_CUDA(cudaMemsetAsync(B.ctl.p, 0, ((size_t)nroute * nstrips + 2) * sizeof(int), c.stream));
    PSB_CUDA(cudaStreamSynchronize(c.stream));  // `loff` is a host temporary
    launch_unpack_db(db, nullptr, nullptr, B.loff.as<long long>(), B.lbytes.as<uint8_t>(), nroute, (unsigned)std::min<int64_t>(nroute, 1024), 256,
                     c.stream);
    c.launches++;
    return launch_wave_subjects(cfg, m, dp->d_query, lq, dp->d_matrix, open, gap, B.lbytes.as<uint8_t>(), B.loff.as<long long>(), nroute,
                                db->d_perm, K, nstrips, B.bnd.as<int>(), B.ctl.as<int>(), B.cand.as<int>(), d_out);
}

// ---- queries of several strips: one sweep of the database per strip; the bottom row of a strip (T and Fh of both
// subjects of a word, one uint2 per column) goes through HBM to the strip below: 16 bytes per column and strip
// boundary against ~K*16*2.5 instructions of fill per column
static int launch_sw16_strips(const std::vector<Sw16Profile> &strips, int open, int gap, psb_db *db, const ScanPlan &P, int *const d_out[6],
                              ScanBufs &B) {
    if (P.nshort == 0 || !P.multi) return PSB_OK;
    Ctx &c = g_ctx;
    if (!db->d_res_off) {
        std::lock_guard<std::mutex> lk(db->mu);
        if (!db->d_res_off) {
            long long *ro = nullptr;
            PSB_CUDA(cudaMallocAsync(&ro, ((size_t)db->n + 1) * sizeof(long long), db->stream));
            if (db->stream != c.stream) PSB_CUDA(cudaStreamSynchronize(db->stream));
            DevMem d_tmp;
            PSB_TRY(exclusive_sum(db->d_len, ro, (int)db->n, d_tmp, c.stream));
            PSB_CUDA(cudaStreamSynchronize(c.stream));
            db->d_res_off = ro;
        }
    }
    PSB_TRY(B.bndA.alloc(((size_t)db->residues + 64) * sizeof(uint2), c.stream));
    PSB_TRY(B.bndB.alloc(((size_t)db->residues + 64) * sizeof(uint2), c.stream));
    for (size_t st = 0; st < strips.size(); ++st) {
        const Sw16Profile &ss = strips[st];
        Sw16Params p = sw16_base_params(ss, open, gap, db, d_out, B);
        sw16_subjects(p, db, P.nroute, P.nshort);
        p.res_off = db->d_res_off + P.nroute;
        p.bnd_in = st == 0 ? nullptr : ((st & 1) ? B.bndA.as<uint2>() : B.bndB.as<uint2>());
        p.bnd_out = st + 1 == strips.size() ? nullptr : ((st & 1) ? B.bndB.as<uint2>() : B.bndA.as<uint2>());
        p.row0 = ss.row0; p.merge = st > 0 ? 1 : 0;
        DevMem d_cnt_st;   // a work counter per launch
        PSB_TRY(d_cnt_st.alloc(sizeof(int), c.stream));
        PSB_CUDA(cudaMemsetAsync(d_cnt_st.p, 0, sizeof(int), c.stream));
        p.counter = d_cnt_st.as<int>();
        const void *fn = sw16_fn(ss.K, true);
        if (!fn) { set_error("sw16: no strip kernel for this query length"); return PSB_EUNSUPPORTED; }
        Sw16Shape s;
        PSB_TRY(sw16_cta_shape(fn, ss, true, 0, &s));
        const long long slots = ((P.nshort + 1) / 2 + 1) / 2;
        PSB_CUDA(launch_persistent(fn, &p, slots, s.wpb, s.smem, s.per_sm, c.sms, c.stream));
        c.launches++;
    }
    return PSB_OK;
}

// a single-strip query: the head launch on the compute stream, then the main launch on `main_stream`
static int launch_sw16(const Sw16Profile &sp, int open, int gap, const psb_db *db, const ScanPlan &P, int *const d_out[6], ScanBufs &B,
                       cudaStream_t main_stream) {
    if (P.nshort == 0 || P.multi) return PSB_OK;
    Ctx &c = g_ctx;
    Sw16Params p = sw16_base_params(sp, open, gap, db, d_out, B);
    const void *fn = sw16_fn(sp.K);
    if (!fn) { set_error("sw16: no kernel for this query length"); return PSB_EUNSUPPORTED; }
    // the head's CTAs request enough shared memory to be alone on their SMs
    const size_t smem_excl = std::max<size_t>(sw16_smem_bytes(sp.nletters, sp.K, 4), 150 * 1024);
    Sw16Shape s;
    PSB_TRY(sw16_cta_shape(fn, sp, false, smem_excl, &s));
    if (debug_timing()) std::fprintf(stderr, "[psb] sw16: K %d, %d warps per CTA, %d CTAs per SM, %zu B shared\n", sp.K, s.wpb, s.per_sm, s.smem);
    if (P.nhead > 0) {
        // head: the longest subjects, 4 warps per CTA (one per sub-partition), each CTA alone on
        // its SM (the shared-memory request keeps the main launch's CTAs away)
        Sw16Params h = p;
        sw16_subjects(h, db, P.nroute, P.nhead);
        h.counter = B.cnt.as<int>() + 2;
        const long long hslots = (P.nhead / 2 + 1) / 2;
        void *hargs[] = {&h};
        PSB_CUDA(cudaLaunchKernel(fn, dim3((unsigned)((hslots + 3) / 4)), dim3(4 * 32), hargs, smem_excl, c.stream));
        c.launches++;
    }
    const int64_t nrest = P.nshort - P.nhead;
    if (nrest > 0) {
        sw16_subjects(p, db, P.nroute + P.nhead, nrest);
        p.counter = B.cnt.as<int>() + 1;
        const long long slots = ((nrest + 1) / 2 + 1) / 2;  // a warp takes two items (four subjects) at a time
        PSB_CUDA(launch_persistent(fn, &p, slots, s.wpb, s.smem, s.per_sm, c.sms, main_stream));
        c.launches++;
    }
    return PSB_OK;
}

// re-run list: launched unconditionally with its length read on the device (usually zero), so the
// scan needs no host round trip in the middle; the count reaches the host with the results
static int launch_rerun(const FnConfig &cfg, const parasail_profile *prof, DevProfile *dp, int open, int gap, psb_db *db, const ScanPlan &P,
                        int *const d_out[6], ScanBufs &B, int64_t *n_retried, int *retried_host) {
    PSB_TRY(scan_general(cfg, prof, dp, open, gap, db, B.retry.as<int>(), (int)db->n, B.cnt.as<int>(), d_out));
    PSB_CUDA(cudaMemcpyAsync(retried_host, B.cnt.p, sizeof(int), cudaMemcpyDeviceToHost, g_ctx.stream));
    *n_retried = P.nroute;   // + *retried_host once the stream has been synchronised
    return PSB_OK;
}

static int scan_sw16(const FnConfig &cfg, const parasail_profile *prof, DevProfile *dp, const std::vector<Sw16Profile> &strips, int open, int gap, psb_db *db,
                     int *const d_out[6], int64_t *n_retried, int *retried_host) {
    Ctx &c = g_ctx;
    const ScanPlan P = plan_scan(strips, (int)prof->query.size(), db);
    if (P.general) {
        // more over-long subjects than the routed head covers: not a workload for the packed kernel
        *n_retried = db->n;
        return scan_general(cfg, prof, dp, open, gap, db, nullptr, 0, nullptr, d_out);
    }
    ScanBufs B;
    PSB_TRY(B.retry.alloc(((size_t)db->n * strips.size() + 2) * sizeof(int), c.stream));
    PSB_TRY(B.cnt.alloc(4 * sizeof(int), c.stream));
    PSB_CUDA(cudaMemsetAsync(B.cnt.p, 0, 4 * sizeof(int), c.stream));
    // The launches that must own their SMs (wavefront strips, head) go on the compute stream, where
    // they start the moment the preceding work ends; the main launch goes on the side stream behind an
    // event, so it reaches the SMs after them.  The other way round, a busy queue lets the main
    // launch's persistent CTAs take every SM first and the head then runs alone AFTER it.
    const bool forked = P.nroute > 0 || P.nhead > 0;
    if (forked) {
        PSB_CUDA(cudaEventRecord(c.ev_fork, c.stream));
        PSB_CUDA(cudaStreamWaitEvent(c.side, c.ev_fork, 0));
    }
    PSB_TRY(launch_route(cfg, prof, dp, open, gap, db, P, d_out, B));
    PSB_TRY(launch_sw16_strips(strips, open, gap, db, P, d_out, B));
    PSB_TRY(launch_sw16(strips[0], open, gap, db, P, d_out, B, forked ? c.side : c.stream));
    if (forked) {
        PSB_CUDA(cudaEventRecord(c.ev_join, c.side));
        PSB_CUDA(cudaStreamWaitEvent(c.stream, c.ev_join, 0));
    }
    return launch_rerun(cfg, prof, dp, open, gap, db, P, d_out, B, n_retried, retried_host);
}

// the packed 16-bit scan serves this function (if its profile can be packed): local score-only at 8/16 bit or "sat"
bool sw16_wanted(const FnConfig &cfg) { return cfg.mode == MODE_SW && !cfg.stats && cfg.width != 32 && cfg.width != 64; }
int scan_enqueue(ScanJob &job, const FnConfig &cfg, const parasail_profile *profile, int open, int gap, psb_db *db,
                        int *const hosts[6], int64_t host_base) {
    Ctx &c = g_ctx;
    DevProfile *dp = nullptr;
    PSB_TRY(get_dev_profile(profile, &dp));
    int *outp[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    const int nout = cfg.stats ? 6 : 3;
    for (int k = 0; k < nout; ++k) { PSB_TRY(job.d_out[k].alloc((size_t)db->n * sizeof(int), c.stream)); outp[k] = job.d_out[k].as<int>(); }
    job.retried_host = (int *)pinned_alloc(64);
    if (!job.retried_host) { set_error("pinned host allocation failed"); return PSB_ENOMEM; }
    *job.retried_host = 0;
    PSB_CUDA(cudaEventCreate(&job.ev0));
    PSB_CUDA(cudaEventCreate(&job.ev1));
    PSB_CUDA(cudaEventRecord(job.ev0, c.stream));
    std::vector<Sw16Profile> sp16;
    const bool fast = sw16_wanted(cfg) && sw16_prepare(profile, dp, open, gap, &sp16);
    int rc;
    if (fast && sp16.size() == 1 && db->nlong == 0) { job.rate_k = sp16[0].K; job.rate_cells = (double)profile->query.size() * (double)db->residues; }
    if (fast) rc = scan_sw16(cfg, profile, dp, sp16, open, gap, db, outp, &job.retried, job.retried_host);
    else rc = scan_general(cfg, profile, dp, open, gap, db, nullptr, 0, nullptr, outp);
    if (rc != PSB_OK) { cudaStreamSynchronize(c.stream); return rc; }
    PSB_CUDA(cudaEventRecord(job.ev1, c.stream));
    for (int k = 0; k < nout && hosts; ++k)
        PSB_CUDA(cudaMemcpyAsync(hosts[k] + host_base, job.d_out[k].p, (size_t)db->n * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    PSB_CUDA(cudaEventCreateWithFlags(&job.done, cudaEventDisableTiming));
    PSB_CUDA(cudaEventRecord(job.done, c.stream));
    return PSB_OK;
}
// the query side, while the compute stream is idle: a profile's first use on a device uploads it and waits for that
// upload, which would otherwise happen inside the first piece's scan_enqueue, behind that piece's whole chain
int prepare_query(const FnConfig &cfg, const parasail_profile_t *profile, int open, int gap) {
    DevProfile *dp = nullptr;
    PSB_TRY(get_dev_profile(profile, &dp));
    std::vector<Sw16Profile> sp;
    if (sw16_wanted(cfg)) sw16_prepare(profile, dp, open, gap, &sp);
    return PSB_OK;
}
// waits until the job's results are on the host
int scan_finish(ScanJob &job) {
    Ctx &c = g_ctx;
    if (job.finished) return PSB_OK;
    job.finished = true;
    cudaError_t e = job.done ? cudaEventSynchronize(job.done) : cudaStreamSynchronize(c.stream);
    if (e != cudaSuccess) { set_error(std::string("psb_scan: ") + cudaGetErrorString(e)); return PSB_ECUDA; }
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, job.ev0, job.ev1) == cudaSuccess) c.last_ms += ms;
    if (debug_timing()) std::fprintf(stderr, "[psb] scan job: %.3f ms, %d re-run at 32 bit\n", ms, *job.retried_host);
    if (job.rate_k > 0) sw16_rate_update(job.rate_k, job.rate_cells, ms);
    job.retried += *job.retried_host;
    return PSB_OK;
}
// what every entry point that runs a profile against a database checks first: a profile function name and a profile
int profile_fn_check(const char *who, const char *fn_name, const parasail_profile_t *profile, FnConfig *cfg) {
    if (!parse_fn_name(fn_name, cfg) || !cfg->profile) { set_error(std::string(who) + ": not a profile function name: " + (fn_name ? fn_name : "(null)")); return PSB_EINVAL; }
    if (!profile) { set_error(std::string(who) + ": NULL profile"); return PSB_EINVAL; }
    return PSB_OK;
}
// and a scan, which produces no traceback
int scan_check(const char *who, const char *fn_name, const parasail_profile_t *profile, FnConfig *cfg) {
    PSB_TRY(profile_fn_check(who, fn_name, profile, cfg));
    if (cfg->trace || cfg->table || cfg->rowcol) { set_error(std::string(who) + ": trace/table/rowcol outputs are not available for database scans"); return PSB_EUNSUPPORTED; }
    return PSB_OK;
}
// a profile run against a resident database: the calling thread's device holds it, and both use the same alphabet
int profile_db_check(const char *who, const parasail_profile_t *profile, const psb_db *db) {
    PSB_TRY(ensure_ctx());
    if (db->device != g_ctx.device) { set_error(std::string(who) + ": database lives on another device"); return PSB_EINVAL; }
    return profile_alphabet_check(who, profile, db);
}
int profile_alphabet_check(const char *who, const parasail_profile_t *profile, const psb_db *db) {
    if (profile->matrix.size != db->msize || std::memcmp(profile->matrix.mapper, db->mapper, 256) != 0) {
        set_error(std::string(who) + ": profile and database were built with different alphabets");
        return PSB_EINVAL;
    }
    return PSB_OK;
}

}  // namespace psb

using namespace psb;

extern "C" {

int psb_scan(const char *fn_name, const parasail_profile_t *profile, int open, int gap, const psb_db_t *db_c, psb_batch_t **out) {
    if (out) *out = nullptr;
    FnConfig cfg;
    PSB_TRY(scan_check("psb_scan", fn_name, profile, &cfg));
    if (!db_c || !out) { set_error("psb_scan: NULL argument"); return PSB_EINVAL; }
    psb_db *db = const_cast<psb_db *>(db_c);
    PSB_TRY(profile_db_check("psb_scan", profile, db));
    Ctx &c = g_ctx;
    c.last_ms = 0.0; c.launches = 0;
    psb_batch_t *b = new_batch(db->n, cfg);
    if (!b) { set_error("pinned host allocation failed"); return PSB_ENOMEM; }
    ScanJob job;
    int rc = scan_enqueue(job, cfg, profile, open, gap, db, batch_outputs(b).data(), 0);
    if (rc == PSB_OK) rc = scan_finish(job);
    if (rc != PSB_OK) { cudaStreamSynchronize(c.stream); free_batch(b); return rc; }
    b->n_retried = job.retried;
    return scan_batch_done(cfg, profile, open, gap, db->residues, [&](int64_t i) { return db->host_len.empty() ? db->maxlen : db->host_len[(size_t)i]; }, b, out);
}

int psb_db_align(const char *fn_name, const parasail_profile_t *profile, int open, int gap, const psb_db_t *db_c,
                 const int64_t *ids, int64_t n, psb_batch_t **out) {
    if (out) *out = nullptr;
    FnConfig cfg;
    PSB_TRY(profile_fn_check("psb_db_align", fn_name, profile, &cfg));
    if (cfg.table || cfg.rowcol) { set_error("psb_db_align: _table/_rowcol outputs exist only on the single-pair API"); return PSB_EUNSUPPORTED; }
    if (!db_c || !out) { set_error("psb_db_align: NULL argument"); return PSB_EINVAL; }
    psb_db *db = const_cast<psb_db *>(db_c);
    PSB_TRY(db_check("psb_db_align", db));
    PSB_TRY(profile_db_check("psb_db_align", profile, db));
    if (n <= 0 || (!ids && n != db->n)) {
        set_error("psb_db_align: " + std::to_string(n) + " ids for a database of " + std::to_string(db->n) + " subjects");
        return PSB_EINVAL;
    }
    // the pairs pass classifies, sorts and cuts by the references' lengths: offsets from the caller-order lengths
    std::vector<int> rid((size_t)n);
    std::vector<int64_t> r_off((size_t)n + 1);
    r_off[0] = 0;
    for (int64_t i = 0; i < n; ++i) {
        const int64_t id = ids ? ids[i] : i;
        if (id < 0 || id >= db->n) {
            set_error("psb_db_align: ids[" + std::to_string(i) + "] = " + std::to_string(id) + " is not a subject of a database of " + std::to_string(db->n));
            return PSB_EINVAL;
        }
        rid[(size_t)i] = (int)id;
        r_off[(size_t)i + 1] = r_off[(size_t)i] + db->host_len[(size_t)id];
    }
    int first_use = 0;
    PSB_TRY(db_inv_perm(db, &first_use));
    const int64_t lq = (int64_t)profile->query.size();
    const int64_t q_off[2] = {0, lq};
    PairsRequest req;
    req.cfg = cfg;
    req.matrix = &profile->matrix; req.open = open; req.gap = gap;
    req.q_cat = profile->query.data(); req.q_off = q_off; req.shared_query = true;
    req.r_off = r_off.data(); req.n = n; req.r_db = db; req.r_ids = rid.data();
    const int rc = run_pairs(req, out);
    g_ctx.launches += first_use;
    if (rc == PSB_OK) flag_saturated(cfg, profile->matrix, open, gap, *out, [&](int64_t i) { return std::make_pair((int)lq, span(r_off.data(), i)); });
    return rc;
}
}  // extern "C"
