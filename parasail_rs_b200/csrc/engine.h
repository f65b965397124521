// engine.h -- the host plumbing that the engine's translation units share.  No CPU fallback exists: every entry
// point fails with PSB_ENODEV / PSB_ECUDA (and psb_last_error text) when the device is unusable.
//
//   ctx.cu        the thread's context, device buffers, uploads, page-locked and staging pools, batches, resident
//                 worker threads, the small C entry points
//   wave32.cu     one long pair, or the scan's routed subjects, over the whole GPU (kern_wave32.cuh)
//   pairs.cu      the pairs pass: psb_align_pairs (SURVEY configs C1/C3/C4), psb_align_pairs_banded, and the
//                 kernels of kern_band32.cuh and kern_util.cuh
//   db.cu         the resident database: construction, psb_db_* and its sort/scan primitives (cub)
//   scan.cu       a resident profile against a resident database: psb_scan (C2), psb_db_align (kern_sw16.cuh), and
//                 the one-warp-per-pair 32-bit kernels (kern_gotoh32.cuh)
//   host_scan.cu  the scan of a database in host memory: psb_scan_host, psb_scan_box
//   pairs16.cu    the packed 16-bit many-pairs kernels (pairs16_host.h)
//
// Each kernel (cub's included) is instantiated in exactly one of them; another file that launches it calls a launcher
// declared here.
// parasail-rs's per-pair Aligner::align [REF src/aligner/mod.rs:397-452] arrives as an n = 1 batch (result.cpp).
#pragma once
#include <cuda_runtime.h>

#include <array>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "psb_db.h"
#include "psb_defs.h"
#include "psb_internal.h"

namespace psb {

struct Gotoh32Params;   // kern_gotoh32.cuh

// ---- per-host-thread context ----------------------------------------------------------------
struct Ctx {
    bool ready = false;
    int device = -1;          // -1: take the current CUDA device on first use
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaStream_t side = nullptr;          // long subjects of a scan run here, beside the main kernel
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaStream_t copy = nullptr;          // host->device uploads of psb_scan_host, beside the kernels
    cudaEvent_t ev_alloc = nullptr;
    int sms = 0;
    double last_ms = 0.0;
    int launches = 0;
    // the big per-pass buffers of psb_align_pairs (decision bytes, CIGAR scratch): kept by the thread from pass to
    // pass of one batch and only grown, so that a lane working through sixteen passes does not put sixteen
    // multi-gigabyte allocations through the stream-ordered pool (KeptMem below)
    struct Kept { void *p = nullptr; size_t cap = 0; } kept[3];
    // two page-locked bounce buffers for uploads out of pageable caller memory (upload_h2d below)
    void *bounce[2] = {nullptr, nullptr};
    cudaEvent_t bounce_free[2] = {nullptr, nullptr};
    int bounce_next = 0;
};
extern thread_local Ctx g_ctx;
// binds the calling thread to its device and creates its streams and events on first use
int ensure_ctx();

#define PSB_CUDA(call)                                                                         \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess) {                                                                \
            set_error(std::string(#call) + ": " + cudaGetErrorString(e_));                      \
            return PSB_ECUDA;                                                                   \
        }                                                                                       \
    } while (0)

// stream-ordered device buffer (RAII)
struct DevMem {
    void *p = nullptr;
    size_t bytes = 0;
    cudaStream_t s = nullptr;
    DevMem() = default;
    DevMem(const DevMem &) = delete;
    DevMem &operator=(const DevMem &) = delete;
    ~DevMem() { release(); }
    int alloc(size_t n, cudaStream_t stream) {
        release();
        s = stream; bytes = n;
        if (n == 0) n = 16;
        cudaError_t e = cudaMallocAsync(&p, n, stream);
        if (e != cudaSuccess) {
            p = nullptr;
            set_error(std::string("cudaMallocAsync(") + std::to_string(n) + "): " + cudaGetErrorString(e));
            return e == cudaErrorMemoryAllocation ? PSB_ENOMEM : PSB_ECUDA;
        }
        return PSB_OK;
    }
    void release() {
        if (p) cudaFreeAsync(p, s);
        p = nullptr;
    }
    template <typename T> T *as() const { return (T *)p; }
};
#define PSB_TRY(expr) do { int rc_ = (expr); if (rc_ != PSB_OK) return rc_; } while (0)

// DevMem's interface over one of the thread's kept slots: alloc() reuses the slot's block when it is large enough
// and replaces it otherwise; nothing is freed when the object goes out of scope (release_kept does that, at the end
// of the batch)
struct KeptMem {
    int slot;
    void *p = nullptr;
    explicit KeptMem(int s) : slot(s) {}
    int alloc(size_t n, cudaStream_t stream) {
        Ctx::Kept &k = g_ctx.kept[slot];
        if (k.cap < n || !k.p) {
            if (k.p) cudaFreeAsync(k.p, stream);
            k.p = nullptr; k.cap = 0;
            const size_t want = n + n / 8 + 256;
            cudaError_t e = cudaMallocAsync(&k.p, want, stream);
            if (e != cudaSuccess) {
                k.p = nullptr;
                set_error(std::string("cudaMallocAsync(") + std::to_string(want) + "): " + cudaGetErrorString(e));
                return e == cudaErrorMemoryAllocation ? PSB_ENOMEM : PSB_ECUDA;
            }
            k.cap = want;
        }
        p = k.p;
        return PSB_OK;
    }
    template <typename T> T *as() const { return (T *)p; }
};
void release_kept();

// PSB_DEBUG_TIMING is set: the engine's "[psb]" lines on stderr and the device timelines behind them
inline bool debug_timing() { return std::getenv("PSB_DEBUG_TIMING") != nullptr; }

// ---- ctx.cu -------------------------------------------------------------------------------------
// host->device copy that does not depend on the caller's memory being page-locked
cudaError_t upload_h2d(void *dst, const void *src, size_t bytes, cudaStream_t stream);
bool is_pageable(const void *p);
// page-locked host blocks, recycled process-wide by size class
void *pinned_alloc(size_t bytes);
void pinned_free(void *p, size_t bytes);
// device staging blocks of psb_scan_host's uploads, recycled process-wide (plain allocations, not stream-ordered)
void *stage_acquire(int device, size_t need, size_t *got);
void stage_release(int device, void *p, size_t bytes);
// what a new device allocation can get (0 if the driver cannot say)
size_t device_mem_available();
psb_batch_t *new_batch(int64_t n, const FnConfig &cfg);
std::array<int *, 6> batch_outputs(psb_batch_t *b);
int span(const int64_t *off, int64_t i);
void fill_lut(unsigned *lut, const uint8_t *mapper);

struct BatchImpl {
    std::vector<std::pair<void *, size_t>> blocks;
    void *take(size_t bytes) {
        void *p = pinned_alloc(bytes);
        if (p) blocks.emplace_back(p, bytes);
        return p;
    }
};

// explicit _8/_16 widths: the pairs whose values do not fit are flagged and their results zeroed (SURVEY A.8), by the
// rule of saturates(); `lens(i)` is pair i's (query, reference) lengths
template <typename Lens>
void flag_saturated(const FnConfig &cfg, const HostMatrix &hm, int open, int gap, psb_batch_t *b, Lens lens) {
    if (cfg.width != 8 && cfg.width != 16) return;
    for (int64_t i = 0; i < b->n; ++i) {
        const std::pair<int, int> l = lens(i);
        if (saturates(cfg, hm, b->score[i], l.first, l.second, open, gap)) {
            b->saturated[i] = 1; b->score[i] = 0; b->end_query[i] = 0; b->end_ref[i] = 0;
        }
    }
}

// the free ends of a traceback or a packed profile: the top edge when local, or semi-global with s1_beg; the left edge
// when local, or semi-global with s2_beg.  `md`: a FnConfig or a Gotoh32Params
struct FreeEnds { bool top, left; };
template <typename Mode> FreeEnds free_ends(const Mode &md) {
    const bool sw = md.mode == MODE_SW, sg = md.mode == MODE_SG;
    return {sw || (sg && md.s1_beg), sw || (sg && md.s2_beg)};
}

// ---- scan.cu: the one-warp-per-pair 32-bit kernels --------------------------------------------------
static constexpr int kNumClass = 13;   // upper bound on classes of either family
struct ClassTable { const int *k; int n; };
ClassTable class_table(bool fine);
int class_of_len(const ClassTable &t, int lq);

enum Variant { V_SCORE = 0, V_STATS32, V_STATS64, V_TRACE, V_TABLE };

static constexpr int kWarpsPerBlock = 4;

int launch_gotoh32(int K, Variant v, Gotoh32Params &p, int nwork, bool prof, long long *grid_warps_out = nullptr);
long long max_grid_warps(long long nwork);

// ---- wave32.cu: one long pair over the whole GPU --------------------------------------------------
static constexpr int kWaveMinLq = 2048;   // below this the per-pair kernel is used

// Long pairs WITH traceback or statistics: the TRACE instantiation of the column-blocked generation leaves 1.25
// bytes per cell (H low bytes + gap open/extend bits) and walk32_kernel follows the path (kern_wave32.cuh).
struct WaveWalk {
    bool stats;                   // count (matches, similar, length) instead of emitting CIGAR runs
    unsigned *rev_ops;
    const long long *rev_off;
    int *nops, *beg_query, *beg_ref;
};

// PSB_DEBUG_TIMING on the pairs path (inert without it): where the host time of a pass goes, the device time of its
// marked launches and its timed region, as "[psb]" lines on stderr (tools/pairs_host_probe.py and
// tools/db_align_probe.py read them).  One per pass, on the calling thread's stream.
struct PassTimeline {
    const bool on = debug_timing();
    std::chrono::steady_clock::time_point h_last = std::chrono::steady_clock::now();
    std::string h_line;
    struct Mark { std::string what; cudaEvent_t begin, end; };
    std::vector<Mark> marks;
    PassTimeline() = default;
    PassTimeline(const PassTimeline &) = delete;
    PassTimeline &operator=(const PassTimeline &) = delete;
    ~PassTimeline() {
        for (Mark &k : marks) { cudaEventDestroy(k.begin); if (k.end) cudaEventDestroy(k.end); }
    }
    void phase(const char *what) {
        if (!on) return;
        const auto now = std::chrono::steady_clock::now();
        char buf[64];
        std::snprintf(buf, sizeof buf, " %s %.3f", what, std::chrono::duration<double, std::milli>(now - h_last).count());
        h_line += buf; h_last = now;
    }
    static cudaEvent_t record() {
        cudaEvent_t ev = nullptr;
        cudaEventCreate(&ev);
        cudaEventRecord(ev, g_ctx.stream);
        return ev;
    }
    void begin(std::string what) { if (on) marks.push_back({std::move(what), record(), nullptr}); }
    void end() { if (on) marks.back().end = record(); }
    // the device time of the last mark, taken off the list (waits for it)
    float take_last_ms() {
        const Mark k = marks.back();
        marks.pop_back();
        float t = 0.f;
        cudaEventSynchronize(k.end);
        cudaEventElapsedTime(&t, k.begin, k.end);
        cudaEventDestroy(k.begin); cudaEventDestroy(k.end);
        return t;
    }
    void report(int64_t lo, int64_t hi, float ms) const {
        if (!on) return;
        std::fprintf(stderr, "[psb] pass %lld..%lld host ms:%s\n", (long long)lo, (long long)hi, h_line.c_str());
        for (const Mark &k : marks) {
            float t = 0.f;
            if (k.end && cudaEventElapsedTime(&t, k.begin, k.end) == cudaSuccess)
                std::fprintf(stderr, "[psb] %-48s %9.3f ms\n", k.what.c_str(), t);
        }
        std::fprintf(stderr, "[psb] pass of %lld pairs: timed region %.3f ms\n", (long long)(hi - lo), ms);
    }
};

// preconditions of the traced wavefront launch for one long pair (psb_align_pairs with traceback or statistics)
bool wave_walk_ok(const HostMatrix &m, int open, int gap, bool is_sw, int lq, int lr, size_t avail);
// one long pair of the pass's Gotoh32Params (byte offsets relative to its biased q / r), result at `out_index`; with
// `ww` the traced launch and the walk
int launch_wave32(const Gotoh32Params &g, const HostMatrix &m, long long q_byte_off, int lq, long long r_byte_off, int lr, int out_index,
                  const WaveWalk *ww, PassTimeline &tl);
// the scan's routed subjects: `nroute` subjects of bytes `lbytes` at offsets `loff` against the query `q`, swept by one
// multi-pair launch of K rows per lane (`nstrips` strips per subject) and reduced into d_out through `out_map`
int launch_wave_subjects(const FnConfig &cfg, const HostMatrix &m, const uint8_t *q, int lq, const int *matrix, int open, int gap,
                         const uint8_t *lbytes, const long long *loff, int64_t nroute, const int *out_map, int K, int nstrips, int *bnd, int *ctl,
                         int *cand, int *const d_out[6]);

// ---- pairs.cu: the pairs pass, and the launchers of the kernels of kern_util.cuh that other files use ---------
// host threads that work through the passes of a large batch side by side.  Measured on 10^6 pairs (tools/
// pairs_host_probe.py; one lane / two / three): sw_trace 250 x 250: 106 / 50 / 47 ms, nw 250 x 250: 45 / 23.7 / 21.8 ms,
// sg_stats 150 x 500: 68 / 34 / 36 ms.  A third lane buys at most 8 % and another set of multi-gigabyte decision
// buffers; two it is.
static constexpr int kPairLanes = 2;
// subjects of a resident database unpacked to matrix codes: `ids` (nullptr: sorted positions 0 .. n-1; with `inv_perm`,
// caller ids) to out + out_off[i]
void launch_unpack_db(const psb_db *db, const int *ids, const int *inv_perm, const long long *out_off, uint8_t *out, long long n, unsigned grid,
                      unsigned block, cudaStream_t stream);
struct DbBuild;
// the packing of a database build's residues (db_finish)
void launch_pack_db(const DbBuild &B, unsigned grid, unsigned block, size_t smem, cudaStream_t stream);
// a database's inverse permutation (db_inv_perm)
void launch_invert_perm(const int *perm, long long n, int *inv, unsigned grid, unsigned block, cudaStream_t stream);

// ---- db.cu: the resident database ------------------------------------------------------------------
struct DbBuild {
    psb_db *db = nullptr;
    DevMem d_raw, d_off, d_len0, d_idx0, d_wcount, d_tmp;
    // copy-stream uploads use recycled staging blocks instead of d_raw / d_off
    void *st_raw = nullptr, *st_off = nullptr;
    size_t st_raw_bytes = 0, st_off_bytes = 0;
    int st_device = 0;
    cudaEvent_t offs_up = nullptr;   // copy stream: the offsets have landed (enough for lengths / sort / word offsets)
    cudaEvent_t res_begin = nullptr; // copy stream: the residue copy begins (timing, feeds the measured upload rate)
    cudaEvent_t uploaded = nullptr;  // copy stream: the residues have landed too
    cudaEvent_t packed = nullptr;    // compute stream: this piece's sort/pack chain has run (gates the next piece's residue upload)
    cudaStream_t up = nullptr;     // the stream the uploads were queued on
    long long raw_base = 0;
    unsigned lut[64];
    uint8_t *raw() const { return st_raw ? (uint8_t *)st_raw : d_raw.as<uint8_t>(); }
    long long *offs() const { return st_off ? (long long *)st_off : d_off.as<long long>(); }
    DbBuild() = default;
    DbBuild(const DbBuild &) = delete;
    DbBuild &operator=(const DbBuild &) = delete;
    // the owner synchronises the streams that used the staging blocks before destroying this
    ~DbBuild() {
        if (uploaded) cudaEventDestroy(uploaded);
        if (offs_up) cudaEventDestroy(offs_up);
        if (res_begin) cudaEventDestroy(res_begin);
        if (packed) cudaEventDestroy(packed);
        stage_release(st_device, st_raw, st_raw_bytes);
        stage_release(st_device, st_off, st_off_bytes);
    }
};

// Phase A1 of a database build: the device-side object and the host->device copies
psb_db *db_upload(DbBuild &B, const uint8_t *cat, const int64_t *off, int64_t n, const HostMatrix &hm, bool use_copy_stream, int force_bits = 0,
                  cudaEvent_t residues_after = nullptr);
// Phase A2: the host pass over the offsets and the remaining device allocations
int db_host_pass(DbBuild &B, const int64_t *off);
struct StreamMarks;
// Phase B: lengths, sort, word offsets and packing on the compute stream; `marks`: psb_scan_host's timeline, or nullptr
int db_finish(DbBuild &B, StreamMarks *marks = nullptr);
int host_db_check(const char *who, const void *arg, const uint8_t *cat, const int64_t *off, int64_t n, bool scan);
int db_check(const char *who, const psb_db *db);
int db_inv_perm(psb_db *db, int *launched);
// exclusive prefix sum of `n` ints into long longs on `stream`, its scratch in `tmp` (cub's scan, instantiated in db.cu)
int exclusive_sum(int *in, long long *out, int n, DevMem &tmp, cudaStream_t stream);

// PSB_DEBUG_TIMING on psb_scan_host (inert without it): a device-side timeline, one event per mark on the stream
// named, reported relative to the first mark
struct StreamMarks {
    const bool on = debug_timing();
    std::vector<cudaEvent_t> ev;
    StreamMarks() = default;
    StreamMarks(const StreamMarks &) = delete;
    StreamMarks &operator=(const StreamMarks &) = delete;
    ~StreamMarks() { for (cudaEvent_t e : ev) cudaEventDestroy(e); }
    void mark(cudaStream_t st) {
        cudaEvent_t e;
        if (on && cudaEventCreate(&e) == cudaSuccess) { cudaEventRecord(e, st); ev.push_back(e); }
    }
    std::string line() const {
        std::string out;
        for (size_t i = 1; i < ev.size(); ++i) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, ev[0], ev[i]);
            char buf[32]; std::snprintf(buf, sizeof buf, " %.3f", ms); out += buf;
        }
        return out;
    }
};

// ---- scan.cu: a resident profile against a resident database -----------------------------------------
bool sw16_wanted(const FnConfig &cfg);
// the query side of a scan, queued while the compute stream is idle: the profile's device copy and packed form
int prepare_query(const FnConfig &cfg, const parasail_profile_t *profile, int open, int gap);
int scan_check(const char *who, const char *fn_name, const parasail_profile_t *profile, FnConfig *cfg);

// one scan of a resident database, in two halves so that psb_scan_host can do host work for the next
// piece while this one runs: scan_enqueue issues the kernels and the device->host copies of the
// per-subject results (to hosts[k] + host_base); scan_finish waits for them.
struct ScanJob {
    DevMem d_out[6];
    int64_t retried = 0;
    int *retried_host = nullptr;   // pinned
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, done = nullptr;   // kernels begin / end, results on the host
    int rate_k = 0;          // > 0: a single-strip packed scan of `rate_cells` cells (feeds the measured rate)
    double rate_cells = 0;
    bool finished = false;   // scan_finish has run
    ScanJob() = default;
    ScanJob(const ScanJob &) = delete;
    ScanJob &operator=(const ScanJob &) = delete;
    ~ScanJob() {
        if (retried_host) pinned_free(retried_host, 64);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (done) cudaEventDestroy(done);
    }
};

int scan_enqueue(ScanJob &job, const FnConfig &cfg, const parasail_profile *profile, int open, int gap, psb_db *db, int *const hosts[6],
                 int64_t host_base);
int scan_finish(ScanJob &job);

// the end of a scan entry point: the batch's cells, the flags of explicit _8 / _16 widths, and the batch handed over;
// `subject_len(i)` is subject i's length
template <typename SubjectLen>
int scan_batch_done(const FnConfig &cfg, const parasail_profile_t *profile, int open, int gap, int64_t residues, SubjectLen subject_len,
                           psb_batch_t *b, psb_batch_t **out) {
    const int lq = (int)profile->query.size();
    b->cells = (double)profile->query.size() * (double)residues;
    flag_saturated(cfg, profile->matrix, open, gap, b, [&](int64_t i) { return std::make_pair(lq, subject_len(i)); });
    *out = b;
    return PSB_OK;
}

// one piece of a host scan (host_scan.cu): its uploads and packed shard, and its scan.  Destroying it gives the packed
// shard, the staging blocks and the result arrays back; the owner has synchronised the streams that used them.
struct HostPiece {
    DbBuild build;
    ScanJob job;
    ~HostPiece() { psb_db_free(build.db); }
};

// ---- resident worker threads: one per device for psb_scan_box, and the lanes of the pairs pass.  The thread keeps
// its context (streams, memory pool, staging blocks) warm across calls --------------------------------------------
struct BoxWorker {
    int device = 0;
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::function<void()> job;
    bool has_job = false, quit = false;
    std::unique_ptr<HostPiece> left;   // device memory of the last piece of the call just reported: given back after the report
    void loop() {
        psb_set_device(device);
        std::unique_lock<std::mutex> lk(mu);
        for (;;) {
            cv.wait(lk, [&] { return has_job || quit; });
            if (quit) return;
            std::function<void()> j = std::move(job);
            lk.unlock();
            j();
            lk.lock();
            has_job = false;
            cv.notify_all();
            lk.unlock();
            left.reset();   // off the caller's critical path (about 0.1 ms of frees and event destruction)
            lk.lock();
        }
    }
    void submit(std::function<void()> j) {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return !has_job; });
        job = std::move(j); has_job = true;
        cv.notify_all();
    }
    void wait() {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return !has_job; });
    }
};
// a new resident worker thread bound to `device`; it lives as long as the process
BoxWorker *start_worker(int device);
// the worker of lane `lane` of the pairs pass on `device`, started on first use
BoxWorker *pair_lane(int device, int lane);

}  // namespace psb
