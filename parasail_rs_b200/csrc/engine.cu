// engine.cu -- host side of the GPU path: device context, batching, kernel launches, the
// resident database and the resident query profile.  No CPU fallback exists: every entry
// point fails with PSB_ENODEV / PSB_ECUDA (and psb_last_error text) when the device is unusable.
//
// Batch entry points: psb_align_pairs (many pairs, SURVEY configs C1/C3/C4) and psb_scan (one
// resident profile vs a resident packed database, C2).  parasail-rs's per-pair
// Aligner::align [REF src/aligner/mod.rs:397-452] arrives here as an n = 1 batch (result.cpp).
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <memory>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <map>
#include <mutex>
#include <limits>
#include <numeric>
#include <condition_variable>
#include <functional>
#include <string>
#include <thread>
#include <future>
#include <vector>

#include "kern_band32.cuh"
#include "kern_gotoh32.cuh"
#include "kern_sw16.cuh"
#include "kern_util.cuh"
#include "kern_wave32.cuh"
#include "pairs16_host.h"
#include "psb_db.h"
#include "psb_internal.h"

namespace psb {

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
static thread_local Ctx g_ctx;

#define PSB_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess) {                                                                \
            set_error(std::string(#call) + ": " + cudaGetErrorString(e_));                      \
            return PSB_ECUDA;                                                                   \
        }                                                                                       \
    } while (0)

static int ensure_ctx() {
    Ctx &c = g_ctx;
    if (c.ready) {
        cudaError_t e = cudaSetDevice(c.device);
        if (e != cudaSuccess) { set_error(std::string("cudaSetDevice: ") + cudaGetErrorString(e)); return PSB_ECUDA; }
        return PSB_OK;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("no CUDA device available: libparasail_b200 has no CPU fallback (needs an sm_100a GPU)");
        return PSB_ENODEV;
    }
    if (c.device < 0) {
        if (cudaGetDevice(&c.device) != cudaSuccess) c.device = 0;
    }
    if (c.device >= ndev) { set_error("psb_set_device: device index out of range"); return PSB_EINVAL; }
    PSB_CUDA(cudaSetDevice(c.device));
    cudaDeviceProp prop;
    PSB_CUDA(cudaGetDeviceProperties(&prop, c.device));
    if (prop.major < 10) {
        set_error(std::string("device ") + prop.name + " is not sm_100-class; this library ships sm_100a code only");
        return PSB_ENODEV;
    }
    c.sms = prop.multiProcessorCount;
    PSB_CUDA(cudaStreamCreateWithFlags(&c.own_stream, cudaStreamNonBlocking));
    if (!c.stream) c.stream = c.own_stream;
    PSB_CUDA(cudaEventCreate(&c.ev0));
    PSB_CUDA(cudaEventCreate(&c.ev1));
    int lo_pri = 0, hi_pri = 0;
    cudaDeviceGetStreamPriorityRange(&lo_pri, &hi_pri);
    // the side stream carries the scan's main launch when a head/wavefront launch must reach the SMs
    // first (scan_sw16): lowest priority, so pending CTAs of the compute stream are placed before it
    (void)hi_pri;
    PSB_CUDA(cudaStreamCreateWithPriority(&c.side, cudaStreamNonBlocking, lo_pri));
    PSB_CUDA(cudaEventCreateWithFlags(&c.ev_fork, cudaEventDisableTiming));
    PSB_CUDA(cudaEventCreateWithFlags(&c.ev_join, cudaEventDisableTiming));
    PSB_CUDA(cudaStreamCreateWithFlags(&c.copy, cudaStreamNonBlocking));
    PSB_CUDA(cudaEventCreateWithFlags(&c.ev_alloc, cudaEventDisableTiming));
    // keep freed stream-ordered allocations cached so repeated batches do not hit the driver
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, c.device) == cudaSuccess) {
        unsigned long long thr = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    c.ready = true;
    return PSB_OK;
}

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

// Host->device copy that does not depend on the caller's memory being page-locked.  cudaMemcpyAsync out of
// pageable memory goes through the driver's own staging at a few GB/s with the calling thread blocked; large
// copies out of such memory are staged here instead, 8 MB at a time through two page-locked bounce buffers of the
// calling thread (memcpy of one chunk while the previous one is on the link).  Page-locked sources (and small
// copies) go straight to cudaMemcpyAsync.
static constexpr size_t kBounceBytes = (size_t)8 << 20;
static bool is_pageable(const void *p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return at.type == cudaMemoryTypeUnregistered;
}
static cudaError_t upload_h2d(void *dst, const void *src, size_t bytes, cudaStream_t stream) {
    if (bytes < ((size_t)1 << 20)) return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream);
    if (!is_pageable(src)) return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream);
    static const bool no_bounce = std::getenv("PSB_NO_BOUNCE") != nullptr;   // A/B knob: leave pageable memory to the driver
    if (no_bounce) return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream);
    Ctx &c = g_ctx;
    for (int k = 0; k < 2; ++k)
        if (!c.bounce[k]) {
            if (cudaMallocHost(&c.bounce[k], kBounceBytes) != cudaSuccess || cudaEventCreateWithFlags(&c.bounce_free[k], cudaEventDisableTiming) != cudaSuccess) {
                cudaGetLastError();
                if (c.bounce[k]) { cudaFreeHost(c.bounce[k]); c.bounce[k] = nullptr; }
                return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream);   // no bounce buffers: the driver's path
            }
            cudaEventRecord(c.bounce_free[k], stream);
        }
    for (size_t done = 0; done < bytes;) {
        const int k = c.bounce_next;
        c.bounce_next ^= 1;
        const size_t len = std::min(kBounceBytes, bytes - done);
        cudaError_t e = cudaEventSynchronize(c.bounce_free[k]);   // the copy that last used this buffer has left it
        if (e != cudaSuccess) return e;
        std::memcpy(c.bounce[k], (const uint8_t *)src + done, len);
        e = cudaMemcpyAsync((uint8_t *)dst + done, c.bounce[k], len, cudaMemcpyHostToDevice, stream);
        if (e != cudaSuccess) return e;
        e = cudaEventRecord(c.bounce_free[k], stream);
        if (e != cudaSuccess) return e;
        done += len;
    }
    return cudaSuccess;
}

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
static void release_kept() {
    Ctx &c = g_ctx;
    for (Ctx::Kept &k : c.kept) {
        if (k.p) cudaFreeAsync(k.p, c.stream);
        k.p = nullptr; k.cap = 0;
    }
}

// pinned host blocks are slow to create; recycle them process-wide by size class
static std::mutex g_pin_mu;
static std::multimap<size_t, void *> g_pin_free;
static void *pinned_alloc(size_t bytes) {
    size_t cls = 4096;
    while (cls < bytes) cls <<= 1;
    {
        std::lock_guard<std::mutex> lk(g_pin_mu);
        auto it = g_pin_free.find(cls);
        if (it != g_pin_free.end()) { void *p = it->second; g_pin_free.erase(it); return p; }
    }
    void *p = nullptr;
    if (cudaMallocHost(&p, cls) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
static void pinned_free(void *p, size_t bytes) {
    if (!p) return;
    size_t cls = 4096;
    while (cls < bytes) cls <<= 1;
    std::lock_guard<std::mutex> lk(g_pin_mu);
    if (g_pin_free.size() < 64) g_pin_free.emplace(cls, p);
    else cudaFreeHost(p);
}

struct BatchImpl {
    std::vector<std::pair<void *, size_t>> blocks;
    void *take(size_t bytes) {
        void *p = pinned_alloc(bytes);
        if (p) blocks.emplace_back(p, bytes);
        return p;
    }
};

// a batch's per-pair result arrays in the order the kernels' outputs use (score, end_query, end_ref, then the statistics)
static std::array<int *, 6> batch_outputs(psb_batch_t *b) { return {b->score, b->end_query, b->end_ref, b->matches, b->similar, b->length}; }
// the length of sequence i of a concatenation
static int span(const int64_t *off, int64_t i) { return (int)(off[i + 1] - off[i]); }
// explicit _8/_16 widths: the pairs whose values do not fit are flagged and their results zeroed (SURVEY A.8), by the
// rule of saturates(); `lens(i)` is pair i's (query, reference) lengths
template <typename Lens>
static void flag_saturated(const FnConfig &cfg, const HostMatrix &hm, int open, int gap, psb_batch_t *b, Lens lens) {
    if (cfg.width != 8 && cfg.width != 16) return;
    for (int64_t i = 0; i < b->n; ++i) {
        const std::pair<int, int> l = lens(i);
        if (saturates(cfg, hm, b->score[i], l.first, l.second, open, gap)) {
            b->saturated[i] = 1; b->score[i] = 0; b->end_query[i] = 0; b->end_ref[i] = 0;
        }
    }
}

static void fill_lut(unsigned *lut, const uint8_t *mapper) {
    for (int i = 0; i < 64; ++i)
        lut[i] = (unsigned)mapper[4 * i] | ((unsigned)mapper[4 * i + 1] << 8) | ((unsigned)mapper[4 * i + 2] << 16) |
                 ((unsigned)mapper[4 * i + 3] << 24);
}

// ---- kernel dispatch --------------------------------------------------------------------------
// Two kernel families.  "fine": per-warp int8 profile, mode-specialised, 13 row-per-lane classes
// (the many-pairs fast path).  "coarse": substitution matrix read directly (values that do not fit
// a byte, PSSMs, table outputs), mode read at run time, 3 classes.
static const int kFineK[] = {1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 12, 14, 16};
static const int kCoarseK[] = {4, 8, 16};
static constexpr int kNumClass = 13;   // upper bound on classes of either family
struct ClassTable { const int *k; int n; };
static ClassTable class_table(bool fine) { return fine ? ClassTable{kFineK, 13} : ClassTable{kCoarseK, 3}; }
static int class_of_len(const ClassTable &t, int lq) {
    for (int c = 0; c < t.n; ++c) if (lq <= 32 * t.k[c]) return c;
    return t.n - 1;
}

enum Variant { V_SCORE = 0, V_STATS32, V_STATS64, V_TRACE, V_TABLE };

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

static constexpr int kWarpsPerBlock = 4;

static int launch_gotoh32(int K, Variant v, Gotoh32Params &p, int nwork, bool prof, long long *grid_warps_out = nullptr) {
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
static long long max_grid_warps(long long nwork) {
    const long long cap = (long long)g_ctx.sms * 16 * kWarpsPerBlock;
    const long long need = ((nwork + kWarpsPerBlock - 1) / kWarpsPerBlock) * kWarpsPerBlock;
    return std::max<long long>(kWarpsPerBlock, std::min(cap, need));
}

// ---- one long pair over the whole GPU (kern_wave32.cuh) -------------------------------------------
static constexpr int kWaveMinLq = 2048;   // below this the per-pair kernel is used

template <int K> static const void *wave32_fn_k(bool v2) { return v2 ? (const void *)wave32v2_kernel<K> : (const void *)wave32_kernel<K>; }
static const void *wave32_fn(int K, bool v2) {
    switch (K) {
        case 1: return wave32_fn_k<1>(v2);
        case 2: return wave32_fn_k<2>(v2);
        case 4: return wave32_fn_k<4>(v2);
        case 8: return wave32_fn_k<8>(v2);
        case 16: return wave32_fn_k<16>(v2);
    }
    return nullptr;
}
static const void *wave32v3_fn(int K, bool is_sw, bool trace = false) {
    if (trace) return K != 8 ? nullptr : (is_sw ? (const void *)wave32v3_kernel<8, 4, true, true> : (const void *)wave32v3_kernel<8, 4, false, true>);
    switch (K) {
        case 4: return is_sw ? (const void *)wave32v3_kernel<4, 4, true> : (const void *)wave32v3_kernel<4, 4, false>;
        case 8: return is_sw ? (const void *)wave32v3_kernel<8, 4, true> : (const void *)wave32v3_kernel<8, 4, false>;
        case 16: return is_sw ? (const void *)wave32v3_kernel<16, 4, true> : (const void *)wave32v3_kernel<16, 4, false>;
    }
    return nullptr;
}
// the latency-optimised generation needs open >= extend and byte-sized (score + open)
static bool wave32_v2_ok(const HostMatrix &m, int open, int gap) {
    return open >= gap && gotoh32_profile_ok(m.size, m.min, m.max, open, m.type == PARASAIL_MATRIX_TYPE_PSSM);
}

// Long pairs WITH traceback or statistics: the TRACE instantiation of the column-blocked generation leaves 1.25
// bytes per cell (H low bytes + gap open/extend bits) and walk32_kernel follows the path (kern_wave32.cuh).
struct WaveWalk {
    bool stats;                   // count (matches, similar, length) instead of emitting CIGAR runs
    unsigned *rev_ops;
    const long long *rev_off;
    int *nops, *beg_query, *beg_ref;
};
static constexpr int kWaveTraceK = 8;
static size_t wave_trace_bytes(int lq, int lr) { return (size_t)wave32v3_trace_records(lq, lr, kWaveTraceK) * 40; }
// preconditions of that path (anything else keeps the one-warp-per-pair kernels): the column-blocked generation's
// own, H bytes that identify a neighbour's value, every strip resident at once, and the trace fits in `avail` bytes
static bool wave_walk_ok(const HostMatrix &m, int open, int gap, bool is_sw, int lq, int lr, size_t avail) {
    if (std::getenv("PSB_NO_WAVE_TRACE")) return false;
    if (!wave32_v2_ok(m, open, gap) || !pairs16_trace_ok(m.min, m.max, open)) return false;
    if ((lq + 32 * kWaveTraceK - 1) / (32 * kWaveTraceK) > g_ctx.sms * 16) return false;
    if (!wave32v3_range_ok(kWaveTraceK, 4, is_sw, lq, lr, m.max, m.min, open, gap)) return false;
    return wave_trace_bytes(lq, lr) + ((size_t)1 << 30) <= avail;
}
// what a new allocation can get: the driver's free figure + what the stream-ordered pool holds idle (0 if the driver
// cannot say).  Counting only the former would make a figure that shrinks as the pool warms up: every call would then
// cut its passes differently, ask for buffers of new sizes, grow the pool again ... -- calls of 2 s instead of 0.3 s.
static size_t device_mem_available() {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); return 0; }
    cudaMemPool_t pool;
    unsigned long long reserved = 0, used = 0;
    if (cudaDeviceGetDefaultMemPool(&pool, g_ctx.device) == cudaSuccess &&
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &reserved) == cudaSuccess &&
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used) == cudaSuccess && reserved > used)
        free_b += (size_t)(reserved - used);
    else cudaGetLastError();
    return free_b;
}

// PSB_DEBUG_TIMING on the pairs path (inert without it): where the host time of a pass goes, the device time of its
// marked launches and its timed region, as "[psb]" lines on stderr (tools/pairs_host_probe.py and
// tools/db_align_probe.py read them).  One per pass, on the calling thread's stream.
struct PassTimeline {
    const bool on = std::getenv("PSB_DEBUG_TIMING") != nullptr;
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

// launch shape of one long pair: generation (1 and 2: wave32_fn; 3: the column-blocked wave32v3_fn), rows per lane
// and warps per CTA
struct WaveShape {
    const void *fn;
    int K, wpb, gen;
};
static WaveShape wave_shape(const HostMatrix &m, int open, int gap, bool is_sw, int lq, int lr, bool traced) {
    const int sms = g_ctx.sms;
    auto strips = [lq](int K) { return (lq + 32 * K - 1) / (32 * K); };
    // the column-blocked generation (K x 4 tiles per lane and step) has the shortest critical path,
    // Lq/K + Lr/4 steps: every mode takes it when its preconditions hold (C5 local 46.5 -> 21.1 ms;
    // 50 kb x 50 kb global 26.6 -> 19.3 ms).  Measured on C5 (tools/c5_probe.py): a step costs about the same for 4
    // and 8 rows per lane (a warp alone on its scheduler is bound by per-step latencies) and twice as much for 16,
    // while every strip adds ~34 steps to the path: 8 rows, 4 warps per CTA (one per scheduler)
    WaveShape s{nullptr, 8, kWarpsPerBlock, wave32_v2_ok(m, open, gap) ? 3 : 1};
    // experiment knobs (tools/c5_probe.py): generation, rows per lane and warps per CTA of the launch
    if (const char *ev = std::getenv("PSB_WAVE_GEN")) { if (std::atoi(ev) == 2 && s.gen == 3) s.gen = 2; }
    if (s.gen == 3) {
        if (strips(s.K) > sms * 16) s.K = 16;
        if (strips(s.K) > sms * 16 || !wave32v3_range_ok(s.K, 4, is_sw, lq, lr, m.max, m.min, open, gap)) s.gen = 2;
    }
    // the older generations: strips of 32*K rows, enough strips to occupy the chip, as few as possible beyond that
    if (s.gen < 3) s.K = lq / 512 >= 2 * sms ? 16 : (lq / 256 >= 2 * sms ? 8 : 4);
    if (const char *ev = std::getenv("PSB_WAVE_K")) {
        const int k = std::atoi(ev);
        if ((k == 1 || k == 2 || k == 4 || k == 8 || k == 16) && (s.gen < 3 || k >= 4)) s.K = k;
    }
    if (const char *ev = std::getenv("PSB_WAVE_WARPS")) { const int w = std::atoi(ev); if (w >= 1 && w <= 32) s.wpb = w; }
    if (traced) { s.gen = 3; s.K = kWaveTraceK; }   // (wave_walk_ok held when the pair was routed here)
    s.fn = s.gen == 3 ? wave32v3_fn(s.K, is_sw, traced) : wave32_fn(s.K, s.gen == 2);
    return s;
}

// What every wavefront launch fills alike in its two parameter blocks: the pair (for several subjects: the query and
// their bytes, lr = 0), scoring, mode and end gaps (`md`: a Gotoh32Params or a FnConfig), the strip buffers (ctl: the
// strip counter, then per-strip progress) and the outputs.  The rest is zero: the multi-pair fields (multi_n, r_off,
// out_map) and the trace records are the caller's to set.
template <typename Mode>
static void wave_params(const Mode &md, const uint8_t *q, const uint8_t *r, int lq, int lr, const int *matrix, int size, int open, int gap,
                        int nstrips, int *bnd, int *ctl, int *cand, int *score, int *end_query, int *end_ref, Wave32Params *p, WaveReduceParams *rp) {
    std::memset(p, 0, sizeof(*p));
    p->q = q; p->r = r; p->Lq = lq; p->Lr = lr;
    p->matrix = matrix; p->size = size; p->open = open; p->gap = gap;
    p->mode = md.mode; p->s1_beg = md.s1_beg; p->s1_end = md.s1_end; p->s2_beg = md.s2_beg; p->s2_end = md.s2_end;
    p->bnd = bnd; p->progress = ctl + 1; p->next_strip = ctl; p->cand = cand;
    std::memset(rp, 0, sizeof(*rp));
    rp->cand = cand; rp->nstrips = nstrips; rp->mode = md.mode; rp->s1_end = md.s1_end; rp->s2_end = md.s2_end; rp->Lr = lr;
    rp->score = score; rp->end_query = end_query; rp->end_ref = end_ref;
}

static int launch_wave32(const Gotoh32Params &g, const HostMatrix &m, long long q_byte_off, int lq, long long r_byte_off, int lr, int out_index,
                         const WaveWalk *ww, PassTimeline &tl) {
    Ctx &c = g_ctx;
    const bool is_sw = g.mode == MODE_SW;
    const WaveShape s = wave_shape(m, g.open, g.gap, is_sw, lq, lr, ww != nullptr);
    const int K = s.K, wpb = s.wpb;
    const bool v3 = s.gen == 3;
    const int nstrips = (lq + 32 * K - 1) / (32 * K);
    DevMem d_bnd, d_ctl, d_cand, d_th, d_tb;
    if (ww) {
        const size_t nrec = (size_t)wave32v3_trace_records(lq, lr, K);
        PSB_TRY(d_th.alloc(nrec * 32, c.stream));
        PSB_TRY(d_tb.alloc(nrec * 8, c.stream));
    }
    PSB_TRY(d_bnd.alloc((size_t)nstrips * 2 * (size_t)lr * sizeof(int), c.stream));
    PSB_TRY(d_ctl.alloc(((size_t)nstrips + 2) * sizeof(int), c.stream));
    PSB_TRY(d_cand.alloc((size_t)nstrips * 8 * sizeof(int), c.stream));
    PSB_CUDA(cudaMemsetAsync(d_ctl.p, 0, ((size_t)nstrips + 2) * sizeof(int), c.stream));
    // generation 3 hands rows over through self-validating words: the lines start out all-zero (invalid)
    if (v3) PSB_CUDA(cudaMemsetAsync(d_bnd.p, 0, (size_t)nstrips * 2 * (size_t)lr * sizeof(int), c.stream));
    Wave32Params p;
    WaveReduceParams r;
    wave_params(g, g.q + q_byte_off, g.r + r_byte_off, lq, lr, g.matrix, g.size, g.open, g.gap, nstrips, d_bnd.as<int>(), d_ctl.as<int>(),
                d_cand.as<int>(), g.score + out_index, g.end_query + out_index, g.end_ref + out_index, &p, &r);
    p.trace_h = d_th.as<uint4>(); p.trace_bits = d_tb.as<uint2>();
    const size_t smem = v3 ? wave32v3_smem_bytes(g.size, wpb, K) : (s.gen == 2 ? wave32v2_smem_bytes(g.size, wpb) : wave32_smem_bytes(g.size, wpb));
    // every launched warp must be resident at once: the strips wait on one another
    int per_sm = 0;
    PSB_CUDA(occupancy_per_sm(s.fn, wpb, smem, &per_sm));
    PSB_CUDA(launch_persistent(s.fn, &p, nstrips, wpb, smem, per_sm, c.sms, c.stream));
    wave32_reduce_kernel<<<1, 32, 0, c.stream>>>(r);
    c.launches += 2;
    if (ww) {
        Walk32Params w;
        std::memset(&w, 0, sizeof(w));
        w.q = p.q; w.r = p.r; w.Lq = lq; w.Lr = lr; w.K = K; w.trace_h = p.trace_h; w.trace_bits = p.trace_bits;
        w.matrix = g.matrix; w.size = g.size; w.open = g.open; w.gap = g.gap; w.is_sw = is_sw ? 1 : 0;
        w.top_free = (is_sw || (g.mode == MODE_SG && g.s1_beg)) ? 1 : 0;
        w.left_free = (is_sw || (g.mode == MODE_SG && g.s2_beg)) ? 1 : 0;
        w.pid = out_index; w.score = g.score; w.end_query = g.end_query; w.end_ref = g.end_ref;
        w.rev_ops = ww->rev_ops; w.rev_off = ww->rev_off; w.nops = ww->nops; w.beg_query = ww->beg_query; w.beg_ref = ww->beg_ref;
        w.matches = g.matches; w.similar = g.similar; w.length = g.length;
        const size_t wsm = walk32_smem_bytes(g.size);
        tl.begin("walk32");
        if (ww->stats) walk32_kernel<true><<<1, 32, wsm, c.stream>>>(w);
        else walk32_kernel<false><<<1, 32, wsm, c.stream>>>(w);
        PSB_CUDA(cudaGetLastError());
        c.launches++;
        tl.end();
        if (tl.on)
            std::fprintf(stderr, "[psb] walk32 of a %d x %d pair: %.3f ms (trace %.2f GB)\n", lq, lr, tl.take_last_ms(),
                         (double)wave_trace_bytes(lq, lr) / 1e9);
    }
    if (v3 && tl.on) {
        // per-strip timeline of the column-blocked kernel: claimed / first columns available / done (us)
        std::vector<int> h((size_t)nstrips * 8);
        PSB_CUDA(cudaMemcpyAsync(h.data(), d_cand.p, h.size() * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
        PSB_CUDA(cudaStreamSynchronize(c.stream));
        const int t0 = h[5];
        for (int k = 0; k < nstrips; k = k < 8 ? k + 1 : k + std::max(1, nstrips / 12))
            std::fprintf(stderr, "[psb] wave strip %4d: claimed %7d us, first columns %7d us, done %7d us\n", k, h[(size_t)k * 8 + 5] - t0,
                         h[(size_t)k * 8 + 6] - t0, h[(size_t)k * 8 + 7] - t0);
    }
    return PSB_OK;
}

// ---- many pairs ---------------------------------------------------------------------------------
struct PairChunk {
    int64_t lo, hi;  // pair range of the caller's batch handled by this pass
};
struct PassOut;
// host threads that work through the passes of a large batch side by side.  Measured on 10^6 pairs (tools/
// pairs_host_probe.py; one lane / two / three): sw_trace 250 x 250: 106 / 50 / 47 ms, nw 250 x 250: 45 / 23.7 / 21.8 ms,
// sg_stats 150 x 500: 68 / 34 / 36 ms.  A third lane buys at most 8 % and another set of multi-gigabyte decision
// buffers; two it is.
static constexpr int kPairLanes = 2;
struct PassCutter;
static int run_pairs_lanes(const PairsRequest &req, PassCutter &cutter, const PairChunk &first, PassOut *first_out, psb_batch_t *b, int lanes);

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
    const bool top_free = req.cfg.mode == MODE_SW || (req.cfg.mode == MODE_SG && req.cfg.s1_beg);
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
            w.top_free = (sw || (cfg.mode == MODE_SG && cfg.s1_beg)) ? 1 : 0; w.left_free = (sw || (cfg.mode == MODE_SG && cfg.s2_beg)) ? 1 : 0;
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
    size_t tmp_bytes = 0;
    auto in_it = B.d_nops.as<int>();
    PSB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, in_it, B.d_csroff.as<long long>(), (int)(n + 1), c.stream));
    PSB_TRY(B.d_scan_tmp.alloc(tmp_bytes, c.stream));
    PSB_CUDA(cub::DeviceScan::ExclusiveSum(B.d_scan_tmp.p, tmp_bytes, in_it, B.d_csroff.as<long long>(), (int)(n + 1), c.stream));
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

static psb_batch_t *new_batch(int64_t n, const FnConfig &cfg) {
    psb_batch_t *b = new psb_batch_t();
    std::memset(b, 0, sizeof(*b));
    BatchImpl *impl = new BatchImpl();
    b->impl = impl;
    b->n = n;
    b->flag = cfg.flag();
    if (cfg.width == 0) b->flag |= PARASAIL_FLAG_BITS_32;
    const size_t ib = (size_t)std::max<int64_t>(n, 1) * sizeof(int);
    b->score = (int *)impl->take(ib); b->end_query = (int *)impl->take(ib); b->end_ref = (int *)impl->take(ib);
    bool ok = b->score && b->end_query && b->end_ref;
    if (cfg.stats) {
        b->matches = (int *)impl->take(ib); b->similar = (int *)impl->take(ib); b->length = (int *)impl->take(ib);
        ok = ok && b->matches && b->similar && b->length;
    }
    if (cfg.trace) {
        b->cigar_off = (int64_t *)impl->take(((size_t)n + 1) * sizeof(int64_t));
        b->beg_query = (int *)impl->take(ib); b->beg_ref = (int *)impl->take(ib);
        ok = ok && b->cigar_off && b->beg_query && b->beg_ref;
        if (ok) b->cigar_off[0] = 0;
    }
    b->saturated = (uint8_t *)impl->take((size_t)std::max<int64_t>(n, 1));
    ok = ok && b->saturated;
    if (!ok) { free_batch(b); return nullptr; }
    std::memset(b->saturated, 0, (size_t)std::max<int64_t>(n, 1));
    return b;
}

void free_batch(psb_batch_t *b) {
    if (!b) return;
    BatchImpl *impl = (BatchImpl *)b->impl;
    if (impl) {
        for (auto &blk : impl->blocks) pinned_free(blk.first, blk.second);
        delete impl;
    }
    delete b;
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
    const bool host_dbg = std::getenv("PSB_DEBUG_TIMING") != nullptr;
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

// ---- resident database ----------------------------------------------------------------------------
}  // namespace psb

namespace psb {

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

__global__ void db_lengths_kernel(const long long *off, long long n, int *len, int *idx) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        len[i] = (int)(off[i + 1] - off[i]);
        idx[i] = (int)i;
    }
}
__global__ void db_wcount_sorted_kernel(const int *len_sorted, long long n, int rpw, long long *wcount) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i <= n; i += stride)
        wcount[i] = i < n ? (len_sorted[i] + rpw - 1) / rpw : 0;
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
    if (!P.general && std::getenv("PSB_DEBUG_TIMING"))
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
    UnpackParams u;
    u.words = db->d_words; u.word_off = db->d_word_off; u.ids = nullptr; u.inv_perm = nullptr; u.out_off = B.loff.as<long long>();
    u.out = B.lbytes.as<uint8_t>(); u.n = nroute; u.bits = db->bits;
    unpack_db_kernel<<<(unsigned)std::min<int64_t>(nroute, 1024), 256, 0, c.stream>>>(u);
    Wave32Params w;
    WaveReduceParams r;
    wave_params(cfg, dp->d_query, B.lbytes.as<uint8_t>(), lq, 0, dp->d_matrix, m.size, open, gap, nstrips, B.bnd.as<int>(), B.ctl.as<int>(),
                B.cand.as<int>(), d_out[0], d_out[1], d_out[2], &w, &r);
    w.multi_n = (int)nroute; w.r_off = B.loff.as<long long>();
    r.multi_n = (int)nroute; r.r_off = B.loff.as<long long>(); r.out_map = db->d_perm;
    const bool v2 = wave32_v2_ok(m, open, gap);
    const void *fn = wave32_fn(K, v2);
    // Full-size CTAs that also reserve most of an SM's shared memory: the strips of the long
    // subjects then own a few SMs outright instead of crawling beside sixteen ALU-bound warps
    // of the main kernel on every SM (each of their steps is a serial dependency).  The main
    // kernel's blocks that find no room start on those SMs as soon as the strips are done.
    const int kRouteWarps = v2 ? 8 : 32;   // generation 2 keeps a 12 KB profile per warp
    const size_t smem = std::max<size_t>(v2 ? wave32v2_smem_bytes(m.size, kRouteWarps) : wave32_smem_bytes(m.size, kRouteWarps), 160 * 1024);
    PSB_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // all warps of this launch must be resident together (strips wait on one another): one CTA
    // per SM at most, issued before the main kernel so that its blocks are placed first
    const long long items = nroute * nstrips;
    long long blocks = std::min<long long>((items + kRouteWarps - 1) / kRouteWarps, (long long)c.sms);
    void *args[] = {&w};
    PSB_CUDA(cudaLaunchKernel(fn, dim3((unsigned)blocks), dim3(kRouteWarps * 32), args, smem, c.stream));
    wave32_reduce_kernel<<<(unsigned)((nroute + 127) / 128), 128, 0, c.stream>>>(r);
    c.launches += 3;
    return PSB_OK;
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
            size_t tb = 0;
            DevMem d_tmp;
            PSB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, db->d_len, ro, (int)db->n, c.stream));
            PSB_TRY(d_tmp.alloc(tb, c.stream));
            PSB_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp.p, tb, db->d_len, ro, (int)db->n, c.stream));
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
    if (std::getenv("PSB_DEBUG_TIMING")) std::fprintf(stderr, "[psb] sw16: K %d, %d warps per CTA, %d CTAs per SM, %zu B shared\n", sp.K, s.wpb, s.per_sm, s.smem);
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

}  // namespace psb

namespace psb {
int db_io_ensure_ctx(int *device, cudaStream_t *stream) {
    const int rc = ensure_ctx();
    if (rc != PSB_OK) return rc;
    *device = g_ctx.device; *stream = g_ctx.stream;
    return PSB_OK;
}
}  // namespace psb

using namespace psb;

extern "C" {

int psb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int psb_set_device(int device) {
    Ctx &c = g_ctx;
    if (c.ready && c.device != device) {
        // a host thread is bound to one device for its lifetime (one process per GPU is the model)
        set_error("psb_set_device: this thread is already bound to another device");
        return PSB_EINVAL;
    }
    c.device = device;
    return ensure_ctx();
}

int psb_set_stream(void *cuda_stream) {
    PSB_TRY(ensure_ctx());
    g_ctx.stream = cuda_stream ? (cudaStream_t)cuda_stream : g_ctx.own_stream;
    return PSB_OK;
}

int psb_synchronize(void) {
    PSB_TRY(ensure_ctx());
    PSB_CUDA(cudaStreamSynchronize(g_ctx.stream));
    return PSB_OK;
}

double psb_last_kernel_ms(void) { return g_ctx.last_ms; }
int psb_last_launches(void) { return g_ctx.launches; }

void psb_batch_free(psb_batch_t *batch) { free_batch(batch); }

}  // extern "C"

namespace psb {
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
}  // namespace psb

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

namespace psb {

// Database construction in two phases so that psb_scan_host can overlap the upload of one piece with
// the scan of the previous one.  Phase A (db_begin): one host pass over the offsets (validation,
// longest lengths, packed size), device allocations, and the host->device copies on `up` (the
// caller's stream or the context's copy stream).  Phase B (db_finish): lengths, stable radix sort
// by decreasing length, word offsets (scan), residue mapping + bit packing, all on the compute
// stream and without any host synchronisation.
// Device staging blocks for psb_scan_host's uploads.  They are filled on the copy stream while the
// compute stream is busy, so they cannot come from a stream-ordered pool without tying the two
// streams together (an allocation that cannot reuse a block freed on the other stream falls back to
// mapping fresh memory, a host-blocking call of tens of milliseconds).  Plain allocations, recycled
// process-wide; a block is handed back only after both streams have been synchronised.
struct StageBlock { void *p; size_t bytes; int device; };
static std::mutex g_stage_mu;
static std::vector<StageBlock> g_stage_free;
static size_t g_stage_cached = 0;
static void *stage_acquire(int device, size_t need, size_t *got) {
    const size_t gran = (size_t)8 << 20;
    const size_t want = (need + gran - 1) / gran * gran;
    {
        std::lock_guard<std::mutex> lk(g_stage_mu);
        int pick = -1;
        for (int i = 0; i < (int)g_stage_free.size(); ++i) {
            const StageBlock &b = g_stage_free[i];
            if (b.device == device && b.bytes >= want && b.bytes <= 2 * want && (pick < 0 || b.bytes < g_stage_free[pick].bytes)) pick = i;
        }
        if (pick >= 0) {
            StageBlock b = g_stage_free[pick];
            g_stage_free.erase(g_stage_free.begin() + pick);
            g_stage_cached -= b.bytes;
            *got = b.bytes;
            return b.p;
        }
    }
    void *p = nullptr;
    if (cudaMalloc(&p, want) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    *got = want;
    return p;
}
static void stage_release(int device, void *p, size_t bytes) {
    if (!p) return;
    {
        std::lock_guard<std::mutex> lk(g_stage_mu);
        if (g_stage_cached + bytes <= ((size_t)4 << 30) && g_stage_free.size() < 256) {
            g_stage_free.push_back({p, bytes, device});
            g_stage_cached += bytes;
            return;
        }
    }
    cudaFree(p);
}

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

// Phase A1: the device-side object and the host->device copies (nothing here looks at the individual offsets,
// so psb_scan_host can queue the upload of piece k+1 before it spends host time on piece k)
static psb_db *db_upload(DbBuild &B, const uint8_t *cat, const int64_t *off, int64_t n, const HostMatrix &hm, bool use_copy_stream, int force_bits = 0,
                         cudaEvent_t residues_after = nullptr) {
    Ctx &c = g_ctx;
    if (hm.size > 32) { set_error("psb_db_create: alphabets above 32 letters cannot be 5-bit packed"); return nullptr; }
    if (off[n] <= off[0]) { set_error("psb_db_create: offsets are not increasing"); return nullptr; }
    psb_db *db = new psb_db();
    db->device = c.device; db->stream = c.stream; db->n = n; db->msize = hm.size;
    std::memcpy(db->mapper, hm.mapper, 256);
    // 2 bit for alphabets of up to 4 letters, 3 bit up to 8 (ACGT + wildcard: DNA ships at 3 bit), else 5
    db->bits = force_bits ? force_bits : db_bits_for(hm.size);
    db->residues = off[n] - off[0];
    const size_t n1 = (size_t)n + 1;
    // with the copy stream, the upload must not queue behind whatever scan is already running on the
    // compute stream: its staging blocks are recycled plain allocations (see StageBlock)
    cudaStream_t up = use_copy_stream ? c.copy : c.stream;
    auto fail = [&](const std::string &what) {
        set_error(what);
        cudaStreamSynchronize(up);
        psb_db_free(db);
        return (psb_db *)nullptr;
    };
    if (use_copy_stream) {
        B.st_device = c.device;
        B.st_raw = stage_acquire(c.device, (size_t)db->residues, &B.st_raw_bytes);
        B.st_off = stage_acquire(c.device, n1 * 8, &B.st_off_bytes);
        if (!B.st_raw || !B.st_off) return fail("psb_scan_host: device allocation of the staging blocks failed");
    } else if (B.d_raw.alloc((size_t)db->residues, up) != PSB_OK || B.d_off.alloc(n1 * 8, up) != PSB_OK) {
        return fail(psb_last_error());
    }
    cudaError_t e = cudaSuccess;
    auto ck = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    // offsets first: lengths, sort and word offsets need nothing else, so that whole chain of small launches runs
    // while the residues (the long copy) are still on the link -- under a saturated link each of those launches
    // costs 30-50 us instead of 5 (measured: 0.6 ms for the chain of the first piece, tools/shard_e2e_probe.py)
    ck(upload_h2d(B.offs(), off, n1 * 8, up));
    if (use_copy_stream) {
        ck(cudaEventCreateWithFlags(&B.offs_up, cudaEventDisableTiming));
        ck(cudaEventRecord(B.offs_up, up));
        // a saturated link makes every small launch on the device wait its turn for the command fetch (30-50 us
        // each, measured), so the residues of this piece stay off the link until the previous piece's sort/pack
        // chain has run; they still have that piece's whole scan to land in
        if (residues_after) ck(cudaStreamWaitEvent(up, residues_after, 0));
        ck(cudaEventCreate(&B.res_begin));
        ck(cudaEventRecord(B.res_begin, up));
    }
    ck(upload_h2d(B.raw(), cat + off[0], (size_t)db->residues, up));
    if (use_copy_stream) {
        ck(cudaEventCreate(&B.uploaded));
        ck(cudaEventRecord(B.uploaded, up));
    }
    if (e != cudaSuccess) return fail(std::string("psb_db_create: ") + cudaGetErrorString(e));
    B.db = db; B.raw_base = off[0]; B.up = up;
    fill_lut(B.lut, hm.mapper);
    return db;
}

// words of `rpw` residues that `l` residues occupy; rpw is one of 16 / 10 / 6 (2, 3, 5 bit): constant
// divisors, because a 64-bit division per subject was most of this pass
template <int RPW> static inline long long words_of(long long l) { return (l + RPW - 1) / RPW; }

// Phase A2: one host pass over the offsets (validation, histogram of lengths for the longest few, exact
// packed size) and the remaining device allocations
static int db_host_pass(DbBuild &B, const int64_t *off) {
    Ctx &c = g_ctx;
    psb_db *db = B.db;
    const int64_t n = db->n;
    const int rpw = db_residues_per_word(db->bits);
    auto fail = [&](const std::string &what) {
        set_error(what);
        cudaStreamSynchronize(B.up);
        cudaStreamSynchronize(c.stream);
        psb_db_free(db);
        B.db = nullptr;
        return PSB_EINVAL;
    };
    thread_local std::vector<int> hist;
    hist.assign(65537, 0);
    std::vector<int> huge;   // lengths above 65535
    long long words = 0;
    int64_t maxlen = 0, bad = -1;
    auto pass = [&](auto wof) {
        for (int64_t i = 0; i < n; ++i) {
            const int64_t l = off[i + 1] - off[i];
            if (l <= 0 || l > 0x7fffffff) { bad = i; return; }
            words += wof(l);
            if (l > 65535) huge.push_back((int)l); else hist[(size_t)l]++;
            maxlen = l > maxlen ? l : maxlen;
        }
    };
    if (rpw == 6) pass(words_of<6>); else if (rpw == 10) pass(words_of<10>); else if (rpw == 16) pass(words_of<16>);
    else pass([rpw](long long l) { return (l + rpw - 1) / rpw; });
    if (bad >= 0) return fail("psb_db_create: empty or oversized subject " + std::to_string(bad));
    std::sort(huge.begin(), huge.end(), [](int a, int b2) { return a > b2; });
    db->maxlen = (int)maxlen; db->nlong = (int)huge.size(); db->words = words;
    db->top_len = huge;
    if (db->top_len.size() > 4096) db->top_len.resize(4096);
    for (int l = (int)std::min<int64_t>(maxlen, 65535); l >= 1 && db->top_len.size() < 4096; --l)
        for (int t = 0; t < hist[l] && db->top_len.size() < 4096; ++t) db->top_len.push_back(l);

    const size_t n1 = (size_t)n + 1;
    if (B.d_len0.alloc((size_t)n * 4, c.stream) != PSB_OK || B.d_idx0.alloc((size_t)n * 4, c.stream) != PSB_OK ||
        B.d_wcount.alloc(n1 * 8, c.stream) != PSB_OK)
        return fail(psb_last_error());
    cudaError_t e = cudaSuccess;
    auto ck = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    ck(cudaMallocAsync(&db->d_word_off, n1 * 8, c.stream));
    ck(cudaMallocAsync(&db->d_perm, (size_t)n * 4, c.stream));
    ck(cudaMallocAsync(&db->d_len, (size_t)n * 4, c.stream));
    ck(cudaMallocAsync(&db->d_words, (size_t)db->words * 4 + 64, c.stream));
    if (e != cudaSuccess) return fail(std::string("psb_db_create: ") + cudaGetErrorString(e));
    return PSB_OK;
}

static psb_db *db_begin(DbBuild &B, const uint8_t *cat, const int64_t *off, int64_t n, const HostMatrix &hm, bool use_copy_stream, int force_bits = 0) {
    if (!db_upload(B, cat, off, n, hm, use_copy_stream, force_bits)) return nullptr;
    if (db_host_pass(B, off) != PSB_OK) return nullptr;
    return B.db;
}

// PSB_DEBUG_TIMING on psb_scan_host (inert without it): a device-side timeline, one event per mark on the stream
// named, reported relative to the first mark
struct StreamMarks {
    const bool on = std::getenv("PSB_DEBUG_TIMING") != nullptr;
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

// PSB_DEBUG_TIMING on psb_scan_host / psb_scan_box (`on` is false without it): the host's milliseconds since construction
struct HostClock {
    const bool on = std::getenv("PSB_DEBUG_TIMING") != nullptr;
    const std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    double ms() const { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); }
};

// `marks`: psb_scan_host's timeline (lengths< >lengths sort> <pack pack>), or nullptr
static int db_finish(DbBuild &B, StreamMarks *marks = nullptr) {
    Ctx &c = g_ctx;
    psb_db *db = B.db;
    const int64_t n = db->n;
    const size_t n1 = (size_t)n + 1;
    const int rpw = db_residues_per_word(db->bits);
    auto mark = [&] { if (marks) marks->mark(c.stream); };
    if (B.offs_up) PSB_CUDA(cudaStreamWaitEvent(c.stream, B.offs_up, 0));
    mark();
    db_lengths_kernel<<<c.sms * 4, 256, 0, c.stream>>>(B.offs(), n, B.d_len0.as<int>(), B.d_idx0.as<int>());
    mark();
    size_t tb = 0, tb2 = 0;
    PSB_CUDA(cub::DeviceRadixSort::SortPairsDescending(nullptr, tb, B.d_len0.as<int>(), db->d_len, B.d_idx0.as<int>(), db->d_perm, (int)n, 0, 32, c.stream));
    PSB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb2, B.d_wcount.as<long long>(), db->d_word_off, (int)n1, c.stream));
    PSB_TRY(B.d_tmp.alloc(std::max(tb, tb2), c.stream));
    PSB_CUDA(cub::DeviceRadixSort::SortPairsDescending(B.d_tmp.p, tb, B.d_len0.as<int>(), db->d_len, B.d_idx0.as<int>(), db->d_perm, (int)n, 0, 32, c.stream));
    mark();
    db_wcount_sorted_kernel<<<c.sms * 4, 256, 0, c.stream>>>(db->d_len, n, rpw, B.d_wcount.as<long long>());
    PSB_CUDA(cub::DeviceScan::ExclusiveSum(B.d_tmp.p, tb2, B.d_wcount.as<long long>(), db->d_word_off, (int)n1, c.stream));
    PackParams pp;
    pp.raw = B.raw(); pp.raw_off = B.offs(); pp.raw_base = B.raw_base; pp.perm = db->d_perm;
    pp.word_off = db->d_word_off; pp.words = db->d_words; pp.n = n; pp.bits = db->bits;
    std::memcpy(pp.lut, B.lut, sizeof(pp.lut));
    if (B.uploaded) PSB_CUDA(cudaStreamWaitEvent(c.stream, B.uploaded, 0));
    mark();
    pack_db_kernel<<<c.sms * 8, 256, 256, c.stream>>>(pp);
    if (B.uploaded) {
        PSB_CUDA(cudaEventCreateWithFlags(&B.packed, cudaEventDisableTiming));
        PSB_CUDA(cudaEventRecord(B.packed, c.stream));
    }
    mark();
    c.launches += 5;
    PSB_CUDA(cudaGetLastError());
    // no synchronisation: later work on this stream is ordered after the packing kernel, and the
    // staging buffers go back to the pool in stream order when B is destroyed
    return PSB_OK;
}

// a database the caller holds in host memory, checked in each entry point's wording; `arg` is the entry point's other
// required pointer.  The host scans (`scan`) report offsets that do not increase as an empty database, before the
// subject count; psb_db_create names them, after it.
static int host_db_check(const char *who, const void *arg, const uint8_t *cat, const int64_t *off, int64_t n, bool scan) {
    const std::string w(who);
    if (!arg || !cat || !off || n <= 0 || (scan && off[n] <= off[0])) { set_error(w + ": NULL argument or empty database"); return PSB_EINVAL; }
    if (n > 0x7ffffffe) { set_error(w + ": more than 2^31-2 subjects"); return PSB_EUNSUPPORTED; }
    if (off[n] <= off[0]) { set_error(w + ": offsets are not increasing"); return PSB_EINVAL; }
    return PSB_OK;
}

}  // namespace psb

extern "C" {

psb_db_t *psb_db_create(const uint8_t *cat, const int64_t *off, int64_t n, const parasail_matrix_t *matrix) {
    if (host_db_check("psb_db_create", matrix, cat, off, n, false) != PSB_OK) return nullptr;
    if (ensure_ctx() != PSB_OK) return nullptr;
    HostMatrix hm(matrix);
    // bits per residue from the residues actually present: a DNA database whose residues are all A/C/G/T
    // (no wildcard, which maps to column 4) packs at 2 bit even though its matrix has 5 columns
    int force_bits = 0;
    if (db_bits_for(hm.size) == 3) {
        bool small = true;
        for (int64_t x = off[0]; x < off[n] && small; ++x) small = hm.mapper[cat[x]] < 4;
        if (small) force_bits = 2;
    }
    DbBuild B;
    psb_db *db = db_begin(B, cat, off, n, hm, false, force_bits);
    if (!db) return nullptr;
    // the caller's buffers must be free to go when this returns: wait for the uploads (not for the packing)
    cudaEvent_t up = nullptr;
    if (cudaEventCreateWithFlags(&up, cudaEventDisableTiming) == cudaSuccess) cudaEventRecord(up, g_ctx.stream);
    db->host_len.resize((size_t)n);
    for (int64_t i = 0; i < n; ++i) db->host_len[(size_t)i] = (int)(off[i + 1] - off[i]);
    const int rc = db_finish(B);
    if (up) { cudaEventSynchronize(up); cudaEventDestroy(up); } else cudaStreamSynchronize(g_ctx.stream);
    if (rc != PSB_OK) { cudaStreamSynchronize(g_ctx.stream); psb_db_free(db); return nullptr; }
    return db;
}

int64_t psb_db_count(const psb_db_t *db) { return db ? db->n : 0; }
int psb_db_bits(const psb_db_t *db) { return db ? db->bits : 0; }
int64_t psb_db_residues(const psb_db_t *db) { return db ? db->residues : 0; }
int64_t psb_db_device_bytes(const psb_db_t *db) {
    return db ? db->words * 4 + (db->n + 1) * 8 + db->n * 8 : 0;
}

void psb_db_free(psb_db_t *db) {
    if (!db) return;
    int cur = 0;
    cudaGetDevice(&cur);
    cudaSetDevice(db->device);
    void *ptrs[] = {db->d_words, db->d_word_off, db->d_perm, db->d_len, db->d_res_off, db->d_inv_perm};
    for (void *p : ptrs) if (p) cudaFreeAsync(p, db->stream);
    cudaSetDevice(cur);
    delete db;
}

}  // extern "C"

namespace psb {
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
// the packed 16-bit scan serves this function (if its profile can be packed): local score-only at 8/16 bit or "sat"
static bool sw16_wanted(const FnConfig &cfg) { return cfg.mode == MODE_SW && !cfg.stats && cfg.width != 32 && cfg.width != 64; }
static int scan_enqueue(ScanJob &job, const FnConfig &cfg, const parasail_profile *profile, int open, int gap, psb_db *db,
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
    for (int k = 0; k < nout; ++k)
        PSB_CUDA(cudaMemcpyAsync(hosts[k] + host_base, job.d_out[k].p, (size_t)db->n * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    PSB_CUDA(cudaEventCreateWithFlags(&job.done, cudaEventDisableTiming));
    PSB_CUDA(cudaEventRecord(job.done, c.stream));
    return PSB_OK;
}
// waits until the job's results are on the host
static int scan_finish(ScanJob &job) {
    Ctx &c = g_ctx;
    if (job.finished) return PSB_OK;
    job.finished = true;
    cudaError_t e = job.done ? cudaEventSynchronize(job.done) : cudaStreamSynchronize(c.stream);
    if (e != cudaSuccess) { set_error(std::string("psb_scan: ") + cudaGetErrorString(e)); return PSB_ECUDA; }
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, job.ev0, job.ev1) == cudaSuccess) c.last_ms += ms;
    if (std::getenv("PSB_DEBUG_TIMING")) std::fprintf(stderr, "[psb] scan job: %.3f ms, %d re-run at 32 bit\n", ms, *job.retried_host);
    if (job.rate_k > 0) sw16_rate_update(job.rate_k, job.rate_cells, ms);
    job.retried += *job.retried_host;
    return PSB_OK;
}
// what every entry point that runs a profile against a database checks first: a profile function name and a profile
static int profile_fn_check(const char *who, const char *fn_name, const parasail_profile_t *profile, FnConfig *cfg) {
    if (!parse_fn_name(fn_name, cfg) || !cfg->profile) { set_error(std::string(who) + ": not a profile function name: " + (fn_name ? fn_name : "(null)")); return PSB_EINVAL; }
    if (!profile) { set_error(std::string(who) + ": NULL profile"); return PSB_EINVAL; }
    return PSB_OK;
}
// and a scan, which produces no traceback
static int scan_check(const char *who, const char *fn_name, const parasail_profile_t *profile, FnConfig *cfg) {
    PSB_TRY(profile_fn_check(who, fn_name, profile, cfg));
    if (cfg->trace || cfg->table || cfg->rowcol) { set_error(std::string(who) + ": trace/table/rowcol outputs are not available for database scans"); return PSB_EUNSUPPORTED; }
    return PSB_OK;
}
// a profile run against a resident database: the calling thread's device holds it, and both use the same alphabet
static int profile_db_check(const char *who, const parasail_profile_t *profile, const psb_db *db) {
    PSB_TRY(ensure_ctx());
    if (db->device != g_ctx.device) { set_error(std::string(who) + ": database lives on another device"); return PSB_EINVAL; }
    if (profile->matrix.size != db->msize || std::memcmp(profile->matrix.mapper, db->mapper, 256) != 0) {
        set_error(std::string(who) + ": profile and database were built with different alphabets");
        return PSB_EINVAL;
    }
    return PSB_OK;
}
// what every call that reads a resident database's subjects by caller id checks: the calling thread's device holds it
static int db_check(const char *who, const psb_db *db) {
    PSB_TRY(ensure_ctx());
    if (db->device != g_ctx.device) { set_error(std::string(who) + ": database lives on another device"); return PSB_EINVAL; }
    if (db->host_len.empty()) { set_error(std::string(who) + ": the database has no subject lengths on the host"); return PSB_EUNSUPPORTED; }
    return PSB_OK;
}
// the end of a scan entry point: the batch's cells, the flags of explicit _8 / _16 widths, and the batch handed over;
// `subject_len(i)` is subject i's length
template <typename SubjectLen>
static int scan_batch_done(const FnConfig &cfg, const parasail_profile_t *profile, int open, int gap, int64_t residues, SubjectLen subject_len,
                           psb_batch_t *b, psb_batch_t **out) {
    const int lq = (int)profile->query.size();
    b->cells = (double)profile->query.size() * (double)residues;
    flag_saturated(cfg, profile->matrix, open, gap, b, [&](int64_t i) { return std::make_pair(lq, subject_len(i)); });
    *out = b;
    return PSB_OK;
}
// The database's inverse permutation, built on first use: the scatter runs on db->stream, behind the sort/pack chain
// psb_db_create queued there (it returns before that chain has finished), and that stream is synchronised before the
// pointer is published.  So whoever sees the pointer -- any host thread, any stream -- also sees finished packed words.
static int db_inv_perm(psb_db *db, int *launched) {
    *launched = 0;
    if (db->d_inv_perm) return PSB_OK;
    std::lock_guard<std::mutex> lk(db->mu);
    if (db->d_inv_perm) return PSB_OK;
    int *inv = nullptr;
    PSB_CUDA(cudaMallocAsync(&inv, (size_t)db->n * sizeof(int), db->stream));
    invert_perm_kernel<<<(unsigned)std::min<int64_t>((db->n + 255) / 256, (int64_t)g_ctx.sms * 8), 256, 0, db->stream>>>(db->d_perm, db->n, inv);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(db->stream);
    if (e != cudaSuccess) {
        cudaFreeAsync(inv, db->stream);
        set_error(std::string("psb_db: inverse permutation: ") + cudaGetErrorString(e));
        return PSB_ECUDA;
    }
    db->d_inv_perm = inv;
    *launched = 1;
    return PSB_OK;
}
}  // namespace psb

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

int64_t psb_db_subject(const psb_db_t *db_c, int64_t id, uint8_t *codes, int64_t cap) {
    if (!db_c || cap < 0 || (cap > 0 && !codes)) { set_error("psb_db_subject: NULL argument or negative capacity"); return PSB_EINVAL; }
    psb_db *db = const_cast<psb_db *>(db_c);
    PSB_TRY(db_check("psb_db_subject", db));
    if (id < 0 || id >= db->n) { set_error("psb_db_subject: id " + std::to_string(id) + " is not a subject of a database of " + std::to_string(db->n)); return PSB_EINVAL; }
    int first_use = 0;
    PSB_TRY(db_inv_perm(db, &first_use));
    const int64_t len = db->host_len[(size_t)id];
    if (cap == 0) return len;
    Ctx &c = g_ctx;
    const int sid = (int)id;
    const long long off[2] = {0, (long long)len};
    DevMem d_id, d_off, d_out;
    PSB_TRY(d_id.alloc(sizeof(int), c.stream));
    PSB_TRY(d_off.alloc(sizeof(off), c.stream));
    PSB_TRY(d_out.alloc((size_t)len, c.stream));
    PSB_CUDA(cudaMemcpyAsync(d_id.p, &sid, sizeof(int), cudaMemcpyHostToDevice, c.stream));
    PSB_CUDA(cudaMemcpyAsync(d_off.p, off, sizeof(off), cudaMemcpyHostToDevice, c.stream));
    UnpackParams u;
    u.words = db->d_words; u.word_off = db->d_word_off; u.ids = d_id.as<int>(); u.inv_perm = db->d_inv_perm;
    u.out_off = d_off.as<long long>(); u.out = d_out.as<uint8_t>(); u.n = 1; u.bits = db->bits;
    unpack_db_kernel<<<1, 32, 0, c.stream>>>(u);
    PSB_CUDA(cudaGetLastError());
    PSB_CUDA(cudaMemcpyAsync(codes, d_out.p, (size_t)std::min(len, cap), cudaMemcpyDeviceToHost, c.stream));
    PSB_CUDA(cudaStreamSynchronize(c.stream));   // (`sid` / `off` are host temporaries)
    return len;
}

}  // extern "C"

namespace psb {
// The scan of a database that lives in HOST memory, on the calling thread's device: the residues are cut
// into pieces whose upload (copy stream), device-side sort + packing and scan are pipelined, and the
// per-subject results land in hosts[k][base ...] (pinned).  Used by psb_scan_host (one device, base 0) and by
// the per-device workers of psb_scan_box (each with its own range of the caller's arrays).
static uint64_t host_scan_key(const FnConfig &cfg, int lq, int open, int gap, int msize) {
    uint64_t h = 1469598103934665603ull;
    for (uint64_t x : {(uint64_t)encode_fn(cfg), (uint64_t)lq, (uint64_t)open, (uint64_t)gap, (uint64_t)msize}) { h ^= x + 1; h *= 1099511628211ull; }
    return h | 1;
}
// piece sizes (bytes) for a host scan of `total` residues: geometric with ratio r = 0.85 v/u (every piece lands
// before its predecessor has been scanned), first piece and count chosen to minimise the exposed time
//   (first piece's upload) + (pieces - 1) x boundary,   boundary = sort/pack chain + the scan kernel's ramp and tail
// e.g. C2 on one GPU (362 MB, 52 GB/s, 27 ms of scan): 22 + 76 + 264 MB; a 1/8 shard (45 MB): 10 + 35 MB.
std::vector<int64_t> plan_pieces(int64_t total, double u, double v) {
    const double boundary_ms = 0.35;
    const int64_t cap = (int64_t)1 << 30;   // bounds the device memory of a piece
    // no piece below ~1 ms of scan: the sweep of a piece's longest subjects is serial, so smaller pieces take that
    // long anyway (measured: 8 MB and 11 MB pieces of C2 both scan in 1.2 ms)
    const int64_t min_piece = std::max<int64_t>((int64_t)4 << 20, (int64_t)(1.0 / v));
    // ratio in steps of 1/4 and sizes in steps of 2 MB: the measured rates move a little from call to call, the
    // plan (and with it every allocation size of the pipeline) should not
    const double r = std::min(16.0, std::max(1.25, std::floor(0.85 * v / u * 4.0) / 4.0));
    const double quantum = (double)((int64_t)2 << 20);
    auto cut_up = [&](double s0) {
        std::vector<int64_t> sizes;
        double s = std::max(quantum, std::floor(s0 / quantum) * quantum);
        for (int64_t left = total; left > 0; s *= r) {
            int64_t sz = std::min<int64_t>((int64_t)(std::floor(std::min(s, (double)cap) / quantum) * quantum), left);
            if (left - sz < min_piece) sz = left;
            sizes.push_back(sz);
            left -= sz;
        }
        return sizes;
    };
    std::vector<int64_t> sizes(1, total);
    double best_cost = (double)total * u;
    for (int m = 2; m <= 8; ++m) {
        double s0 = (double)total * (r - 1.0) / (std::pow(r, m) - 1.0);
        const bool floor_hit = s0 < (double)min_piece;
        if (floor_hit) s0 = (double)min_piece;
        if (s0 + (double)min_piece > (double)total) break;
        std::vector<int64_t> cand = cut_up(s0);
        const double cost = (double)cand[0] * u + (double)(cand.size() - 1) * boundary_ms;
        if (cost < best_cost) { best_cost = cost; sizes.swap(cand); }
        if (floor_hit) break;
    }
    return sizes;
}

// subject cuts of the database off[0 .. n] at residue targets (counted from off[0], increasing): 0, then for each target
// the first subject boundary at or past it but at least one subject past the previous cut, then n.  A cut that would
// leave no subject after it ends the list.
static std::vector<int64_t> cut_subjects(const int64_t *off, int64_t n, const std::vector<int64_t> &targets) {
    std::vector<int64_t> cut(1, 0);
    for (const int64_t t : targets) {
        const int64_t at = std::max<int64_t>(std::lower_bound(off, off + n + 1, off[0] + t) - off, cut.back() + 1);
        if (at >= n) break;
        cut.push_back(at);
    }
    cut.push_back(n);
    return cut;
}

// The pieces of a host scan: the upload of piece k+1 (copy stream) runs under the scan of piece k, and nothing on the
// host waits for the GPU until the last piece is queued.  The sizes follow from two measured rates (HostScanState): with
// u = upload time and v = scan time per residue, piece k+1 may be r = 0.85 v/u times piece k and still land before
// piece k has been scanned; the first piece and the number of pieces minimise
// (upload of the first piece) + (pieces - 1) x (cost of a piece boundary).  plan_pieces() above.
struct PiecePlan {
    uint64_t rate_key = 0;              // host_scan_key of the scan
    double u_rate = 0, v_rate = 0;      // upload and scan ms per residue the sizes were planned with
    std::vector<int64_t> cut;           // piece k is subjects cut[k] .. cut[k + 1] - 1
};
// what this thread's host scans are planned from: the measured rates of its device and the previous plan
struct HostScanState {
    double h2d_ms_per_byte = 0;     // residue uploads of >= 4 MB
    uint64_t key = 0;               // the scan (function, query length, penalties) scan_ms_per_byte belongs to
    double scan_ms_per_byte = 0;    // kernel time per database residue of that scan
    int64_t last_total = 0;         // the previous plan: residues, scan and piece sizes
    uint64_t last_key = 0;
    std::vector<int64_t> last_sizes;
    // the rates are exponential averages: a new figure counts half
    static double average(double old, double now) { return old > 0 ? 0.5 * old + 0.5 * now : now; }
    // a finished piece's residue upload (both events have completed by now), counted once
    void note_upload(DbBuild &B) {
        if (!B.res_begin || !B.uploaded || !B.db || B.db->residues < ((int64_t)4 << 20)) return;
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, B.res_begin, B.uploaded) != cudaSuccess || ms <= 0.f) { cudaGetLastError(); return; }
        h2d_ms_per_byte = average(h2d_ms_per_byte, (double)ms / (double)B.db->residues);
        cudaEventDestroy(B.res_begin); B.res_begin = nullptr;
    }
    // a host scan of `total` residues whose kernels took `ms`
    void note_scan(uint64_t scan_key, double ms, int64_t total) {
        scan_ms_per_byte = average(key == scan_key ? scan_ms_per_byte : 0, ms / (double)total);
        key = scan_key;
    }
    // the pieces of a call, from the measured rates (defaults for what has not been measured yet)
    PiecePlan plan(const FnConfig &cfg, const parasail_profile_t *profile, int open, int gap, const int64_t *off, int64_t n) {
        PiecePlan pl;
        const int64_t total = off[n] - off[0];
        pl.rate_key = host_scan_key(cfg, (int)profile->query.size(), open, gap, profile->matrix.size);
        const double u_rate = pl.u_rate = h2d_ms_per_byte > 0 ? h2d_ms_per_byte : 1e3 / 50e9;
        const double v_rate = pl.v_rate = (key == pl.rate_key && scan_ms_per_byte > 0)
                                              ? scan_ms_per_byte
                                              : (double)profile->query.size() * 1e3 / (sw16_wanted(cfg) ? 4.9e12 : 1.5e12);
        std::vector<int64_t> sizes = plan_pieces(total, u_rate, v_rate);
        // hysteresis: the rates are measured and move a little from call to call; a plan that is still within 5 % of
        // the best one is kept, so that a service repeating a scan keeps its allocation sizes (a new size can mean a
        // host-blocking growth of the memory pool)
        auto exposed = [&](const std::vector<int64_t> &sz) {
            double t = (double)sz[0] * u_rate + 0.35 * (double)(sz.size() - 1);
            for (size_t k = 0; k + 1 < sz.size(); ++k) t += std::max(0.0, (double)sz[k + 1] * u_rate - (double)sz[k] * v_rate);
            return t;
        };
        if (last_total == total && last_key == pl.rate_key && !last_sizes.empty() && exposed(last_sizes) <= 1.05 * exposed(sizes) + 0.05) sizes = last_sizes;
        last_total = total; last_key = pl.rate_key; last_sizes = sizes;
        std::vector<int64_t> ends(sizes.size() - 1);   // residues up to the end of every piece but the last
        std::partial_sum(sizes.begin(), sizes.end() - 1, ends.begin());
        pl.cut = cut_subjects(off, n, ends);
        return pl;
    }
};
static thread_local HostScanState g_hs;

// one piece of a host scan: its uploads and packed shard, and its scan.  Destroying it gives the packed shard, the
// staging blocks and the result arrays back; the owner has synchronised the streams that used them.
struct HostPiece {
    DbBuild build;
    ScanJob job;
    ~HostPiece() { psb_db_free(build.db); }
};

// the query side, while the compute stream is idle: a profile's first use on a device uploads it and waits for that
// upload, which would otherwise happen inside the first piece's scan_enqueue, behind that piece's whole chain
static int prepare_query(const FnConfig &cfg, const parasail_profile_t *profile, int open, int gap) {
    DevProfile *dp = nullptr;
    PSB_TRY(get_dev_profile(profile, &dp));
    std::vector<Sw16Profile> sp;
    if (sw16_wanted(cfg)) sw16_prepare(profile, dp, open, gap, &sp);
    return PSB_OK;
}

// piece k's host pass over its offsets and its sort/pack chain.  PSB_DEBUG_TIMING also makes the chain's first mark
// wait for the piece's offsets, so that the timeline shows when they landed.
static int build_piece(HostPiece &p, const int64_t *off, int k, StreamMarks &tl, const HostClock &clk) {
    Ctx &c = g_ctx;
    const double h0 = clk.on ? clk.ms() : 0.0;
    int rc = db_host_pass(p.build, off);
    const double h1 = clk.on ? clk.ms() : 0.0;
    if (clk.on) { cudaStreamWaitEvent(c.stream, p.build.offs_up, 0); tl.mark(c.stream); }
    if (rc == PSB_OK) rc = db_finish(p.build, &tl);
    if (clk.on) std::fprintf(stderr, "[psb] scan_host(dev %d): piece %d host: offsets pass + allocations %.3f ms, chain launches %.3f ms\n", c.device, k, h1 - h0, clk.ms() - h1);
    tl.mark(c.stream);
    return rc;
}

// waits until the piece's results are on the host; its re-runs and its upload time are counted once
static int finish_piece(HostPiece &p, int64_t *n_retried) {
    int rc = PSB_OK;
    if (p.job.ev0 && !p.job.finished) { rc = scan_finish(p.job); *n_retried += p.job.retried; }
    g_hs.note_upload(p.build);
    return rc;
}

// `keep_last`: takes over the last piece once its results are on the host, for a caller with a better moment to give
// its device memory back (psb_scan_box's workers, after they have reported completion)
static int scan_host_into(const FnConfig &cfg, const parasail_profile_t *profile, int open, int gap, const uint8_t *cat,
                          const int64_t *off, int64_t n, int *const hosts[6], int64_t base, int64_t *n_retried,
                          std::unique_ptr<HostPiece> *keep_last = nullptr) {
    Ctx &c = g_ctx;
    const HostClock clk{};
    const PiecePlan pl = g_hs.plan(cfg, profile, open, gap, off, n);
    const std::vector<int64_t> &cut = pl.cut;
    const int npieces = (int)cut.size() - 1;
    const double ms_at_entry = c.last_ms;
    const bool pageable = is_pageable(cat + off[0]);
    if (clk.on) {
        std::string line;
        for (int k = 0; k < npieces; ++k) line += " " + std::to_string((off[cut[k + 1]] - off[cut[k]]) >> 20);
        std::fprintf(stderr, "[psb] scan_host(dev %d): pieces (MB):%s; upload %.1f GB/s, scan %.1f GB/s of residues\n", c.device, line.c_str(),
                     1e-6 / pl.u_rate, 1e-6 / pl.v_rate);
    }
    // a finished piece gives its device memory back, so at most kDepth pieces are resident however large the host
    // database is
    const int kDepth = 4;
    std::vector<std::unique_ptr<HostPiece>> pieces(npieces);
    int rc = PSB_OK;
    auto finish = [&](int k) {
        if (!pieces[k]) return;
        const int r = finish_piece(*pieces[k], n_retried);
        if (rc == PSB_OK) rc = r;
        pieces[k].reset();
    };
    // PSB_DEBUG_TIMING: a device-side timeline (upload landed / packing begins / scan begins / scan ends / results
    // on the host), relative to an event recorded on the idle compute stream at entry
    StreamMarks tl;
    // piece k goes up after piece k - kDepth is finished; its residues wait for piece k-1's chain
    auto upload = [&](int k) {
        if (k >= npieces || rc != PSB_OK) return;
        if (k >= kDepth) finish(k - kDepth);
        if (rc != PSB_OK) return;
        pieces[k].reset(new HostPiece());
        cudaEvent_t gate = k > 0 ? pieces[k - 1]->build.packed : nullptr;
        if (!db_upload(pieces[k]->build, cat, off + cut[k], cut[k + 1] - cut[k], profile->matrix, true, 0, gate)) rc = PSB_ECUDA;
        else tl.mark(c.copy);
    };
    auto scan = [&](int k) {
        if (rc == PSB_OK) rc = scan_enqueue(pieces[k]->job, cfg, profile, open, gap, pieces[k]->build.db, hosts, base + cut[k]);
        tl.mark(c.stream);
    };
    tl.mark(c.stream);
    upload(0);
    if (rc == PSB_OK) rc = prepare_query(cfg, profile, open, gap);
    if (clk.on) std::fprintf(stderr, "[psb] scan_host(dev %d): %d pieces, first upload queued at %.3f ms\n", c.device, npieces, clk.ms());
    for (int k = 0; k < npieces && rc == PSB_OK; ++k) {
        rc = build_piece(*pieces[k], off + cut[k], k, tl, clk);
        // the next upload goes in as soon as its gate (this piece's chain) exists -- unless the caller's memory is
        // pageable: then the upload is a memcpy loop on this thread (upload_h2d) and this piece's scan has to be on the
        // device first
        if (pageable) { scan(k); upload(k + 1); } else { upload(k + 1); scan(k); }
        if (clk.on) std::fprintf(stderr, "[psb] scan_host(dev %d): piece %d queued at %.3f ms\n", c.device, k, clk.ms());
    }
    // everything is queued: the host finishes the earlier pieces while the last ones are still being scanned
    for (int k = 0; k + 1 < npieces; ++k) finish(k);
    cudaStreamSynchronize(c.copy);
    if (clk.on) std::fprintf(stderr, "[psb] scan_host(dev %d): uploads done at %.3f ms\n", c.device, clk.ms());
    if (rc == PSB_OK) rc = finish_piece(*pieces[npieces - 1], n_retried);
    cudaStreamSynchronize(c.stream);
    if (clk.on) std::fprintf(stderr, "[psb] scan_host(dev %d): all done at %.3f ms\n", c.device, clk.ms());
    // order of the marks: entry | upload 0 | per piece k: [upload k+1] upload-k-landed (lengths< >lengths sort> <pack pack>) pack-end results-on-host
    if (clk.on && !tl.ev.empty()) std::fprintf(stderr, "[psb] scan_host(dev %d): device timeline (ms after entry):%s\n", c.device, tl.line().c_str());
    const int64_t total = off[n] - off[0];
    if (rc == PSB_OK && total >= ((int64_t)8 << 20) && c.last_ms > ms_at_entry) g_hs.note_scan(pl.rate_key, c.last_ms - ms_at_entry, total);
    if (keep_last && rc == PSB_OK) *keep_last = std::move(pieces[npieces - 1]);
    for (int k = 0; k < npieces; ++k) finish(k);
    return rc;
}

// ---- one worker thread per device for psb_scan_box: the thread keeps its context (streams, memory pool,
// staging blocks) warm across calls -----------------------------------------------------------------------
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
static BoxWorker *start_worker(int device) {
    BoxWorker *w = new BoxWorker();
    w->device = device;
    w->th = std::thread([w] { w->loop(); });
    w->th.detach();
    return w;
}
// ---- lanes for the passes of a large psb_align_pairs batch ------------------------------------------------
// Each lane is a resident host thread bound to the caller's device, with its own context (streams, events): the
// passes are handed out in order, so that while one lane's pass is in its kernels the other lane uploads and
// prepares the next one.  The passes write disjoint slices of the batch; what is not a slice comes back in PassOut.
static std::mutex g_lane_mu;
static std::map<std::pair<int, int>, BoxWorker *> g_lanes;   // (device, lane) -> worker; never destroyed
static BoxWorker *pair_lane(int device, int lane) {
    std::lock_guard<std::mutex> lk(g_lane_mu);
    BoxWorker *&w = g_lanes[{device, lane}];
    if (!w) w = start_worker(device);
    return w;
}
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

static std::mutex g_box_mu;
static std::vector<BoxWorker *> g_box;   // index = device; never destroyed (the threads live as long as the process)
static BoxWorker *box_worker(int device) {
    std::lock_guard<std::mutex> lk(g_box_mu);
    if ((int)g_box.size() <= device) g_box.resize(device + 1, nullptr);
    if (!g_box[device]) g_box[device] = start_worker(device);
    return g_box[device];
}
}  // namespace psb

extern "C" {

int psb_scan_host(const char *fn_name, const parasail_profile_t *profile, int open, int gap, const uint8_t *cat,
                  const int64_t *off, int64_t n, psb_batch_t **out) {
    if (out) *out = nullptr;
    FnConfig cfg;
    PSB_TRY(scan_check("psb_scan_host", fn_name, profile, &cfg));
    PSB_TRY(host_db_check("psb_scan_host", out, cat, off, n, true));
    PSB_TRY(ensure_ctx());
    Ctx &c = g_ctx;
    c.last_ms = 0.0; c.launches = 0;
    psb_batch_t *b = new_batch(n, cfg);
    if (!b) { set_error("pinned host allocation failed"); return PSB_ENOMEM; }
    const int rc = scan_host_into(cfg, profile, open, gap, cat, off, n, batch_outputs(b).data(), 0, &b->n_retried);
    if (rc != PSB_OK) { free_batch(b); return rc; }
    return scan_batch_done(cfg, profile, open, gap, off[n] - off[0], [&](int64_t i) { return span(off, i); }, b, out);
}

// The whole box from one process and one call (SURVEY 8b/8e): the database is cut into n_gpus contiguous
// ranges of equal residue count (contiguous, so every device uploads straight from the caller's arrays and
// writes straight into the caller-order result arrays -- no gather on either side), one resident worker
// thread per device runs the pipelined host scan on its range, and the call returns ONE batch in the
// caller's subject order.  No data-path collective: the ranges are independent.
int psb_scan_box(const char *fn_name, const parasail_profile_t *profile, int open, int gap, const uint8_t *cat,
                 const int64_t *off, int64_t n, int n_gpus, psb_batch_t **out) {
    if (out) *out = nullptr;
    FnConfig cfg;
    PSB_TRY(scan_check("psb_scan_box", fn_name, profile, &cfg));
    PSB_TRY(host_db_check("psb_scan_box", out, cat, off, n, true));
    const int ndev = psb_device_count();
    if (ndev <= 0) { set_error("no CUDA device available: libparasail_b200 has no CPU fallback (needs an sm_100a GPU)"); return PSB_ENODEV; }
    if (n_gpus <= 0 || n_gpus > ndev) n_gpus = ndev;
    if ((int64_t)n_gpus > n) n_gpus = (int)n;
    const HostClock clk{};
    PSB_TRY(ensure_ctx());   // the batch's pinned arrays are allocated by the calling thread
    psb_batch_t *b = new_batch(n, cfg);
    if (!b) { set_error("pinned host allocation failed"); return PSB_ENOMEM; }
    if (clk.on) std::fprintf(stderr, "[psb] scan_box: batch ready at %.3f ms\n", clk.ms());
    const int64_t total = off[n] - off[0];
    std::vector<int64_t> targets;
    for (int d = 1; d < n_gpus; ++d) targets.push_back(total * d / n_gpus);
    // device d scans range d; the devices past the last range have no work
    const std::vector<int64_t> cut = cut_subjects(off, n, targets);
    const int nranges = (int)cut.size() - 1;
    const std::array<int *, 6> hosts = batch_outputs(b);
    struct DeviceResult { int rc = PSB_OK, launches = 0; int64_t retried = 0; double ms = 0.0; std::string err; };
    std::vector<DeviceResult> res(nranges);
    for (int d = 0; d < nranges; ++d) {
        BoxWorker *w = box_worker(d);
        w->submit([&, d, w] {
            DeviceResult &r = res[d];
            r.rc = ensure_ctx();
            if (r.rc == PSB_OK) {
                g_ctx.last_ms = 0.0; g_ctx.launches = 0;
                r.rc = scan_host_into(cfg, profile, open, gap, cat, off + cut[d], cut[d + 1] - cut[d], hosts.data(), cut[d], &r.retried, &w->left);
                r.ms = g_ctx.last_ms; r.launches = g_ctx.launches;
            }
            if (r.rc != PSB_OK) r.err = psb_last_error();
        });
    }
    int rc = PSB_OK;
    Ctx &c = g_ctx;
    c.last_ms = 0.0; c.launches = 0;
    if (clk.on) std::fprintf(stderr, "[psb] scan_box: %d ranges submitted at %.3f ms\n", n_gpus, clk.ms());
    for (int d = 0; d < nranges; ++d) {
        box_worker(d)->wait();
        if (clk.on) std::fprintf(stderr, "[psb] scan_box: device %d done at %.3f ms\n", d, clk.ms());
        const DeviceResult &r = res[d];
        if (r.rc != PSB_OK && rc == PSB_OK) { rc = r.rc; set_error("psb_scan_box (device " + std::to_string(d) + "): " + r.err); }
        b->n_retried += r.retried;
        c.last_ms = std::max(c.last_ms, r.ms);   // the devices run side by side: the slowest one
        c.launches += r.launches;
    }
    if (rc != PSB_OK) { free_batch(b); return rc; }
    return scan_batch_done(cfg, profile, open, gap, total, [&](int64_t i) { return span(off, i); }, b, out);
}

int psb_batch_topk(const psb_batch_t *batch, int k, int64_t *idx_out, int *score_out) {
    if (!batch || k <= 0 || !idx_out) { set_error("psb_batch_topk: bad argument"); return PSB_EINVAL; }
    const int64_t n = batch->n;
    std::vector<int64_t> idx(n);
    std::iota(idx.begin(), idx.end(), 0);
    const int64_t kk = std::min<int64_t>(k, n);
    auto better = [&](int64_t a, int64_t b) { return batch->score[a] != batch->score[b] ? batch->score[a] > batch->score[b] : a < b; };
    std::partial_sort(idx.begin(), idx.begin() + kk, idx.end(), better);
    for (int64_t i = 0; i < kk; ++i) { idx_out[i] = idx[i]; if (score_out) score_out[i] = batch->score[idx[i]]; }
    return (int)kk;
}

int psb_trim(void) {
    PSB_TRY(ensure_ctx());
    Ctx &c = g_ctx;
    // this thread's kept buffers and those of the device's lanes
    release_kept();
    for (int t = 0; t < kPairLanes; ++t) {
        BoxWorker *w = nullptr;
        {
            std::lock_guard<std::mutex> lk(g_lane_mu);
            auto it = g_lanes.find({c.device, t});
            if (it != g_lanes.end()) w = it->second;
        }
        if (!w) continue;
        std::promise<void> done;
        w->submit([&] { if (ensure_ctx() == PSB_OK) { release_kept(); cudaStreamSynchronize(g_ctx.stream); } done.set_value(); });
        done.get_future().wait();
    }
    PSB_CUDA(cudaStreamSynchronize(c.stream));
    // recycled staging blocks of this device, recycled page-locked blocks, then the pool itself
    {
        std::lock_guard<std::mutex> lk(g_stage_mu);
        for (size_t i = 0; i < g_stage_free.size();) {
            if (g_stage_free[i].device == c.device) {
                cudaFree(g_stage_free[i].p);
                g_stage_cached -= g_stage_free[i].bytes;
                g_stage_free.erase(g_stage_free.begin() + (long)i);
            } else ++i;
        }
    }
    {
        std::lock_guard<std::mutex> lk(g_pin_mu);
        for (auto &kv : g_pin_free) cudaFreeHost(kv.second);
        g_pin_free.clear();
    }
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, c.device) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
    cudaGetLastError();
    return PSB_OK;
}

int psb_host_scan_plan(int64_t total, double upload_ms_per_byte, double scan_ms_per_byte, int64_t *sizes_out, int cap) {
    if (total <= 0 || upload_ms_per_byte <= 0 || scan_ms_per_byte <= 0 || !sizes_out || cap <= 0) { set_error("psb_host_scan_plan: bad argument"); return PSB_EINVAL; }
    const std::vector<int64_t> sizes = plan_pieces(total, upload_ms_per_byte, scan_ms_per_byte);
    for (size_t k = 0; k < sizes.size() && (int)k < cap; ++k) sizes_out[k] = sizes[k];
    return (int)sizes.size();
}

int psb_shard_plan(const int64_t *off, int64_t n, int n_shards, int *shard_of) {
    if (!off || !shard_of || n <= 0 || n_shards <= 0) { set_error("psb_shard_plan: bad argument"); return PSB_EINVAL; }
    // longest-processing-time first on residue counts: sort by length, give each subject to
    // the currently lightest shard (SURVEY 8e)
    std::vector<int64_t> order(n);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int64_t a, int64_t b) { return off[a + 1] - off[a] > off[b + 1] - off[b]; });
    std::vector<int64_t> load(n_shards, 0);
    for (int64_t t = 0; t < n; ++t) {
        const int64_t i = order[t];
        int best = 0;
        for (int s = 1; s < n_shards; ++s) if (load[s] < load[best]) best = s;
        shard_of[i] = best;
        load[best] += off[i + 1] - off[i];
    }
    return PSB_OK;
}

}  // extern "C"
