// ctx.cu -- the calling thread's context (device, streams, events), its device buffers and uploads, the process-wide
// page-locked and staging pools, batches, the resident worker threads, and the small C entry points.
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <cstring>
#include <future>
#include <map>
#include <numeric>

#include "engine.h"

namespace psb {

thread_local Ctx g_ctx;

int ensure_ctx() {
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

// Host->device copy that does not depend on the caller's memory being page-locked.  cudaMemcpyAsync out of
// pageable memory goes through the driver's own staging at a few GB/s with the calling thread blocked; large
// copies out of such memory are staged here instead, 8 MB at a time through two page-locked bounce buffers of the
// calling thread (memcpy of one chunk while the previous one is on the link).  Page-locked sources (and small
// copies) go straight to cudaMemcpyAsync.
static constexpr size_t kBounceBytes = (size_t)8 << 20;
bool is_pageable(const void *p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return at.type == cudaMemoryTypeUnregistered;
}
cudaError_t upload_h2d(void *dst, const void *src, size_t bytes, cudaStream_t stream) {
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

void release_kept() {
    Ctx &c = g_ctx;
    for (Ctx::Kept &k : c.kept) {
        if (k.p) cudaFreeAsync(k.p, c.stream);
        k.p = nullptr; k.cap = 0;
    }
}

// pinned host blocks are slow to create; recycle them process-wide by size class
static std::mutex g_pin_mu;
static std::multimap<size_t, void *> g_pin_free;
void *pinned_alloc(size_t bytes) {
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
void pinned_free(void *p, size_t bytes) {
    if (!p) return;
    size_t cls = 4096;
    while (cls < bytes) cls <<= 1;
    std::lock_guard<std::mutex> lk(g_pin_mu);
    if (g_pin_free.size() < 64) g_pin_free.emplace(cls, p);
    else cudaFreeHost(p);
}

// a batch's per-pair result arrays in the order the kernels' outputs use (score, end_query, end_ref, then the statistics)
std::array<int *, 6> batch_outputs(psb_batch_t *b) { return {b->score, b->end_query, b->end_ref, b->matches, b->similar, b->length}; }
// the length of sequence i of a concatenation
int span(const int64_t *off, int64_t i) { return (int)(off[i + 1] - off[i]); }

void fill_lut(unsigned *lut, const uint8_t *mapper) {
    for (int i = 0; i < 64; ++i)
        lut[i] = (unsigned)mapper[4 * i] | ((unsigned)mapper[4 * i + 1] << 8) | ((unsigned)mapper[4 * i + 2] << 16) |
                 ((unsigned)mapper[4 * i + 3] << 24);
}

// what a new allocation can get: the driver's free figure + what the stream-ordered pool holds idle (0 if the driver
// cannot say).  Counting only the former would make a figure that shrinks as the pool warms up: every call would then
// cut its passes differently, ask for buffers of new sizes, grow the pool again ... -- calls of 2 s instead of 0.3 s.
size_t device_mem_available() {
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

psb_batch_t *new_batch(int64_t n, const FnConfig &cfg) {
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

// Device staging blocks for psb_scan_host's uploads.  They are filled on the copy stream while the
// compute stream is busy, so they cannot come from a stream-ordered pool without tying the two
// streams together (an allocation that cannot reuse a block freed on the other stream falls back to
// mapping fresh memory, a host-blocking call of tens of milliseconds).  Plain allocations, recycled
// process-wide; a block is handed back only after both streams have been synchronised.
struct StageBlock { void *p; size_t bytes; int device; };
static std::mutex g_stage_mu;
static std::vector<StageBlock> g_stage_free;
static size_t g_stage_cached = 0;
void *stage_acquire(int device, size_t need, size_t *got) {
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
void stage_release(int device, void *p, size_t bytes) {
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

BoxWorker *start_worker(int device) {
    BoxWorker *w = new BoxWorker();
    w->device = device;
    w->th = std::thread([w] { w->loop(); });
    w->th.detach();
    return w;
}

// the lanes of the pairs pass (run_pairs_lanes, pairs.cu)
static std::mutex g_lane_mu;
static std::map<std::pair<int, int>, BoxWorker *> g_lanes;   // (device, lane) -> worker; never destroyed
BoxWorker *pair_lane(int device, int lane) {
    std::lock_guard<std::mutex> lk(g_lane_mu);
    BoxWorker *&w = g_lanes[{device, lane}];
    if (!w) w = start_worker(device);
    return w;
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
