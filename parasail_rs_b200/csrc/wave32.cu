// wave32.cu -- one long pair over the whole GPU (kern_wave32.cuh), and the scan's subjects too long for the packed
// kernel: the three wavefront generations, their reduction and the walk of the traced launch.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "engine.h"
#include "kern_gotoh32.cuh"
#include "kern_wave32.cuh"
#include "pairs16_host.h"

namespace psb {

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

// Long pairs with traceback or statistics (WaveWalk) take the TRACE instantiation of the column-blocked generation
static constexpr int kWaveTraceK = 8;
static size_t wave_trace_bytes(int lq, int lr) { return (size_t)wave32v3_trace_records(lq, lr, kWaveTraceK) * 40; }
// preconditions of that path (anything else keeps the one-warp-per-pair kernels): the column-blocked generation's
// own, H bytes that identify a neighbour's value, every strip resident at once, and the trace fits in `avail` bytes
bool wave_walk_ok(const HostMatrix &m, int open, int gap, bool is_sw, int lq, int lr, size_t avail) {
    if (std::getenv("PSB_NO_WAVE_TRACE")) return false;
    if (!wave32_v2_ok(m, open, gap) || !pairs16_trace_ok(m.min, m.max, open)) return false;
    if ((lq + 32 * kWaveTraceK - 1) / (32 * kWaveTraceK) > g_ctx.sms * 16) return false;
    if (!wave32v3_range_ok(kWaveTraceK, 4, is_sw, lq, lr, m.max, m.min, open, gap)) return false;
    return wave_trace_bytes(lq, lr) + ((size_t)1 << 30) <= avail;
}

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

int launch_wave32(const Gotoh32Params &g, const HostMatrix &m, long long q_byte_off, int lq, long long r_byte_off, int lr, int out_index,
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
        const FreeEnds fe = free_ends(g);
        w.top_free = fe.top ? 1 : 0; w.left_free = fe.left ? 1 : 0;
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

int launch_wave_subjects(const FnConfig &cfg, const HostMatrix &m, const uint8_t *q, int lq, const int *matrix, int open, int gap,
                         const uint8_t *lbytes, const long long *loff, int64_t nroute, const int *out_map, int K, int nstrips, int *bnd, int *ctl,
                         int *cand, int *const d_out[6]) {
    Ctx &c = g_ctx;
    Wave32Params w;
    WaveReduceParams r;
    wave_params(cfg, q, lbytes, lq, 0, matrix, m.size, open, gap, nstrips, bnd, ctl, cand, d_out[0], d_out[1], d_out[2], &w, &r);
    w.multi_n = (int)nroute; w.r_off = loff;
    r.multi_n = (int)nroute; r.r_off = loff; r.out_map = out_map;
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
    c.launches += 2;
    return PSB_OK;
}

}  // namespace psb
