// emu_kernels.cpp -- TEST ONLY.  Compiles the product's kernel sources with -DPSB_EMULATE
// (every lane an OS thread, see csrc/psb_simt.h) so that the warp programs can be stepped
// on a CPU-only box and compared with the oracle before any GPU time is spent.
#define PSB_EMULATE 1
#ifdef EMU_NO_PINGPONG
#define SW16_PINGPONG 0
#endif
#include "../../parasail_rs_b200/csrc/kern_gotoh32.cuh"
#include <cstdio>

using namespace psb;

static bool g_prof = false;
template <int K, bool STATS, bool TRACE, typename W>
static void run32(const Gotoh32Params &p, int nblocks) {
    size_t smem = gotoh32_smem_bytes(p.size, 1, STATS, sizeof(W), g_prof);
    if (p.tabH) emu::launch(nblocks, smem, [&]() { gotoh32_kernel<K, STATS, TRACE, true, W>(p); });
    else if (g_prof) emu::launch(nblocks, smem, [&]() { gotoh32_kernel<K, STATS, TRACE, false, W, true>(p); });
    else emu::launch(nblocks, smem, [&]() { gotoh32_kernel<K, STATS, TRACE, false, W>(p); });
}

extern "C" void emu_gotoh32_use_profile(int on) { g_prof = on != 0; }

extern "C" int emu_gotoh32(int K, int stats, int trace, int wide_stats, const Gotoh32Params *pp, int nblocks) {
    Gotoh32Params p = *pp;
#define CASE(KK)                                                                              \
    case KK:                                                                                  \
        if (trace) run32<KK, false, true, unsigned>(p, nblocks);                              \
        else if (stats && wide_stats) run32<KK, true, false, unsigned long long>(p, nblocks); \
        else if (stats) run32<KK, true, false, unsigned>(p, nblocks);                         \
        else run32<KK, false, false, unsigned>(p, nblocks);                                   \
        return 0;
    switch (K) {
        CASE(1) CASE(2) CASE(3) CASE(4) CASE(8) CASE(16)
    }
    return -1;
}
extern "C" int emu_sizeof_params() { return (int)sizeof(Gotoh32Params); }

// ---- packed 16-bit scan kernel ------------------------------------------------------------------
#include "../../parasail_rs_b200/csrc/kern_sw16.cuh"

extern "C" int emu_sw16_build(const uint8_t *mapped_query, int lq, const int *table, int size, int open,
                              int8_t *out, int cap, int *K, int *max_score, int *chunks) {
    Sw16Profile pr;
    std::vector<int8_t> host;
    if (!sw16_build_profile(mapped_query, lq, table, size, open, &pr, &host)) return -1;
    if ((int)host.size() > cap) return -2;
    std::memcpy(out, host.data(), host.size());
    *K = pr.K; *max_score = pr.max_score; *chunks = pr.chunks;
    return (int)host.size();
}

extern "C" int emu_sw16(int K, const Sw16Params *pp, int nblocks) {
    Sw16Params p = *pp;
    size_t smem = sw16_smem_bytes(p.nletters, K, 1);
#define SCASE(KK) case KK: emu::launch(nblocks, smem, [&]() { sw16_scan_kernel<KK>(p); }); return 0;
    switch (K) { SCASE(4) SCASE(8) SCASE(12) SCASE(16) SCASE(20) SCASE(25) SCASE(28) SCASE(32) }
    return -1;
}
extern "C" int emu_sizeof_sw16() { return (int)sizeof(Sw16Params); }

// ---- long-pair wavefront kernel -------------------------------------------------------------------
#include "../../parasail_rs_b200/csrc/kern_wave32.cuh"

static bool g_wave_v2 = false;
static int g_wave_gen = 1;   // 1, 2, or 3 (column-blocked, local alignment only)
extern "C" void emu_wave32_use_v2(int on) { g_wave_v2 = on == 1; g_wave_gen = on == 2 ? 3 : (on == 1 ? 2 : 1); }
extern "C" int emu_wave32(int K, const Wave32Params *pp, const WaveReduceParams *rp, int nblocks) {
    Wave32Params p = *pp;
    if (g_wave_gen == 3) {
        size_t smem3 = wave32v3_smem_bytes(p.size, 1, K);
        switch (K) {
#define W3CASE(KK) case KK: if (p.mode == MODE_SW) emu::launch(nblocks, smem3, [&]() { wave32v3_kernel<KK, 4, true>(p); }); else emu::launch(nblocks, smem3, [&]() { wave32v3_kernel<KK, 4, false>(p); }); break;
            W3CASE(4) W3CASE(8) W3CASE(16)
            default: return -1;
        }
        WaveReduceParams r3 = *rp;
        emu::launch((r3.multi_n + 31) / 32 + (r3.multi_n == 0), 64, [&]() { wave32_reduce_kernel(r3); });
        return 0;
    }
    size_t smem = g_wave_v2 ? wave32v2_smem_bytes(p.size, 1) : wave32_smem_bytes(p.size, 1);
#define WCASE(KK) case KK: if (g_wave_v2) emu::launch(nblocks, smem, [&]() { wave32v2_kernel<KK>(p); }); else emu::launch(nblocks, smem, [&]() { wave32_kernel<KK>(p); }); break;
    switch (K) { WCASE(1) WCASE(2) WCASE(4) WCASE(8) default: return -1; }
    WaveReduceParams r = *rp;
    emu::launch((r.multi_n + 31) / 32 + (r.multi_n == 0), 64, [&]() { wave32_reduce_kernel(r); });
    return 0;
}
extern "C" int emu_sizeof_wave32() { return (int)sizeof(Wave32Params); }
extern "C" int emu_sizeof_wavereduce() { return (int)sizeof(WaveReduceParams); }

// long pair WITH traceback / statistics: TRACE instantiation of the column-blocked kernel + walk32_kernel.
// q / r are mapped residues.  what: 1 = CIGAR walk (rev_ops: lq + lr + 2 words, reversed run list), 2 = statistics walk.
// out: score, end_query, end_ref, then (what == 1) nops, beg_query, beg_ref or (what == 2) matches, similar, length.
extern "C" int emu_wave32_trace(const uint8_t *q, int lq, const uint8_t *r, int lr, const int *table, int size, int open, int gap,
                                int mode, int s1_beg, int s1_end, int s2_beg, int s2_end, int what, int nblocks, int *out, unsigned *rev_ops) {
    constexpr int K = 8;
    const int nstrips = (lq + 32 * K - 1) / (32 * K);
    std::vector<long long> bnd((size_t)nstrips * lr + 8, 0);
    std::vector<int> cand((size_t)nstrips * 8 + 8, 0);
    int next = 0;
    const long long nrec = wave32v3_trace_records(lq, lr, K);
    std::vector<uint4> th((size_t)nrec * 2 + 2);
    std::vector<uint2> tb((size_t)nrec + 2);
    std::memset(th.data(), 0xee, th.size() * sizeof(uint4));
    std::memset(tb.data(), 0xee, tb.size() * sizeof(uint2));
    Wave32Params p;
    std::memset(&p, 0, sizeof(p));
    p.q = q; p.r = r; p.Lq = lq; p.Lr = lr; p.matrix = table; p.size = size; p.open = open; p.gap = gap;
    p.mode = mode; p.s1_beg = s1_beg; p.s1_end = s1_end; p.s2_beg = s2_beg; p.s2_end = s2_end;
    p.bnd = (int *)bnd.data(); p.next_strip = &next; p.cand = cand.data();
    p.trace_h = th.data(); p.trace_bits = tb.data();
    const size_t smem = wave32v3_smem_bytes(size, 1, K);
    if (mode == MODE_SW) emu::launch(nblocks, smem, [&]() { wave32v3_kernel<K, 4, true, true>(p); });
    else emu::launch(nblocks, smem, [&]() { wave32v3_kernel<K, 4, false, true>(p); });
    WaveReduceParams rp;
    std::memset(&rp, 0, sizeof(rp));
    rp.cand = cand.data(); rp.nstrips = nstrips; rp.mode = mode; rp.s1_end = s1_end; rp.s2_end = s2_end; rp.Lr = lr;
    rp.score = out; rp.end_query = out + 1; rp.end_ref = out + 2;
    emu::launch(1, 64, [&]() { wave32_reduce_kernel(rp); });
    const long long rev_off = 0;
    Walk32Params w;
    std::memset(&w, 0, sizeof(w));
    w.q = q; w.r = r; w.Lq = lq; w.Lr = lr; w.K = K; w.trace_h = th.data(); w.trace_bits = tb.data();
    w.matrix = table; w.size = size; w.open = open; w.gap = gap; w.is_sw = mode == MODE_SW;
    w.top_free = (mode == MODE_SW || (mode == MODE_SG && s1_beg)) ? 1 : 0;
    w.left_free = (mode == MODE_SW || (mode == MODE_SG && s2_beg)) ? 1 : 0;
    w.pid = 0; w.score = out; w.end_query = out + 1; w.end_ref = out + 2;
    w.rev_ops = rev_ops; w.rev_off = &rev_off; w.nops = out + 3; w.beg_query = out + 4; w.beg_ref = out + 5;
    w.matches = out + 3; w.similar = out + 4; w.length = out + 5;
    if (what == 2) emu::launch(1, walk32_smem_bytes(size), [&]() { walk32_kernel<true>(w); });
    else emu::launch(1, walk32_smem_bytes(size), [&]() { walk32_kernel<false>(w); });
    return 0;
}

// ---- packed 16-bit many-pairs kernel + walk -------------------------------------------------------------
#include "../../parasail_rs_b200/csrc/kern_pairs16.cuh"

template <int G, int K> static void run_p16(const Pairs16Params &p, bool sw, bool trace, int nblocks, size_t smem) {
    if (sw && trace) emu::launch(nblocks, smem, [&]() { pairs16_kernel<G, K, true, true>(p); });
    else if (sw) emu::launch(nblocks, smem, [&]() { pairs16_kernel<G, K, true, false>(p); });
    else if (trace) emu::launch(nblocks, smem, [&]() { pairs16_kernel<G, K, false, true>(p); });
    else emu::launch(nblocks, smem, [&]() { pairs16_kernel<G, K, false, false>(p); });
}

// pairs are taken two at a time in the given order; q / r are already mapped to matrix indices.
// what: 0 = score only, 1 = trace + CIGAR walk (rev_ops: per pair region of lq+lr+2 words, reversed run list),
// 2 = trace + statistics walk.  Returns 0, -1 for an unsupported class, -2 when a pair does not fit 16 bit.
extern "C" int emu_pairs16(int G, int K, int mode, int s1_beg, int s1_end, int s2_beg, int s2_end, int what, int n,
                           const uint8_t *q, const long long *q_off, const uint8_t *r, const long long *r_off,
                           const int *table, int size, int mat_min, int mat_max, int open, int gap, int nblocks,
                           int *score, int *end_query, int *end_ref, int *matches, int *similar, int *length,
                           unsigned *rev_ops, const long long *rev_off, int *nops, int *beg_query, int *beg_ref) {
    const bool sw = mode == MODE_SW, trace = what != 0;
    if (!pairs16_scheme_ok(size, mat_min, mat_max, open, gap, false) || (what != 0 && !pairs16_trace_ok(mat_min, mat_max, open))) return -2;
    std::vector<int> items;
    for (int i = 0; i < n; i += 2) { items.push_back(i); items.push_back(i + 1 < n ? i + 1 : -1); }
    const int nitems = (int)items.size() / 2;
    std::vector<long long> toff(nitems + 1, 0);
    std::vector<int> slot_of(n);
    for (int w = 0; w < nitems; ++w) {
        int lrmax = 0;
        for (int h = 0; h < 2; ++h) {
            const int pid = items[2 * w + h];
            if (pid < 0) continue;
            const int lq = (int)(q_off[pid + 1] - q_off[pid]), lr = (int)(r_off[pid + 1] - r_off[pid]);
            if (lq > G * K || !pairs16_fits(G * K, lq, lr, mat_max, mat_min, open, gap, sw)) return -2;
            lrmax = std::max(lrmax, lr);
            slot_of[pid] = 2 * w + h;
        }
        toff[w + 1] = toff[w] + (trace ? pairs16_item_trace_words(G, K, lrmax) : 0);
    }
    std::vector<unsigned> tr((size_t)toff[nitems] + 16, 0xdeadbeefu);
    std::vector<int8_t> mat8(33 * 32);
    const bool top_free = sw || (mode == MODE_SG && s1_beg);
    pairs16_build_mat8(table, size, open, top_free, mat8.data());
    int counter = 0;
    Pairs16Params p;
    std::memset(&p, 0, sizeof(p));
    p.q = q; p.q_off = q_off; p.r = r; p.r_off = r_off; p.shared_query = 0;
    p.items = items.data(); p.nitems = nitems; p.mat8 = mat8.data(); p.size = size; p.open = open; p.gap = gap;
    p.mode = mode; p.s1_beg = s1_beg; p.s1_end = s1_end; p.s2_beg = s2_beg; p.s2_end = s2_end;
    p.score = score; p.end_query = end_query; p.end_ref = end_ref;
    p.trace = tr.data(); p.trace_off = toff.data(); p.counter = &counter;
    const size_t smem = pairs16_smem_bytes(K, size + 1, sw, 1);
#define PCASE(GG, KK) if (G == GG && K == KK) { run_p16<GG, KK>(p, sw, trace, nblocks, smem); } else
    PCASE(16, 1) PCASE(16, 3) PCASE(16, 4) PCASE(16, 8) PCASE(16, 10) PCASE(16, 19) PCASE(32, 2) PCASE(32, 9) PCASE(32, 16) { return -1; }
    if (trace) {
        std::vector<int> ids(n);
        for (int i = 0; i < n; ++i) ids[i] = i;
        Walk16Params w;
        std::memset(&w, 0, sizeof(w));
        w.q = q; w.q_off = q_off; w.r = r; w.r_off = r_off; w.pair_ids = ids.data(); w.pair_slot = slot_of.data(); w.n = n;
        w.G = G; w.K = K; w.trace = tr.data(); w.trace_off = toff.data(); w.matrix = table; w.size = size;
        w.open = open; w.gap = gap; w.is_sw = sw ? 1 : 0; w.top_free = top_free ? 1 : 0; w.left_free = (sw || (mode == MODE_SG && s2_beg)) ? 1 : 0; w.score = score; w.end_query = end_query; w.end_ref = end_ref;
        w.rev_ops = rev_ops; w.rev_off = rev_off; w.nops = nops; w.beg_query = beg_query; w.beg_ref = beg_ref;
        w.matches = matches; w.similar = similar; w.length = length;
        if (what == 2) emu::launch((n + 31) / 32, walk16_smem_bytes(size), [&]() { walk16_kernel<true>(w); });
        else emu::launch((n + 31) / 32, walk16_smem_bytes(size), [&]() { walk16_kernel<false>(w); });
    }
    return 0;
}

// ---- strip-wise scan of a long query (STRIP instantiations of the scan kernel), host loop as in scan.cu ----
extern "C" int emu_sw16_strips(const uint8_t *mapped_query, int lq, const int *table, int size, int open, int gap, int rows_per_strip,
                               const unsigned *words, const long long *word_off, const int *len, int bits, long long n,
                               const int *out_map, int *score, int *end_query, int *end_ref, int *retry, int *retry_count, int nblocks) {
    std::vector<long long> res_off((size_t)n + 1, 0);
    for (long long i = 0; i < n; ++i) res_off[(size_t)i + 1] = res_off[(size_t)i] + len[i];
    std::vector<uint2> bndA((size_t)res_off[(size_t)n] + 64), bndB((size_t)res_off[(size_t)n] + 64);
    const int nstrips = (lq + rows_per_strip - 1) / rows_per_strip;
    if (rows_per_strip % SW16_G != 0 || sw16_pick_k(rows_per_strip) * SW16_G != rows_per_strip) return -4;   // full strips only
    for (int st = 0; st < nstrips; ++st) {
        const int r0 = st * rows_per_strip, nr = std::min(rows_per_strip, lq - r0);
        Sw16Profile pr;
        std::vector<int8_t> host;
        if (!sw16_build_profile(mapped_query + r0, nr, table, size, open, &pr, &host)) return -1;
        if (!sw16_supported(pr, open, gap)) return -2;
        int counter = 0;
        Sw16Params p;
        std::memset(&p, 0, sizeof(p));
        p.prof = host.data(); p.nletters = pr.nletters; p.lq = nr; p.open = open; p.gap = gap; p.max_score = pr.max_score;
        p.words = words; p.word_off = word_off; p.len = len; p.bits = bits; p.n = n; p.out_map = out_map;
        p.score = score; p.end_query = end_query; p.end_ref = end_ref; p.retry = retry; p.retry_count = retry_count;
        p.counter = &counter; p.mul_one = 1u; p.mul_64k = 65536u;
        p.res_off = res_off.data();
        p.bnd_in = st == 0 ? nullptr : ((st & 1) ? bndA.data() : bndB.data());
        p.bnd_out = st + 1 == nstrips ? nullptr : ((st & 1) ? bndB.data() : bndA.data());
        p.row0 = r0; p.merge = st > 0;
        const size_t smem = sw16_smem_bytes(p.nletters, pr.K, 1, true);
        switch (pr.K) {
#define STCASE(KK) case KK: emu::launch(nblocks, smem, [&]() { sw16_scan_kernel<KK, true>(p); }); break;
            STCASE(4) STCASE(8) STCASE(12) STCASE(16)
            default: return -3;
        }
    }
    return 0;
}
