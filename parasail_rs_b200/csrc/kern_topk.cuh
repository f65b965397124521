// kern_topk.cuh -- selection of the kk best subjects of one query's scan on the device (psb_db_search, search.cu).
//
// The rule is psb_batch_topk's: score descending, then smaller caller id.  A radix select on the order-preserving key
// score ^ 0x80000000 decides the key T of the kk-th best subject eight bits per pass (four histogram / pick pairs),
// and leaves in TopkState how many subjects lie above T and how many are still needed from T.  An ordered compaction
// then takes every subject above T and the first `need` subjects equal to T in caller-id order, so that ties at the
// threshold go to the smaller ids.  Each warp owns a contiguous chunk of ids; its counts go through an exclusive sum
// (exclusive_sum, db.cu) and give it its output offsets.  Every launch reads the previous one's result from device
// memory: nothing returns to the host between a scan and its selection.  The kk rows come out in caller-id order
// within each class (above T, then equal to T), not in score order.
#pragma once
#include "psb_simt.h"

namespace psb {

static constexpr int kTopkBins = 256;

struct TopkState {
    unsigned prefix;   // the key bits decided so far; after the last pass, T itself
    unsigned mask;     // which bits those are
    int need;          // subjects still wanted among those whose key matches prefix under mask
    int above;         // subjects whose key is above every key that matches
    int hist[kTopkBins];
};

// explicit _8 / _16 widths: the rule of saturates() (result.cpp) for one query against every subject, in the form
// a kernel can apply.  A subject saturates when score > score_hi, score < score_lo, or max(qlen, its length) > len_hi;
// its score, end_query and end_ref then read 0 (flag_saturated), before the selection sees them.
struct TopkSat {
    int score_hi, score_lo, len_hi, qlen;
    const int *len_sorted;   // subject lengths in sorted order (psb_db::d_len)
    const int *inv_perm;     // caller id -> sorted position
};

struct TopkParams {
    int *score, *end_query, *end_ref;   // the scan's n per-subject results, caller order
    long long n;
    int kk;
    TopkState *st;
    int shift;                 // histogram / pick: the byte of the key this pass decides (24, 16, 8, 0)
    long long chunk;           // count / write: ids per warp (a multiple of 32)
    int nwarps;
    int *counts;               // 2 * nwarps: per warp, its subjects above T, then its subjects equal to T
    const long long *offs;     // exclusive sum of counts
    int *sat;                  // n flags of the saturation pass, or nullptr
    int *out_id, *out_score, *out_end_query, *out_end_ref, *out_sat;   // kk rows
};

PSB_HD unsigned topk_key(int score) { return (unsigned)score ^ 0x80000000u; }
// ids per warp of the compaction for `nwarps` warps over n subjects
PSB_HD long long topk_chunk(long long n, int nwarps) { return ((n + nwarps - 1) / nwarps + 31) / 32 * 32; }

// explicit widths: zero the results that do not fit and flag them
PSB_KERNEL void topk_saturate_kernel(TopkParams p, TopkSat s) {
    const long long stride = (long long)grid_blocks() * threads_per_block();
    for (long long i = (long long)block_id() * threads_per_block() + thread_in_block(); i < p.n; i += stride) {
        const int sc = p.score[i];
        const int lr = s.len_sorted[s.inv_perm[i]];
        const bool bad = sc > s.score_hi || sc < s.score_lo || (s.qlen > lr ? s.qlen : lr) > s.len_hi;
        p.sat[i] = bad ? 1 : 0;
        if (bad) { p.score[i] = 0; p.end_query[i] = 0; p.end_ref[i] = 0; }
    }
}

// one pass of the radix select: the histogram of the byte at `shift` over the keys that match the prefix so far.
// Dynamic shared memory: kTopkBins ints.
PSB_KERNEL void topk_hist_kernel(TopkParams p) {
    PSB_SHARED_DECL(smem_raw);
    int *h = (int *)smem_raw;
    const unsigned prefix = p.st->prefix, mask = p.st->mask;
    for (int b = thread_in_block(); b < kTopkBins; b += threads_per_block()) h[b] = 0;
    sync_block();
    const long long stride = (long long)grid_blocks() * threads_per_block();
    for (long long i = (long long)block_id() * threads_per_block() + thread_in_block(); i < p.n; i += stride) {
        const unsigned key = topk_key(p.score[i]);
        if ((key & mask) == prefix) atomic_add(&h[(key >> p.shift) & 255u], 1);
    }
    sync_block();
    for (int b = thread_in_block(); b < kTopkBins; b += threads_per_block())
        if (h[b]) atomic_add(&p.st->hist[b], h[b]);
}

// and its decision (one block): the highest byte value at which the count from the top reaches `need`.  The first
// pass (shift 24) starts from need = kk on a zeroed state.  The histogram is cleared for the next pass.
PSB_KERNEL void topk_pick_kernel(TopkParams p) {
    TopkState *st = p.st;
    if (thread_in_block() == 0) {
        int need = p.shift == 24 ? p.kk : st->need, above = p.shift == 24 ? 0 : st->above;
        int b = kTopkBins - 1;
        for (; b > 0; --b) {
            const int h = st->hist[b];
            if (h >= need) break;
            need -= h; above += h;
        }
        st->need = need; st->above = above;
        st->prefix |= (unsigned)b << p.shift;
        st->mask |= 255u << p.shift;
    }
    sync_block();
    for (int b = thread_in_block(); b < kTopkBins; b += threads_per_block()) st->hist[b] = 0;
}

// the compaction, warp by warp over contiguous chunks of ids: COUNT the warp's subjects above T and equal to T, or
// (WRITE, offsets known) write the rows: subjects above T at their rank among those, subjects equal to T at
// above + their rank among those while that is below kk
template <bool WRITE> PSB_KERNEL void topk_take_kernel(TopkParams p) {
    const int w = block_id() * warps_per_block() + warp_in_block();
    if (w >= p.nwarps) return;
    const unsigned T = p.st->prefix;
    const long long lo = (long long)w * p.chunk < p.n ? (long long)w * p.chunk : p.n;
    const long long hi = lo + p.chunk < p.n ? lo + p.chunk : p.n;
    long long na = WRITE ? p.offs[w] : 0, ne = WRITE ? p.offs[p.nwarps + w] : 0;
    const unsigned below = (1u << lane_id()) - 1u;
    for (long long base = lo; base < hi; base += 32) {
        const long long i = base + lane_id();
        const unsigned key = i < hi ? topk_key(p.score[i]) : 0u;
        const bool a = i < hi && key > T, e = i < hi && key == T;
        const unsigned ba = ballot(a), be = ballot(e);
        if (WRITE && (a || e)) {
            const long long pos = a ? na + pop_count(ba & below) : ne + pop_count(be & below);
            if (pos < p.kk) {
                p.out_id[pos] = (int)i;
                p.out_score[pos] = p.score[i];
                p.out_end_query[pos] = p.end_query[i];
                p.out_end_ref[pos] = p.end_ref[i];
                p.out_sat[pos] = p.sat ? p.sat[i] : 0;
            }
        }
        na += pop_count(ba);
        ne += pop_count(be);
    }
    if (!WRITE && lane_id() == 0) { p.counts[w] = (int)na; p.counts[p.nwarps + w] = (int)ne; }
}

}  // namespace psb
