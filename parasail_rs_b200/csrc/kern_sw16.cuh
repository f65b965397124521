// kern_sw16.cuh -- the database-scan hot kernel: Smith-Waterman score + end cell of ONE resident
// query profile against the resident bit-packed database, in packed 16-bit lanes
// (DPX VIADDMNMX.S16x2 / VIMNMX3.S16x2), two subjects per 16-lane group, two groups per warp.
//
// Replaces upstream parasail_sw_{striped,scan}_profile_{16,sat} as reached from parasail-rs's
// profile aligner [REF src/aligner/mod.rs:431-450]; results follow SURVEY.md Appendix A
// (score; smallest end_ref among maxima; smallest end_query in that column).
//
// Design (B200-first; nothing here mirrors parasail's striped CPU layout):
//   * a group of G = 16 lanes is a 16-stage systolic array: lane t owns K consecutive query rows
//     in registers and fills reference column j = s - t at step s; the bottom row of a lane
//     travels to the next lane by shfl_up.  A warp runs two groups (four subjects) at once.
//   * each 32-bit register holds the same cell of TWO different subjects (lo/hi half), so one
//     DPX instruction updates two cells and there is no dependency inside a word.
//   * values are kept shifted by `open`:  X = H + o,  T = X - o = H,  E' = E + o,  F' = F + o.
//     In that space the local-alignment floor is the constant o, every value stays inside
//     [0, 32767] (no -inf sentinels), and T = X - (o,o) is a plain 32-bit operation that can never
//     borrow across the halves:
//        E' = max(E' - e, Tleft)      F' = max(F'up - e, Tup)       h = max(Tdiag + (S+o), E')
//        X  = max(h, F', o)           T  = X - o              (4 DPX ops + 1 add per two cells)
//   * query profile: int8 (S+o) in shared memory, laid out [letter][16-row chunk][lane][16 B] so
//     that one LDS.128 fetches 16 rows of one subject letter and the 8 lanes of a quarter-warp
//     always hit 8 different 16-byte bank groups (conflict free whatever the letters are); PRMT
//     with sign-replicating selectors interleaves the two subjects' scores into one 16x2 word.
//   * end cell: only the column maximum is formed per step (VIMNMX3 over the lane's rows) and
//     compared with a threshold that is the larger of the lane's own best and (the group's best,
//     published through shared memory) - 1.  Beating it is rare (a few dozen times per subject),
//     so the bookkeeping sits in a cold branch that records score and column and parks the
//     lane's column of H values in shared memory; the row is resolved once per subject from the
//     parked column of the winning lane.  Lanes are merged with parasail's tie-break (score,
//     then smaller end_ref, then smaller end_query).
//   * 16-bit overflow: subjects whose score reaches 32767 - o - max(S) are re-run at 32 bit.
#pragma once
#include "psb_defs.h"
#include "psb_simt.h"

#include <vector>

namespace psb {

static constexpr int SW16_G = 16;  // lanes per group

// SW16_PROF32=1: the profile holds one 32-bit word (S+o, zero-extended 16 bit) per letter and row, and
// the two subjects' scores are joined by (b << 16) + a, an add-class instruction that issues at twice
// the rate of the DPX/PRMT pipe the recurrence saturates.  SW16_PROF32=0: int8 profile joined by PRMT
// (4x less shared-memory traffic, one more instruction per row on the saturated pipe).
#ifndef SW16_PROF32
#define SW16_PROF32 1
#endif
// SW16_DECOUPLE=1: the recurrence is kept in true (unshifted) space with the vertical gap carried as
// Fh = F + open, so that the only loop-carried dependency between the rows of a lane is ONE instruction:
//    E  = max(E - e, Tleft)            Tleft = H[i][j-1] - o
//    h  = max(Tdiag + (S+o), E)        = max(H[i-1][j-1] + S, E)
//    H  = max(Fh - o, h, 0)            VIADDMNMX.S16x2.RELU
//    Fh'= max(Fh - e, h)               the chain; equals max(Fh - e, H) wherever it can matter (needs o >= e)
//    T  = H - o                        VIADD.16x2, off the chain
// (4 DPX + 1 packed add per two cells, as before, but the X -> T -> F' chain of three dependent
// instructions per row becomes one, so a warp needs far fewer partners to keep its scheduler busy.)
#ifndef SW16_DECOUPLE
#define SW16_DECOUPLE 1
#endif
// rows of one letter that one LDS.128 fetches for a lane
static constexpr int SW16_ROWS_PER_LOAD = SW16_PROF32 ? 4 : 16;
inline constexpr int sw16_chunks(int K) { return (K + SW16_ROWS_PER_LOAD - 1) / SW16_ROWS_PER_LOAD; }
// words per lane and half of the parked H column (>= K, a multiple of 4)
inline constexpr int sw16_park_words(int K) { return SW16_PROF32 ? ((K + 3) / 4) * 4 : ((K + 15) / 16) * 16; }

struct Sw16Profile {
    int8_t *prof = nullptr;  // device: [nletters][chunks][16 lanes][16 bytes] of (S + open); pad letter last
    int lq = 0;
    int K = 0;               // rows per lane
    int chunks = 0;          // sw16_chunks(K): 16-byte loads per lane and letter
    int nletters = 0;        // alphabet size + 1 (the pad letter)
    int max_score = 0, min_score = 0;
    int open_baked = -1;
    int row0 = 0;            // first query row this profile covers (strip profiles of long queries)
};

static const int kSw16K[] = {4, 8, 12, 16, 20, 25, 28, 32};
inline int sw16_pick_k(int lq) {
    for (int k : kSw16K) if (SW16_G * k >= lq) return k;
    return 0;
}
inline bool sw16_supported(const Sw16Profile &p, int open, int gap) {
    if (SW16_DECOUPLE && open < gap) return false;
    return p.K > 0 && open >= 0 && gap >= 0 && gap <= 4096 && open + p.max_score <= 127 && open + p.min_score >= -127;
}
inline size_t sw16_letter_stride(int chunks) { return (size_t)chunks * SW16_G * 16; }
// host-side build of the packed profile with `open` folded in
inline bool sw16_build_profile(const uint8_t *mapped_query, int lq, const int *table, int size, int open,
                               Sw16Profile *out, std::vector<int8_t> *host) {
    const int K = sw16_pick_k(lq);
    if (K == 0 || size + 1 > 32) return false;
    out->lq = lq; out->K = K; out->chunks = sw16_chunks(K); out->nletters = size + 1; out->open_baked = open;
    int mx = -1000000, mn = 1000000;
    for (int i = 0; i < size * size; ++i) { mx = table[i] > mx ? table[i] : mx; mn = table[i] < mn ? table[i] : mn; }
    out->max_score = mx; out->min_score = mn;
    if (!sw16_supported(*out, open, 0)) return false;
    const size_t ls = sw16_letter_stride(out->chunks);
#if SW16_PROF32
    // rows past the query and the pad letter score S+o = -128, as in the int8 layout
    host->assign((size_t)(size + 1) * ls, (int8_t)0);
    unsigned *w = (unsigned *)host->data();
    for (size_t x = 0; x < host->size() / 4; ++x) w[x] = 0xff80u;
    for (int a = 0; a < size; ++a)
        for (int lane = 0; lane < SW16_G; ++lane)
            for (int k = 0; k < K; ++k) {
                const int i = lane * K + k;
                if (i < lq)
                    w[((size_t)a * ls + ((size_t)(k >> 2) * SW16_G + lane) * 16) / 4 + (k & 3)] =
                        (unsigned)(table[(size_t)mapped_query[i] * size + a] + open) & 0xffffu;
            }
#else
    host->assign((size_t)(size + 1) * ls, (int8_t)-128);
    for (int a = 0; a < size; ++a)
        for (int lane = 0; lane < SW16_G; ++lane)
            for (int k = 0; k < K; ++k) {
                const int i = lane * K + k;
                if (i < lq)
                    (*host)[(size_t)a * ls + ((size_t)(k >> 4) * SW16_G + lane) * 16 + (k & 15)] =
                        (int8_t)(table[(size_t)mapped_query[i] * size + a] + open);
            }
#endif
    return true;
}

struct Sw16Params {
    const int8_t *prof;
    int nletters;
    int lq;
    int open, gap;
    int max_score;
    const unsigned *words;        // packed database (sorted by length, descending)
    const long long *word_off;    // n+1
    const int *len;               // n
    int bits;                     // 5, 3 or 2
    long long n;                  // subjects; work item w = subjects 2w and 2w+1
    const int *out_map;           // sorted position -> caller's subject id
    int *score, *end_query, *end_ref;
    int *retry;                   // sorted positions that overflowed 16 bit
    int *retry_count;
    int sid_base;                 // added to a subject index before it is pushed to `retry`
    int *counter;                 // dynamic work queue over pairs of items
    // STRIP kernels (queries longer than one strip of 16*K rows are swept strip by strip, one launch each):
    const long long *res_off;     // first residue of each sorted subject (n+1): an item's boundary line starts at
                                  // res_off of its first subject and has one uint2 (T, Fh of both subjects) per column
    const uint2 *bnd_in;          // bottom row of the strip above (NULL for the first strip)
    uint2 *bnd_out;               // this strip's bottom row (NULL for the last strip)
    int row0;                     // first query row of this strip
    int merge;                    // 1: combine with the result already stored for the subject (strips after the first)
    unsigned mul_one;             // the constant 1, kept opaque so that T = X*1 - o can be an IMAD
    unsigned mul_64k;             // the constant 65536, opaque for the same reason: (b << 16) + a as an IMAD
};

// per warp: 2 rings of 64 words, 2 published group bests (padded to 16 B), 2 halves x 32 lanes x
// sw16_park_words(K) words of parked H columns, and (strip kernels) 2 rings of 64 boundary columns
inline size_t sw16_warp_smem(int K, bool strip = false) { return 2 * 64 * 4 + 16 + (size_t)2 * 32 * sw16_park_words(K) * 4 + (strip ? 2 * 64 * 8 : 0); }
inline size_t sw16_smem_bytes(int nletters, int K, int warps, bool strip = false) {
    return (size_t)nletters * sw16_letter_stride(sw16_chunks(K)) + (size_t)warps * sw16_warp_smem(K, strip);
}

PSB_DEV unsigned sw16_fetch_code(const unsigned *words, long long w0, int len, int c, int bits, int pad_code) {
    if (c >= len) return (unsigned)pad_code;
    if (bits == 2) return (words[w0 + (c >> 4)] >> (2 * (c & 15))) & 3u;
    if (bits == 3) {
        const int w = (int)(((unsigned long long)(unsigned)c * 0xCCCCCCCDull) >> 35);  // c / 10
        return (words[w0 + w] >> (3 * (c - 10 * w))) & 7u;
    }
    const int w = (int)(((unsigned long long)(unsigned)c * 0xAAAAAAABull) >> 34);  // c / 6
    return (words[w0 + w] >> (5 * (c - 6 * w))) & 31u;
}

// tuning knobs (overridable at build time for experiments)
#ifndef SW16_UNROLL
#define SW16_UNROLL 2
#endif
#ifndef SW16_PINGPONG
#define SW16_PINGPONG 1   // two register copies of the column (measured +3 %: no moves at the back-edge)
#endif
#define PSB_PRAGMA_(x) _Pragma(#x)
#define PSB_UNROLL(n) PSB_PRAGMA_(unroll n)
#ifndef SW16_WARPS_PER_BLOCK
#define SW16_WARPS_PER_BLOCK 8
#endif
#if defined(SW16_MIN_BLOCKS) && !defined(PSB_EMULATE)
#define SW16_BOUNDS __launch_bounds__(SW16_WARPS_PER_BLOCK * 32, SW16_MIN_BLOCKS)
#else
#define SW16_BOUNDS
#endif

template <int K, bool STRIP = false>
PSB_KERNEL void SW16_BOUNDS sw16_scan_kernel(Sw16Params p) {
    constexpr int G = SW16_G;
    constexpr int CH = (K + SW16_ROWS_PER_LOAD - 1) / SW16_ROWS_PER_LOAD;   // = sw16_chunks(K): 16-byte profile loads per lane and letter
    constexpr unsigned LSTRIDE = CH * G * 16;         // bytes per letter
    PSB_SHARED_DECL(smem_raw);
    const int lane = lane_id();
    const int lg = lane & (G - 1);                    // lane inside the group
    const int grp = lane >> 4;                        // which of the warp's two groups
    // ---- stage the profile (shared by all warps of the block) ----------------------------------
    {
        const uint4 *src = (const uint4 *)p.prof;
        uint4 *dst = (uint4 *)smem_raw;
        const int n16 = p.nletters * (int)(LSTRIDE / 16);
        for (int x = thread_in_block(); x < n16; x += threads_per_block()) dst[x] = src[x];
    }
    sync_block();
    const unsigned char *lane_base = smem_raw + lg * 16;
    constexpr int PARKW = SW16_PROF32 ? ((K + 3) / 4) * 4 : ((K + 15) / 16) * 16;   // = sw16_park_words(K)
    unsigned char *wsm = smem_raw + (size_t)p.nletters * LSTRIDE + (size_t)warp_in_block() * (2 * 64 * 4 + 16 + 2 * 32 * PARKW * 4 + (STRIP ? 2 * 64 * 8 : 0));
    uint2 *bring = (uint2 *)(wsm + 2 * 64 * 4 + 16 + 2 * 32 * PARKW * 4) + grp * 64;   // STRIP: boundary columns of the strip above
    unsigned *ring = (unsigned *)wsm + grp * 64;
    volatile unsigned *gpub = (volatile unsigned *)(wsm + 2 * 64 * 4) + grp;   // group best - 1, per half
    uint4 *park = (uint4 *)(wsm + 2 * 64 * 4 + 16);   // [half][chunk4][lane] 16-byte slots
    const int pad_code = p.nletters - 1;
    const unsigned O2 = (unsigned)p.open * 0x10001u;
    const unsigned NEGE = ((unsigned)(-p.gap) & 0xffffu) * 0x10001u;
    const unsigned NEGO = SW16_DECOUPLE ? ((unsigned)(-p.open) & 0xffffu) * 0x10001u   // (-o, -o) as two halves
                                        : 0u - O2;                                       // 32-bit -(o, o): X - o never borrows
    (void)O2;
    const unsigned one = p.mul_one;
    (void)one;
    const unsigned m64k = p.mul_64k;
    (void)m64k;
    const long long nitems = (p.n + 1) >> 1;
    const long long nslots = (nitems + 1) >> 1;       // a warp takes two items at a time
    const int limit = 32767 - p.open - p.max_score;   // scores from here on may have wrapped

    for (;;) {
        int slot = 0;
        if (lane == 0) slot = atomic_add(p.counter, 1);
        slot = shfl(slot, 0);
        if (slot >= nslots) break;
        const long long item = 2ll * slot + grp;
        const long long sa = 2 * item, sb = sa + 1;
        const int lenA = sa < p.n ? p.len[sa] : 0;
        const int lenB = sb < p.n ? p.len[sb] : 0;
        const long long wA = sa < p.n ? p.word_off[sa] : 0, wB = sb < p.n ? p.word_off[sb] : 0;
        const int Lmax = lenA > lenB ? lenA : lenB;    // this group's columns
        const int Lother = shfl_xor(Lmax, 16);
        const int nsteps = (Lmax > Lother ? Lmax : Lother) + G - 1;  // warp-uniform
        const long long bbase = STRIP ? p.res_off[sa < p.n ? sa : 0] : 0;   // this item's boundary line

        // boundary values of a local alignment: H = 0, so T = H - o (decoupled form) or T = H (shifted form)
        const unsigned TB = SW16_DECOUPLE ? NEGO : 0u;
        unsigned T[K], E[K];
#pragma unroll
        for (int k = 0; k < K; ++k) { T[k] = TB; E[k] = TB; }
#if SW16_PINGPONG
        unsigned T2[K];
#pragma unroll
        for (int k = 0; k < K; ++k) T2[k] = TB;
#endif
        unsigned Tdiag_in = TB, Tout = TB, Fout = 0;
        unsigned thr = 0;                     // per half: a column maximum must exceed this to matter
        unsigned best = 0, bestj = 0;         // per half: own best score and its column
        sync_warp();
        if (lg == 0) *gpub = 0;

        for (int s0 = 0; s0 < nsteps; s0 += 32) {
            // every 32 steps: stage the next 32 columns of both subjects as profile byte offsets
            sync_warp();
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int c = s0 + lg + u * G;
                const unsigned ca = sw16_fetch_code(p.words, wA, lenA, c, p.bits, pad_code);
                const unsigned cb = sw16_fetch_code(p.words, wB, lenB, c, p.bits, pad_code);
                ring[c & 63] = (ca * LSTRIDE) | ((cb * LSTRIDE) << 16);
                if (STRIP) {
                    uint2 bv; bv.x = TB; bv.y = 0u;   // first strip: the table's top boundary (H = 0, F opened from it)
                    if (p.bnd_in && c < Lmax) bv = p.bnd_in[bbase + c];
                    bring[c & 63] = bv;
                }
            }
            sync_warp();
            const int send = (s0 + 32 < nsteps) ? s0 + 32 : nsteps;
            // one step of the systolic sweep: reads the previous column's T from Tin, writes the new
            // column into Tnew (the same array, or the other one of a ping-pong pair)
            auto step = [&](const int s, unsigned (&Tin)[K], unsigned (&Tnew)[K]) {
                const int j = s - lg;
                unsigned Tup = shfl_up(Tout, 1);
                unsigned Fup = shfl_up(Fout, 1);
                if (lg == 0) {
                    if (STRIP) { const uint2 bv = bring[j & 63]; Tup = bv.x; Fup = bv.y; }
                    else { Tup = TB; Fup = 0; }
                }
                if (j >= 0 && j < Lmax) {
                    const unsigned w = ring[j & 63];
                    const unsigned char *pa = lane_base + (w & 0xffffu);
                    const unsigned char *pb = lane_base + (w >> 16);
                    unsigned was[CH * 4], wbs[CH * 4];
#pragma unroll
                    for (int c = 0; c < CH; ++c) {
                        const uint4 a = *(const uint4 *)(pa + c * (G * 16));
                        const uint4 b = *(const uint4 *)(pb + c * (G * 16));
                        was[4 * c] = a.x; was[4 * c + 1] = a.y; was[4 * c + 2] = a.z; was[4 * c + 3] = a.w;
                        wbs[4 * c] = b.x; wbs[4 * c + 1] = b.y; wbs[4 * c + 2] = b.z; wbs[4 * c + 3] = b.w;
                    }
                    unsigned Td = Tdiag_in, Tu = Tup, Fu = Fup;
                    unsigned cmax = 0, tprev = 0;
#pragma unroll
                    for (int k = 0; k < K; ++k) {
#if SW16_PROF32
                        const unsigned So = wbs[k] * m64k + was[k];
#else
                        constexpr unsigned SEL0 = 0xC480u;
                        const unsigned sel = SEL0 + (unsigned)(k & 3) * 0x1111u;
                        const unsigned So = prmt(was[k >> 2], wbs[k >> 2], sel);
#endif
                        const unsigned Tl = Tin[k];
                        const unsigned En = viaddmax2(E[k], NEGE, Tl);
#if SW16_DECOUPLE
                        const unsigned h = viaddmax2(Td, So, En);
                        const unsigned Hn = viaddmax2_relu(Fu, NEGO, h);
                        const unsigned Fn = viaddmax2(Fu, NEGE, h);
                        const unsigned Tn = vadd2(Hn, NEGO);
                        if (k & 1) cmax = vimax3_2(cmax, tprev, Hn);
                        else tprev = Hn;
#else
                        const unsigned Fn = viaddmax2(Fu, NEGE, Tu);
                        const unsigned h = viaddmax2(Td, So, En);
                        const unsigned X = vimax3_2(h, Fn, O2);
                        const unsigned Tn = X * one + NEGO;
                        if (k & 1) cmax = vimax3_2(cmax, tprev, Tn);
                        else tprev = Tn;
#endif
                        Td = Tl; Tnew[k] = Tn; E[k] = En; Tu = Tn; Fu = Fn;
                    }
                    if (K & 1) cmax = vimax2(cmax, tprev);
                    Tdiag_in = Tup; Tout = Tu; Fout = Fu;
                    if (STRIP) {
                        if (lg == G - 1 && p.bnd_out) { uint2 bv; bv.x = Tu; bv.y = Fu; p.bnd_out[bbase + j] = bv; }
                    }
                    thr = vimax2(thr, *gpub);
                    const unsigned m = vimax2(thr, cmax);
                    if (m != thr) {
                        // cold: a half beat the threshold.  Record score and column, park the column
                        // of H values (the row is resolved after the last step) and publish the score.
                        const unsigned diff = m ^ thr;
                        const unsigned mask = ((diff & 0xffffu) ? 0xffffu : 0u) | ((diff >> 16) ? 0xffff0000u : 0u);
                        best = (best & ~mask) | (cmax & mask);
                        bestj = (bestj & ~mask) | (((unsigned)j * 0x10001u) & mask);
                        thr = m;
#pragma unroll
                        for (int c4 = 0; c4 < (K + 3) / 4; ++c4) {
                            uint4 v;
                            v.x = Tnew[4 * c4];
                            v.y = 4 * c4 + 1 < K ? Tnew[4 * c4 + 1] : 0u;
                            v.z = 4 * c4 + 2 < K ? Tnew[4 * c4 + 2] : 0u;
                            v.w = 4 * c4 + 3 < K ? Tnew[4 * c4 + 3] : 0u;
                            if (mask & 0xffffu) park[(0 * (PARKW / 4) + c4) * 32 + lane] = v;
                            if (mask >> 16) park[(1 * (PARKW / 4) + c4) * 32 + lane] = v;
                        }
                        // publish (best - 1) so that the other lanes ignore anything smaller; a lost
                        // race only leaves the published value lower, which is always safe
                        const unsigned pub = vimax2(*gpub, vimax2(best, 0x00010001u) - 0x00010001u);
                        *gpub = pub;
                    }
                }
            };
#if SW16_PINGPONG
            // two register copies of the column: even steps read T and write T2, odd steps the
            // reverse, so no value has to be moved at the loop's back-edge.  The chunk always starts
            // on an even step; a trailing odd step past the end has no active lane.
            for (int s = s0; s < send; s += 2) {
                step(s, T, T2);
                step(s + 1, T2, T);
            }
#else
            PSB_UNROLL(SW16_UNROLL)
            for (int s = s0; s < send; ++s) step(s, T, T);
#endif
        }
        // ---- merge the group's lanes: (score desc, end_ref asc, end_query asc), each half separately --
        sync_warp();
        unsigned long long comps[2];
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const unsigned sc = half ? (best >> 16) : (best & 0xffffu);
            const unsigned col = half ? (bestj >> 16) : (bestj & 0xffffu);
            // first row of the parked column that holds the lane's best
            unsigned rowk = 0;
            if (sc != 0) {
                const unsigned *pk = (const unsigned *)park;
                // the parked words hold T: H itself (shifted form) or H - o (decoupled form)
                const unsigned want = SW16_DECOUPLE ? ((sc - (unsigned)p.open) & 0xffffu) : sc;
                for (int k = K - 1; k >= 0; --k) {
                    const unsigned wv = pk[(((half * (PARKW / 4) + (k >> 2)) * 32 + lane) << 2) + (k & 3)];
                    if ((half ? (wv >> 16) : (wv & 0xffffu)) == want) rowk = (unsigned)k;
                }
            }
            const unsigned row = (unsigned)(lg * K) + rowk;
            // 16 bits score | 16 bits inverted column | 10 bits inverted row
            unsigned long long comp = ((unsigned long long)sc << 26) | ((unsigned long long)(0xffffu - col) << 10) |
                                      (unsigned long long)(1023u - row);
#pragma unroll
            for (int m = G / 2; m >= 1; m >>= 1) {
                const unsigned long long other = (unsigned long long)shfl_xor((long long)comp, m);
                comp = other > comp ? other : comp;
            }
            comps[half] = comp;
        }
        if (lg == 0) {
            // a half that leaves the 16-bit range re-runs both subjects of the item at 32 bit
            const bool overflow = (int)(comps[0] >> 26) >= limit || (int)(comps[1] >> 26) >= limit;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const long long sid = half ? sb : sa;
                if (sid >= p.n) continue;
                const unsigned long long comp = comps[half];
                const int sc = (int)(comp >> 26);
                const int oid = p.out_map ? p.out_map[sid] : (int)sid;
                // STRIP: a strip that lists an item stores the score -1 for both its subjects; the strips below leave
                // such an item alone, so it is listed once and the re-run alone writes its results
                const int osc = STRIP && p.merge ? p.score[oid] : 0;
                if (osc < 0) continue;
                if (overflow) {
                    const int slot_r = atomic_add(p.retry_count, 1);
                    p.retry[slot_r] = (int)sid + p.sid_base;
                    if (STRIP) p.score[oid] = -1;
                } else {
                    int er = sc == 0 ? 0 : (int)(0xffffu - (unsigned)((comp >> 10) & 0xffffu));
                    int eq = sc == 0 ? 0 : 1023 - (int)(comp & 1023u) + (STRIP ? p.row0 : 0);
                    int best_sc = sc;
                    if (STRIP && p.merge) {
                        // the strips above have stored their best: (score, smaller end_ref, smaller end_query) decides
                        const int oer = p.end_ref[oid], oeq = p.end_query[oid];
                        if (osc > sc || (osc == sc && (sc == 0 || oer < er || (oer == er && oeq < eq)))) { best_sc = osc; er = oer; eq = oeq; }
                    }
                    p.score[oid] = best_sc; p.end_query[oid] = eq; p.end_ref[oid] = er;
                }
            }
        }
    }
}

}  // namespace psb
