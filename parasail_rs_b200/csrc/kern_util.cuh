// kern_util.cuh -- residue mapping, database bit-packing and the device-side trace walk.
#pragma once
#include "psb_defs.h"
#include "psb_simt.h"

namespace psb {

// raw residue bytes -> matrix column indices through the matrix's 256-entry mapper
// (parasail applies matrix->mapper to every residue before the fill; SURVEY A.1)
struct MapParams {
    uint8_t *data;
    long long n;
    unsigned lut[64];  // 256 bytes
};
PSB_KERNEL void map_residues_kernel(MapParams p) {
    const long long stride = (long long)grid_blocks() * threads_per_block();
    for (long long i = (long long)block_id() * threads_per_block() + thread_in_block(); i < p.n; i += stride) {
        const unsigned b = p.data[i];
        p.data[i] = (uint8_t)((p.lut[b >> 2] >> (8 * (b & 3))) & 0xff);
    }
}

// ---- database packing -----------------------------------------------------------------------
// A subject is stored as 32-bit words of RPW residues of BITS bits each (5 bit: 6 per word, 3 bit: 10 per
// word, 2 bit: 16 per word), first residue in the low bits, each subject starting on a fresh word.
PSB_DEV constexpr int residues_per_word(int bits) { return bits == 2 ? 16 : (bits == 3 ? 10 : 6); }
// residue c of a packed subject whose first word is words[w0]
PSB_DEV unsigned packed_residue(const unsigned *words, long long w0, int c, int bits) {
    if (bits == 2) return (words[w0 + (c >> 4)] >> (2 * (c & 15))) & 3u;
    if (bits == 3) {
        const int w = (int)(((unsigned long long)(unsigned)c * 0xCCCCCCCDull) >> 35);   // c / 10
        return (words[w0 + w] >> (3 * (c - 10 * w))) & 7u;
    }
    const int w = (int)(((unsigned long long)(unsigned)c * 0xAAAAAAABull) >> 34);       // c / 6
    return (words[w0 + w] >> (5 * (c - 6 * w))) & 31u;
}

struct PackParams {
    const uint8_t *raw;          // original residues (caller order), unmapped
    const long long *raw_off;    // n+1, as given by the caller
    long long raw_base;          // raw_off[0]: `raw` starts at that residue
    const int *perm;             // sorted position -> original subject id
    const long long *word_off;   // n+1, in words, sorted order
    unsigned *words;
    long long n;
    int bits;
    unsigned lut[64];
};
// one warp per subject, lanes stride over its words.  256 bytes of dynamic shared memory hold the byte -> code
// table (indexing the kernel parameter itself with a per-lane byte would serialise on the constant cache:
// 0.68 ms for 253 MB before, profiles/README.md r2r).
PSB_KERNEL void pack_db_kernel(PackParams p) {
    PSB_SHARED_DECL(smem);
    uint8_t *slut = smem;
    for (int b = thread_in_block(); b < 256; b += threads_per_block()) slut[b] = (uint8_t)((p.lut[b >> 2] >> (8 * (b & 3))) & 0xff);
    sync_block();
    const int rpw = residues_per_word(p.bits);
    const long long warp = ((long long)block_id() * threads_per_block() + thread_in_block()) >> 5;
    const long long nwarps = ((long long)grid_blocks() * threads_per_block()) >> 5;
    const int lane = lane_id();
    for (long long s = warp; s < p.n; s += nwarps) {
        const long long o0 = p.raw_off[p.perm[s]];
        const uint8_t *src = p.raw + (o0 - p.raw_base);
        const int len = (int)(p.raw_off[p.perm[s] + 1] - o0);
        const long long w0 = p.word_off[s];
        const int nw = (int)(p.word_off[s + 1] - w0);
        for (int w = lane; w < nw; w += 32) {
            unsigned word = 0;
            const int i0 = w * rpw;
            if (i0 + rpw <= len) {
#pragma unroll 2
                for (int t = 0; t < rpw; ++t) word |= (unsigned)slut[src[i0 + t]] << (p.bits * t);
            } else {
                for (int t = 0; i0 + t < len; ++t) word |= (unsigned)slut[src[i0 + t]] << (p.bits * t);
            }
            p.words[w0 + w] = word;
        }
    }
}

// sorted position -> caller id (a database's permutation) inverted: inv[perm[s]] = s
PSB_KERNEL void invert_perm_kernel(const int *perm, long long n, int *inv) {
    const long long stride = (long long)grid_blocks() * threads_per_block();
    for (long long s = (long long)block_id() * threads_per_block() + thread_in_block(); s < n; s += stride) inv[perm[s]] = (int)s;
}

// packed subjects -> matrix codes, one warp per subject
struct UnpackParams {
    const unsigned *words;
    const long long *word_off;   // sorted order
    const int *ids;              // which subjects to unpack (NULL: all sorted subjects, 0..n-1)
    const int *inv_perm;         // non-NULL: `ids` are caller-order ids, resolved to sorted positions through it
    const long long *out_off;    // n+1 byte offsets of the outputs
    uint8_t *out;
    long long n;
    int bits;
};
PSB_KERNEL void unpack_db_kernel(UnpackParams p) {
    const int rpw = residues_per_word(p.bits);
    const unsigned mask = (1u << p.bits) - 1u;
    const long long warp = ((long long)block_id() * threads_per_block() + thread_in_block()) >> 5;
    const long long nwarps = ((long long)grid_blocks() * threads_per_block()) >> 5;
    const int lane = lane_id();
    for (long long s = warp; s < p.n; s += nwarps) {
        const long long sid = p.ids ? (p.inv_perm ? p.inv_perm[p.ids[s]] : p.ids[s]) : s;
        const long long w0 = p.word_off[sid];
        const long long o0 = p.out_off[s];
        const int len = (int)(p.out_off[s + 1] - o0);
        for (int idx = lane; idx < len; idx += 32) {
            const unsigned word = p.words[w0 + idx / rpw];
            p.out[o0 + idx] = (uint8_t)((word >> (p.bits * (idx % rpw))) & mask);
        }
    }
}

// ---- device-side trace walk (SURVEY A.7) ------------------------------------------------------
// One thread per pair walks the [strip][step][lane][K] trace bytes written by gotoh32_kernel
// from the end cell and run-length encodes the path in reverse into a per-pair scratch region;
// compact_cigar_kernel then reverses each run list into the CSR the caller receives.
struct WalkParams {
    const uint8_t *q;
    const long long *q_off;
    const uint8_t *r;
    const long long *r_off;
    int shared_query;
    const int *ids;              // pair ids of this launch
    int n;
    int K;
    const uint8_t *trace;
    const long long *trace_off;  // indexed by pair id
    const int *end_query, *end_ref;   // indexed by pair id
    unsigned *rev_ops;           // scratch
    const long long *rev_off;    // indexed by pair id: start of the pair's scratch region
    int *nops, *beg_query, *beg_ref;  // indexed by pair id
};
PSB_KERNEL void walk_trace_kernel(WalkParams p) {
    const long long t = (long long)block_id() * threads_per_block() + thread_in_block();
    if (t >= p.n) return;
    const int pid = p.ids ? p.ids[t] : (int)t;
    const long long qo = p.shared_query ? p.q_off[0] : p.q_off[pid];
    const uint8_t *q = p.q + qo;
    const long long ro = p.r_off[pid];
    const uint8_t *r = p.r + ro;
    const int Lr = (int)(p.r_off[pid + 1] - ro);
    const int K = p.K, rows = 32 * K, nsteps = Lr + 31;
    const uint8_t *tr = p.trace + p.trace_off[pid];
    unsigned *out = p.rev_ops + p.rev_off[pid];
    int i = p.end_query[pid], j = p.end_ref[pid];
    int where = TR_DIAG, cur = -1, n = 0;
    unsigned len = 0;
    while (i >= 0 || j >= 0) {
        int op;
        if (i < 0) { op = 2; --j; }
        else if (j < 0) { op = 1; --i; }
        else {
            const int strip = i / rows, rem = i - strip * rows, lane = rem / K, k = rem - lane * K;
            const int tf = tr[(((size_t)strip * nsteps + (j + lane)) * 32 + lane) * K + k];
            if (where == TR_DIAG) {
                if (tf & TR_DIAG) { op = (q[i] == r[j]) ? 7 : 8; --i; --j; }
                else if (tf & TR_INS) { where = TR_INS; continue; }
                else if (tf & TR_DEL) { where = TR_DEL; continue; }
                else break;
            } else if (where == TR_INS) { op = 2; where = (tf & TR_DIAG_E) ? TR_DIAG : TR_INS; --j; }
            else { op = 1; where = (tf & TR_DIAG_F) ? TR_DIAG : TR_DEL; --i; }
        }
        if (op == cur) ++len;
        else {
            if (cur >= 0) out[n++] = (len << 4) | (unsigned)cur;
            cur = op; len = 1;
        }
    }
    if (cur >= 0) out[n++] = (len << 4) | (unsigned)cur;
    p.nops[pid] = n;
    p.beg_query[pid] = i + 1;
    p.beg_ref[pid] = j + 1;
}

// The same walk over the band-layout trace bytes of band32_kernel (row i, offset t = j - i - lo at byte i * W + t),
// from the corner (Lq - 1, Lr - 1); `K` of the parameters is unused, `k` is the band's half-width.  Same run lists,
// same scratch: compact_cigar_kernel and the CIGAR CSR build take them as they are.
PSB_KERNEL void walk_band_kernel(WalkParams p, int k) {
    const long long t = (long long)block_id() * threads_per_block() + thread_in_block();
    if (t >= p.n) return;
    const int pid = p.ids ? p.ids[t] : (int)t;
    const long long qo = p.shared_query ? p.q_off[0] : p.q_off[pid];
    const uint8_t *q = p.q + qo;
    const int Lq = (int)((p.shared_query ? p.q_off[1] : p.q_off[pid + 1]) - qo);
    const long long ro = p.r_off[pid];
    const uint8_t *r = p.r + ro;
    const int Lr = (int)(p.r_off[pid + 1] - ro);
    const int d = Lr - Lq, lo = -k + (d < 0 ? d : 0), W = 2 * k + (d < 0 ? -d : d) + 1;
    const uint8_t *tr = p.trace + p.trace_off[pid];
    unsigned *out = p.rev_ops + p.rev_off[pid];
    int i = Lq - 1, j = Lr - 1;
    int where = TR_DIAG, cur = -1, n = 0;
    unsigned len = 0;
    while (i >= 0 || j >= 0) {
        int op;
        if (i < 0) { op = 2; --j; }
        else if (j < 0) { op = 1; --i; }
        else {
            const int tf = tr[(size_t)i * W + (j - i - lo)];
            if (where == TR_DIAG) {
                if (tf & TR_DIAG) { op = (q[i] == r[j]) ? 7 : 8; --i; --j; }
                else if (tf & TR_INS) { where = TR_INS; continue; }
                else if (tf & TR_DEL) { where = TR_DEL; continue; }
                else break;
            } else if (where == TR_INS) { op = 2; where = (tf & TR_DIAG_E) ? TR_DIAG : TR_INS; --j; }
            else { op = 1; where = (tf & TR_DIAG_F) ? TR_DIAG : TR_DEL; --i; }
        }
        if (op == cur) ++len;
        else {
            if (cur >= 0) out[n++] = (len << 4) | (unsigned)cur;
            cur = op; len = 1;
        }
    }
    if (cur >= 0) out[n++] = (len << 4) | (unsigned)cur;
    p.nops[pid] = n;
    p.beg_query[pid] = i + 1;
    p.beg_ref[pid] = j + 1;
}

struct CompactParams {
    const unsigned *rev_ops;
    const long long *rev_off;   // by pair id
    const long long *csr_off;   // by pair id (n+1): exclusive scan of nops
    unsigned *csr_ops;
    int n;
};
PSB_KERNEL void compact_cigar_kernel(CompactParams p) {
    const long long warp = ((long long)block_id() * threads_per_block() + thread_in_block()) >> 5;
    const long long nwarps = ((long long)grid_blocks() * threads_per_block()) >> 5;
    const int lane = lane_id();
    for (long long pid = warp; pid < p.n; pid += nwarps) {
        const long long a = p.csr_off[pid];
        const int cnt = (int)(p.csr_off[pid + 1] - a);
        const unsigned *src = p.rev_ops + p.rev_off[pid];
        for (int k = lane; k < cnt; k += 32) p.csr_ops[a + k] = src[cnt - 1 - k];
    }
}

}  // namespace psb
