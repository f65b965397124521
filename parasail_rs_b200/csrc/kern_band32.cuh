// kern_band32.cuh -- banded global alignment (nw) that fills only the band: one warp per pair, 32-bit scores,
// optional statistics, optional trace bytes in band layout.  Work per pair is O(W * (Lq + Lr)), not O(Lq * Lr).
//
// Band of a pair (oracle rule band_rule = 0): with d = Lr - Lq, lo = -k + min(d, 0) and hi = k + max(d, 0), cell
// (i, j) is in the band iff lo <= j - i <= hi; the band has W = hi - lo + 1 offsets t = j - i - lo.
//
// Layout of the computation:
//   * the warp sweeps anti-diagonals s = i + j.  Offset t holds a cell on every second anti-diagonal (those with
//     s - t - lo even), so a step is two half-steps, one per parity class of offsets;
//   * lane l owns the R consecutive offsets l*R .. l*R + R - 1 (R even, so the first and last offset of a lane are
//     of different parity).  At anti-diagonal s a cell reads its left neighbour (t - 1: H, E) and its upper
//     neighbour (t + 1: H, F) as they were on s - 1, and its own H of s - 2 (the diagonal): cells update in place,
//     and only a lane's edge offsets cross lanes -- one shuffle up (H, E of the last offset) before the even
//     half-step, one shuffle down (H, F of the first offset) before the odd one;
//   * no prefix scan along a row: every tie rule stays cell-local, exactly as in oracle/gotoh_oracle.c (H source
//     diag >= F >= E, a gap opens only when strictly better than extending, the E / F "opened" trace bits);
//   * an offset whose cell lies outside the table holds that cell's boundary value (row -1 / column -1: the nw gap
//     penalties, corner 0) or -inf, so the table's edges need no special case in the cell update; offsets t >= W
//     (padding of the last lanes) are -inf, statistics 0: outside the band;
//   * SMEM: the offsets of a lane live in shared memory, [r][lane] (conflict-free), instead of registers, for bands
//     wider than 32 * 16 up to kBandMaxW.  A lane only ever touches its own column (the edges still cross lanes by
//     shuffle), so the variants differ in nothing but where the offsets are kept.
// Boundary values, statistics rules and trace-flag bits are those of gotoh32_kernel (nw).  Trace bytes: row i,
// offset t at byte i * W + t of the pair's block (psb::band_cell_index); positions outside the table hold 0.
#pragma once
#include "kern_gotoh32.cuh"

namespace psb {

static constexpr int kBandRegMaxW = 32 * 16;   // register variants: R = 2, 4, 8, 16 offsets per lane
static constexpr int kBandMaxW = 4096;         // shared-memory variant beyond that

struct BandGeom {
    int lo, hi, W;
};
PSB_HD BandGeom band_geom(int lq, int lr, int k) {
    const int d = lr - lq;
    BandGeom g;
    g.lo = -k + (d < 0 ? d : 0);
    g.hi = k + (d > 0 ? d : 0);
    g.W = g.hi - g.lo + 1;
    return g;
}

struct Band32Params {
    const uint8_t *q;           // residues already mapped to matrix column indices
    const long long *q_off;     // n+1 offsets (shared_query: only [0],[1] are read)
    const uint8_t *r;
    const long long *r_off;     // n+1 offsets
    const int *order;           // pair ids handled by this launch (NULL: 0..n-1)
    int n;
    int shared_query;
    const int *matrix;          // square: size*size; pssm: qlen*size (global memory)
    int size;
    int is_pssm;
    int open, gap;
    int k;                      // band half-width
    int *score, *end_query, *end_ref;   // indexed by pair id
    int *matches, *similar, *length;    // STATS only
    uint8_t *trace;             // TRACE only: per pair Lq x W bytes, band layout
    const long long *trace_off; // byte offset of each pair's trace block (indexed by pair id)
    int *counter;               // dynamic work queue
    int rr;                     // SMEM only: offsets per lane (even, 32 * rr >= W of every pair of the launch)
};

// dynamic shared memory: the square matrix, then (SMEM) each warp's band state
PSB_HD size_t band32_warp_smem(int rr, bool stats) { return (size_t)32 * rr * (3 * sizeof(int) + (stats ? 3 * sizeof(unsigned long long) : 0)); }
inline size_t band32_smem_bytes(int size, int warps, bool smem, int rr, bool stats) {
    const size_t m = ((size_t)size * size * sizeof(int) + 15) & ~(size_t)15;
    return m + (smem ? (size_t)warps * band32_warp_smem(rr, stats) : 0);
}

// the R offsets of a lane: registers, or a lane's column of a [r][32] shared-memory array
template <typename T, int R, bool SMEM> struct BandArr {
    T v[R];
    PSB_DEV void place(T *) {}
    PSB_DEV T &operator[](int r) { return v[r]; }
};
template <typename T, int R> struct BandArr<T, R, true> {
    T *p;
    PSB_DEV void place(T *col) { p = col; }   // the lane's column: offset r at col[32 * r]
    PSB_DEV T &operator[](int r) { return p[r * 32]; }
};

template <int R, bool SMEM, bool STATS, bool TRACE>
PSB_KERNEL void band32_kernel(Band32Params p) {
    typedef unsigned long long SWord;
    typedef StatPack<SWord> SP;
    PSB_SHARED_DECL(smem_raw);
    const int lane = lane_id();
    const int size = p.size, o = p.open, e = p.gap;
    int *smat = (int *)smem_raw;
    const size_t mat_bytes = p.is_pssm ? 0 : (((size_t)size * size * sizeof(int) + 15) & ~(size_t)15);
    if (!p.is_pssm)
        for (int x = thread_in_block(); x < size * size; x += threads_per_block()) smat[x] = p.matrix[x];
    sync_block();

    const int RR = SMEM ? p.rr : R;
    BandArr<int, R, SMEM> H, E, F;
    BandArr<SWord, R, SMEM> Hs, Es, Fs;
    if (SMEM) {
        unsigned char *base = smem_raw + mat_bytes + (size_t)warp_in_block() * band32_warp_smem(RR, STATS);
        int *ib = (int *)base + lane;
        H.place(ib); E.place(ib + 32 * RR); F.place(ib + 64 * RR);
        SWord *sb = (SWord *)(base + (size_t)32 * RR * 3 * sizeof(int)) + lane;
        Hs.place(sb); Es.place(sb + 32 * RR); Fs.place(sb + 64 * RR);
    }

    for (;;) {
        int slot = 0;
        if (lane == 0) slot = atomic_add(p.counter, 1);
        slot = shfl(slot, 0);
        if (slot >= p.n) break;
        const int pid = p.order ? p.order[slot] : slot;
        const long long qo = p.shared_query ? p.q_off[0] : p.q_off[pid];
        const int Lq = (int)((p.shared_query ? p.q_off[1] : p.q_off[pid + 1]) - qo);
        const long long ro = p.r_off[pid];
        const int Lr = (int)(p.r_off[pid + 1] - ro);
        const uint8_t *q = p.q + qo, *r = p.r + ro;
        const BandGeom g = band_geom(Lq, Lr, p.k);
        const int lo = g.lo, W = g.W;
        uint8_t *tr = TRACE ? p.trace + p.trace_off[pid] : nullptr;
        const int t0 = lane * RR;
        // the value an offset holds for a cell outside the table: the boundary row / column (nw) or -inf
        auto outside = [&](int r_, int t, int i, int j) {
            int h = NEG_INF32;
            if (t < W) {
                if (i == -1 && j == -1) h = 0;
                else if (i == -1 && j >= 0) h = -o - j * e;
                else if (j == -1 && i >= 0) h = -o - i * e;
            }
            H[r_] = h; E[r_] = NEG_INF32; F[r_] = NEG_INF32;
            if (STATS) { Hs[r_] = 0; Es[r_] = 0; Fs[r_] = 0; }
        };
        if (TRACE) {
            // the positions of the block outside the table (offset t of row i is column i + lo + t): flag byte 0
            for (int t = lane; t < W; t += 32) {
                for (int i = 0; i < Lq && i + lo + t < 0; ++i) tr[(size_t)i * W + t] = 0;
                for (int i = Lr - lo - t > 0 ? Lr - lo - t : 0; i < Lq; ++i) tr[(size_t)i * W + t] = 0;
            }
        }
        // the first half-step is on anti-diagonal s0 (s0 - lo even: the even offsets are its cells); before it, even
        // offsets hold their cell of s0 - 2 and odd ones their cell of s0 - 1 (every one outside the table)
        const int s0 = (lo & 1) ? -1 : 0;
#pragma unroll
        for (int r_ = 0; r_ < RR; ++r_) {
            const int t = t0 + r_, s = s0 - 2 + (r_ & 1);
            const int i = (s - t - lo) >> 1;
            outside(r_, t, i, s - i);
        }
        const int nsteps = (Lq + Lr - 2 - s0) / 2 + 1;
        for (int step = 0; step < nsteps; ++step) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int s = s0 + 2 * step + h;
                // the neighbour across the lane edge, as it was on s - 1: even half-step, the left neighbour
                // (H, E) of offset t0; odd half-step, the upper neighbour (H, F) of offset t0 + RR - 1
                int Hx, Gx;
                SWord Hsx = 0, Gsx = 0;
                if (h == 0) {
                    Hx = shfl_up(H[RR - 1], 1); Gx = shfl_up(E[RR - 1], 1);
                    if (STATS) { Hsx = shfl_up(Hs[RR - 1], 1); Gsx = shfl_up(Es[RR - 1], 1); }
                    if (lane == 0) { Hx = NEG_INF32; Gx = NEG_INF32; Hsx = 0; Gsx = 0; }
                } else {
                    Hx = shfl(H[0], lane + 1); Gx = shfl(F[0], lane + 1);
                    if (STATS) { Hsx = shfl(Hs[0], lane + 1); Gsx = shfl(Fs[0], lane + 1); }
                    if (lane == 31) { Hx = NEG_INF32; Gx = NEG_INF32; Hsx = 0; Gsx = 0; }
                }
#pragma unroll
                for (int r_ = h; r_ < RR; r_ += 2) {
                    const int t = t0 + r_;
                    const int i = (s - t - lo) >> 1, j = s - i;
                    if (t >= W || (unsigned)i >= (unsigned)Lq || (unsigned)j >= (unsigned)Lr) { outside(r_, t, i, j); continue; }
                    const bool edge_l = h == 0 && r_ == 0, edge_u = h == 1 && r_ == RR - 1;
                    const int Hl = edge_l ? Hx : H[r_ - (r_ > 0)], El = edge_l ? Gx : E[r_ - (r_ > 0)];
                    const int Hu = edge_u ? Hx : H[r_ + (r_ < RR - 1)], Fu = edge_u ? Gx : F[r_ + (r_ < RR - 1)];
                    const int qi = (int)q[i], letter = (int)r[j];
                    const int S = p.is_pssm ? ld_ro(p.matrix + (size_t)i * size + letter) : smat[qi * size + letter];
                    const int hd = H[r_] + S;
                    if (!STATS && !TRACE) {
                        const int En = viaddmax(El, -e, Hl - o), Fn = viaddmax(Fu, -e, Hu - o);
                        H[r_] = vimax3(hd, En, Fn); E[r_] = En; F[r_] = Fn;
                    } else {
                        const int Eext = El - e, Eopn = Hl - o, Fext = Fu - e, Fopn = Hu - o;
                        const bool eopen = Eopn > Eext, fopen = Fopn > Fext;
                        const int En = eopen ? Eopn : Eext, Fn = fopen ? Fopn : Fext;
                        const bool isdiag = hd >= En && hd >= Fn;
                        const bool isf = !isdiag && Fn >= En;
                        if (STATS) {
                            const SWord one = (SWord)1 << SP::LS;
                            const SWord Hsl = edge_l ? Hsx : Hs[r_ - (r_ > 0)], Esl = edge_l ? Gsx : Es[r_ - (r_ > 0)];
                            const SWord Hsu = edge_u ? Hsx : Hs[r_ + (r_ < RR - 1)], Fsu = edge_u ? Gsx : Fs[r_ + (r_ < RR - 1)];
                            const SWord es = (eopen ? Hsl : Esl) + one, fs = (fopen ? Hsu : Fsu) + one;
                            SWord inc = one;
                            if (qi == letter) inc += 1;
                            if (S > 0) inc += (SWord)1 << SP::SS;
                            Hs[r_] = isdiag ? Hs[r_] + inc : (isf ? fs : es);
                            Es[r_] = es; Fs[r_] = fs;
                        }
                        if (TRACE) {
                            const unsigned tf = (eopen ? TR_DIAG_E : TR_INS_E) | (fopen ? TR_DIAG_F : TR_DEL_F) |
                                                (isdiag ? TR_DIAG : (isf ? TR_DEL : TR_INS));
                            tr[(size_t)i * W + t] = (uint8_t)tf;
                        }
                        H[r_] = isdiag ? hd : (isf ? Fn : En); E[r_] = En; F[r_] = Fn;
                    }
                    if (i == Lq - 1 && j == Lr - 1) {
                        p.score[pid] = H[r_]; p.end_query[pid] = i; p.end_ref[pid] = j;
                        if (STATS) {
                            p.matches[pid] = (int)(Hs[r_] & SP::MM);
                            p.similar[pid] = (int)((Hs[r_] >> SP::SS) & SP::SM);
                            p.length[pid] = (int)((Hs[r_] >> SP::LS) & SP::LM);
                        }
                    }
                }
            }
        }
    }
}

}  // namespace psb
