// band32_kernels.cpp -- TEST ONLY.  The band kernel (csrc/kern_band32.cuh) and its walk (walk_band_kernel,
// csrc/kern_util.cuh) compiled with -DPSB_EMULATE (every lane an OS thread, see csrc/psb_simt.h), so that they can be
// stepped on a CPU-only box and compared with the oracle.  Driven by tests/emu_band32.py.
#define PSB_EMULATE 1
#include <cstring>

#include "../../parasail_rs_b200/csrc/kern_band32.cuh"
#include "../../parasail_rs_b200/csrc/kern_util.cuh"

using namespace psb;

template <int R, bool SMEM> static void run_band(const Band32Params &p, bool stats, bool trace, int nblocks, size_t smem) {
    if (stats && trace) emu::launch(nblocks, smem, [&]() { band32_kernel<R, SMEM, true, true>(p); });
    else if (stats) emu::launch(nblocks, smem, [&]() { band32_kernel<R, SMEM, true, false>(p); });
    else if (trace) emu::launch(nblocks, smem, [&]() { band32_kernel<R, SMEM, false, true>(p); });
    else emu::launch(nblocks, smem, [&]() { band32_kernel<R, SMEM, false, false>(p); });
}

// R: 2 / 4 / 8 / 16 (registers) or 0 (shared memory, p.rr offsets per lane).  With trace, the walk follows and
// writes rev_ops (per pair lq + lr + 2 words at rev_off, reversed run list), nops, beg_query, beg_ref.
extern "C" int emu_band32(int R, int stats, int trace, const Band32Params *pp, int nblocks, unsigned *rev_ops,
                          const long long *rev_off, int *nops, int *beg_query, int *beg_ref) {
    Band32Params p = *pp;
    const size_t smem = band32_smem_bytes(p.is_pssm ? 0 : p.size, 1, R == 0, p.rr, stats != 0);
    switch (R) {
        case 0: run_band<2, true>(p, stats, trace, nblocks, smem); break;
        case 2: run_band<2, false>(p, stats, trace, nblocks, smem); break;
        case 4: run_band<4, false>(p, stats, trace, nblocks, smem); break;
        case 8: run_band<8, false>(p, stats, trace, nblocks, smem); break;
        case 16: run_band<16, false>(p, stats, trace, nblocks, smem); break;
        default: return -1;
    }
    if (trace) {
        WalkParams w;
        std::memset(&w, 0, sizeof(w));
        w.q = p.q; w.q_off = p.q_off; w.r = p.r; w.r_off = p.r_off; w.shared_query = p.shared_query;
        w.ids = nullptr; w.n = p.n; w.trace = p.trace; w.trace_off = p.trace_off; w.end_query = p.end_query; w.end_ref = p.end_ref;
        w.rev_ops = rev_ops; w.rev_off = rev_off; w.nops = nops; w.beg_query = beg_query; w.beg_ref = beg_ref;
        emu::launch((p.n + 31) / 32, 64, [&]() { walk_band_kernel(w, p.k); });
    }
    return 0;
}
extern "C" int emu_sizeof_band32() { return (int)sizeof(Band32Params); }
