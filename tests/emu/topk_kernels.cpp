// topk_kernels.cpp -- TEST ONLY.  The selection of a query's best subjects (csrc/kern_topk.cuh) compiled with
// -DPSB_EMULATE (every lane an OS thread, see csrc/psb_simt.h), with the host flow of search.cu, so that it can be
// stepped on a CPU-only box and compared with np.lexsort.  Driven by tests/emu_topk.py.
#define PSB_EMULATE 1
#include <cstring>
#include <vector>

#include "../../parasail_rs_b200/csrc/kern_topk.cuh"

using namespace psb;

// score / end_query / end_ref: n results in caller order; `nblocks` histogram blocks, `nwarps` compaction warps.
// Writes kk rows (ids, scores, end_query, end_ref) in the kernel's order.  -1: the radix select's state does not add
// up to kk, or the warps' counts disagree with it.
extern "C" int emu_topk(int *score, int *end_query, int *end_ref, long long n, int kk, int nblocks, int nwarps, int *out_id, int *out_score,
                        int *out_end_query, int *out_end_ref) {
    TopkState st;
    std::memset(&st, 0, sizeof(st));
    std::vector<int> counts(2 * (size_t)nwarps), sat_rows((size_t)kk);
    std::vector<long long> offs(2 * (size_t)nwarps);
    TopkParams p;
    std::memset(&p, 0, sizeof(p));
    p.score = score; p.end_query = end_query; p.end_ref = end_ref; p.n = n; p.kk = kk; p.st = &st;
    p.chunk = topk_chunk(n, nwarps); p.nwarps = nwarps; p.counts = counts.data(); p.offs = offs.data();
    p.out_id = out_id; p.out_score = out_score; p.out_end_query = out_end_query; p.out_end_ref = out_end_ref; p.out_sat = sat_rows.data();
    for (int shift = 24; shift >= 0; shift -= 8) {
        p.shift = shift;
        emu::launch(nblocks, kTopkBins * sizeof(int), [&]() { topk_hist_kernel(p); });
        emu::launch(1, 0, [&]() { topk_pick_kernel(p); });
    }
    emu::launch(nwarps, 0, [&]() { topk_take_kernel<false>(p); });
    long long run = 0;
    for (size_t w = 0; w < counts.size(); ++w) { offs[w] = run; run += counts[w]; }
    if (offs[(size_t)nwarps] != st.above || st.above + st.need != kk) return -1;
    emu::launch(nwarps, 0, [&]() { topk_take_kernel<true>(p); });
    return 0;
}
