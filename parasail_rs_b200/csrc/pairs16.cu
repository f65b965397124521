// pairs16.cu -- instantiations and launch code of the packed 16-bit many-pairs kernels (kern_pairs16.cuh).
#include "pairs16_host.h"

#include <algorithm>
#include <cstdlib>

#include "../../include/parasail_b200.h"

namespace psb {

// rows = G*K, ascending; 16-lane groups carry four pairs per warp, 32-lane groups two
static const P16Class kClasses[] = {{16, 4},  {16, 8},  {16, 10}, {16, 12}, {16, 16}, {16, 19}, {16, 22},
                                    {16, 25}, {32, 8},  {32, 10}, {32, 12}, {32, 14}, {32, 16}};
static constexpr int kNumClasses = (int)(sizeof(kClasses) / sizeof(kClasses[0]));
int p16_num_classes() { return kNumClasses; }
P16Class p16_class(int idx) { return kClasses[idx]; }

int p16_pick_class(int lq, bool prefer_wide) {
    int best = -1;
    for (int pass = 0; pass < 2 && best < 0; ++pass) {
        const int want_g = (prefer_wide ? (pass == 0 ? 32 : 16) : (pass == 0 ? 16 : 32));
        for (int c = 0; c < kNumClasses; ++c) {
            if (kClasses[c].G != want_g || kClasses[c].G * kClasses[c].K < lq) continue;
            if (best < 0 || kClasses[c].G * kClasses[c].K < kClasses[best].G * kClasses[best].K) best = c;
        }
        // a wide class wastes rows on short queries: only take it when it is not much larger than the narrow fit
        if (best >= 0 && prefer_wide && pass == 0) {
            int narrow = -1;
            for (int c = 0; c < kNumClasses; ++c)
                if (kClasses[c].G == 16 && kClasses[c].G * kClasses[c].K >= lq && (narrow < 0 || kClasses[c].K < kClasses[narrow].K)) narrow = c;
            if (narrow >= 0 && kClasses[best].G * kClasses[best].K > kClasses[narrow].G * kClasses[narrow].K + 32) best = narrow;
        }
    }
    return best;
}

template <int G, int K> static const void *p16_fn_gk(bool sw, bool trace) {
    if (sw) return trace ? (const void *)pairs16_kernel<G, K, true, true> : (const void *)pairs16_kernel<G, K, true, false>;
    return trace ? (const void *)pairs16_kernel<G, K, false, true> : (const void *)pairs16_kernel<G, K, false, false>;
}
static const void *p16_fn(int cls, bool sw, bool trace) {
    switch (cls) {
        case 0: return p16_fn_gk<16, 4>(sw, trace);
        case 1: return p16_fn_gk<16, 8>(sw, trace);
        case 2: return p16_fn_gk<16, 10>(sw, trace);
        case 3: return p16_fn_gk<16, 12>(sw, trace);
        case 4: return p16_fn_gk<16, 16>(sw, trace);
        case 5: return p16_fn_gk<16, 19>(sw, trace);
        case 6: return p16_fn_gk<16, 22>(sw, trace);
        case 7: return p16_fn_gk<16, 25>(sw, trace);
        case 8: return p16_fn_gk<32, 8>(sw, trace);
        case 9: return p16_fn_gk<32, 10>(sw, trace);
        case 10: return p16_fn_gk<32, 12>(sw, trace);
        case 11: return p16_fn_gk<32, 14>(sw, trace);
        case 12: return p16_fn_gk<32, 16>(sw, trace);
    }
    return nullptr;
}

int p16_launch(int cls, bool sw, bool trace, const Pairs16Params &p, int sms, cudaStream_t stream, std::string *err,
               int *warps_per_sm_out) {
    const void *fn = p16_fn(cls, sw, trace);
    if (!fn) { *err = "pairs16: no kernel for this class"; return PSB_EUNSUPPORTED; }
    const P16Class c = kClasses[cls];
    const int nletters = p.size + 1;
    // warps per CTA: as many as keep the SM's shared memory well used (every warp carries its own profiles)
    int wpb = 4;
    if (const char *ev = std::getenv("PSB_P16_WARPS")) { const int w = std::atoi(ev); if (w >= 1 && w <= 16) wpb = w; }
    size_t smem = pairs16_smem_bytes(c.K, nletters, sw, wpb);
    while (wpb > 1 && (smem > 100 * 1024 || (227 * 1024 / smem) * wpb < (227 * 1024 / pairs16_smem_bytes(c.K, nletters, sw, wpb / 2)) * (wpb / 2))) {
        wpb /= 2;
        smem = pairs16_smem_bytes(c.K, nletters, sw, wpb);
    }
    int per_sm = 0;
    cudaError_t e = occupancy_per_sm(fn, wpb, smem, &per_sm);
    if (e != cudaSuccess) { *err = std::string("pairs16 launch setup: ") + cudaGetErrorString(e); return PSB_ECUDA; }
    if (warps_per_sm_out) *warps_per_sm_out = per_sm * wpb;
    const int ng = 32 / c.G;
    const long long slots = ((long long)p.nitems + ng - 1) / ng;
    Pairs16Params pp = p;
    e = launch_persistent(fn, &pp, slots, wpb, smem, per_sm, sms, stream);
    if (e != cudaSuccess) { *err = std::string("pairs16 launch: ") + cudaGetErrorString(e); return PSB_ECUDA; }
    return PSB_OK;
}

int p16_launch_walk(const Walk16Params &w, bool stats, cudaStream_t stream, std::string *err) {
    if (w.n <= 0) return PSB_OK;
    const size_t smem = walk16_smem_bytes(w.size);
    if (stats) walk16_kernel<true><<<(unsigned)((w.n + 127) / 128), 128, smem, stream>>>(w);
    else walk16_kernel<false><<<(unsigned)((w.n + 127) / 128), 128, smem, stream>>>(w);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { *err = std::string("walk16 launch: ") + cudaGetErrorString(e); return PSB_ECUDA; }
    return PSB_OK;
}

}  // namespace psb
