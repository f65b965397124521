// pairs16_host.h -- launch interface of the packed 16-bit many-pairs kernels (pairs16.cu), kept in its own
// translation unit so that its ~50 template instantiations compile beside engine.cu, not after it; and the
// persistent-grid launch both translation units use.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <string>

#include "kern_pairs16.cuh"

namespace psb {

// CTAs of `fn` (`wpb` warps, `smem` bytes of dynamic shared memory) that one SM holds at once, at least 1.  Raises the
// kernel's shared-memory limit to `smem` first when that is above the 48 KB default.
inline cudaError_t occupancy_per_sm(const void *fn, int wpb, size_t smem, int *per_sm) {
    cudaError_t e = cudaSuccess;
    if (smem > 48 * 1024) e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    *per_sm = 0;
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, fn, wpb * 32, smem);
    if (*per_sm < 1) *per_sm = 1;
    return e;
}
// A persistent grid of CTAs of `wpb` warps: one warp per work item, capped at `per_sm` CTAs on each of `sms` SMs (the
// kernel's warps then loop over the items left), at least one CTA.  *blocks_out: the grid launched.
inline cudaError_t launch_persistent(const void *fn, void *params, long long items, int wpb, size_t smem, int per_sm, int sms,
                                     cudaStream_t stream, long long *blocks_out = nullptr) {
    const long long blocks = std::max<long long>(1, std::min<long long>((items + wpb - 1) / wpb, (long long)sms * per_sm));
    if (blocks_out) *blocks_out = blocks;
    void *args[] = {params};
    return cudaLaunchKernel(fn, dim3((unsigned)blocks), dim3(wpb * 32), args, smem, stream);
}

struct P16Class { int G, K; };
int p16_num_classes();
P16Class p16_class(int idx);
// smallest class whose G*K rows hold a query of lq residues; prefer_wide chooses the 32-lane groups (half
// the profile bytes per warp, two pairs per warp) when both group widths could hold it.  -1: none.
int p16_pick_class(int lq, bool prefer_wide);
// grid = min(work, resident capacity) persistent warps; returns PSB_OK or a PSB_E* code with *err filled
int p16_launch(int cls, bool sw, bool trace, const Pairs16Params &p, int sms, cudaStream_t stream, std::string *err,
               int *warps_per_sm_out = nullptr);
int p16_launch_walk(const Walk16Params &w, bool stats, cudaStream_t stream, std::string *err);

}  // namespace psb
