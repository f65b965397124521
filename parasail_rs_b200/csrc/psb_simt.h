// psb_simt.h -- the handful of SIMT primitives the kernels use, in two spellings:
//   * nvcc / sm_100a: the real intrinsics (this is the only thing the product library uses);
//   * -DPSB_EMULATE (g++, tests only): every lane of a warp is an OS thread and the warp
//     primitives are rendezvous points, so the *same kernel source* can be stepped on a CPU
//     box that has no GPU.  The emulation exists to catch logic errors before GPU time is
//     spent; it is never linked into libparasail_b200.so.
#pragma once
#include <stdint.h>

#if !defined(PSB_EMULATE)
// ------------------------------------------------------------------------------------------
#include <cuda_runtime.h>
#define PSB_DEV __device__ __forceinline__
#define PSB_HD __host__ __device__ __forceinline__   // shared by a kernel and its host-side launcher
#define PSB_KERNEL __global__
#define PSB_SHARED_DECL(name) extern __shared__ __align__(16) unsigned char name[]

namespace psb {
PSB_DEV int lane_id() { return (int)(threadIdx.x & 31u); }
PSB_DEV int warp_in_block() { return (int)(threadIdx.x >> 5); }
PSB_DEV int warps_per_block() { return (int)(blockDim.x >> 5); }
PSB_DEV int block_id() { return (int)blockIdx.x; }
PSB_DEV int grid_blocks() { return (int)gridDim.x; }
PSB_DEV int thread_in_block() { return (int)threadIdx.x; }
PSB_DEV int threads_per_block() { return (int)blockDim.x; }
PSB_DEV void sync_warp() { __syncwarp(); }
PSB_DEV void sync_block() { __syncthreads(); }
template <typename T> PSB_DEV T shfl_up(T v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }
template <typename T> PSB_DEV T shfl(T v, int src) { return __shfl_sync(0xffffffffu, v, src); }
template <typename T> PSB_DEV T shfl_xor(T v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
PSB_DEV unsigned ballot(bool p) { return __ballot_sync(0xffffffffu, p); }
PSB_DEV unsigned long long atomic_add(unsigned long long *p, unsigned long long v) { return atomicAdd(p, v); }
PSB_DEV int atomic_add(int *p, int v) { return atomicAdd(p, v); }
template <typename T> PSB_DEV T ld_cg(const T *p) { return __ldcg(p); }
template <typename T> PSB_DEV void st_cg(T *p, T v) { __stcg(p, v); }
template <typename T> PSB_DEV T ld_ro(const T *p) { return __ldg(p); }
// DPX (sm_90+: VIADDMNMX / VIMNMX3 and their .S16x2 forms)
PSB_DEV int viaddmax(int a, int b, int c) { return __viaddmax_s32(a, b, c); }            // max(a+b, c)
PSB_DEV int viaddmax_relu(int a, int b, int c) { return __viaddmax_s32_relu(a, b, c); }  // max(a+b, c, 0)
PSB_DEV int vimax3(int a, int b, int c) { return __vimax3_s32(a, b, c); }
PSB_DEV unsigned viaddmax2(unsigned a, unsigned b, unsigned c) { return __viaddmax_s16x2(a, b, c); }
PSB_DEV unsigned viaddmax2_relu(unsigned a, unsigned b, unsigned c) { return __viaddmax_s16x2_relu(a, b, c); }
PSB_DEV unsigned vimax3_2(unsigned a, unsigned b, unsigned c) { return __vimax3_s16x2(a, b, c); }
PSB_DEV unsigned vimax2(unsigned a, unsigned b) { return __vmaxs2(a, b); }
PSB_DEV unsigned vimax2_relu(unsigned a, unsigned b) { return __vimax_s16x2_relu(a, b); }   // max(a, b, 0) per half
PSB_DEV void st_cs(uint4 *p, uint4 v) { __stcs(p, v); }   // streaming: written once, read by a later kernel
PSB_DEV void st_cs(uint2 *p, uint2 v) { __stcs(p, v); }
PSB_DEV void st_cg(uint4 *p, uint4 v) { __stcg(p, v); }
PSB_DEV void st_cg(uint2 *p, uint2 v) { __stcg(p, v); }
PSB_DEV unsigned vadd2(unsigned a, unsigned b) { return __vadd2(a, b); }
PSB_DEV int find_first_set(unsigned v) { return __ffs((int)v); }   // 1-based position of the lowest set bit, 0 for 0
PSB_DEV int pop_count(unsigned v) { return __popc(v); }
PSB_DEV unsigned funnel_l1(unsigned lo, unsigned hi) { return __funnelshift_l(lo, hi, 1); }   // (hi << 1) | (lo >> 31)
// prmt.b32 with the sign-replicate selector bit (the __byte_perm intrinsic masks it off)
PSB_DEV unsigned prmt(unsigned a, unsigned b, unsigned sel) {
    unsigned d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}
}  // namespace psb

#else  // PSB_EMULATE ------------------------------------------------------------------------
#include <algorithm>
#include <atomic>
#include <barrier>
#include <cstring>
#include <functional>
#include <thread>
#include <vector>
#define PSB_DEV inline
#define PSB_HD inline
#define PSB_KERNEL
#define PSB_SHARED_DECL(name) unsigned char *name = psb::emu::tls().smem

struct uint4 { unsigned x, y, z, w; };
struct uint2 { unsigned x, y; };
namespace psb {
namespace emu {
struct Block {
    std::barrier<> bar{32};
    unsigned long long slots[32];
    std::vector<unsigned char> smem;
};
struct Tls {
    int lane = 0, block = 0, nblocks = 1;
    Block *blk = nullptr;
    unsigned char *smem = nullptr;
};
inline Tls &tls() {
    static thread_local Tls t;
    return t;
}
// run `fn` as a grid of `nblocks` one-warp blocks, blocks one after another
inline void launch(int nblocks, size_t smem_bytes, const std::function<void()> &fn) {
    for (int b = 0; b < nblocks; ++b) {
        Block blk;
        blk.smem.assign(smem_bytes + 64, 0);
        std::vector<std::thread> th;
        for (int l = 0; l < 32; ++l)
            th.emplace_back([&, l]() {
                Tls &t = tls();
                t.lane = l; t.block = b; t.nblocks = nblocks; t.blk = &blk;
                t.smem = (unsigned char *)(((uintptr_t)blk.smem.data() + 15) & ~(uintptr_t)15);
                fn();
            });
        for (auto &t : th) t.join();
    }
}
template <typename T> inline T exchange(T v, int src_lane_or_neg) {
    Tls &t = tls();
    unsigned long long raw = 0;
    std::memcpy(&raw, &v, sizeof(T));
    t.blk->slots[t.lane] = raw;
    t.blk->bar.arrive_and_wait();
    unsigned long long got = (src_lane_or_neg >= 0 && src_lane_or_neg < 32) ? t.blk->slots[src_lane_or_neg] : raw;
    t.blk->bar.arrive_and_wait();
    T r;
    std::memcpy(&r, &got, sizeof(T));
    return r;
}
}  // namespace emu

inline int lane_id() { return emu::tls().lane; }
inline int warp_in_block() { return 0; }
inline int warps_per_block() { return 1; }
inline int block_id() { return emu::tls().block; }
inline int grid_blocks() { return emu::tls().nblocks; }
inline int thread_in_block() { return emu::tls().lane; }
inline int threads_per_block() { return 32; }
inline void sync_warp() { emu::tls().blk->bar.arrive_and_wait(); }
inline void sync_block() { emu::tls().blk->bar.arrive_and_wait(); }
template <typename T> inline T shfl_up(T v, int d) { int l = lane_id(); return emu::exchange(v, l >= d ? l - d : -1); }
template <typename T> inline T shfl(T v, int src) { return emu::exchange(v, src & 31); }
template <typename T> inline T shfl_xor(T v, int m) { return emu::exchange(v, lane_id() ^ m); }
inline unsigned ballot(bool p) {
    unsigned mine = p ? (1u << lane_id()) : 0u, all = 0;
    for (int l = 0; l < 32; ++l) all |= emu::exchange(mine, l);
    return all;
}
inline unsigned long long atomic_add(unsigned long long *p, unsigned long long v) { return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
inline int atomic_add(int *p, int v) { return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
template <typename T> inline T ld_cg(const T *p) { return *(const volatile T *)p; }
template <typename T> inline void st_cg(T *p, T v) { *(volatile T *)p = v; }
template <typename T> inline T ld_ro(const T *p) { return *p; }
inline int viaddmax(int a, int b, int c) { return std::max(a + b, c); }
inline int viaddmax_relu(int a, int b, int c) { return std::max(std::max(a + b, c), 0); }
inline int vimax3(int a, int b, int c) { return std::max(a, std::max(b, c)); }
inline int16_t lo16(unsigned a) { return (int16_t)(a & 0xffffu); }
inline int16_t hi16(unsigned a) { return (int16_t)(a >> 16); }
inline unsigned pack16(int lo, int hi) { return ((unsigned)lo & 0xffffu) | ((unsigned)hi << 16); }
inline unsigned viaddmax2(unsigned a, unsigned b, unsigned c) {
    int l = std::max((int)(int16_t)(lo16(a) + lo16(b)), (int)lo16(c));
    int h = std::max((int)(int16_t)(hi16(a) + hi16(b)), (int)hi16(c));
    return pack16(l, h);
}
inline unsigned viaddmax2_relu(unsigned a, unsigned b, unsigned c) {
    int l = std::max(std::max((int)(int16_t)(lo16(a) + lo16(b)), (int)lo16(c)), 0);
    int h = std::max(std::max((int)(int16_t)(hi16(a) + hi16(b)), (int)hi16(c)), 0);
    return pack16(l, h);
}
inline unsigned vimax3_2(unsigned a, unsigned b, unsigned c) {
    return pack16(std::max((int)lo16(a), std::max((int)lo16(b), (int)lo16(c))),
                  std::max((int)hi16(a), std::max((int)hi16(b), (int)hi16(c))));
}
inline unsigned vimax2(unsigned a, unsigned b) {
    return pack16(std::max((int)lo16(a), (int)lo16(b)), std::max((int)hi16(a), (int)hi16(b)));
}
inline unsigned vadd2(unsigned a, unsigned b) { return pack16(lo16(a) + lo16(b), hi16(a) + hi16(b)); }
inline int find_first_set(unsigned v) { return __builtin_ffs((int)v); }
inline int pop_count(unsigned v) { return __builtin_popcount(v); }
inline unsigned funnel_l1(unsigned lo, unsigned hi) { return (hi << 1) | (lo >> 31); }
inline unsigned vimax2_relu(unsigned a, unsigned b) {
    return pack16(std::max(std::max((int)lo16(a), (int)lo16(b)), 0), std::max(std::max((int)hi16(a), (int)hi16(b)), 0));
}
inline void st_cs(uint4 *p, uint4 v) { *p = v; }
inline void st_cs(uint2 *p, uint2 v) { *p = v; }
inline void st_cg(uint4 *p, uint4 v) { *p = v; }
inline void st_cg(uint2 *p, uint2 v) { *p = v; }
inline unsigned prmt(unsigned a, unsigned b, unsigned sel) {
    unsigned long long src = ((unsigned long long)b << 32) | a;
    unsigned d = 0;
    for (int k = 0; k < 4; ++k) {
        unsigned s = (sel >> (4 * k)) & 0xf;
        unsigned byte = (unsigned)((src >> (8 * (s & 7))) & 0xff);
        if (s & 8) byte = (byte & 0x80) ? 0xff : 0x00;
        d |= byte << (8 * k);
    }
    return d;
}
}  // namespace psb
#endif
