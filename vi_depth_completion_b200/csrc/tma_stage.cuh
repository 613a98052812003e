// tma_stage.cuh -- Blackwell/Hopper TMA staging of a tile's source footprint into shared memory.
//
// The gather of the warp kernels is limited by the L1 data pipe: a 32-lane bilinear tap load touches
// ~3.6 cache lines, 12-16 such requests per row segment.  Here ONE thread issues a tiled bulk tensor copy
// (cp.async.bulk.tensor, SASS UTMALDG) of the footprint's bounding box -- all planes at once, completion
// on an mbarrier -- and the taps are then read from shared memory with immediate offsets and no bounds
// tests: the TMA unit zero-fills everything outside the tensor, which IS padding_mode='zeros'.
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace vidc_k {

constexpr int TMA_BW = 64;                           // box width in floats (smem row pitch)
constexpr int TMA_NH = 4;                            // box-height classes
__host__ __device__ constexpr int tma_box_h(int cls) { return cls == 0 ? 24 : cls == 1 ? 32 : cls == 2 ? 40 : 48; }
constexpr int TMA_BH_MAX = 48;

struct TmaMaps {                                     // one tensor map per box-height class
    CUtensorMap a[TMA_NH];                           // planes of image A (RGB or normals), box (64, h, C, 1)
    CUtensorMap d[TMA_NH];                           // depth, box (64, h, 1, 1)
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // make the init visible to the async (TMA) proxy
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t phase) {
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(smem_u32(bar)), "r"(phase) : "memory");
    }
}
// 4-D tiled load: coordinates (x, y, plane, frame); out-of-range elements are written as zeros.
// Measured on the B200 (tools/tma_probe4.cu): x * sizeof(float) must be a multiple of 16 bytes -- an unaligned
// innermost coordinate raises 'illegal instruction'; negative and out-of-range coordinates are fine.
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, unsigned long long* bar,
                                            int x, int y, int c, int n) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
        ::"r"(smem_u32(smem_dst)), "l"((unsigned long long)map), "r"(x), "r"(y), "r"(c), "r"(n), "r"(smem_u32(bar))
        : "memory");
}


// ---- tiled bulk tensor STORES (shared -> global, SASS UTMASTG): the write-out of the sheared kernels ----------------------
// Elements of the box that fall outside the tensor are not written.  Every thread that wrote the staged tile through the
// generic proxy fences (fence_async_smem) before the barrier; one thread then issues the stores, commits the group and waits
// until the TMA unit has READ the tile (the CTA must not exit -- and hand its shared memory to the next CTA -- earlier).
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
#ifndef VIDC_TMA_STORE_HINT
#define VIDC_TMA_STORE_HINT 0     // 1: L2::evict_first on the stores (the outputs are never re-read by these kernels): measured neutral
                                  // (forward 0.4934 / 0.4925 ms, inverse 0.4392 / 0.4397 ms, bench 271.9 / 271.6 K frames/s), so off
#endif
__device__ __forceinline__ unsigned long long l2_evict_first_policy() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* smem_src, int x, int y, int c, int n) {
#if VIDC_TMA_STORE_HINT
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group.L2::cache_hint [%0, {%2, %3, %4, %5}], [%1], %6;"
                 ::"l"((unsigned long long)map), "r"(smem_u32(smem_src)), "r"(x), "r"(y), "r"(c), "r"(n), "l"(l2_evict_first_policy()) : "memory");
#else
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                 ::"l"((unsigned long long)map), "r"(smem_u32(smem_src)), "r"(x), "r"(y), "r"(c), "r"(n) : "memory");
#endif
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* smem_src, int x, int y, int n) {
#if VIDC_TMA_STORE_HINT
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group.L2::cache_hint [%0, {%2, %3, %4}], [%1], %5;"
                 ::"l"((unsigned long long)map), "r"(smem_u32(smem_src)), "r"(x), "r"(y), "r"(n), "l"(l2_evict_first_policy()) : "memory");
#else
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"((unsigned long long)map), "r"(smem_u32(smem_src)), "r"(x), "r"(y), "r"(n) : "memory");
#endif
}
__device__ __forceinline__ void tma_store_commit_and_wait_read() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// ---- tiled bulk tensor PREFETCH into L2 (SASS UTMAPF): the L2 prefetch of the sheared kernels -------------------------------
// One instruction from one thread asks the TMA unit for a whole box; no shared memory, no barrier, nothing to wait for, a hint
// only.  Elements of the box outside the tensor are not fetched.
__device__ __forceinline__ void tma_prefetch_l2_4d(const CUtensorMap* map, int x, int y, int c, int n) {
    asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global.tile [%0, {%1, %2, %3, %4}];"
                 ::"l"((unsigned long long)map), "r"(x), "r"(y), "r"(c), "r"(n) : "memory");
}
__device__ __forceinline__ void tma_prefetch_l2_3d(const CUtensorMap* map, int x, int y, int n) {
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];"
                 ::"l"((unsigned long long)map), "r"(x), "r"(y), "r"(n) : "memory");
}

// plain arrive (no transaction bytes) and arrive from a consumer warp
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_init_only(unsigned long long* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

}  // namespace vidc_k
