// TMA / mbarrier helpers shared by the streaming scan (detect_scan_tma.cu) and the piece filter (detect_cluster.cu); sm_100a.
// The CPU emulation build (-DMOCAP_EMU, tests/emu) gets stand-ins for what the piece filter uses, see the end of the file.
#pragma once
#include "common.cuh"
#ifndef MOCAP_EMU
#include <cuda.h>

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity)
{
    asm volatile("{\n\t.reg .pred P1;\n\tLAB_WAIT:\n\tmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t@P1 bra DONE;\n\tbra LAB_WAIT;\n\tDONE:\n\t}"
                 :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
// makes the barriers thread 0 initialised visible to the TMA unit before the first copy completes on them
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// one box of a 3-D tensor [z][y][x] -> shared memory, completion on `bar` (bytes), with / without an L2 cache policy
__device__ __forceinline__ void tma_load_box(void* dst, const CUtensorMap* map, int x, int y, int z, uint64_t* bar, uint64_t policy)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
                 :: "r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(x), "r"(y), "r"(z), "l"(policy) : "memory");
}
__device__ __forceinline__ void tma_load_box(void* dst, const CUtensorMap* map, int x, int y, int z, uint64_t* bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 :: "r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(x), "r"(y), "r"(z) : "memory");
}
#else
// Stand-ins of the CPU emulation build, for the piece filter's source window.  tma_load_box copies the whole box before it
// returns, so the barrier calls have nothing to do.  That is only valid where the issuing thread then reaches a __syncthreads()
// that every reader of the box passes after its mbar_wait and before it reads: a reader can then never see a box in flight.
#define __grid_constant__
struct CUtensorMap {                   // a frame batch viewed as u8 [n][H][W], frames fstride bytes apart; boxes box_w x box_h
    const uint8_t* base;
    int n, H, W;
    int64_t fstride;
    int box_w, box_h;
};
static inline void mbar_init(uint64_t*, unsigned) {}
static inline void mbar_init_fence() {}
static inline void mbar_expect_tx(uint64_t*, unsigned) {}
static inline void mbar_wait(uint64_t*, unsigned) {}
// box at (x, y) of frame z -> dst; every byte outside [0, W) x [0, H) of frame z reads 0, as the TMA unit fills it
static inline void tma_load_box(void* dst, const CUtensorMap* map, int x, int y, int z, uint64_t*, uint64_t)
{
    uint8_t* out = (uint8_t*)dst;
    memset(out, 0, (size_t)map->box_w * map->box_h);
    if (z < 0 || z >= map->n) return;
    const int x0 = max(x, 0), x1 = min(x + map->box_w, map->W);                    // the columns inside the frame
    if (x0 >= x1) return;
    for (int r = 0; r < map->box_h; ++r) {
        const int gy = y + r;
        if (gy >= 0 && gy < map->H)
            memcpy(out + (size_t)r * map->box_w + (x0 - x), map->base + z * map->fstride + (int64_t)gy * map->W + x0, x1 - x0);
    }
}
#endif

// tensor map of a frame batch viewed as u8 [n][H][W] with boxes of box_w x box_h x 1 (detect_scan_tma.cu); false when the driver entry point
// is missing or the batch cannot be described; l2_promotion: bytes (0, 64, 128, 256) a fetch is widened to in L2 (rows / frame stride / base not multiples of 16 bytes)
bool frames_tensor_map(CUtensorMap* out, const uint8_t* frames, int n, int H, int W, int64_t fstride, int box_w, int box_h, int l2_promotion);
