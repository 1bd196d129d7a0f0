// TMA (cp.async.bulk.tensor) and mbarrier primitives of the kernels that stage padded plane rows in shared memory:
// the ellipse morphology producers (lt_morph.cu) and the vertical threshold ring (lt_filter.cu).
#pragma once
#include <cuda.h>                    // CUtensorMap (types only: the encoder is fetched with cudaGetDriverEntryPoint)
#include "lt_common.cuh"

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
// makes the barriers initialised above visible to the async proxy (the bulk copies that complete on them)
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n.reg .pred p;\nWAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@!p bra WAIT_%=;\n}\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
}
// box at column x, row y of `map` -> smem_dst; completes `bar`'s transaction count
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int x, int y, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(map), "r"(x), "r"(y),
                   "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
// orders this thread's generic-proxy accesses to shared memory before the bulk copies it issues next
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Tensor map of the padded plane allocation behind `plane` (lt_morph.cu): 2-D uint32 [rows][pp] over all streams, box =
// box_w columns x 8 rows.  Packed column x, row y of stream s is map column LT_HALO_X + x, map row
// s * (bv_h + 2 * LT_HALO_Y) + LT_HALO_Y + y.  Cached per (device, allocation, geometry).
int lt_plane_tensor_map(lt_handle* h, const uint32_t* plane, int box_w, CUtensorMap* out);
