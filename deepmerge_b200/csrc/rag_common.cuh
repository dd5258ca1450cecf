// Shared between the raster kernels of R1 (rag.cu, rag_blocks.cu): launch parameters, mbarrier / TMA wrappers, tensor-map
// encoding.
#pragma once
#include <cuda.h>
#include <stdlib.h>
#include <string.h>
#include "common.cuh"

namespace dm {
namespace rag {

constexpr int STRIP_W = 128;            // pixels per warp row: 32 lanes x 4
constexpr int LAB_PITCH = STRIP_W + 4;  // + halo columns (TMA inner box must be a multiple of 16 B)
constexpr int RS = 32;                  // region table slots per warp (power of two)
constexpr int ES = 64;                  // edge table slots per warp (power of two)
constexpr int FLUSH_ROWS = 256;         // forced drain period: 128 px * 256 rows * 255^2 < 2^32
constexpr int EMPTY_LABEL = -1;
constexpr unsigned long long EMPTY_KEY = ~0ull;
constexpr int SLOT_NONE = -1;

constexpr int align128(int x) { return (x + 127) / 128 * 128; }

struct Params {
    const int32_t* labels;
    int64_t ld;
    const uint8_t* image;
    int64_t image_pitch;
    int rows_own, rows_avail, W;
    int n_regions;
    int top_border, bottom_border;
    unsigned long long* area;
    unsigned long long* border;
    unsigned long long* bsum;
    unsigned long long* bsq;
    unsigned long long* raw_keys;
    uint32_t* raw_cnt;
    long long capacity;
    unsigned long long* counters;   // [1] raw entries, [2] overflow, [3] bad label / internal error
    int tiles_x, tiles_y, tiles_per_cta;   // strips, row blocks per strip, units per warp
};

// ------------------------------------------------------------------------------------ //
// mbarrier / TMA wrappers
// ------------------------------------------------------------------------------------ //
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, unsigned parity) {
    unsigned ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(100000u)   // suspend-time hint (ns): sleep in HW, do not spin
        : "memory");
    return ok != 0;
}
// Bounded wait: a TMA that never lands must become an error, not a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity, unsigned long long* counters) {
    unsigned spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 20)) {
            atomicExch(&counters[3], 2ull);
            __trap();
        }
    }
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int x, int y, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(dst)),
        "l"((uint64_t)map), "r"(x), "r"(y), "r"(smem_u32(bar))
        : "memory");
}


// host side: tensor maps (rag.cu)
bool make_map_2d(CUtensorMap* m, const void* base, uint64_t dim0, uint64_t dim1, uint64_t pitch_bytes, uint32_t box0,
                 uint32_t box1);
void set_last_path(int path);
int run_blocks(const Params& P, int C, cudaStream_t s);   // rag_blocks.cu

}  // namespace rag
}  // namespace dm
