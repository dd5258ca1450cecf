// Kernels shared by the two tracers of boundary chains, the polygonizer (polygon.cu) and the boundary-line tracer
// (lines.cu).  Both give every pixel a 4-bit mask of the boundary elements it owns (8 pixels per uint32, one element
// count per 32-pixel word of a row), scan the word counts into word bases, so that element (pixel p, bit s) has the
// dense index base[word] + popc(masks of the word before p) + popc(mask[p] below s), and follow successor pointers by
// pointer jumping.  counts is the int64 [4] word of both entry points: [2] elements found, [3] status.
#pragma once
#include "common.cuh"

namespace dm {
namespace chain {

constexpr int NT = 256;
constexpr int MAX_PASSES = 64;

__device__ __forceinline__ uint64_t ld_relaxed(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed(uint64_t* p, uint64_t v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__device__ __forceinline__ bool failed(const int64_t* counts) { return *(volatile const int64_t*)(counts + 3) != 0; }

// One pass over the labels: Rule::mask(L, H, W, ld, x, y) is the 4-bit mask of pixel (x, y).  Writes the masks, the
// count per word, adds the total to counts[2] and sets status 1 for a label >= n_regions.
template <class Rule>
static __global__ void __launch_bounds__(NT) mask_kernel(const int32_t* __restrict__ L, int64_t H, int64_t W, int64_t ld,
                                                         int64_t wpr, int64_t n_regions, uint32_t* __restrict__ masks,
                                                         uint32_t* __restrict__ wcnt, int64_t* __restrict__ counts,
                                                         int64_t* __restrict__ n_words_dev) {
    const int lane = threadIdx.x & 31;
    const int64_t n_words = H * wpr;
    const int64_t warp0 = ((int64_t)blockIdx.x * NT + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * NT) >> 5;
    if (blockIdx.x == 0 && threadIdx.x == 0) *n_words_dev = n_words;
    unsigned long long total = 0;
    bool bad = false;
    for (int64_t w = warp0; w < n_words; w += nwarps) {
        const int64_t y = w / wpr, x = (w - y * wpr) * 32 + lane;
        unsigned m = 0;
        if (x < W) {
            bad |= L[y * ld + x] >= n_regions;
            m = Rule::mask(L, H, W, ld, x, y);
        }
        unsigned v = m << (4 * (lane & 7));
        v |= __shfl_xor_sync(0xffffffffu, v, 1);
        v |= __shfl_xor_sync(0xffffffffu, v, 2);
        v |= __shfl_xor_sync(0xffffffffu, v, 4);
        if ((lane & 7) == 0) masks[w * 4 + (lane >> 3)] = v;
        const unsigned c = __reduce_add_sync(0xffffffffu, (unsigned)__popc(m));
        if (lane == 0) wcnt[w] = c;
        total += c;
    }
    if (__any_sync(0xffffffffu, bad) && lane == 0) atomicExch((unsigned long long*)(counts + 3), 1ull);
    if (lane == 0 && total) atomicAdd((unsigned long long*)(counts + 2), total);
}

// dense index of element s of pixel (x, y)
__device__ __forceinline__ uint32_t dense_index(const uint32_t* masks, const uint32_t* wbase, int64_t wpr, int64_t x,
                                                int64_t y, int s) {
    const int64_t w = y * wpr + (x >> 5);
    const int k = (int)(x & 31);
    const uint32_t* m = masks + w * 4;
    uint32_t i = wbase[w];
    for (int j = 0; j < (k >> 3); ++j) i += __popc(m[j]);
    return i + __popc(m[k >> 3] & ((1u << (4 * (k & 7) + s)) - 1u));
}

// One pointer-jumping pass over the counts[2] elements, in place on packed (value << 32 | pointer) words.  phase 0:
// value = minimum over the elements [i, pointer); phase 1: value = sum over (i, pointer], where an element that ends its
// chain points at itself with value 0.  Every pass at least doubles the span a word covers, so ceil(log2(capacity))
// passes suffice; a pass that changes nothing ends the phase early (the remaining launches return at once).  A word
// read while its owner rewrites it is an older or newer (value, pointer) pair, both of which hold the invariant.
static __global__ void __launch_bounds__(NT) jump_kernel(uint64_t* jw, const int64_t* __restrict__ counts, int* changed,
                                                         int phase, int pass) {
    if (failed(counts)) return;
    int* ch_flags = changed + phase * MAX_PASSES;
    if (pass > 0 && !ch_flags[pass - 1]) return;
    const int64_t n = counts[2];
    bool ch = false;
    for (int64_t i = (int64_t)blockIdx.x * NT + threadIdx.x; i < n; i += (int64_t)gridDim.x * NT) {
        const uint64_t w = ld_relaxed(jw + i);
        const uint32_t p = (uint32_t)w;
        const uint64_t t = ld_relaxed(jw + p);
        uint64_t nw;
        if (phase == 0) {
            const uint64_t mn = min(w >> 32, t >> 32);
            ch |= mn != (w >> 32);
            nw = (mn << 32) | (uint32_t)t;
        } else {
            ch |= (uint32_t)t != p;
            nw = (((w >> 32) + (t >> 32)) << 32) | (uint32_t)t;
        }
        st_relaxed(jw + i, nw);
    }
    if (__syncthreads_or(ch) && threadIdx.x == 0) ch_flags[pass] = 1;
}

inline int ceil_log2(int64_t x) {
    int b = 0;
    while (((int64_t)1 << b) < x) ++b;
    return b;
}

}  // namespace chain
}  // namespace dm
