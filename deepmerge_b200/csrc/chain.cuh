// The machinery shared by the two tracers of boundary chains, the polygonizer (polygon.cu) and the boundary-line tracer
// (lines.cu).  Both give every pixel a 4-bit mask of the boundary elements it owns (8 pixels per uint32, one element
// count per 32-pixel word of a row), scan the word counts into word bases, so that element (pixel p, bit s) has the
// dense index base[word] + popc(masks of the word before p) + popc(mask[p] below s), and follow successor pointers by
// pointer jumping.  counts is the int64 [4] word of both entry points: [0] chains listed, [2] elements found, [3] status.
//
// A tracer is a rule type Rule with
//   Ws                                 its workspace, which starts with Front and is carved by carve_front first;
//   mask(L, H, W, ld, x, y)            the 4-bit mask of the elements pixel (x, y) owns;
//   emit(L, H, W, ld, wpr, masks, wbase, x, y, s, i, ws)
//                                      element i, bit s of pixel (x, y): its head vertex, successor, flags and phase-0
//                                      word;
//   start(counts, W, cap, ws, i)       after phase 0: lists the chain element i starts, if any, and turns its word into
//                                      phase 1's.
// trace<Rule> runs the front half of an entry point on them: mask -> scan -> emit -> jump phase 0 -> starts -> jump
// phase 1.
#pragma once
#include "common.cuh"
#include "prims.cuh"

namespace dm {
namespace chain {

constexpr int NT = 256;
constexpr int MAX_PASSES = 64;

// The front of both workspaces: the mask pass and its scan, the jump flags, and per element its head vertex index
// y (W + 1) + x, its successor, its flags and its pointer-jumping word (value << 32 | pointer).
struct Front {
    uint32_t *masks, *wcnt, *wbase;
    void* scan;
    int64_t* n_words_dev;
    int* changed;                       // [2][MAX_PASSES]: pass k of phase f changed a word
    uint32_t *hv, *nxt;
    uint8_t* flags;
    uint64_t* jw;
};

// cap elements; scan_cap is the longest scan the tracer runs after the word counts'.
inline void carve_front(Front& f, Carver& c, int64_t H, int64_t W, int64_t cap, int64_t scan_cap) {
    const int64_t n_words = H * ceil_div(W, 32);
    f.masks = c.take<uint32_t>((size_t)n_words * 4);
    f.wcnt = c.take<uint32_t>((size_t)n_words);
    f.wbase = c.take<uint32_t>((size_t)n_words);
    f.scan = c.take<char>(prims::scan_ws_bytes(imax64(n_words, scan_cap)));
    f.n_words_dev = c.take<int64_t>(1);
    f.changed = c.take<int>(2 * MAX_PASSES);
    f.hv = c.take<uint32_t>((size_t)cap);
    f.nxt = c.take<uint32_t>((size_t)cap);
    f.flags = c.take<uint8_t>((size_t)cap);
    f.jw = c.take<uint64_t>((size_t)cap);
}

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

// One warp per 32-pixel word: every element of the word gets its dense index from the word base and a scan of the
// lanes' element counts, and Rule::emit writes it.  Sets status 2 instead when counts[2] elements exceed cap.
template <class Rule>
static __global__ void __launch_bounds__(NT) emit_kernel(const int32_t* __restrict__ L, int64_t H, int64_t W, int64_t ld,
                                                         int64_t wpr, int64_t cap, const uint32_t* __restrict__ masks,
                                                         const uint32_t* __restrict__ wbase,
                                                         int64_t* __restrict__ counts, typename Rule::Ws ws) {
    if (failed(counts)) return;
    if (counts[2] > cap) {
        if (blockIdx.x == 0 && threadIdx.x == 0) counts[3] = 2;
        return;
    }
    const int lane = threadIdx.x & 31;
    const int64_t n_words = H * wpr;
    const int64_t warp0 = ((int64_t)blockIdx.x * NT + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * NT) >> 5;
    for (int64_t w = warp0; w < n_words; w += nwarps) {
        const int64_t y = w / wpr, x = (w - y * wpr) * 32 + lane;
        const unsigned m = (masks[w * 4 + (lane >> 3)] >> (4 * (lane & 7))) & 15u;
        if (!__any_sync(0xffffffffu, m)) continue;
        const unsigned c = __popc(m);
        unsigned inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        uint32_t i = wbase[w] + inc - c;
        for (int s = 0; s < 4; ++s) {
            if (!((m >> s) & 1u)) continue;
            Rule::emit(L, H, W, ld, wpr, masks, wbase, x, y, s, i, ws);
            ++i;
        }
    }
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

// After phase 0: Rule::start for every element.
template <class Rule>
static __global__ void __launch_bounds__(NT) starts_kernel(int64_t* __restrict__ counts, int64_t W, int64_t cap,
                                                           typename Rule::Ws ws) {
    if (failed(counts)) return;
    const int64_t n = counts[2];
    for (int64_t i = (int64_t)blockIdx.x * NT + threadIdx.x; i < n; i += (int64_t)gridDim.x * NT)
        Rule::start(counts, W, cap, ws, i);
}

inline int ceil_log2(int64_t x) {
    int b = 0;
    while (((int64_t)1 << b) < x) ++b;
    return b;
}

// Extents and capacities both tracers accept: every vertex index (H + 1) (W + 1) and every element fit 32 bits.
inline bool extent_ok(int64_t H, int64_t W, int64_t cap) {
    return H >= 0 && W >= 0 && H < (1ll << 31) && W < (1ll << 31) && (H + 1) * (W + 1) <= (1ll << 32) && cap >= 0 &&
           cap < (1ll << 31);
}

// The scalar arguments of both entry points.
inline bool args_ok(int64_t H, int64_t W, int64_t ld, int64_t n_regions, int64_t cap) {
    return extent_ok(H, W, cap) && ld >= W && n_regions >= 0 && n_regions < (1ll << 31);
}

// An empty raster has no elements and no chains: counts and the first offset are cleared where given.
inline int clear_empty(int64_t* counts, int64_t* offsets, cudaStream_t s) {
    if (counts) DM_CUDA(cudaMemsetAsync(counts, 0, 4 * sizeof(int64_t), s));
    if (offsets) DM_CUDA(cudaMemsetAsync(offsets, 0, sizeof(int64_t), s));
    return DM_OK;
}

// The front half of both entry points, on a workspace w carved for cap elements: clears counts and the jump flags,
// then runs mask -> scan -> emit -> jump phase 0 -> starts -> jump phase 1, the per-element kernels on one grid.
template <class Rule>
int trace(const int32_t* labels, int64_t H, int64_t W, int64_t ld, int64_t n_regions, int64_t cap, int64_t* counts,
          const typename Rule::Ws& w, cudaStream_t s) {
    const int64_t wpr = ceil_div(W, 32), n_words = H * wpr;
    DM_CUDA(cudaMemsetAsync(counts, 0, 4 * sizeof(int64_t), s));
    DM_CUDA(cudaMemsetAsync(w.changed, 0, 2 * MAX_PASSES * sizeof(int), s));
    const unsigned g_words = grid_for(n_words * 32, NT, 16), g_elems = grid_for(cap, NT, 16);
    DM_TRY(launch(mask_kernel<Rule>, g_words, NT, 0, s, labels, H, W, ld, wpr, n_regions, w.masks, w.wcnt, counts,
                  w.n_words_dev));
    DM_TRY(prims::scan_exclusive_u32(w.wcnt, w.wbase, w.n_words_dev, n_words, nullptr, w.scan, s));
    DM_TRY(launch(emit_kernel<Rule>, g_words, NT, 0, s, labels, H, W, ld, wpr, cap, w.masks, w.wbase, counts, w));
    const int passes = ceil_log2(cap) + 1;
    for (int phase = 0; phase < 2; ++phase) {
        for (int k = 0; k < passes; ++k)
            DM_TRY(launch(jump_kernel, g_elems, NT, 0, s, w.jw, counts, w.changed, phase, k));
        if (phase == 0) DM_TRY(launch(starts_kernel<Rule>, g_elems, NT, 0, s, counts, W, cap, w));
    }
    return DM_OK;
}

}  // namespace chain
}  // namespace dm
