// Polygonizer: label raster -> closed rings of pixel-corner vertices, one set per region (dm_polygonize in
// include/deepmerge_b200.h).  The per-side rule lives in polygon_core.cuh.
//
// 1. mask_kernel    one pass over the labels: a 4-bit mask of boundary sides per pixel (8 pixels per uint32), one side
//                   count per 32-pixel word of a row, the exact total and the label range check.
// 2. scan           word counts -> word bases, so side (pixel p, side s) has the dense index
//                   base[word] + popc(masks of the word before p) + popc(mask[p] below s).
// 3. emit_kernel    per side: head vertex, region, corner flag and the dense index of its successor (no search).
// 4. jump_kernel    pointer jumping over the successor cycles, in place on packed (value, pointer) words: first the
//                   minimum head vertex of every ring (its canonical start), then, with every cycle cut at its start,
//                   the number of corners from each side to the start.  Every pass at least doubles the span a word
//                   covers, so ceil(log2(capacity)) passes suffice; a pass that changes nothing ends the phase early
//                   (the remaining launches return at once).
// 5. starts_kernel  one ring per start side, listed with its start vertex; sort_pairs orders the list by start vertex
//                   (radix), then stably by region (bucket + rank), whose CSR offsets are region_rings.
// 6. vertex_kernel  corners scattered to ring offset + rank, ring areas as the sum of x * dy over the vertical sides.
#include "common.cuh"
#include "polygon_core.cuh"
#include "prims.cuh"

namespace dm {
namespace poly {
using namespace polycore;

constexpr int NT = 256;
constexpr int MAX_PASSES = 64;
constexpr uint8_t CORNER = 4;   // flags: bits 0-1 side / direction, bit 2 head vertex is a corner

__device__ __forceinline__ uint64_t ld_relaxed(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed(uint64_t* p, uint64_t v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

struct Ws {
    uint32_t *masks, *wcnt, *wbase;
    void* scan;
    int64_t* n_words_dev;
    int* changed;                       // [2][MAX_PASSES]: pass k of phase f changed a word
    uint32_t *hv, *nxt, *ring_of;       // per side: head vertex index y (W+1) + x, successor, ring of a start side
    int32_t* reg;
    uint8_t* flags;
    uint64_t* jw;                       // per side: the pointer-jumping word (value << 32 | pointer)
    uint64_t* rkeys;                    // per ring
    uint32_t *rvals, *ccount, *offs;
    void* sort;
};

size_t carve(Ws& w, void* base, int64_t H, int64_t W, int64_t n_regions, int64_t cap) {
    Carver c(base);
    const int64_t n_words = H * ceil_div(W, 32), ring_cap = cap / 4;
    w.masks = c.take<uint32_t>((size_t)n_words * 4);
    w.wcnt = c.take<uint32_t>((size_t)n_words);
    w.wbase = c.take<uint32_t>((size_t)n_words);
    w.scan = c.take<char>(prims::scan_ws_bytes(imax64(n_words, ring_cap)));
    w.n_words_dev = c.take<int64_t>(1);
    w.changed = c.take<int>(2 * MAX_PASSES);
    w.hv = c.take<uint32_t>((size_t)cap);
    w.nxt = c.take<uint32_t>((size_t)cap);
    w.ring_of = c.take<uint32_t>((size_t)cap);
    w.reg = c.take<int32_t>((size_t)cap);
    w.flags = c.take<uint8_t>((size_t)cap);
    w.jw = c.take<uint64_t>((size_t)cap);
    w.rkeys = c.take<uint64_t>((size_t)ring_cap);
    w.rvals = c.take<uint32_t>((size_t)ring_cap);
    w.ccount = c.take<uint32_t>((size_t)ring_cap);
    w.offs = c.take<uint32_t>((size_t)ring_cap);
    w.sort = c.take<char>(prims::ws_bytes(ring_cap, false, n_regions + 1));
    return c.used();
}

__device__ __forceinline__ bool failed(const int64_t* counts) { return *(volatile const int64_t*)(counts + 3) != 0; }

__global__ void __launch_bounds__(NT) mask_kernel(const int32_t* __restrict__ L, int64_t H, int64_t W, int64_t ld,
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
            m = side_mask(L, H, W, ld, x, y);
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

// dense index of side s of pixel (x, y)
__device__ __forceinline__ uint32_t dense_index(const uint32_t* masks, const uint32_t* wbase, int64_t wpr, int64_t x,
                                                int64_t y, int s) {
    const int64_t w = y * wpr + (x >> 5);
    const int k = (int)(x & 31);
    const uint32_t* m = masks + w * 4;
    uint32_t i = wbase[w];
    for (int j = 0; j < (k >> 3); ++j) i += __popc(m[j]);
    return i + __popc(m[k >> 3] & ((1u << (4 * (k & 7) + s)) - 1u));
}

__global__ void __launch_bounds__(NT) emit_kernel(const int32_t* __restrict__ L, int64_t H, int64_t W, int64_t ld,
                                                  int64_t wpr, int64_t cap, const uint32_t* __restrict__ masks,
                                                  const uint32_t* __restrict__ wbase, int64_t* __restrict__ counts, Ws ws) {
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
            const Succ q = successor(L, H, W, ld, x, y, s);
            const uint32_t j = dense_index(masks, wbase, wpr, q.x, q.y, q.s);
            const uint32_t hv = (uint32_t)(head_y(y, s) * (W + 1) + head_x(x, s));
            ws.hv[i] = hv;
            ws.nxt[i] = j;
            ws.reg[i] = L[y * ld + x];
            ws.flags[i] = (uint8_t)(s | (q.corner ? CORNER : 0));
            ws.jw[i] = ((uint64_t)hv << 32) | j;   // phase 0: minimum head vertex over [i, pointer) = own head
            ++i;
        }
    }
}

// One pointer-jumping pass, in place.  phase 0: value = minimum head vertex over the sides [i, pointer);
// phase 1: value = corners over (i, pointer], the start side of every ring points at itself with value 0.
// A word read while its owner rewrites it is an older or newer (value, pointer) pair, both of which hold the invariant.
__global__ void __launch_bounds__(NT) jump_kernel(uint64_t* jw, const int64_t* __restrict__ counts, int* changed,
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

// After phase 0: the side whose head is its ring's minimum vertex starts the ring.  The word becomes phase 1's.
__global__ void __launch_bounds__(NT) starts_kernel(int64_t* __restrict__ counts, int64_t ring_cap, Ws ws) {
    if (failed(counts)) return;
    const int64_t n = counts[2];
    for (int64_t i = (int64_t)blockIdx.x * NT + threadIdx.x; i < n; i += (int64_t)gridDim.x * NT) {
        const uint32_t hv = ws.hv[i];
        if ((ws.jw[i] >> 32) == hv) {
            ws.jw[i] = (uint64_t)i;
            const unsigned long long r = atomicAdd((unsigned long long*)counts, 1ull);
            if ((int64_t)r < ring_cap) {
                ws.rkeys[r] = hv;
                ws.rvals[r] = (uint32_t)i;
            }
        } else {
            const uint32_t j = ws.nxt[i];
            ws.jw[i] = ((uint64_t)((ws.flags[j] & CORNER) ? 1 : 0) << 32) | j;
        }
    }
}

__global__ void __launch_bounds__(NT) region_keys_kernel(const int64_t* __restrict__ counts, Ws ws) {
    const int64_t n = counts[0];
    for (int64_t r = (int64_t)blockIdx.x * NT + threadIdx.x; r < n; r += (int64_t)gridDim.x * NT)
        ws.rkeys[r] = (uint64_t)(uint32_t)ws.reg[ws.rvals[r]];
}

// per ring in final order: region, corner count (corners over (j, start] plus j itself, j = the start's successor)
__global__ void __launch_bounds__(NT) ring_info_kernel(const int64_t* __restrict__ counts, int32_t* __restrict__ ring_region,
                                                       Ws ws) {
    const int64_t n = counts[0];
    for (int64_t r = (int64_t)blockIdx.x * NT + threadIdx.x; r < n; r += (int64_t)gridDim.x * NT) {
        const uint32_t s0 = ws.rvals[r], j = ws.nxt[s0];
        ring_region[r] = ws.reg[s0];
        ws.ccount[r] = (uint32_t)(ws.jw[j] >> 32) + ((ws.flags[j] & CORNER) ? 1u : 0u);
        ws.ring_of[s0] = (uint32_t)r;
    }
}

__global__ void __launch_bounds__(NT) vertex_kernel(const int64_t* __restrict__ counts, int64_t W, Ws ws,
                                                    int32_t* __restrict__ vertices, int64_t* __restrict__ ring_offsets,
                                                    int64_t* __restrict__ ring_area) {
    const int64_t n_rings = counts[0];
    const int64_t gtid = (int64_t)blockIdx.x * NT + threadIdx.x, gstride = (int64_t)gridDim.x * NT;
    for (int64_t r = gtid; r <= n_rings; r += gstride) ring_offsets[r] = r < n_rings ? (int64_t)ws.offs[r] : counts[1];
    if (failed(counts)) return;
    const int64_t n = counts[2];
    for (int64_t i = gtid; i < n; i += gstride) {
        const uint64_t w = ws.jw[i];
        const uint32_t s0 = (uint32_t)w, r = ws.ring_of[s0];
        const uint8_t f = ws.flags[i];
        const uint32_t hv = ws.hv[i];
        const int64_t hx = hv % (uint32_t)(W + 1), hy = hv / (uint32_t)(W + 1);
        if (f & CORNER) {
            const uint32_t rank = (uint32_t)i == s0 ? 0u : ws.ccount[r] - (uint32_t)(w >> 32);
            const int64_t pos = (int64_t)ws.offs[r] + rank;
            vertices[2 * pos] = (int32_t)hx;
            vertices[2 * pos + 1] = (int32_t)hy;
        }
        // shoelace area = sum of x dy: south sides (direction 1) add x, north sides (3) subtract it
        if ((f & 3) == 1) atomicAdd((unsigned long long*)(ring_area + r), (unsigned long long)hx);
        else if ((f & 3) == 3) atomicAdd((unsigned long long*)(ring_area + r), (unsigned long long)(-hx));
    }
}

int ceil_log2(int64_t x) {
    int b = 0;
    while (((int64_t)1 << b) < x) ++b;
    return b;
}

}  // namespace poly
}  // namespace dm

using namespace dm;

static bool poly_extent_ok(int64_t H, int64_t W) {
    return H >= 0 && W >= 0 && H < (1ll << 31) && W < (1ll << 31) && (H + 1) * (W + 1) <= (1ll << 32);
}

extern "C" size_t dm_polygonize_workspace_bytes(int64_t H, int64_t W, int64_t n_regions, int64_t capacity) {
    if (!poly_extent_ok(H, W) || n_regions < 0 || capacity < 0 || capacity >= (1ll << 31)) return 0;
    poly::Ws w;
    return poly::carve(w, nullptr, H, W, n_regions, capacity);
}

extern "C" int dm_polygonize(const int32_t* labels, int64_t H, int64_t W, int64_t ld, int64_t n_regions, int64_t capacity,
                             int32_t* ring_region, int64_t* ring_offsets, int64_t* ring_area, int32_t* vertices,
                             int64_t* region_rings, int64_t* counts, void* ws, size_t ws_bytes, dm_stream_t stream) {
    if (!poly_extent_ok(H, W) || ld < W || n_regions < 0 || n_regions >= (1ll << 31) || capacity < 0 ||
        capacity >= (1ll << 31))
        return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    if (H == 0 || W == 0) {
        if (counts) DM_CUDA(cudaMemsetAsync(counts, 0, 4 * sizeof(int64_t), s));
        if (ring_offsets) DM_CUDA(cudaMemsetAsync(ring_offsets, 0, sizeof(int64_t), s));
        if (region_rings) DM_CUDA(cudaMemsetAsync(region_rings, 0, (size_t)(n_regions + 1) * sizeof(int64_t), s));
        return DM_OK;
    }
    if (!labels || !ring_offsets || !region_rings || !counts || !ws || (capacity > 0 && !vertices) ||
        (capacity >= 4 && (!ring_region || !ring_area)))
        return DM_ERR_BAD_ARG;
    if (ws_bytes < dm_polygonize_workspace_bytes(H, W, n_regions, capacity)) return DM_ERR_WORKSPACE;
    poly::Ws w;
    poly::carve(w, ws, H, W, n_regions, capacity);
    const int64_t wpr = ceil_div(W, 32), n_words = H * wpr, ring_cap = capacity / 4;
    DM_CUDA(cudaMemsetAsync(counts, 0, 4 * sizeof(int64_t), s));
    DM_CUDA(cudaMemsetAsync(w.changed, 0, 2 * poly::MAX_PASSES * sizeof(int), s));
    if (ring_cap) DM_CUDA(cudaMemsetAsync(ring_area, 0, (size_t)ring_cap * sizeof(int64_t), s));
    const unsigned g_words = grid_for(n_words * 32, poly::NT, 16), g_sides = grid_for(capacity, poly::NT, 16);
    const unsigned g_rings = grid_for(ring_cap + 1, poly::NT, 16);
    DM_TRY(launch(poly::mask_kernel, g_words, poly::NT, 0, s, labels, H, W, ld, wpr, n_regions, w.masks, w.wcnt, counts,
        w.n_words_dev));
    DM_TRY(prims::scan_exclusive_u32(w.wcnt, w.wbase, w.n_words_dev, n_words, nullptr, w.scan, s));
    DM_TRY(launch(poly::emit_kernel, g_words, poly::NT, 0, s, labels, H, W, ld, wpr, capacity, w.masks, w.wbase, counts, w));
    const int passes = poly::ceil_log2(capacity) + 1;
    for (int phase = 0; phase < 2; ++phase) {
        for (int k = 0; k < passes; ++k) {
            DM_TRY(launch(poly::jump_kernel, g_sides, poly::NT, 0, s, w.jw, counts, w.changed, phase, k));
        }
        if (phase == 0) {
            DM_TRY(launch(poly::starts_kernel, g_sides, poly::NT, 0, s, counts, ring_cap, w));
        }
    }
    // rings in raster order of their start vertex, then stably by region
    DM_TRY(prims::sort_pairs(w.rkeys, w.rvals, counts, ring_cap, bits_for((H + 1) * (W + 1)), bits_for((H + 1) * (W + 1)),
                             w.sort, s));
    DM_TRY(launch(poly::region_keys_kernel, g_rings, poly::NT, 0, s, counts, w));
    const int rb = bits_for(n_regions + 1);
    DM_TRY(prims::sort_pairs(w.rkeys, w.rvals, counts, ring_cap, rb, rb, w.sort, s, n_regions + 1, region_rings, nullptr));
    if (ring_cap == 0) DM_CUDA(cudaMemsetAsync(region_rings, 0, (size_t)(n_regions + 1) * sizeof(int64_t), s));
    DM_TRY(launch(poly::ring_info_kernel, g_rings, poly::NT, 0, s, counts, ring_region, w));
    DM_TRY(prims::scan_exclusive_u32(w.ccount, w.offs, counts, ring_cap, counts + 1, w.scan, s));
    return launch(poly::vertex_kernel, imax64(g_sides, g_rings), poly::NT, 0, s, counts, W, w, vertices, ring_offsets,
        ring_area);
}
