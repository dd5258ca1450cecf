// Polygonizer: label raster -> closed rings of pixel-corner vertices, one set per region (dm_polygonize in
// include/deepmerge_b200.h).  The per-side arithmetic lives in polygon_core.cuh.  Steps 1 to 5 are the kernels and the
// launch sequence (chain::trace) of chain.cuh, shared with the boundary-line tracer (lines.cu); SideRule is their
// per-side part.
//
// 1. mask_kernel    one pass over the labels: a 4-bit mask of boundary sides per pixel (8 pixels per uint32), one side
//                   count per 32-pixel word of a row, the exact total and the label range check.
// 2. scan           word counts -> word bases: every side has a dense index.
// 3. emit_kernel    per side: head vertex, region, corner flag and the dense index of its successor (no search).
// 4. jump_kernel    pointer jumping over the successor cycles: first the minimum head vertex of every ring (its
//                   canonical start), then, with every cycle cut at its start, the number of corners from each side to
//                   the start.
// 5. starts_kernel  one ring per start side, listed with its start vertex; sort_pairs orders the list by start vertex
//                   (radix), then stably by region (bucket + rank), whose CSR offsets are region_rings.
// 6. vertex_kernel  corners scattered to ring offset + rank, ring areas as the sum of x * dy over the vertical sides.
// dm_polygonize_simplified traces with NodeSideRule, which also emits (and flags) the head vertices that are nodes in
// the sense of dm_lines, writes the rings of step 6 to its workspace and simplifies them (simplify.cuh) into the output.
#include <cmath>
#include <type_traits>

#include "chain.cuh"
#include "lines_core.cuh"
#include "polygon_core.cuh"
#include "prims.cuh"
#include "simplify.cuh"

namespace dm {
namespace poly {
using namespace polycore;
using namespace chain;

constexpr uint8_t CORNER = 4;   // flags: bits 0-1 side / direction, bit 2 head vertex is a vertex of the ring
constexpr uint8_t NODE = 8;     // NodeSideRule: the head vertex is a node

struct Ws : Front {
    uint32_t* ring_of;                  // per side: ring of a start side
    int32_t* reg;
    uint64_t* rkeys;                    // per ring
    uint32_t *rvals, *ccount, *offs;
    void* sort;
};

void take(Ws& w, Carver& c, int64_t H, int64_t W, int64_t n_regions, int64_t cap) {
    const int64_t ring_cap = cap / 4;
    carve_front(w, c, H, W, cap, ring_cap);
    w.ring_of = c.take<uint32_t>((size_t)cap);
    w.reg = c.take<int32_t>((size_t)cap);
    w.rkeys = c.take<uint64_t>((size_t)ring_cap);
    w.rvals = c.take<uint32_t>((size_t)ring_cap);
    w.ccount = c.take<uint32_t>((size_t)ring_cap);
    w.offs = c.take<uint32_t>((size_t)ring_cap);
    w.sort = c.take<char>(prims::ws_bytes(ring_cap, false, n_regions + 1));
}

size_t carve(Ws& w, void* base, int64_t H, int64_t W, int64_t n_regions, int64_t cap) {
    Carver c(base);
    take(w, c, H, W, n_regions, cap);
    return c.used();
}

// dm_polygonize_simplified: the tracer's workspace, then the simplifier's with the unsimplified rings (cap vertices).
size_t carve_simplified(Ws& w, simplify::Ws& sw, void* base, int64_t H, int64_t W, int64_t n_regions, int64_t cap) {
    Carver c(base);
    take(w, c, H, W, n_regions, cap);
    simplify::carve(sw, c, cap, cap / 4, true);
    return c.used();
}

struct SideRule {
    using Ws = poly::Ws;

    static __device__ __forceinline__ unsigned mask(const int32_t* L, int64_t H, int64_t W, int64_t ld, int64_t x, int64_t y) {
        return side_mask(L, H, W, ld, x, y);
    }

    // side s of pixel (x, y): head vertex, region, corner flag and the dense index of its successor (no search)
    static __device__ __forceinline__ void emit(const int32_t* L, int64_t H, int64_t W, int64_t ld, int64_t wpr,
                                                const uint32_t* masks, const uint32_t* wbase, int64_t x, int64_t y,
                                                int s, uint32_t i, const Ws& ws) {
        const Succ q = successor(L, H, W, ld, x, y, s);
        const uint32_t j = dense_index(masks, wbase, wpr, q.x, q.y, q.s);
        const uint32_t hv = (uint32_t)(head_y(y, s) * (W + 1) + head_x(x, s));
        ws.hv[i] = hv;
        ws.nxt[i] = j;
        ws.reg[i] = L[y * ld + x];
        ws.flags[i] = (uint8_t)(s | (q.corner ? CORNER : 0));
        ws.jw[i] = ((uint64_t)hv << 32) | j;   // phase 0: minimum head vertex over [i, pointer) = own head
    }

    // the side whose head is its ring's minimum vertex starts the ring; one ring per 4 sides at most
    static __device__ __forceinline__ void start(int64_t* counts, int64_t W, int64_t cap, const Ws& ws, int64_t i) {
        const uint32_t hv = ws.hv[i];
        if ((ws.jw[i] >> 32) == hv) {
            ws.jw[i] = (uint64_t)i;
            const unsigned long long r = atomicAdd((unsigned long long*)counts, 1ull);
            if ((int64_t)r < cap / 4) {
                ws.rkeys[r] = hv;
                ws.rvals[r] = (uint32_t)i;
            }
        } else {
            const uint32_t j = ws.nxt[i];
            ws.jw[i] = ((uint64_t)((ws.flags[j] & CORNER) ? 1 : 0) << 32) | j;
        }
    }
};

// SideRule with every head vertex that is a node (linecore::node_arms) made a ring vertex and flagged NODE.
struct NodeSideRule : SideRule {
    static __device__ __forceinline__ void emit(const int32_t* L, int64_t H, int64_t W, int64_t ld, int64_t wpr,
                                                const uint32_t* masks, const uint32_t* wbase, int64_t x, int64_t y,
                                                int s, uint32_t i, const Ws& ws) {
        SideRule::emit(L, H, W, ld, wpr, masks, wbase, x, y, s, i, ws);
        if (linecore::node_arms(linecore::arms(L, H, W, ld, head_x(x, s), head_y(y, s)))) ws.flags[i] |= CORNER | NODE;
    }
};

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

// node (NodeSideRule only): per vertex, whether it is a node
template <bool Nodes>
__global__ void __launch_bounds__(NT) vertex_kernel(const int64_t* __restrict__ counts, int64_t W, Ws ws,
                                                    int32_t* __restrict__ vertices, int64_t* __restrict__ ring_offsets,
                                                    int64_t* __restrict__ ring_area, uint8_t* __restrict__ node) {
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
            if (Nodes) node[pos] = (f & NODE) ? 1 : 0;
        }
        // shoelace area = sum of x dy: south sides (direction 1) add x, north sides (3) subtract it
        if ((f & 3) == 1) atomicAdd((unsigned long long*)(ring_area + r), (unsigned long long)hx);
        else if ((f & 3) == 3) atomicAdd((unsigned long long*)(ring_area + r), (unsigned long long)(-hx));
    }
}

// The whole tracer on workspace w, with rule SideRule or NodeSideRule; node receives NodeSideRule's node flags.
template <class Rule>
int polygonize(const int32_t* labels, int64_t H, int64_t W, int64_t ld, int64_t n_regions, int64_t capacity,
               int32_t* ring_region, int64_t* ring_offsets, int64_t* ring_area, int32_t* vertices,
               int64_t* region_rings, int64_t* counts, uint8_t* node, Ws& w, cudaStream_t s) {
    const int64_t ring_cap = capacity / 4;
    if (ring_cap) DM_CUDA(cudaMemsetAsync(ring_area, 0, (size_t)ring_cap * sizeof(int64_t), s));
    DM_TRY(chain::trace<Rule>(labels, H, W, ld, n_regions, capacity, counts, w, s));
    const unsigned g_sides = grid_for(capacity, poly::NT, 16), g_rings = grid_for(ring_cap + 1, poly::NT, 16);
    // rings in raster order of their start vertex, then stably by region
    DM_TRY(prims::sort_pairs(w.rkeys, w.rvals, counts, ring_cap, bits_for((H + 1) * (W + 1)), bits_for((H + 1) * (W + 1)),
                             w.sort, s));
    DM_TRY(launch(poly::region_keys_kernel, g_rings, poly::NT, 0, s, counts, w));
    const int rb = bits_for(n_regions + 1);
    DM_TRY(prims::sort_pairs(w.rkeys, w.rvals, counts, ring_cap, rb, rb, w.sort, s, n_regions + 1, region_rings, nullptr));
    if (ring_cap == 0) DM_CUDA(cudaMemsetAsync(region_rings, 0, (size_t)(n_regions + 1) * sizeof(int64_t), s));
    DM_TRY(launch(poly::ring_info_kernel, g_rings, poly::NT, 0, s, counts, ring_region, w));
    DM_TRY(prims::scan_exclusive_u32(w.ccount, w.offs, counts, ring_cap, counts + 1, w.scan, s));
    return launch(vertex_kernel<std::is_same<Rule, NodeSideRule>::value>, imax64(g_sides, g_rings), NT, 0, s, counts, W,
                  w, vertices, ring_offsets, ring_area, node);
}

}  // namespace poly
}  // namespace dm

using namespace dm;

extern "C" size_t dm_polygonize_workspace_bytes(int64_t H, int64_t W, int64_t n_regions, int64_t capacity) {
    if (!chain::extent_ok(H, W, capacity) || n_regions < 0) return 0;
    poly::Ws w;
    return poly::carve(w, nullptr, H, W, n_regions, capacity);
}

extern "C" int dm_polygonize(const int32_t* labels, int64_t H, int64_t W, int64_t ld, int64_t n_regions, int64_t capacity,
                             int32_t* ring_region, int64_t* ring_offsets, int64_t* ring_area, int32_t* vertices,
                             int64_t* region_rings, int64_t* counts, void* ws, size_t ws_bytes, dm_stream_t stream) {
    if (!chain::args_ok(H, W, ld, n_regions, capacity)) return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    if (H == 0 || W == 0) {
        DM_TRY(chain::clear_empty(counts, ring_offsets, s));
        if (region_rings) DM_CUDA(cudaMemsetAsync(region_rings, 0, (size_t)(n_regions + 1) * sizeof(int64_t), s));
        return DM_OK;
    }
    if (!labels || !ring_offsets || !region_rings || !counts || !ws || (capacity > 0 && !vertices) ||
        (capacity >= 4 && (!ring_region || !ring_area)))
        return DM_ERR_BAD_ARG;
    if (ws_bytes < dm_polygonize_workspace_bytes(H, W, n_regions, capacity)) return DM_ERR_WORKSPACE;
    poly::Ws w;
    poly::carve(w, ws, H, W, n_regions, capacity);
    return poly::polygonize<poly::SideRule>(labels, H, W, ld, n_regions, capacity, ring_region, ring_offsets, ring_area,
                                            vertices, region_rings, counts, nullptr, w, s);
}

extern "C" size_t dm_polygonize_simplified_workspace_bytes(int64_t H, int64_t W, int64_t n_regions, int64_t capacity) {
    if (!chain::extent_ok(H, W, capacity) || !simplify::extent_ok(H, W) || n_regions < 0) return 0;
    poly::Ws w;
    simplify::Ws sw;
    return poly::carve_simplified(w, sw, nullptr, H, W, n_regions, capacity);
}

extern "C" int dm_polygonize_simplified(const int32_t* labels, int64_t H, int64_t W, int64_t ld, int64_t n_regions,
                                        int64_t capacity, double tolerance, int32_t* ring_region, int64_t* ring_offsets,
                                        int64_t* ring_area, int32_t* vertices, int64_t* region_rings, int64_t* counts,
                                        void* ws, size_t ws_bytes, dm_stream_t stream) {
    if (!chain::args_ok(H, W, ld, n_regions, capacity) || !simplify::extent_ok(H, W) || !std::isfinite(tolerance) ||
        tolerance < 0)
        return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    if (H == 0 || W == 0) {
        DM_TRY(chain::clear_empty(counts, ring_offsets, s));
        if (region_rings) DM_CUDA(cudaMemsetAsync(region_rings, 0, (size_t)(n_regions + 1) * sizeof(int64_t), s));
        return DM_OK;
    }
    if (!labels || !ring_offsets || !region_rings || !counts || !ws || (capacity > 0 && !vertices) ||
        (capacity >= 4 && (!ring_region || !ring_area)))
        return DM_ERR_BAD_ARG;
    if (ws_bytes < dm_polygonize_simplified_workspace_bytes(H, W, n_regions, capacity)) return DM_ERR_WORKSPACE;
    poly::Ws w;
    simplify::Ws sw;
    poly::carve_simplified(w, sw, ws, H, W, n_regions, capacity);
    DM_TRY(poly::polygonize<poly::NodeSideRule>(labels, H, W, ld, n_regions, capacity, ring_region, sw.in.off,
                                                ring_area, sw.in.v, region_rings, counts, sw.in.node, w, s));
    return simplify::run(counts, H, W, simpcore::quantize_tolerance(tolerance, H, W), capacity, capacity / 4, sw,
                         vertices, ring_offsets, s);
}
