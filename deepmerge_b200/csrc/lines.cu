// Boundary-line tracer: label raster -> one polyline per maximal chain of boundary segments between nodes, with the
// values on its left and right (dm_lines in include/deepmerge_b200.h).  The per-vertex arithmetic lives in
// lines_core.cuh.  Steps 1 to 5 are the kernels and the launch sequence (chain::trace) of chain.cuh, shared with the
// polygonizer (polygon.cu); SegmentRule is their per-segment part.
//
// 1. mask_kernel    one pass over the labels: a 4-bit mask of the segments each pixel owns, counts per word, the
//                   label range check.
// 2. scan           word counts -> word bases: every segment has a dense index.
// 3. emit_kernel    per segment: orientation, head vertex, flags (direction, emits a vertex, head / tail is a node)
//                   and the dense index of its successor at the head; a segment whose head is a node points at itself.
// 4. jump_kernel    phase 0: the minimum over the rest of the chain of key(head vertex), with 0 at every segment
//                   that ends at a node, so that open lines reach 0 and every cycle its smallest vertex.
// 5. starts_kernel  one line per segment whose tail is a node, and one per cycle, starting after the segment whose
//                   head is the cycle's smallest vertex; that segment and every one ending at a node end their chain.
//    jump_kernel    phase 1: the number of vertex-emitting segments after each segment up to the end of its line.
// 6. sort_pairs     lines by (start vertex, first direction) (radix); info_kernel: per line its values, vertex count
//                   and the line of its end segment; scan -> vertex offsets.
// 7. vertex_kernel  start vertices and emitted head vertices scattered to line offset + rank, lengths counted.
// dm_lines_simplified writes the vertices of step 7 to its workspace and simplifies them (simplify.cuh) into the output.
#include <cmath>

#include "chain.cuh"
#include "lines_core.cuh"
#include "prims.cuh"
#include "simplify.cuh"

namespace dm {
namespace lines {
using namespace linecore;
using namespace chain;

// flags: bits 0-1 direction, then:
constexpr uint8_t EMIT = 4;        // the head vertex is a vertex of the line (a corner or the line's end)
constexpr uint8_t NODE_HEAD = 8;
constexpr uint8_t NODE_TAIL = 16;

struct Ws : Front {
    uint32_t* line_of;                  // per segment: line ended by the segment
    uint64_t* lkeys;                    // per line: start vertex << 32 | direction of the first segment
    uint32_t *lvals, *vcount, *offs;    // per line: first segment, vertices, vertex offset
    void* sort;
};

void take(Ws& w, Carver& c, int64_t H, int64_t W, int64_t cap) {
    carve_front(w, c, H, W, cap, cap);
    w.line_of = c.take<uint32_t>((size_t)cap);
    w.lkeys = c.take<uint64_t>((size_t)cap);
    w.lvals = c.take<uint32_t>((size_t)cap);
    w.vcount = c.take<uint32_t>((size_t)cap);
    w.offs = c.take<uint32_t>((size_t)cap);
    w.sort = c.take<char>(prims::ws_bytes(cap, false));
}

size_t carve(Ws& w, void* base, int64_t H, int64_t W, int64_t cap) {
    Carver c(base);
    take(w, c, H, W, cap);
    return c.used();
}

// dm_lines_simplified: the tracer's workspace, then the simplifier's with the unsimplified lines (2 cap vertices).
size_t carve_simplified(Ws& w, simplify::Ws& sw, void* base, int64_t H, int64_t W, int64_t cap) {
    Carver c(base);
    take(w, c, H, W, cap);
    simplify::carve(sw, c, 2 * cap, cap, false);
    return c.used();
}

// Phase-0 key of a head vertex: 1 + its index, 0 is kept for the ends of open lines.  The clamp can only merge the
// last two vertices of the last vertex row (when (H + 1) (W + 1) = 2^32), and no cycle has its smallest vertex there.
__device__ __forceinline__ uint64_t vertex_key(uint32_t hv) { return hv == 0xffffffffu ? hv : (uint64_t)hv + 1; }

struct SegmentRule {
    using Ws = lines::Ws;

    static __device__ __forceinline__ unsigned mask(const int32_t* L, int64_t H, int64_t W, int64_t ld, int64_t x, int64_t y) {
        return owned_mask(L, H, W, ld, x, y);
    }

    // segment b of pixel (x, y): orientation, head vertex, flags and the dense index of its successor at the head; a
    // segment whose head is a node points at itself
    static __device__ __forceinline__ void emit(const int32_t* L, int64_t H, int64_t W, int64_t ld, int64_t wpr,
                                                const uint32_t* masks, const uint32_t* wbase, int64_t x, int64_t y,
                                                int b, uint32_t i, const Ws& ws) {
        const Seg s = orient(L, H, W, ld, x, y, b);
        const int64_t hx = s.x + step_x(s.d), hy = s.y + step_y(s.d);
        const Next q = next_at(L, H, W, ld, hx, hy, s.d);
        uint32_t j = i;
        if (!q.node) {
            const Owner o = owner_of(H, W, hx, hy, q.d);
            j = dense_index(masks, wbase, wpr, o.x, o.y, o.b);
        }
        const uint32_t hv = (uint32_t)(hy * (W + 1) + hx);
        uint8_t f = (uint8_t)s.d;
        if (q.node || q.d != s.d) f |= EMIT;
        if (q.node) f |= NODE_HEAD;
        if (node_arms(arms(L, H, W, ld, s.x, s.y))) f |= NODE_TAIL;
        ws.hv[i] = hv;
        ws.nxt[i] = j;
        ws.flags[i] = f;
        ws.jw[i] = ((q.node ? 0 : vertex_key(hv)) << 32) | j;
    }

    // list the line segment i starts, if any, and turn its word into phase 1's
    static __device__ __forceinline__ void start(int64_t* counts, int64_t W, int64_t cap, const Ws& ws, int64_t i) {
        const uint32_t hv = ws.hv[i], j = ws.nxt[i];
        const uint8_t f = ws.flags[i];
        const bool anchor = (ws.jw[i] >> 32) == vertex_key(hv);   // its head is its cycle's smallest vertex
        if (anchor || (f & NODE_TAIL)) {
            uint64_t key;
            uint32_t first;
            if (anchor) {
                key = ((uint64_t)hv << 32) | (ws.flags[j] & 3u);
                first = j;
            } else {
                const int d = f & 3;
                const int64_t hx = hv % (uint32_t)(W + 1), hy = hv / (uint32_t)(W + 1);
                key = ((uint64_t)((hy - step_y(d)) * (W + 1) + hx - step_x(d)) << 32) | (uint32_t)d;
                first = (uint32_t)i;
            }
            const unsigned long long r = atomicAdd((unsigned long long*)counts, 1ull);
            if ((int64_t)r < cap) {
                ws.lkeys[r] = key;
                ws.lvals[r] = first;
            }
        }
        ws.jw[i] = anchor || (f & NODE_HEAD) ? (uint64_t)i : ((uint64_t)((ws.flags[j] & EMIT) ? 1 : 0) << 32) | j;
    }
};

// per line in final order: values, length cleared, vertex count (start + emitting segments from the first to the end)
__global__ void __launch_bounds__(NT) info_kernel(const int32_t* __restrict__ L, int64_t H, int64_t W, int64_t ld,
                                                  const int64_t* __restrict__ counts, int32_t* __restrict__ line_left,
                                                  int32_t* __restrict__ line_right, int64_t* __restrict__ line_length,
                                                  Ws ws) {
    const int64_t n = counts[0];
    for (int64_t r = (int64_t)blockIdx.x * NT + threadIdx.x; r < n; r += (int64_t)gridDim.x * NT) {
        const uint32_t f = ws.lvals[r];
        const uint64_t w = ws.jw[f];
        const uint64_t k = ws.lkeys[r];
        const uint32_t sv = (uint32_t)(k >> 32);
        const Seg s = {(int64_t)(sv % (uint32_t)(W + 1)), (int64_t)(sv / (uint32_t)(W + 1)), (int)(k & 3u)};
        line_left[r] = left_value(L, H, W, ld, s);
        line_right[r] = right_value(L, H, W, ld, s);
        line_length[r] = 0;
        ws.line_of[(uint32_t)w] = (uint32_t)r;
        ws.vcount[r] = 1u + (uint32_t)(w >> 32) + ((ws.flags[f] & EMIT) ? 1u : 0u);
    }
}

__global__ void __launch_bounds__(NT) vertex_kernel(const int64_t* __restrict__ counts, int64_t W, Ws ws,
                                                    int32_t* __restrict__ vertices, int64_t* __restrict__ line_offsets,
                                                    int64_t* __restrict__ line_length) {
    const int64_t n_lines = counts[0];
    const int64_t gtid = (int64_t)blockIdx.x * NT + threadIdx.x, gstride = (int64_t)gridDim.x * NT;
    for (int64_t r = gtid; r <= n_lines; r += gstride) {
        line_offsets[r] = r < n_lines ? (int64_t)ws.offs[r] : counts[1];
        if (r < n_lines) {
            const uint32_t sv = (uint32_t)(ws.lkeys[r] >> 32);
            vertices[2 * ws.offs[r]] = (int32_t)(sv % (uint32_t)(W + 1));
            vertices[2 * ws.offs[r] + 1] = (int32_t)(sv / (uint32_t)(W + 1));
        }
    }
    if (failed(counts)) return;
    const int64_t n = counts[2];
    for (int64_t i = gtid; i < n; i += gstride) {
        const uint64_t w = ws.jw[i];
        const uint32_t r = ws.line_of[(uint32_t)w];
        if (ws.flags[i] & EMIT) {
            const int64_t pos = (int64_t)ws.offs[r] + ws.vcount[r] - 1u - (uint32_t)(w >> 32);
            const uint32_t hv = ws.hv[i];
            vertices[2 * pos] = (int32_t)(hv % (uint32_t)(W + 1));
            vertices[2 * pos + 1] = (int32_t)(hv / (uint32_t)(W + 1));
        }
        // segments of a line often sit side by side in raster order: one atomic per line and warp
        const unsigned peers = __match_any_sync(__activemask(), r);
        if ((threadIdx.x & 31) == __ffs(peers) - 1)
            atomicAdd((unsigned long long*)(line_length + r), (unsigned long long)__popc(peers));
    }
}

}  // namespace lines
}  // namespace dm

using namespace dm;

extern "C" size_t dm_lines_workspace_bytes(int64_t H, int64_t W, int64_t capacity) {
    if (!chain::extent_ok(H, W, capacity)) return 0;
    lines::Ws w;
    return lines::carve(w, nullptr, H, W, capacity);
}

namespace dm {
namespace lines {

// The back half of both entry points after the trace: the lines' sort, info and vertices.
int finish(const int32_t* labels, int64_t H, int64_t W, int64_t ld, int64_t capacity, int32_t* line_left,
           int32_t* line_right, int64_t* line_length, int64_t* line_offsets, int32_t* vertices, int64_t* counts,
           Ws& w, cudaStream_t s) {
    const unsigned g_lines = grid_for(capacity + 1, chain::NT, 16);
    // lines by start vertex (high half), then by the direction of their first segment (low half)
    const int vb = bits_for((H + 1) * (W + 1));
    DM_TRY(prims::sort_pairs(w.lkeys, w.lvals, counts, capacity, vb, 2 * vb, w.sort, s));
    DM_TRY(launch(lines::info_kernel, g_lines, chain::NT, 0, s, labels, H, W, ld, counts, line_left, line_right,
                  line_length, w));
    DM_TRY(prims::scan_exclusive_u32(w.vcount, w.offs, counts, capacity, counts + 1, w.scan, s));
    return launch(lines::vertex_kernel, g_lines, chain::NT, 0, s, counts, W, w, vertices, line_offsets, line_length);
}

}  // namespace lines
}  // namespace dm

extern "C" int dm_lines(const int32_t* labels, int64_t H, int64_t W, int64_t ld, int64_t n_regions, int64_t capacity,
                        int32_t* line_left, int32_t* line_right, int64_t* line_length, int64_t* line_offsets,
                        int32_t* vertices, int64_t* counts, void* ws, size_t ws_bytes, dm_stream_t stream) {
    if (!chain::args_ok(H, W, ld, n_regions, capacity)) return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    if (H == 0 || W == 0) return chain::clear_empty(counts, line_offsets, s);
    if (!labels || !line_offsets || !counts || !ws ||
        (capacity > 0 && (!line_left || !line_right || !line_length || !vertices)))
        return DM_ERR_BAD_ARG;
    if (ws_bytes < dm_lines_workspace_bytes(H, W, capacity)) return DM_ERR_WORKSPACE;
    lines::Ws w;
    lines::carve(w, ws, H, W, capacity);
    DM_TRY(chain::trace<lines::SegmentRule>(labels, H, W, ld, n_regions, capacity, counts, w, s));
    return lines::finish(labels, H, W, ld, capacity, line_left, line_right, line_length, line_offsets, vertices, counts,
                         w, s);
}

extern "C" size_t dm_lines_simplified_workspace_bytes(int64_t H, int64_t W, int64_t capacity) {
    if (!chain::extent_ok(H, W, capacity) || !simplify::extent_ok(H, W)) return 0;
    lines::Ws w;
    simplify::Ws sw;
    return lines::carve_simplified(w, sw, nullptr, H, W, capacity);
}

extern "C" int dm_lines_simplified(const int32_t* labels, int64_t H, int64_t W, int64_t ld, int64_t n_regions,
                                   int64_t capacity, double tolerance, int32_t* line_left, int32_t* line_right,
                                   int64_t* line_length, int64_t* line_offsets, int32_t* vertices, int64_t* counts,
                                   void* ws, size_t ws_bytes, dm_stream_t stream) {
    if (!chain::args_ok(H, W, ld, n_regions, capacity) || !simplify::extent_ok(H, W) || !std::isfinite(tolerance) ||
        tolerance < 0)
        return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    if (H == 0 || W == 0) return chain::clear_empty(counts, line_offsets, s);
    if (!labels || !line_offsets || !counts || !ws ||
        (capacity > 0 && (!line_left || !line_right || !line_length || !vertices)))
        return DM_ERR_BAD_ARG;
    if (ws_bytes < dm_lines_simplified_workspace_bytes(H, W, capacity)) return DM_ERR_WORKSPACE;
    lines::Ws w;
    simplify::Ws sw;
    lines::carve_simplified(w, sw, ws, H, W, capacity);
    DM_TRY(chain::trace<lines::SegmentRule>(labels, H, W, ld, n_regions, capacity, counts, w, s));
    DM_TRY(lines::finish(labels, H, W, ld, capacity, line_left, line_right, line_length, sw.in.off, sw.in.v, counts, w,
                         s));
    return simplify::run(counts, H, W, simpcore::quantize_tolerance(tolerance, H, W), 2 * capacity, capacity, sw,
                         vertices, line_offsets, s);
}
