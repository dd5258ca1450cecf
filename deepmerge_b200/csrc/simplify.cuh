// Douglas-Peucker simplification of boundary chains, shared by dm_polygonize_simplified (polygon.cu) and
// dm_lines_simplified (lines.cu).  The contract is in include/deepmerge_b200.h, the exact arithmetic in simplify_core.cuh.
//
// Input: chains as offsets into pixel-corner vertices, counts[0] chains and counts[1] vertices on the device.  Lines are
// open lists whose ends are anchors (a closed line repeats its start); rings are cyclic lists whose anchors are the
// vertices flagged as nodes, or the start of a ring without one.  Vertices on the image border are anchors in both.
//
// 1. anchors_kernel  one warp per chain: keep = anchor, and one piece per pair of consecutive anchors with a vertex
//                    between them (a ring with one anchor is one piece from it back to itself).
// 2. dp_kernel       one warp per piece, depth first with an explicit stack in per-vertex workspace (the pending
//                    intervals of a piece are disjoint, each holds an interior vertex, so a piece of n segments never
//                    has more than n / 2 of them): the top vertex of the piece (and, when its ends coincide, of both
//                    halves) is kept, then every interval keeps its top vertex when it lies farther than t and splits.
// 3. scan            keep -> output positions; counts[1] = kept vertices.
// 4. compact_kernel  kept vertices to their positions, chain offsets.
// The launch sequence is fixed and nothing is read back: the element counts come from the device.
#pragma once
#include "chain.cuh"
#include "prims.cuh"
#include "simplify_core.cuh"

namespace dm {
namespace simplify {
using namespace simpcore;

constexpr int NT = 256;

// The vertices before simplification: chain c has vertices [off[c], off[c + 1]); rings flag their nodes in `node`.
struct Chains {
    int32_t* v;             // [vcap, 2]
    int64_t* off;           // [chain_cap + 1]
    uint8_t* node;          // [vcap] for rings, null for lines
};

struct Ws {
    Chains in;
    uint32_t *keep, *rank;  // per vertex
    uint64_t* stack;        // per vertex: pending intervals of the piece that owns the slot
    uint4* pieces;          // first vertex of the chain, chain length, first position, segments
    int64_t *n_pieces, *n_vertices;
    void* scan;
};

inline void carve(Ws& w, Carver& c, int64_t vcap, int64_t chain_cap, bool rings) {
    w.in.v = c.take<int32_t>((size_t)vcap * 2);
    w.in.off = c.take<int64_t>((size_t)chain_cap + 1);
    w.in.node = rings ? c.take<uint8_t>((size_t)vcap) : nullptr;
    w.keep = c.take<uint32_t>((size_t)vcap);
    w.rank = c.take<uint32_t>((size_t)vcap);
    w.stack = c.take<uint64_t>((size_t)vcap);
    w.pieces = c.take<uint4>((size_t)vcap);
    w.n_pieces = c.take<int64_t>(1);
    w.n_vertices = c.take<int64_t>(1);
    w.scan = c.take<char>(prims::scan_ws_bytes(vcap));
}

// Extents whose distances the exact comparison covers.
inline bool extent_ok(int64_t H, int64_t W) { return H < MAX_EXTENT && W < MAX_EXTENT; }

__device__ __forceinline__ bool on_border(int64_t x, int64_t y, int64_t H, int64_t W) {
    return x == 0 || y == 0 || x == W || y == H;
}

// pieces from anchor a to anchor b of the chain at s0 with len vertices, for the lanes with want set
__device__ __forceinline__ void emit_piece(bool want, uint32_t s0, uint32_t len, int64_t a, int64_t b, const Ws& w) {
    const unsigned m = __ballot_sync(0xffffffffu, want);
    if (!m) return;
    unsigned long long base = 0;
    if (lane_id() == 0) base = atomicAdd((unsigned long long*)w.n_pieces, (unsigned long long)__popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (want) w.pieces[base + __popc(m & lanemask_lt())] = make_uint4(s0, len, (uint32_t)a, (uint32_t)(b - a));
}

static __global__ void __launch_bounds__(NT) anchors_kernel(const int64_t* __restrict__ counts, int64_t H, int64_t W,
                                                            Ws w) {
    const bool cyclic = w.in.node != nullptr;
    const bool bad = chain::failed(counts);
    if (blockIdx.x == 0 && threadIdx.x == 0) *w.n_vertices = bad ? 0 : counts[1];
    if (bad) return;
    const int lane = threadIdx.x & 31;
    const int64_t n = counts[0];
    const int64_t warp0 = ((int64_t)blockIdx.x * NT + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * NT) >> 5;
    for (int64_t c = warp0; c < n; c += nwarps) {
        const int64_t s0 = w.in.off[c], len = w.in.off[c + 1] - s0;
        bool has_node = false;
        if (cyclic)
            for (int64_t j0 = 0; j0 < len && !has_node; j0 += 32)
                has_node = __any_sync(0xffffffffu, j0 + lane < len && w.in.node[s0 + j0 + lane]);
        int64_t first = -1, prev = -1;
        for (int64_t j0 = 0; j0 < len; j0 += 32) {
            const int64_t j = j0 + lane;
            bool a = false;
            if (j < len) {
                const int64_t x = w.in.v[2 * (s0 + j)], y = w.in.v[2 * (s0 + j) + 1];
                a = on_border(x, y, H, W) || (cyclic ? (w.in.node[s0 + j] || (!has_node && j == 0)) : (j == 0 || j == len - 1));
                w.keep[s0 + j] = a;
            }
            const unsigned m = __ballot_sync(0xffffffffu, a);
            const unsigned below = m & lanemask_lt();
            const int64_t pred = below ? j0 + 31 - __clz(below) : prev;
            emit_piece(a && pred >= 0 && j - pred >= 2, (uint32_t)s0, (uint32_t)len, pred, j, w);
            if (m) {
                if (first < 0) first = j0 + __ffs(m) - 1;
                prev = j0 + 31 - __clz(m);
            }
        }
        if (cyclic) emit_piece(lane == 0 && first + len - prev >= 2, (uint32_t)s0, (uint32_t)len, prev, first + len, w);
    }
}

// One warp: the top vertex of the interval [lo, hi] (hi - lo >= 2 segments) of a piece -> its position, num and the
// interval's den.
struct Top {
    int64_t k;
    u128 num, den;
};

__device__ __forceinline__ Top top_of(const Ws& w, int64_t W, uint4 pc, int64_t lo, int64_t hi) {
    auto at = [&](int64_t k) -> int64_t {
        int64_t j = (int64_t)pc.z + k;
        if (j >= (int64_t)pc.y) j -= pc.y;
        return (int64_t)pc.x + j;
    };
    const int2 A = *(const int2*)(w.in.v + 2 * at(lo)), B = *(const int2*)(w.in.v + 2 * at(hi));
    Cand best = {0, ~0ull, ~0ull};
    int64_t bk = -1;
    for (int64_t k = lo + 1 + lane_id(); k < hi; k += 32) {
        const int2 P = *(const int2*)(w.in.v + 2 * at(k));
        const Cand c = {seg_num(A.x, A.y, B.x, B.y, P.x, P.y), mid_rank(k - lo, hi - lo),
                        (uint64_t)P.y * (uint64_t)(W + 1) + (uint64_t)P.x};
        if (above(c, best)) {
            best = c;
            bk = k;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        Cand t;
        const uint64_t nh = __shfl_xor_sync(0xffffffffu, (uint64_t)(best.num >> 64), o);
        const uint64_t nl = __shfl_xor_sync(0xffffffffu, (uint64_t)best.num, o);
        t.num = ((u128)nh << 64) | nl;
        t.mid = __shfl_xor_sync(0xffffffffu, best.mid, o);
        t.idx = __shfl_xor_sync(0xffffffffu, best.idx, o);
        const int64_t tk = __shfl_xor_sync(0xffffffffu, bk, o);
        if (above(t, best)) {
            best = t;
            bk = tk;
        }
    }
    return {bk, best.num, seg_den(A.x, A.y, B.x, B.y)};
}

static __global__ void __launch_bounds__(NT) dp_kernel(const int64_t* __restrict__ counts, int64_t W, uint64_t T, Ws w) {
    if (chain::failed(counts)) return;
    const int64_t n = *w.n_pieces;
    const int64_t warp0 = ((int64_t)blockIdx.x * NT + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * NT) >> 5;
    const bool leader = lane_id() == 0;
    for (int64_t q = warp0; q < n; q += nwarps) {
        const uint4 pc = w.pieces[q];
        auto at = [&](int64_t k) -> int64_t {
            int64_t j = (int64_t)pc.z + k;
            if (j >= (int64_t)pc.y) j -= pc.y;
            return (int64_t)pc.x + j;
        };
        int64_t sp = 0;
        auto push = [&](int64_t lo, int64_t hi) {
            if (hi - lo < 2) return;
            if (leader) w.stack[at(sp)] = ((uint64_t)lo << 32) | (uint64_t)hi;
            ++sp;
        };
        // the guard: the piece's top vertex, and with coinciding ends the top vertices of both halves, are kept
        const int64_t nseg = pc.w;
        const Top t0 = top_of(w, W, pc, 0, nseg);
        if (leader) w.keep[at(t0.k)] = 1;
        const int2 A = *(const int2*)(w.in.v + 2 * at(0)), B = *(const int2*)(w.in.v + 2 * at(nseg));
        if (A.x == B.x && A.y == B.y) {
            const int64_t lo[2] = {0, t0.k}, hi[2] = {t0.k, nseg};
            for (int h = 0; h < 2; ++h) {
                if (hi[h] - lo[h] < 2) continue;
                const Top t = top_of(w, W, pc, lo[h], hi[h]);
                if (leader) w.keep[at(t.k)] = 1;
                push(lo[h], t.k);
                push(t.k, hi[h]);
            }
        } else {
            push(0, t0.k);
            push(t0.k, nseg);
        }
        while (sp > 0) {
            --sp;
            uint64_t e = 0;
            if (leader) e = w.stack[at(sp)];
            e = __shfl_sync(0xffffffffu, e, 0);
            const int64_t lo = (int64_t)(e >> 32), hi = (int64_t)(uint32_t)e;
            const Top t = top_of(w, W, pc, lo, hi);
            if (!exceeds(t.num, t.den, T)) continue;
            if (leader) w.keep[at(t.k)] = 1;
            push(lo, t.k);
            push(t.k, hi);
        }
    }
}

static __global__ void __launch_bounds__(NT) compact_kernel(const int64_t* __restrict__ counts, Ws w,
                                                            int32_t* __restrict__ vertices, int64_t* __restrict__ offsets) {
    const int64_t n_chains = counts[0], nv = *w.n_vertices;
    const int64_t gtid = (int64_t)blockIdx.x * NT + threadIdx.x, gstride = (int64_t)gridDim.x * NT;
    for (int64_t c = gtid; c <= n_chains; c += gstride)
        offsets[c] = c < n_chains ? (int64_t)w.rank[w.in.off[c]] : counts[1];
    for (int64_t i = gtid; i < nv; i += gstride) {
        if (!w.keep[i]) continue;
        const int64_t r = w.rank[i];
        vertices[2 * r] = w.in.v[2 * i];
        vertices[2 * r + 1] = w.in.v[2 * i + 1];
    }
}

// Simplifies the chains of w.in (counts[0] chains, counts[1] vertices) into vertices / offsets with tolerance T
// (quantize_tolerance); counts[1] becomes the number of kept vertices.  vcap bounds the vertices, chain_cap the chains.
inline int run(int64_t* counts, int64_t H, int64_t W, uint64_t T, int64_t vcap, int64_t chain_cap, const Ws& w,
               int32_t* vertices, int64_t* offsets, cudaStream_t s) {
    DM_CUDA(cudaMemsetAsync(w.n_pieces, 0, sizeof(int64_t), s));
    DM_TRY(launch(anchors_kernel, grid_for(chain_cap * 32, NT, 16), NT, 0, s, counts, H, W, w));
    DM_TRY(launch(dp_kernel, grid_for(vcap * 32, NT, 16), NT, 0, s, counts, W, T, w));
    DM_TRY(prims::scan_exclusive_u32(w.keep, w.rank, w.n_vertices, vcap, counts + 1, w.scan, s));
    return launch(compact_kernel, grid_for(imax64(vcap, chain_cap + 1), NT, 16), NT, 0, s, counts, w, vertices, offsets);
}

}  // namespace simplify
}  // namespace dm
