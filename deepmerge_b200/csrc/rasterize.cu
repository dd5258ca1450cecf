// Rasterizer: polygon rings in map coordinates -> int32 label raster (dm_rasterize in include/deepmerge_b200.h), the
// contract of shapefile.rasterize_polygons.  The per-segment arithmetic lives in rasterize_core.cuh.
//
// Every closed ring crosses each row an even number of times under the half-open rule, and the crossing column is
// monotone in the crossing x, so pairing the crossings of one (polygon, row) by column gives the spans the reference
// fills by pairing them by x.  The whole raster therefore takes one integer sort instead of a scanline loop per polygon:
//
// 1. count_kernel  per vertex (= per segment, the vertex to its successor in the ring): the rows in [0, H) the segment
//                  crosses, the exact total, status 1 / 4 for a non-finite coordinate / a malformed ring.
// 2. scan          counts -> the first key of every segment.
// 3. emit_kernel   one u64 key per crossing: record << 32 | row (W + 1) + column.  Status 2 when the total exceeds the
//                  capacity.
// 4. sort_pairs    by (record, row, column): bucket + rank, one bucket per record.
// 5. span_kernel   the sorted keys in pairs (2m, 2m + 1) are the spans [c0, c1) of one (record, row); each is painted
//                  with max(record) into the raster, which starts at -1, so the later record wins.
// 6. map_kernel    only for ids or nodata != -1: -1 -> nodata, record -> ids[record].
#include "prims.cuh"
#include "rasterize_core.cuh"

namespace dm {
namespace rast {
using namespace rastcore;

constexpr int NT = 256;

struct Ws {
    uint32_t *cnt, *first;              // per vertex: crossings of its segment, the index of its first key
    uint64_t* keys;                     // per crossing
    int64_t* n_dev;                     // [0] vertices (the scan's count), [1] keys to sort (0 when nothing is painted),
                                        // [2] a crossing x is not finite
    void *scan, *sort;
};

size_t carve(Ws& w, void* base, int64_t n_vertices, int64_t n_records, int64_t cap) {
    Carver c(base);
    w.cnt = c.take<uint32_t>((size_t)n_vertices);
    w.first = c.take<uint32_t>((size_t)n_vertices);
    w.keys = c.take<uint64_t>((size_t)cap);
    w.n_dev = c.take<int64_t>(3);
    w.scan = c.take<char>(prims::scan_ws_bytes(n_vertices));
    w.sort = c.take<char>(prims::ws_bytes(cap, false, n_records));
    return c.used();
}

struct Rings {
    const double* xy;
    const int64_t* offsets;
    const int32_t* record;
    int64_t n_rings, n_vertices, n_records;
    double gt0, gt1, gt3, gt5;
};

struct Seg {
    double x0, y0, x1, y1;
    int32_t rec;
};

enum { ST_NONFINITE = 1, ST_CAPACITY = 2, ST_PAIRING = 3, ST_RINGS = 4 };

__device__ __forceinline__ bool failed(const int64_t* counts) { return *(volatile const int64_t*)(counts + 3) != 0; }
__device__ __forceinline__ void set_status(int64_t* counts, int st) {
    atomicExch((unsigned long long*)(counts + 3), (unsigned long long)st);
}

// The segment that starts at vertex v: to the next vertex of its ring, or from the last vertex back to the first when
// the ring's first and last pixel coordinates differ.  false when v starts none (outside every ring, a ring of fewer
// than 3 vertices, the last vertex of a closed ring) or on an error, which *st receives.
__device__ __forceinline__ bool segment(const Rings& g, int64_t v, Seg& s, int* st) {
    const int64_t* off = g.offsets;
    if (off[0] > v) return false;
    int64_t lo = 0, hi = g.n_rings;                 // the last ring k with off[k] <= v
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (off[mid] <= v) lo = mid;
        else hi = mid;
    }
    const int64_t b = off[lo], e = off[lo + 1];
    if (v >= e) return false;
    s.rec = g.record[lo];
    if (b < 0 || e > g.n_vertices || s.rec < 0 || s.rec >= g.n_records) {
        *st = ST_RINGS;
        return false;
    }
    if (e - b < 3) return false;
    s.x0 = rz_pixel(g.xy[2 * v], g.gt0, g.gt1);
    s.y0 = rz_pixel(g.xy[2 * v + 1], g.gt3, g.gt5);
    if (!rz_finite(s.x0) || !rz_finite(s.y0)) {
        *st = ST_NONFINITE;
        return false;
    }
    const int64_t u = v + 1 < e ? v + 1 : b;
    s.x1 = rz_pixel(g.xy[2 * u], g.gt0, g.gt1);
    s.y1 = rz_pixel(g.xy[2 * u + 1], g.gt3, g.gt5);
    if (u == b && s.x1 == s.x0 && s.y1 == s.y0) return false;    // explicitly closed: no closing segment
    return rz_finite(s.x1) && rz_finite(s.y1);                  // u's own thread reports it
}

__global__ void __launch_bounds__(NT) count_kernel(Rings g, int64_t H, uint32_t* __restrict__ cnt,
                                                   int64_t* __restrict__ counts, int64_t* __restrict__ n_dev) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        n_dev[0] = g.n_vertices;
        n_dev[2] = 0;
    }
    unsigned long long total = 0;
    int st = 0;
    for (int64_t v = (int64_t)blockIdx.x * NT + threadIdx.x; v < g.n_vertices; v += (int64_t)gridDim.x * NT) {
        Seg s;
        int64_t r0, n = 0;
        if (segment(g, v, s, &st)) n = rz_rows(s.y0, s.y1, H, &r0);
        cnt[v] = (uint32_t)n;
        total += (unsigned long long)n;
    }
    if (st) set_status(counts, st);
    for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
    if ((threadIdx.x & 31) == 0 && total) atomicAdd((unsigned long long*)(counts + 2), total);
}

// One key per crossing, record << 32 | row (W + 1) + column, at the segment's first index.  Sets status 2 and sorts
// nothing when the counts[2] crossings exceed cap.  Every block takes the same decision, as nothing it reads changes
// during the launch: a crossing x that is not finite (the interpolation overflowed) is flagged in n_dev[2] and still
// gets a valid key, and span_kernel reports it.
__global__ void __launch_bounds__(NT) emit_kernel(Rings g, int64_t H, int64_t W, int64_t cap,
                                                  const uint32_t* __restrict__ first, uint64_t* __restrict__ keys,
                                                  int64_t* __restrict__ counts, int64_t* __restrict__ n_dev) {
    const bool over = counts[2] > cap;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (over && !failed(counts)) counts[3] = ST_CAPACITY;
        n_dev[1] = over || failed(counts) ? 0 : counts[2];
    }
    if (over || failed(counts)) return;
    bool nonfinite = false;
    for (int64_t v = (int64_t)blockIdx.x * NT + threadIdx.x; v < g.n_vertices; v += (int64_t)gridDim.x * NT) {
        Seg s;
        int st = 0;                                 // the count kernel has reported every ring error
        if (!segment(g, v, s, &st)) continue;
        int64_t r0;
        const int64_t n = rz_rows(s.y0, s.y1, H, &r0);
        uint64_t* out = keys + first[v];
        for (int64_t k = 0; k < n; ++k) {
            const int64_t r = r0 + k;
            const double xi = rz_xi(s.x0, s.y0, s.x1, s.y1, rz_add((double)r, 0.5));
            nonfinite |= !rz_finite(xi);
            out[k] = ((uint64_t)(uint32_t)s.rec << 32) | (uint64_t)(r * (W + 1) + rz_col(xi, W));
        }
    }
    if (nonfinite) n_dev[2] = 1;
}

// One lane per pair of sorted keys; the warp then paints the 32 spans one after another, one column per lane.
__global__ void __launch_bounds__(NT) span_kernel(const uint64_t* __restrict__ keys, const int64_t* __restrict__ n_dev,
                                                  int64_t W, int64_t ld, int32_t* __restrict__ labels,
                                                  int64_t* __restrict__ counts) {
    if (failed(counts)) return;
    const int64_t n = n_dev[1];
    if (n_dev[2] || (n & 1)) {
        if (blockIdx.x == 0 && threadIdx.x == 0) set_status(counts, n_dev[2] ? ST_NONFINITE : ST_PAIRING);
        return;
    }
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * NT + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * NT) >> 5;
    unsigned long long spans = 0, pixels = 0;
    bool bad = false;
    for (int64_t p0 = warp0 * 32; p0 < n / 2; p0 += nwarps * 32) {
        const int64_t p = p0 + lane;
        int64_t row = 0, c0 = 0, c1 = 0;
        int32_t rec = 0;
        if (p < n / 2) {
            const ulonglong2 k = reinterpret_cast<const ulonglong2*>(keys)[p];
            const uint32_t la = (uint32_t)k.x, lb = (uint32_t)k.y;
            row = la / (uint32_t)(W + 1);
            if ((k.x >> 32) != (k.y >> 32) || lb / (uint32_t)(W + 1) != row) {
                bad = true;                                         // not one (record, row): paint nothing
            } else {
                rec = (int32_t)(k.x >> 32);
                c0 = la - row * (W + 1);
                c1 = lb - row * (W + 1);
                if (c1 > c0) {
                    ++spans;
                    pixels += (unsigned long long)(c1 - c0);
                }
            }
        }
        for (int j = 0; j < 32; ++j) {
            const int64_t a = __shfl_sync(0xffffffffu, c0, j), b = __shfl_sync(0xffffffffu, c1, j);
            if (a >= b) continue;
            int32_t* dst = labels + __shfl_sync(0xffffffffu, row, j) * ld;
            const int32_t v = __shfl_sync(0xffffffffu, rec, j);
            for (int64_t c = a + lane; c < b; c += 32) atomicMax(dst + c, v);
        }
    }
    if (__any_sync(0xffffffffu, bad) && lane == 0) set_status(counts, ST_PAIRING);
    for (int o = 16; o > 0; o >>= 1) {
        spans += __shfl_xor_sync(0xffffffffu, spans, o);
        pixels += __shfl_xor_sync(0xffffffffu, pixels, o);
    }
    if (lane == 0 && spans) {
        atomicAdd((unsigned long long*)counts, spans);
        atomicAdd((unsigned long long*)(counts + 1), pixels);
    }
}

// -1 -> nodata, record -> ids[record] (the record itself when ids is null); one block per row.
__global__ void __launch_bounds__(NT) map_kernel(int32_t* __restrict__ labels, int64_t H, int64_t W, int64_t ld,
                                                 const int32_t* __restrict__ ids, int32_t nodata) {
    for (int64_t y = blockIdx.x; y < H; y += gridDim.x) {
        int32_t* row = labels + y * ld;
        for (int64_t x = threadIdx.x; x < W; x += NT) {
            const int32_t v = row[x];
            row[x] = v < 0 ? nodata : ids ? ids[v] : v;
        }
    }
}

bool sizes_ok(int64_t n_vertices, int64_t n_records, int64_t cap) {
    return n_vertices >= 0 && n_vertices < (1ll << 31) && n_records >= 0 && n_records < (1ll << 31) && cap >= 0 &&
           cap < (1ll << 31);
}

}  // namespace rast
}  // namespace dm

using namespace dm;

extern "C" size_t dm_rasterize_workspace_bytes(int64_t n_vertices, int64_t n_records, int64_t capacity) {
    if (!rast::sizes_ok(n_vertices, n_records, capacity)) return 0;
    rast::Ws w;
    return rast::carve(w, nullptr, n_vertices, n_records, capacity);
}

extern "C" int dm_rasterize(const double* xy, int64_t n_vertices, const int64_t* ring_offsets, const int32_t* ring_record,
                            int64_t n_rings, int64_t n_records, double gt0, double gt1, double gt3, double gt5,
                            const int32_t* ids, int32_t nodata, int64_t H, int64_t W, int64_t ld, int64_t capacity,
                            int32_t* labels, int64_t* counts, void* ws, size_t ws_bytes, dm_stream_t stream) {
    if (!rast::sizes_ok(n_vertices, n_records, capacity) || n_rings < 0 || n_rings >= (1ll << 31) || H < 0 || W < 0 ||
        H >= (1ll << 31) || W >= (1ll << 31) || (H + 1) * (W + 1) > (1ll << 32) || ld < W || gt1 == 0.0 || gt5 == 0.0)
        return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    if (H == 0 || W == 0) {
        if (counts) DM_CUDA(cudaMemsetAsync(counts, 0, 4 * sizeof(int64_t), s));
        return DM_OK;
    }
    const bool work = n_rings > 0 && n_vertices > 0;
    if (!labels || !counts || (work && (!xy || !ring_offsets || !ring_record || !ws))) return DM_ERR_BAD_ARG;
    if (work && ws_bytes < dm_rasterize_workspace_bytes(n_vertices, n_records, capacity)) return DM_ERR_WORKSPACE;
    DM_CUDA(cudaMemsetAsync(counts, 0, 4 * sizeof(int64_t), s));
    // -1 everywhere before any polygon; the output has a row pitch
    DM_CUDA(cudaMemset2DAsync(labels, (size_t)ld * sizeof(int32_t), 0xff, (size_t)W * sizeof(int32_t), (size_t)H, s));
    if (work) {
        rast::Ws w;
        rast::carve(w, ws, n_vertices, n_records, capacity);
        const rast::Rings g{xy, ring_offsets, ring_record, n_rings, n_vertices, n_records, gt0, gt1, gt3, gt5};
        const unsigned g_verts = grid_for(n_vertices, rast::NT, 16);
        DM_TRY(launch(rast::count_kernel, g_verts, rast::NT, 0, s, g, H, w.cnt, counts, w.n_dev));
        DM_TRY(prims::scan_exclusive_u32(w.cnt, w.first, w.n_dev, n_vertices, nullptr, w.scan, s));
        DM_TRY(launch(rast::emit_kernel, g_verts, rast::NT, 0, s, g, H, W, capacity, w.first, w.keys, counts, w.n_dev));
        // by record (one bucket per record), then by row and column
        const int id_bits = bits_for(imax64(n_records, H * (W + 1)));
        DM_TRY(prims::sort_pairs(w.keys, nullptr, w.n_dev + 1, capacity, id_bits, 2 * id_bits, w.sort, s, n_records));
        DM_TRY(launch(rast::span_kernel, grid_for(capacity / 2 + 1, rast::NT, 16), rast::NT, 0, s, w.keys, w.n_dev, W,
                      ld, labels, counts));
    }
    if (ids == nullptr && nodata == -1) return DM_OK;
    return launch(rast::map_kernel, (unsigned)imin64(H, (int64_t)num_sms() * 16), rast::NT, 0, s, labels, H, W, ld, ids,
                  nodata);
}
