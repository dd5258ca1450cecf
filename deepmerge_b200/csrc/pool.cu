// R3-R5: region -> sample-point membership and mean pooling; per-pixel embedding pooling.
#include <cuda_bf16.h>
#include "common.cuh"
#include "prims.cuh"

namespace dm {
namespace pool {

__global__ void points_region_kernel(const int32_t* __restrict__ labels, int64_t H, int64_t W, int64_t ld,
                                     const int32_t* __restrict__ xs, const int32_t* __restrict__ ys, int64_t n,
                                     int32_t* __restrict__ out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int x = xs[i], y = ys[i];
        int l = -1;
        if (x >= 0 && x < W && y >= 0 && y < H) l = labels[(int64_t)y * ld + x];
        out[i] = l < 0 ? -1 : l;
    }
}

// key = region (invalid -> n_regions, sorts last), value = point id
__global__ void csr_keys_kernel(const int32_t* __restrict__ rop, int64_t n, int64_t n_regions, uint64_t* __restrict__ keys,
                                uint32_t* __restrict__ vals, int64_t* __restrict__ n_dev) {
    if (blockIdx.x == 0 && threadIdx.x == 0) *n_dev = n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int r = rop[i];
        keys[i] = (r >= 0 && r < n_regions) ? (uint64_t)r : (uint64_t)n_regions;
        vals[i] = (uint32_t)i;
    }
}

// One warp per region, lanes over the feature dimension, points visited in membership
// order: sum = ((f0 + f1) + f2) + ...  exactly like np.mean's row-by-row reduction
// (ExtractFeatures.py:211-212).  K*32 feature columns per pass starting at d_base.
template <int K>
__global__ void __launch_bounds__(256) pool_points_kernel(const int64_t* __restrict__ offsets,
                                                          const int32_t* __restrict__ ids, const float* __restrict__ feats,
                                                          int64_t ld, int64_t R_all, int D, int d_base, float* __restrict__ sum,
                                                          int32_t* __restrict__ cnt, const int64_t* __restrict__ range,
                                                          float* __restrict__ mean, float* __restrict__ norm2) {
    const int lane = threadIdx.x & 31;
    // range (row tiles of a sharded scene: ids are global, the tile's points fall into a small id interval): only
    // regions [range[0], range[1]] are visited; rows and counts outside are the caller's
    const int64_t r_first = range ? imax64(range[0], 0) : 0, R = range ? imin64(range[1], R_all - 1) + 1 : R_all;
    // An empty interval -- (INT64_MAX, -1) from dm_points_id_range for a tile without points -- visits nothing: return
    // before r_first + warp index can overflow (the same decision in every thread, before any shuffle).
    if (r_first >= R) return;
    const int64_t warp0 = r_first + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    // A region costs three dependent round trips (offsets -> point ids -> rows).  The warp therefore looks one region
    // ahead: the next region's offsets are requested before this region's rows, and its point ids (one per lane) as
    // soon as those offsets arrive, while the rows are still in flight.
    int64_t r = warp0, a = 0, b = 0;
    int my = 0;                                            // lane l holds the id of the region's point a + l
    if (r < R) {
        a = offsets[r];
        b = offsets[r + 1];
        my = a + lane < b ? ids[a + lane] : 0;
    }
    auto rows4 = [&](float (&v)[4][K], int id_lane, int u0, int n) {   // rows u0 .. u0+3 of the (<= 32) ids held by the lanes
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (u0 + u < n) {                              // (n is the same in every lane)
                const float* row = feats + (int64_t)__shfl_sync(0xffffffffu, id_lane, u0 + u) * ld + d_base;
#pragma unroll
                for (int k = 0; k < K; ++k) v[u][k] = (d_base + lane + 32 * k < D) ? row[lane + 32 * k] : 0.f;
            }
        }
    };
    auto add4 = [&](float (&acc)[K], const float (&v)[4][K], int u0, int n) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (u0 + u < n) {
#pragma unroll
                for (int k = 0; k < K; ++k) acc[k] += v[u][k];
            }
        }
    };
    while (r < R) {
        const int64_t rn = r + nwarps;
        int64_t an = 0, bn = 0;
        if (rn < R) {
            an = offsets[rn];
            bn = offsets[rn + 1];
        }
        float acc[K];
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] = 0.f;
        const int n0 = (int)imin64(b - a, 32);
        float v[4][K];
        rows4(v, my, 0, n0);
        const int myn = (rn < R && an + lane < bn) ? ids[an + lane] : 0;    // waits for an / bn beside the rows above
        add4(acc, v, 0, n0);
        for (int u0 = 4; u0 < n0; u0 += 4) {
            rows4(v, my, u0, n0);
            add4(acc, v, u0, n0);
        }
        for (int64_t j = a + 32; j < b; j += 32) {         // more than 32 points: further chunks of ids
            const int n1 = (int)imin64(b - j, 32);
            const int more = j + lane < b ? ids[j + lane] : 0;
            for (int u0 = 0; u0 < n1; u0 += 4) {
                rows4(v, more, u0, n1);
                add4(acc, v, u0, n1);
            }
        }
#pragma unroll
        for (int k = 0; k < K; ++k)
            if (d_base + lane + 32 * k < D) sum[r * D + d_base + lane + 32 * k] = acc[k];
        if (lane == 0 && d_base == 0) cnt[r] = (int32_t)(b - a);
        if (mean) {     // D <= 128: the whole row is in this pass -- mean and norm exactly as region_mean_kernel forms them
            const int n = (int)(b - a);
            const float c = n > 0 ? (float)n : __int_as_float(0x7fc00000);
            float n2 = 0.f;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                if (lane + 32 * k < D) {
                    const float v = n > 0 ? __fdiv_rn(acc[k], c) : c;
                    mean[r * D + lane + 32 * k] = v;
                    n2 = __fmaf_rn(v, v, n2);
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) n2 += __shfl_xor_sync(0xffffffffu, n2, o);
            if (lane == 0) norm2[r] = n2;
        }
        r = rn;
        a = an;
        b = bn;
        my = myn;
    }
}

// mean = sum / max(cnt,1) with an IEEE fp32 division (np.mean divides the fp32 sum by n),
// norm2 = sum_d mean^2 reduced in a fixed lane/shuffle order (deterministic).
__global__ void __launch_bounds__(256) region_mean_kernel(const float* __restrict__ sum, const int32_t* __restrict__ cnt,
                                                          int64_t R, int D, float* __restrict__ mean,
                                                          float* __restrict__ norm2, const uint8_t* __restrict__ only) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    auto one = [&](int64_t r) {
        // A region without sample points has no embedding: its mean (and norm) is NaN, what np.mean over no rows gives
        // (ExtractFeatures.py:211-212; the reference itself raises earlier on an empty PointID field).  NaN scores fail
        // `< tau`, NaN logits fail `o1 > o0`: such a region never merges on the strength of a made-up zero vector.
        const int n = cnt[r];
        const float c = n > 0 ? (float)n : __int_as_float(0x7fc00000);
        float n2 = 0.f;
        for (int d0 = 0; d0 < D; d0 += 128) {          // four loads in flight per lane; same order of the norm's terms
            float x[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) x[k] = (n > 0 && d0 + 32 * k + lane < D) ? sum[r * D + d0 + 32 * k + lane] : 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int d = d0 + 32 * k + lane;
                if (d < D) {
                    const float v = n > 0 ? __fdiv_rn(x[k], c) : c;
                    mean[r * D + d] = v;
                    n2 = __fmaf_rn(v, v, n2);
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) n2 += __shfl_xor_sync(0xffffffffu, n2, o);
        if (lane == 0) norm2[r] = n2;
    };
    if (!only) {                                   // every region: one warp per region
        for (int64_t r = warp0; r < R; r += nwarps) one(r);
        return;
    }
    // sparse update: a warp takes 32 consecutive regions -- one coalesced look at the flags, then the flagged ones in turn
    for (int64_t r0 = warp0 * 32; r0 < R; r0 += nwarps * 32) {
        unsigned m = __ballot_sync(0xffffffffu, r0 + lane < R && only[r0 + lane]);
        while (m) {
            one(r0 + __ffs(m) - 1);
            m &= m - 1;
        }
    }
}

// Per-pixel embedding pooling.  A warp walks a run of pixels of one raster row; lanes hold
// 32-column slices of the current label's partial sum in registers and flush it with one
// fp32 atomic per column only when the label changes (run-length pre-aggregation).
template <typename T, int K>
__global__ void __launch_bounds__(256) pool_dense_kernel(const int32_t* __restrict__ labels, int64_t H, int64_t W,
                                                         int64_t ld, const T* __restrict__ emb, int D, int d_base,
                                                         int64_t n_regions, float* __restrict__ sum,
                                                         int32_t* __restrict__ cnt, int chunk) {
    const int lane = threadIdx.x & 31;
    const int64_t chunks_per_row = (W + chunk - 1) / chunk;
    const int64_t total = H * chunks_per_row;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t w = warp0; w < total; w += nwarps) {
        const int64_t y = w / chunks_per_row;
        const int64_t xa = (w - y * chunks_per_row) * chunk;
        const int64_t xb = min(W, xa + chunk);
        float acc[K];
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] = 0.f;
        int cur = -1, run = 0;
        for (int64_t x = xa; x < xb; ++x) {
            int l = labels[y * ld + x];
            if (l >= n_regions) l = -1;
            if (l != cur) {
                if (cur >= 0) {
#pragma unroll
                    for (int k = 0; k < K; ++k)
                        if (d_base + lane + 32 * k < D) atomicAdd(&sum[(int64_t)cur * D + d_base + lane + 32 * k], acc[k]);
                    if (lane == 0 && d_base == 0) atomicAdd(&cnt[cur], run);
                }
#pragma unroll
                for (int k = 0; k < K; ++k) acc[k] = 0.f;
                cur = l;
                run = 0;
            }
            if (l >= 0) {
                const T* e = emb + (y * W + x) * (int64_t)D + d_base;
#pragma unroll
                for (int k = 0; k < K; ++k)
                    if (d_base + lane + 32 * k < D) acc[k] += (float)e[lane + 32 * k];
                ++run;
            }
        }
        if (cur >= 0) {
#pragma unroll
            for (int k = 0; k < K; ++k)
                if (d_base + lane + 32 * k < D) atomicAdd(&sum[(int64_t)cur * D + d_base + lane + 32 * k], acc[k]);
            if (lane == 0 && d_base == 0) atomicAdd(&cnt[cur], run);
        }
    }
}

// Per-boundary pooling of a dense embedding grid (north-star "per-boundary feature vectors"; the reference
// only writes a scalar per boundary, ExtractFeatures.py:217-219).  For every 4-adjacent pixel pair whose two
// valid labels differ, both pixels' embeddings are added to the edge of that label pair.  A warp takes 32
// consecutive pixels of a row; lanes flag their (right, down) pairs, then the warp serves the flagged pairs
// one after another: the edge index comes from a binary search in the sorted unique edge keys (every lane
// runs the same search: no divergence), and the lanes add the two embedding rows slice by slice.
template <typename T>
__global__ void __launch_bounds__(256) pool_boundary_kernel(const int32_t* __restrict__ labels, int64_t H, int64_t W,
                                                            int64_t ld, int64_t rows_avail, const T* __restrict__ emb,
                                                            int D, const uint64_t* __restrict__ keys,
                                                            const int64_t* __restrict__ n_edges_dev,
                                                            float* __restrict__ bsum, int32_t* __restrict__ bcnt) {
    const int lane = threadIdx.x & 31;
    const int64_t E = *n_edges_dev;
    const int64_t chunks_per_row = (W + 31) / 32;
    const int64_t total = H * chunks_per_row;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t w = warp0; w < total; w += nwarps) {
        const int64_t y = w / chunks_per_row;
        const int64_t x = (w - y * chunks_per_row) * 32 + lane;
        int a = -1, r = -1, d = -1;
        if (x < W) {
            a = labels[y * ld + x];
            if (x + 1 < W) r = labels[y * ld + x + 1];
            if (y + 1 < rows_avail) d = labels[(y + 1) * ld + x];
        }
        const bool pr = a >= 0 && r >= 0 && a != r, pd = a >= 0 && d >= 0 && a != d;
        unsigned mr = __ballot_sync(0xffffffffu, pr), md = __ballot_sync(0xffffffffu, pd);
        for (int dir = 0; dir < 2; ++dir) {
            unsigned m = dir == 0 ? mr : md;
            while (m) {
                const int src = __ffs(m) - 1;
                m &= m - 1;
                const int la = __shfl_sync(0xffffffffu, a, src);
                const int lb = __shfl_sync(0xffffffffu, dir == 0 ? r : d, src);
                const uint64_t key = pack_key(la, lb);
                int64_t lo = 0, hi = E;                       // first index with keys[i] >= key
                while (lo < hi) {
                    const int64_t mid = (lo + hi) >> 1;
                    if (keys[mid] < key) lo = mid + 1;
                    else hi = mid;
                }
                if (lo >= E || keys[lo] != key) continue;     // not an edge of this list (e.g. a foreign tile's)
                const int64_t xp = (w - y * chunks_per_row) * 32 + src;
                const T* e0 = emb + (y * W + xp) * (int64_t)D;
                const T* e1 = dir == 0 ? e0 + D : e0 + W * (int64_t)D;
                for (int k = lane; k < D; k += 32) atomicAdd(&bsum[lo * D + k], (float)e0[k] + (float)e1[k]);
                if (lane == 0) atomicAdd(&bcnt[lo], 2);
            }
        }
    }
}

// N1 (first piece): batched zero-padded window cut around sample points, the semantics of
// ExtractFeatureDataset.cut_image (MyUtils2.py:330-360) on a band-major uint8 raster [C, H, W]:
// out[i, c, v, u] = image[c, y0_i + v, x0_i + u] inside the raster, 0 outside.  One warp per output row.
__global__ void __launch_bounds__(256) cut_windows_kernel(const uint8_t* __restrict__ image, int C, int64_t H, int64_t W,
                                                          const int32_t* __restrict__ x0s, const int32_t* __restrict__ y0s,
                                                          int64_t n, int size, uint8_t* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t rows = n * C * size;
    for (int64_t w = warp0; w < rows; w += nwarps) {
        const int64_t i = w / ((int64_t)C * size);
        const int c = (int)((w / size) % C), v = (int)(w % size);
        const int64_t y = (int64_t)y0s[i] + v, x0 = x0s[i];
        uint8_t* dst = out + w * size;
        const bool row_in = y >= 0 && y < H;
        const uint8_t* src = image + ((int64_t)c * H + (row_in ? y : 0)) * W;
        for (int u = lane; u < size; u += 32) {
            const int64_t x = x0 + u;
            dst[u] = (row_in && x >= 0 && x < W) ? src[x] : (uint8_t)0;
        }
    }
}

// N2: bounding boxes of the regions (for the designed attributes len / width / smooth / compact / border, MyUtils1.py:79-114).
// A warp walks down a 32-pixel column strip; a lane keeps the vertical run of its column (label, first row) and publishes
// it with four integer atomics when the label changes: min / max column, first / last row.
__global__ void __launch_bounds__(256) region_bbox_kernel(const int32_t* __restrict__ labels, int64_t H, int64_t W, int64_t ld,
                                                          int64_t R, int32_t* __restrict__ bbox, int rows_per_warp,
                                                          unsigned long long* __restrict__ bad) {
    const int lane = threadIdx.x & 31;
    const int64_t strips = (W + 31) / 32, chunks = (H + rows_per_warp - 1) / rows_per_warp;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t w = warp0; w < strips * chunks; w += nwarps) {
        const int64_t sx = w % strips, cy = w / strips;
        const int64_t x = sx * 32 + lane, y0 = cy * rows_per_warp, y1 = imin64(H, y0 + rows_per_warp);
        if (x >= W) continue;
        int cur = -1;
        int64_t ys = y0;
        auto flush = [&](int64_t ylast) {
            if (cur < 0) return;
            if (cur >= R) { atomicExch(bad, 1ull); return; }
            int32_t* b = bbox + (int64_t)cur * 4;
            atomicMin(&b[0], (int)x);
            atomicMin(&b[1], (int)ys);
            atomicMax(&b[2], (int)x);
            atomicMax(&b[3], (int)ylast);
        };
        for (int64_t y = y0; y < y1; ++y) {
            const int l = labels[y * ld + x];
            if (l != cur) {
                flush(y - 1);
                cur = l;
                ys = y;
            }
        }
        flush(y1 - 1);
    }
}
__global__ void region_bbox_init_kernel(int32_t* __restrict__ bbox, int64_t R) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (int64_t)gridDim.x * blockDim.x) {
        bbox[4 * r] = 0x7fffffff;
        bbox[4 * r + 1] = 0x7fffffff;
        bbox[4 * r + 2] = -1;
        bbox[4 * r + 3] = -1;
    }
}

}  // namespace pool
}  // namespace dm

using namespace dm;

extern "C" int dm_points_region(const int32_t* labels, int64_t H, int64_t W, int64_t ld, const int32_t* xs,
                                const int32_t* ys, int64_t n, int32_t* out, dm_stream_t stream) {
    if (n < 0 || H < 0 || W < 0 || ld < W) return DM_ERR_BAD_ARG;
    if (n == 0) return DM_OK;
    if (!labels || !xs || !ys || !out) return DM_ERR_BAD_ARG;
    return launch(pool::points_region_kernel, grid_for(n), 256, 0, S(stream), labels, H, W, ld, xs, ys, n, out);
}

namespace {
struct CsrWs {
    uint64_t* keys;
    uint32_t* vals;
    int64_t* n_dev;
    void* sort;
    size_t bytes;
};
CsrWs csr_ws(void* base, int64_t n_points, int64_t n_regions) {
    const int64_t cap = imax64(n_points, 1);
    Carver c(base);
    // the bucket sort keeps per-id arrays for the n_regions + 1 keys (region ids and the "no region" key)
    return {c.take<uint64_t>(cap), c.take<uint32_t>(cap), c.take<int64_t>(1),
            c.take<char>(prims::ws_bytes(cap, false, n_regions + 1)), c.used()};
}
}  // namespace

extern "C" size_t dm_csr_workspace_bytes(int64_t n_points, int64_t n_regions) {
    return csr_ws(nullptr, n_points, n_regions).bytes;
}

extern "C" int dm_csr_build(const int32_t* rop, int64_t n, int64_t R, int64_t* offsets, int32_t* point_ids, void* ws,
                            size_t ws_bytes, dm_stream_t stream) {
    if (n < 0 || n > INT32_MAX || R < 0 || !offsets) return DM_ERR_BAD_ARG;   // point ids are int32
    cudaStream_t s = S(stream);
    if (n == 0) {
        DM_CUDA(cudaMemsetAsync(offsets, 0, (size_t)(R + 1) * sizeof(int64_t), s));
        return DM_OK;
    }
    if (!rop || !point_ids || !ws) return DM_ERR_BAD_ARG;
    const CsrWs w = csr_ws(ws, n, R);
    if (ws_bytes < w.bytes) return DM_ERR_WORKSPACE;
    DM_TRY(launch(pool::csr_keys_kernel, grid_for(n), 256, 0, s, rop, n, R, w.keys, w.vals, w.n_dev));
    // stable sort by region only (input is in ascending point id): low bits_for(R+1) bits
    const int b = bits_for(R + 1);
    // bucket + rank in one cooperative launch, offsets and point ids included
    return prims::sort_pairs(w.keys, w.vals, w.n_dev, n, b, b, w.sort, s, R + 1, offsets, point_ids);
}

template <int K>
static int pool_points_groups(const int64_t* offsets, const int32_t* ids, const float* feats, int64_t ld, int64_t R, int D,
                              int d0, float* sum, int32_t* cnt, const int64_t* range, float* mean, float* norm2,
                              cudaStream_t s) {
    return launch(pool::pool_points_kernel<K>, grid_for(R * 32), 256, 0, s, offsets, ids, feats, ld, R, D, d0, sum, cnt, range,
                  mean, norm2);
}

// One pass of the pooling kernel over feature columns [d0, min(D, d0 + 128)): K = 1..4 groups of 32 columns.
static int pool_points_pass(const int64_t* offsets, const int32_t* ids, const float* feats, int64_t ld, int64_t R, int D,
                            int d0, float* sum, int32_t* cnt, const int64_t* range, float* mean, float* norm2,
                            cudaStream_t s) {
    const int rem = D - d0;
    if (rem > 96) return pool_points_groups<4>(offsets, ids, feats, ld, R, D, d0, sum, cnt, range, mean, norm2, s);
    if (rem > 64) return pool_points_groups<3>(offsets, ids, feats, ld, R, D, d0, sum, cnt, range, mean, norm2, s);
    if (rem > 32) return pool_points_groups<2>(offsets, ids, feats, ld, R, D, d0, sum, cnt, range, mean, norm2, s);
    return pool_points_groups<1>(offsets, ids, feats, ld, R, D, d0, sum, cnt, range, mean, norm2, s);
}

extern "C" int dm_pool_points_csr_tile(const int64_t* offsets, const int32_t* ids, const float* feats, int64_t ld, int64_t R,
                                       int64_t D, float* sum, int32_t* cnt, const int64_t* region_range, dm_stream_t stream) {
    if (R < 0 || D <= 0 || ld < D || D > (1 << 20)) return DM_ERR_BAD_ARG;
    if (R == 0) return DM_OK;
    if (!offsets || !sum || !cnt) return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    if (region_range) DM_CUDA(cudaMemsetAsync(cnt, 0, (size_t)R * sizeof(int32_t), s));   // no points outside the range
    for (int d0 = 0; d0 < D; d0 += 128)
        DM_TRY(pool_points_pass(offsets, ids, feats, ld, R, (int)D, d0, sum, cnt, region_range, nullptr, nullptr, s));
    return DM_OK;
}

extern "C" int dm_pool_points_csr_mean(const int64_t* offsets, const int32_t* ids, const float* feats, int64_t ld, int64_t R,
                                       int64_t D, float* sum, int32_t* cnt, float* mean, float* norm2, dm_stream_t stream) {
    if (R < 0 || D <= 0 || ld < D) return DM_ERR_BAD_ARG;
    if (D > 128) return DM_ERR_UNSUPPORTED;                 // the row must fit one pass of the pooling kernel
    if (R == 0) return DM_OK;
    if (!offsets || !sum || !cnt || !mean || !norm2) return DM_ERR_BAD_ARG;
    return pool_points_pass(offsets, ids, feats, ld, R, (int)D, 0, sum, cnt, nullptr, mean, norm2, S(stream));
}

extern "C" int dm_pool_points_csr(const int64_t* offsets, const int32_t* ids, const float* feats, int64_t ld, int64_t R,
                                  int64_t D, float* sum, int32_t* cnt, dm_stream_t stream) {
    return dm_pool_points_csr_tile(offsets, ids, feats, ld, R, D, sum, cnt, nullptr, stream);
}

// [first, last] region id that has a point (first > last: none); the argument of dm_pool_points_csr_tile
namespace dm { namespace pool {
__global__ void id_range_kernel(const int32_t* __restrict__ rop, int64_t n, int64_t R, long long* __restrict__ range) {
    long long lo = 0x7fffffffffffffffll, hi = -1;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int r = rop[i];
        if (r >= 0 && r < R) {
            lo = lo < r ? lo : r;
            hi = hi > r ? hi : r;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const long long l2 = __shfl_xor_sync(0xffffffffu, lo, o), h2 = __shfl_xor_sync(0xffffffffu, hi, o);
        lo = lo < l2 ? lo : l2;
        hi = hi > h2 ? hi : h2;
    }
    if ((threadIdx.x & 31) == 0 && hi >= 0) {
        atomicMin(range, lo);
        atomicMax(range + 1, hi);
    }
}
__global__ void id_range_init_kernel(long long* range) {
    range[0] = 0x7fffffffffffffffll;
    range[1] = -1;
}
}}  // namespace dm::pool

extern "C" int dm_points_id_range(const int32_t* region_of_point, int64_t n_points, int64_t n_regions, int64_t* range,
                                  dm_stream_t stream) {
    if (n_points < 0 || n_regions < 0 || !range || (n_points > 0 && !region_of_point)) return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    DM_TRY(launch(pool::id_range_init_kernel, 1, 1, 0, s, (long long*)range));
    if (n_points == 0) return DM_OK;
    return launch(pool::id_range_kernel, grid_for(n_points, 256, 4), 256, 0, s, region_of_point, n_points, n_regions,
        (long long*)range);
}

extern "C" int dm_region_mean(const float* sum, const int32_t* cnt, int64_t R, int64_t D, float* mean, float* norm2,
                              const uint8_t* only, dm_stream_t stream) {
    if (R < 0 || D <= 0) return DM_ERR_BAD_ARG;
    if (R == 0) return DM_OK;
    if (!sum || !cnt || !mean || !norm2) return DM_ERR_BAD_ARG;
    return launch(pool::region_mean_kernel, grid_for(R * 32), 256, 0, S(stream), sum, cnt, R, (int)D, mean, norm2,
        only);
}

template <typename T>
static int pool_dense_t(const int32_t* labels, int64_t H, int64_t W, int64_t ld, const T* emb, int64_t D, int64_t R,
                        float* sum, int32_t* cnt, cudaStream_t s) {
    const int chunk = 64;
    const int64_t warps = H * ceil_div(W, chunk);
    const unsigned g = grid_for(warps * 32);
    for (int d0 = 0; d0 < D; d0 += 128) {
        const int rem = (int)D - d0;
        if (rem > 96) {
            DM_TRY(launch(pool::pool_dense_kernel<T, 4>, g, 256, 0, s, labels, H, W, ld, emb, (int)D, d0, R, sum, cnt, chunk));
        } else if (rem > 64) {
            DM_TRY(launch(pool::pool_dense_kernel<T, 3>, g, 256, 0, s, labels, H, W, ld, emb, (int)D, d0, R, sum, cnt, chunk));
        } else if (rem > 32) {
            DM_TRY(launch(pool::pool_dense_kernel<T, 2>, g, 256, 0, s, labels, H, W, ld, emb, (int)D, d0, R, sum, cnt, chunk));
        } else {
            DM_TRY(launch(pool::pool_dense_kernel<T, 1>, g, 256, 0, s, labels, H, W, ld, emb, (int)D, d0, R, sum, cnt, chunk));
        }
    }
    return DM_OK;
}

extern "C" int dm_pool_dense(const int32_t* labels, int64_t H, int64_t W, int64_t ld, const void* emb, int dtype_bf16,
                             int64_t D, int64_t R, float* sum, int32_t* cnt, dm_stream_t stream) {
    if (H < 0 || W < 0 || ld < W || D <= 0 || R < 0) return DM_ERR_BAD_ARG;
    if (H == 0 || W == 0) return DM_OK;
    if (!labels || !emb || !sum || !cnt) return DM_ERR_BAD_ARG;
    if (dtype_bf16) return pool_dense_t<__nv_bfloat16>(labels, H, W, ld, (const __nv_bfloat16*)emb, D, R, sum, cnt, S(stream));
    return pool_dense_t<float>(labels, H, W, ld, (const float*)emb, D, R, sum, cnt, S(stream));
}

extern "C" int dm_pool_boundary(const int32_t* labels, int64_t rows_own, int64_t rows_avail, int64_t W, int64_t ld,
                                const void* emb, int dtype_bf16, int64_t D, const uint64_t* edge_keys,
                                const int64_t* n_edges_dev, int64_t capacity, float* bsum, int32_t* bcnt,
                                dm_stream_t stream) {
    if (rows_own < 0 || W < 0 || ld < W || D <= 0 || capacity < 0) return DM_ERR_BAD_ARG;
    if (rows_avail != rows_own && rows_avail != rows_own + 1) return DM_ERR_BAD_ARG;
    if (rows_own == 0 || W == 0 || capacity == 0) return DM_OK;
    if (!labels || !emb || !edge_keys || !n_edges_dev || !bsum || !bcnt) return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    const unsigned g = grid_for(rows_own * ceil_div(W, 32) * 32);
    if (dtype_bf16)
        return launch(pool::pool_boundary_kernel<__nv_bfloat16>, g, 256, 0, s, labels, rows_own, W, ld, rows_avail,
            (const __nv_bfloat16*)emb, (int)D, edge_keys, n_edges_dev, bsum, bcnt);
    return launch(pool::pool_boundary_kernel<float>, g, 256, 0, s, labels, rows_own, W, ld, rows_avail, (const float*)emb,
        (int)D, edge_keys, n_edges_dev, bsum, bcnt);
}

extern "C" int dm_cut_windows(const uint8_t* image, int64_t C, int64_t H, int64_t W, const int32_t* x0, const int32_t* y0,
                              int64_t n, int64_t size, uint8_t* out, dm_stream_t stream) {
    if (C < 1 || H < 0 || W < 0 || n < 0 || size < 1 || size > (1 << 14)) return DM_ERR_BAD_ARG;
    if (n == 0) return DM_OK;
    if (!image || !x0 || !y0 || !out) return DM_ERR_BAD_ARG;
    return launch(pool::cut_windows_kernel, grid_for(n * C * size * 32), 256, 0, S(stream), image, (int)C, H, W, x0,
        y0, n, (int)size, out);
}

extern "C" int dm_region_bbox(const int32_t* labels, int64_t H, int64_t W, int64_t ld, int64_t n_regions, int32_t* bbox,
                              int64_t* bad_label, dm_stream_t stream) {
    if (H < 0 || W < 0 || ld < W || n_regions < 0 || H > 0x7ffffff0 || W > 0x7ffffff0) return DM_ERR_BAD_ARG;
    const bool pixels = H > 0 && W > 0;
    if (n_regions > 0 && (!bbox || !bad_label || (pixels && !labels))) return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    if (bad_label) DM_CUDA(cudaMemsetAsync(bad_label, 0, sizeof(int64_t), s));
    if (n_regions == 0) return DM_OK;
    DM_TRY(launch(pool::region_bbox_init_kernel, grid_for(n_regions), 256, 0, s, bbox, n_regions));
    if (!pixels) return DM_OK;
    const int rows_per_warp = 128;
    const int64_t warps = ceil_div(W, 32) * ceil_div(H, rows_per_warp);
    return launch(pool::region_bbox_kernel, grid_for(warps * 32), 256, 0, s, labels, H, W, ld, n_regions, bbox, rows_per_warp,
        (unsigned long long*)bad_label);
}
