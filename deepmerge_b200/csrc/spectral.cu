// Region merging by spectral and shape heterogeneity (Baatz & Schaepe 2000, the fusion criterion of multiresolution
// segmentation): fusion values of the edges from the integer region statistics of the raster pass, local mutual best
// fitting selection, and the integer merge of those statistics.  Per-edge arithmetic in spectral_core.cuh.
#include "common.cuh"
#include "spectral_core.cuh"

namespace dm {
namespace spectral {

// One thread per edge: the two regions' area, perimeter and box, then the C band sums and sums of squares of both,
// contiguous int64 rows (32 bytes a row for C = 4).  fp64 throughout; the result is rounded to fp32 once.
__global__ void __launch_bounds__(256) score_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ lens,
                                                   const int64_t* __restrict__ n_dev, const int64_t* __restrict__ area,
                                                   const int64_t* __restrict__ perim, const uint64_t* __restrict__ bsum,
                                                   const uint64_t* __restrict__ bsq, int C, const int32_t* __restrict__ bbox,
                                                   const float* __restrict__ band_w, double w_shape, double w_cmpct,
                                                   const uint8_t* __restrict__ rescore, float* __restrict__ scores) {
    const int64_t n = *n_dev;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t k = keys[e];
        const int a = key_lo(k), b = key_hi(k);
        if (rescore && !rescore[a] && !rescore[b]) continue;
        const int64_t na = area[a], nb = area[b];
        const uint64_t *Sa = bsum + (int64_t)a * C, *Sb = bsum + (int64_t)b * C;
        const uint64_t *Qa = bsq + (int64_t)a * C, *Qb = bsq + (int64_t)b * C;
        double hc = 0.0;
        for (int c = 0; c < C; ++c)
            hc = sp_add(hc, sp_color_band(band_w ? (double)band_w[c] : 1.0, na, Sa[c], Qa[c], nb, Sb[c], Qb[c]));
        int32_t ba[4], bb[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            ba[j] = bbox[4 * (int64_t)a + j];
            bb[j] = bbox[4 * (int64_t)b + j];
        }
        scores[e] = __double2float_rn(sp_fusion(hc, na, perim[a], ba, nb, perim[b], bb, (int64_t)lens[e], w_shape, w_cmpct));
    }
}

// Order-preserving key of (score, edge index): the fp32 bits mapped so that unsigned order is float order (both zeros
// map to +0), the edge index below them.  Only called for scores below the threshold, so never for NaN.
__device__ __forceinline__ uint64_t mutual_key(float s, int64_t e) {
    unsigned u = __float_as_uint(s);
    u = s == 0.0f ? 0x80000000u : ((u & 0x80000000u) ? ~u : (u | 0x80000000u));
    return ((uint64_t)u << 32) | (uint64_t)e;
}

// pass 1: best[r] = min over the candidate edges of r of their keys
__global__ void mutual_min_kernel(const float* __restrict__ scores, float thr, const uint64_t* __restrict__ keys,
                                  const int64_t* __restrict__ n_dev, int64_t R, unsigned long long* __restrict__ best) {
    const int64_t n = *n_dev;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const float s = scores[e];
        if (!(s < thr)) continue;
        const uint64_t k = keys[e];
        if ((k >> 32) >= (uint64_t)R || (k & 0xffffffffu) >= (uint64_t)R) continue;
        const unsigned long long m = mutual_key(s, e);
        atomicMin(&best[key_lo(k)], m);
        atomicMin(&best[key_hi(k)], m);
    }
}

// pass 2: an edge is selected when its key is the minimum at both of its endpoints
__global__ void mutual_select_kernel(const float* __restrict__ scores, float thr, const uint64_t* __restrict__ keys,
                                     const int64_t* __restrict__ n_dev, int64_t R, const unsigned long long* __restrict__ best,
                                     uint8_t* __restrict__ selected, unsigned long long* __restrict__ n_sel) {
    const int64_t n = *n_dev;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x - (threadIdx.x & 31); e0 < n; e0 += stride) {
        const int64_t e = e0 + (threadIdx.x & 31);
        bool sel = false;
        if (e < n) {
            const float s = scores[e];
            const uint64_t k = keys[e];
            if (s < thr && (k >> 32) < (uint64_t)R && (k & 0xffffffffu) < (uint64_t)R) {
                const unsigned long long m = mutual_key(s, e);
                sel = best[key_lo(k)] == m && best[key_hi(k)] == m;
            }
            selected[e] = sel ? 1 : 0;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, sel);
        if (bal && (threadIdx.x & 31) == 0) atomicAdd(n_sel, (unsigned long long)__popc(bal));
    }
}

// Every region absorbed this round adds its integer statistics into its root and widens the root's box; all updates
// commute, so no order is needed.
__global__ void apply_regions_kernel(const int32_t* __restrict__ parent, uint8_t* __restrict__ alive,
                                     uint8_t* __restrict__ changed, unsigned long long* __restrict__ area,
                                     unsigned long long* __restrict__ perim, unsigned long long* __restrict__ bsum,
                                     unsigned long long* __restrict__ bsq, int C, int32_t* __restrict__ bbox, int64_t R,
                                     unsigned long long* __restrict__ n_moved) {
    for (int64_t x0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x - (threadIdx.x & 31); x0 < R;
         x0 += (int64_t)gridDim.x * blockDim.x) {
        const int64_t x = x0 + (threadIdx.x & 31);
        int r = 0;
        const bool moved = x < R && alive[x] && (r = parent[x]) != (int)x;
        const unsigned bal = __ballot_sync(0xffffffffu, moved);
        if (bal && (threadIdx.x & 31) == 0) atomicAdd(n_moved, (unsigned long long)__popc(bal));
        if (!moved) continue;
        alive[x] = 0;
        changed[r] = 1;
        atomicAdd(&area[r], area[x]);
        atomicAdd(&perim[r], perim[x]);
        for (int c = 0; c < C; ++c) {
            atomicAdd(&bsum[(int64_t)r * C + c], bsum[x * C + c]);
            atomicAdd(&bsq[(int64_t)r * C + c], bsq[x * C + c]);
        }
        atomicMin(&bbox[4 * (int64_t)r + 0], bbox[4 * x + 0]);
        atomicMin(&bbox[4 * (int64_t)r + 1], bbox[4 * x + 1]);
        atomicMax(&bbox[4 * (int64_t)r + 2], bbox[4 * x + 2]);
        atomicMax(&bbox[4 * (int64_t)r + 3], bbox[4 * x + 3]);
    }
}

}  // namespace spectral
}  // namespace dm

using namespace dm;

extern "C" int dm_score_spectral(const uint64_t* keys, const uint32_t* lens, const int64_t* n_dev, int64_t capacity,
                                 const int64_t* area, const int64_t* perimeter, const uint64_t* band_sum,
                                 const uint64_t* band_sumsq, int64_t C, const int32_t* bbox, const float* band_weights,
                                 float w_shape, float w_cmpct, const uint8_t* rescore, float* scores, dm_stream_t stream) {
    if (C <= 0 || C > 0x7fffffff || capacity < 0 || !(w_shape >= 0.f && w_shape <= 1.f) || !(w_cmpct >= 0.f && w_cmpct <= 1.f))
        return DM_ERR_BAD_ARG;
    if (capacity == 0) return DM_OK;
    if (!keys || !lens || !n_dev || !area || !perimeter || !band_sum || !band_sumsq || !bbox || !scores) return DM_ERR_BAD_ARG;
    return launch(spectral::score_kernel, grid_for(capacity), 256, 0, S(stream), keys, lens, n_dev, area, perimeter, band_sum,
        band_sumsq, (int)C, bbox, band_weights, (double)w_shape, (double)w_cmpct, rescore, scores);
}

namespace {
struct MutualWs {
    unsigned long long* best;
    size_t bytes;
};
MutualWs select_mutual_ws(void* base, int64_t R) {
    Carver c(base);
    return {c.take<unsigned long long>(imax64(R, 1)), c.used()};
}
}  // namespace

extern "C" size_t dm_merge_select_mutual_workspace_bytes(int64_t R) { return select_mutual_ws(nullptr, R).bytes; }

extern "C" int dm_merge_select_mutual(const float* scores, float threshold, const uint64_t* keys, const int64_t* n_dev,
                                      int64_t capacity, int64_t R, uint8_t* selected, int64_t* n_sel, void* ws,
                                      size_t ws_bytes, dm_stream_t stream) {
    // edge indices travel in the low 32 bits of the selection key
    if (capacity < 0 || capacity > 0xffffffffll || R < 0 || R > 0x7fffffff || !n_sel) return DM_ERR_BAD_ARG;
    const MutualWs w = select_mutual_ws(ws, R);
    if (capacity > 0) {
        if (!scores || !keys || !n_dev || !selected || !ws) return DM_ERR_BAD_ARG;
        if (ws_bytes < w.bytes) return DM_ERR_WORKSPACE;
    }
    cudaStream_t s = S(stream);
    DM_CUDA(cudaMemsetAsync(n_sel, 0, sizeof(int64_t), s));
    if (capacity == 0) return DM_OK;
    DM_CUDA(cudaMemsetAsync(w.best, 0xff, sizeof(unsigned long long) * (size_t)imax64(R, 1), s));
    DM_TRY(launch(spectral::mutual_min_kernel, grid_for(capacity), 256, 0, s, scores, threshold, keys, n_dev, R, w.best));
    return launch(spectral::mutual_select_kernel, grid_for(capacity), 256, 0, s, scores, threshold, keys, n_dev, R, w.best,
        selected, (unsigned long long*)n_sel);
}

extern "C" int dm_merge_apply_regions(const int32_t* parent, uint8_t* alive, uint8_t* changed, int64_t* area,
                                      int64_t* perimeter, uint64_t* band_sum, uint64_t* band_sumsq, int64_t C, int32_t* bbox,
                                      int64_t R, int64_t* n_merged, dm_stream_t stream) {
    if (R < 0 || C <= 0 || C > 0x7fffffff || !n_merged) return DM_ERR_BAD_ARG;
    if (R > 0 && (!parent || !alive || !changed || !area || !perimeter || !band_sum || !band_sumsq || !bbox))
        return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    DM_CUDA(cudaMemsetAsync(n_merged, 0, sizeof(int64_t), s));
    if (R == 0) return DM_OK;
    DM_CUDA(cudaMemsetAsync(changed, 0, (size_t)R, s));
    return launch(spectral::apply_regions_kernel, grid_for(R), 256, 0, s, parent, alive, changed, (unsigned long long*)area,
        (unsigned long long*)perimeter, (unsigned long long*)band_sum, (unsigned long long*)band_sumsq, (int)C, bbox, R,
        (unsigned long long*)n_merged);
}
