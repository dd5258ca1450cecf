// R6: edge score = Euclidean distance between pooled region means, with the reference's
// expanded formula sqrt(max(0, |x|^2 + |y|^2 - 2 x.y)) in fp32 (ExtractFeatures.py:139-147).
#include "common.cuh"

namespace dm {
namespace score {

// One warp per edge: 2 x D fp32 gathered with coalesced row reads, dot product reduced
// with warp shuffles; |x|^2, |y|^2 come precomputed per region (dm_region_mean).
__global__ void __launch_bounds__(256) score_l2_kernel(const float* __restrict__ mean, const float* __restrict__ norm2,
                                                       int D, const uint64_t* __restrict__ keys,
                                                       const int64_t* __restrict__ n_dev, const uint8_t* __restrict__ rescore,
                                                       float* __restrict__ scores) {
    const int64_t n = *n_dev;
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t e = warp0; e < n; e += nwarps) {
        const uint64_t k = keys[e];
        const int lo = key_lo(k), hi = key_hi(k);
        if (rescore && !rescore[lo] && !rescore[hi]) continue;
        const float* x = mean + (int64_t)lo * D;
        const float* y = mean + (int64_t)hi * D;
        float dot = 0.f;
        for (int d = lane; d < D; d += 32) dot = __fmaf_rn(x[d], y[d], dot);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
        if (lane == 0) {
            float v = (norm2[lo] + norm2[hi]) - 2.0f * dot;
            v = v < 0.f ? 0.f : v;
            scores[e] = __fsqrt_rn(v);
        }
    }
}

// D % 4 == 0 and 16-byte aligned rows: 8 lanes per edge, 4 edges per warp trip, 128-bit gathers.  Every load of a
// trip (key, both rows, both norms) is issued before the first use, so a trip costs two memory round trips (key, then
// rows) instead of one per 32 floats; the kernel was latency bound, not bandwidth bound, in the one-warp-per-edge form.
// The summation order of an edge is fixed (lane-strided float4 chunks, xor tree over 8 lanes): a score does not depend
// on which warp computed it.
__global__ void __launch_bounds__(256) score_l2_vec_kernel(const float* __restrict__ mean, const float* __restrict__ norm2,
                                                           int D4, const uint64_t* __restrict__ keys,
                                                           const int64_t* __restrict__ n_dev,
                                                           const uint8_t* __restrict__ rescore, float* __restrict__ scores) {
    const int64_t n = *n_dev;
    const int lane = threadIdx.x & 31, sub = lane & 7, grp = lane >> 3;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t e0 = warp0 * 4; e0 < n; e0 += nwarps * 4) {
        const int64_t e = e0 + grp;
        const bool live = e < n;
        const uint64_t k = live ? keys[e] : 0ull;
        const int lo = key_lo(k), hi = key_hi(k);
        const bool need = live && !(rescore && !rescore[lo] && !rescore[hi]);
        const float4* x = (const float4*)mean + (int64_t)lo * D4;
        const float4* y = (const float4*)mean + (int64_t)hi * D4;
        const float nn = (need && sub == 0) ? norm2[lo] + norm2[hi] : 0.f;
        float dot = 0.f;
        for (int c0 = sub; c0 < D4; c0 += 32) {               // 4 chunks of 8 lanes x 16 B per trip (one trip for D <= 128)
            float4 a[4], b[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = c0 + 8 * j;
                const bool ok = need && c < D4;
                a[j] = ok ? x[c] : make_float4(0.f, 0.f, 0.f, 0.f);
                b[j] = ok ? y[c] : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                dot = __fmaf_rn(a[j].x, b[j].x, dot);
                dot = __fmaf_rn(a[j].y, b[j].y, dot);
                dot = __fmaf_rn(a[j].z, b[j].z, dot);
                dot = __fmaf_rn(a[j].w, b[j].w, dot);
            }
        }
        dot += __shfl_xor_sync(0xffffffffu, dot, 4);
        dot += __shfl_xor_sync(0xffffffffu, dot, 2);
        dot += __shfl_xor_sync(0xffffffffu, dot, 1);
        if (need && sub == 0) {
            float v = nn - 2.0f * dot;
            v = v < 0.f ? 0.f : v;
            scores[e] = __fsqrt_rn(v);
        }
    }
}

// Dense distance matrix D[i,j] for X[n,p], Y[m,p]: one warp per output element.
__global__ void __launch_bounds__(256) euclid_matrix_kernel(const float* __restrict__ X, const float* __restrict__ Y,
                                                            int64_t n, int64_t m, int64_t p, float* __restrict__ Dm) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t w = warp0; w < n * m; w += nwarps) {
        const int64_t i = w / m, j = w - i * m;
        const float* x = X + i * p;
        const float* y = Y + j * p;
        float xx = 0.f, yy = 0.f, xy = 0.f;
        for (int64_t d = lane; d < p; d += 32) {
            const float a = x[d], b = y[d];
            xx = __fmaf_rn(a, a, xx);
            yy = __fmaf_rn(b, b, yy);
            xy = __fmaf_rn(a, b, xy);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            xx += __shfl_xor_sync(0xffffffffu, xx, o);
            yy += __shfl_xor_sync(0xffffffffu, yy, o);
            xy += __shfl_xor_sync(0xffffffffu, xy, o);
        }
        if (lane == 0) {
            float v = (xx + yy) - 2.0f * xy;
            v = v < 0.f ? 0.f : v;
            Dm[w] = __fsqrt_rn(v);
        }
    }
}

}  // namespace score
}  // namespace dm

using namespace dm;

extern "C" int dm_score_l2(const float* mean, const float* norm2, int64_t D, const uint64_t* keys, const int64_t* n_dev,
                           int64_t capacity, const uint8_t* rescore, float* scores, dm_stream_t stream) {
    if (D <= 0 || capacity < 0) return DM_ERR_BAD_ARG;
    if (capacity == 0) return DM_OK;
    if (!mean || !norm2 || !keys || !n_dev || !scores) return DM_ERR_BAD_ARG;
    if (D % 4 == 0 && (uintptr_t)mean % 16 == 0)
        return launch(score::score_l2_vec_kernel, grid_for(capacity * 8), 256, 0, S(stream), mean, norm2, (int)(D / 4), keys,
            n_dev, rescore, scores);
    return launch(score::score_l2_kernel, grid_for(capacity * 32), 256, 0, S(stream), mean, norm2, (int)D, keys, n_dev, rescore,
        scores);
}

extern "C" int dm_euclidean_matrix(const float* X, const float* Y, int64_t n, int64_t m, int64_t p, float* Dm,
                                   dm_stream_t stream) {
    if (n < 0 || m < 0 || p < 0) return DM_ERR_BAD_ARG;
    if (n == 0 || m == 0) return DM_OK;
    if (!X || !Y || !Dm) return DM_ERR_BAD_ARG;
    return launch(score::euclid_matrix_kernel, grid_for(n * m * 32), 256, 0, S(stream), X, Y, n, m, p, Dm);
}
