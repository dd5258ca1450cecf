// R11: contrastive pair loss forward + backward (Losses.py:34-38) and the row gather that
// feeds it from pooled features (R10 pair sampler output).
#include "common.cuh"

namespace dm {
namespace loss {

// One warp per pair: d = sum_k (a-b)^2 (shuffle reduction), per-pair loss and both gradients.
// Block partials are combined in a fixed order; a single block keeps the mean deterministic.
__global__ void __launch_bounds__(1024) contrastive_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                           const int64_t* __restrict__ flag, int64_t B, int D, float margin,
                                                           float* __restrict__ loss, float* __restrict__ ga,
                                                           float* __restrict__ gb) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    __shared__ float part[32];
    float acc = 0.f;
    const float invB = 1.0f / (float)B;
    for (int64_t i = warp; i < B; i += nw) {
        const float* x = a + i * D;
        const float* y = b + i * D;
        float d = 0.f;
        for (int k = lane; k < D; k += 32) {
            const float t = x[k] - y[k];
            d = __fmaf_rn(t, t, d);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
        const float f = (float)flag[i];
        const float hinge = fmaxf(margin - d, 0.f);
        acc += f * d + (1.f - f) * hinge;
        if (ga || gb) {
            // dL/da = (2/B) (a-b) (flag - (1-flag)[d < margin]) = -dL/db
            const float coef = 2.0f * invB * (f - (1.f - f) * (d < margin ? 1.f : 0.f));
            for (int k = lane; k < D; k += 32) {
                const float g = coef * (x[k] - y[k]);
                if (ga) ga[i * D + k] = g;
                if (gb) gb[i * D + k] = -g;
            }
        }
    }
    if (lane == 0) part[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f;
        for (int w = 0; w < nw; ++w) s += part[w];
        *loss = s * invB;
    }
}

__global__ void gather_rows_kernel(const float* __restrict__ table, int D, const int64_t* __restrict__ idx, int64_t n,
                                   float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp0; i < n; i += nwarps) {
        const float* row = table + idx[i] * D;
        for (int k = lane; k < D; k += 32) out[i * D + k] = row[k];
    }
}

}  // namespace loss
}  // namespace dm

using namespace dm;

extern "C" int dm_contrastive_fwd_bwd(const float* a, const float* b, const int64_t* flag, int64_t B, int64_t D, float margin,
                                      float* loss, float* ga, float* gb, dm_stream_t stream) {
    if (B <= 0 || D <= 0 || !a || !b || !flag || !loss) return DM_ERR_BAD_ARG;
    return launch(loss::contrastive_kernel, 1, 1024, 0, S(stream), a, b, flag, B, (int)D, margin, loss, ga, gb);
}

extern "C" int dm_gather_rows(const float* table, int64_t D, const int64_t* idx, int64_t n, float* out, dm_stream_t stream) {
    if (n < 0 || D <= 0) return DM_ERR_BAD_ARG;
    if (n == 0) return DM_OK;
    if (!table || !idx || !out) return DM_ERR_BAD_ARG;
    return launch(loss::gather_rows_kernel, grid_for(n * 32), 256, 0, S(stream), table, (int)D, idx, n, out);
}
