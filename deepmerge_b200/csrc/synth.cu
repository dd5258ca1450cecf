// Synthetic scenes of SURVEY.md section 8(d), bit-identical to oracle/oracle_np.py
// (jittered-grid Voronoi labels, object-coherent image bands and embeddings).
// Bench / test utility: lets full-size scenes be created directly in HBM.
#include "common.cuh"
#include "../../include/deepmerge_b200_synth.h"

// libdeepmerge_b200_synth.so is linked on its own (bench / test utility, see the header): the few helpers of the product
// library it uses are defined here.
namespace dm {
thread_local int g_last_cuda_error = 0;
long long g_launch_count = 0;
int num_sms() {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
        return 148;
    return n;
}
}  // namespace dm


namespace dm {
namespace synth {

__host__ __device__ __forceinline__ uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}
__host__ __device__ __forceinline__ uint32_t hash32(uint32_t seed, uint32_t a, uint32_t b = 0, uint32_t c = 0) {
    uint32_t h = mix32(c + 0xc2b2ae35u);
    h = mix32((b + 0x85ebca6bu) ^ h);
    h = mix32((a + 0x9e3779b9u) ^ h);
    return mix32(seed ^ h);
}

struct Grid {
    int g, ncx, ncy;
    uint32_t seed;
    __device__ __forceinline__ void seed_of(int cx, int cy, long long& sx, long long& sy) const {
        sx = (long long)cx * g + hash32(seed, cx, cy, 0) % (uint32_t)g;
        sy = (long long)cy * g + hash32(seed, cx, cy, 1) % (uint32_t)g;
    }
    // nearest seed among the 3x3 neighbouring cells; ties -> lower id (ascending scan, strict <)
    __device__ __forceinline__ int nearest(long long x, long long y) const {
        int cx0 = (int)imin64(imax64(x / g, 0), ncx - 1);
        int cy0 = (int)imin64(imax64(y / g, 0), ncy - 1);
        long long best = 0x7fffffffffffffffll;
        int id = 0;
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
            for (int dx = -1; dx <= 1; ++dx) {
                const int cx = cx0 + dx, cy = cy0 + dy;
                if (cx < 0 || cx >= ncx || cy < 0 || cy >= ncy) continue;
                long long sx, sy;
                seed_of(cx, cy, sx, sy);
                const long long d = (x - sx) * (x - sx) + (y - sy) * (y - sy);
                if (d < best) { best = d; id = cy * ncx + cx; }
            }
        return id;
    }
};

static Grid make_grid(int64_t H, int64_t W, int64_t g, uint32_t seed) {
    Grid G;
    G.g = (int)g;
    G.ncx = (int)ceil_div(W, g);
    G.ncy = (int)ceil_div(H, g);
    G.seed = seed;
    return G;
}

__global__ void labels_kernel(int32_t* __restrict__ out, int64_t y0, int64_t rows, int64_t W, int64_t ld, Grid G) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < rows * W; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / W, x = i - r * W;
        out[r * ld + x] = G.nearest(x, y0 + r);
    }
}

__global__ void region_objects_kernel(int32_t* __restrict__ out, Grid G, Grid O) {
    const int n = G.ncx * G.ncy;
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < n; r += gridDim.x * blockDim.x) {
        long long sx, sy;
        G.seed_of(r % G.ncx, r / G.ncx, sx, sy);
        out[r] = O.nearest(sx, sy);
    }
}

__global__ void image_kernel(uint8_t* __restrict__ img, const int32_t* __restrict__ labels, int64_t y0, int64_t rows,
                             int64_t W, int64_t ld, int C, const int32_t* __restrict__ region_obj, uint32_t seed) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < rows * W; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / W, x = i - r * W;
        const int l = labels[r * ld + x];
        const uint32_t pix = (uint32_t)(((y0 + r) * W + x) & 0xffffffffll);
        for (int c = 0; c < C; ++c) {
            int v = 0;
            if (l >= 0) {
                const int obj = region_obj[l];
                const int col = 32 + (int)(hash32(seed + 2, obj, c) % 192u);
                const int off = (int)(hash32(seed + 3, l, c) % 9u) - 4;
                const int noi = (int)(hash32(seed + 4, pix, c) % 17u) - 8;
                v = min(255, max(0, col + off + noi));
            }
            img[i * C + c] = (uint8_t)v;
        }
    }
}

__global__ void points_kernel(int32_t* __restrict__ xs, int32_t* __restrict__ ys, int64_t H, int64_t W, Grid G, int P,
                              uint32_t seed) {
    const int64_t n = (int64_t)G.ncx * G.ncy * P;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / P), k = (int)(i - (int64_t)r * P);
        long long sx, sy;
        G.seed_of(r % G.ncx, r / G.ncx, sx, sy);
        long long dx = 0, dy = 0;
        if (k > 0) {
            const uint32_t span = G.g / 2 + 1;
            dx = (long long)(hash32(seed + 5, r, k, 0) % span) - G.g / 4;
            dy = (long long)(hash32(seed + 5, r, k, 1) % span) - G.g / 4;
        }
        xs[i] = (int32_t)imin64(imax64(sx + dx, 0), W - 1);
        ys[i] = (int32_t)imin64(imax64(sy + dy, 0), H - 1);
    }
}

__global__ void feats_kernel(float* __restrict__ feats, const int32_t* __restrict__ rop, const int32_t* __restrict__ region_obj,
                             const int64_t* __restrict__ point_ids, int64_t n, int D, uint32_t seed) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n * D; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p = i / D;
        const int d = (int)(i - p * D);
        const int r = rop[p];
        const int obj = r >= 0 ? region_obj[r] : 0;
        const uint32_t gid = (uint32_t)(point_ids ? point_ids[p] : p);   // global point id: the scene does not depend on sharding
        const uint32_t hc = hash32(seed + 6, obj, d), hn = hash32(seed + 7, gid, d);
        const int ci = (int)(hc & 0xffff) + (int)(hc >> 16) - 65535;
        const int ni = (int)(hn & 0xffff) + (int)(hn >> 16) - 65535;
        feats[i] = (float)(ci * 128 + ni) * (1.0f / 2097152.0f);
    }
}

}  // namespace synth
}  // namespace dm

using namespace dm;

extern "C" int dm_synth_labels(int32_t* labels, int64_t y0, int64_t rows, int64_t H, int64_t W, int64_t ld, int64_t g,
                               uint32_t seed, dm_stream_t stream) {
    if (!labels || rows < 0 || W <= 0 || H <= 0 || g <= 0 || ld < W) return DM_ERR_BAD_ARG;
    if (rows == 0) return DM_OK;
    return launch(synth::labels_kernel, grid_for(rows * W, 256, 16), 256, 0, S(stream), labels, y0, rows, W, ld,
        synth::make_grid(H, W, g, seed));
}

extern "C" int dm_synth_region_objects(int32_t* region_obj, int64_t H, int64_t W, int64_t g, uint32_t seed, dm_stream_t stream) {
    if (!region_obj || W <= 0 || H <= 0 || g <= 0) return DM_ERR_BAD_ARG;
    synth::Grid G = synth::make_grid(H, W, g, seed), O = synth::make_grid(H, W, 4 * g, seed + 1);
    return launch(synth::region_objects_kernel, grid_for((int64_t)G.ncx * G.ncy, 256, 16), 256, 0, S(stream), region_obj, G, O);
}

extern "C" int dm_synth_image(uint8_t* image, const int32_t* labels, int64_t y0, int64_t rows, int64_t W, int64_t ld,
                              int64_t C, const int32_t* region_obj, uint32_t seed, dm_stream_t stream) {
    if (!image || !labels || !region_obj || rows < 0 || W <= 0 || C <= 0 || ld < W) return DM_ERR_BAD_ARG;
    if (rows == 0) return DM_OK;
    return launch(synth::image_kernel, grid_for(rows * W, 256, 16), 256, 0, S(stream), image, labels, y0, rows, W, ld, (int)C,
        region_obj, seed);
}

extern "C" int dm_synth_points(int32_t* xs, int32_t* ys, int64_t H, int64_t W, int64_t g, int64_t P, uint32_t seed,
                               dm_stream_t stream) {
    if (!xs || !ys || W <= 0 || H <= 0 || g <= 0 || P <= 0) return DM_ERR_BAD_ARG;
    synth::Grid G = synth::make_grid(H, W, g, seed);
    return launch(synth::points_kernel, grid_for((int64_t)G.ncx * G.ncy * P, 256, 16), 256, 0, S(stream), xs, ys, H, W, G, (int)P,
        seed);
}

extern "C" int dm_synth_feats(float* feats, const int32_t* rop, const int32_t* region_obj, const int64_t* point_ids,
                              int64_t n, int64_t D, uint32_t seed, dm_stream_t stream) {
    if (n < 0 || D <= 0) return DM_ERR_BAD_ARG;
    if (n == 0) return DM_OK;
    if (!feats || !rop || !region_obj) return DM_ERR_BAD_ARG;
    return launch(synth::feats_kernel, grid_for(n * D, 256, 16), 256, 0, S(stream), feats, rop, region_obj, point_ids, n, (int)D,
        seed);
}
