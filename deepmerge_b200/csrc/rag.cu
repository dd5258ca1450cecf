// R1: region adjacency graph from a label raster, fused with per-region band pooling -- host side and C ABI.
// The raster kernel is rag_blocks.cu (per-block arithmetic in rag_core.cuh, hash tables in rag_tables.cuh); this file
// encodes the tensor maps, carves the workspace and chains the raster pass with the sort / run reduction of the raw
// (edge key, count) entries (prims.cu).
#include "rag_common.cuh"
#include "prims.cuh"

namespace dm {
namespace rag {

// ------------------------------------------------------------------------------------ //
// host side
// ------------------------------------------------------------------------------------ //
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

static thread_local int g_last_path = -1;     // 1 = TMA staging, 0 = ld.global staging
static thread_local int g_last_encode_error = 0;
int last_path() { return g_last_path; }
void set_last_path(int path) { g_last_path = path; }
int last_encode_error() { return g_last_encode_error; }

bool make_map_2d(CUtensorMap* m, const void* base, uint64_t dim0, uint64_t dim1, uint64_t pitch_bytes,
                        uint32_t box0, uint32_t box1) {
    EncodeTiledFn enc = get_encode();
    if (!enc) {
        g_last_encode_error = -1;
        return false;
    }
    cuuint64_t dims[2] = {dim0, dim1};
    cuuint64_t strides[1] = {pitch_bytes};
    cuuint32_t box[2] = {box0, box1};
    cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_INT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    g_last_encode_error = (int)r;
    return r == CUDA_SUCCESS;
}

}  // namespace rag
}  // namespace dm

using namespace dm;

extern "C" int dm_rag_last_path(void) { return rag::last_path(); }
extern "C" int dm_rag_last_encode_error(void) { return rag::last_encode_error(); }

namespace {
struct RagWs {
    uint64_t* raw_keys;
    uint32_t* raw_cnt;
    void* sort;
    size_t bytes;
};
RagWs rag_ws(void* base, int64_t capacity) {
    const int64_t cap = imax64(capacity, 1);
    Carver c(base);
    return {c.take<uint64_t>(cap), c.take<uint32_t>(cap), c.take<char>(prims::ws_bytes(cap, true)), c.used()};
}
}  // namespace

extern "C" size_t dm_rag_workspace_bytes(int64_t capacity) { return rag_ws(nullptr, capacity).bytes; }

extern "C" int dm_rag_scan(const int32_t* labels, int64_t rows_own, int64_t rows_avail, int64_t W, int64_t ld,
                           const uint8_t* image, int64_t C, int64_t image_pitch, int64_t n_regions, int top_border,
                           int bottom_border, int64_t* area, int64_t* border, uint64_t* band_sum, uint64_t* band_sumsq,
                           int64_t capacity, int64_t* counts, void* ws, size_t ws_bytes, dm_stream_t stream) {
    if (rows_own < 0 || W < 0 || ld < W || n_regions < 0 || n_regions > 0x7fffffff || capacity < 0) return DM_ERR_BAD_ARG;
    if (rows_avail != rows_own && rows_avail != rows_own + 1) return DM_ERR_BAD_ARG;
    if (rows_own > 0x7ffffff0 || W > 0x7ffffff0) return DM_ERR_BAD_ARG;
    if (!counts) return DM_ERR_BAD_ARG;
    if (!image) C = 0;
    if (C < 0 || C > 4) return DM_ERR_BAD_ARG;
    if (C > 0 && (!band_sum || !band_sumsq || image_pitch < W * C)) return DM_ERR_BAD_ARG;
    const bool empty = rows_own == 0 || W == 0;
    const RagWs w = rag_ws(ws, capacity);
    if (!empty) {
        if (!labels || !area || !border || !ws) return DM_ERR_BAD_ARG;
        if (ws_bytes < w.bytes) return DM_ERR_WORKSPACE;
    }
    cudaStream_t s = S(stream);
    DM_CUDA(cudaMemsetAsync(counts, 0, 4 * sizeof(int64_t), s));
    if (empty) return DM_OK;
    rag::Params P;
    P.labels = labels;
    P.ld = ld;
    P.image = image;
    P.image_pitch = image_pitch;
    P.rows_own = (int)rows_own;
    P.rows_avail = (int)rows_avail;
    P.W = (int)W;
    P.n_regions = (int)n_regions;
    P.top_border = top_border;
    P.bottom_border = bottom_border;
    P.area = (unsigned long long*)area;
    P.border = (unsigned long long*)border;
    P.bsum = (unsigned long long*)band_sum;
    P.bsq = (unsigned long long*)band_sumsq;
    P.raw_keys = (unsigned long long*)w.raw_keys;
    P.raw_cnt = w.raw_cnt;
    P.capacity = capacity;
    P.counters = (unsigned long long*)counts;
    P.tiles_x = P.tiles_y = P.tiles_per_cta = 0;
    return rag::run_blocks(P, (int)C, s);
}

extern "C" int dm_rag_finish(uint64_t* edge_keys, uint32_t* boundary_len, int64_t capacity, int64_t n_regions,
                             int64_t* counts, void* ws, size_t ws_bytes, dm_stream_t stream) {
    if (capacity < 0 || n_regions < 0 || !counts) return DM_ERR_BAD_ARG;
    if (capacity == 0) return DM_OK;
    if (!edge_keys || !boundary_len || !ws) return DM_ERR_BAD_ARG;
    const RagWs w = rag_ws(ws, capacity);
    if (ws_bytes < w.bytes) return DM_ERR_WORKSPACE;
    prims::Reduce r;
    r.out = {edge_keys, boundary_len, nullptr, counts};
    const int b = bits_for(n_regions);
    // counts[1] may exceed capacity (an overflowed raw list): sort_unique reads min(counts[1], capacity) entries
    return prims::sort_unique(w.raw_keys, w.raw_cnt, counts + 1, capacity, b, 2 * b, w.sort, r, S(stream), n_regions);
}

extern "C" int dm_rag_build(const int32_t* labels, int64_t rows_own, int64_t rows_avail, int64_t W, int64_t ld,
                            const uint8_t* image, int64_t C, int64_t image_pitch, int64_t n_regions, int top_border,
                            int bottom_border, int64_t* area, int64_t* border, uint64_t* band_sum, uint64_t* band_sumsq,
                            uint64_t* edge_keys, uint32_t* boundary_len, int64_t capacity, int64_t* counts, void* ws,
                            size_t ws_bytes, dm_stream_t stream) {
    if (capacity > 0 && (!edge_keys || !boundary_len)) return DM_ERR_BAD_ARG;
    DM_TRY(dm_rag_scan(labels, rows_own, rows_avail, W, ld, image, C, image_pitch, n_regions, top_border, bottom_border,
                       area, border, band_sum, band_sumsq, capacity, counts, ws, ws_bytes, stream));
    if (rows_own == 0 || W == 0) return DM_OK;
    return dm_rag_finish(edge_keys, boundary_len, capacity, n_regions, counts, ws, ws_bytes, stream);
}

namespace dm {
namespace rag {
__global__ void concat_kernel(const uint64_t* __restrict__ sk, const uint32_t* __restrict__ sl,
                              const int64_t* __restrict__ counts, int n_lists, int64_t slot_cap,
                              uint64_t* __restrict__ dk, uint32_t* __restrict__ dl, int64_t dst_cap,
                              int64_t* __restrict__ n_out) {
    // every thread recomputes the (few) slot offsets; lists are short compared with the grid-stride work
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)n_lists * slot_cap;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int g = (int)(i / slot_cap);
        const int64_t j = i - (int64_t)g * slot_cap;
        if (j >= counts[g]) continue;
        int64_t off = 0;
        for (int h = 0; h < g; ++h) off += imin64(counts[h], slot_cap);
        if (off + j < dst_cap) {
            dk[off + j] = sk[i];
            dl[off + j] = sl[i];
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        int64_t tot = 0, bad = 0;
        for (int h = 0; h < n_lists; ++h) {
            if (counts[h] > slot_cap) bad = 1;
            tot += imin64(counts[h], slot_cap);
        }
        if (tot > dst_cap) { bad = 1; tot = dst_cap; }
        n_out[0] = tot;
        n_out[1] = bad;
    }
}
}  // namespace rag
}  // namespace dm

extern "C" int dm_edges_concat(const uint64_t* src_keys, const uint32_t* src_lens, const int64_t* counts, int64_t n_lists,
                               int64_t slot_capacity, uint64_t* dst_keys, uint32_t* dst_lens, int64_t dst_capacity,
                               int64_t* n_out_dev, dm_stream_t stream) {
    if (n_lists < 0 || n_lists > 4096 || slot_capacity < 0 || dst_capacity < 0 || !n_out_dev) return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    if (n_lists == 0 || slot_capacity == 0) {
        DM_CUDA(cudaMemsetAsync(n_out_dev, 0, 2 * sizeof(int64_t), s));
        return DM_OK;
    }
    if (!src_keys || !src_lens || !counts || !dst_keys || !dst_lens) return DM_ERR_BAD_ARG;
    return launch(rag::concat_kernel, grid_for(n_lists * slot_capacity), 256, 0, s, src_keys, src_lens, counts, (int)n_lists,
        slot_capacity, dst_keys, dst_lens, dst_capacity, n_out_dev);
}

namespace {
struct UniqueWs {
    uint64_t* out_keys;
    uint32_t* out_lens;
    int64_t* n_new;
    void* sort;
    size_t bytes;
};
UniqueWs edges_unique_ws(void* base, int64_t capacity) {
    const int64_t cap = imax64(capacity, 1);
    Carver c(base);
    return {c.take<uint64_t>(cap), c.take<uint32_t>(cap), c.take<int64_t>(1), c.take<char>(prims::ws_bytes(cap, true)),
            c.used()};
}
}  // namespace

extern "C" size_t dm_edges_unique_workspace_bytes(int64_t capacity) { return edges_unique_ws(nullptr, capacity).bytes; }

extern "C" int dm_edges_sort_unique(uint64_t* keys, uint32_t* lens, const int64_t* n_in, int64_t capacity, int64_t n_regions,
                                    int64_t* n_out, void* ws, size_t ws_bytes, dm_stream_t stream) {
    if (capacity < 0 || n_regions < 0 || !n_out) return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    if (capacity == 0) {
        DM_CUDA(cudaMemsetAsync(n_out, 0, sizeof(int64_t), s));
        return DM_OK;
    }
    if (!keys || !lens || !n_in || !ws) return DM_ERR_BAD_ARG;
    const UniqueWs w = edges_unique_ws(ws, capacity);
    if (ws_bytes < w.bytes) return DM_ERR_WORKSPACE;
    prims::Reduce r;
    r.out = {w.out_keys, w.out_lens, nullptr, w.n_new};
    r.back = {keys, lens, nullptr, n_out};
    const int b = bits_for(n_regions);
    return prims::sort_unique(keys, lens, n_in, capacity, b, 2 * b, w.sort, r, s, n_regions);
}
