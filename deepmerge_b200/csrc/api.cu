// Library-level entry points: version, errors, device query, exported primitives.
#include "common.cuh"
#include "prims.cuh"

namespace dm {
thread_local int g_last_cuda_error = 0;
long long g_launch_count = 0;

int num_sms() {
    static thread_local int cached_dev = -1, cached = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev != cached_dev) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached = n;
        cached_dev = dev;
    }
    return cached;
}
}  // namespace dm

using namespace dm;

extern "C" int dm_version(void) { return 100; }

extern "C" const char* dm_error_string(int code) {
    switch (code) {
        case DM_OK: return "ok";
        case DM_ERR_BAD_ARG: return "bad argument";
        case DM_ERR_WORKSPACE: return "workspace too small";
        case DM_ERR_CUDA: return "CUDA error (see dm_last_cuda_error)";
        case DM_ERR_UNSUPPORTED: return "unsupported device or driver";
        case DM_ERR_CAPACITY: return "capacity too small";
        default: return "unknown error";
    }
}

extern "C" int64_t dm_launch_count(void) { return (int64_t)__atomic_load_n(&g_launch_count, __ATOMIC_RELAXED); }
extern "C" void dm_launch_count_add(int64_t n) { __atomic_add_fetch(&g_launch_count, (long long)n, __ATOMIC_RELAXED); }

extern "C" int dm_last_cuda_error(void) { return g_last_cuda_error; }

extern "C" int dm_num_sms(void) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return DM_ERR_CUDA;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return DM_ERR_CUDA;
    return n;
}

extern "C" size_t dm_sort_edges_workspace_bytes(int64_t capacity) { return prims::ws_bytes(capacity, false); }

extern "C" int dm_sort_edges(uint64_t* keys, uint32_t* vals, const int64_t* n_dev, int64_t capacity, int64_t n_regions,
                             void* ws, size_t ws_bytes, dm_stream_t stream) {
    if (capacity < 0 || n_regions < 1) return DM_ERR_BAD_ARG;
    if (capacity == 0) return DM_OK;
    if (!keys || !n_dev || !ws) return DM_ERR_BAD_ARG;
    if (ws_bytes < prims::ws_bytes(capacity, false)) return DM_ERR_WORKSPACE;
    const int b = bits_for(n_regions);
    return prims::sort_pairs(keys, vals, n_dev, capacity, b, 2 * b, ws, S(stream));
}

extern "C" size_t dm_scan_workspace_bytes(int64_t capacity) { return prims::scan_ws_bytes(capacity); }

extern "C" int dm_scan_exclusive_u32(const uint32_t* in, uint32_t* out, const int64_t* n_dev, int64_t capacity,
                                     int64_t* total_dev, void* ws, size_t ws_bytes, dm_stream_t stream) {
    if (capacity < 0) return DM_ERR_BAD_ARG;
    if (capacity > 0 && (!in || !out || !n_dev || !ws)) return DM_ERR_BAD_ARG;
    if (ws_bytes < prims::scan_ws_bytes(capacity)) return DM_ERR_WORKSPACE;
    return prims::scan_exclusive_u32(in, out, n_dev, capacity, total_dev, ws, S(stream));
}
