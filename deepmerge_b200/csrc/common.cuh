// Shared helpers for the deepmerge_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/deepmerge_b200.h"

namespace dm {

extern thread_local int g_last_cuda_error;
extern long long g_launch_count;   // kernels accepted by the runtime from this library in this process

inline int cuda_fail(cudaError_t e) {
    g_last_cuda_error = (int)e;
    return DM_ERR_CUDA;
}

#define DM_CUDA(expr)                                   \
    do {                                                \
        cudaError_t _e = (expr);                        \
        if (_e != cudaSuccess) return dm::cuda_fail(_e); \
    } while (0)

#define DM_TRY(expr)             \
    do {                         \
        int _r = (expr);         \
        if (_r != DM_OK) return _r; \
    } while (0)

inline cudaStream_t S(dm_stream_t s) { return (cudaStream_t)s; }

__host__ __device__ inline long long imin64(long long a, long long b) { return a < b ? a : b; }
__host__ __device__ inline long long imax64(long long a, long long b) { return a > b ? a : b; }

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

int num_sms();

// Grid of a grid-stride kernel: one thread per item, but at most per_sm blocks per SM.
inline unsigned grid_for(int64_t items, int threads = 256, int per_sm = 8) {
    return (unsigned)imax64(1, imin64(ceil_div(items, threads), (int64_t)num_sms() * per_sm));
}

// Outcome of a launch whose own result is e: the thread's CUDA error is read and cleared, so a refused launch is
// reported once, as DM_ERR_CUDA, and is not seen again by the next check of this library or of the caller.  Only a
// launch the runtime accepted is counted.
inline int launched(cudaError_t e) {
    const cudaError_t pending = cudaGetLastError();
    if (e == cudaSuccess) e = pending;
    if (e != cudaSuccess) return cuda_fail(e);
    __atomic_add_fetch(&g_launch_count, 1, __ATOMIC_RELAXED);
    return DM_OK;
}

// Keeps P out of template argument deduction: the kernel alone fixes the parameter types, and the arguments are
// converted to them at the call, as in a triple-chevron launch.
template <typename T> struct param { using type = T; };

// Every kernel of the library is launched through here or launch_cooperative.  Dynamic shared memory above the 48 KB
// a kernel gets by default is opted into first.
template <typename... P>
int launch(void (*k)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, typename param<P>::type... args) {
    if (smem > 48 * 1024) DM_CUDA(cudaFuncSetAttribute((const void*)k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<grid, block, smem, s>>>(args...);
    return launched(cudaSuccess);
}

// A kernel whose blocks meet at grid-wide barriers: the runtime refuses the launch unless all of grid fits on the GPU
// at once.
template <typename... P>
int launch_cooperative(void (*k)(P...), dim3 grid, dim3 block, cudaStream_t s, typename param<P>::type... args) {
    void* argv[] = {(void*)&args...};
    return launched(cudaLaunchCooperativeKernel((const void*)k, grid, block, argv, 0, s));
}

// Carves a caller-provided workspace into 256-byte aligned pieces.  Each workspace has one layout function that takes
// its pieces in order and returns them with used(): from the caller's base it gives the pieces, from a null base the
// bytes they span, which is what the workspace query returns.
struct Carver {
    char* base;
    size_t off = 0;
    explicit Carver(void* p) : base((char*)p) {}
    template <typename T>
    T* take(size_t n) {
        off = align_up(off, 256);
        T* r = (T*)(base + off);
        off += n * sizeof(T);
        return r;
    }
    size_t used() const { return align_up(off, 256); }
};

__device__ __forceinline__ uint64_t pack_key(int a, int b) {
    unsigned lo = (unsigned)min(a, b), hi = (unsigned)max(a, b);
    return ((uint64_t)lo << 32) | hi;
}
__device__ __forceinline__ int key_lo(uint64_t k) { return (int)(k >> 32); }
__device__ __forceinline__ int key_hi(uint64_t k) { return (int)(k & 0xffffffffu); }

__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ unsigned lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// streaming 128-bit global accesses that do not allocate in L1
__device__ __forceinline__ int4 ldg_stream(const int4* p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream(int4* p, const int4& v) {
    asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// number of bits needed to represent ids in [0, n)
inline int bits_for(int64_t n) {
    int b = 1;
    while (b < 32 && ((int64_t)1 << b) < n) ++b;
    return b;
}

}  // namespace dm
