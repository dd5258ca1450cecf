// Device-wide primitives used by the graph stages: exclusive scan, stable LSD radix
// sort of packed edge keys, and sorted-run reduction (unique + sum).  All take their
// element count from device memory so that stages chain without host round trips.
#pragma once
#include "common.cuh"

namespace dm {
namespace prims {

constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

constexpr int SORT_THREADS = 256;
constexpr int SORT_ITEMS = 8;
constexpr int SORT_TILE = SORT_THREADS * SORT_ITEMS;

// Workspace of scan_exclusive_u32 over `cap` items (at least one).
size_t scan_ws_bytes(int64_t cap);
int scan_exclusive_u32(const uint32_t* in, uint32_t* out, const int64_t* n_dev, int64_t cap,
                       int64_t* total_dev, void* ws, cudaStream_t s);

// sort_pairs and sort_unique each run as ONE cooperative launch (persistent blocks meeting at grid barriers).  On a
// device without cooperative launch they return DM_ERR_UNSUPPORTED; a refused launch is DM_ERR_CUDA with the CUDA
// error recorded.  Which kernel runs depends on the input only.

// Workspace of sort_pairs (unique = false) or sort_unique (unique = true; adds the tile heads and the hash table of
// the run reduction) over `cap` pairs.  Its per-id arrays hold max(4 cap + 65536, n_ids) ids.
size_t ws_bytes(int64_t cap, bool unique, int64_t n_ids = 0);

// Stable sort of (keys, vals) in place by the low key_bits bits of the compacted key ((hi32 << id_bits) | lo32); both
// 32-bit halves of every key must be < 2^id_bits.  key_bits = 2*id_bits sorts by (hi, lo); key_bits = id_bits sorts by
// lo only.  n = min(*n_dev, cap) pairs; vals may be null; ws holds ws_bytes(cap, false, n_ids) bytes.
// n_ids > 0 with key_bits = id_bits or 2 id_bits and cap < 2^31: the sort runs as bucket + rank (bucket_sort_fused in
// prims.cu), one bucket per primary id (the lo half for id_bits, hi for 2 id_bits) below n_ids; it takes the radix
// path inside the same launch when a bucket is too large or an id is >= n_ids.  Otherwise: the LSD radix sort
// (radix_sort_fused).  csr_offsets / csr_ids need the bucket sort (DM_ERR_BAD_ARG otherwise): they also receive
// offsets[id] = first sorted position of primary id `id`, for id < n_ids, and the sorted values as int32.
int sort_pairs(uint64_t* keys, uint32_t* vals, const int64_t* n_dev, int64_t cap, int id_bits, int key_bits,
               void* ws, cudaStream_t s, int64_t n_ids = 0, int64_t* csr_offsets = nullptr, int32_t* csr_ids = nullptr);

// A list of runs: keys[r], lens[r], scores[r] for r < *n.
struct RunList {
    uint64_t* keys = nullptr;
    uint32_t* lens = nullptr;
    float* scores = nullptr;
    int64_t* n = nullptr;
};

// What sort_unique gathers and drops, and where it writes the runs.  The defaults gather nothing and drop nothing
// (~0 is not the key of two ids below 2^31).
struct Reduce {
    RunList out;                              // keys, lens and n are required; scores is written when set
    RunList back;                             // a copy of out, e.g. over the input arrays: see sort_unique
    const uint32_t* gather_lens = nullptr;
    const float* gather_scores = nullptr;
    uint64_t sentinel = ~0ull;
};

// Sort + run reduction of n = min(*n_dev, cap) pairs; ws holds ws_bytes(cap, true) bytes.  For every run of equal keys
// (runs of r.sentinel are dropped), in ascending key order:
//   out.keys[i] = key, out.lens[i] = sum of the run's lengths, out.scores[i] = score of the run's first pair;
// *out.n = number of runs.  r.gather_lens == null: the values are the lengths.  Otherwise the values are a permutation
// and lengths / scores are gathered through it (gather_lens[vals[i]], gather_scores[vals[i]]; out.scores needs
// gather_scores).  r.back.keys set: the keys and lens of the list are copied there, and the scores when both out.scores
// and back.scores are set; r.back.n set: the number of runs is written there too.  keys / vals are left sorted or
// untouched.
// n_ids in (0, 4 cap + 65536] with key_bits = 2 id_bits and cap < 2^31: both halves of every key that is not the
// sentinel are ids < n_ids, and the run reduction goes through a hash table + per-id buckets without sorting the raw
// pairs (edge_unique_hashed in prims.cu), which takes the radix path inside the same launch when a bucket is too large
// or an id is out of range.  Otherwise: the LSD radix sort of the pairs, then the reduction (radix_sort_fused).
int sort_unique(uint64_t* keys, uint32_t* vals, const int64_t* n_dev, int64_t cap, int id_bits, int key_bits, void* ws,
                const Reduce& r, cudaStream_t s, int64_t n_ids = 0);

// ---- device helpers -------------------------------------------------------------------

// Block-wide exclusive scan of one uint32 per thread.  smem needs NT/32 + 1 words.
template <int NT>
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t* smem, uint32_t& total) {
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
    }
    if (lane == 31) smem[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = lane < NT / 32 ? smem[lane] : 0;
        uint32_t winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= (unsigned)o) winc += t;
        }
        if (lane < NT / 32) smem[lane] = winc - w;
        if (lane == 31) smem[NT / 32] = winc;
    }
    __syncthreads();
    uint32_t r = smem[warp] + inc - v;
    total = smem[NT / 32];
    __syncthreads();
    return r;
}

}  // namespace prims
}  // namespace dm
