// Scan / radix sort / run reduction (see prims.cuh).  Hand-written for sm_100a; no CUB.
#include <cstdio>
#include "prims.cuh"
#include <map>
#include <stdlib.h>
#include <string.h>
#include <utility>

namespace dm {
namespace prims {

// ------------------------------------------------------------------------------------ //
// exclusive scan: tile sums -> single-block scan of tile sums -> tile scan + offset; n = min(*n_dev, cap) as in the sorts
// ------------------------------------------------------------------------------------ //

__global__ void __launch_bounds__(SCAN_THREADS) scan_tile_sums(const uint32_t* __restrict__ in,
                                                               const int64_t* __restrict__ n_dev, int64_t cap,
                                                               uint32_t* __restrict__ tile_sum) {
    const int64_t n = imin64(*n_dev, cap);
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
    if (base >= n) return;
    uint32_t s = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        int64_t idx = base + i * SCAN_THREADS + threadIdx.x;
        if (idx < n) s += in[idx];
    }
    __shared__ uint32_t sm[SCAN_THREADS / 32 + 1];
    uint32_t total;
    block_excl_scan<SCAN_THREADS>(s, sm, total);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = total;
}

__global__ void __launch_bounds__(1024) scan_tile_offsets(uint32_t* __restrict__ tile_sum,
                                                          const int64_t* __restrict__ n_dev, int64_t cap,
                                                          int64_t* __restrict__ total_dev) {
    const int64_t n = imin64(*n_dev, cap);
    const int64_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    __shared__ uint32_t sm[1024 / 32 + 1];
    uint32_t carry = 0;
    for (int64_t b0 = 0; b0 < tiles; b0 += 1024) {
        int64_t b = b0 + threadIdx.x;
        uint32_t v = b < tiles ? tile_sum[b] : 0;
        uint32_t total;
        uint32_t ex = block_excl_scan<1024>(v, sm, total);
        if (b < tiles) tile_sum[b] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0 && total_dev) *total_dev = (int64_t)carry;
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_apply(const uint32_t* __restrict__ in, uint32_t* __restrict__ out,
                                                           const int64_t* __restrict__ n_dev, int64_t cap,
                                                           const uint32_t* __restrict__ tile_off) {
    const int64_t n = imin64(*n_dev, cap);
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
    if (base >= n) return;
    // blocked arrangement: thread t owns items [t*ITEMS, (t+1)*ITEMS)
    uint32_t v[SCAN_ITEMS];
    uint32_t s = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        int64_t idx = base + (int64_t)threadIdx.x * SCAN_ITEMS + i;
        v[i] = idx < n ? in[idx] : 0;
        s += v[i];
    }
    __shared__ uint32_t sm[SCAN_THREADS / 32 + 1];
    uint32_t total;
    uint32_t ex = block_excl_scan<SCAN_THREADS>(s, sm, total) + tile_off[blockIdx.x];
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        int64_t idx = base + (int64_t)threadIdx.x * SCAN_ITEMS + i;
        if (idx < n) out[idx] = ex;
        ex += v[i];
    }
}

size_t scan_ws_bytes(int64_t cap) {
    Carver c(nullptr);
    c.take<uint32_t>(ceil_div(imax64(cap, 1), SCAN_TILE) + 1);   // tile sums
    return c.used();
}

int scan_exclusive_u32(const uint32_t* in, uint32_t* out, const int64_t* n_dev, int64_t cap, int64_t* total_dev,
                       void* ws, cudaStream_t s) {
    if (cap <= 0) {
        if (total_dev) DM_CUDA(cudaMemsetAsync(total_dev, 0, sizeof(int64_t), s));
        return DM_OK;
    }
    uint32_t* tile_sum = (uint32_t*)ws;
    const unsigned tiles = (unsigned)ceil_div(cap, SCAN_TILE);
    DM_TRY(launch(scan_tile_sums, tiles, SCAN_THREADS, 0, s, in, n_dev, cap, tile_sum));
    DM_TRY(launch(scan_tile_offsets, 1, 1024, 0, s, tile_sum, n_dev, cap, total_dev));
    return launch(scan_apply, tiles, SCAN_THREADS, 0, s, in, out, n_dev, cap, tile_sum);
}

// ------------------------------------------------------------------------------------ //
// LSD radix sort, 9-bit digits.  Per pass: tile histograms, per-digit offsets over tiles, scatter.
// radix_sort_fused runs the whole sort (and, optionally, the run reduction that follows it) as ONE
// cooperative launch; persistent blocks walk their tiles and meet at grid barriers between the
// phases.  At the sizes of the graph stages (<= a few million pairs) a pass is launch/latency
// bound, so the 12 + 6 launches of a one-launch-per-phase driver collapse into one.
// Buffers written inside the fused kernel are read back with ld.global.cg (L2): L1 is not coherent
// across blocks and `const __restrict__` loads could take the non-coherent path.
// ------------------------------------------------------------------------------------ //
constexpr int RADIX_BITS = 9;
constexpr int RADIX = 1 << RADIX_BITS;
constexpr int SORT_WARPS = SORT_THREADS / 32;

__device__ __forceinline__ unsigned digit_of(uint64_t key, int id_bits, int shift) {
    uint64_t ck = ((key >> 32) << id_bits) | (key & ((1ull << id_bits) - 1));
    return (unsigned)(ck >> shift) & (unsigned)(RADIX - 1);
}
__device__ __forceinline__ uint64_t ldcg64(const uint64_t* p) { return __ldcg((const unsigned long long*)p); }

struct SortSmem {
    uint32_t wcnt[SORT_WARPS][RADIX];   // per-warp digit counters (the first row doubles as the tile histogram)
    uint32_t goff[RADIX];
    uint32_t scan[SORT_THREADS / 32 + 1];
};

// hist is digit-major: hist[d * tiles_cap + tile], so that the per-digit scan over tiles is coalesced
__device__ __forceinline__ void hist_tile(SortSmem& sm, const uint64_t* keys, int64_t n, int tile, int id_bits, int shift,
                                          uint32_t* hist, int tiles_cap) {
    uint32_t* h = sm.wcnt[0];
    for (int i = threadIdx.x; i < RADIX; i += SORT_THREADS) h[i] = 0;
    __syncthreads();
    const int64_t base = (int64_t)tile * SORT_TILE;
    uint64_t key[SORT_ITEMS];                              // all loads first: one round trip, not SORT_ITEMS
#pragma unroll
    for (int i = 0; i < SORT_ITEMS; ++i) {
        const int64_t idx = base + i * SORT_THREADS + threadIdx.x;
        key[i] = idx < n ? ldcg64(keys + idx) : 0;
    }
#pragma unroll
    for (int i = 0; i < SORT_ITEMS; ++i) {
        const int64_t idx = base + i * SORT_THREADS + threadIdx.x;
        if (idx < n) atomicAdd(&h[digit_of(key[i], id_bits, shift)], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < RADIX; i += SORT_THREADS) hist[(size_t)i * tiles_cap + tile] = h[i];
    __syncthreads();
}

// One warp per digit: turns the per-tile counts of that digit into an exclusive prefix over tiles
// (in place) and writes the digit's total to totals[d].  The digit bases (exclusive scan of the
// totals) are computed by every scatter block itself.
__device__ __forceinline__ void offsets_digit(uint32_t* hist, uint32_t* totals, int d, int tiles, int tiles_cap) {
    const int lane = threadIdx.x & 31;
    uint32_t* row = hist + (size_t)d * tiles_cap;
    uint32_t carry = 0;
    constexpr int UN = 8;                                  // 8 x 32 tiles in flight: the loads are the latency here
    for (int t0 = 0; t0 < tiles; t0 += 32 * UN) {
        uint32_t c[UN];
#pragma unroll
        for (int j = 0; j < UN; ++j) {
            const int t = t0 + 32 * j + lane;
            c[j] = t < tiles ? __ldcg(row + t) : 0;
        }
#pragma unroll
        for (int j = 0; j < UN; ++j) {
            const int t = t0 + 32 * j + lane;
            uint32_t inc = c[j];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += v;
            }
            if (t < tiles) row[t] = carry + inc - c[j];
            carry += __shfl_sync(0xffffffffu, inc, 31);
        }
    }
    if (lane == 0) totals[d] = carry;
}

__device__ __forceinline__ void scatter_tile(SortSmem& sm, const uint64_t* kin, const uint32_t* vin, uint64_t* kout,
                                             uint32_t* vout, int64_t n, int tile, int id_bits, int shift,
                                             const uint32_t* hist, const uint32_t* totals, int tiles_cap) {
    constexpr int PER = RADIX / SORT_THREADS;             // digits per thread in the block-wide steps
    const int64_t tile_base = (int64_t)tile * SORT_TILE;
    for (int i = threadIdx.x; i < SORT_WARPS * RADIX; i += SORT_THREADS) (&sm.wcnt[0][0])[i] = 0;
    {   // digit base = exclusive scan of the digit totals (thread t owns digits [t*PER, (t+1)*PER))
        uint32_t t[PER], sum = 0;
#pragma unroll
        for (int k = 0; k < PER; ++k) {
            t[k] = __ldcg(totals + threadIdx.x * PER + k);
            sum += t[k];
        }
        uint32_t tot;
        uint32_t base = block_excl_scan<SORT_THREADS>(sum, sm.scan, tot);
#pragma unroll
        for (int k = 0; k < PER; ++k) {
            const int d = threadIdx.x * PER + k;
            sm.goff[d] = base + __ldcg(hist + (size_t)d * tiles_cap + tile);
            base += t[k];
        }
    }
    __syncthreads();
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t wbase = tile_base + (int64_t)warp * (32 * SORT_ITEMS);
    uint64_t key[SORT_ITEMS];
    uint32_t val[SORT_ITEMS];
    uint32_t rank[SORT_ITEMS];
    unsigned dig[SORT_ITEMS];
#pragma unroll
    for (int i = 0; i < SORT_ITEMS; ++i) {
        const int64_t idx = wbase + i * 32 + lane;
        key[i] = idx < n ? ldcg64(kin + idx) : 0;
        val[i] = (vin && idx < n) ? __ldcg(vin + idx) : 0;     // with the keys: one round trip for all loads
    }
#pragma unroll
    for (int i = 0; i < SORT_ITEMS; ++i) {
        const int64_t idx = wbase + i * 32 + lane;
        const bool valid = idx < n;
        const unsigned vmask = __ballot_sync(0xffffffffu, valid);
        dig[i] = 0;
        rank[i] = 0;
        if (valid) {
            dig[i] = digit_of(key[i], id_bits, shift);
            const unsigned peers = __match_any_sync(vmask, dig[i]);
            const int leader = __ffs(peers) - 1;
            uint32_t pre = 0;
            if ((int)lane == leader) {
                pre = sm.wcnt[warp][dig[i]];
                sm.wcnt[warp][dig[i]] = pre + __popc(peers);
            }
            pre = __shfl_sync(peers, pre, leader);
            rank[i] = pre + __popc(peers & lanemask_lt());
        }
        __syncwarp();
    }
    __syncthreads();
    for (int d = threadIdx.x; d < RADIX; d += SORT_THREADS) {   // exclusive prefix over warps, per digit
        uint32_t run = 0;
#pragma unroll
        for (int w = 0; w < SORT_WARPS; ++w) {
            uint32_t c = sm.wcnt[w][d];
            sm.wcnt[w][d] = run;
            run += c;
        }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < SORT_ITEMS; ++i) {
        const int64_t idx = wbase + i * 32 + lane;
        if (idx < n) {
            const uint32_t pos = sm.goff[dig[i]] + sm.wcnt[warp][dig[i]] + rank[i];
            kout[pos] = key[i];
            if (vin) vout[pos] = val[i];
        }
    }
    __syncthreads();
}

// ---- the fused (single cooperative launch) driver ---------------------------------------

struct FusedArgs {
    uint64_t* k0; uint32_t* v0;          // the pairs (in place); v0 may be null
    uint64_t* k1; uint32_t* v1;          // ping-pong buffers
    const int64_t* n_dev; int64_t n_max; // n = min(*n_dev, n_max)
    uint32_t* hist; uint32_t* totals;
    unsigned* bar;                       // [0] arrivals (zeroed before the launch), [1] error flag
    int id_bits, passes, tiles_cap;
    // run reduction of the sorted pairs (do_unique): see sort_unique in prims.cuh
    int do_unique;
    const uint32_t* gather_lens;         // null: the sorted values are the lengths; else lengths / scores are
    const float* gather_scores;          //       gathered through the sorted values (a permutation)
    uint64_t sentinel;
    uint64_t* out_keys; uint32_t* out_lens; float* out_scores; int64_t* n_out;
    uint32_t* tile_heads;                // [tiles_cap]
    // optional copy of the reduced list back over caller arrays (after one more barrier)
    uint64_t* back_keys; uint32_t* back_lens; float* back_scores; int64_t* back_n;
};

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// All blocks of the (co-resident) grid meet here.  Arrivals only ever grow: barrier k completes at k * gridDim.x.
// The wait is bounded: a grid that cannot meet becomes an error + trap, not a hung GPU.
__device__ __forceinline__ void grid_barrier(unsigned* bar, unsigned& target) {
    __syncthreads();
    target += gridDim.x;
    if (threadIdx.x == 0) {
        // release / acquire at gpu scope; bar.sync on both sides extends the ordering to the whole block
        asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(bar), "r"(1u) : "memory");
        unsigned spins = 0;
        while (ld_acquire_u32(bar) < target) {
            if (++spins > (1u << 23)) {
                atomicExch(bar + 1, 1u);
                __trap();
            }
        }
    }
    __syncthreads();
}

__device__ __forceinline__ void lsd_body(const FusedArgs& A, SortSmem& sm, unsigned& target) {
    const int64_t n = imin64(*A.n_dev, A.n_max);
    const int tiles = (int)((n + SORT_TILE - 1) / SORT_TILE);
    const int G = (int)gridDim.x;
    uint64_t *ka = A.k0, *kb = A.k1;
    uint32_t *va = A.v0, *vb = A.v0 ? A.v1 : nullptr;
    for (int p = 0; p < A.passes; ++p) {
        const int shift = RADIX_BITS * p;
        for (int t = blockIdx.x; t < tiles; t += G) hist_tile(sm, ka, n, t, A.id_bits, shift, A.hist, A.tiles_cap);
        grid_barrier(A.bar, target);
        for (int d = blockIdx.x * SORT_WARPS + (threadIdx.x >> 5); d < RADIX; d += G * SORT_WARPS)
            offsets_digit(A.hist, A.totals, d, tiles, A.tiles_cap);
        grid_barrier(A.bar, target);
        for (int t = blockIdx.x; t < tiles; t += G)
            scatter_tile(sm, ka, va, kb, vb, n, t, A.id_bits, shift, A.hist, A.totals, A.tiles_cap);
        grid_barrier(A.bar, target);
        uint64_t* tk = ka; ka = kb; kb = tk;
        uint32_t* tv = va; va = vb; vb = tv;
    }
    if (!A.do_unique) {
        if (ka != A.k0) {                                  // odd number of passes: move the result home
            for (int64_t i = (int64_t)blockIdx.x * SORT_THREADS + threadIdx.x; i < n; i += (int64_t)G * SORT_THREADS) {
                A.k0[i] = ldcg64(ka + i);
                if (va) A.v0[i] = __ldcg(va + i);
            }
        }
        return;
    }
    // ---- run reduction: heads per tile -> (barrier) -> tile bases, in-tile scan, scatter + length sums ----
    // blocked arrangement: thread t owns items [t*ITEMS, (t+1)*ITEMS) of its tile
    for (int t = blockIdx.x; t < tiles; t += G) {
        const int64_t base = (int64_t)t * SORT_TILE + (int64_t)threadIdx.x * SORT_ITEMS;
        uint32_t heads = 0;
        uint64_t prev = (base > 0 && base - 1 < n) ? ldcg64(ka + base - 1) : 0;
        uint64_t key[SORT_ITEMS];
#pragma unroll
        for (int i = 0; i < SORT_ITEMS; ++i) key[i] = base + i < n ? ldcg64(ka + base + i) : 0;
#pragma unroll
        for (int i = 0; i < SORT_ITEMS; ++i) {
            const int64_t idx = base + i;
            if (idx < n) {
                heads += (key[i] != A.sentinel && (idx == 0 || key[i] != prev)) ? 1u : 0u;
                prev = key[i];
                A.out_lens[idx] = 0;
            }
        }
        uint32_t total;
        block_excl_scan<SORT_THREADS>(heads, sm.scan, total);
        if (threadIdx.x == 0) A.tile_heads[t] = total;
    }
    grid_barrier(A.bar, target);
    if (blockIdx.x == 0) {                                 // number of runs = heads in all tiles
        uint32_t part = 0, n_runs;
        for (int u = threadIdx.x; u < tiles; u += SORT_THREADS) part += __ldcg(A.tile_heads + u);
        block_excl_scan<SORT_THREADS>(part, sm.scan, n_runs);
        if (threadIdx.x == 0) *A.n_out = (int64_t)n_runs;
    }
    for (int t = blockIdx.x; t < tiles; t += G) {
        uint32_t part = 0, tile_base;                      // heads in the tiles before this one
        for (int u = threadIdx.x; u < t; u += SORT_THREADS) part += __ldcg(A.tile_heads + u);
        block_excl_scan<SORT_THREADS>(part, sm.scan, tile_base);
        const int64_t base = (int64_t)t * SORT_TILE + (int64_t)threadIdx.x * SORT_ITEMS;
        uint64_t key[SORT_ITEMS];
        uint32_t flag[SORT_ITEMS];
        uint32_t heads = 0;
        uint64_t prev = (base > 0 && base - 1 < n) ? ldcg64(ka + base - 1) : 0;
#pragma unroll
        for (int i = 0; i < SORT_ITEMS; ++i) {
            const int64_t idx = base + i;
            key[i] = idx < n ? ldcg64(ka + idx) : A.sentinel;
            flag[i] = (idx < n && key[i] != A.sentinel && (idx == 0 || key[i] != prev)) ? 1u : 0u;
            heads += flag[i];
            prev = key[i];
        }
        uint32_t src[SORT_ITEMS], len[SORT_ITEMS];          // every load before the first store (they may alias)
        float sc[SORT_ITEMS];
#pragma unroll
        for (int i = 0; i < SORT_ITEMS; ++i) {
            const int64_t idx = base + i;
            const bool live = idx < n && key[i] != A.sentinel;
            const uint32_t v = (live && va) ? __ldcg(va + idx) : 0u;
            src[i] = A.gather_lens ? v : (uint32_t)idx;
            len[i] = v;
        }
        if (A.gather_lens) {
#pragma unroll
            for (int i = 0; i < SORT_ITEMS; ++i) {
                const bool live = base + i < n && key[i] != A.sentinel;
                len[i] = live ? A.gather_lens[src[i]] : 0u;
                sc[i] = (live && flag[i] && A.gather_scores) ? A.gather_scores[src[i]] : 0.f;
            }
        }
        uint32_t total;
        uint32_t excl = block_excl_scan<SORT_THREADS>(heads, sm.scan, total) + tile_base;
        uint32_t acc = 0, acc_run = 0xffffffffu;            // lengths of one run are summed locally first
#pragma unroll
        for (int i = 0; i < SORT_ITEMS; ++i) {
            const int64_t idx = base + i;
            if (idx < n && key[i] != A.sentinel) {
                const uint32_t run = excl + flag[i] - 1;
                if (flag[i]) {
                    A.out_keys[run] = key[i];
                    if (A.gather_scores) A.out_scores[run] = sc[i];
                }
                if (run != acc_run) {
                    if (acc) atomicAdd(&A.out_lens[acc_run], acc);
                    acc = 0;
                    acc_run = run;
                }
                acc += len[i];
            }
            excl += flag[i];
        }
        if (acc) atomicAdd(&A.out_lens[acc_run], acc);
    }
    if (!A.back_keys) return;
    grid_barrier(A.bar, target);
    const int64_t m = (int64_t)__ldcg((const long long*)A.n_out);
    for (int64_t i = (int64_t)blockIdx.x * SORT_THREADS + threadIdx.x; i < m; i += (int64_t)G * SORT_THREADS) {
        A.back_keys[i] = ldcg64(A.out_keys + i);
        A.back_lens[i] = __ldcg(A.out_lens + i);
        if (A.back_scores && A.out_scores) A.back_scores[i] = __ldcg(A.out_scores + i);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && A.back_n) *A.back_n = m;
}

__global__ void __launch_bounds__(SORT_THREADS, 3) radix_sort_fused(const FusedArgs A) {
    __shared__ SortSmem sm;
    unsigned target = 0;
    lsd_body(A, sm, target);
}

// ------------------------------------------------------------------------------------ //
// Run reduction of an edge list WITHOUT sorting the raw entries (one cooperative launch, 4 grid barriers instead of
// the 14 of four LSD passes + reduction).  The raw list holds every edge a few times (per-warp tables of the raster
// pass, parallel edges after a merge); what is wanted is the sorted list of the UNIQUE keys with summed lengths:
//   0  clear a hash table sized for this call's n (16 B slots: key | length sum | smallest raw position)
//   A  every raw entry: CAS-insert its key, add its length, min its position; the inserter counts deg[lo]
//   B  exclusive scan of deg over the ids (chunk per block; chunk bases are summed by every block itself): the
//      unique keys of `lo` will occupy out[off[lo] .. off[lo] + deg[lo])  -- the output offsets are known before
//      anything is ordered
//   C  table slots -> bucket of their lo (any order inside the bucket)
//   D  every entry ranks itself among the deg[lo] (<= a handful in a planar graph) entries of its bucket and goes
//      to its final place.  Buckets above HUB_MIN entries are ranked by a whole block through shared memory.
// Fallback inside the same launch (decided after B, the raw list is still untouched): a bucket above HUB_MAX
// entries, more than HUB_CAP hubs, or an id outside [0, n_ids) -> the LSD radix path above.
// ------------------------------------------------------------------------------------ //
constexpr unsigned HUB_MIN = 48, HUB_MAX = 4096, HUB_CAP = 1024;
constexpr int HASH_MAX_GRID = 1024;
constexpr int HASH_BLOCKS_PER_SM = 4;
static_assert(HUB_MAX * sizeof(uint32_t) <= sizeof(SortSmem::wcnt), "hub staging aliases the sort counters");

struct HashArgs {
    FusedArgs F;
    uint4* tab; int tab_cap_log2;
    uint32_t *deg, *off, *cur;          // [n_ids]
    uint32_t* chunk_tot;                // [HASH_MAX_GRID]
    uint32_t* hubs;                     // [HUB_CAP]
    unsigned* misc;                     // [0] hubs, [1] fall back (zeroed before the launch)
    uint4* t_ent;                       // [cap] bucket entries: lo | hi | length | score bits
    uint2* t_bkt;                       // [cap] the entry's bucket: first position | size
    int64_t n_ids;
};

__device__ __forceinline__ void hashed_write(const FusedArgs& F, uint32_t p, const uint4& e) {
    const uint64_t key = ((uint64_t)e.x << 32) | e.y;
    F.out_keys[p] = key;
    F.out_lens[p] = e.z;
    if (F.out_scores) F.out_scores[p] = __uint_as_float(e.w);
    if (F.back_keys) {
        F.back_keys[p] = key;
        F.back_lens[p] = e.z;
        if (F.back_scores && F.out_scores) F.back_scores[p] = __uint_as_float(e.w);
    }
}

__device__ __forceinline__ void bucket_offsets_phase(const HashArgs& H, SortSmem& sm, int shift, unsigned hub_max) {
    const int64_t c0 = (int64_t)blockIdx.x << shift, c1 = imin64(H.n_ids, c0 + (1ll << shift));
    uint32_t carry = 0;
    for (int64_t t0 = c0; t0 < c1; t0 += SORT_THREADS) {
        const int64_t id = t0 + threadIdx.x;
        const uint32_t d = id < c1 ? __ldcg(H.deg + id) : 0u;
        if (d > HUB_MIN) {
            if (d > hub_max) {
                atomicExch(H.misc + 1, 1u);
            } else {
                const unsigned slot = atomicAdd(H.misc, 1u);
                if (slot < HUB_CAP) H.hubs[slot] = (uint32_t)id;
                else atomicExch(H.misc + 1, 1u);
            }
        }
        uint32_t tot;
        const uint32_t ex = block_excl_scan<SORT_THREADS>(d, sm.scan, tot);
        if (id < c1) H.off[id] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) H.chunk_tot[blockIdx.x] = carry;
}

__device__ __forceinline__ uint32_t bucket_chunk_bases(const HashArgs& H, SortSmem& sm, uint32_t* chunk_base) {
    const int G = (int)gridDim.x;
    uint32_t carry = 0;
    for (int t0 = 0; t0 < G; t0 += SORT_THREADS) {
        const int b = t0 + threadIdx.x;
        const uint32_t v = b < G ? __ldcg(H.chunk_tot + b) : 0u;
        uint32_t tot;
        const uint32_t ex = block_excl_scan<SORT_THREADS>(v, sm.scan, tot);
        if (b < G) chunk_base[b] = carry + ex;
        carry += tot;
    }
    __syncthreads();
    return carry;
}

__device__ __forceinline__ void phase_stamp(unsigned* misc, int k) {      // DM_HASH_TS=1 prints them (profiling aid)
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        ((unsigned long long*)(misc + 4))[k] = t;
    }
}

// Every global round trip of this kernel is a dependent L2 access, so each phase works on HB items per thread at a
// time: all loads (or atomics) of a step are issued before the first result is used.
constexpr int HB = 4;

__global__ void __launch_bounds__(SORT_THREADS, HASH_BLOCKS_PER_SM) edge_unique_hashed(const HashArgs H) {
    __shared__ SortSmem sm;
    __shared__ uint32_t chunk_base[HASH_MAX_GRID];
    const FusedArgs& F = H.F;
    const int64_t n = imin64(*F.n_dev, F.n_max);
    const int G = (int)gridDim.x;
    const int64_t gtid = (int64_t)blockIdx.x * SORT_THREADS + threadIdx.x, gstride = (int64_t)G * SORT_THREADS;
    unsigned target = 0;
    int logT = 10;
    while (logT < H.tab_cap_log2 && (1ll << logT) < n + n / 2 + 1) ++logT;
    const int64_t T = 1ll << logT;
    const uint32_t Tmask = (uint32_t)(T - 1);
    int shift = 0;                                         // ids per chunk = 1 << shift, at most G chunks
    while (((H.n_ids - 1) >> shift) >= G) ++shift;
    const bool want_sc = F.gather_lens && F.gather_scores && F.out_scores;
    // ---- 0: clear ----
    phase_stamp(H.misc, 0);
    for (int64_t i = gtid; i < T; i += gstride) H.tab[i] = make_uint4(~0u, ~0u, 0u, ~0u);
    for (int64_t i = gtid; i < H.n_ids; i += gstride) {
        H.deg[i] = 0;
        H.cur[i] = 0;
    }
    grid_barrier(F.bar, target);
    phase_stamp(H.misc, 1);
    // ---- A: insert ----
    for (int64_t i0 = gtid; i0 < n; i0 += HB * gstride) {
        uint64_t key[HB];
        uint32_t val[HB], h[HB];
        bool pend[HB];
#pragma unroll
        for (int u = 0; u < HB; ++u) {
            const int64_t i = i0 + u * gstride;
            key[u] = i < n ? ldcg64(F.k0 + i) : F.sentinel;
            val[u] = i < n ? __ldcg(F.v0 + i) : 0u;
        }
        if (F.gather_lens) {
#pragma unroll
            for (int u = 0; u < HB; ++u) val[u] = key[u] != F.sentinel ? F.gather_lens[val[u]] : 0u;
        }
        bool any = false;
#pragma unroll
        for (int u = 0; u < HB; ++u) {
            const uint32_t lo = (uint32_t)(key[u] >> 32);
            pend[u] = key[u] != F.sentinel;
            if (pend[u] && ((int64_t)lo >= H.n_ids || key[u] == ~0ull)) {
                atomicExch(H.misc + 1, 1u);
                pend[u] = false;
            }
            const uint64_t ck = ((uint64_t)lo << F.id_bits) | (uint32_t)key[u];
            h[u] = (uint32_t)((ck * 0x9E3779B97F4A7C15ull) >> (64 - logT));
            any |= pend[u];
        }
        while (any) {
            unsigned long long prev[HB];
#pragma unroll
            for (int u = 0; u < HB; ++u)
                if (pend[u]) prev[u] = atomicCAS((unsigned long long*)(H.tab + h[u]), ~0ull, (unsigned long long)key[u]);
            any = false;
#pragma unroll
            for (int u = 0; u < HB; ++u) {
                if (!pend[u]) continue;
                if (prev[u] == ~0ull) atomicAdd(H.deg + (uint32_t)(key[u] >> 32), 1u);
                if (prev[u] == ~0ull || prev[u] == key[u]) {
                    uint32_t* e = (uint32_t*)(H.tab + h[u]);
                    if (val[u]) atomicAdd(e + 2, val[u]);
                    if (want_sc) atomicMin(e + 3, (uint32_t)(i0 + u * gstride));
                    pend[u] = false;
                } else {
                    h[u] = (h[u] + 1) & Tmask;
                    any = true;
                }
            }
        }
    }
    grid_barrier(F.bar, target);
    phase_stamp(H.misc, 2);
    // ---- B: offsets inside this block's chunk of ids, hubs, chunk total ----
    bucket_offsets_phase(H, sm, shift, HUB_MAX);
    grid_barrier(F.bar, target);
    phase_stamp(H.misc, 3);
    if (__ldcg(H.misc + 1)) {                              // every block reads the same word after the same barrier
        lsd_body(F, sm, target);
        return;
    }
    const uint32_t n_unique = bucket_chunk_bases(H, sm, chunk_base);
    // ---- C: table -> buckets (any order inside a bucket) ----
    for (int64_t i0 = gtid; i0 < T; i0 += HB * gstride) {
        uint4 e[HB];
        uint32_t off[HB], m[HB], c[HB], pos[HB];
#pragma unroll
        for (int u = 0; u < HB; ++u) {
            const int64_t i = i0 + u * gstride;
            e[u] = i < T ? __ldcg(H.tab + i) : make_uint4(~0u, ~0u, 0u, 0u);
        }
#pragma unroll
        for (int u = 0; u < HB; ++u) {
            if (e[u].x == ~0u && e[u].y == ~0u) continue;
            off[u] = __ldcg(H.off + e[u].y);
            m[u] = __ldcg(H.deg + e[u].y);
            c[u] = atomicAdd(H.cur + e[u].y, 1u);
            pos[u] = want_sc ? __ldcg(F.v0 + e[u].w) : 0u;
        }
        if (want_sc) {
#pragma unroll
            for (int u = 0; u < HB; ++u)
                if (!(e[u].x == ~0u && e[u].y == ~0u)) pos[u] = __float_as_uint(F.gather_scores[pos[u]]);
        }
#pragma unroll
        for (int u = 0; u < HB; ++u) {
            if (e[u].x == ~0u && e[u].y == ~0u) continue;
            const uint32_t base = chunk_base[e[u].y >> shift] + off[u];
            H.t_ent[base + c[u]] = make_uint4(e[u].y, e[u].x, e[u].z, pos[u]);
            H.t_bkt[base + c[u]] = make_uint2(base, m[u]);
        }
    }
    grid_barrier(F.bar, target);
    phase_stamp(H.misc, 4);
    if (blockIdx.x == 0 && threadIdx.x == 0) {             // (every block has read *n_dev long ago: back_n may alias it)
        *F.n_out = (int64_t)n_unique;
        if (F.back_n) *F.back_n = (int64_t)n_unique;
    }
    // ---- D: every entry ranks itself inside its bucket ----
    for (int64_t e0 = (int64_t)blockIdx.x * (SORT_THREADS * 2) + threadIdx.x; e0 < (int64_t)n_unique; e0 += 2 * gstride) {
        uint4 ent[2];
        uint2 bk[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int64_t e = e0 + u * SORT_THREADS;
            ent[u] = e < (int64_t)n_unique ? __ldcg(H.t_ent + e) : make_uint4(0u, 0u, 0u, 0u);
            bk[u] = e < (int64_t)n_unique ? __ldcg(H.t_bkt + e) : make_uint2(0u, HUB_MAX);
        }
        uint32_t o[2][8];
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int k = 0; k < 8; ++k) o[u][k] = (uint32_t)k < bk[u].y && bk[u].y <= HUB_MIN ? __ldcg(&H.t_ent[bk[u].x + k].y) : ~0u;
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            if (bk[u].y > HUB_MIN) continue;               // a hub (or past the end)
            uint32_t rank = 0;
#pragma unroll
            for (int k = 0; k < 8; ++k) rank += o[u][k] < ent[u].y ? 1u : 0u;
            for (uint32_t k0 = 8; k0 < bk[u].y; k0 += 8) {
                uint32_t q[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) q[k] = k0 + k < bk[u].y ? __ldcg(&H.t_ent[bk[u].x + k0 + k].y) : ~0u;
#pragma unroll
                for (int k = 0; k < 8; ++k) rank += q[k] < ent[u].y ? 1u : 0u;
            }
            hashed_write(F, bk[u].x + rank, ent[u]);
        }
    }
    const unsigned n_hubs = __ldcg(H.misc);
    uint32_t* stage = &sm.wcnt[0][0];
    for (unsigned hb = blockIdx.x; hb < n_hubs; hb += G) {
        const uint32_t lo = __ldcg(H.hubs + hb);
        const uint32_t m = __ldcg(H.deg + lo);
        const uint32_t base = chunk_base[lo >> shift] + __ldcg(H.off + lo);
        __syncthreads();
        for (uint32_t j = threadIdx.x; j < m; j += SORT_THREADS) stage[j] = __ldcg(&H.t_ent[base + j].y);
        __syncthreads();
        for (uint32_t j = threadIdx.x; j < m; j += SORT_THREADS) {
            const uint32_t hi = stage[j];
            uint32_t rank = 0;
            for (uint32_t k = 0; k < m; ++k) rank += stage[k] < hi ? 1u : 0u;
            hashed_write(F, base + rank, __ldcg(H.t_ent + base + j));
        }
    }
    phase_stamp(H.misc, 5);
}

// ------------------------------------------------------------------------------------ //
// Stable sort of pairs by bucket + rank (same skeleton as edge_unique_hashed, no hash table): a pair goes to the
// bucket of its primary id (the high half of the key for key_bits = 2 id_bits, the low half for key_bits = id_bits)
// and ranks itself there by (secondary half, raw position).  Fast when the buckets are small -- the members of a
// merged component, the sample points of a region -- and takes the radix path when they are not.  With csr_offsets
// the bucket offsets come out as well (offsets[id] for id < n_ids; CSR of the sample points).
// ------------------------------------------------------------------------------------ //
constexpr unsigned HUB_MAX_SORT = 2048;
static_assert(HUB_MAX_SORT * sizeof(uint64_t) <= sizeof(SortSmem::wcnt), "hub staging aliases the sort counters");

struct BucketSortExtra {
    int by_low;
    int64_t* csr_offsets;
    int32_t* csr_ids;
};

__global__ void __launch_bounds__(SORT_THREADS, HASH_BLOCKS_PER_SM) bucket_sort_fused(const HashArgs H, const BucketSortExtra X) {
    __shared__ SortSmem sm;
    __shared__ uint32_t chunk_base[HASH_MAX_GRID];
    const FusedArgs& F = H.F;
    const int64_t n = imin64(*F.n_dev, F.n_max);
    const int G = (int)gridDim.x;
    const int64_t gtid = (int64_t)blockIdx.x * SORT_THREADS + threadIdx.x, gstride = (int64_t)G * SORT_THREADS;
    unsigned target = 0;
    int shift = 0;
    while (((H.n_ids - 1) >> shift) >= G) ++shift;
    // ---- 0: clear ----
    for (int64_t i = gtid; i < H.n_ids; i += gstride) {
        H.deg[i] = 0;
        H.cur[i] = 0;
    }
    grid_barrier(F.bar, target);
    // ---- A: bucket sizes ----
    for (int64_t i0 = gtid; i0 < n; i0 += HB * gstride) {
        uint64_t key[HB];
#pragma unroll
        for (int u = 0; u < HB; ++u) key[u] = i0 + u * gstride < n ? ldcg64(F.k0 + i0 + u * gstride) : 0ull;
#pragma unroll
        for (int u = 0; u < HB; ++u) {
            if (i0 + u * gstride >= n) continue;
            const uint32_t p = X.by_low ? (uint32_t)key[u] : (uint32_t)(key[u] >> 32);
            if ((int64_t)p >= H.n_ids) atomicExch(H.misc + 1, 1u);
            else atomicAdd(H.deg + p, 1u);
        }
    }
    grid_barrier(F.bar, target);
    bucket_offsets_phase(H, sm, shift, HUB_MAX_SORT);
    grid_barrier(F.bar, target);
    if (__ldcg(H.misc + 1)) {                              // the radix path, then the CSR outputs from the sorted list
        lsd_body(F, sm, target);
        if (!X.csr_offsets) return;
        grid_barrier(F.bar, target);
        for (int64_t id = gtid; id < H.n_ids; id += gstride) {
            int64_t a = 0, b = n;                          // first position whose primary id is >= id
            while (a < b) {
                const int64_t mid = (a + b) >> 1;
                const uint64_t k = ldcg64(F.k0 + mid);
                if ((int64_t)(X.by_low ? (uint32_t)k : (uint32_t)(k >> 32)) < id) a = mid + 1;
                else b = mid;
            }
            X.csr_offsets[id] = a;
        }
        if (X.csr_ids && F.v0)
            for (int64_t i = gtid; i < n; i += gstride) X.csr_ids[i] = (int32_t)__ldcg(F.v0 + i);
        return;
    }
    bucket_chunk_bases(H, sm, chunk_base);
    // ---- C: pairs -> buckets ----
    for (int64_t i0 = gtid; i0 < n; i0 += HB * gstride) {
        uint64_t key[HB];
        uint32_t val[HB], off[HB], m[HB], c[HB];
#pragma unroll
        for (int u = 0; u < HB; ++u) {
            const int64_t i = i0 + u * gstride;
            key[u] = i < n ? ldcg64(F.k0 + i) : 0ull;
            val[u] = (i < n && F.v0) ? __ldcg(F.v0 + i) : 0u;
        }
#pragma unroll
        for (int u = 0; u < HB; ++u) {
            if (i0 + u * gstride >= n) continue;
            const uint32_t p = X.by_low ? (uint32_t)key[u] : (uint32_t)(key[u] >> 32);
            off[u] = __ldcg(H.off + p);
            m[u] = __ldcg(H.deg + p);
            c[u] = atomicAdd(H.cur + p, 1u);
        }
#pragma unroll
        for (int u = 0; u < HB; ++u) {
            const int64_t i = i0 + u * gstride;
            if (i >= n) continue;
            const uint32_t p = X.by_low ? (uint32_t)key[u] : (uint32_t)(key[u] >> 32);
            const uint32_t sec = X.by_low ? (uint32_t)(key[u] >> 32) : (uint32_t)key[u];
            const uint32_t base = chunk_base[p >> shift] + off[u];
            H.t_ent[base + c[u]] = make_uint4(p, sec, val[u], (uint32_t)i);
            H.t_bkt[base + c[u]] = make_uint2(base, m[u]);
        }
    }
    grid_barrier(F.bar, target);
    // ---- D: rank by (secondary half, raw position); by_low: the secondary half is not part of the order ----
    auto token = [&](const uint4& e) { return ((uint64_t)(X.by_low ? 0u : e.y) << 32) | e.w; };
    auto put = [&](uint32_t pos, const uint4& e) {
        F.k0[pos] = X.by_low ? (((uint64_t)e.y << 32) | e.x) : (((uint64_t)e.x << 32) | e.y);
        if (F.v0) F.v0[pos] = e.z;
        if (X.csr_ids) X.csr_ids[pos] = (int32_t)e.z;
    };
    for (int64_t e0 = (int64_t)blockIdx.x * (SORT_THREADS * 2) + threadIdx.x; e0 < n; e0 += 2 * gstride) {
        uint4 ent[2];
        uint2 bk[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int64_t e = e0 + u * SORT_THREADS;
            ent[u] = e < n ? __ldcg(H.t_ent + e) : make_uint4(0u, 0u, 0u, 0u);
            bk[u] = e < n ? __ldcg(H.t_bkt + e) : make_uint2(0u, ~0u);
        }
        uint4 o[2][4];
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int k = 0; k < 4; ++k)
                o[u][k] = ((uint32_t)k < bk[u].y && bk[u].y <= HUB_MIN) ? __ldcg(H.t_ent + bk[u].x + k) : make_uint4(0u, ~0u, 0u, ~0u);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            if (bk[u].y > HUB_MIN) continue;
            const uint64_t tk = token(ent[u]);
            uint32_t rank = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) rank += ((uint32_t)k < bk[u].y && token(o[u][k]) < tk) ? 1u : 0u;
            for (uint32_t k0 = 4; k0 < bk[u].y; k0 += 4) {
                uint4 q[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) q[k] = k0 + k < bk[u].y ? __ldcg(H.t_ent + bk[u].x + k0 + k) : make_uint4(0u, ~0u, 0u, ~0u);
#pragma unroll
                for (int k = 0; k < 4; ++k) rank += (k0 + k < bk[u].y && token(q[k]) < tk) ? 1u : 0u;
            }
            put(bk[u].x + rank, ent[u]);
        }
    }
    const unsigned n_hubs = __ldcg(H.misc);
    uint64_t* stage = (uint64_t*)&sm.wcnt[0][0];
    for (unsigned hb = blockIdx.x; hb < n_hubs; hb += G) {
        const uint32_t id = __ldcg(H.hubs + hb);
        const uint32_t m = __ldcg(H.deg + id);
        const uint32_t base = chunk_base[id >> shift] + __ldcg(H.off + id);
        __syncthreads();
        for (uint32_t j = threadIdx.x; j < m; j += SORT_THREADS) stage[j] = token(__ldcg(H.t_ent + base + j));
        __syncthreads();
        for (uint32_t j = threadIdx.x; j < m; j += SORT_THREADS) {
            const uint64_t tk = stage[j];
            uint32_t rank = 0;
            for (uint32_t k = 0; k < m; ++k) rank += stage[k] < tk ? 1u : 0u;
            put(base + rank, __ldcg(H.t_ent + base + j));
        }
    }
    if (X.csr_offsets) {
        const int64_t c0 = (int64_t)blockIdx.x << shift, c1 = imin64(H.n_ids, c0 + (1ll << shift));
        for (int64_t id = c0 + threadIdx.x; id < c1; id += SORT_THREADS)
            X.csr_offsets[id] = (int64_t)chunk_base[blockIdx.x] + __ldcg(H.off + id);
    }
}


// ------------------------------------------------------------------------------------ //
// host side: one workspace layout, one cooperative launch per call
// ------------------------------------------------------------------------------------ //
namespace {
int ceil_log2_i64(int64_t x) {
    int l = 0;
    while ((1ll << l) < x) ++l;
    return l;
}
// ids the per-id arrays of a workspace sized for `cap` entries hold at least
int64_t hash_ids_cap(int64_t cap) { return 4 * cap + 65536; }
int hash_tab_log2(int64_t cap) { return ceil_log2_i64(imax64(1024, cap + cap / 2 + 1)); }

// The layout ws_bytes measures, carved into the workspace pointers of H; returns the bytes it spans.  The per-id
// arrays hold max(hash_ids_cap(cap), ids) ids; the tile heads and the hash table exist only for the run reduction.
size_t carve_ws(HashArgs& H, void* ws, int64_t cap, bool unique, int64_t ids) {
    FusedArgs& A = H.F;
    Carver c(ws);
    A.k1 = c.take<uint64_t>(cap);
    A.v1 = c.take<uint32_t>(cap);
    A.tiles_cap = (int)ceil_div(cap, SORT_TILE);
    A.hist = c.take<uint32_t>((size_t)A.tiles_cap * RADIX);
    A.totals = c.take<uint32_t>(RADIX);
    A.bar = c.take<unsigned>(2);
    if (unique) {
        A.tile_heads = c.take<uint32_t>(A.tiles_cap);
        H.tab_cap_log2 = hash_tab_log2(cap);
        H.tab = c.take<uint4>((size_t)1 << H.tab_cap_log2);
    }
    const size_t n_ids = (size_t)imax64(hash_ids_cap(cap), ids);
    H.deg = c.take<uint32_t>(n_ids);
    H.off = c.take<uint32_t>(n_ids);
    H.cur = c.take<uint32_t>(n_ids);
    H.chunk_tot = c.take<uint32_t>(HASH_MAX_GRID);
    H.hubs = c.take<uint32_t>(HUB_CAP);
    H.t_ent = c.take<uint4>(cap);
    H.t_bkt = c.take<uint2>(cap);
    H.misc = c.take<unsigned>(16);
    return c.used();
}

// Kernel arguments of one call: the carved workspace and the pairs (the run-reduction fields stay zero).
HashArgs make_args(void* ws, int64_t cap, bool unique, int64_t ws_ids, uint64_t* keys, uint32_t* vals,
                   const int64_t* n_dev, int id_bits, int key_bits, int64_t n_ids) {
    HashArgs H;
    memset(&H, 0, sizeof(H));
    carve_ws(H, ws, cap, unique, ws_ids);
    FusedArgs& A = H.F;
    A.k0 = keys; A.v0 = vals;
    A.n_dev = n_dev; A.n_max = cap;
    A.id_bits = id_bits; A.passes = (key_bits + RADIX_BITS - 1) / RADIX_BITS;
    H.n_ids = n_ids;
    return H;
}

// Blocks of `kernel` (SORT_THREADS threads) that are co-resident on the current device, at most per_sm_cap per SM;
// 0 when the device has no cooperative launch.
int coop_grid_limit(const void* kernel, int per_sm_cap) {
    static thread_local std::map<std::pair<int, const void*>, int> cache;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    const auto hit = cache.find({dev, kernel});
    if (hit != cache.end()) return hit->second;
    int coop = 0, per_sm = 0, limit = 0;
    if (cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev) == cudaSuccess && coop &&
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, SORT_THREADS, 0) == cudaSuccess)
        limit = (per_sm < per_sm_cap ? per_sm : per_sm_cap) * num_sms();
    cache[{dev, kernel}] = limit;
    return limit;
}

// Zeroes the grid barrier words (and, when given, the hub count and fall-back flag of misc) and launches `kernel`
// cooperatively on `grid` blocks.  grid < 1 means the device has no cooperative launch: DM_ERR_UNSUPPORTED.  A refused
// launch is DM_ERR_CUDA with the CUDA error recorded; there is no other path to fall back to.
template <typename... P>
int launch_coop(void (*kernel)(P...), int64_t grid, unsigned* bar, unsigned* misc, cudaStream_t s, const P&... args) {
    if (grid < 1) return DM_ERR_UNSUPPORTED;
    DM_CUDA(cudaMemsetAsync(bar, 0, 2 * sizeof(unsigned), s));
    if (misc) DM_CUDA(cudaMemsetAsync(misc, 0, 4 * sizeof(unsigned), s));
    return launch_cooperative(kernel, (unsigned)grid, SORT_THREADS, s, args...);
}

int launch_radix(FusedArgs& A, int64_t cap, cudaStream_t s) {
    // measured: a third block per SM costs more in the barriers than it saves in the phases
    const int64_t grid = imin64(ceil_div(cap, SORT_TILE), coop_grid_limit((const void*)radix_sort_fused, 2));
    return launch_coop(radix_sort_fused, grid, A.bar, nullptr, s, A);
}
}  // namespace

size_t ws_bytes(int64_t cap, bool unique, int64_t n_ids) {
    HashArgs H;
    return carve_ws(H, nullptr, imax64(cap, 1), unique, n_ids);
}

int sort_pairs(uint64_t* keys, uint32_t* vals, const int64_t* n_dev, int64_t cap, int id_bits, int key_bits, void* ws,
               cudaStream_t s, int64_t n_ids, int64_t* csr_offsets, int32_t* csr_ids) {
    if (cap <= 0) return DM_OK;
    if (id_bits < 1 || id_bits > 32 || key_bits < 1 || key_bits > 2 * id_bits) return DM_ERR_BAD_ARG;
    HashArgs H = make_args(ws, cap, false, n_ids, keys, vals, n_dev, id_bits, key_bits, n_ids);
    const bool bucket = n_ids > 0 && (key_bits == 2 * id_bits || key_bits == id_bits) && cap < (1ll << 31);
    if (!bucket) return csr_offsets ? DM_ERR_BAD_ARG : launch_radix(H.F, cap, s);
    BucketSortExtra X;
    X.by_low = key_bits == id_bits ? 1 : 0;
    X.csr_offsets = csr_offsets; X.csr_ids = csr_ids;
    // one id-scan tile per block, but not more than ~2.5 blocks per SM: beyond that the barriers cost more than the
    // shorter phases save (measured: 98 k members 31.6 us at 96 blocks, 20.5 at 383; 392 k points 24.3 us at 383
    // blocks, 26.4 at 592)
    const int64_t limit = imin64(coop_grid_limit((const void*)bucket_sort_fused, HASH_BLOCKS_PER_SM), HASH_MAX_GRID);
    const int64_t grid = imin64(imin64(ceil_div(imax64(cap, n_ids), SORT_THREADS), limit), 5 * num_sms() / 2);
    return launch_coop(bucket_sort_fused, grid, H.F.bar, H.misc, s, H, X);
}

int sort_unique(uint64_t* keys, uint32_t* vals, const int64_t* n_dev, int64_t cap, int id_bits, int key_bits, void* ws,
                const Reduce& r, cudaStream_t s, int64_t n_ids) {
    if (cap <= 0) {
        DM_CUDA(cudaMemsetAsync(r.out.n, 0, sizeof(int64_t), s));
        if (r.back.n) DM_CUDA(cudaMemsetAsync(r.back.n, 0, sizeof(int64_t), s));
        return DM_OK;
    }
    if (!vals || id_bits < 1 || id_bits > 32 || key_bits < 1 || key_bits > 2 * id_bits) return DM_ERR_BAD_ARG;
    HashArgs H = make_args(ws, cap, true, 0, keys, vals, n_dev, id_bits, key_bits, n_ids);
    FusedArgs& A = H.F;
    A.do_unique = 1;
    A.gather_lens = r.gather_lens; A.gather_scores = r.gather_lens ? r.gather_scores : nullptr;
    A.sentinel = r.sentinel;
    A.out_keys = r.out.keys; A.out_lens = r.out.lens; A.out_scores = r.out.scores; A.n_out = r.out.n;
    A.back_keys = r.back.keys; A.back_lens = r.back.lens; A.back_scores = r.back.scores; A.back_n = r.back.n;
    if (!(n_ids > 0 && n_ids <= hash_ids_cap(cap) && key_bits == 2 * id_bits && cap < (1ll << 31)))
        return launch_radix(A, cap, s);
    const int64_t limit = imin64(coop_grid_limit((const void*)edge_unique_hashed, HASH_BLOCKS_PER_SM), HASH_MAX_GRID);
    const int64_t grid = imin64(ceil_div(imax64(cap, n_ids), SORT_THREADS * 4), limit);
    DM_TRY(launch_coop(edge_unique_hashed, grid, A.bar, H.misc, s, H));
    static const bool print_ts = getenv("DM_HASH_TS") != nullptr;
    if (print_ts) {                                        // profiling aid: phase boundaries seen by block 0 (ns)
        unsigned long long t[6];
        cudaStreamSynchronize(s);
        cudaMemcpy(t, H.misc + 4, sizeof(t), cudaMemcpyDeviceToHost);
        fprintf(stderr, "edge_unique_hashed grid %d: clear %llu insert %llu offsets %llu buckets %llu rank %llu ns\n",
                (int)grid, t[1] - t[0], t[2] - t[1], t[3] - t[2], t[4] - t[3], t[5] - t[4]);
    }
    return DM_OK;
}

}  // namespace prims
}  // namespace dm
