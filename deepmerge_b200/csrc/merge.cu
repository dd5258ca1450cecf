// R9: merge loop building blocks -- selection, lock-free union-find with minimum-id roots,
// merged statistics with a deterministic fp32 summation order, edge re-keying, and the
// final LUT relabel of the raster.  Spec: SURVEY.md section 8(a) R9 (the reference only
// scores edges, ExtractFeatures.py:150-225, and never merges).
#include "common.cuh"
#include "prims.cuh"

namespace dm {
namespace merge {

// ---- selection ------------------------------------------------------------------------
template <bool MLP>
__global__ void select_kernel(const float* __restrict__ v, float tau, int n_out, const int64_t* __restrict__ n_dev,
                              uint8_t* __restrict__ selected, unsigned long long* __restrict__ n_sel) {
    const int64_t n = *n_dev;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t start = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int64_t e0 = start - threadIdx.x % 32; e0 < n; e0 += stride) {
        const int64_t e = e0 + threadIdx.x % 32;
        bool sel = false;
        if (e < n) {
            if (MLP) sel = v[e * n_out + 1] > v[e * n_out];   // argmax == 1 (ties go to class 0)
            else sel = v[e] < tau;
            selected[e] = sel ? 1 : 0;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, sel);
        if (bal && (threadIdx.x & 31) == 0) atomicAdd(n_sel, (unsigned long long)__popc(bal));
    }
}

// ---- union-find ---------------------------------------------------------------------------
__device__ __forceinline__ int uf_find(const int32_t* parent, int x) {
    int p = ((const volatile int32_t*)parent)[x];
    while (p != x) {
        x = p;
        p = ((const volatile int32_t*)parent)[x];
    }
    return x;
}

// Hook the larger root under the smaller with atomicCAS and retry on contention: parent[x] <= x
// always holds, so there are no cycles and every tree's root is its component's minimum id.
__global__ void uf_union_kernel(int32_t* __restrict__ parent, const uint64_t* __restrict__ keys,
                                const uint8_t* __restrict__ selected, const int64_t* __restrict__ n_dev) {
    const int64_t n = *n_dev;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        if (!selected[e]) continue;
        const uint64_t k = keys[e];
        int a = uf_find(parent, key_lo(k));
        int b = uf_find(parent, key_hi(k));
        while (a != b) {
            if (a > b) { int t = a; a = b; b = t; }          // a < b: hook b under a
            const int old = atomicCAS(&parent[b], b, a);
            if (old == b) break;
            b = uf_find(parent, old);                         // b got hooked elsewhere meanwhile
            a = uf_find(parent, a);
        }
    }
}

__device__ __forceinline__ void uf_unite(int32_t* parent, int a, int b) {
    a = uf_find(parent, a);
    b = uf_find(parent, b);
    while (a != b) {
        if (a > b) { int t = a; a = b; b = t; }
        const int old = atomicCAS(&parent[b], b, a);
        if (old == b) break;
        b = uf_find(parent, old);
        a = uf_find(parent, a);
    }
}

// Distributed union-find, frontier exchange.  A component can span two row tiles only through a region both ranks see,
// so after the local unions every rank publishes, for each alive component it shares with another rank, the pair
// (component, its local root); every rank then unites ALL ranks' pairs into its own forest.  The pairs carry the whole
// cross-rank connectivity (a local root is the minimum id of its local component, and the global minimum is the minimum
// of the local roots), so no iteration and no convergence test are needed.
__global__ void shard_frontier_pairs_kernel(const int32_t* __restrict__ parent, const uint8_t* __restrict__ alive,
                                            const int32_t* __restrict__ mask, int my_bit, int64_t R,
                                            uint64_t* __restrict__ pairs, int64_t cap, unsigned long long* __restrict__ n_out) {
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < R; x += (int64_t)gridDim.x * blockDim.x) {
        if (!alive[x]) continue;
        const int m = mask[x];
        if (!(m & my_bit) || !(m & ~my_bit)) continue;             // not seen here, or seen here only
        const int r = parent[x];
        if (r == (int)x) continue;
        const unsigned long long i = atomicAdd(n_out, 1ull);
        if ((long long)i < cap) pairs[i] = ((uint64_t)(unsigned)x << 32) | (unsigned)r;
    }
}
__global__ void uf_union_slots_kernel(int32_t* __restrict__ parent, const unsigned char* __restrict__ slots, int n_slots,
                                      int64_t slot_bytes, int64_t cap, int64_t R) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)n_slots * cap;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int slot = (int)(i / cap);
        const int64_t j = i - (int64_t)slot * cap;
        const unsigned char* sb = slots + (size_t)slot * slot_bytes;
        const long long n = *(const long long*)sb;
        if (j >= n || j >= cap) continue;
        const uint64_t k = ((const uint64_t*)(sb + 80))[j];
        const int a = key_lo(k), b = key_hi(k);
        if ((unsigned)a < (unsigned)R && (unsigned)b < (unsigned)R) uf_unite(parent, a, b);
    }
}

__global__ void uf_compress_kernel(int32_t* __restrict__ parent, int64_t n) {
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (int64_t)gridDim.x * blockDim.x) {
        // roots never change here, so racing writes of final roots are benign
        parent[x] = uf_find(parent, (int)x);
    }
}

// ---- merged statistics ------------------------------------------------------------------------
__global__ void collect_members_kernel(const int32_t* __restrict__ parent, uint8_t* __restrict__ alive,
                                       uint8_t* __restrict__ changed, int32_t* __restrict__ cnt,
                                       unsigned long long* __restrict__ area, unsigned long long* __restrict__ perimeter,
                                       int64_t R, uint64_t* __restrict__ list, unsigned long long* __restrict__ n_list,
                                       unsigned long long* __restrict__ n_moved, const uint8_t* __restrict__ root_mask) {
    for (int64_t x0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x - (threadIdx.x & 31); x0 < R;
         x0 += (int64_t)gridDim.x * blockDim.x) {
        const int64_t x = x0 + (threadIdx.x & 31);
        bool moved = false;
        int r = 0;
        if (x < R && alive[x]) {
            r = parent[x];
            moved = r != (int)x;
        }
        const unsigned bal_moved = __ballot_sync(0xffffffffu, moved);
        if (!bal_moved) continue;
        // root_mask (row-tile sharding): only components this rank sees get their embedding sums merged here
        const bool listed = moved && (!root_mask || root_mask[r]);
        const unsigned bal = __ballot_sync(0xffffffffu, listed);
        unsigned long long base = 0;
        if ((threadIdx.x & 31) == 0) {
            if (bal) base = atomicAdd(n_list, (unsigned long long)__popc(bal));
            atomicAdd(n_moved, (unsigned long long)__popc(bal_moved));
        }
        base = __shfl_sync(0xffffffffu, base, 0);
        if (moved) {
            alive[x] = 0;
            changed[r] = 1;
            atomicAdd(&cnt[r], cnt[x]);
            atomicAdd(&area[r], area[x]);
            atomicAdd(&perimeter[r], perimeter[x]);
            if (listed) list[base + __popc(bal & lanemask_lt())] = ((uint64_t)(unsigned)r << 32) | (unsigned)x;
        }
    }
}

// list sorted by (root, member).  The warp that lands on the head of a root's run adds the
// members' sums into the root's sum one after another (ascending member id): a fixed fp32
// summation order, so results do not depend on scheduling.  The run is read 32 entries at a time
// (one entry per lane: the run's end is a ballot, the member ids travel by shuffle), each lane keeps
// up to 4 feature columns in registers and 8 member rows of loads are in flight; the adds stay in order.
__global__ void __launch_bounds__(256) merge_sums_kernel(const uint64_t* __restrict__ list,
                                                         const int64_t* __restrict__ n_dev, float* __restrict__ sum,
                                                         int D) {
    const int64_t n = *n_dev;
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp0; i < n; i += nwarps) {
        const int root = key_lo(list[i]);
        if (i > 0 && key_lo(list[i - 1]) == root) continue;
        for (int d0 = 0; d0 < D; d0 += 128) {
            float acc[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[k] = (d0 + lane + 32 * k < D) ? sum[(int64_t)root * D + d0 + lane + 32 * k] : 0.f;
            int64_t j = i;
            while (true) {
                const int64_t idx = j + lane;
                const uint64_t kk = idx < n ? list[idx] : 0ull;
                const unsigned same = __ballot_sync(0xffffffffu, idx < n && key_lo(kk) == root);
                const int len = same == 0xffffffffu ? 32 : __ffs(~same) - 1;    // entries of this run among the 32
                const int member = key_hi(kk);
                for (int u0 = 0; u0 < len; u0 += 8) {
                    float v[8][4];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        if (u0 + u < len) {                                    // (len is the same in every lane)
                            const float* row = sum + (int64_t)__shfl_sync(0xffffffffu, member, u0 + u) * D + d0;
#pragma unroll
                            for (int k = 0; k < 4; ++k) v[u][k] = (d0 + lane + 32 * k < D) ? row[lane + 32 * k] : 0.f;
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        if (u0 + u < len) {
#pragma unroll
                            for (int k = 0; k < 4; ++k) acc[k] += v[u][k];
                        }
                    }
                }
                j += len;
                if (len < 32) break;
            }
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (d0 + lane + 32 * k < D) sum[(int64_t)root * D + d0 + lane + 32 * k] = acc[k];
        }
    }
}

// ---- edge re-keying -----------------------------------------------------------------------------
__global__ void rekey_kernel(const int32_t* __restrict__ parent, const uint64_t* __restrict__ keys,
                             const uint32_t* __restrict__ lens, const int64_t* __restrict__ n_dev, uint64_t sentinel,
                             unsigned long long* __restrict__ perimeter, uint64_t* __restrict__ new_keys,
                             uint32_t* __restrict__ perm) {
    const int64_t n = *n_dev;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t k = keys[e];
        const int a = parent[key_lo(k)], b = parent[key_hi(k)];
        perm[e] = (uint32_t)e;
        if (a == b) {   // the boundary became internal: both of its sides leave the perimeter
            atomicAdd(&perimeter[a], (unsigned long long)(-2ll * (long long)lens[e]));
            new_keys[e] = sentinel;
        } else {
            new_keys[e] = pack_key(a, b);
        }
    }
}


// ---- relabel ------------------------------------------------------------------------------------
__device__ __forceinline__ int lut(const int32_t* __restrict__ root, int l, int R) {
    return (unsigned)l < (unsigned)R ? __ldg(root + l) : l;
}

// 128-bit streaming loads/stores; the root LUT (4 B x R) stays in L2 / L1.
// gate (may be null): the kernel does nothing when *gate != 0 -- a relabel enqueued BEFORE the host has read the merge
// loop's last selection count runs only if that count is zero (no further round), so the loop's last read-back does not
// leave the GPU idle.
__global__ void __launch_bounds__(256) relabel_vec_kernel(const int4* __restrict__ in, int64_t n4,
                                                          const int32_t* __restrict__ root, int R, int4* __restrict__ out,
                                                          const int64_t* __restrict__ gate) {
    if (gate && *gate != 0) return;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < n4; i += 4 * stride) {   // 4 independent 16-byte loads in flight per thread
        int4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = ldg_stream(in + i + u * stride);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            v[u].x = lut(root, v[u].x, R);
            v[u].y = lut(root, v[u].y, R);
            v[u].z = lut(root, v[u].z, R);
            v[u].w = lut(root, v[u].w, R);
            stg_stream(out + i + u * stride, v[u]);
        }
    }
    for (; i < n4; i += stride) {
        int4 v = ldg_stream(in + i);
        v.x = lut(root, v.x, R);
        v.y = lut(root, v.y, R);
        v.z = lut(root, v.z, R);
        v.w = lut(root, v.w, R);
        stg_stream(out + i, v);
    }
}

__global__ void relabel_scalar_kernel(const int32_t* __restrict__ in, int64_t H, int64_t W, int64_t ld_in,
                                      const int32_t* __restrict__ root, int R, int32_t* __restrict__ out, int64_t ld_out,
                                      const int64_t* __restrict__ gate) {
    if (gate && *gate != 0) return;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < H * W; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t y = i / W, x = i - y * W;
        out[y * ld_out + x] = lut(root, in[y * ld_in + x], R);
    }
}

__global__ void root_flags_kernel(const int32_t* __restrict__ root, int64_t R, uint32_t* __restrict__ flags,
                                  int64_t* __restrict__ n_dev) {
    if (blockIdx.x == 0 && threadIdx.x == 0) *n_dev = R;
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < R; x += (int64_t)gridDim.x * blockDim.x)
        flags[x] = root[x] == (int)x ? 1u : 0u;
}
__global__ void compact_kernel(const int32_t* __restrict__ root, int64_t R, const uint32_t* __restrict__ excl,
                               int32_t* __restrict__ compact) {
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < R; x += (int64_t)gridDim.x * blockDim.x) {
        const int r = root[x];
        compact[x] = (unsigned)r < (unsigned)R ? (int)excl[r] : -1;
    }
}

__global__ void perimeter_init_kernel(const int64_t* __restrict__ border, int64_t* __restrict__ perimeter, int64_t R) {
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < R; x += (int64_t)gridDim.x * blockDim.x)
        perimeter[x] = border[x];
}
__global__ void perimeter_edges_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ lens,
                                       const int64_t* __restrict__ n_dev, unsigned long long* __restrict__ perimeter,
                                       int64_t R) {
    const int64_t n = *n_dev;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t k = keys[e];
        if ((k >> 32) >= (uint64_t)R || (k & 0xffffffffu) >= (uint64_t)R) continue;   // sentinels and foreign keys
        atomicAdd(&perimeter[key_lo(k)], (unsigned long long)lens[e]);
        atomicAdd(&perimeter[key_hi(k)], (unsigned long long)lens[e]);
    }
}

// ---- row-tile sharding helpers ------------------------------------------------------------------------
__global__ void mark_endpoints_kernel(const uint64_t* __restrict__ keys, const int64_t* __restrict__ n_dev, int64_t R,
                                      uint8_t* __restrict__ flags) {
    const int64_t n = *n_dev;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t k = keys[e];
        if ((k >> 32) < (uint64_t)R && (k & 0xffffffffu) < (uint64_t)R) {   // both ids in [0, R), compared unsigned
            flags[key_lo(k)] = 1;
            flags[key_hi(k)] = 1;
        }
    }
}

// one warp per region: flagged rows are appended (id, row) to the slot buffer; order inside the slot is arbitrary
__global__ void __launch_bounds__(256) rows_pack_kernel(const uint8_t* __restrict__ flag, const float* __restrict__ rows,
                                                        int64_t R, int D, int32_t* __restrict__ out_ids,
                                                        float* __restrict__ out_rows, int64_t cap,
                                                        unsigned long long* __restrict__ n_out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r0 = warp0 * 32; r0 < R; r0 += nwarps * 32) {
        const int64_t r = r0 + lane;
        const bool f = r < R && flag[r];
        unsigned m = __ballot_sync(0xffffffffu, f);
        if (!m) continue;
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(n_out, (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        int j = 0;
        while (m) {
            const int src = __ffs(m) - 1;
            m &= m - 1;
            const unsigned long long slot = base + j++;
            if ((long long)slot < cap) {                       // overflow is visible in the count
                if (lane == 0) out_ids[slot] = (int32_t)(r0 + src);
                for (int d = lane; d < D; d += 32) out_rows[slot * D + d] = rows[(r0 + src) * D + d];
            }
        }
    }
}

// one warp per packed entry: rows[id] = row (add == 0) or rows[id] += row (add != 0; ids are distinct inside one slot)
__global__ void __launch_bounds__(256) rows_unpack_kernel(const int32_t* __restrict__ ids, const float* __restrict__ in_rows,
                                                          const int64_t* __restrict__ n_dev, int64_t cap, int64_t R, int D,
                                                          float* __restrict__ rows, int add) {
    const int64_t n = imin64(*n_dev, cap);
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp0; i < n; i += nwarps) {
        const int64_t r = ids[i];
        if (r < 0 || r >= R) continue;
        for (int d = lane; d < D; d += 32) {
            const float v = in_rows[i * D + d];
            rows[r * D + d] = add ? rows[r * D + d] + v : v;
        }
    }
}

// rank-visibility masks: bit g of mask[r] = rank g sees region r.  A component is seen by every rank that sees a member.
__global__ void shard_propagate_kernel(const int32_t* __restrict__ parent, const uint8_t* __restrict__ alive,
                                       int32_t* __restrict__ mask, uint8_t* __restrict__ grew, int64_t R) {
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < R; x += (int64_t)gridDim.x * blockDim.x) {
        const int p = parent[x];
        if (alive[x] && p != (int)x) {
            atomicOr(&mask[p], mask[x]);
            grew[p] = 1;
        }
    }
}
// send[x]: this rank ships region x's embedding sum -- x belongs to a component that grew this round and is seen by
// at least two ranks, and this rank is the lowest one that held x's sum before the round.
__global__ void shard_plan_kernel(const int32_t* __restrict__ parent, const uint8_t* __restrict__ alive,
                                  const int32_t* __restrict__ mask_old, const int32_t* __restrict__ mask_new,
                                  const uint8_t* __restrict__ grew, int my_bit, int64_t R, uint8_t* __restrict__ send,
                                  uint8_t* __restrict__ seen_comp) {
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < R; x += (int64_t)gridDim.x * blockDim.x) {
        const int p = parent[x];
        const int mo = mask_old[x], mp = mask_new[p];
        seen_comp[x] = (mask_new[x] & my_bit) ? 1 : 0;
        send[x] = (alive[x] && grew[p] && (mp & (mp - 1)) != 0 && (mo & -mo) == my_bit) ? 1 : 0;
    }
}

// All slots of an all-gathered exchange buffer in one launch.  Slot layout: int64 count | pad to 16 B | int32 ids[cap] |
// float rows[cap][D].  zero != 0 writes zeros (ids may repeat across slots: benign), else copies (ids distinct overall).
__global__ void __launch_bounds__(256) rows_unpack_slots_kernel(const unsigned char* __restrict__ buf, int n_slots,
                                                                int64_t slot_bytes, int64_t cap, int64_t R, int D,
                                                                float* __restrict__ rows, int zero) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t w = warp0; w < (int64_t)n_slots * cap; w += nwarps) {
        const int g = (int)(w / cap);
        const int64_t i = w - (int64_t)g * cap;
        const unsigned char* slot = buf + (size_t)g * slot_bytes;
        if (i >= *(const int64_t*)slot) continue;
        const int64_t r = ((const int32_t*)(slot + 16))[i];
        if (r < 0 || r >= R) continue;
        const float* src = (const float*)(slot + 16 + 4 * cap) + i * D;
        for (int d = lane; d < D; d += 32) rows[r * D + d] = zero ? 0.f : src[d];
    }
}

// fused R-sized glue of the distributed merge loop (one launch each instead of a string of elementwise kernels)
__global__ void shard_seen_kernel(const int64_t* __restrict__ area, uint8_t* __restrict__ seen, const int32_t* __restrict__ cnt,
                                  int my_bit, int64_t R, int32_t* __restrict__ mask_cnt, int32_t* __restrict__ cnt_local) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (int64_t)gridDim.x * blockDim.x) {
        const bool sees = seen[r] || area[r] > 0;            // an endpoint of a tile edge, or pixels in the tile
        seen[r] = sees ? 1 : 0;
        mask_cnt[r] = sees ? my_bit : 0;
        const int c = cnt[r];
        mask_cnt[R + r] = c;
        cnt_local[r] = c;
    }
}
__global__ void shard_frontier_kernel(const int32_t* __restrict__ mask_cnt, const int32_t* __restrict__ cnt_local, int64_t R,
                                      int32_t* __restrict__ cnt, uint8_t* __restrict__ send) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (int64_t)gridDim.x * blockDim.x) {
        const int m = mask_cnt[r];
        cnt[r] = mask_cnt[R + r];
        send[r] = ((m & (m - 1)) != 0 && cnt_local[r] > 0) ? 1 : 0;   // seen by two ranks, and this one has points of it
    }
}
// Fused "all-gather" of fixed-layout slots over NVLink peer memory: this rank's slot -- a header and up to two segments
// whose used length is the header's leading count -- is stored straight into slot `rank` of EVERY rank's gathered buffer
// (peer_bases[p] = base address of rank p's buffer, mapped into this process; p == rank is the local copy).  Only the
// used part travels.  A barrier over all ranks (signal pads) after this kernel makes the stores visible.
__global__ void __launch_bounds__(256) peer_put_kernel(const unsigned char* __restrict__ src, const long long* __restrict__ peer_bases,
                                                       int world, int rank, int64_t slot_bytes, int64_t hdr_units,
                                                       int64_t seg0_off, int64_t seg0_elem, int64_t seg1_off, int64_t seg1_elem,
                                                       int64_t cap) {
    const long long n = imin64(*(const long long*)src, cap);
    const int64_t u0 = (n * seg0_elem + 15) >> 4, u1 = (n * seg1_elem + 15) >> 4;
    const int64_t total = hdr_units + u0 + u1;
    for (int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; u < total; u += (int64_t)gridDim.x * blockDim.x) {
        int64_t off;
        if (u < hdr_units) off = u << 4;
        else if (u < hdr_units + u0) off = seg0_off + ((u - hdr_units) << 4);
        else off = seg1_off + ((u - hdr_units - u0) << 4);
        const uint4 v = *(const uint4*)(src + off);
        for (int p = 0; p < world; ++p)
            *(uint4*)((unsigned char*)peer_bases[p] + (size_t)rank * slot_bytes + off) = v;
    }
}

// Two-shot all-reduce of an int32 array that lives at the same offset of every rank's symmetric buffer, over NVLink peer
// memory: rank g reduces slice g of all ranks' arrays (peer loads) and stores the result into slice g of EVERY rank's
// array (peer stores), in place.  A barrier over all ranks before this kernel (every rank's array is complete) and one
// after it (every slice has landed) are the caller's.  Slices are whole 16-byte units; op 0 = sum, 1 = min.
__device__ __forceinline__ int4 ld_peer_v4(const int4* p) {
    int4 v;
    asm volatile("ld.volatile.global.v4.s32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
__global__ void __launch_bounds__(256) peer_allreduce_i32_kernel(const long long* __restrict__ peer_bases, int world, int rank,
                                                                 int64_t offset_bytes, int64_t n4, int op) {
    const int64_t per = (n4 + world - 1) / world;
    const int64_t lo = (int64_t)rank * per, hi = imin64(n4, lo + per);
    for (int64_t i = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (int64_t)gridDim.x * blockDim.x) {
        int4 acc = op ? make_int4(0x7fffffff, 0x7fffffff, 0x7fffffff, 0x7fffffff) : make_int4(0, 0, 0, 0);
        for (int p0 = 0; p0 < world; p0 += 8) {            // up to 8 peer loads in flight
            int4 v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (p0 + j < world) v[j] = ld_peer_v4((const int4*)((const unsigned char*)peer_bases[p0 + j] + offset_bytes) + i);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                if (p0 + j < world) {
                    if (op) {
                        acc.x = min(acc.x, v[j].x); acc.y = min(acc.y, v[j].y); acc.z = min(acc.z, v[j].z); acc.w = min(acc.w, v[j].w);
                    } else {
                        acc.x += v[j].x; acc.y += v[j].y; acc.z += v[j].z; acc.w += v[j].w;
                    }
                }
            }
        }
        for (int p = 0; p < world; ++p) *((int4*)((unsigned char*)peer_bases[p] + offset_bytes) + i) = acc;
    }
}

// The flag words of one round of the distributed loop, filled from the engine's counters in ONE launch (they were a
// dozen elementwise launches from the host): flags[0] = edges selected; first round: [3] tile edge-list overflow, [4] bad
// label, [5] internal error, [6] raw entries needed; then flags -> the header of the frontier slot.
__global__ void shard_round_flags_kernel(const int64_t* __restrict__ counts, int64_t* __restrict__ flags, int first_round,
                                         int64_t* __restrict__ slot_flags) {
    const int i = threadIdx.x;
    if (i >= 8) return;
    int64_t v = flags[i];
    if (i == 0) v = counts[4];
    if (first_round) {
        if (i == 3) v = counts[2] != 0;
        if (i == 4) v = counts[3] == 1;
        if (i == 6) v = counts[1];
    }
    if (i == 5 && counts[3] > 1) v = 1;                       // internal error (raster pass, pair-MLP status): any round
    flags[i] = v;
    slot_flags[i] = v;
}
// flag = max(flag, any slot's entry count > capacity)
__global__ void slots_overflow_kernel(const unsigned char* __restrict__ slots, int n_slots, int64_t slot_bytes, int64_t cap,
                                      int64_t* __restrict__ flag) {
    bool over = false;
    for (int g = threadIdx.x; g < n_slots; g += blockDim.x) over |= *(const int64_t*)(slots + (size_t)g * slot_bytes) > cap;
    if (over) *flag = 1;
}

// out = max over the slots of the int64 word at word_offset bytes of every slot (e.g. "edges selected" of every rank)
__global__ void slots_word_max_kernel(const unsigned char* __restrict__ slots, int n_slots, int64_t slot_bytes,
                                      int64_t word_offset, int64_t* __restrict__ out) {
    long long m = 0;
    for (int g = threadIdx.x; g < n_slots; g += blockDim.x) {
        const long long v = *(const long long*)(slots + (size_t)g * slot_bytes + word_offset);
        m = v > m ? v : m;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const long long v = __shfl_xor_sync(0xffffffffu, m, o);
        m = v > m ? v : m;
    }
    if (threadIdx.x == 0) *out = m;
}

}  // namespace merge
}  // namespace dm

using namespace dm;

extern "C" int dm_shard_seen(const int64_t* area, uint8_t* seen, const int32_t* cnt, int rank, int64_t n_regions,
                             int32_t* mask_cnt, int32_t* cnt_local, dm_stream_t stream) {
    if (n_regions < 0 || rank < 0 || rank > 30) return DM_ERR_BAD_ARG;
    if (n_regions == 0) return DM_OK;
    if (!area || !seen || !cnt || !mask_cnt || !cnt_local) return DM_ERR_BAD_ARG;
    return launch(merge::shard_seen_kernel, grid_for(n_regions), 256, 0, S(stream), area, seen, cnt, 1 << rank, n_regions,
        mask_cnt, cnt_local);
}

extern "C" int dm_shard_frontier(const int32_t* mask_cnt, const int32_t* cnt_local, int64_t n_regions, int32_t* cnt,
                                 uint8_t* send, dm_stream_t stream) {
    if (n_regions < 0) return DM_ERR_BAD_ARG;
    if (n_regions == 0) return DM_OK;
    if (!mask_cnt || !cnt_local || !cnt || !send) return DM_ERR_BAD_ARG;
    return launch(merge::shard_frontier_kernel, grid_for(n_regions), 256, 0, S(stream), mask_cnt, cnt_local, n_regions, cnt,
        send);
}

extern "C" int dm_shard_frontier_pairs(const int32_t* parent, const uint8_t* alive, const int32_t* mask, int rank,
                                       int64_t n_regions, void* slot, int64_t capacity, dm_stream_t stream) {
    if (n_regions < 0 || capacity < 0 || rank < 0 || rank > 30 || !slot || ((uintptr_t)slot & 15)) return DM_ERR_BAD_ARG;
    if (n_regions > 0 && (!parent || !alive || !mask)) return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    DM_CUDA(cudaMemsetAsync(slot, 0, 16, s));                       // count; the caller owns the 8 flag words behind it
    if (n_regions == 0) return DM_OK;
    return launch(merge::shard_frontier_pairs_kernel, grid_for(n_regions), 256, 0, s, parent, alive, mask, 1 << rank, n_regions,
        (uint64_t*)((unsigned char*)slot + 80), capacity, (unsigned long long*)slot);
}

extern "C" int dm_uf_union_slots(int32_t* parent, const void* slots, int64_t n_slots, int64_t slot_bytes, int64_t capacity,
                                 int64_t n_regions, dm_stream_t stream) {
    if (n_slots < 0 || capacity < 0 || n_regions < 0 || slot_bytes < 80 + 8 * capacity || (slot_bytes & 15)) return DM_ERR_BAD_ARG;
    if (n_slots == 0 || capacity == 0 || n_regions == 0) return DM_OK;
    if (!parent || !slots) return DM_ERR_BAD_ARG;
    return launch(merge::uf_union_slots_kernel, grid_for(n_slots * capacity), 256, 0, S(stream), parent,
        (const unsigned char*)slots, (int)n_slots, slot_bytes, capacity, n_regions);
}

extern "C" int dm_peer_put_slot(const void* slot, const int64_t* peer_bases_dev, int64_t world, int64_t rank, int64_t slot_bytes,
                                int64_t header_bytes, int64_t seg0_offset, int64_t seg0_elem_bytes, int64_t seg1_offset,
                                int64_t seg1_elem_bytes, int64_t capacity, dm_stream_t stream) {
    if (world < 1 || world > 31 || rank < 0 || rank >= world || capacity < 0 || header_bytes < 16 || (header_bytes & 15) ||
        (slot_bytes & 15) || (seg0_offset & 15) || (seg1_offset & 15) || seg0_elem_bytes < 0 || seg1_elem_bytes < 0 ||
        seg0_offset + capacity * seg0_elem_bytes > slot_bytes || seg1_offset + capacity * seg1_elem_bytes > slot_bytes)
        return DM_ERR_BAD_ARG;
    if (!slot || !peer_bases_dev || ((uintptr_t)slot & 15)) return DM_ERR_BAD_ARG;
    const int64_t units = header_bytes / 16 + (capacity * seg0_elem_bytes + 15) / 16 + (capacity * seg1_elem_bytes + 15) / 16;
    return launch(merge::peer_put_kernel, grid_for(units), 256, 0, S(stream), (const unsigned char*)slot,
        (const long long*)peer_bases_dev, (int)world, (int)rank, slot_bytes, header_bytes / 16, seg0_offset, seg0_elem_bytes,
        seg1_offset, seg1_elem_bytes, capacity);
}

extern "C" int dm_peer_allreduce_i32(const void* peer_bases_dev, int64_t world, int64_t rank, int64_t offset_bytes, int64_t n,
                                     int op, dm_stream_t stream) {
    if (world < 1 || world > 64 || rank < 0 || rank >= world || offset_bytes < 0 || (offset_bytes & 15) || n < 0 || (n & 3) ||
        (op != 0 && op != 1))
        return DM_ERR_BAD_ARG;
    if (n == 0) return DM_OK;
    if (!peer_bases_dev) return DM_ERR_BAD_ARG;
    const int64_t n4 = n / 4, per = ceil_div(n4, world);
    return launch(merge::peer_allreduce_i32_kernel, grid_for(per), 256, 0, S(stream), (const long long*)peer_bases_dev,
        (int)world, (int)rank, offset_bytes, n4, op);
}

extern "C" int dm_shard_round_flags(const int64_t* counts, int64_t* flags, int first_round, int64_t* slot_flags,
                                    dm_stream_t stream) {
    if (!counts || !flags || !slot_flags) return DM_ERR_BAD_ARG;
    return launch(merge::shard_round_flags_kernel, 1, 32, 0, S(stream), counts, flags, first_round, slot_flags);
}

extern "C" int dm_slots_overflow(const void* slots, int64_t n_slots, int64_t slot_bytes, int64_t capacity, int64_t* flag_dev,
                                 dm_stream_t stream) {
    if (n_slots < 0 || n_slots > 4096 || slot_bytes < 16 || capacity < 0 || !flag_dev) return DM_ERR_BAD_ARG;
    if (n_slots == 0) return DM_OK;
    if (!slots) return DM_ERR_BAD_ARG;
    return launch(merge::slots_overflow_kernel, 1, 64, 0, S(stream), (const unsigned char*)slots, (int)n_slots, slot_bytes,
        capacity, flag_dev);
}

extern "C" int dm_slots_word_max(const void* slots, int64_t n_slots, int64_t slot_bytes, int64_t word_offset, int64_t* out_dev,
                                 dm_stream_t stream) {
    if (n_slots < 0 || n_slots > 4096 || slot_bytes < 8 || word_offset < 0 || (word_offset & 7) || word_offset + 8 > slot_bytes ||
        !out_dev)
        return DM_ERR_BAD_ARG;
    if (n_slots > 0 && !slots) return DM_ERR_BAD_ARG;
    return launch(merge::slots_word_max_kernel, 1, 32, 0, S(stream), (const unsigned char*)slots, (int)n_slots, slot_bytes,
        word_offset, out_dev);
}

extern "C" int dm_rows_unpack_slots(const void* slots, int64_t n_slots, int64_t slot_bytes, int64_t slot_capacity,
                                    int64_t n_regions, int64_t D, float* rows, int zero, dm_stream_t stream) {
    if (n_slots < 0 || slot_capacity < 0 || n_regions < 0 || D <= 0 || slot_bytes < 16 + 4 * slot_capacity * (D + 1) ||
        (slot_bytes & 15))
        return DM_ERR_BAD_ARG;
    if (n_slots == 0 || slot_capacity == 0 || n_regions == 0) return DM_OK;
    if (!slots || !rows) return DM_ERR_BAD_ARG;
    return launch(merge::rows_unpack_slots_kernel, grid_for(n_slots * slot_capacity * 32), 256, 0, S(stream),
        (const unsigned char*)slots, (int)n_slots, slot_bytes, slot_capacity, n_regions, (int)D, rows, zero);
}

extern "C" int dm_shard_propagate(const int32_t* parent, const uint8_t* alive, int32_t* mask, uint8_t* grew, int64_t n_regions,
                                  dm_stream_t stream) {
    if (n_regions < 0) return DM_ERR_BAD_ARG;
    if (n_regions == 0) return DM_OK;
    if (!parent || !alive || !mask || !grew) return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    DM_CUDA(cudaMemsetAsync(grew, 0, (size_t)n_regions, s));
    return launch(merge::shard_propagate_kernel, grid_for(n_regions), 256, 0, s, parent, alive, mask, grew, n_regions);
}

extern "C" int dm_shard_plan(const int32_t* parent, const uint8_t* alive, const int32_t* mask_old, const int32_t* mask_new,
                             const uint8_t* grew, int rank, int64_t n_regions, uint8_t* send, uint8_t* seen_comp,
                             dm_stream_t stream) {
    if (n_regions < 0 || rank < 0 || rank > 30) return DM_ERR_BAD_ARG;
    if (n_regions == 0) return DM_OK;
    if (!parent || !alive || !mask_old || !mask_new || !grew || !send || !seen_comp) return DM_ERR_BAD_ARG;
    return launch(merge::shard_plan_kernel, grid_for(n_regions), 256, 0, S(stream), parent, alive, mask_old, mask_new, grew,
        1 << rank, n_regions, send, seen_comp);
}

extern "C" int dm_mark_endpoints(const uint64_t* edge_keys, const int64_t* n_edges_dev, int64_t capacity, int64_t n_regions,
                                 uint8_t* flags, dm_stream_t stream) {
    if (capacity < 0 || n_regions < 0) return DM_ERR_BAD_ARG;
    if (capacity == 0 || n_regions == 0) return DM_OK;
    if (!edge_keys || !n_edges_dev || !flags) return DM_ERR_BAD_ARG;
    return launch(merge::mark_endpoints_kernel, grid_for(capacity), 256, 0, S(stream), edge_keys, n_edges_dev, n_regions, flags);
}

extern "C" int dm_rows_pack(const uint8_t* flag, const float* rows, int64_t n_regions, int64_t D, int32_t* out_ids,
                            float* out_rows, int64_t capacity, int64_t* n_out_dev, dm_stream_t stream) {
    if (n_regions < 0 || D <= 0 || capacity < 0 || !n_out_dev) return DM_ERR_BAD_ARG;
    if (n_regions > 0 && (!flag || !rows || (capacity > 0 && (!out_ids || !out_rows)))) return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    DM_CUDA(cudaMemsetAsync(n_out_dev, 0, sizeof(int64_t), s));
    if (n_regions == 0) return DM_OK;
    return launch(merge::rows_pack_kernel, grid_for(n_regions), 256, 0, s, flag, rows, n_regions, (int)D, out_ids, out_rows,
        capacity, (unsigned long long*)n_out_dev);
}

extern "C" int dm_rows_unpack(const int32_t* ids, const float* in_rows, const int64_t* n_dev, int64_t capacity,
                              int64_t n_regions, int64_t D, float* rows, int add, dm_stream_t stream) {
    if (n_regions < 0 || D <= 0 || capacity < 0) return DM_ERR_BAD_ARG;
    if (capacity == 0 || n_regions == 0) return DM_OK;
    if (!ids || !in_rows || !n_dev || !rows) return DM_ERR_BAD_ARG;
    return launch(merge::rows_unpack_kernel, grid_for(capacity * 32), 256, 0, S(stream), ids, in_rows, n_dev, capacity, n_regions,
        (int)D, rows, add);
}

extern "C" int dm_merge_select_l2(const float* scores, float tau, const int64_t* n_dev, int64_t capacity, uint8_t* selected,
                                  int64_t* n_sel, dm_stream_t stream) {
    if (capacity < 0 || !n_sel) return DM_ERR_BAD_ARG;
    if (capacity > 0 && (!scores || !n_dev || !selected)) return DM_ERR_BAD_ARG;
    DM_CUDA(cudaMemsetAsync(n_sel, 0, sizeof(int64_t), S(stream)));
    if (capacity == 0) return DM_OK;
    return launch(merge::select_kernel<false>, grid_for(capacity), 256, 0, S(stream), scores, tau, 1, n_dev, selected,
        (unsigned long long*)n_sel);
}

extern "C" int dm_merge_select_mlp(const float* o, int64_t n_out, const int64_t* n_dev, int64_t capacity, uint8_t* selected,
                                   int64_t* n_sel, dm_stream_t stream) {
    if (capacity < 0 || !n_sel || n_out < 2) return DM_ERR_BAD_ARG;
    if (capacity > 0 && (!o || !n_dev || !selected)) return DM_ERR_BAD_ARG;
    DM_CUDA(cudaMemsetAsync(n_sel, 0, sizeof(int64_t), S(stream)));
    if (capacity == 0) return DM_OK;
    return launch(merge::select_kernel<true>, grid_for(capacity), 256, 0, S(stream), o, 0.f, (int)n_out, n_dev, selected,
        (unsigned long long*)n_sel);
}

extern "C" int dm_uf_union(int32_t* parent, const uint64_t* keys, const uint8_t* selected, const int64_t* n_dev,
                           int64_t capacity, dm_stream_t stream) {
    if (capacity < 0) return DM_ERR_BAD_ARG;
    if (capacity == 0) return DM_OK;
    if (!parent || !keys || !selected || !n_dev) return DM_ERR_BAD_ARG;
    return launch(merge::uf_union_kernel, grid_for(capacity), 256, 0, S(stream), parent, keys, selected, n_dev);
}

extern "C" int dm_uf_compress(int32_t* parent, int64_t R, dm_stream_t stream) {
    if (R < 0) return DM_ERR_BAD_ARG;
    if (R == 0) return DM_OK;
    if (!parent) return DM_ERR_BAD_ARG;
    return launch(merge::uf_compress_kernel, grid_for(R), 256, 0, S(stream), parent, R);
}

namespace {
struct ApplyWs {
    uint64_t* list;
    void* sort;
    int64_t* n_list;
    size_t bytes;
};
ApplyWs merge_apply_ws(void* base, int64_t R) {
    const int64_t cap = imax64(R, 1);
    Carver c(base);
    return {c.take<uint64_t>(cap), c.take<char>(prims::ws_bytes(cap, false)), c.take<int64_t>(1), c.used()};
}
}  // namespace

extern "C" size_t dm_merge_apply_workspace_bytes(int64_t R) { return merge_apply_ws(nullptr, R).bytes; }

extern "C" int dm_merge_apply_masked(const int32_t* parent, uint8_t* alive, uint8_t* changed, float* sum, int32_t* cnt,
                                     int64_t* area, int64_t* perimeter, int64_t R, int64_t D, int64_t* n_merged,
                                     const uint8_t* root_mask, void* ws, size_t ws_bytes, dm_stream_t stream) {
    if (R < 0 || D <= 0 || !n_merged) return DM_ERR_BAD_ARG;
    const ApplyWs w = merge_apply_ws(ws, R);
    if (R > 0) {
        if (!parent || !alive || !changed || !sum || !cnt || !area || !perimeter || !ws) return DM_ERR_BAD_ARG;
        if (ws_bytes < w.bytes) return DM_ERR_WORKSPACE;
    }
    cudaStream_t s = S(stream);
    DM_CUDA(cudaMemsetAsync(n_merged, 0, sizeof(int64_t), s));
    if (R == 0) return DM_OK;
    DM_CUDA(cudaMemsetAsync(changed, 0, (size_t)R, s));
    DM_CUDA(cudaMemsetAsync(w.n_list, 0, sizeof(int64_t), s));
    DM_TRY(launch(merge::collect_members_kernel, grid_for(R), 256, 0, s, parent, alive, changed, cnt, (unsigned long long*)area,
        (unsigned long long*)perimeter, R, w.list, (unsigned long long*)w.n_list, (unsigned long long*)n_merged, root_mask));
    const int b = bits_for(R);
    DM_TRY(prims::sort_pairs(w.list, nullptr, w.n_list, R, b, 2 * b, w.sort, s, R));
    return launch(merge::merge_sums_kernel, grid_for(R * 32), 256, 0, s, w.list, w.n_list, sum, (int)D);
}

extern "C" int dm_merge_apply(const int32_t* parent, uint8_t* alive, uint8_t* changed, float* sum, int32_t* cnt,
                              int64_t* area, int64_t* perimeter, int64_t R, int64_t D, int64_t* n_merged, void* ws,
                              size_t ws_bytes, dm_stream_t stream) {
    return dm_merge_apply_masked(parent, alive, changed, sum, cnt, area, perimeter, R, D, n_merged, nullptr, ws, ws_bytes,
                                 stream);
}

namespace {
struct RekeyWs {
    uint64_t *new_keys, *out_keys;
    uint32_t *perm, *out_lens;
    float* out_scores;
    void* sort;
    int64_t* n_new;
    size_t bytes;
};
RekeyWs edges_rekey_ws(void* base, int64_t capacity) {
    const int64_t cap = imax64(capacity, 1);
    Carver c(base);
    return {c.take<uint64_t>(cap), c.take<uint64_t>(cap), c.take<uint32_t>(cap), c.take<uint32_t>(cap), c.take<float>(cap),
            c.take<char>(prims::ws_bytes(cap, true)), c.take<int64_t>(1), c.used()};
}
}  // namespace

extern "C" size_t dm_edges_rekey_workspace_bytes(int64_t capacity) { return edges_rekey_ws(nullptr, capacity).bytes; }

extern "C" int dm_edges_rekey(const int32_t* parent, uint64_t* keys, uint32_t* lens, float* scores, int64_t* n_dev,
                              int64_t capacity, int64_t R, int64_t* perimeter, void* ws, size_t ws_bytes,
                              dm_stream_t stream) {
    if (capacity < 0 || R < 0) return DM_ERR_BAD_ARG;
    if (capacity == 0) return DM_OK;
    if (!parent || !keys || !lens || !n_dev || !perimeter || !ws) return DM_ERR_BAD_ARG;
    const RekeyWs w = edges_rekey_ws(ws, capacity);
    if (ws_bytes < w.bytes) return DM_ERR_WORKSPACE;
    cudaStream_t s = S(stream);
    prims::Reduce r;
    r.sentinel = ((uint64_t)R << 32) | (uint64_t)R;
    r.gather_lens = lens;
    r.gather_scores = scores;
    r.out = {w.out_keys, w.out_lens, scores ? w.out_scores : nullptr, w.n_new};
    r.back = {keys, lens, scores, n_dev};
    DM_TRY(launch(merge::rekey_kernel, grid_for(capacity), 256, 0, s, parent, keys, lens, n_dev, r.sentinel,
        (unsigned long long*)perimeter, w.new_keys, w.perm));
    const int b = bits_for(R + 1);
    return prims::sort_unique(w.new_keys, w.perm, n_dev, capacity, b, 2 * b, w.sort, r, s, R);
}

extern "C" int dm_relabel_gated(const int32_t* labels, int64_t H, int64_t W, int64_t ld_in, const int32_t* root, int64_t R,
                                int32_t* out, int64_t ld_out, const int64_t* skip_if_nonzero, dm_stream_t stream) {
    if (H < 0 || W < 0 || ld_in < W || ld_out < W || R < 0 || R > 0x7fffffff) return DM_ERR_BAD_ARG;
    if (H == 0 || W == 0) return DM_OK;
    if (!labels || !out || (!root && R > 0)) return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    const bool dense = (ld_in == W && ld_out == W);
    const int64_t n = H * W;
    if (dense && n % 4 == 0 && (uintptr_t)labels % 16 == 0 && (uintptr_t)out % 16 == 0) {
        const int64_t n4 = n / 4;
        // 4 x 16 B per thread per trip: a block covers 1024 int4
        return launch(merge::relabel_vec_kernel, grid_for(n4, 1024), 256, 0, s, (const int4*)labels, n4, root, (int)R,
            (int4*)out, skip_if_nonzero);
    }
    return launch(merge::relabel_scalar_kernel, grid_for(n), 256, 0, s, labels, H, W, ld_in, root, (int)R, out, ld_out,
        skip_if_nonzero);
}

extern "C" int dm_relabel(const int32_t* labels, int64_t H, int64_t W, int64_t ld_in, const int32_t* root, int64_t R,
                          int32_t* out, int64_t ld_out, dm_stream_t stream) {
    return dm_relabel_gated(labels, H, W, ld_in, root, R, out, ld_out, nullptr, stream);
}

namespace {
struct RootsWs {
    uint32_t *flags, *excl;
    void* scan;
    int64_t* n_dev;
    size_t bytes;
};
RootsWs compact_roots_ws(void* base, int64_t R) {
    const int64_t cap = imax64(R, 1);
    Carver c(base);
    return {c.take<uint32_t>(cap), c.take<uint32_t>(cap), c.take<char>(prims::scan_ws_bytes(cap)), c.take<int64_t>(1),
            c.used()};
}
}  // namespace

extern "C" size_t dm_compact_roots_workspace_bytes(int64_t R) { return compact_roots_ws(nullptr, R).bytes; }

extern "C" int dm_compact_roots(const int32_t* root, int64_t R, int32_t* compact, int64_t* n_roots, void* ws,
                                size_t ws_bytes, dm_stream_t stream) {
    if (R < 0 || !n_roots) return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    if (R == 0) {
        DM_CUDA(cudaMemsetAsync(n_roots, 0, sizeof(int64_t), s));
        return DM_OK;
    }
    if (!root || !compact || !ws) return DM_ERR_BAD_ARG;
    const RootsWs w = compact_roots_ws(ws, R);
    if (ws_bytes < w.bytes) return DM_ERR_WORKSPACE;
    DM_TRY(launch(merge::root_flags_kernel, grid_for(R), 256, 0, s, root, R, w.flags, w.n_dev));
    DM_TRY(prims::scan_exclusive_u32(w.flags, w.excl, w.n_dev, R, n_roots, w.scan, s));
    return launch(merge::compact_kernel, grid_for(R), 256, 0, s, root, R, w.excl, compact);
}

extern "C" int dm_perimeter(const uint64_t* keys, const uint32_t* lens, const int64_t* n_dev, int64_t capacity,
                            const int64_t* border, int64_t* perimeter, int64_t R, dm_stream_t stream) {
    if (capacity < 0 || R < 0) return DM_ERR_BAD_ARG;
    if (R == 0) return DM_OK;
    if (!border || !perimeter || (capacity > 0 && (!keys || !lens || !n_dev))) return DM_ERR_BAD_ARG;
    cudaStream_t s = S(stream);
    DM_TRY(launch(merge::perimeter_init_kernel, grid_for(R), 256, 0, s, border, perimeter, R));
    if (capacity == 0) return DM_OK;
    return launch(merge::perimeter_edges_kernel, grid_for(capacity), 256, 0, s, keys, lens, n_dev,
        (unsigned long long*)perimeter, R);
}
