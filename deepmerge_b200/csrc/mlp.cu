// R8: pair-MLP scorer with the layer structure of Nets.MLP.forward (Nets.py:28-35) on the
// 5th-generation tensor cores: three Linear + leaky_relu(0.01), bf16 operands, fp32 accumulation
// in TMEM.
//
// One persistent CTA per SM walks over tiles of 128 rows (edges).  Twenty-six warps, four roles:
//   warp 0      weight loader: streams the pre-packed bf16 weight chunks (K = 64 columns of all
//               256 output features, 32 KB, already in the UMMA SWIZZLE_128B K-major image) from
//               global memory into a 3-stage shared-memory ring with 1-D TMA bulk copies
//               (cp.async.bulk + mbarrier complete_tx);
//   warp 1      MMA issuer: one thread issues tcgen05.mma (M=128, N=256 / 16, K=16) on the ring's
//               A / B chunks, tcgen05.commit releases ring stages and signals the accumulator;
//               owns the TMEM allocation (512 columns: D1 at 0, D2 and then D3 at 256).  Layer 1 of
//               the NEXT tile is issued between layers 2 and 3 of this one, so the tensor core works
//               while the epilogue warps are busy;
//   warps 2-9   epilogue: tcgen05.ld the accumulator (each warp its TMEM lane quadrant), add the bias,
//               apply the leaky ReLU, and either re-pack the activations as the next layer's bf16 A
//               operand in shared memory or store the fp32 result;
//   warps 10-25 producers (layer 1): gather the tile's rows -- x_e = concat(mean[lo], mean[hi]) --
//               convert to bf16 and write them as swizzled A chunks into the ring, running ahead of
//               the tile in flight as far as the ring allows.
// Layers 2 and 3 never leave the SM: h1 and h2 go TMEM -> registers -> shared memory -> tensor core.
#include <cuda_bf16.h>
#include "common.cuh"

namespace dm {
namespace mlp {

constexpr int M_TILE = 128;                  // rows (edges) per tile = UMMA M
constexpr int N_HID = 256;                   // hidden width padded to the UMMA N of layers 1 and 2
constexpr int N_OUT = 16;                    // output width padded to the UMMA N of layer 3
constexpr int KC = 64;                       // K columns per chunk = one 128-byte swizzle row of bf16
constexpr int UMMA_K = 16;
constexpr int STAGES = 3;
constexpr int A_CHUNK_BYTES = M_TILE * KC * 2;               // 16 KB
constexpr int B_CHUNK_BYTES = N_HID * KC * 2;                // 32 KB
constexpr int STAGE_BYTES = A_CHUNK_BYTES + B_CHUNK_BYTES;   // 48 KB
constexpr int A2_BYTES = M_TILE * N_HID * 2;                 // 64 KB: h1 / h2 as bf16 A operand (4 chunks)
constexpr int W3_CHUNK_BYTES = N_OUT * KC * 2;               // 2 KB
constexpr int W3_BYTES = (N_HID / KC) * W3_CHUNK_BYTES;      // 8 KB
constexpr int BIAS_FLOATS = N_HID + N_HID + N_OUT;
constexpr int OFF_RING = 0;
constexpr int OFF_A2 = OFF_RING + STAGES * STAGE_BYTES;
constexpr int OFF_W3 = OFF_A2 + A2_BYTES;
constexpr int OFF_BIAS = OFF_W3 + W3_BYTES;
constexpr int OFF_BARS = OFF_BIAS + BIAS_FLOATS * 4;
constexpr int N_BARS = 3 * STAGES + 3 + 8;                   // full_b, full_a, empty per stage; d1/d2/d3_full; a1/a2_ready per K chunk
constexpr int OFF_TMEM = OFF_BARS + N_BARS * 8;
constexpr int SMEM_BYTES = 1024 + OFF_TMEM + 16;
constexpr int EPI_WARPS = 8;                 // two per TMEM lane quadrant, each half of the columns
constexpr int PROD_WARPS = 16;               // each gathers 128 / PROD_WARPS rows of a chunk
constexpr int THREADS = (2 + EPI_WARPS + PROD_WARPS) * 32;   // loader, MMA issuer, epilogue warps, producer warps
constexpr int TMEM_COLS = 512;
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
static_assert(OFF_A2 % 1024 == 0 && OFF_W3 % 1024 == 0 && STAGE_BYTES % 1024 == 0 && A_CHUNK_BYTES % 1024 == 0, "swizzle atoms");

// Packed weight blob: W1 chunks | W2 chunks | W3 chunks | b1[256] b2[256] b3[16] (fp32)
__host__ __device__ inline int64_t nk_for(int64_t in_features) { return (in_features + KC - 1) / KC; }
__host__ __device__ inline size_t off_w2(int64_t nk1) { return (size_t)nk1 * B_CHUNK_BYTES; }
__host__ __device__ inline size_t off_w3(int64_t nk1) { return off_w2(nk1) + (size_t)(N_HID / KC) * B_CHUNK_BYTES; }
__host__ __device__ inline size_t off_bias(int64_t nk1) { return off_w3(nk1) + W3_BYTES; }
__host__ __device__ inline size_t packed_bytes(int64_t nk1) { return off_bias(nk1) + BIAS_FLOATS * 4; }

struct Params {
    const float* src;          // mean [R, ld] (edge mode) or x [B, ld] (dense mode)
    int64_t ld;
    const uint64_t* keys;      // edge keys, or null in dense mode
    const int64_t* n_dev;      // device-side row count, or null
    int64_t n_host;
    int D;                     // features per endpoint (edge mode: in_features = 2 D)
    int in_features, nk1, hidden, n_out;
    const unsigned char* packed;
    float* o;
    float* h2;
    int* status;               // set to 1 when a bounded wait expires (never a hang)
};

// ------------------------------------------------------------------------------------ //
// PTX wrappers
// ------------------------------------------------------------------------------------ //
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, unsigned parity) {
    unsigned ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"(20000u)
        : "memory");
    return ok != 0;
}
// Bounded, without a trap: a lost signal must become an error CODE -- not a hung GPU and not a dead context.  When a
// wait expires the thread raises the CTA's abort flag (shared memory) and the status word behind the packed weights
// (global memory: 1 = a bounded wait expired, the outputs are invalid); every other wait that does not succeed at
// once sees the flag and returns, every role leaves its tile loop at the next tile, and the kernel ends normally.
// The host reads the status word at its next synchronisation (PackedMLP.check / dm_mlp_status_offset).
struct Bail {
    uint32_t flag;     // shared-memory address of the CTA's abort flag
    int* status;
};
__device__ __forceinline__ bool aborted(const Bail& b) {
    unsigned v;
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(b.flag) : "memory");
    return v != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, unsigned parity, const Bail& b) {
    unsigned spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (aborted(b)) return;
        if (++spins > (1u << 20)) {
            asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(b.flag), "r"(1u) : "memory");
            atomicExch(b.status, 1);
            return;
        }
    }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, unsigned bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
        : "memory");
}
// K-major SWIZZLE_128B operand tile: rows of 128 bytes, 8-row groups 1024 bytes apart
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3fffu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// kind::f16 instruction descriptor: D = f32, A = B = bf16, both K-major
__host__ __device__ constexpr uint32_t umma_idesc(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float lrelu(float x) { return fmaxf(x, x * 0.01f); }        // F.leaky_relu, default slope 0.01
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);                                // .x = a (low half)
    return *(const uint32_t*)&h;
}
// byte offset of the 16-byte piece p (8 bf16) of row r inside a [rows x 64] swizzled chunk
__device__ __forceinline__ uint32_t swz(int r, int p) { return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((p ^ (r & 7)) << 4)); }

// epilogue half 0 writes chunks 0, 1 while half 1 writes 2, 3: the i-th chunk to be complete is kc_order(i)
__host__ __device__ constexpr int kc_order(int i) { return ((i & 1) << 1) | (i >> 1); }

struct Ring {            // every role walks the same sequence of ring uses
    int stage = 0;
    unsigned phase = 0;
    __device__ __forceinline__ void advance(int n = 1) {
        for (int i = 0; i < n; ++i)
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
    }
};

// ------------------------------------------------------------------------------------ //
// the kernel
// ------------------------------------------------------------------------------------ //
__global__ void __launch_bounds__(THREADS, 1) pair_mlp_kernel(const Params P) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* bias = (float*)(smem + OFF_BIAS);
    uint32_t* tmem_slot = (uint32_t*)(smem + OFF_TMEM);
    const Bail bail{sbase + OFF_TMEM + 4u, P.status};           // the abort flag sits beside the TMEM base address
    const uint32_t bar0 = sbase + OFF_BARS;
    auto full_b = [&](int s) { return bar0 + 8u * s; };
    auto full_a = [&](int s) { return bar0 + 8u * (STAGES + s); };
    auto empty = [&](int s) { return bar0 + 8u * (2 * STAGES + s); };
    // accumulator / activation hand-offs, each completing once per tile (parity = tile iteration & 1)
    const uint32_t d1_full = bar0 + 8u * (3 * STAGES), d2_full = d1_full + 8u, d3_full = d1_full + 16u;
    // activations are handed over per 64-column chunk (= one K chunk of the next layer): a1_ready(kc), a2_ready(kc)
    auto a1_ready = [&](int kc) { return d1_full + 24u + 8u * kc; };
    auto a2_ready = [&](int kc) { return d1_full + 24u + 32u + 8u * kc; };

    const int64_t n_rows = P.n_dev ? *P.n_dev : P.n_host;
    const int64_t tiles = (n_rows + M_TILE - 1) / M_TILE;
    const int nk1 = P.nk1, nk2 = N_HID / KC;

    // ---- one-time setup ------------------------------------------------------------------------
    {   // W3 and the biases stay resident
        const uint4* src = (const uint4*)(P.packed + off_w3(nk1));
        uint4* dst = (uint4*)(smem + OFF_W3);
        for (int i = threadIdx.x; i < (W3_BYTES + BIAS_FLOATS * 4) / 16; i += THREADS) dst[i] = src[i];
    }
    if (threadIdx.x == 0) {
        tmem_slot[1] = 0;                     // abort flag
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_b(s), 1);
            mbar_init(full_a(s), PROD_WARPS);
            mbar_init(empty(s), 1);
        }
        mbar_init(d1_full, 1);
        mbar_init(d2_full, 1);
        mbar_init(d3_full, 1);
        for (int kc = 0; kc < N_HID / KC; ++kc) {
            mbar_init(a1_ready(kc), 4);       // the four warps (TMEM lane quadrants) that write that 64-column chunk
            mbar_init(a2_ready(kc), 4);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "n"(TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_async_smem();          // W3 was written with generic stores, the tensor core reads it through the async proxy
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        // ===== weight loader =====================================================================
        Ring ring;
        for (int64_t tile = blockIdx.x; tile < tiles && !aborted(bail); tile += gridDim.x) {
            for (int kc = 0; kc < nk1 + nk2; ++kc) {
                mbar_wait(empty(ring.stage), ring.phase ^ 1u, bail);
                if (lane == 0) {
                    // W1 chunks in order, then W2 chunks in the order the epilogue halves finish them: 0, 2, 1, 3
                    const int ck = kc < nk1 ? kc : nk1 + kc_order(kc - nk1);
                    const unsigned char* src = P.packed + (size_t)ck * B_CHUNK_BYTES;
                    mbar_expect_tx(full_b(ring.stage), B_CHUNK_BYTES);
                    bulk_g2s(sbase + OFF_RING + ring.stage * STAGE_BYTES + A_CHUNK_BYTES, src, B_CHUNK_BYTES,
                             full_b(ring.stage));
                }
                __syncwarp();
                ring.advance();
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer ========================================================================
        // Issue order: L1(0) | L2(0) L1(1) L3(0) | L2(1) L1(2) L3(1) | ...  Layer 1 of the NEXT tile runs on the
        // tensor core while the epilogue warps are busy with this tile's h2 (D1 is free once E1 has read it).
        Ring ring;
        unsigned fa_bits = 0;             // full_a[s] completes on layer-1 ring uses only: its own phase per stage
        constexpr uint32_t idesc_hid = umma_idesc(M_TILE, N_HID), idesc_out = umma_idesc(M_TILE, N_OUT);
        auto issue_l1 = [&]() {           // D1 = X W1^T, both operands from the ring
            for (int kc = 0; kc < nk1; ++kc) {
                mbar_wait(full_b(ring.stage), ring.phase, bail);
                mbar_wait(full_a(ring.stage), (fa_bits >> ring.stage) & 1u, bail);
                fa_bits ^= 1u << ring.stage;
                tc_fence_after();
                if (lane == 0) {
                    const uint32_t a0 = sbase + OFF_RING + ring.stage * STAGE_BYTES, b0 = a0 + A_CHUNK_BYTES;
#pragma unroll
                    for (int k = 0; k < KC / UMMA_K; ++k)
                        tc_mma(tmem, umma_desc(a0 + k * 32), umma_desc(b0 + k * 32), idesc_hid, (kc | k) ? 1u : 0u);
                    tc_commit(empty(ring.stage));
                    if (kc == nk1 - 1) tc_commit(d1_full);
                }
                __syncwarp();
                ring.advance();
            }
        };
        if ((int64_t)blockIdx.x < tiles) issue_l1();
        unsigned it = 0;
        for (int64_t tile = blockIdx.x; tile < tiles && !aborted(bail); tile += gridDim.x, ++it) {
            // layer 2: D2 = h1 W2^T, A from the resident activation buffer, B from the ring
            for (int i = 0; i < nk2; ++i) {
                const int kc = kc_order(i);                               // h1 chunk kc is ready as soon as its half wrote it
                mbar_wait(a1_ready(kc), it & 1u, bail);
                mbar_wait(full_b(ring.stage), ring.phase, bail);
                tc_fence_after();
                if (lane == 0) {
                    const uint32_t a0 = sbase + OFF_A2 + kc * A_CHUNK_BYTES;
                    const uint32_t b0 = sbase + OFF_RING + ring.stage * STAGE_BYTES + A_CHUNK_BYTES;
#pragma unroll
                    for (int k = 0; k < KC / UMMA_K; ++k)
                        tc_mma(tmem + N_HID, umma_desc(a0 + k * 32), umma_desc(b0 + k * 32), idesc_hid, (i | k) ? 1u : 0u);
                    tc_commit(empty(ring.stage));
                    if (i == nk2 - 1) tc_commit(d2_full);
                }
                __syncwarp();
                ring.advance();
            }
            if (tile + gridDim.x < tiles) issue_l1();          // next tile's layer 1 overlaps this tile's epilogue 2
            // layer 3: D3 = h2 W3^T, both operands resident; D3 takes over D2's columns (E2 has read them)
            // (D3 overwrites D2's first 16 columns: wait for ALL of epilogue 2 before the first layer-3 MMA)
            for (int i = 0; i < nk2; ++i) mbar_wait(a2_ready(i), it & 1u, bail);
            tc_fence_after();
            if (lane == 0) {
                for (int kc = 0; kc < nk2; ++kc) {
                    const uint32_t a0 = sbase + OFF_A2 + kc * A_CHUNK_BYTES, b0 = sbase + OFF_W3 + kc * W3_CHUNK_BYTES;
#pragma unroll
                    for (int k = 0; k < KC / UMMA_K; ++k)
                        tc_mma(tmem + N_HID, umma_desc(a0 + k * 32), umma_desc(b0 + k * 32), idesc_out, (kc | k) ? 1u : 0u);
                }
                tc_commit(d3_full);
            }
            __syncwarp();
        }
    } else if (warp >= 2 + EPI_WARPS) {
        // ===== producers: gather the tile's rows, convert to bf16, write swizzled A chunks (layer 1) ========
        Ring ring;
        const int w = warp - (2 + EPI_WARPS);         // 0 .. PROD_WARPS-1
        constexpr int RPW = M_TILE / PROD_WARPS;      // rows per producer warp
        constexpr int ITS = RPW / 4;                  // 4 rows per warp instruction (8 lanes x 16 bytes per row chunk)
        const int piece = lane & 7, rsub = lane >> 3; // 16-byte piece / row within a 4-row group
        for (int64_t tile = blockIdx.x; tile < tiles && !aborted(bail); tile += gridDim.x) {
            const int64_t row0 = tile * M_TILE;
            // rows this thread gathers: w*RPW + it*4 + rsub
            const float* base_lo[ITS];
            const float* base_hi[ITS];
#pragma unroll
            for (int it = 0; it < ITS; ++it) {
                const int64_t e = row0 + w * RPW + it * 4 + rsub;
                base_lo[it] = base_hi[it] = nullptr;
                if (e < n_rows) {
                    if (P.keys) {
                        const uint64_t k = P.keys[e];
                        base_lo[it] = P.src + (int64_t)(k >> 32) * P.ld;
                        base_hi[it] = P.src + (int64_t)(k & 0xffffffffu) * P.ld;
                    } else {
                        base_lo[it] = P.src + e * P.ld;
                    }
                }
            }
            const int D = P.keys ? P.D : P.in_features, K = P.in_features;
            const bool vec4 = (D % 4 == 0) && (K % 4 == 0) && (P.ld % 4 == 0) && (((uintptr_t)P.src & 15) == 0);
            for (int kc = 0; kc < nk1; ++kc) {
                mbar_wait(empty(ring.stage), ring.phase ^ 1u, bail);
                unsigned char* a_st = smem + OFF_RING + ring.stage * STAGE_BYTES;
                const int k0 = kc * KC + piece * 8;
#pragma unroll
                for (int it = 0; it < ITS; ++it) {
                    float v[8];
                    if (vec4) {                       // D, ld multiples of 4 and a 16-byte aligned base: 128-bit gathers
#pragma unroll
                        for (int q = 0; q < 2; ++q) {
                            const int k = k0 + 4 * q;
                            float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (base_lo[it] && k < K)
                                x = k < D ? __ldg((const float4*)(base_lo[it] + k)) : __ldg((const float4*)(base_hi[it] + (k - D)));
                            v[4 * q] = x.x; v[4 * q + 1] = x.y; v[4 * q + 2] = x.z; v[4 * q + 3] = x.w;
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const int k = k0 + j;
                            float x = 0.f;
                            if (base_lo[it] && k < K) x = k < D ? __ldg(base_lo[it] + k) : __ldg(base_hi[it] + (k - D));
                            v[j] = x;
                        }
                    }
                    const int r = w * RPW + it * 4 + rsub;
                    *(uint4*)(a_st + swz(r, piece)) =
                        make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
                }
                fence_async_smem();                   // generic writes -> visible to the tensor core's async proxy
                __syncwarp();
                if (lane == 0) mbar_arrive(full_a(ring.stage));
                ring.advance();
            }
            // layer 2's ring uses carry no A chunk, but the producers still pace themselves on them: running more
            // than one ring round ahead of the MMA warp would alias the mbarrier phase parity
            for (int kc = 0; kc < nk2; ++kc) {
                mbar_wait(empty(ring.stage), ring.phase ^ 1u, bail);
                ring.advance();
            }
        }
    } else {
        // ===== epilogue warps: accumulator -> bias, leaky ReLU -> next layer's A operand / result ============
        const int quad = warp & 3;                    // TMEM lane quadrant this warp may read
        const int half = (warp - 2) >> 2;             // which half of the 256 columns this warp handles
        unsigned it = 0;
        for (int64_t tile = blockIdx.x; tile < tiles && !aborted(bail); tile += gridDim.x, ++it) {
            const int64_t row0 = tile * M_TILE;
            const int r = quad * 32 + lane;           // accumulator row of this thread
            const int64_t e = row0 + r;
            const uint32_t t_row = tmem + ((uint32_t)(quad * 32) << 16);
            // ---- epilogue 1 / 2: h = lrelu(D + b) -> bf16 A operand (and fp32 h2) ---------------------
#pragma unroll 1
            for (int layer = 0; layer < 2; ++layer) {
                mbar_wait(layer == 0 ? d1_full : d2_full, it & 1u, bail);
                tc_fence_after();
                const float* b = bias + layer * N_HID;
#pragma unroll 1
                for (int c0 = half * (N_HID / 2); c0 < (half + 1) * (N_HID / 2); c0 += 32) {
                    uint32_t v[32];
                    tmem_ld32(t_row + layer * N_HID + c0, v);
                    tmem_ld_wait();
                    float h[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) h[j] = lrelu(__uint_as_float(v[j]) + b[c0 + j]);
                    if (layer == 1 && P.h2 && e < n_rows) {
                        float* dst = P.h2 + e * P.hidden + c0;
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (c0 + j < P.hidden) dst[j] = h[j];
                    }
                    unsigned char* a2 = smem + OFF_A2 + (c0 / KC) * A_CHUNK_BYTES;
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        *(uint4*)(a2 + swz(r, (c0 % KC) / 8 + i)) =
                            make_uint4(pack_bf16(h[8 * i], h[8 * i + 1]), pack_bf16(h[8 * i + 2], h[8 * i + 3]),
                                       pack_bf16(h[8 * i + 4], h[8 * i + 5]), pack_bf16(h[8 * i + 6], h[8 * i + 7]));
                    if ((c0 & (KC - 1)) == KC - 32) {                     // a 64-column chunk is complete: hand it over
                        tc_fence_before();
                        fence_async_smem();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(layer == 0 ? a1_ready(c0 / KC) : a2_ready(c0 / KC));
                    }
                }
            }
            // ---- epilogue 3: o = lrelu(D3 + b3) ------------------------------------------------------
            // every epilogue warp waits (the next tile's h1 must not overwrite h2 before layer 3 has read it)
            mbar_wait(d3_full, it & 1u, bail);
            tc_fence_after();
            if (half == 0) {
                uint32_t v[16];
                tmem_ld16(t_row + N_HID, v);
                tmem_ld_wait();
                if (e < n_rows) {
                    const float* b = bias + 2 * N_HID;
#pragma unroll
                    for (int j = 0; j < N_OUT; ++j)
                        if (j < P.n_out) P.o[e * P.n_out + j] = lrelu(__uint_as_float(v[j]) + b[j]);
                }
            }
            tc_fence_before();
            __syncwarp();
        }
    }

    // ---- teardown -------------------------------------------------------------------------------
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TMEM_COLS) : "memory");
    }
}

// fp32 nn.Linear weights -> padded bf16 chunks in the shared-memory image the tensor core reads
__global__ void pack_kernel(const float* __restrict__ W1, const float* __restrict__ b1, const float* __restrict__ W2,
                            const float* __restrict__ b2, const float* __restrict__ W3, const float* __restrict__ b3,
                            int in_features, int hidden, int n_out, int nk1, unsigned char* __restrict__ packed) {
    const int64_t n_w12 = (int64_t)(nk1 + N_HID / KC) * (B_CHUNK_BYTES / 2);      // bf16 elements of W1 and W2
    const int64_t n_w3 = W3_BYTES / 2;
    const int64_t total = n_w12 + n_w3 + BIAS_FLOATS;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        if (i < n_w12 + n_w3) {
            const bool is3 = i >= n_w12;
            const int64_t j = is3 ? i - n_w12 : i;
            const int chunk_elems = is3 ? W3_CHUNK_BYTES / 2 : B_CHUNK_BYTES / 2;
            const int chunk = (int)(j / chunk_elems);
            const int o = (int)(j % chunk_elems) * 2;                              // byte offset inside the chunk
            const int rr = (o % 1024) / 128, n = (o / 1024) * 8 + rr;
            const int kk = ((((o % 128) / 16) ^ rr) * 8) + (o % 16) / 2;
            float v = 0.f;
            if (is3) {
                const int k = chunk * KC + kk;
                if (n < n_out && k < hidden) v = W3[(int64_t)n * hidden + k];
            } else if (chunk < nk1) {
                const int k = chunk * KC + kk;
                if (n < hidden && k < in_features) v = W1[(int64_t)n * in_features + k];
            } else {
                const int k = (chunk - nk1) * KC + kk;
                if (n < hidden && k < hidden) v = W2[(int64_t)n * hidden + k];
            }
            ((__nv_bfloat16*)packed)[i] = __float2bfloat16_rn(v);
        } else {
            const int t = (int)(i - n_w12 - n_w3);
            float v = 0.f;
            if (t < N_HID) v = t < hidden ? b1[t] : 0.f;
            else if (t < 2 * N_HID) v = (t - N_HID) < hidden ? b2[t - N_HID] : 0.f;
            else v = (t - 2 * N_HID) < n_out ? b3[t - 2 * N_HID] : 0.f;
            ((float*)(packed + off_bias(nk1)))[t] = v;
        }
    }
}

static int check_dims(int64_t in_features, int64_t hidden, int64_t n_out) {
    if (in_features < 1 || in_features > (1 << 20) || hidden < 1 || hidden > N_HID || n_out < 1 || n_out > N_OUT)
        return DM_ERR_BAD_ARG;
    return DM_OK;
}

static int run(const Params& P, int64_t rows_cap, cudaStream_t s) {
    const int64_t tiles = ceil_div(rows_cap, M_TILE);
    const int grid = (int)imax64(1, imin64(tiles, num_sms()));
    return launch(pair_mlp_kernel, grid, THREADS, SMEM_BYTES, s, P);
}

}  // namespace mlp
}  // namespace dm

using namespace dm;

extern "C" size_t dm_mlp_packed_bytes(int64_t in_features, int64_t hidden, int64_t n_out) {
    if (mlp::check_dims(in_features, hidden, n_out) != DM_OK) return 0;
    return mlp::packed_bytes(mlp::nk_for(in_features)) + 16;      // + the status word of the kernel's bounded waits
}

extern "C" size_t dm_mlp_status_offset(int64_t in_features, int64_t hidden, int64_t n_out) {
    if (mlp::check_dims(in_features, hidden, n_out) != DM_OK) return 0;
    return mlp::packed_bytes(mlp::nk_for(in_features));
}

extern "C" int dm_mlp_pack(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                           const float* b3, int64_t in_features, int64_t hidden, int64_t n_out, void* packed,
                           dm_stream_t stream) {
    DM_TRY(mlp::check_dims(in_features, hidden, n_out));
    if (!W1 || !b1 || !W2 || !b2 || !W3 || !b3 || !packed || ((uintptr_t)packed & 15)) return DM_ERR_BAD_ARG;
    const int nk1 = (int)mlp::nk_for(in_features);
    cudaStream_t s = S(stream);
    DM_CUDA(cudaMemsetAsync((unsigned char*)packed + mlp::packed_bytes(nk1), 0, 16, s));
    return launch(mlp::pack_kernel, num_sms() * 4, 256, 0, s, W1, b1, W2, b2, W3, b3, (int)in_features, (int)hidden,
                  (int)n_out, nk1, (unsigned char*)packed);
}

extern "C" int dm_score_mlp_bf16(const float* mean, int64_t D, const uint64_t* edge_keys, const int64_t* n_edges_dev,
                                 int64_t capacity, const void* packed, int64_t in_features, int64_t hidden,
                                 int64_t n_out, float* o, float* h2, dm_stream_t stream) {
    DM_TRY(mlp::check_dims(in_features, hidden, n_out));
    if (capacity < 0 || D < 1 || in_features != 2 * D) return DM_ERR_BAD_ARG;
    if (capacity == 0) return DM_OK;
    if (!mean || !edge_keys || !n_edges_dev || !packed || !o || ((uintptr_t)packed & 15)) return DM_ERR_BAD_ARG;
    mlp::Params P;
    P.src = mean;
    P.ld = D;
    P.keys = edge_keys;
    P.n_dev = n_edges_dev;
    P.n_host = 0;
    P.D = (int)D;
    P.in_features = (int)in_features;
    P.nk1 = (int)mlp::nk_for(in_features);
    P.hidden = (int)hidden;
    P.n_out = (int)n_out;
    P.packed = (const unsigned char*)packed;
    P.o = o;
    P.h2 = h2;
    P.status = (int*)((unsigned char*)packed + mlp::packed_bytes(P.nk1));
    return mlp::run(P, capacity, S(stream));
}

extern "C" int dm_mlp_forward_bf16(const float* x, int64_t B, const void* packed, int64_t in_features, int64_t hidden,
                                   int64_t n_out, float* o, float* h2, dm_stream_t stream) {
    DM_TRY(mlp::check_dims(in_features, hidden, n_out));
    if (B < 0) return DM_ERR_BAD_ARG;
    if (B == 0) return DM_OK;
    if (!x || !packed || !o || ((uintptr_t)packed & 15)) return DM_ERR_BAD_ARG;
    mlp::Params P;
    P.src = x;
    P.ld = in_features;
    P.keys = nullptr;
    P.n_dev = nullptr;
    P.n_host = B;
    P.D = (int)in_features;
    P.in_features = (int)in_features;
    P.nk1 = (int)mlp::nk_for(in_features);
    P.hidden = (int)hidden;
    P.n_out = (int)n_out;
    P.packed = (const unsigned char*)packed;
    P.o = o;
    P.h2 = h2;
    P.status = (int*)((unsigned char*)packed + mlp::packed_bytes(P.nk1));
    return mlp::run(P, B, S(stream));
}
