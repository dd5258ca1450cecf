// R1: region adjacency graph from a label raster, fused with per-region band pooling -- the block / work-list
// formulation of the raster pass.
//
// Why this shape.  The previous kernel (rag.cu) kept a 2-entry label cache per lane and paid for every rare event
// (label change in one lane, junction, boundary crossing a lane edge) with a divergent code path that the whole warp
// waits for: 307 warp instructions per 128-pixel row at 18 active lanes per instruction, 0.32 of the HBM roofline.
// Here rare work is never executed where it is found; it is COMPACTED and executed 32 wide:
//   * a warp walks down a 128-pixel strip in block rows of 4 rows; a lane owns one 4 x 4 block per block row
//     (4 x LDS.128 of labels, 4 x LDS.128 of image bytes from the warp's own TMA-fed stage ring);
//   * fast path (convergent, ~70 % of the blocks): the block's window -- its 16 pixels, the 4 above, the 4 to the right --
//     is one label (12 LOP3 over the 24 values): no pixel pair differs, the 16 pixels are added unmasked (PRMT
//     transposes + DP4A) to the lane's accumulators of its current label; a label change pushes them to the warp's
//     hash table (once per lane per region, batched per block row);
//   * every other block (a boundary, a junction, nodata, an image border) is copied out of the registers into the
//     warp's item buffer as a self-contained ITEM (24 labels, 16 pixels, position; 11 conflict-free STS.128), and as
//     soon as 32 items wait the warp processes them, one per lane, with rag_core.cuh:process_item -- position masks
//     per distinct label, masked DP4A statistics, pair counts by shifted-mask popcounts -- straight into the warp's
//     private shared-memory hash tables (region -> accumulators, edge key -> pair count);
//   * tables drain to global memory (64-bit atomics for regions, appended (key, count) entries for edges) when half
//     full; the appended entries are then sorted and run-reduced (prims.cu) into the sorted unique edge list.
// Staging is unchanged: lane 0 of every warp feeds the warp's own ring with cp.async.bulk.tensor (TH label rows x 132
// columns -- a 4-column halo for the right neighbour -- and TH image rows), completion on the warp's own mbarriers; no
// block-level barrier exists.  The row above a block row is carried in registers.
//
// HBM traffic: labels 4 B/px + image C B/px read once.
#include "rag_tables.cuh"

namespace dm {
namespace rag {
namespace blk {

template <int C_, int TH_, int NS_, int NW_, int ICAP_>
struct Cfg {
    static constexpr int C = C_, TH = TH_, NS = NS_, NWARPS = NW_, ICAP = ICAP_;
    static constexpr int CW = C_ > 0 ? C_ : 1;               // words of image bytes per lane-row
    static constexpr int THREADS = NWARPS * 32;
    static constexpr int LAB_BOX = align128(TH * LAB_PITCH * 4);
    static constexpr int IMG_ROW_WORDS = STRIP_W * C / 4;    // 32*C
    static constexpr int IMG_BOX = align128(TH * IMG_ROW_WORDS * 4);
    static constexpr int STAGE_BYTES = LAB_BOX + IMG_BOX;
    static constexpr int ITEM_VECS = 7 + C;                  // above | 4 own rows | right column | C image vectors | position
    static constexpr int ITEM_BYTES = ICAP * ITEM_VECS * 16;
    static constexpr int TABLE_WORDS = RS * (3 + 2 * C) + ES * 3 + 4;     // + used[2] + pad
    static constexpr int TABLE_BYTES = align128(TABLE_WORDS * 4 + NS * 8);   // + full barriers
    static constexpr int WARP_BYTES = NS * STAGE_BYTES + ITEM_BYTES + TABLE_BYTES;
    static constexpr int SMEM_BYTES = 128 + NWARPS * WARP_BYTES;
    static constexpr int TX_BYTES = TH * LAB_PITCH * 4 + (C > 0 ? TH * IMG_ROW_WORDS * 4 : 0);
    static constexpr int FLUSH_UNITS = FLUSH_ROWS / TH > 0 ? FLUSH_ROWS / TH : 1;
    static_assert(TH % 4 == 0, "a stage holds whole block rows");
    static_assert(ICAP % 8 == 0 && ICAP >= 40, "item buffer: the rest of a pass (< 32 items) plus a block row of new ones");
    static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};

__device__ __noinline__ void slow_wait(uint64_t* bar, unsigned parity, unsigned long long* counters) {
    mbar_wait(bar, parity, counters);
}

// One pass over the newest min(32, icount) items, one per lane.
template <typename CF>
__device__ __noinline__ void item_pass(uint4* items, unsigned* tab, const Params* Pp, int icount, int lane) {
    constexpr int C = CF::C, CW = CF::CW, ICAP = CF::ICAP;
    const Params& P = *Pp;
    const Tab<C> T = Tab<C>::from(tab);
    __syncwarp();
    const int n = min(32, icount), base = icount - n;
    if (lane < n) {
        const int j = base + lane;
        const uint4* it = items + j;
        int lab[ragcore::WIN];
        unsigned img[4 * CW];
        uint4 v = it[0];
        lab[20] = (int)v.x; lab[21] = (int)v.y; lab[22] = (int)v.z; lab[23] = (int)v.w;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            v = it[(1 + r) * ICAP];
            lab[5 * r] = (int)v.x; lab[5 * r + 1] = (int)v.y; lab[5 * r + 2] = (int)v.z; lab[5 * r + 3] = (int)v.w;
        }
        v = it[5 * ICAP];
        lab[4] = (int)v.x; lab[9] = (int)v.y; lab[14] = (int)v.z; lab[19] = (int)v.w;
#pragma unroll
        for (int vi = 0; vi < C; ++vi) {
            v = it[(6 + vi) * ICAP];
            img[4 * vi] = v.x; img[4 * vi + 1] = v.y; img[4 * vi + 2] = v.z; img[4 * vi + 3] = v.w;
        }
        v = it[(6 + C) * ICAP];
        const ragcore::Geo g{P.W, P.rows_own, P.rows_avail, P.top_border, P.bottom_border};
        Sink<C> sink{T, P};
        const ItemPick<ICAP> pick{(const int*)items, j};
        ragcore::process_item<C>(lab, img, (int)v.x, (int)v.y, g, sink, pick);
    }
    __syncwarp();
}

// ------------------------------------------------------------------------------------ //
// the kernel
// ------------------------------------------------------------------------------------ //
template <typename CF, bool USE_TMA>
__global__ void __launch_bounds__(CF::THREADS, 1)
rag_blocks_kernel(const __grid_constant__ CUtensorMap mapL, const __grid_constant__ CUtensorMap mapI,
                  const __grid_constant__ Params P) {
    constexpr int C = CF::C, CW = CF::CW, TH = CF::TH, NS = CF::NS, ICAP = CF::ICAP;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // align by OFFSET (no integer round trip) so that every derived pointer keeps the shared address space
    unsigned char* smem = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);
    // the warp index through a shuffle: provably warp-uniform, so the TMA operands stay in uniform registers
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;
    unsigned char* wbase = smem + (size_t)warp * CF::WARP_BYTES;       // this warp's private arena
    uint4* items = (uint4*)(wbase + NS * CF::STAGE_BYTES);
    unsigned* tab = (unsigned*)(wbase + NS * CF::STAGE_BYTES + CF::ITEM_BYTES);
    const Tab<C> T = Tab<C>::from(tab);
    uint64_t* full_bar = (uint64_t*)(tab + ((CF::TABLE_WORDS + 1) & ~1));

    // ---- this warp's run of units (unit = TH rows of one strip, column-major order) -------
    const long long total_units = (long long)P.tiles_x * P.tiles_y;
    const long long gw = (long long)blockIdx.x * CF::NWARPS + warp;
    // even split over all warps of the grid: runs differ by at most one unit, no SM is left without a CTA
    const long long n_warps = (long long)gridDim.x * CF::NWARPS;
    const long long u_begin = total_units / n_warps * gw + min(gw, total_units % n_warps);
    const long long u_end = u_begin + total_units / n_warps + (gw < total_units % n_warps ? 1 : 0);
    const int my_units = (int)(u_end - u_begin);

    // ---- init (warp-private, no block barrier needed) ---------------------------------------
    T.rkey[lane] = EMPTY_LABEL;
    T.rarea[lane] = 0;
    T.rborder[lane] = 0;
#pragma unroll
    for (int c = 0; c < C; ++c) {
        T.rsum[c * RS + lane] = 0;
        T.rsq[c * RS + lane] = 0;
    }
    T.ekey[lane] = EMPTY_KEY;
    T.ekey[lane + 32] = EMPTY_KEY;
    T.ecnt[lane] = 0;
    T.ecnt[lane + 32] = 0;
    if (lane == 0) {
        T.used[0] = T.used[1] = 0;
        if (USE_TMA) {
            for (int s = 0; s < NS; ++s) mbar_init(&full_bar[s], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
    }
    __syncwarp();
    if (my_units == 0) return;

    // (strip, row block) of the next unit to fetch, advanced incrementally (column-major order)
    int isx = (int)(u_begin / P.tiles_y), ij = (int)(u_begin - (long long)isx * P.tiles_y), issued = 0;
    auto issue = [&]() {          // TMA loads of this warp's next unit into stage issued % NS (lane 0 issues)
        if (lane == 0) {
            const int st = issued % NS;
            unsigned char* sb = wbase + (size_t)st * CF::STAGE_BYTES;
            mbar_expect_tx(&full_bar[st], (unsigned)CF::TX_BYTES);
            tma_load_2d(sb, &mapL, isx * STRIP_W, ij * TH, &full_bar[st]);
            if (C > 0) tma_load_2d(sb + CF::LAB_BOX, &mapI, isx * STRIP_W * C / 4, ij * TH, &full_bar[st]);
        }
        ++issued;
        if (ij + 1 < P.tiles_y) ++ij;
        else { ij = 0; ++isx; }
    };
    if (USE_TMA) {
        for (int k = 0; k < NS && k < my_units; ++k) issue();
    }

    // ---- lane state: the row above, the current label's accumulators, the item count ----------
    int4 up = make_int4(0, 0, 0, 0);
    int cur = EMPTY_LABEL;
    unsigned area = 0, s[CW], q[CW];
#pragma unroll
    for (int c = 0; c < CW; ++c) s[c] = q[c] = 0;
    int icount = 0;                     // items waiting in the buffer (warp-uniform)
    auto lane_flush = [&]() {
        if (cur >= 0 && area) table_region_add<C>(T, P, cur, area, 0u, s, q);
        area = 0;
#pragma unroll
        for (int c = 0; c < CW; ++c) s[c] = q[c] = 0;
    };

    int units_since_flush = 0;
    int sx = (int)(u_begin / P.tiles_y), j = (int)(u_begin - (long long)sx * P.tiles_y);
    bool contiguous = false;            // `up` carries over from the previous unit

    for (int i = 0; i < my_units; ++i) {
        const int st = USE_TMA ? i % NS : 0;
        unsigned char* sb = wbase + (size_t)st * CF::STAGE_BYTES;
        const int strip_x0 = sx * STRIP_W, unit_y0 = j * TH;
        int* Lw = (int*)sb;
        if (USE_TMA) {
            if (!mbar_try_wait(&full_bar[st], (unsigned)(i / NS) & 1u)) slow_wait(&full_bar[st], (unsigned)(i / NS) & 1u, P.counters);
        } else {
            // fallback staging for rasters whose pitch/base TMA cannot describe
            __syncwarp();
            for (int k = lane; k < TH * LAB_PITCH; k += 32) {
                const int r = k / LAB_PITCH, cidx = k - r * LAB_PITCH;
                const int gy = unit_y0 + r, gx = strip_x0 + cidx;
                Lw[k] = (gy < P.rows_avail && gx < P.W) ? P.labels[(int64_t)gy * P.ld + gx] : 0;
            }
            if constexpr (C > 0) {
                unsigned char* Ib = sb + CF::LAB_BOX;
                for (int k = lane; k < TH * CF::IMG_ROW_WORDS * 4; k += 32) {
                    const int r = k / (CF::IMG_ROW_WORDS * 4), bidx = k - r * (CF::IMG_ROW_WORDS * 4);
                    const int gy = unit_y0 + r;
                    const int64_t gb = (int64_t)strip_x0 * C + bidx;
                    Ib[k] = (gy < P.rows_own && gb < (int64_t)P.W * C) ? P.image[(int64_t)gy * P.image_pitch + gb] : 0;
                }
            }
            __syncwarp();
        }

        const int x0 = strip_x0 + 4 * lane;                 // first column of this lane's blocks
        const bool in_img = x0 < P.W;
        const bool forced_x = (x0 == 0) || (x0 + 4 >= P.W);
        if (!contiguous) {
            // first unit of the run / of a strip: the row above comes straight from global memory
            up = make_int4(0, 0, 0, 0);
            if (unit_y0 > 0) {
                const int32_t* row = P.labels + (int64_t)(unit_y0 - 1) * P.ld;
                if (x0 < P.W) up.x = row[x0];
                if (x0 + 1 < P.W) up.y = row[x0 + 1];
                if (x0 + 2 < P.W) up.z = row[x0 + 2];
                if (x0 + 3 < P.W) up.w = row[x0 + 3];
            }
        }

#pragma unroll
        for (int b = 0; b < TH / 4; ++b) {
            const int y0 = unit_y0 + 4 * b;
            if (y0 >= P.rows_avail) break;                          // warp-uniform
            const int* Lp = Lw + (4 * b) * LAB_PITCH + 4 * lane;
            const int4 a0 = *(const int4*)Lp;
            const int4 a1 = *(const int4*)(Lp + LAB_PITCH);
            const int4 a2 = *(const int4*)(Lp + 2 * LAB_PITCH);
            const int4 a3 = *(const int4*)(Lp + 3 * LAB_PITCH);
            int r0 = __shfl_down_sync(0xffffffffu, a0.x, 1);
            int r1 = __shfl_down_sync(0xffffffffu, a1.x, 1);
            int r2 = __shfl_down_sync(0xffffffffu, a2.x, 1);
            int r3 = __shfl_down_sync(0xffffffffu, a3.x, 1);
            if (lane == 31) {                                       // the strip's halo columns start right after lane 31's pixels
                r0 = Lp[4];
                r1 = Lp[LAB_PITCH + 4];
                r2 = Lp[2 * LAB_PITCH + 4];
                r3 = Lp[3 * LAB_PITCH + 4];
            }
            unsigned px[4][CW];
            if constexpr (C > 0) {
                const unsigned* Ip = (const unsigned*)(sb + CF::LAB_BOX) + (4 * b) * CF::IMG_ROW_WORDS + CW * lane;
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    if constexpr (C == 4) {
                        const uint4 v = *(const uint4*)(Ip + r * CF::IMG_ROW_WORDS);
                        px[r][0] = v.x; px[r][1] = v.y; px[r][2] = v.z; px[r][3] = v.w;
                    } else {
#pragma unroll
                        for (int c = 0; c < C; ++c) px[r][c] = Ip[r * CF::IMG_ROW_WORDS + c];
                    }
                }
            }
            // one label in the whole window?  (a closed chain of equalities over the 24 values)
            const unsigned d = or3(or3(or3(eq3(up.x, up.y, up.z), eq3(up.z, up.w, a0.x), eq3(a0.x, a0.y, a0.z)),
                                       or3(eq3(a0.z, a0.w, r0), eq3(r0, a1.x, a1.y), eq3(a1.y, a1.z, a1.w)),
                                       or3(eq3(a1.w, r1, a2.x), eq3(a2.x, a2.y, a2.z), eq3(a2.z, a2.w, r2))),
                                   or3(eq3(r2, a3.x, a3.y), eq3(a3.y, a3.z, a3.w), eq3(a3.w, r3, up.x)), 0u);
            const bool forced = forced_x || (y0 == 0) || (y0 + 4 >= P.rows_own);
            const bool is_item = in_img && (forced || d != 0u);
            const bool is_fast = in_img && !is_item;
            const int ref = a0.x;
            if (is_fast && ref != cur) {                            // the lane enters another region
                lane_flush();
                cur = ref;
            }
            __syncwarp();
            if (is_fast) {
                area += 16u;
                if constexpr (C > 0) {
#pragma unroll
                    for (int r = 0; r < 4; ++r) ragcore::row_stats<C>(px[r], s, q);
                }
            }
            const unsigned bal = __ballot_sync(0xffffffffu, is_item);
            if (bal) {
                if (icount + __popc(bal) > ICAP) {                  // no room: a pass over the waiting items first
                    item_pass<CF>(items, tab, &P, icount, lane);
                    icount -= min(32, icount);
                }
                if (is_item) {
                    uint4* it = items + (icount + __popc(bal & lanemask_lt()));
                    it[0] = make_uint4((unsigned)up.x, (unsigned)up.y, (unsigned)up.z, (unsigned)up.w);
                    it[1 * ICAP] = make_uint4((unsigned)a0.x, (unsigned)a0.y, (unsigned)a0.z, (unsigned)a0.w);
                    it[2 * ICAP] = make_uint4((unsigned)a1.x, (unsigned)a1.y, (unsigned)a1.z, (unsigned)a1.w);
                    it[3 * ICAP] = make_uint4((unsigned)a2.x, (unsigned)a2.y, (unsigned)a2.z, (unsigned)a2.w);
                    it[4 * ICAP] = make_uint4((unsigned)a3.x, (unsigned)a3.y, (unsigned)a3.z, (unsigned)a3.w);
                    it[5 * ICAP] = make_uint4((unsigned)r0, (unsigned)r1, (unsigned)r2, (unsigned)r3);
                    if constexpr (C > 0) {
                        const unsigned* Wf = &px[0][0];
#pragma unroll
                        for (int vi = 0; vi < C; ++vi)
                            it[(6 + vi) * ICAP] = make_uint4(Wf[4 * vi], Wf[4 * vi + 1], Wf[4 * vi + 2], Wf[4 * vi + 3]);
                    }
                    it[(6 + C) * ICAP] = make_uint4((unsigned)x0, (unsigned)y0, 0u, 0u);
                }
                icount += __popc(bal);
            }
            up = a3;
        }
        contiguous = (j + 1 < P.tiles_y);

        // next unit of this warp's run
        if (j + 1 < P.tiles_y) ++j;
        else { j = 0; ++sx; }

        // ---- recycle the stage: this warp is its only reader, so it refills it itself ----------
        __syncwarp();
        if (USE_TMA && i + NS < my_units) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic reads before async writes
            issue();
        }

        // ---- full passes over the waiting items; tables -> global when they fill up -------------
        ++units_since_flush;
        const bool forced_flush = units_since_flush >= CF::FLUSH_UNITS || (i + 1 == my_units);
        if (icount >= 32 || forced_flush) {
            while (icount >= 32 || (forced_flush && icount > 0)) {
                item_pass<CF>(items, tab, &P, icount, lane);
                icount -= min(32, icount);
                if (icount > 0 && (T.used[0] > RS / 2 || T.used[1] > ES / 2)) drain_tables<C>(tab, &P, lane);
            }
            if (forced_flush) {
                lane_flush();
                units_since_flush = 0;
            }
        }
        __syncwarp();
        const uint2 used = *(const uint2*)T.used;
        if (forced_flush || used.x > RS / 2 || used.y > ES / 2) drain_tables<C>(tab, &P, lane);
    }
}

template <typename CF>
static int run(const Params& Pin, cudaStream_t s) {
    Params P = Pin;
    P.tiles_x = (int)ceil_div(P.W, STRIP_W);            // strips
    P.tiles_y = (int)ceil_div(P.rows_avail, CF::TH);    // units per strip (a halo row below counts)
    const long long total = (long long)P.tiles_x * P.tiles_y;
    if (total == 0) return DM_OK;
    // one persistent CTA per SM; every warp takes one contiguous run of units
    const long long max_warps = (long long)num_sms() * CF::NWARPS;
    const long long per = ceil_div(total, max_warps);
    if (per > 0x7fffffff) return DM_ERR_BAD_ARG;
    P.tiles_per_cta = (int)per;
    const int grid = (int)imin64(num_sms(), ceil_div(total, CF::NWARPS));   // (a tiny raster: one unit per warp)

    CUtensorMap mapL, mapI;
    memset(&mapL, 0, sizeof(mapL));
    memset(&mapI, 0, sizeof(mapI));
    // TMA needs 16-byte aligned bases and row pitches; anything else takes the ld.global staging path
    bool tma = ((uintptr_t)P.labels % 16 == 0) && ((P.ld * 4) % 16 == 0) && P.ld >= P.W;
    if (CF::C > 0)
        tma = tma && ((uintptr_t)P.image % 16 == 0) && (P.image_pitch % 16 == 0) && (((int64_t)P.W * CF::C) % 4 == 0);
    if (tma)
        tma = make_map_2d(&mapL, P.labels, (uint64_t)P.W, (uint64_t)P.rows_avail, (uint64_t)P.ld * 4, LAB_PITCH, CF::TH);
    if (tma && CF::C > 0)
        tma = make_map_2d(&mapI, P.image, (uint64_t)P.W * CF::C / 4, (uint64_t)P.rows_own, (uint64_t)P.image_pitch,
                          CF::IMG_ROW_WORDS, CF::TH);
    set_last_path(tma ? 1 : 0);
    return launch(tma ? rag_blocks_kernel<CF, true> : rag_blocks_kernel<CF, false>, grid, CF::THREADS, CF::SMEM_BYTES, s,
                  mapL, mapI, P);
}

}  // namespace blk

// Kernel shapes per band count: <bands, rows per stage, stages, warps per CTA, item capacity>.
int run_blocks(const Params& P, int C, cudaStream_t s) {
    using namespace blk;
    switch (C) {
        case 0: return run<Cfg<0, 8, 2, 14, 48>>(P, s);
        case 1: return run<Cfg<1, 4, 2, 16, 48>>(P, s);
        case 2: return run<Cfg<2, 4, 2, 14, 48>>(P, s);
        case 3: return run<Cfg<3, 4, 2, 12, 48>>(P, s);
        case 4: return run<Cfg<4, 4, 2, 12, 48>>(P, s);
        default: return DM_ERR_BAD_ARG;
    }
}

}  // namespace rag
}  // namespace dm
