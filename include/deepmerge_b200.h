/*
 * deepmerge_b200 -- C ABI of the B200-native DeepMerge region-merging hot path.
 *
 * The reference (lvxianwei/DeepMerge) is pure Python and has no FFI: its callers use
 * plain Python callables.  "Drop-in" therefore means same-named Python callables
 * (package deepmerge_b200, see INTEGRATION.md) backed by this library.  Each entry
 * point below names the reference code it replaces (file:line in /root/reference) or
 * the SURVEY.md section 8(a) row whose written spec it implements when the reference
 * has no code for the stage.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless its name ends in _host;
 *  - the caller owns every buffer including workspaces (query *_workspace_bytes, allocate,
 *    pass); the library allocates nothing persistent and keeps no mutable state between calls -- except three
 *    DIAGNOSTICS that no result depends on: dm_launch_count() (a process-wide counter, incremented atomically),
 *    dm_last_cuda_error() and dm_rag_last_path() / dm_rag_last_encode_error() (thread-local: they describe the last call
 *    of the calling thread).  Everything else is re-entrant: concurrent calls from different host threads on different
 *    streams / devices are safe;
 *  - all work is enqueued on `stream` (a cudaStream_t) and is asynchronous;
 *  - variable-size results use capacity + device-side counts: `counts` arrays live on
 *    the device so that dependent calls chain without a host round trip;
 *  - return value 0 = DM_OK, negative = error (dm_error_string); no exception crosses
 *    the ABI, the library never exits the process;
 *  - region ids are int32 in [0, n_regions); negative labels are nodata;
 *  - an edge key is (uint64)min(u,v) << 32 | max(u,v).
 */
#ifndef DEEPMERGE_B200_H
#define DEEPMERGE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* dm_stream_t; /* cudaStream_t */

enum {
    DM_OK = 0,
    DM_ERR_BAD_ARG = -1,      /* null pointer, negative extent, unsupported C / D ...       */
    DM_ERR_WORKSPACE = -2,    /* workspace smaller than *_workspace_bytes reports           */
    DM_ERR_CUDA = -3,         /* a CUDA call failed; dm_last_cuda_error() holds the code    */
    DM_ERR_UNSUPPORTED = -4,  /* device is not sm_100 class, or driver lacks a needed entry */
    DM_ERR_CAPACITY = -5      /* capacity argument too small to even start                  */
};

int dm_version(void);
const char* dm_error_string(int code);
int dm_last_cuda_error(void);   /* cudaError_t of the last DM_ERR_CUDA on this thread */
int dm_num_sms(void);           /* SM count of the current device (148 on B200), <0 on error */
int64_t dm_launch_count(void);  /* kernels of this library accepted by the runtime in this process (all threads) */
void dm_launch_count_add(int64_t n);  /* a host layer that replays a CUDA graph captured from n of this library's launches
                                         reports them here (the counter itself only sees the capture) */

/* ----------------------------------------------------------------------------------- *
 * Primitives (exported so that tests can pin them individually)
 * ----------------------------------------------------------------------------------- */

/* Stable LSD radix sort of (key,value) pairs on the bit range implied by n_regions
 * (both 32-bit halves of an edge key are < n_regions), one cooperative launch.
 * n = min(n_dev[0], capacity) is read on the device.  Sorted output is left in keys/vals
 * (vals nullable).  DM_ERR_UNSUPPORTED on a device without cooperative launch. */
size_t dm_sort_edges_workspace_bytes(int64_t capacity);
int dm_sort_edges(uint64_t* keys, uint32_t* vals, const int64_t* n_dev, int64_t capacity,
                  int64_t n_regions, void* ws, size_t ws_bytes, dm_stream_t stream);

/* Exclusive prefix sum of uint32 -> uint32; total written to total_dev[0] (int64). */
size_t dm_scan_workspace_bytes(int64_t capacity);
int dm_scan_exclusive_u32(const uint32_t* in, uint32_t* out, const int64_t* n_dev, int64_t capacity,
                          int64_t* total_dev, void* ws, size_t ws_bytes, dm_stream_t stream);

/* ----------------------------------------------------------------------------------- *
 * R1  Region adjacency graph from a label raster, fused with band pooling.
 *     Replaces the edge list the reference READS from lines.shp
 *     (MyUtils2.py:155-193 PolygonConnectPointDataset.add_data; LEFT_FID/RIGHT_FID,
 *     -1 rows dropped :184-186) and the area / peri / mean* / std* attribute-table
 *     fields it reads per polygon (MyUtils1.py:79-114).  Raster semantics: SURVEY.md
 *     section 8(a) R1 (4-adjacency, nodata < 0 skipped).
 *
 * labels   int32 [rows_avail, ld]; the tile OWNS rows [0, rows_own); rows_avail is
 *          rows_own or rows_own+1 (one halo row below, used only as lower neighbour).
 * image    uint8 [rows_own, W, C] with row pitch image_pitch bytes, or NULL (C ignored).
 * top_border / bottom_border: whether row 0 / row rows_own-1 touch the image border
 *          (false for interior row tiles of a sharded scene).
 * area, border, band_sum, band_sumsq: int64/uint64 accumulators [n_regions(,C)], ADDED to
 *          (caller zeroes them).  border counts pixel sides facing the image border or
 *          nodata; perimeter = border + sum of incident boundary lengths (dm_perimeter).
 * edge_keys / boundary_len [capacity]: sorted unique edges and their pixel-pair counts.
 * counts   int64 [4] device: [0] = E unique edges, [1] = raw per-CTA entries produced,
 *          [2] = overflow flag (raw entries exceeded capacity: results invalid, retry
 *          with capacity >= counts[1]), [3] = reserved.
 * ----------------------------------------------------------------------------------- */
size_t dm_rag_workspace_bytes(int64_t capacity);
int dm_rag_build(const int32_t* labels, int64_t rows_own, int64_t rows_avail, int64_t W, int64_t ld,
                 const uint8_t* image, int64_t C, int64_t image_pitch, int64_t n_regions,
                 int top_border, int bottom_border,
                 int64_t* area, int64_t* border, uint64_t* band_sum, uint64_t* band_sumsq,
                 uint64_t* edge_keys, uint32_t* boundary_len, int64_t capacity, int64_t* counts,
                 void* ws, size_t ws_bytes, dm_stream_t stream);

/* The two phases of dm_rag_build, exported separately so that the raster pass (one kernel,
 * the HBM-bound part) can be timed and profiled on its own:
 *   dm_rag_scan   zeroes counts, runs the fused raster kernel: accumulators updated, raw
 *                 per-CTA (key,count) entries appended inside the workspace, counts[1..3] set;
 *   dm_rag_finish run reduction of the raw entries (one cooperative launch, normally through a
 *                 hash table and per-region buckets instead of a sort) -> ascending unique
 *                 edge_keys, summed boundary_len, counts[0].  Same ws / capacity as the scan call. */
int dm_rag_scan(const int32_t* labels, int64_t rows_own, int64_t rows_avail, int64_t W, int64_t ld,
                const uint8_t* image, int64_t C, int64_t image_pitch, int64_t n_regions,
                int top_border, int bottom_border,
                int64_t* area, int64_t* border, uint64_t* band_sum, uint64_t* band_sumsq,
                int64_t capacity, int64_t* counts, void* ws, size_t ws_bytes, dm_stream_t stream);
int dm_rag_finish(uint64_t* edge_keys, uint32_t* boundary_len, int64_t capacity, int64_t n_regions,
                  int64_t* counts, void* ws, size_t ws_bytes, dm_stream_t stream);

/* Which staging path the last dm_rag_scan on this thread took: 1 = TMA (cp.async.bulk.tensor),
 * 0 = ld.global (pitch / base not 16-byte aligned), -1 = none yet; and the
 * CUresult of the last cuTensorMapEncodeTiled (-1: driver entry point missing). */
int dm_rag_last_path(void);
int dm_rag_last_encode_error(void);

/* Sort + unique (summing lengths) an arbitrary concatenation of (key,len) lists: used to
 * merge the per-tile lists of a sharded scene and inside the merge loop.  In place. */
size_t dm_edges_unique_workspace_bytes(int64_t capacity);
int dm_edges_sort_unique(uint64_t* keys, uint32_t* lens, const int64_t* n_in_dev, int64_t capacity,
                         int64_t n_regions, int64_t* n_out_dev, void* ws, size_t ws_bytes, dm_stream_t stream);

/* Concatenate `n_lists` edge lists that sit in equal-sized slots of one buffer (slot g = entries
 * [g*slot_capacity, g*slot_capacity + counts[g])), e.g. the all-gathered per-tile lists of a sharded scene,
 * into dst (valid entries only, slot order kept); n_out_dev[0] = total.  counts: int64 [n_lists] on the
 * device.  No host round trip: the lengths never leave the GPU.  A slot count above slot_capacity or a
 * total above dst_capacity sets n_out_dev[1] = 1 (n_out_dev has 2 entries). */
int dm_edges_concat(const uint64_t* src_keys, const uint32_t* src_lens, const int64_t* counts, int64_t n_lists,
                    int64_t slot_capacity, uint64_t* dst_keys, uint32_t* dst_lens, int64_t dst_capacity,
                    int64_t* n_out_dev, dm_stream_t stream);

/* perimeter[r] = border[r] + sum of boundary_len over edges incident to r; a key whose two ids are not both in
 * [0, n_regions) (the (R, R) sentinel, ~0) adds nothing. */
int dm_perimeter(const uint64_t* edge_keys, const uint32_t* boundary_len, const int64_t* n_edges_dev,
                 int64_t capacity, const int64_t* border, int64_t* perimeter, int64_t n_regions,
                 dm_stream_t stream);

/* ----------------------------------------------------------------------------------- *
 * R3-R5  Region -> sample-point membership and mean pooling.
 *     dm_points_region: raster form of the PointID membership (ExtractFeatures.py:175-179):
 *         region_of_point[i] = labels[ys[i], xs[i]]  (-1 when outside or nodata).
 *     dm_csr_build: group point ids by region, ascending point id inside a region.
 *     dm_pool_points_csr: ExtractFeatures.py:188-212 -- rows gathered in membership order,
 *         sequential fp32 accumulation (np.mean(axis=0) semantics), one warp per region.
 *         sum fp32 [R,D], cnt int32 [R].  Bit-exact with the reference's np.mean after
 *         dm_region_mean.
 * ----------------------------------------------------------------------------------- */
int dm_points_region(const int32_t* labels, int64_t H, int64_t W, int64_t ld, const int32_t* xs,
                     const int32_t* ys, int64_t n_points, int32_t* region_of_point, dm_stream_t stream);
/* Grows with n_regions once n_regions + 1 exceeds 4 n_points + 65536 (per-region arrays of
 * the bucket sort).  dm_csr_build: n_points <= INT32_MAX (point ids are int32). */
size_t dm_csr_workspace_bytes(int64_t n_points, int64_t n_regions);
int dm_csr_build(const int32_t* region_of_point, int64_t n_points, int64_t n_regions, int64_t* offsets,
                 int32_t* point_ids, void* ws, size_t ws_bytes, dm_stream_t stream);
int dm_pool_points_csr(const int64_t* offsets, const int32_t* point_ids, const float* feats, int64_t feat_ld,
                       int64_t n_regions, int64_t D, float* sum, int32_t* cnt, dm_stream_t stream);
/* The same for the engine of one row tile of a sharded scene (ids are global, the tile's points fall into a small interval
 * of them): region_range (device, int64[2] = first and last region id with a point, from dm_points_id_range; NULL = every
 * region, which is dm_pool_points_csr) limits the pass to that interval: cnt becomes 0 for every region outside it and
 * the sum rows outside are left untouched, so that the pass costs what the tile's own regions cost. */
int dm_pool_points_csr_tile(const int64_t* offsets, const int32_t* point_ids, const float* feats, int64_t feat_ld,
                            int64_t n_regions, int64_t D, float* sum, int32_t* cnt, const int64_t* region_range,
                            dm_stream_t stream);
int dm_points_id_range(const int32_t* region_of_point, int64_t n_points, int64_t n_regions, int64_t* range,
                       dm_stream_t stream);
/* dm_pool_points_csr followed by dm_region_mean(only = NULL) in one pass over the points (D <= 128, else
 * DM_ERR_UNSUPPORTED): the same sum, cnt, mean and norm2, bit for bit. */
int dm_pool_points_csr_mean(const int64_t* offsets, const int32_t* point_ids, const float* feats, int64_t feat_ld,
                            int64_t n_regions, int64_t D, float* sum, int32_t* cnt, float* mean, float* norm2,
                            dm_stream_t stream);
/* mean[r] = sum[r] / cnt[r] (IEEE fp32 division), norm2[r] = sum_d mean[r,d]^2.  A region without sample points
 * (cnt[r] == 0) gets mean = norm2 = NaN -- what np.mean over no rows gives -- so that its edges score NaN
 * (dm_score_l2) / NaN logits (dm_score_mlp_bf16) and are never selected by dm_merge_select_*.
 * `only` (nullable) restricts the update to regions with only[r] != 0. */
int dm_region_mean(const float* sum, const int32_t* cnt, int64_t n_regions, int64_t D, float* mean,
                   float* norm2, const uint8_t* only, dm_stream_t stream);

/* Per-pixel embedding pooling (north-star raster form of R5): emb is fp32 or bf16
 * [H, W, D] (dtype_bf16 != 0 selects bf16); accumulates fp32 sums [R,D] and int32 counts. */
int dm_pool_dense(const int32_t* labels, int64_t H, int64_t W, int64_t ld, const void* emb, int dtype_bf16,
                  int64_t D, int64_t n_regions, float* sum, int32_t* cnt, dm_stream_t stream);

/* Per-boundary pooling of a dense embedding grid (north-star "per-boundary feature vectors"; the reference
 * itself only writes one scalar per boundary, ExtractFeatures.py:217-219): for every 4-adjacent pixel pair
 * with two different valid labels, both pixels' embeddings are ADDED to bsum[e] (fp32 [E, D]) of the edge e
 * of that label pair and bcnt[e] (int32) grows by 2, so that mean = bsum / bcnt and bcnt = 2 * boundary_len.
 * edge_keys must be the sorted unique list of dm_rag_build; pairs whose key is not in it are skipped.
 * Row tiles: the tile owns pairs (y, y+1) for its rows y; emb must then hold rows_avail rows. */
int dm_pool_boundary(const int32_t* labels, int64_t rows_own, int64_t rows_avail, int64_t W, int64_t ld,
                     const void* emb, int dtype_bf16, int64_t D, const uint64_t* edge_keys,
                     const int64_t* n_edges_dev, int64_t capacity, float* bsum, int32_t* bcnt, dm_stream_t stream);

/* "Next" row N1, first piece: batched zero-padded window cut around sample points with the semantics of
 * ExtractFeatureDataset.cut_image (MyUtils2.py:330-360) on a band-major uint8 raster [C, H, W] (what GDAL
 * ReadAsArray returns): out uint8 [n, C, size, size], out[i,c,v,u] = image[c, y0[i]+v, x0[i]+u] or 0 outside.
 * (x0, y0) = calculate_left_top_point_and_size(XPixel, YLine, size), MyUtils2.py:379-383. */
int dm_cut_windows(const uint8_t* image, int64_t C, int64_t H, int64_t W, const int32_t* x0, const int32_t* y0,
                   int64_t n, int64_t size, uint8_t* out, dm_stream_t stream);

/* "Next" row N1, second piece: ExtractFeatureDataset.resize_data (MyUtils2.py:362-376) for a batch of square
 * uint8 planes [n_planes, s, s] (windows x bands of dm_cut_windows): cv2.resize(.., (t, t), INTER_AREA) bit for
 * bit, then float32 / 255 -> out float32 [n_planes, t, t].
 *   mode 0: s % t == 0 (integer shrink or copy), no tables.
 *   mode 1: fractional shrink; ti = start[t + 1] ++ src[E] (int32), tf = weight[E] (float32): entries
 *           start[d] .. start[d + 1] - 1 of destination index d, the same table for both axes.
 *   mode 2: enlargement; ti = sx[t] ++ a0[t] ++ a1[t] ++ xmax (int32), tf unused.
 * The tables depend on (s, t) only; deepmerge_b200.MyUtils2.area_tables builds them. */
int dm_resize_area(const uint8_t* patches, int64_t n_planes, int64_t s, int64_t t, int mode, const int32_t* ti,
                   const float* tf, float* out, dm_stream_t stream);

/* ----------------------------------------------------------------------------------- *
 * R6  Edge score = Euclidean distance between pooled means, the reference's expanded
 *     formula sqrt(max(0,|x|^2+|y|^2-2x.y)) in fp32 (ExtractFeatures.py:119-147, called
 *     with n=m=1 per edge at :215).  One warp per edge.
 *     `rescore` (nullable, uint8 [R]): when given, only edges with a flagged endpoint are
 *     recomputed; the others keep scores[e].
 * ----------------------------------------------------------------------------------- */
int dm_score_l2(const float* mean, const float* norm2, int64_t D, const uint64_t* edge_keys,
                const int64_t* n_edges_dev, int64_t capacity, const uint8_t* rescore, float* scores,
                dm_stream_t stream);
/* Dense [n,m] distance matrix with the same formula: the Euclidean_distance(X,Y) /
 * MC_Lyu_2020(X,Y) drop-in (ExtractFeatures.py:119, :228). */
int dm_euclidean_matrix(const float* X, const float* Y, int64_t n, int64_t m, int64_t p, float* D,
                        dm_stream_t stream);

/* ----------------------------------------------------------------------------------- *
 * R8  Pair-MLP scorer with the layer structure of Nets.MLP.forward (Nets.py:28-35):
 *     three Linear + leaky_relu(0.01).  x_e = concat(mean[lo], mean[hi]) (K = 2D), hidden
 *     H1 = H2 <= 256, out <= 16.  bf16 operands, fp32 accumulation on tcgen05 tensor cores
 *     with TMEM accumulators.  Weights are fp32 row-major [out_features, in_features] as in
 *     torch.nn.Linear; dm_mlp_pack converts them once into the padded bf16 UMMA layout.
 *     o [E, n_out] fp32; h2 (nullable) [E, hidden] fp32.
 *     Every wait inside the kernel is bounded.  A wait that expires (a lost TMA / tensor-core signal) neither hangs nor
 *     traps: the CTA abandons its remaining tiles and the int32 STATUS WORD at byte dm_mlp_status_offset(...) of the
 *     packed blob becomes 1 (outputs invalid).  dm_mlp_pack clears it; read it after synchronising the stream.
 */
size_t dm_mlp_packed_bytes(int64_t in_features, int64_t hidden, int64_t n_out);
size_t dm_mlp_status_offset(int64_t in_features, int64_t hidden, int64_t n_out);
int dm_mlp_pack(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                const float* b3, int64_t in_features, int64_t hidden, int64_t n_out, void* packed,
                dm_stream_t stream);
int dm_score_mlp_bf16(const float* mean, int64_t D, const uint64_t* edge_keys, const int64_t* n_edges_dev,
                      int64_t capacity, const void* packed, int64_t in_features, int64_t hidden,
                      int64_t n_out, float* o, float* h2, dm_stream_t stream);
/* Same network on rows of a dense matrix x [B, in_features] (the Nets.MLP()(x) drop-in). */
int dm_mlp_forward_bf16(const float* x, int64_t B, const void* packed, int64_t in_features, int64_t hidden,
                        int64_t n_out, float* o, float* h2, dm_stream_t stream);

/* ----------------------------------------------------------------------------------- *
 * R9  Merge loop building blocks (spec: SURVEY.md section 8(a) R9; the reference scores
 *     edges, ExtractFeatures.py:150-225, and never merges).
 *
 * dm_merge_select_l2 / _mlp: flag edges with score < tau / o[e,1] > o[e,0]; counts[0] =
 *     number selected.
 * dm_uf_union: lock-free union over the selected edges, hooking the larger root under
 *     the smaller (atomicCAS), so every component's root is its minimum id.
 * dm_uf_compress: parent[x] = root(x) for all x.
 * dm_merge_apply: for every region that stopped being a root this round: add its cnt /
 *     area / perimeter into the root (integer atomics), emit (root, member) pairs; then
 *     sums are accumulated per root in ASCENDING member id (sequential fp32), and
 *     changed[root] = 1.  alive[x] is cleared for absorbed regions.
 * dm_edges_rekey: edges -> (root(u), root(v)); self loops removed and 2*len subtracted
 *     from perimeter[root]; result sorted + unique with lengths summed.
 * dm_relabel: labels_out[p] = root[labels[p]] (nodata kept), 128-bit loads/stores.
 * ----------------------------------------------------------------------------------- */
int dm_merge_select_l2(const float* scores, float tau, const int64_t* n_edges_dev, int64_t capacity,
                       uint8_t* selected, int64_t* n_selected_dev, dm_stream_t stream);
int dm_merge_select_mlp(const float* o, int64_t n_out, const int64_t* n_edges_dev, int64_t capacity,
                        uint8_t* selected, int64_t* n_selected_dev, dm_stream_t stream);
int dm_uf_union(int32_t* parent, const uint64_t* edge_keys, const uint8_t* selected,
                const int64_t* n_edges_dev, int64_t capacity, dm_stream_t stream);
int dm_uf_compress(int32_t* parent, int64_t n_regions, dm_stream_t stream);
size_t dm_merge_apply_workspace_bytes(int64_t n_regions);
int dm_merge_apply(const int32_t* parent, uint8_t* alive, uint8_t* changed, float* sum, int32_t* cnt,
                   int64_t* area, int64_t* perimeter, int64_t n_regions, int64_t D, int64_t* n_merged_dev,
                   void* ws, size_t ws_bytes, dm_stream_t stream);
/* dm_merge_apply restricted for row-tile sharding: counts / areas / perimeters of every absorbed region are merged,
 * but embedding sums only for components whose root has root_mask[root] != 0 (nullable = all). */
int dm_merge_apply_masked(const int32_t* parent, uint8_t* alive, uint8_t* changed, float* sum, int32_t* cnt,
                          int64_t* area, int64_t* perimeter, int64_t n_regions, int64_t D, int64_t* n_merged_dev,
                          const uint8_t* root_mask, void* ws, size_t ws_bytes, dm_stream_t stream);
size_t dm_edges_rekey_workspace_bytes(int64_t capacity);
int dm_edges_rekey(const int32_t* parent, uint64_t* edge_keys, uint32_t* boundary_len, float* scores,
                   int64_t* n_edges_dev, int64_t capacity, int64_t n_regions, int64_t* perimeter,
                   void* ws, size_t ws_bytes, dm_stream_t stream);
int dm_relabel(const int32_t* labels, int64_t H, int64_t W, int64_t ld_in, const int32_t* root,
               int64_t n_regions, int32_t* labels_out, int64_t ld_out, dm_stream_t stream);
/* The same, enqueued before the host knows whether the merge loop goes on: the kernel does nothing when
 * *skip_if_nonzero != 0 (device memory: the count of edges the last selection picked; NULL = dm_relabel).  The loop's last
 * read-back then does not leave the device idle. */
int dm_relabel_gated(const int32_t* labels, int64_t H, int64_t W, int64_t ld_in, const int32_t* root, int64_t n_regions,
                     int32_t* out, int64_t ld_out, const int64_t* skip_if_nonzero, dm_stream_t stream);
/* compact[r] = rank of root(r) among roots (ascending); n_roots_dev[0] = number of roots. */
size_t dm_compact_roots_workspace_bytes(int64_t n_regions);
int dm_compact_roots(const int32_t* root, int64_t n_regions, int32_t* compact, int64_t* n_roots_dev,
                     void* ws, size_t ws_bytes, dm_stream_t stream);

/* ----------------------------------------------------------------------------------- *
 * Merge by spectral and shape heterogeneity: the fusion criterion of multiresolution segmentation (Baatz, M. and
 * Schaepe, A., 2000, "Multiresolution Segmentation: an optimization approach for high quality multi-scale image
 * segmentation"), computed from the statistics of the raster pass alone, so that no embedding is needed.  It
 * reproduces, for merged candidates, the area / peri / mean<c> / std<c> / smooth / compact columns of the reference's
 * polygon tables (MyUtils1.py:79-114), which the multiresolution segmentation behind its initial segments wrote.
 *
 * Region i: n = area, l = perimeter, b = 2 (w + h) of its bounding box (bbox int32 [R, 4] as dm_region_bbox), per band
 * c the exact sums S_ic, Q_ic (band_sum / band_sumsq [R, C]) and sigma_ic = sqrt(max(Q/n - (S/n)^2, 0)).  The merged
 * candidate m of an edge (a, b) with boundary length L has n_a + n_b pixels, the summed band sums, l_a + l_b - 2 L and
 * the union of the two boxes; then, all in fp64 from the integers (every operation rounded once, no fused multiply-add):
 *     h_color  = sum_c w_c (n_m sigma_mc - (n_a sigma_ac + n_b sigma_bc))          (c ascending, from 0.0)
 *     h_cmpct  = n_m l_m / sqrt(n_m) - (n_a l_a / sqrt(n_a) + n_b l_b / sqrt(n_b))
 *     h_smooth = n_m l_m / b_m - (n_a l_a / b_a + n_b l_b / b_b)
 *     f = (1 - w_shape) h_color + w_shape (w_cmpct h_cmpct + (1 - w_cmpct) h_smooth)
 * dm_score_spectral: scores[e] = (float) f(e); w_shape, w_cmpct in [0, 1], band_weights float [C] (NULL = ones) are
 *     widened exactly.  `rescore` (nullable, uint8 [R]) as for dm_score_l2.
 * dm_merge_select_mutual: local mutual best fitting.  Edge e is selected iff scores[e] < threshold and e holds the
 *     minimum of (score, edge index) over the edges of both of its endpoints (edges not below the threshold, NaN
 *     included, take no part; -0 and +0 are equal).  Every region takes part in at most one merge per round, and
 *     the global minimum edge is always selected while any edge is below the threshold.  One atomicMin pass on
 *     (ordered score bits << 32 | edge index) keys into the workspace (8 bytes a region), one decision pass;
 *     n_selected_dev[0] = number selected.  capacity < 2^32.
 * dm_merge_apply_regions: the integer-only counterpart of dm_merge_apply for a loop without embeddings: every region
 *     that stopped being a root this round adds its area, perimeter, band sums and sums of squares into the root
 *     (integer atomics) and widens the root's box (atomicMin / atomicMax); alive[x] cleared, changed[root] = 1 (changed
 *     is cleared first), n_merged_dev[0] = regions absorbed.  No workspace.
 * A round: select -> dm_uf_union + dm_uf_compress -> dm_merge_apply_regions -> dm_edges_rekey -> dm_score_spectral
 * (rescore = changed) -> select.
 * ----------------------------------------------------------------------------------- */
int dm_score_spectral(const uint64_t* edge_keys, const uint32_t* boundary_len, const int64_t* n_edges_dev,
                      int64_t capacity, const int64_t* area, const int64_t* perimeter, const uint64_t* band_sum,
                      const uint64_t* band_sumsq, int64_t C, const int32_t* bbox, const float* band_weights,
                      float w_shape, float w_cmpct, const uint8_t* rescore, float* scores, dm_stream_t stream);
size_t dm_merge_select_mutual_workspace_bytes(int64_t n_regions);
int dm_merge_select_mutual(const float* scores, float threshold, const uint64_t* edge_keys, const int64_t* n_edges_dev,
                           int64_t capacity, int64_t n_regions, uint8_t* selected, int64_t* n_selected_dev, void* ws,
                           size_t ws_bytes, dm_stream_t stream);
int dm_merge_apply_regions(const int32_t* parent, uint8_t* alive, uint8_t* changed, int64_t* area, int64_t* perimeter,
                           uint64_t* band_sum, uint64_t* band_sumsq, int64_t C, int32_t* bbox, int64_t n_regions,
                           int64_t* n_merged_dev, dm_stream_t stream);

/* ----------------------------------------------------------------------------------- *
 * Row-tile sharding helpers (SURVEY.md section 8(e)): the sparse exchanges of the owner-free
 * distributed merge loop (deepmerge_b200/sharded.py).
 * dm_mark_endpoints: flags[lo] = flags[hi] = 1 for every edge of the list (regions this tile sees); a key whose two ids
 *                    are not both in [0, n_regions) (the (R, R) sentinel, ~0) is skipped.
 * dm_rows_pack:  rows of the regions with flag[r] != 0 -> (out_ids, out_rows) in arbitrary order;
 *                n_out_dev[0] = number of flagged regions (> capacity: the slot overflowed).
 * dm_rows_unpack: rows[ids[i]] = in_rows[i] (add == 0) or += (add != 0); ids distinct within a call.
 * ----------------------------------------------------------------------------------- */
 /* dm_shard_propagate: mask[root] |= mask[x] for every region absorbed this round (bit g = rank g sees it);
 *                     grew[root] = 1.   dm_shard_plan: send[x] = this rank ships x's embedding sum (see sharded.py),
 *                     seen_comp[r] = this rank sees component r. */
int dm_shard_propagate(const int32_t* parent, const uint8_t* alive, int32_t* mask, uint8_t* grew, int64_t n_regions,
                       dm_stream_t stream);
int dm_shard_plan(const int32_t* parent, const uint8_t* alive, const int32_t* mask_old, const int32_t* mask_new,
                  const uint8_t* grew, int rank, int64_t n_regions, uint8_t* send, uint8_t* seen_comp,
                  dm_stream_t stream);
/* fused per-region glue: dm_shard_seen: seen[r] |= area[r] > 0; mask_cnt[r] = seen ? 1 << rank : 0; mask_cnt[R + r] =
 * cnt_local[r] = cnt[r] (the buffer that is all-reduced).  dm_shard_frontier (after the all-reduce): cnt[r] = global count,
 * send[r] = region seen by two ranks and this rank has points of it. */
int dm_shard_seen(const int64_t* area, uint8_t* seen, const int32_t* cnt, int rank, int64_t n_regions,
                  int32_t* mask_cnt, int32_t* cnt_local, dm_stream_t stream);
int dm_shard_frontier(const int32_t* mask_cnt, const int32_t* cnt_local, int64_t n_regions, int32_t* cnt, uint8_t* send,
                      dm_stream_t stream);
/* Distributed union-find by FRONTIER EXCHANGE (one all-gather of a few hundred pairs per round, no iteration): a component
 * can span two row tiles only through a region both ranks see.  After its local unions (dm_uf_union + dm_uf_compress) a
 * rank writes, for every alive component x it shares with another rank (mask[x] has its bit and another one) and whose
 * local root differs from x, the pair (x << 32 | root) into a slot [int64 count | int64 pad | int64 flags[8] | u64
 * pairs[capacity]] (dm_shard_frontier_pairs; count > capacity = overflow, nothing is written beyond capacity; the eight
 * flag words are the caller's: the round's "edges selected" count and error flags travel with the pairs).  The slots of all ranks are
 * all-gathered and dm_uf_union_slots unites every pair of every slot into the rank's own forest; after dm_uf_compress the
 * regions a rank sees point at their GLOBAL root (the minimum id of the component: a local root is the minimum of its
 * local component and it is part of a pair).  One all_reduce(MIN) of parent then fills in the regions a rank does not see. */
int dm_shard_frontier_pairs(const int32_t* parent, const uint8_t* alive, const int32_t* mask, int rank, int64_t n_regions,
                            void* slot, int64_t capacity, dm_stream_t stream);
int dm_uf_union_slots(int32_t* parent, const void* slots, int64_t n_slots, int64_t slot_bytes, int64_t capacity,
                      int64_t n_regions, dm_stream_t stream);
/* The exchange step of the sharded path as ONE kernel over NVLink peer memory instead of a collective call: the slot of
 * this rank -- a header (header_bytes, its first int64 the entry count) and up to two segments holding count entries of
 * segK_elem_bytes each at segK_offset -- is stored into slot `rank` of every rank's gathered buffer [world x slot_bytes];
 * peer_bases_dev[p] is the device address of rank p's buffer as mapped into this process (CUDA IPC / symmetric memory;
 * the caller's communicator stays opaque to the library).  Only the used part travels: the header, and of each segment
 * min(count, capacity) * segK_elem_bytes rounded up to a multiple of 16 bytes.  The caller runs a barrier over
 * the ranks after it (and alternates two buffers, so that a buffer is rewritten only after every rank has passed the
 * barrier that follows its last read).  All offsets / sizes in bytes, multiples of 16 where they are addresses. */
/* Two-shot all-reduce of an int32 array over NVLink peer memory (the replicated per-region state of the sharded merge
 * loop: visibility masks + point counts (sum), the parent array (min); replaces torch.distributed.all_reduce there).
 * The array sits at offset_bytes of every rank's symmetric buffer (peer_bases_dev[p] = rank p's buffer mapped into this
 * process, as for dm_peer_put_slot); n int32 values, n a multiple of 4, offset a multiple of 16.  Rank g reduces slice g of
 * all ranks' arrays and stores it into every rank's array.  The caller brackets the call with barriers over all ranks
 * (before: every rank's array is complete; after: every slice has landed).  op 0 = sum, 1 = min. */
int dm_peer_allreduce_i32(const void* peer_bases_dev, int64_t world, int64_t rank, int64_t offset_bytes, int64_t n, int op,
                          dm_stream_t stream);

/* host-side glue of the distributed loop as single launches: dm_shard_round_flags fills the eight flag words of a round
 * from the engine's counters (flags[0] = counts[4] edges selected; first round also [3] = counts[2] != 0 overflow, [4] =
 * counts[3] == 1 bad label, [6] = counts[1] raw entries needed; every round [5] |= counts[3] > 1 internal error) and copies them into
 * the frontier slot's header; dm_slots_overflow sets *flag_dev when any gathered slot's entry count exceeds capacity. */
int dm_shard_round_flags(const int64_t* counts, int64_t* flags, int first_round, int64_t* slot_flags, dm_stream_t stream);
int dm_slots_overflow(const void* slots, int64_t n_slots, int64_t slot_bytes, int64_t capacity, int64_t* flag_dev,
                      dm_stream_t stream);
/* *out_dev = max over the gathered slots of the (non-negative) int64 word at word_offset of every slot -- "did any rank
 * select an edge", computed where dm_relabel_gated can read it. */
int dm_slots_word_max(const void* slots, int64_t n_slots, int64_t slot_bytes, int64_t word_offset, int64_t* out_dev,
                      dm_stream_t stream);
int dm_peer_put_slot(const void* slot, const int64_t* peer_bases_dev, int64_t world, int64_t rank, int64_t slot_bytes,
                     int64_t header_bytes, int64_t seg0_offset, int64_t seg0_elem_bytes, int64_t seg1_offset,
                     int64_t seg1_elem_bytes, int64_t capacity, dm_stream_t stream);
int dm_mark_endpoints(const uint64_t* edge_keys, const int64_t* n_edges_dev, int64_t capacity, int64_t n_regions,
                      uint8_t* flags, dm_stream_t stream);
int dm_rows_pack(const uint8_t* flag, const float* rows, int64_t n_regions, int64_t D, int32_t* out_ids,
                 float* out_rows, int64_t capacity, int64_t* n_out_dev, dm_stream_t stream);
int dm_rows_unpack(const int32_t* ids, const float* in_rows, const int64_t* n_dev, int64_t capacity,
                   int64_t n_regions, int64_t D, float* rows, int add, dm_stream_t stream);
/* every slot of an all-gathered exchange buffer in one launch; slot = int64 count | pad to 16 B | int32 ids[cap] |
 * float rows[cap][D]; zero != 0: the listed rows are cleared, else copied (ids distinct over all slots). */
int dm_rows_unpack_slots(const void* slots, int64_t n_slots, int64_t slot_bytes, int64_t slot_capacity,
                         int64_t n_regions, int64_t D, float* rows, int zero, dm_stream_t stream);

/* ----------------------------------------------------------------------------------- *
 * N2  Bounding boxes of the regions, for the bounding-box attributes of the reference's polygon tables (len, width, smooth,
 *     compact, border; MyUtils1.py:79-114 reads them, their formulas are not in the repository: DESIGN.md section 4.5).
 *     bbox int32 [R, 4] = (min column, min row, max column, max row), (INT32_MAX, INT32_MAX, -1, -1) for a region
 *     without pixels; *bad_label != 0 when a label >= n_regions was met.  Not part of the merge step.
 * ----------------------------------------------------------------------------------- */
int dm_region_bbox(const int32_t* labels, int64_t H, int64_t W, int64_t ld, int64_t n_regions, int32_t* bbox,
                   int64_t* bad_label, dm_stream_t stream);

/* ----------------------------------------------------------------------------------- *
 * Polygonize a label raster: the way back from a merged label map to the polygons of the reference's tile.shp (one
 * polygon per segment).  Not part of the merge step.
 *
 * labels int32 [H, ld] (ld >= W); negative labels are nodata and get no polygon; a label >= n_regions sets status 1.
 *  - Rings: every region present gets its boundary as closed rings of pixel-corner vertices, int32 (x, y) with
 *    x in [0, W], y in [0, H].  A boundary side is a pixel side facing another label, nodata or the image border
 *    (the sides dm_rag_build counts in the perimeter).
 *  - Connectivity: regions are 4-connected.  At a saddle vertex (a 2 x 2 block with the same label on one diagonal
 *    only) each region's ring turns so that it stays on its own pixel, so diagonal pixels are never joined.  A ring may
 *    touch itself or another ring of its region at such a vertex.
 *  - Orientation: in pixel coordinates (y down) the region lies on the right of the direction of travel: outer rings
 *    have positive shoelace area 1/2 sum(x_i y_{i+1} - x_{i+1} y_i), holes negative; the sum over a region's rings is
 *    its pixel count.
 *  - Vertices: corners only (the direction changes at every vertex), the ring is not explicitly closed; every ring has
 *    an even number >= 4 of vertices and its edges alternate between horizontal and vertical.
 *  - Canonical form (deterministic): each ring starts at its smallest vertex in (y, x) order, which a ring passes only
 *    once; rings are ordered by (region id, start y, start x), a total order.
 * Outputs (device, caller-owned), with ring_cap = capacity / 4 (a ring has at least 4 boundary sides, and at most one
 * vertex per side):
 *    ring_region  int32 [ring_cap]          ring_offsets int64 [ring_cap + 1] (into vertices)
 *    ring_area    int64 [ring_cap] (signed, pixels)    vertices int32 [capacity, 2]
 *    region_rings int64 [n_regions + 1]: rings of region r are [region_rings[r], region_rings[r + 1])
 *    counts int64 [4]: [0] rings, [1] vertices, [2] boundary sides found (exact, also above capacity),
 *           [3] status: 0 ok, 1 a label >= n_regions, 2 capacity exceeded (outputs invalid; retry with
 *           capacity >= counts[2]).
 * capacity bounds the boundary sides, < 2^31.  (H + 1) (W + 1) <= 2^32.  The workspace grows with H W / 4 bytes, the
 * capacity and n_regions (per-region arrays of the ring sort).  The empty raster writes zero counts (when the outputs
 * are given) and returns 0.
 * ----------------------------------------------------------------------------------- */
size_t dm_polygonize_workspace_bytes(int64_t H, int64_t W, int64_t n_regions, int64_t capacity);
int dm_polygonize(const int32_t* labels, int64_t H, int64_t W, int64_t ld, int64_t n_regions, int64_t capacity,
                  int32_t* ring_region, int64_t* ring_offsets, int64_t* ring_area, int32_t* vertices,
                  int64_t* region_rings, int64_t* counts, void* ws, size_t ws_bytes, dm_stream_t stream);

/* ----------------------------------------------------------------------------------- *
 * R11 Contrastive pair loss forward + backward (Losses.py:34-38):
 *     d = sum_k (a-b)^2 ; L = mean(flag*d + (1-flag)*relu(margin-d)).
 *     loss fp32 [1]; grad_a, grad_b fp32 [B,D] (nullable).  flag int64 as collated.
 * ----------------------------------------------------------------------------------- */
int dm_contrastive_fwd_bwd(const float* a, const float* b, const int64_t* flag, int64_t B, int64_t D,
                           float margin, float* loss, float* grad_a, float* grad_b, dm_stream_t stream);
/* Row gather used by the pair sampler path (R10): out[i] = table[idx[i]]. */
int dm_gather_rows(const float* table, int64_t D, const int64_t* idx, int64_t n, float* out, dm_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DEEPMERGE_B200_H */
