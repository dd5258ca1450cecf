/* polygon_oracle.c -- a plain sequential restatement of dm_polygonize (include/deepmerge_b200.h), written from its
 * contract and sharing no code with deepmerge_b200/csrc/polygon.cu.  TEST INFRASTRUCTURE ONLY: compiled with gcc by
 * tests/polygon_oracle.py into a temporary directory; nothing in deepmerge_b200 links it. */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

/* ---- polygonize: label raster -> canonical rings (include/deepmerge_b200.h, dm_polygonize) ----
 * A plain sequential tracer.  Boundary sides are walked in raster order (pixel, then side top / right / bottom / left);
 * an untraced one starts a ring, which follows the successor rule until it closes.  Side d of a pixel is travelled in
 * direction d (0 east, 1 south, 2 west, 3 north; y down) with the pixel on its right.  At the head vertex the 2 x 2
 * block decides: the pixel behind on the right carries the region; when the pixel ahead on the right does not, turn
 * right (stay on the pixel: diagonal pixels are never joined); else when the pixel ahead on the left does not, go
 * straight on; else turn left. */
static int32_t plab(const int32_t* L, int64_t H, int64_t W, int64_t x, int64_t y) {
    return (x < 0 || y < 0 || x >= W || y >= H) ? -1 : L[y * W + x];
}

static int pside(const int32_t* L, int64_t H, int64_t W, int64_t x, int64_t y, int d) {
    static const int nx[4] = {0, 1, 0, -1}, ny[4] = {-1, 0, 1, 0};   /* neighbour across side d */
    const int32_t a = L[y * W + x];
    return a >= 0 && plab(L, H, W, x + nx[d], y + ny[d]) != a;
}

/* Successor of side d of pixel (x, y): out = (pixel x, pixel y, side, head vertex is a corner).  Returns 0 when
 * (x, y, d) is not a boundary side. */
int dmo_poly_successor(const int32_t* L, int64_t H, int64_t W, int64_t x, int64_t y, int d, int64_t* out) {
    /* head vertex of side d and the quadrants around it (0 NW, 1 NE, 2 SW, 3 SE) that lie behind-right, ahead-right
     * and ahead-left of the direction of travel */
    static const int hx[4] = {1, 1, 0, 0}, hy[4] = {0, 1, 1, 0};
    static const int ahead_r[4] = {3, 2, 0, 1}, ahead_l[4] = {1, 3, 2, 0};
    if (!pside(L, H, W, x, y, d)) return 0;
    const int64_t vx = x + hx[d], vy = y + hy[d];
    const int64_t qx[4] = {vx - 1, vx, vx - 1, vx}, qy[4] = {vy - 1, vy - 1, vy, vy};
    const int32_t a = L[y * W + x];
    int q, nd;
    if (plab(L, H, W, qx[ahead_r[d]], qy[ahead_r[d]]) != a) {
        out[0] = x; out[1] = y; nd = (d + 1) & 3;
    } else if (plab(L, H, W, qx[ahead_l[d]], qy[ahead_l[d]]) != a) {
        q = ahead_r[d]; out[0] = qx[q]; out[1] = qy[q]; nd = d;
    } else {
        q = ahead_l[d]; out[0] = qx[q]; out[1] = qy[q]; nd = (d + 3) & 3;
    }
    out[2] = nd;
    out[3] = nd != d;
    return 1;
}

typedef struct {
    int64_t region, y0, x0, off, n, area;
} PRing;

static int cmp_ring(const void* a, const void* b) {
    const PRing *p = (const PRing*)a, *q = (const PRing*)b;
    if (p->region != q->region) return p->region < q->region ? -1 : 1;
    if (p->y0 != q->y0) return p->y0 < q->y0 ? -1 : 1;
    return (p->x0 > q->x0) - (p->x0 < q->x0);
}

/* labels [H, W] (pitch W).  With S the number of boundary sides: ring_region / ring_offsets (+1) / ring_area hold
 * S / 4 + 1 entries, verts S pairs,
 * region_rings R + 1.  counts[0..3] as dm_polygonize (counts[3] = 1 and nothing else written when a label >= R).
 * Returns 0, or -1 when out of memory. */
int dmo_polygonize(const int32_t* L, int64_t H, int64_t W, int64_t R, int32_t* ring_region, int64_t* ring_offsets,
                   int64_t* ring_area, int32_t* verts, int64_t* region_rings, int64_t* counts) {
    static const int hx[4] = {1, 1, 0, 0}, hy[4] = {0, 1, 1, 0};
    memset(counts, 0, 4 * sizeof(int64_t));
    memset(region_rings, 0, (size_t)(R + 1) * sizeof(int64_t));
    ring_offsets[0] = 0;
    for (int64_t p = 0; p < H * W; ++p)
        if (L[p] >= R) { counts[3] = 1; return 0; }
    int64_t total = 0;                                               /* boundary sides: bounds vertices and rings */
    for (int64_t y = 0; y < H; ++y)
        for (int64_t x = 0; x < W; ++x)
            for (int d = 0; d < 4; ++d) total += pside(L, H, W, x, y, d);
    uint8_t* seen = (uint8_t*)calloc((size_t)(H * W + 1), 1);
    int32_t* tmp = (int32_t*)malloc((size_t)(2 * total + 8) * sizeof(int32_t));
    int32_t* raw = (int32_t*)malloc((size_t)(2 * total + 8) * sizeof(int32_t));
    PRing* rings = (PRing*)malloc((size_t)(total / 4 + 1) * sizeof(PRing));
    if (!seen || !tmp || !raw || !rings) { free(seen); free(tmp); free(raw); free(rings); return -1; }
    int64_t n_rings = 0, n_verts = 0, n_sides = 0;
    for (int64_t y = 0; y < H; ++y)
        for (int64_t x = 0; x < W; ++x)
            for (int d = 0; d < 4; ++d) {
                if (!pside(L, H, W, x, y, d)) continue;
                ++n_sides;
                if (seen[y * W + x] & (1 << d)) continue;
                int64_t cx = x, cy = y, k = 0, nxt[4];
                int cd = d;
                do {                                                 /* trace, collecting the corners */
                    seen[cy * W + cx] |= (uint8_t)(1 << cd);
                    dmo_poly_successor(L, H, W, cx, cy, cd, nxt);
                    if (nxt[3]) {
                        tmp[2 * k] = (int32_t)(cx + hx[cd]);
                        tmp[2 * k + 1] = (int32_t)(cy + hy[cd]);
                        ++k;
                    }
                    cx = nxt[0]; cy = nxt[1]; cd = (int)nxt[2];
                } while (!(cx == x && cy == y && cd == d));
                int64_t m = 0;                                       /* rotate to the smallest (y, x) vertex */
                for (int64_t i = 1; i < k; ++i)
                    if (tmp[2 * i + 1] < tmp[2 * m + 1] || (tmp[2 * i + 1] == tmp[2 * m + 1] && tmp[2 * i] < tmp[2 * m])) m = i;
                int64_t a2 = 0;
                for (int64_t i = 0; i < k; ++i) {
                    const int64_t j = (m + i) % k, j1 = (m + i + 1) % k;
                    raw[2 * (n_verts + i)] = tmp[2 * j];
                    raw[2 * (n_verts + i) + 1] = tmp[2 * j + 1];
                    a2 += (int64_t)tmp[2 * j] * tmp[2 * j1 + 1] - (int64_t)tmp[2 * j1] * tmp[2 * j + 1];
                }
                PRing* r = &rings[n_rings++];
                r->region = L[y * W + x]; r->y0 = tmp[2 * m + 1]; r->x0 = tmp[2 * m];
                r->off = n_verts; r->n = k; r->area = a2 / 2;
                n_verts += k;
            }
    qsort(rings, (size_t)n_rings, sizeof(PRing), cmp_ring);
    int64_t o = 0;
    for (int64_t i = 0; i < n_rings; ++i) {
        ring_region[i] = (int32_t)rings[i].region;
        ring_area[i] = rings[i].area;
        ring_offsets[i] = o;
        memcpy(verts + 2 * o, raw + 2 * rings[i].off, (size_t)(2 * rings[i].n) * sizeof(int32_t));
        o += rings[i].n;
        region_rings[rings[i].region + 1] += 1;
    }
    ring_offsets[n_rings] = o;
    for (int64_t r = 0; r < R; ++r) region_rings[r + 1] += region_rings[r];
    counts[0] = n_rings; counts[1] = n_verts; counts[2] = n_sides;
    free(seen); free(tmp); free(raw); free(rings);
    return 0;
}
