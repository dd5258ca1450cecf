/* lines_oracle.c -- a plain sequential restatement of dm_lines (include/deepmerge_b200.h), written from its contract
 * and sharing no code with deepmerge_b200/csrc/lines.cu.  TEST INFRASTRUCTURE ONLY: compiled with gcc by
 * tests/lines_oracle.py into a temporary directory; nothing in deepmerge_b200 links it.
 *
 * Segments are numbered: horizontal ones (on vertex row y, between columns x and x + 1) first, h = y W + x for
 * y in [0, H], then vertical ones (on vertex column x, between rows y and y + 1), (H + 1) W + y (W + 1) + x.  The
 * degree of every vertex is counted from the segments present; a line is traced from every segment whose tail is a node
 * until a segment ends at a node, and every segment left over lies on a cycle, which is rotated to start at its
 * smallest vertex. */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static int32_t lval(const int32_t* L, int64_t H, int64_t W, int64_t x, int64_t y) {
    if (x < 0 || y < 0 || x >= W || y >= H) return -1;
    return L[y * W + x] < 0 ? -1 : L[y * W + x];
}

typedef struct {
    int64_t H, W, nh, n;
    const int32_t* L;
    uint8_t* present;
    uint8_t* deg;          /* [(H + 1) (W + 1)] */
} Grid;

/* tail vertex and direction (0 E, 1 S, 2 W, 3 N) of segment s, the larger value on the right */
static void seg_dir(const Grid* g, int64_t s, int64_t* tx, int64_t* ty, int* d) {
    if (s < g->nh) {
        const int64_t y = s / g->W, x = s % g->W;
        const int32_t up = lval(g->L, g->H, g->W, x, y - 1), dn = lval(g->L, g->H, g->W, x, y);
        if (dn > up) { *tx = x; *ty = y; *d = 0; }      /* east: the pixel below is on the right */
        else { *tx = x + 1; *ty = y; *d = 2; }
    } else {
        const int64_t k = s - g->nh, y = k / (g->W + 1), x = k % (g->W + 1);
        const int32_t lf = lval(g->L, g->H, g->W, x - 1, y), rt = lval(g->L, g->H, g->W, x, y);
        if (lf > rt) { *tx = x; *ty = y; *d = 1; }      /* south: the pixel to the left is on the right */
        else { *tx = x; *ty = y + 1; *d = 3; }
    }
}

static void seg_head(const Grid* g, int64_t s, int64_t* hx, int64_t* hy, int* d) {
    int64_t tx, ty;
    seg_dir(g, s, &tx, &ty, d);
    *hx = tx + (*d == 0) - (*d == 2);
    *hy = ty + (*d == 1) - (*d == 3);
}

/* the up to four segments at vertex (x, y), -1 where absent: east, south, west, north */
static void around(const Grid* g, int64_t x, int64_t y, int64_t out[4]) {
    const int64_t W = g->W, H = g->H;
    out[0] = (x < W) ? y * W + x : -1;
    out[1] = (y < H) ? g->nh + y * (W + 1) + x : -1;
    out[2] = (x > 0) ? y * W + x - 1 : -1;
    out[3] = (y > 0) ? g->nh + (y - 1) * (W + 1) + x : -1;
    for (int i = 0; i < 4; ++i)
        if (out[i] >= 0 && !g->present[out[i]]) out[i] = -1;
}

/* successor of s at its head: -1 at a node */
static int64_t succ(const Grid* g, int64_t s) {
    int64_t hx, hy, a[4];
    int d;
    seg_head(g, s, &hx, &hy, &d);
    if (g->deg[hy * (g->W + 1) + hx] != 2) return -1;
    around(g, hx, hy, a);
    for (int i = 0; i < 4; ++i)
        if (a[i] >= 0 && a[i] != s) return a[i];
    return -1;
}

static int grid_init(Grid* g, const int32_t* L, int64_t H, int64_t W) {
    g->L = L; g->H = H; g->W = W;
    g->nh = (H + 1) * W;
    g->n = g->nh + H * (W + 1);
    g->present = (uint8_t*)calloc((size_t)g->n + 1, 1);
    g->deg = (uint8_t*)calloc((size_t)((H + 1) * (W + 1)), 1);
    if (!g->present || !g->deg) return -1;
    for (int64_t y = 0; y <= H; ++y)
        for (int64_t x = 0; x < W; ++x)
            if (lval(L, H, W, x, y - 1) != lval(L, H, W, x, y)) {
                g->present[y * W + x] = 1;
                g->deg[y * (W + 1) + x]++;
                g->deg[y * (W + 1) + x + 1]++;
            }
    for (int64_t y = 0; y < H; ++y)
        for (int64_t x = 0; x <= W; ++x)
            if (lval(L, H, W, x - 1, y) != lval(L, H, W, x, y)) {
                g->present[g->nh + y * (W + 1) + x] = 1;
                g->deg[y * (W + 1) + x]++;
                g->deg[(y + 1) * (W + 1) + x]++;
            }
    return 0;
}

static void grid_free(Grid* g) {
    free(g->present);
    free(g->deg);
}

/* Every segment: tail x, tail y, direction, head is a node, tail is a node, successor's tail x, y, direction (-1s at a
 * node), head is a vertex of the line (corner or end).  out [n_segments][9]; returns the number of segments (rows in
 * the oracle's numbering), or -1 when out of memory. */
int64_t dmo_line_segments(const int32_t* L, int64_t H, int64_t W, int64_t* out) {
    Grid g;
    if (grid_init(&g, L, H, W) != 0) { grid_free(&g); return -1; }
    int64_t k = 0;
    for (int64_t s = 0; s < g.n; ++s) {
        if (!g.present[s]) continue;
        int64_t tx, ty, hx, hy, *o = out + 9 * k++;
        int d;
        seg_dir(&g, s, &tx, &ty, &d);
        seg_head(&g, s, &hx, &hy, &d);
        const int64_t q = succ(&g, s);
        o[0] = tx; o[1] = ty; o[2] = d;
        o[3] = g.deg[hy * (W + 1) + hx] >= 3;
        o[4] = g.deg[ty * (W + 1) + tx] >= 3;
        if (q >= 0) {
            int qd;
            seg_dir(&g, q, &o[5], &o[6], &qd);
            o[7] = qd;
            o[8] = qd != d;
        } else {
            o[5] = o[6] = o[7] = -1;
            o[8] = 1;
        }
    }
    grid_free(&g);
    return k;
}

typedef struct {
    int64_t y0, x0, d0, left, right, len, off, nv;
} OLine;

static int cmp_line(const void* a, const void* b) {
    const OLine *p = (const OLine*)a, *q = (const OLine*)b;
    if (p->y0 != q->y0) return p->y0 < q->y0 ? -1 : 1;
    if (p->x0 != q->x0) return p->x0 < q->x0 ? -1 : 1;
    return (p->d0 > q->d0) - (p->d0 < q->d0);
}

/* Append the line whose segments are chain[0 .. m) to the output lists. */
static void add_line(const Grid* g, const int64_t* chain, int64_t m, OLine* lines, int64_t* n_lines, int32_t* raw,
                     int64_t* n_raw) {
    OLine* l = &lines[(*n_lines)++];
    int64_t tx, ty, hx, hy;
    int d, nd;
    seg_dir(g, chain[0], &tx, &ty, &d);
    l->x0 = tx; l->y0 = ty; l->d0 = d; l->len = m; l->off = *n_raw;
    /* values: the right of the first segment's direction */
    {
        static const int rx[4] = {0, -1, -1, 0}, ry[4] = {0, 0, -1, -1}, lx[4] = {0, 0, -1, -1}, ly[4] = {-1, 0, 0, -1};
        l->right = lval(g->L, g->H, g->W, tx + rx[d], ty + ry[d]);
        l->left = lval(g->L, g->H, g->W, tx + lx[d], ty + ly[d]);
    }
    raw[2 * *n_raw] = (int32_t)tx; raw[2 * *n_raw + 1] = (int32_t)ty; ++*n_raw;
    for (int64_t i = 0; i < m; ++i) {
        seg_head(g, chain[i], &hx, &hy, &d);
        int emit = i == m - 1;
        if (!emit) {
            seg_dir(g, chain[i + 1], &tx, &ty, &nd);
            emit = nd != d;
        }
        if (emit) { raw[2 * *n_raw] = (int32_t)hx; raw[2 * *n_raw + 1] = (int32_t)hy; ++*n_raw; }
    }
    l->nv = *n_raw - l->off;
}

/* labels [H, W] (pitch W).  With S the number of boundary segments: left / right / length hold S entries, offsets
 * S + 1, verts 2 S pairs.  counts[0..3] as dm_lines (counts[3] = 1 and nothing else written when a label >= R).
 * Returns 0, or -1 when out of memory. */
int dmo_lines(const int32_t* L, int64_t H, int64_t W, int64_t R, int32_t* left, int32_t* right, int64_t* length,
              int64_t* offsets, int32_t* verts, int64_t* counts) {
    memset(counts, 0, 4 * sizeof(int64_t));
    offsets[0] = 0;
    for (int64_t p = 0; p < H * W; ++p)
        if (L[p] >= R) { counts[3] = 1; return 0; }
    if (H == 0 || W == 0) return 0;
    Grid g;
    if (grid_init(&g, L, H, W) != 0) { grid_free(&g); return -1; }
    int64_t S = 0;
    for (int64_t s = 0; s < g.n; ++s) S += g.present[s];
    uint8_t* used = (uint8_t*)calloc((size_t)g.n + 1, 1);
    int64_t* chain = (int64_t*)malloc((size_t)(S + 1) * sizeof(int64_t));
    OLine* lines = (OLine*)malloc((size_t)(S + 1) * sizeof(OLine));
    int32_t* raw = (int32_t*)malloc((size_t)(4 * S + 4) * sizeof(int32_t));
    if (!used || !chain || !lines || !raw) {
        free(used); free(chain); free(lines); free(raw); grid_free(&g);
        return -1;
    }
    int64_t n_lines = 0, n_raw = 0;
    for (int64_t s = 0; s < g.n; ++s) {                      /* open lines: from every segment leaving a node */
        int64_t tx, ty;
        int d;
        if (!g.present[s]) continue;
        seg_dir(&g, s, &tx, &ty, &d);
        if (g.deg[ty * (W + 1) + tx] < 3) continue;
        int64_t m = 0;
        for (int64_t c = s; c >= 0; c = succ(&g, c)) { chain[m++] = c; used[c] = 1; }
        add_line(&g, chain, m, lines, &n_lines, raw, &n_raw);
    }
    for (int64_t s = 0; s < g.n; ++s) {                      /* cycles */
        if (!g.present[s] || used[s]) continue;
        int64_t m = 0, best = 0, bk = -1;
        int64_t c = s;
        do { chain[m++] = c; used[c] = 1; c = succ(&g, c); } while (c != s);
        for (int64_t i = 0; i < m; ++i) {                    /* rotate to the segment leaving the smallest vertex */
            int64_t tx, ty;
            int d;
            seg_dir(&g, chain[i], &tx, &ty, &d);
            const int64_t k = ty * (W + 1) + tx;
            if (bk < 0 || k < bk) { bk = k; best = i; }
        }
        int64_t* rot = (int64_t*)malloc((size_t)m * sizeof(int64_t));
        if (!rot) { free(used); free(chain); free(lines); free(raw); grid_free(&g); return -1; }
        for (int64_t i = 0; i < m; ++i) rot[i] = chain[(best + i) % m];
        add_line(&g, rot, m, lines, &n_lines, raw, &n_raw);
        free(rot);
    }
    qsort(lines, (size_t)n_lines, sizeof(OLine), cmp_line);
    int64_t o = 0;
    for (int64_t i = 0; i < n_lines; ++i) {
        left[i] = (int32_t)lines[i].left;
        right[i] = (int32_t)lines[i].right;
        length[i] = lines[i].len;
        offsets[i] = o;
        memcpy(verts + 2 * o, raw + 2 * lines[i].off, (size_t)(2 * lines[i].nv) * sizeof(int32_t));
        o += lines[i].nv;
    }
    offsets[n_lines] = o;
    counts[0] = n_lines; counts[1] = o; counts[2] = S;
    free(used); free(chain); free(lines); free(raw); grid_free(&g);
    return 0;
}
