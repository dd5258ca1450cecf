/* Sequential, recursive simplifier of boundary chains: the contract of dm_polygonize_simplified / dm_lines_simplified
 * (include/deepmerge_b200.h), written independently of deepmerge_b200/csrc/simplify_core.cuh.  TEST INFRASTRUCTURE
 * ONLY.
 *
 * Distances are kept as fractions n / d of squared lengths with d = 1 (distance to an end point, n < 2^54) or
 * d = |AB|^2 (distance to the line, n = cross^2 < 2^107), and two fractions are compared by cross-multiplying only when
 * their denominators differ, where one of them is 1.  Nodes of a ring are found from the labels: a vertex where three
 * or four of the unit segments around it separate different values. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

typedef unsigned __int128 u128;

typedef struct {
    const int32_t* v;   /* vertices of the chain, [len, 2] */
    int64_t len, start, W;
    uint64_t T;
    uint8_t* keep;
} Piece;

static int64_t pos(const Piece* p, int64_t k) { return (p->start + k) % p->len; }
static int64_t X(const Piece* p, int64_t k) { return p->v[2 * pos(p, k)]; }
static int64_t Y(const Piece* p, int64_t k) { return p->v[2 * pos(p, k) + 1]; }

static u128 sq128(int64_t a) { u128 u = (u128)(a < 0 ? -a : a); return u * u; }

/* squared distance of position k to the segment of positions lo .. hi, as n / d */
static void dist2(const Piece* p, int64_t lo, int64_t hi, int64_t k, u128* n, u128* d) {
    const int64_t ax = X(p, lo), ay = Y(p, lo), bx = X(p, hi), by = Y(p, hi), px = X(p, k), py = Y(p, k);
    const int64_t abx = bx - ax, aby = by - ay, apx = px - ax, apy = py - ay;
    const int64_t len2 = abx * abx + aby * aby;
    *d = 1;
    if (len2 == 0) { *n = sq128(apx) + sq128(apy); return; }
    const int64_t t = apx * abx + apy * aby;
    if (t <= 0) { *n = sq128(apx) + sq128(apy); return; }
    if (t >= len2) { *n = sq128(px - bx) + sq128(py - by); return; }
    *n = sq128(abx * apy - aby * apx);
    *d = (u128)len2;
}

/* n1 / d1 vs n2 / d2: -1, 0, 1 */
static int cmp_frac(u128 n1, u128 d1, u128 n2, u128 d2) {
    u128 a = n1, b = n2;
    if (d1 != d2) {
        if (d1 == 1) a = n1 * d2;
        else b = n2 * d1;
    }
    return a > b ? 1 : (a < b ? -1 : 0);
}

/* the top position of lo .. hi (hi - lo >= 2); its distance in *n / *d */
static int64_t top(const Piece* p, int64_t lo, int64_t hi, u128* bn, u128* bd) {
    int64_t best = -1, bmid = 0, bidx = 0;
    const int64_t m = hi - lo;
    for (int64_t k = lo + 1; k < hi; ++k) {
        u128 n, d;
        dist2(p, lo, hi, k, &n, &d);
        const int64_t mid = llabs(2 * (k - lo) - m), idx = Y(p, k) * (p->W + 1) + X(p, k);
        int better = best < 0;
        if (!better) {
            const int c = cmp_frac(n, d, *bn, *bd);
            better = c > 0 || (c == 0 && (mid < bmid || (mid == bmid && idx < bidx)));
        }
        if (better) { best = k; *bn = n; *bd = d; bmid = mid; bidx = idx; }
    }
    return best;
}

static void keep_at(const Piece* p, int64_t k) { p->keep[pos(p, k)] = 1; }

static void dp(const Piece* p, int64_t lo, int64_t hi) {
    if (hi - lo < 2) return;
    u128 n, d;
    const int64_t k = top(p, lo, hi, &n, &d);
    /* d(top)^2 > (T / 2^10)^2 */
    if (!(n * ((u128)1 << 20) > (u128)p->T * (u128)p->T * d)) return;
    keep_at(p, k);
    dp(p, lo, k);
    dp(p, k, hi);
}

/* the piece of n segments from position 0 of p */
static void piece(const Piece* p, int64_t n) {
    if (n < 2) return;
    u128 bn, bd;
    const int64_t k = top(p, 0, n, &bn, &bd);
    keep_at(p, k);
    if (X(p, 0) == X(p, n) && Y(p, 0) == Y(p, n)) {
        const int64_t lo[2] = {0, k}, hi[2] = {k, n};
        for (int h = 0; h < 2; ++h) {
            if (hi[h] - lo[h] < 2) continue;
            const int64_t kk = top(p, lo[h], hi[h], &bn, &bd);
            keep_at(p, kk);
            dp(p, lo[h], kk);
            dp(p, kk, hi[h]);
        }
    } else {
        dp(p, 0, k);
        dp(p, k, n);
    }
}

/* Keep flags of n_chains chains (vertices v, offsets off).  cyclic: rings, whose nodes are flagged in node; else lines
 * (open lists, a closed line repeats its start).  Returns the number of kept vertices, -1 on a bad tolerance. */
int64_t dmo_simplify(const int32_t* v, const int64_t* off, int64_t n_chains, const uint8_t* node, int cyclic, int64_t H,
                     int64_t W, double t, uint8_t* keep) {
    if (!isfinite(t) || t < 0) return -1;
    const double lim = (double)(H + W);
    const uint64_t T = (uint64_t)floor((t < lim ? t : lim) * 1024.0 + 0.5);
    int64_t kept = 0;
    for (int64_t c = 0; c < n_chains; ++c) {
        const int64_t s0 = off[c], len = off[c + 1] - s0;
        const int32_t* cv = v + 2 * s0;
        uint8_t* ck = keep + s0;
        int has_node = 0;
        if (cyclic)
            for (int64_t j = 0; j < len; ++j) has_node |= node[s0 + j] != 0;
        int64_t first = -1, prev = -1;
        for (int64_t j = 0; j < len; ++j) {
            const int64_t x = cv[2 * j], y = cv[2 * j + 1];
            int a = x == 0 || y == 0 || x == W || y == H;
            if (cyclic) a |= node[s0 + j] || (!has_node && j == 0);
            else a |= j == 0 || j == len - 1;
            ck[j] = (uint8_t)a;
            if (!a) continue;
            if (prev >= 0) {
                Piece p = {cv, len, prev, W, T, ck};
                piece(&p, j - prev);
            } else {
                first = j;
            }
            prev = j;
        }
        if (cyclic) {
            Piece p = {cv, len, prev, W, T, ck};
            piece(&p, first + len - prev);
        }
    }
    for (int64_t i = 0; i < off[n_chains]; ++i) kept += keep[i];
    return kept;
}

static int32_t value(const int32_t* L, int64_t H, int64_t W, int64_t x, int64_t y) {
    if (x < 0 || y < 0 || x >= W || y >= H) return -1;
    return L[y * W + x] < 0 ? -1 : L[y * W + x];
}

/* vertex (x, y) has three or four boundary segments around it */
static int is_node(const int32_t* L, int64_t H, int64_t W, int64_t x, int64_t y) {
    const int32_t nw = value(L, H, W, x - 1, y - 1), ne = value(L, H, W, x, y - 1);
    const int32_t sw = value(L, H, W, x - 1, y), se = value(L, H, W, x, y);
    return (nw != ne) + (ne != se) + (se != sw) + (sw != nw) >= 3;
}

/* The rings of dm_polygonize (corners only, labels L [H, W]) with their nodes: every corner, and every vertex between
 * two corners that is a node, found by walking each straight edge.  Writes v_out [n, 2], off_out [n_rings + 1] and
 * node_out [n]; returns n. */
int64_t dmo_ring_nodes(const int32_t* L, int64_t H, int64_t W, const int32_t* v, const int64_t* off, int64_t n_rings,
                       int32_t* v_out, int64_t* off_out, uint8_t* node_out) {
    int64_t n = 0;
    for (int64_t r = 0; r < n_rings; ++r) {
        off_out[r] = n;
        const int64_t s0 = off[r], len = off[r + 1] - s0;
        for (int64_t j = 0; j < len; ++j) {
            const int64_t x0 = v[2 * (s0 + j)], y0 = v[2 * (s0 + j) + 1];
            const int64_t x1 = v[2 * (s0 + (j + 1) % len)], y1 = v[2 * (s0 + (j + 1) % len) + 1];
            const int64_t dx = x1 > x0 ? 1 : (x1 < x0 ? -1 : 0), dy = y1 > y0 ? 1 : (y1 < y0 ? -1 : 0);
            for (int64_t x = x0, y = y0; x != x1 || y != y1; x += dx, y += dy) {
                const int nd = is_node(L, H, W, x, y);
                if (!nd && (x != x0 || y != y0)) continue;
                v_out[2 * n] = (int32_t)x;
                v_out[2 * n + 1] = (int32_t)y;
                node_out[n++] = (uint8_t)nd;
            }
        }
    }
    off_out[n_rings] = n;
    return n;
}

/* The top position of the interval of vertices v [n + 1, 2] (n >= 2) and whether it lies farther than T / 2^10 px. */
int64_t dmo_top(const int32_t* v, int64_t n, int64_t W, uint64_t T, int* exceeds) {
    const Piece p = {v, n + 1, 0, W, T, NULL};
    u128 bn, bd;
    const int64_t k = top(&p, 0, n, &bn, &bd);
    *exceeds = bn * ((u128)1 << 20) > (u128)T * (u128)T * bd;
    return k;
}

uint64_t dmo_quantize(double t, int64_t H, int64_t W) {
    const double lim = (double)(H + W);
    return (uint64_t)floor((t < lim ? t : lim) * 1024.0 + 0.5);
}
