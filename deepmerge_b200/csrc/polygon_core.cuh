// Per-side arithmetic of the polygonizer (polygon.cu), host/device.
//
// A boundary side is a side of a pixel with a valid label that faces another label, nodata or the image border.  Side s
// of pixel (x, y) is travelled in direction s with the pixel on its right (pixel coordinates, y down):
//   s = 0 top    (x, y)     -> (x+1, y)     east
//   s = 1 right  (x+1, y)   -> (x+1, y+1)   south
//   s = 2 bottom (x+1, y+1) -> (x, y+1)     west
//   s = 3 left   (x, y+1)   -> (x, y)       north
// At the head vertex the ring continues on the first of: a right turn (same pixel, side s+1) when the pixel ahead on the
// right does not carry the label; straight on (that pixel, side s) when the pixel ahead on the left does not; otherwise a
// left turn (the pixel ahead on the left, side s+3).  Taking the right turn first keeps a ring on its own pixel at a
// saddle vertex, so diagonal pixels are never joined (4-connectivity).  The head vertex is a corner unless the ring
// goes straight on.
//
// The same source is compiled by g++ in the CPU test suite (tests/polygon_core_host.cpp) and checked against the
// sequential tracer of tests/polygon_oracle.c.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define DM_PHD __host__ __device__ __forceinline__
#else
#define DM_PHD inline
#endif

namespace dm {
namespace polycore {

DM_PHD int step_x(int d) { return d == 0 ? 1 : (d == 2 ? -1 : 0); }
DM_PHD int step_y(int d) { return d == 1 ? 1 : (d == 3 ? -1 : 0); }

// label at (x, y), -1 outside the image (the border counts like nodata: it is never traced)
DM_PHD int32_t label_at(const int32_t* L, int64_t H, int64_t W, int64_t ld, int64_t x, int64_t y) {
    return (x < 0 || y < 0 || x >= W || y >= H) ? -1 : L[y * ld + x];
}

// 4-bit mask of the boundary sides of pixel (x, y): bit s set when side s is a boundary side
DM_PHD unsigned side_mask(const int32_t* L, int64_t H, int64_t W, int64_t ld, int64_t x, int64_t y) {
    const int32_t a = L[y * ld + x];
    if (a < 0) return 0u;
    unsigned m = 0;
    for (int s = 0; s < 4; ++s) {   // the neighbour across side s lies in direction s + 3 (left of the travel)
        const int n = (s + 3) & 3;
        if (label_at(L, H, W, ld, x + step_x(n), y + step_y(n)) != a) m |= 1u << s;
    }
    return m;
}

// Successor of side s of a pixel labelled a, given the labels of the pixel ahead on the right (rf) and ahead on the
// left (lf).  Returns the turn: 1 = right (same pixel), 0 = straight (the rf pixel), 3 = left (the lf pixel); the
// successor side is (s + turn) & 3.
DM_PHD int turn_of(int32_t a, int32_t rf, int32_t lf) {
    if (rf != a) return 1;
    if (lf != a) return 0;
    return 3;
}

struct Succ {
    int64_t x, y;   // pixel of the successor side
    int s;          // its side
    bool corner;    // the head vertex of the current side is a corner
};

DM_PHD Succ successor(const int32_t* L, int64_t H, int64_t W, int64_t ld, int64_t x, int64_t y, int s) {
    const int32_t a = L[y * ld + x];
    const int64_t rx = x + step_x(s), ry = y + step_y(s);                                   // ahead on the right
    const int l = (s + 3) & 3;
    const int64_t lx = rx + step_x(l), ly = ry + step_y(l);                                 // ahead on the left
    const int t = turn_of(a, label_at(L, H, W, ld, rx, ry), label_at(L, H, W, ld, lx, ly));
    Succ r;
    r.s = (s + t) & 3;
    r.corner = t != 0;
    r.x = t == 1 ? x : (t == 0 ? rx : lx);
    r.y = t == 1 ? y : (t == 0 ? ry : ly);
    return r;
}

// head vertex of side s of pixel (x, y)
DM_PHD int64_t head_x(int64_t x, int s) { return x + (s == 0 || s == 1 ? 1 : 0); }
DM_PHD int64_t head_y(int64_t y, int s) { return y + (s == 1 || s == 2 ? 1 : 0); }

}  // namespace polycore
}  // namespace dm
