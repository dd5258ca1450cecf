// Per-vertex arithmetic of the boundary-line tracer (lines.cu), host/device.
//
// Every pixel position has a value: its label when >= 0, else -1; positions outside the image are -1.  A boundary
// segment is a unit side between two 4-adjacent positions whose values differ.  Pixel (x, y) owns the segments on its
// top and left side, and, in the last column / row, the one on its right / bottom side (mask bits TOP, LEFT, RIGHT,
// BOTTOM).  A segment is travelled with the larger value on its right (pixel coordinates, y down; directions 0 E, 1 S,
// 2 W, 3 N as in polygon_core.cuh).  The degree of a vertex is the number of segments that meet there; a vertex of
// degree >= 3 is a node, where lines end.  At a vertex of degree 2 a line goes on along the other segment, whose
// orientation carries on: the same two values stay on the same sides.
//
// The same source is compiled by g++ in the CPU test suite (tests/lines_core_host.cpp) and checked against the
// sequential tracer of tests/lines_oracle.c.
#pragma once
#include "polygon_core.cuh"

namespace dm {
namespace linecore {
using polycore::label_at;
using polycore::step_x;
using polycore::step_y;

enum { TOP = 0, LEFT = 1, RIGHT = 2, BOTTOM = 3 };

DM_PHD int32_t value_at(const int32_t* L, int64_t H, int64_t W, int64_t ld, int64_t x, int64_t y) {
    const int32_t v = label_at(L, H, W, ld, x, y);
    return v < 0 ? -1 : v;
}

// 4-bit mask of the segments pixel (x, y) owns
DM_PHD unsigned owned_mask(const int32_t* L, int64_t H, int64_t W, int64_t ld, int64_t x, int64_t y) {
    const int32_t a = value_at(L, H, W, ld, x, y);
    unsigned m = 0;
    if (value_at(L, H, W, ld, x, y - 1) != a) m |= 1u << TOP;
    if (value_at(L, H, W, ld, x - 1, y) != a) m |= 1u << LEFT;
    if (x == W - 1 && a >= 0) m |= 1u << RIGHT;
    if (y == H - 1 && a >= 0) m |= 1u << BOTTOM;
    return m;
}

// Bit d set: a segment leaves vertex (vx, vy) in direction d.  Quadrants: NW (vx-1, vy-1), NE (vx, vy-1),
// SW (vx-1, vy), SE (vx, vy).
DM_PHD unsigned arms(const int32_t* L, int64_t H, int64_t W, int64_t ld, int64_t vx, int64_t vy) {
    const int32_t nw = value_at(L, H, W, ld, vx - 1, vy - 1), ne = value_at(L, H, W, ld, vx, vy - 1);
    const int32_t sw = value_at(L, H, W, ld, vx - 1, vy), se = value_at(L, H, W, ld, vx, vy);
    return (ne != se ? 1u : 0u) | (sw != se ? 2u : 0u) | (nw != sw ? 4u : 0u) | (nw != ne ? 8u : 0u);
}

DM_PHD bool node_arms(unsigned a) { return ((a & 1u) + ((a >> 1) & 1u) + ((a >> 2) & 1u) + ((a >> 3) & 1u)) >= 3; }

// A directed segment: tail vertex and direction.
struct Seg {
    int64_t x, y;
    int d;
};

// The values on the right and the left of a directed segment.
DM_PHD int32_t right_value(const int32_t* L, int64_t H, int64_t W, int64_t ld, Seg s) {
    const int64_t px = s.x - (s.d == 1 || s.d == 2 ? 1 : 0), py = s.y - (s.d == 2 || s.d == 3 ? 1 : 0);
    return value_at(L, H, W, ld, px, py);
}
DM_PHD int32_t left_value(const int32_t* L, int64_t H, int64_t W, int64_t ld, Seg s) {
    const int64_t px = s.x - (s.d == 2 || s.d == 3 ? 1 : 0), py = s.y - (s.d == 0 || s.d == 3 ? 1 : 0);
    return value_at(L, H, W, ld, px, py);
}

// Orientation of segment b of pixel (x, y): the larger value on the right.
DM_PHD Seg orient(const int32_t* L, int64_t H, int64_t W, int64_t ld, int64_t x, int64_t y, int b) {
    const int32_t a = value_at(L, H, W, ld, x, y);
    Seg s;
    if (b == TOP) {              // east has the pixel below on its right
        const bool east = a > value_at(L, H, W, ld, x, y - 1);
        s.x = east ? x : x + 1; s.y = y; s.d = east ? 0 : 2;
    } else if (b == LEFT) {      // south has the pixel to the left on its right
        const bool south = value_at(L, H, W, ld, x - 1, y) > a;
        s.x = x; s.y = south ? y : y + 1; s.d = south ? 1 : 3;
    } else if (b == RIGHT) {     // the image border on the right of the pixel: south
        s.x = x + 1; s.y = y; s.d = 1;
    } else {                     // the border below: west
        s.x = x + 1; s.y = y + 1; s.d = 2;
    }
    return s;
}

// Owner (pixel, bit) of the segment that leaves vertex (vx, vy) in direction d.
struct Owner {
    int64_t x, y;
    int b;
};
DM_PHD Owner owner_of(int64_t H, int64_t W, int64_t vx, int64_t vy, int d) {
    Owner o;
    if (d == 0 || d == 2) {      // horizontal: the top side of the pixel below, or the bottom side in the last row
        o.x = d == 0 ? vx : vx - 1;
        o.y = vy < H ? vy : H - 1;
        o.b = vy < H ? TOP : BOTTOM;
    } else {                     // vertical: the left side of the pixel to the right, or the right side in the last column
        o.x = vx < W ? vx : W - 1;
        o.y = d == 1 ? vy : vy - 1;
        o.b = vx < W ? LEFT : RIGHT;
    }
    return o;
}

// What follows a segment that arrives at vertex (hx, hy) travelling in direction d: nothing at a node, else the other
// segment of the vertex, leaving it in direction `d` of the result.
struct Next {
    bool node;
    int d;
};
DM_PHD Next next_at(const int32_t* L, int64_t H, int64_t W, int64_t ld, int64_t hx, int64_t hy, int d) {
    const unsigned a = arms(L, H, W, ld, hx, hy);
    Next n;
    n.node = node_arms(a);
    const unsigned o = a & ~(1u << ((d + 2) & 3));
    n.d = o & 1u ? 0 : (o & 2u ? 1 : (o & 4u ? 2 : 3));
    return n;
}

}  // namespace linecore
}  // namespace dm
