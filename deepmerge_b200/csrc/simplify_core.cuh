// Exact arithmetic of the chain simplifier (simplify.cuh), host/device: the tolerance rounding, the distance of a vertex
// to the segment of its interval and the order that picks an interval's top vertex (dm_polygonize_simplified and
// dm_lines_simplified in include/deepmerge_b200.h).
//
// Vertices are integer pixel corners with 0 <= x, y < 2^26, so every coordinate difference fits 27 bits.  For an interval
// A..B (v = B - A) and a vertex P (w = P - A) the squared distance to the segment AB is num / den with
//   A = B:                   num = |w|^2,            den = 1
//   projection before A:     num = |w|^2 |v|^2,      den = |v|^2
//   projection after B:      num = |P - B|^2 |v|^2,  den = |v|^2
//   otherwise:               num = cross(v, w)^2,    den = |v|^2
// so that all vertices of one interval share den and compare by num alone.  num < 2^107.  The tolerance is t_q = T / 2^10
// px (T an integer <= (W + H) 2^10 < 2^37), and d > t_q is num 2^20 > T^2 den: both sides stay below 2^128.
//
// The same source is compiled by g++ in the CPU test suite (tests/simplify_core_host.cpp) and checked against the
// sequential simplifier of tests/simplify_oracle.c.
#pragma once
#include <stdint.h>

#include "polygon_core.cuh"

namespace dm {
namespace simpcore {

typedef unsigned __int128 u128;

// Coordinates the exact comparison covers: W, H < 2^26.
constexpr int64_t MAX_EXTENT = (int64_t)1 << 26;

// t (finite, >= 0) in units of 2^-10 px, rounded to nearest (halves up), clamped to W + H: no distance in the raster
// exceeds its diagonal, so the clamp changes no decision.
DM_PHD uint64_t quantize_tolerance(double t, int64_t H, int64_t W) {
    const double lim = (double)(H + W);
    const double c = t < lim ? t : lim;
    return (uint64_t)(c * 1024.0 + 0.5);
}

DM_PHD u128 sq(int64_t a) { return (u128)(uint64_t)(a < 0 ? -a : a) * (uint64_t)(a < 0 ? -a : a); }

// den of the interval A..B
DM_PHD u128 seg_den(int64_t ax, int64_t ay, int64_t bx, int64_t by) {
    const u128 v2 = sq(bx - ax) + sq(by - ay);
    return v2 == 0 ? (u128)1 : v2;
}

// num of vertex P in the interval A..B
DM_PHD u128 seg_num(int64_t ax, int64_t ay, int64_t bx, int64_t by, int64_t px, int64_t py) {
    const int64_t vx = bx - ax, vy = by - ay, wx = px - ax, wy = py - ay;
    const u128 w2 = sq(wx) + sq(wy);
    if (vx == 0 && vy == 0) return w2;
    const u128 v2 = sq(vx) + sq(vy);
    const int64_t dot = wx * vx + wy * vy;                      // |dot| < 2^55
    if (dot <= 0) return w2 * v2;
    if ((u128)(uint64_t)dot >= v2) return (sq(px - bx) + sq(py - by)) * v2;
    return sq(vx * wy - vy * wx);
}

// d > t_q for tolerance T (quantize_tolerance)
DM_PHD bool exceeds(u128 num, u128 den, uint64_t T) { return (num << 20) > (u128)T * T * den; }

// A top-vertex candidate: num, |2k - n| for position k of an interval of n segments, vertex index y (W + 1) + x.
struct Cand {
    u128 num;
    uint64_t mid;
    uint64_t idx;
};

// a ranks above b: the larger distance, then the position nearer the middle, then the smaller vertex index
DM_PHD bool above(const Cand& a, const Cand& b) {
    if (a.num != b.num) return a.num > b.num;
    if (a.mid != b.mid) return a.mid < b.mid;
    return a.idx < b.idx;
}

DM_PHD uint64_t mid_rank(int64_t k, int64_t n) { return (uint64_t)(2 * k > n ? 2 * k - n : n - 2 * k); }

}  // namespace simpcore
}  // namespace dm
