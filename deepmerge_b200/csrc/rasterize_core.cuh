// Arithmetic of dm_rasterize: the pixel transform, the crossing predicate, the rows and the crossing column of one polygon
// segment, in the operation order of shapefile.rasterize_polygons (include/deepmerge_b200.h states it).  Plain C++ that
// compiles for the device (rasterize.cu) and for the host: tests/test_rasterize_cpu.py builds this very header with g++
// and checks it bit for bit against numpy's own expressions, so that only the CUDA indexing around it is left to the
// GPU tests.  Every fp64 operation is a single IEEE add, subtract, multiply or divide (no fused multiply-add): on the
// device through the _rn intrinsics, on the host through -ffp-contract=off.
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define DM_RASTER_FN __host__ __device__ __forceinline__
#else
#define DM_RASTER_FN static inline
#endif

namespace dm {
namespace rastcore {

DM_RASTER_FN double rz_add(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
DM_RASTER_FN double rz_sub(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
DM_RASTER_FN double rz_mul(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
DM_RASTER_FN double rz_div(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}

DM_RASTER_FN bool rz_finite(double v) { return isfinite(v); }

// map coordinate -> pixel coordinate: (X - gt0) / gt1 for x, (Y - gt3) / gt5 for y
DM_RASTER_FN double rz_pixel(double v, double origin, double size) { return rz_div(rz_sub(v, origin), size); }

// the half-open rule: segment (., y0) -> (., y1) crosses the row whose centre is yc
DM_RASTER_FN bool rz_crosses(double y0, double y1, double yc) { return (y0 <= yc) != (y1 <= yc); }

// The rows r in [0, H) the segment crosses (yc = r + 0.5) are the n rows from *first on; returns n.  The candidates
// ceil(min y - 0.5) .. floor(max y - 0.5) hold every crossed row, and every candidate strictly between the two ends is
// crossed (the rounding of y - 0.5 is below one unit for |y| < 2^52, and rows beyond that are outside [0, H)), so only
// the two ends are checked against the predicate.  y0 and y1 must be finite.
DM_RASTER_FN int64_t rz_rows(double y0, double y1, int64_t H, int64_t* first) {
    const double lo = y0 < y1 ? y0 : y1, hi = y0 < y1 ? y1 : y0;
    double a = ceil(rz_sub(lo, 0.5)), b = floor(rz_sub(hi, 0.5));
    if (a < 0.0) a = 0.0;
    if (b > (double)(H - 1)) b = (double)(H - 1);
    *first = 0;
    if (!(a <= b)) return 0;
    int64_t r0 = (int64_t)a, n = (int64_t)b - r0 + 1;
    if (!rz_crosses(y0, y1, rz_add((double)r0, 0.5))) {
        ++r0;
        --n;
    }
    if (n > 0 && !rz_crosses(y0, y1, rz_add((double)(r0 + n - 1), 0.5))) --n;
    *first = r0;
    return n;
}

// x of the crossing with row centre yc: x0 + ((yc - y0) (x1 - x0)) / (y1 - y0)
DM_RASTER_FN double rz_xi(double x0, double y0, double x1, double y1, double yc) {
    return rz_add(x0, rz_div(rz_mul(rz_sub(yc, y0), rz_sub(x1, x0)), rz_sub(y1, y0)));
}

// the first column whose centre is >= xi: clip(ceil(xi - 0.5), 0, W) (0 for NaN, which the caller reports)
DM_RASTER_FN int64_t rz_col(double xi, int64_t W) {
    const double c = ceil(rz_sub(xi, 0.5));
    if (!(c > 0.0)) return 0;
    if (c > (double)W) return W;
    return (int64_t)c;
}

}  // namespace rastcore
}  // namespace dm
