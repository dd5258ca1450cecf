// Arithmetic of dm_score_spectral: the Baatz-Schaepe fusion value of one edge from the integer statistics of its two
// regions.  Plain C++ that compiles for the device (spectral.cu) and for the host: tests/test_spectral_core_cpu.py
// builds this very header with g++ and checks it bit for bit against spectral_fusion of tests/spectral_oracle.py, so
// that only the CUDA indexing around it is left to the GPU tests.  Every fp64 operation is a single IEEE add,
// subtract, multiply, divide or square root (no fused multiply-add): on the device through the _rn intrinsics, on
// the host through -ffp-contract=off.  The operation order below is the one include/deepmerge_b200.h states.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define DM_SPECTRAL_FN __host__ __device__ __forceinline__
#else
#include <math.h>
#define DM_SPECTRAL_FN static inline
#endif

namespace dm {
namespace spectral {

DM_SPECTRAL_FN double sp_add(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
DM_SPECTRAL_FN double sp_sub(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
DM_SPECTRAL_FN double sp_mul(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
DM_SPECTRAL_FN double sp_div(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}
DM_SPECTRAL_FN double sp_sqrt(double a) {
#if defined(__CUDA_ARCH__)
    return __dsqrt_rn(a);
#else
    return sqrt(a);
#endif
}

// population deviation of one band: sqrt(max(Q/n - (S/n)^2, 0)), the formula of RAG.attributes()
DM_SPECTRAL_FN double sp_sigma(double n, uint64_t S, uint64_t Q) {
    const double m = sp_div((double)S, n);
    const double v = sp_sub(sp_div((double)Q, n), sp_mul(m, m));
    return sp_sqrt(v < 0.0 ? 0.0 : v);
}

// w_c (n_m sigma_mc - (n_a sigma_ac + n_b sigma_bc)): band c's term of h_color; the caller adds the terms in ascending c
DM_SPECTRAL_FN double sp_color_band(double w, int64_t na, uint64_t Sa, uint64_t Qa, int64_t nb, uint64_t Sb, uint64_t Qb) {
    const double da = (double)na, db = (double)nb, dm = (double)(na + nb);
    const double ta = sp_mul(da, sp_sigma(da, Sa, Qa));
    const double tb = sp_mul(db, sp_sigma(db, Sb, Qb));
    const double tm = sp_mul(dm, sp_sigma(dm, Sa + Sb, Qa + Qb));
    return sp_mul(w, sp_sub(tm, sp_add(ta, tb)));
}

// n l / sqrt(n) and n l / b of one region; b = 2 (w + h) of its bounding box (min col, min row, max col, max row)
DM_SPECTRAL_FN double sp_cmpct(double n, double l) { return sp_div(sp_mul(n, l), sp_sqrt(n)); }
DM_SPECTRAL_FN double sp_smooth(double n, double l, int32_t x0, int32_t y0, int32_t x1, int32_t y1) {
    const int64_t b = 2 * (((int64_t)x1 - x0 + 1) + ((int64_t)y1 - y0 + 1));
    return sp_div(sp_mul(n, l), (double)b);
}

// f = (1 - w_shape) h_color + w_shape (w_cmpct h_cmpct + (1 - w_cmpct) h_smooth) of the edge (a, b) with shared
// boundary length L; ba / bb are the two bounding boxes.  h_color comes from the band loop above.
DM_SPECTRAL_FN double sp_fusion(double h_color, int64_t na, int64_t la, const int32_t* ba, int64_t nb, int64_t lb,
                                const int32_t* bb, int64_t L, double w_shape, double w_cmpct) {
    const int64_t nm = na + nb, lm = la + lb - 2 * L;
    const double da = (double)na, db = (double)nb, dm = (double)nm;
    const double fa = (double)la, fb = (double)lb, fm = (double)lm;
    const int32_t x0 = ba[0] < bb[0] ? ba[0] : bb[0], y0 = ba[1] < bb[1] ? ba[1] : bb[1];
    const int32_t x1 = ba[2] > bb[2] ? ba[2] : bb[2], y1 = ba[3] > bb[3] ? ba[3] : bb[3];
    const double h_cmpct = sp_sub(sp_cmpct(dm, fm), sp_add(sp_cmpct(da, fa), sp_cmpct(db, fb)));
    const double h_smooth = sp_sub(sp_smooth(dm, fm, x0, y0, x1, y1),
                                   sp_add(sp_smooth(da, fa, ba[0], ba[1], ba[2], ba[3]), sp_smooth(db, fb, bb[0], bb[1], bb[2], bb[3])));
    const double h_shape = sp_add(sp_mul(w_cmpct, h_cmpct), sp_mul(sp_sub(1.0, w_cmpct), h_smooth));
    return sp_add(sp_mul(sp_sub(1.0, w_shape), h_color), sp_mul(w_shape, h_shape));
}

}  // namespace spectral
}  // namespace dm
