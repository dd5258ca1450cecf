// Host harness around deepmerge_b200/csrc/rasterize_core.cuh (TEST INFRASTRUCTURE): each function of the header applied
// elementwise to arrays, on the CPU.  Built by tests/test_rasterize_cpu.py with g++ -ffp-contract=off.
#include "../deepmerge_b200/csrc/rasterize_core.cuh"

using namespace dm::rastcore;

extern "C" void pixel_host(const double* v, long n, double origin, double size, double* out) {
    for (long i = 0; i < n; ++i) out[i] = rz_pixel(v[i], origin, size);
}

extern "C" void crosses_host(const double* y0, const double* y1, const double* yc, long n, unsigned char* out) {
    for (long i = 0; i < n; ++i) out[i] = rz_crosses(y0[i], y1[i], yc[i]);
}

extern "C" void rows_host(const double* y0, const double* y1, long n, long H, long* first, long* count) {
    for (long i = 0; i < n; ++i) {
        int64_t f;
        count[i] = (long)rz_rows(y0[i], y1[i], H, &f);
        first[i] = (long)f;
    }
}

extern "C" void xi_host(const double* x0, const double* y0, const double* x1, const double* y1, const double* yc, long n,
                        double* out) {
    for (long i = 0; i < n; ++i) out[i] = rz_xi(x0[i], y0[i], x1[i], y1[i], yc[i]);
}

extern "C" void col_host(const double* xi, long n, long W, long* out) {
    for (long i = 0; i < n; ++i) out[i] = (long)rz_col(xi[i], W);
}
