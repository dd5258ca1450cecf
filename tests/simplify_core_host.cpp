// Host build of deepmerge_b200/csrc/simplify_core.cuh for tests/test_simplify_cpu.py: the top vertex of an interval and
// its keep decision as the simplifier's kernels compute them, to be compared with the oracle's.
#include "../deepmerge_b200/csrc/simplify_core.cuh"

using namespace dm::simpcore;

// The top position of the interval of vertices v [n + 1, 2] (n >= 2) and whether it lies farther than T / 2^10 px.
extern "C" long core_top(const int32_t* v, long n, long W, uint64_t T, int* exceeds_out) {
    const long ax = v[0], ay = v[1], bx = v[2 * n], by = v[2 * n + 1];
    Cand best = {0, ~0ull, ~0ull};
    long bk = -1;
    for (long k = 1; k < n; ++k) {
        const long px = v[2 * k], py = v[2 * k + 1];
        const Cand c = {seg_num(ax, ay, bx, by, px, py), mid_rank(k, n), (uint64_t)py * (uint64_t)(W + 1) + (uint64_t)px};
        if (above(c, best)) {
            best = c;
            bk = k;
        }
    }
    *exceeds_out = exceeds(best.num, seg_den(ax, ay, bx, by), T);
    return bk;
}

extern "C" uint64_t core_quantize(double t, long H, long W) { return quantize_tolerance(t, H, W); }
