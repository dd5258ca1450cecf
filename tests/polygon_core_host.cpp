// Host build of deepmerge_b200/csrc/polygon_core.cuh for tests/test_polygonize_cpu.py: the side masks and successors the
// polygonizer's kernels compute, for every pixel and side of a raster, to be compared with the oracle's.
#include "../deepmerge_b200/csrc/polygon_core.cuh"

// out [H * W * 4][4] = (successor pixel x, y, side, corner) of every boundary side, -1s elsewhere; returns the sides
extern "C" long poly_core_successors(const int32_t* L, long H, long W, long ld, long* out) {
    long n = 0;
    for (long y = 0; y < H; ++y)
        for (long x = 0; x < W; ++x) {
            const unsigned m = dm::polycore::side_mask(L, H, W, ld, x, y);
            for (int s = 0; s < 4; ++s) {
                long* o = out + 4 * ((y * W + x) * 4 + s);
                if (!((m >> s) & 1u)) {
                    o[0] = o[1] = o[2] = o[3] = -1;
                    continue;
                }
                const dm::polycore::Succ q = dm::polycore::successor(L, H, W, ld, x, y, s);
                o[0] = q.x; o[1] = q.y; o[2] = q.s; o[3] = q.corner ? 1 : 0;
                ++n;
            }
        }
    return n;
}
