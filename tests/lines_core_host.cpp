// Host build of deepmerge_b200/csrc/lines_core.cuh for tests/test_lines_cpu.py: for every segment a pixel owns, what the
// line tracer's kernels compute from the per-vertex rule, to be compared with the oracle's.
#include "../deepmerge_b200/csrc/lines_core.cuh"

using namespace dm::linecore;

// out [H * W * 4][9] = (tail x, tail y, direction, head is a node, tail is a node, successor's tail x, y, direction
// (-1s at a node), head is a vertex of the line) of every owned segment, rows of unowned ones untouched; returns the
// number of segments
extern "C" long line_core_segments(const int32_t* L, long H, long W, long ld, long* out) {
    long n = 0;
    for (long y = 0; y < H; ++y)
        for (long x = 0; x < W; ++x) {
            const unsigned m = owned_mask(L, H, W, ld, x, y);
            for (int b = 0; b < 4; ++b) {
                if (!((m >> b) & 1u)) continue;
                long* o = out + 9 * ((y * W + x) * 4 + b);
                const Seg s = orient(L, H, W, ld, x, y, b);
                const long hx = s.x + step_x(s.d), hy = s.y + step_y(s.d);
                const Next q = next_at(L, H, W, ld, hx, hy, s.d);
                o[0] = s.x; o[1] = s.y; o[2] = s.d;
                o[3] = q.node ? 1 : 0;
                o[4] = node_arms(arms(L, H, W, ld, s.x, s.y)) ? 1 : 0;
                if (q.node) {
                    o[5] = o[6] = o[7] = -1;
                } else {
                    const Owner w = owner_of(H, W, hx, hy, q.d);
                    if (!((owned_mask(L, H, W, ld, w.x, w.y) >> w.b) & 1u)) return -1;   // successor not owned there
                    const Seg t = orient(L, H, W, ld, w.x, w.y, w.b);
                    o[5] = t.x; o[6] = t.y; o[7] = t.d;
                }
                o[8] = (q.node || q.d != s.d) ? 1 : 0;
                ++n;
            }
        }
    return n;
}
