// Host harness around deepmerge_b200/csrc/spectral_core.cuh (TEST INFRASTRUCTURE): the loop of the score kernel of
// dm_score_spectral run sequentially on the CPU over the same per-edge functions the kernel calls.  Built by
// tests/test_spectral_core_cpu.py with g++ -ffp-contract=off.
#include "../deepmerge_b200/csrc/spectral_core.cuh"

extern "C" int score_spectral_host(const uint64_t* keys, const uint32_t* lens, long n, const int64_t* area,
                                   const int64_t* perim, const uint64_t* bsum, const uint64_t* bsq, int C,
                                   const int32_t* bbox, const float* band_w, float w_shape, float w_cmpct, float* scores) {
    using namespace dm::spectral;
    for (long e = 0; e < n; ++e) {
        const int a = (int)(keys[e] >> 32), b = (int)(keys[e] & 0xffffffffu);
        double hc = 0.0;
        for (int c = 0; c < C; ++c)
            hc = sp_add(hc, sp_color_band(band_w ? (double)band_w[c] : 1.0, area[a], bsum[(long)a * C + c], bsq[(long)a * C + c],
                                          area[b], bsum[(long)b * C + c], bsq[(long)b * C + c]));
        scores[e] = (float)sp_fusion(hc, area[a], perim[a], bbox + 4L * a, area[b], perim[b], bbox + 4L * b, (int64_t)lens[e],
                                     (double)w_shape, (double)w_cmpct);
    }
    return 0;
}
