// "Next" row N1, second piece: the patch resize of the reference's loader, ExtractFeatureDataset.resize_data
// (MyUtils2.py:362-376): per band cv2.resize(band, (t, t), interpolation=cv2.INTER_AREA) on a square uint8 patch,
// then astype(float32) / 255.  OpenCV's arithmetic for 8-bit input is reproduced bit for bit (the CPU checker is
// oracle/resize_area.py, pinned against the executed reference and against cv2):
//   mode 0  integer shrink factor k = s / t: k == 1 copies, k == 2 is (block sum + 2) >> 2, any other k is the
//           integer block sum times float(1 / k^2) rounded half to even;
//   mode 1  fractional shrink: per axis a table of (source index, float weight) runs, reduced first along x into
//           float rows (one multiply and one add per entry, in table order, no fused multiply-add), then along y;
//   mode 2  enlargement ("area-mode" bilinear): 11-bit fixed-point coefficients and the fixed-point vertical pass
//           ((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2.
// The tables depend only on (s, t) and are built on the host (deepmerge_b200/MyUtils2.py: area_tables).
// One CTA per plane (window x band); HBM traffic is the patch bytes in and 4 t^2 bytes out.
#include "common.cuh"
#include "resize_core.cuh"

namespace dm {
namespace resize {

// ti (mode 1): start[0..t] then src[0..E);  tf: weight[0..E)
// ti (mode 2): sx[0..t), a0[0..t), a1[0..t), xmax
__global__ void __launch_bounds__(256) resize_area_kernel(const uint8_t* __restrict__ patches, int s, int t, int mode,
                                                          const int32_t* __restrict__ ti, const float* __restrict__ tf,
                                                          float* __restrict__ out) {
    extern __shared__ float buf[];                           // mode 1: [s][t] horizontally reduced rows
    const uint8_t* P = patches + (size_t)blockIdx.x * s * s;
    float* O = out + (size_t)blockIdx.x * t * t;
    if (mode == 0) {
        for (int o = threadIdx.x; o < t * t; o += blockDim.x) O[o] = shrink_integer(P, s, t, o / t, o % t);
    } else if (mode == 1) {
        const int32_t* start = ti;
        const int32_t* src = ti + t + 1;
        for (int o = threadIdx.x; o < s * t; o += blockDim.x) buf[o] = shrink_row(P, s, t, o / t, o % t, start, src, tf);
        __syncthreads();
        for (int o = threadIdx.x; o < t * t; o += blockDim.x) O[o] = shrink_col(buf, s, t, o / t, o % t, start, src, tf);
    } else {
        for (int o = threadIdx.x; o < t * t; o += blockDim.x) O[o] = enlarge(P, s, t, o / t, o % t, ti);
    }
}

}  // namespace resize
}  // namespace dm

using namespace dm;

extern "C" int dm_resize_area(const uint8_t* patches, int64_t n_planes, int64_t s, int64_t t, int mode, const int32_t* ti,
                              const float* tf, float* out, dm_stream_t stream) {
    if (n_planes < 0 || s < 1 || t < 1 || s > 4096 || t > 1024 || mode < 0 || mode > 2) return DM_ERR_BAD_ARG;
    if (mode == 0 && s % t != 0) return DM_ERR_BAD_ARG;
    if (n_planes == 0) return DM_OK;
    if (!patches || !out || (mode != 0 && !ti) || (mode == 1 && !tf)) return DM_ERR_BAD_ARG;
    if (n_planes > 0x7fffffff) return DM_ERR_BAD_ARG;
    size_t smem = 0;
    if (mode == 1) {
        smem = (size_t)s * t * sizeof(float);
        if (smem > 200 * 1024) return DM_ERR_UNSUPPORTED;     // rows of one plane must fit in shared memory
    }
    return launch(resize::resize_area_kernel, (unsigned)n_planes, 256, smem, S(stream), patches, (int)s, (int)t, mode, ti, tf,
                  out);
}
