// TEST INFRASTRUCTURE ONLY — not part of librt_b200.so and never reachable from the product API.
//
// The per-pixel functions of dual-buffer denoising (rt_denoise.cuh: dual_out, dual_error, filtered_pixel_done) compiled as
// plain C++ (RTB_HOST_EMULATION), so that the `-m "not gpu"` suite can compare them with numpy restatements.  Built by
// tests/test_dual_denoise.py into a temporary directory.
#define RTB_HOST_EMULATION 1
#include <cstdint>

#include "../../mu-lambda-raytracer_b200/csrc/rt_denoise.cuh"

using namespace rtb;

extern "C" {

// out and eps of `count` values from F_A and F_B at their nine neighbours each (count x 9)
void emul_dual(const float* fa, const float* fb, int64_t count, float* out, float* eps) {
    for (int64_t i = 0; i < count; ++i) {
        out[i] = dual_out(fa[9 * i + 4], fb[9 * i + 4]);
        eps[i] = dual_error(fa + 9 * i, fb + 9 * i);
    }
}

// the filtered stop rule of `count` pixels with counts n, filtered values out and error estimates eps (count x 3)
void emul_filtered_pixel_done(const uint32_t* n, uint32_t n_max, const float* out, const float* eps, int64_t count, double threshold,
                              uint8_t* done) {
    for (int64_t i = 0; i < count; ++i) done[i] = filtered_pixel_done(n[i], n_max, out + 3 * i, eps + 3 * i, threshold) ? 1 : 0;
}

}  // extern "C"
