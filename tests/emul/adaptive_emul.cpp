// TEST INFRASTRUCTURE ONLY — not part of librt_b200.so and never reachable from the product API.
//
// The exact integer and f64 functions of adaptive sampling (rt_device.cuh: moment2_fixed, adaptive_pixel_done) compiled as
// plain C++ (RTB_HOST_EMULATION), so that the `-m "not gpu"` suite can compare them with Python restatements.  Built by
// tests/test_adaptive.py into a temporary directory.
#define RTB_HOST_EMULATION 1
#include <cstdint>

#include "../../mu-lambda-raytracer_b200/csrc/rt_device.cuh"

using namespace rtb;

extern "C" {

void emul_moment2_fixed(const uint64_t* q, int64_t n, uint64_t* out) {
    for (int64_t i = 0; i < n; ++i) out[i] = moment2_fixed((AccumFx)q[i]);
}

void emul_adaptive_done(const uint32_t* n, uint32_t n_max, const uint64_t* s1, const uint64_t* s2, int64_t count, double threshold, uint8_t* out) {
    for (int64_t i = 0; i < count; ++i)
        out[i] = adaptive_pixel_done(n[i], n_max, (const AccumFx*)s1 + 3 * i, (const AccumFx*)s2 + 3 * i, threshold) ? 1 : 0;
}

}  // extern "C"
