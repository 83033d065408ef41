// TEST INFRASTRUCTURE ONLY — not part of librt_b200.so and never reachable from the product API.
//
// The per-pixel functions of feature guidance (rt_denoise.cuh: feature_accumulate, feature_mean_var, guide_scale,
// guide_distance) compiled as plain C++ (RTB_HOST_EMULATION), so that the `-m "not gpu"` suite can compare them with numpy
// restatements.  Built by tests/test_guided_denoise.py into a temporary directory.
#define RTB_HOST_EMULATION 1
#include <cstdint>

#include "../../mu-lambda-raytracer_b200/csrc/rt_denoise.cuh"

using namespace rtb;

extern "C" {

// samples f[i][k], k < n, of `count` channels, accumulated in ascending k -> mean and variance of the mean
void emul_feature_mean_var(const float* f, int64_t count, uint32_t n, float* mu, float* v) {
    for (int64_t i = 0; i < count; ++i) {
        double s1 = 0.0, s2 = 0.0;
        for (uint32_t k = 0; k < n; ++k) feature_accumulate(&s1, &s2, f[i * n + k]);
        feature_mean_var(s1, s2, n, mu + i, v + i);
    }
}

// d(p, q) of one feature for `count` pairs: m_p, s_p, m_q, s_q, gx, gy are count x 3
void emul_guide_distance(const float* m_p, const float* s_p, const float* m_q, const float* s_q, const float* gx, const float* gy, int64_t count,
                         float kf2_3, float tau, float* out) {
    for (int64_t i = 0; i < count; ++i) {
        float scale[3];
        for (int c = 0; c < 3; ++c) scale[c] = guide_scale(s_p[3 * i + c], gx[3 * i + c], gy[3 * i + c], kf2_3, tau);
        out[i] = guide_distance(m_p + 3 * i, s_p + 3 * i, scale, m_q + 3 * i, s_q + 3 * i);
    }
}

int64_t emul_sizeof_rt_guide() { return (int64_t)sizeof(RtGuide); }

}  // extern "C"
