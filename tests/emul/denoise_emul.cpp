// TEST INFRASTRUCTURE ONLY — not part of librt_b200.so and never reachable from the product API.
//
// The per-pixel functions of the denoiser (rt_denoise.cuh: denoise_mean_var, denoise_x_terms, denoise_term) compiled as plain
// C++ (RTB_HOST_EMULATION), so that the `-m "not gpu"` suite can compare them with numpy restatements.  Built by
// tests/test_denoise.py into a temporary directory.
#define RTB_HOST_EMULATION 1
#include <cstdint>

#include "../../mu-lambda-raytracer_b200/csrc/rt_denoise.cuh"

using namespace rtb;

extern "C" {

void emul_denoise_mean_var(const uint64_t* s1, const uint64_t* s2, const uint32_t* n, int64_t count, float* mu, float* v) {
    for (int64_t i = 0; i < count; ++i) denoise_mean_var(s1[i], s2[i], n[i], mu + i, v + i);
}

// one channel's share of e for count pairs (x, y)
void emul_denoise_term(const float* mu_x, const float* v_x, const float* mu_y, const float* v_y, int64_t count, float alpha, float k2, float* out) {
    for (int64_t i = 0; i < count; ++i) {
        float ax, cx;
        denoise_x_terms(v_x[i], alpha, k2, &ax, &cx);
        out[i] = denoise_term(mu_x[i], v_x[i], ax, cx, mu_y[i], v_y[i], alpha, k2);
    }
}

int64_t emul_sizeof_rt_denoise() { return (int64_t)sizeof(RtDenoise); }

}  // extern "C"
