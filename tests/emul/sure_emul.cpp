// TEST INFRASTRUCTURE ONLY — not part of librt_b200.so and never reachable from the product API.
//
// The per-pixel functions of the SURE filter (rt_denoise.cuh: sure_risk, sure_out_risk, sure_select, dual_out) compiled as
// plain C++ (RTB_HOST_EMULATION), so that the `-m "not gpu"` suite can compare them with numpy restatements.  Built by
// tests/test_sure_denoise.py into a temporary directory.
#define RTB_HOST_EMULATION 1
#include <cstdint>

#include "../../mu-lambda-raytracer_b200/csrc/rt_denoise.cuh"

using namespace rtb;

namespace {
int clampi(int x, int hi) { return x < 0 ? 0 : (x > hi ? hi : x); }
}  // namespace

extern "C" {

// R of `count` values: (f - mu)^2 + v (2 / w - 1)
void emul_sure_risk(const float* f, const float* mu, const float* v, const float* w, int64_t count, float* r) {
    for (int64_t i = 0; i < count; ++i) r[i] = sure_risk(f[i], mu[i], v[i], w[i]);
}

// s_hat of `count` values from R_A and R_B
void emul_sure_out_risk(const float* ra, const float* rb, int64_t count, float* s) {
    for (int64_t i = 0; i < count; ++i) s[i] = sure_out_risk(ra[i], rb[i]);
}

// the selection of sure_select_kernel on a W x H image: risk [H][W][9] (candidate-major), fa and fb [3][H][W][3]
void emul_sure_select(const float* risk, const float* fa, const float* fb, int W, int H, int b, float* out, float* err, int32_t* choice) {
    const int64_t npix = (int64_t)W * H;
    const int side = 2 * b + 1;
    for (int64_t p = 0; p < npix; ++p) {
        const int x = (int)(p % W), y = (int)(p / W);
        float e[3];
        const int j = sure_select(side * side, [&](int k) { return risk + 9 * ((int64_t)clampi(y + k / side - b, H - 1) * W + clampi(x + k % side - b, W - 1)); }, e);
        for (int c = 0; c < 3; ++c) {
            const int64_t v = 3 * p + c;
            out[v] = dual_out(fa[3 * npix * j + v], fb[3 * npix * j + v]);
            err[v] = e[c];
        }
        choice[p] = j;
    }
}

}  // extern "C"
