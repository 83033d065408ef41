// TEST INFRASTRUCTURE ONLY — not part of librt_b200.so and never reachable from the product API.
//
// The per-pixel functions of the neighbourhood variance prior (rt_denoise.cuh: prior_term, prior_pool, prior_posterior,
// prior_pixel_done, prior_var_of_mean, sure_window_err) compiled as plain C++ (RTB_HOST_EMULATION), and the evaluations of
// prior_eval_kernel, prior_var_kernel and prior_sure_err_kernel over whole images, so that the `-m "not gpu"` suite can compare
// them with numpy restatements and the GPU suite can replay the rounds.  Built by tests/test_adaptive_prior.py into a temporary
// directory.
#define RTB_HOST_EMULATION 1
#include <cstdint>

#include "../../mu-lambda-raytracer_b200/csrc/rt_denoise.cuh"

using namespace rtb;

namespace {
int clampi(int x, int hi) { return x < 0 ? 0 : (x > hi ? hi : x); }
}  // namespace

extern "C" {

// the terms of `count` pixels: s1, s2 [count][3], n [count] -> t [count][4]
void emul_prior_term(const uint64_t* s1, const uint64_t* s2, const uint32_t* n, int64_t count, double* t) {
    for (int64_t i = 0; i < count; ++i) prior_term(s1 + 3 * i, s2 + 3 * i, n[i], t + 4 * i);
}

// the pool of every pixel of a W x H image of terms [H][W][4] -> sums [H][W][4]
void emul_prior_pool(const double* terms, int W, int H, int b, double* sums) {
    for (int64_t p = 0; p < (int64_t)W * H; ++p)
        prior_pool((int)(p % W), (int)(p / W), W, H, b, [&](size_t q) { return terms + 4 * q; }, sums + 4 * p);
}

void emul_prior_posterior(const double* N, const double* d, const double* sum_n, const double* sum_d, double n0, int64_t count, double* out) {
    for (int64_t i = 0; i < count; ++i) out[i] = prior_posterior(N[i], d[i], sum_n[i], sum_d[i], n0);
}

void emul_prior_done(const uint32_t* n, uint32_t n_max, const uint64_t* s1, const double* var, int64_t count, double threshold, uint8_t* out) {
    for (int64_t i = 0; i < count; ++i) out[i] = prior_pixel_done(n[i], n_max, s1 + 3 * i, var + 3 * i, threshold) ? 1 : 0;
}

// prior_term_kernel then prior_eval_kernel for EVERY pixel of a W x H image with its own count: done [H][W] and the posterior
// variances [H][W][3]
void emul_prior_eval(const uint64_t* s1, const uint64_t* s2, const uint32_t* n, int W, int H, int b, double n0, uint32_t n_max, double threshold,
                     uint8_t* done, double* var) {
    const int64_t npix = (int64_t)W * H;
    double* terms = new double[4 * npix];
    for (int64_t p = 0; p < npix; ++p) prior_term(s1 + 3 * p, s2 + 3 * p, n[p], terms + 4 * p);
    for (int64_t p = 0; p < npix; ++p) {
        double sum[4];
        prior_pool((int)(p % W), (int)(p / W), W, H, b, [&](size_t q) { return terms + 4 * q; }, sum);
        const double* t = terms + 4 * p;
        for (int c = 0; c < 3; ++c) var[3 * p + c] = prior_posterior(t[c], t[3], sum[c], sum[3], n0);
        done[p] = prior_pixel_done(n[p], n_max, s1 + 3 * p, var + 3 * p, threshold) ? 1 : 0;
    }
    delete[] terms;
}

// v~ of one half (prior_var_kernel) for every pixel: sums [H][W][3] and counts [H][W] of the half -> vt [H][W][3]
void emul_prior_var(const uint64_t* s1, const uint64_t* s2, const uint32_t* n, int W, int H, int b, double n0, float* vt) {
    const int64_t npix = (int64_t)W * H;
    double* terms = new double[4 * npix];
    for (int64_t p = 0; p < npix; ++p) prior_term(s1 + 3 * p, s2 + 3 * p, n[p], terms + 4 * p);
    for (int64_t p = 0; p < npix; ++p) {
        double sum[4];
        prior_pool((int)(p % W), (int)(p / W), W, H, b, [&](size_t q) { return terms + 4 * q; }, sum);
        const double* t = terms + 4 * p;
        for (int c = 0; c < 3; ++c) vt[3 * p + c] = prior_var_of_mean(prior_posterior(t[c], t[3], sum[c], sum[3], n0), n[p]);
    }
    delete[] terms;
}

// err' of prior_sure_err_kernel: risk [H][W][9] (candidate-major), choice [H][W] -> err [H][W][3]
void emul_sure_window_err(const float* risk, const int32_t* choice, int W, int H, int b, float* err) {
    const int side = 2 * b + 1;
    for (int64_t p = 0; p < (int64_t)W * H; ++p) {
        const int x = (int)(p % W), y = (int)(p / W);
        sure_window_err(side * side, choice[p], [&](int k) { return risk + 9 * ((int64_t)clampi(y + k / side - b, H - 1) * W + clampi(x + k % side - b, W - 1)); },
                        err + 3 * p);
    }
}

}  // extern "C"
