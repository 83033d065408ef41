// EXTENSION: the per-pixel functions of the non-local-means denoiser (rt_denoise.cu; the definition is in
// include/rt_b200.h).
//
// Like rt_device.cuh, the file also compiles as plain C++ (RTB_HOST_EMULATION) so that tests/emul/denoise_emul.cpp can
// run the very same functions on the CPU; that build is test infrastructure only.
#pragma once
#include <math.h>
#include <stdint.h>

#include "../../include/rt_b200.h"

#if defined(__CUDACC__) && !defined(RTB_HOST_EMULATION)
#define RTD_DEV __device__ __forceinline__
#define RTD_DMUL __dmul_rn
#define RTD_DSUB __dsub_rn
#define RTD_DDIV __ddiv_rn
#define RTD_F32 __double2float_rn
#define RTD_FDIV __fdividef  // x * MUFU.RCP(y): the library builds without --use_fast_math, so the approximation is explicit
#define RTD_DADD __dadd_rn
#define RTD_FRCP __frcp_rn
#define RTD_FADD __fadd_rn
#define RTD_FSUB __fsub_rn
#define RTD_FMUL __fmul_rn
#define RTD_FDIV_RN __fdiv_rn
#define RTD_DSQRT __dsqrt_rn
#else
#define RTD_FADD(a, b) ((float)(a) + (float)(b))
#define RTD_FSUB(a, b) ((float)(a) - (float)(b))
#define RTD_FMUL(a, b) ((float)(a) * (float)(b))
#define RTD_FDIV_RN(a, b) ((float)(a) / (float)(b))
#define RTD_DSQRT(a) sqrt((double)(a))
#define RTD_DADD(a, b) ((double)(a) + (double)(b))
#define RTD_FRCP(a) (1.0f / (a))
#define RTD_DEV inline
#define RTD_DMUL(a, b) ((double)(a) * (double)(b))
#define RTD_DSUB(a, b) ((double)(a) - (double)(b))
#define RTD_DDIV(a, b) ((double)(a) / (double)(b))
#define RTD_F32(a) ((float)(a))
#define RTD_FDIV(a, b) ((a) / (b))
#endif

#define RTD_EPS 1e-10f

namespace rtb {

// Mean and variance of the mean of one channel from its fixed-point sums over n >= 2 samples, in the f64 arithmetic of
// adaptive_pixel_done (every operation rounded on its own), each rounded once to f32:
//   mu = S1 2^-32 / n,   v = max(0, (S2 2^-24 - n mu^2) / (n - 1)) / n
RTD_DEV void denoise_mean_var(uint64_t s1, uint64_t s2, uint32_t n, float* mu_out, float* v_out) {
    const double dn = (double)n;
    const double mu = RTD_DDIV(RTD_DMUL((double)s1, 2.3283064365386963e-10), dn);
    const double m2 = RTD_DMUL((double)s2, 5.9604644775390625e-08);
    double var = RTD_DDIV(RTD_DSUB(m2, RTD_DMUL(dn, RTD_DMUL(mu, mu))), RTD_DSUB(dn, 1.0));
    var = var > 0.0 ? var : 0.0;
    *mu_out = RTD_F32(mu);
    *v_out = RTD_F32(RTD_DDIV(var, dn));
}

// The terms of x in one channel of e_d(x), which do not depend on the offset d: ax = alpha v_x, cx = eps + k^2 v_x
RTD_DEV void denoise_x_terms(float v_x, float alpha, float k2, float* ax, float* cx) {
    *ax = alpha * v_x;
    *cx = fmaf(k2, v_x, RTD_EPS);
}

// One channel's share of e_d(x):
//   [(mu_x - mu_y)^2 - alpha (v_x + min(v_x, v_y))] / (eps + k^2 (v_x + v_y))
// as (d^2 - ax - alpha min(v_x, v_y)) / (cx + k^2 v_y), in f32.
RTD_DEV float denoise_term(float mu_x, float v_x, float ax, float cx, float mu_y, float v_y, float alpha, float k2) {
    const float d = mu_x - mu_y;
    const float num = fmaf(-alpha, fminf(v_x, v_y), fmaf(d, d, -ax));
    return RTD_FDIV(num, fmaf(k2, v_y, cx));
}

// ---- feature guidance (rt_features.cu, rt_denoise_guided_device)

// One sample f of one feature channel added to its f64 sums: s1 += f, s2 += f^2 (each operation rounded on its own)
RTD_DEV void feature_accumulate(double* s1, double* s2, float f) {
    *s1 = RTD_DADD(*s1, (double)f);
    *s2 = RTD_DADD(*s2, RTD_DMUL((double)f, (double)f));
}

// Mean and variance of the mean of one feature channel from its f64 sums over n >= 1 samples, each rounded once to f32:
//   mu = s1 / n,   v = max(0, (s2 - n mu^2) / (n - 1)) / n,   v = 0 for n = 1
RTD_DEV void feature_mean_var(double s1, double s2, uint32_t n, float* mu_out, float* v_out) {
    const double dn = (double)n;
    const double mu = RTD_DDIV(s1, dn);
    double var = 0.0;
    if (n > 1) {
        var = RTD_DDIV(RTD_DSUB(s2, RTD_DMUL(dn, RTD_DMUL(mu, mu))), RTD_DSUB(dn, 1.0));
        var = var > 0.0 ? var : 0.0;
    }
    *mu_out = RTD_F32(mu);
    *v_out = RTD_F32(RTD_DDIV(var, dn));
}

// The per-pixel scale of one feature channel at p: 1 / (3 k_f^2 max(tau, s(p), g(p)^2)), with the central differences
// gx, gy of the channel's mean and kf2_3 = 3 k_f^2 (a k_f^2 beyond the f32 range gives 0: the feature never matters)
RTD_DEV float guide_scale(float s_p, float gx, float gy, float kf2_3, float tau) {
    const float g2 = fmaf(gx, gx, gy * gy);
    return RTD_FRCP(kf2_3 * fmaxf(tau, fmaxf(s_p, g2)));
}

// d_j(p, q) of one feature from the three channels' means m, variances of the mean s and scales (guide_scale) at p:
//   sum_c [(m_c(p) - m_c(q))^2 - (s_c(p) + min(s_c(p), s_c(q)))] scale_c(p)
RTD_DEV float guide_distance(const float m_p[3], const float s_p[3], const float scale_p[3], const float m_q[3], const float s_q[3]) {
    float d = 0.0f;
#if defined(__CUDACC__)
#pragma unroll
#endif
    for (int c = 0; c < 3; ++c) {
        const float e = m_p[c] - m_q[c];
        d = fmaf(fmaf(e, e, -(s_p[c] + fminf(s_p[c], s_q[c]))), scale_p[c], d);
    }
    return d;
}

// ---- dual buffers (rt_denoise_cross_device, rt_render_denoised_dual)

// out of one channel from the two cross-filtered halves: (F_A + F_B) / 2
RTD_DEV float dual_out(float fa, float fb) { return RTD_FMUL(RTD_FADD(fa, fb), 0.5f); }

// eps of one channel from F_A and F_B at the nine neighbours of p (clamped to the image, in row order from the bottom left):
// the mean of ((F_A - F_B) / 2)^2, every f32 operation rounded on its own (no contraction), so that the sum has one order
RTD_DEV float dual_error(const float fa[9], const float fb[9]) {
    float s = 0.0f;
#if defined(__CUDACC__)
#pragma unroll
#endif
    for (int k = 0; k < 9; ++k) {
        const float d = RTD_FMUL(RTD_FSUB(fa[k], fb[k]), 0.5f);
        s = RTD_FADD(s, RTD_FMUL(d, d));
    }
    return RTD_FDIV_RN(s, 9.0f);
}

// The filtered stop rule for a pixel that holds n of at most n_max samples, from its filtered value `out` and error estimate
// `eps` per channel: the rule of adaptive_pixel_done with (out, eps) in place of (mu, se^2),
//   e = sqrt(eps) / (2 sqrt(max(out, 2^-16))),
// done when n == n_max or, for every channel, e <= threshold or out - 3 sqrt(eps) >= 1.  f64, every operation rounded on its own.
RTD_DEV bool filtered_pixel_done(uint32_t n, uint32_t n_max, const float out[3], const float eps[3], double threshold) {
    if (n >= n_max) return true;
    for (int c = 0; c < 3; ++c) {
        const double o = (double)out[c];
        const double se = RTD_DSQRT((double)eps[c]);
        const double e = RTD_DDIV(se, RTD_DMUL(2.0, RTD_DSQRT(o > 1.52587890625e-05 ? o : 1.52587890625e-05)));
        if (!(e <= threshold || RTD_DSUB(o, RTD_DMUL(3.0, se)) >= 1.0)) return false;
    }
    return true;
}

// ---- SURE selection (rt_denoise_sure_device, rt_render_denoised_sure)

// R of one half, candidate and channel from its filtered value f, its own mean mu and variance of the mean v, and its weight
// sum w >= 1: (f - mu)^2 + v (2 / w - 1), every f32 operation rounded on its own (w = 1 and f = mu give v exactly)
RTD_DEV float sure_risk(float f, float mu, float v, float w) {
    const float d = RTD_FSUB(f, mu);
    return RTD_FADD(RTD_FMUL(d, d), RTD_FMUL(v, RTD_FSUB(RTD_FDIV_RN(2.0f, w), 1.0f)));
}

// s_hat of one candidate and channel from the risks of the two halves: (R_A + R_B) / 2
RTD_DEV float sure_out_risk(float ra, float rb) { return RTD_FMUL(RTD_FADD(ra, rb), 0.5f); }

// The selection at p from s_hat at the n neighbours of its window (clamped to the image, in row order from the bottom left):
// risk(k) points to the nine s_hat of neighbour k, candidate-major ([j][c]).  S_j = sum_k ((s_j,0 + s_j,1) + s_j,2) / n and
// the per-channel window means, in f32 with every operation rounded on its own; returns j* = argmin S_j (ties to the smaller
// j) and err_c = max(0, the window mean of s_hat_j*,c).
template <class Risk>
RTD_DEV int sure_select(int n, Risk risk, float err[3]) {
    float S[3] = {0.0f, 0.0f, 0.0f}, E[3][3] = {{0.0f, 0.0f, 0.0f}, {0.0f, 0.0f, 0.0f}, {0.0f, 0.0f, 0.0f}};
    for (int k = 0; k < n; ++k) {
        const float* s = risk(k);
#if defined(__CUDACC__)
#pragma unroll
#endif
        for (int j = 0; j < 3; ++j) {
            S[j] = RTD_FADD(S[j], RTD_FADD(RTD_FADD(s[3 * j], s[3 * j + 1]), s[3 * j + 2]));
#if defined(__CUDACC__)
#pragma unroll
#endif
            for (int c = 0; c < 3; ++c) E[j][c] = RTD_FADD(E[j][c], s[3 * j + c]);
        }
    }
    const float fn = (float)n;
    int best = 0;
    float s_best = RTD_FDIV_RN(S[0], fn);
#if defined(__CUDACC__)
#pragma unroll
#endif
    for (int j = 1; j < 3; ++j) {
        const float s = RTD_FDIV_RN(S[j], fn);
        if (s < s_best) best = j, s_best = s;
    }
#if defined(__CUDACC__)
#pragma unroll
#endif
    for (int c = 0; c < 3; ++c) {
        const float e = RTD_FDIV_RN(best == 0 ? E[0][c] : best == 1 ? E[1][c] : E[2][c], fn);
        err[c] = e > 0.0f ? e : 0.0f;
    }
    return best;
}

// err_c = max(0, the window mean of s_hat_j,c) for a given j, in the order and f32 arithmetic of sure_select (with j = j* it is
// sure_select's err bit for bit)
template <class Risk>
RTD_DEV void sure_window_err(int n, int j, Risk risk, float err[3]) {
    float E[3] = {0.0f, 0.0f, 0.0f};
    for (int k = 0; k < n; ++k) {
        const float* s = risk(k) + 3 * j;
#if defined(__CUDACC__)
#pragma unroll
#endif
        for (int c = 0; c < 3; ++c) E[c] = RTD_FADD(E[c], s[c]);
    }
    const float fn = (float)n;
#if defined(__CUDACC__)
#pragma unroll
#endif
    for (int c = 0; c < 3; ++c) {
        const float e = RTD_FDIV_RN(E[c], fn);
        err[c] = e > 0.0f ? e : 0.0f;
    }
}

// ---- neighbourhood variance prior (rt_render_adaptive_prior, rt_render_denoised_sure_prior)

// The term of one pixel holding n >= 2 samples: N_c = max(0, S2 2^-24 - n mu^2) per channel, with mu as in adaptive_pixel_done,
// and d = n - 1, into t[4] = (N_r, N_g, N_b, d).  f64, every operation rounded on its own.
RTD_DEV void prior_term(const uint64_t s1[3], const uint64_t s2[3], uint32_t n, double t[4]) {
    const double dn = (double)n;
    for (int c = 0; c < 3; ++c) {
        const double mu = RTD_DDIV(RTD_DMUL((double)s1[c], 2.3283064365386963e-10), dn);
        const double m2 = RTD_DMUL((double)s2[c], 5.9604644775390625e-08);
        const double x = RTD_DSUB(m2, RTD_DMUL(dn, RTD_DMUL(mu, mu)));
        t[c] = x > 0.0 ? x : 0.0;
    }
    t[3] = RTD_DSUB(dn, 1.0);
}

// The pool of pixel (x, y) of a W x H image: sums of the terms of the (2b + 1)^2 window without (x, y), neighbours outside the
// image skipped, in row order from the bottom left; term(q) points to the four f64 of pixel q.  sum[4] = (sum N_c, sum d).
template <class Term>
RTD_DEV void prior_pool(int x, int y, int W, int H, int b, Term term, double sum[4]) {
    sum[0] = sum[1] = sum[2] = sum[3] = 0.0;
    for (int dy = -b; dy <= b; ++dy) {
        const int qy = y + dy;
        if (qy < 0 || qy >= H) continue;
        for (int dx = -b; dx <= b; ++dx) {
            const int qx = x + dx;
            if (qx < 0 || qx >= W || (dx | dy) == 0) continue;
            const double* t = term((size_t)qy * W + qx);
#if defined(__CUDACC__)
#pragma unroll
#endif
            for (int k = 0; k < 4; ++k) sum[k] = RTD_DADD(sum[k], t[k]);
        }
    }
}

// The posterior per-sample variance of one channel from the pixel's term (N, d) and its pool (sum_n, sum_d) with n0 pseudo-samples:
// (N + n0 P) / (d + n0), P = sum_n / sum_d; N / d (s^2, no prior) when the window holds no pixel
RTD_DEV double prior_posterior(double N, double d, double sum_n, double sum_d, double n0) {
    if (sum_d == 0.0) return RTD_DDIV(N, d);
    const double P = RTD_DDIV(sum_n, sum_d);
    return RTD_DDIV(RTD_DADD(N, RTD_DMUL(n0, P)), RTD_DADD(d, n0));
}

// The prior rule for a pixel that holds n of at most n_max samples: the rule of adaptive_pixel_done with the posterior per-sample
// variances var[3] in place of s^2
RTD_DEV bool prior_pixel_done(uint32_t n, uint32_t n_max, const uint64_t s1[3], const double var[3], double threshold) {
    if (n >= n_max) return true;
    const double dn = (double)n;
    for (int c = 0; c < 3; ++c) {
        const double mu = RTD_DDIV(RTD_DMUL((double)s1[c], 2.3283064365386963e-10), dn);
        const double se = RTD_DSQRT(RTD_DDIV(var[c], dn));
        const double e = RTD_DDIV(se, RTD_DMUL(2.0, RTD_DSQRT(mu > 1.52587890625e-05 ? mu : 1.52587890625e-05)));
        if (!(e <= threshold || RTD_DSUB(mu, RTD_DMUL(3.0, se)) >= 1.0)) return false;
    }
    return true;
}

// v~ of one channel of a half holding n >= 2 samples from its posterior per-sample variance: s~^2 / n, rounded once to f32
// (with s~^2 = s^2 it is denoise_mean_var's v bit for bit)
RTD_DEV float prior_var_of_mean(double var, uint32_t n) { return RTD_F32(RTD_DDIV(var, (double)n)); }

}  // namespace rtb
