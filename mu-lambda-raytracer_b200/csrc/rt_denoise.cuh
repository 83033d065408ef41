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
#else
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

}  // namespace rtb
