// EXTENSION (no counterpart in the reference): a non-local-means denoiser guided by the exact per-pixel variance of the
// moments family (Rousselle, Knaus & Zwicker 2012; the definition is in include/rt_b200.h, the per-pixel functions in
// rt_denoise.cuh).
//
// denoise_nlm_kernel: one block of 32 x 8 threads filters a tile of 32 x 16 pixels.  It loads mu and v of the tile plus a halo of
// r + f pixels (clamped to the image) into shared memory as six planes, then loops over the offsets d of the search window:
//   1. e_d on the tile plus a halo of f (each thread keeps the terms of its own locations x in registers), into E;
//   2. the horizontal box sums of E over 2f + 1 columns, into H;
//   3. per output pixel, the vertical box sum of H over 2f + 1 rows gives D; w = exp(-max(0, D)) and w mu(q) are
//      accumulated in registers.
// Two barriers per offset; no atomics, and every sum runs in a fixed order, so the output is reproducible bit for bit.
// d = 0 has weight 1 and is not evaluated; an offset that puts every candidate of the tile outside the image is skipped.
//
// denoise_nlm_guided_kernel (rt_denoise_guided_device): the same body (nlm_body) with step 3's weight bounded by the feature
// weight of the candidate (guide_weight).  Each thread keeps the features and per-channel scales of its two output pixels in
// registers and reads the candidates' features through L1 (__ldg), so the shared memory and the radius bounds are those of
// the colour-only filter.  The colour-only instances are compiled from the same body with the feature code removed at compile
// time; their instructions are unchanged.
//
// denoise_nlm_cross_kernel (rt_denoise_cross_device): the dual-buffer cross filter, the same body with the weights computed
// from one half's (mu, v) and the averaged values taken from the other half's mu, staged as three more planes of shared memory
// (at most 173 KB at r = 15, f = 7).  blockIdx.z picks the direction (F_A or F_B); colour-only and guided, every
// locations-per-thread count.  dual_combine_kernel then writes out = (F_A + F_B) / 2 and the 3 x 3 error estimate.
//
// rt_render_denoised renders through the moments family (rt_adaptive.cu), converts the sums (denoise_mean_var), filters and
// tonemaps.  rt_render_denoised_dual renders two halves of every range of samples, in the rounds of rt_render_adaptive's
// schedule (adaptive_round_count), and cross-filters the whole image after each round; dual_eval_kernel applies the filtered
// stop rule (filtered_pixel_done) to the active pixels.
#include <cuda_runtime.h>

#include <cub/device/device_select.cuh>

#include <algorithm>
#include <cmath>
#include <cstring>

#include "rt_denoise.cuh"
#include "rt_device.cuh"
#include "scene_internal.h"

using namespace rtb;

namespace rtb {
// The feature buffers of the guided filter (f32 [H][W][3] each) and its constants (a kernel parameter)
struct GuideIn {
    const float *albedo, *albedo_var, *normal, *normal_var;
    float kf2_3, tau;  // 3 k_f^2, tau
};
}  // namespace rtb

namespace {

constexpr int kTileX = 32, kTileY = 16, kThreadsY = 8, kThreads = kTileX * kThreadsY;
static_assert(RT_DENOISE_MAX_HEIGHT == 65535 * kTileY, "the grid's y dimension holds at most 65 535 tiles");

// shared-memory locations of e per thread: ceil((32 + 2f)(16 + 2f) / 256)
constexpr int locations_per_thread(int f) { return ((kTileX + 2 * f) * (kTileY + 2 * f) + kThreads - 1) / kThreads; }

// planes: 6 (mu and v), or 9 for the cross filter (plus the values' mu)
size_t smem_bytes(int r, int f, int planes = 6) {
    const size_t R = (size_t)r + f;
    return sizeof(float) * (planes * (kTileX + 2 * R) * (kTileY + 2 * R) + (size_t)(kTileX + 2 * f) * (kTileY + 2 * f) + (size_t)kTileX * (kTileY + 2 * f));
}

__device__ __forceinline__ int clampi(int x, int hi) { return x < 0 ? 0 : (x > hi ? hi : x); }

// mean m, variance of the mean s and scale (guide_scale) of both features at pixel (x, y)
struct GuideAt {
    float m[2][3], s[2][3], scale[2][3];
};

__device__ __forceinline__ void guide_load(const GuideIn& g, size_t i, float m[2][3], float s[2][3]) {
#pragma unroll
    for (int c = 0; c < 3; ++c)
        m[0][c] = __ldg(g.albedo + 3 * i + c), s[0][c] = __ldg(g.albedo_var + 3 * i + c), m[1][c] = __ldg(g.normal + 3 * i + c),
        s[1][c] = __ldg(g.normal_var + 3 * i + c);
}

__device__ __forceinline__ GuideAt guide_at(const GuideIn& g, int W, int H, int x, int y) {
    GuideAt a;
    guide_load(g, (size_t)y * W + x, a.m, a.s);
    const size_t xl = (size_t)y * W + clampi(x - 1, W - 1), xr = (size_t)y * W + clampi(x + 1, W - 1);
    const size_t yd = (size_t)clampi(y - 1, H - 1) * W + x, yu = (size_t)clampi(y + 1, H - 1) * W + x;
    const float* planes[2] = {g.albedo, g.normal};
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float* m = planes[j];
            const float gx = 0.5f * (__ldg(m + 3 * xr + c) - __ldg(m + 3 * xl + c)), gy = 0.5f * (__ldg(m + 3 * yu + c) - __ldg(m + 3 * yd + c));
            a.scale[j][c] = guide_scale(a.s[j][c], gx, gy, g.kf2_3, g.tau);
        }
    return a;
}

// the feature weight of candidate q for the output pixel described by p: min over the features of exp(-max(0, d_j))
__device__ __forceinline__ float guide_weight(const GuideIn& g, int W, const GuideAt& p, int qx, int qy) {
    float m[2][3], s[2][3];
    guide_load(g, (size_t)qy * W + qx, m, s);
    const float d = fmaxf(guide_distance(p.m[0], p.s[0], p.scale[0], m[0], s[0]), guide_distance(p.m[1], p.s[1], p.scale[1], m[1], s[1]));
    return __expf(-fmaxf(d, 0.0f));
}

}  // namespace

namespace rtb {  // kernels with stable names (profiles)

// The body of all filters.  GUIDED adds the feature weight to step 3 and nothing else: the sums keep their order, so with
// feature weights of 1 the output is the colour-only filter's bit for bit.  CROSS computes the weights from (mean, var) and
// averages `values` (a third mu, staged as planes 6-8): with values == mean the output is the filter's bit for bit.
template <int NE, bool GUIDED, bool CROSS = false>
__device__ __forceinline__ void nlm_body(const float* __restrict__ mean, const float* __restrict__ var, const float* __restrict__ values, int W, int H, int r,
                                         int f, float k2, float alpha, float inv_norm, float* __restrict__ out, const GuideIn& gd) {
    extern __shared__ float smem[];
    constexpr int V = CROSS ? 6 : 0;  // the first plane of the averaged mu
    const int R = r + f;
    const int SW = kTileX + 2 * R, SH = kTileY + 2 * R, plane = SW * SH;
    const int EW = kTileX + 2 * f, EH = kTileY + 2 * f, n_e = EW * EH;
    float* E = smem + (CROSS ? 9 : 6) * plane;
    float* Hs = E + n_e;
    const int tid = threadIdx.y * kTileX + threadIdx.x;
    const int x0 = blockIdx.x * kTileX, y0 = blockIdx.y * kTileY;
    const int sx0 = x0 - R, sy0 = y0 - R;

    // mu and v of the tile plus its halo, clamped to the image, as planes mu_r mu_g mu_b v_r v_g v_b
    for (int i = tid; i < plane; i += kThreads) {
        const int gx = clampi(sx0 + i % SW, W - 1), gy = clampi(sy0 + i / SW, H - 1);
        const size_t g = 3 * ((size_t)gy * W + gx);
        for (int c = 0; c < 3; ++c) smem[c * plane + i] = mean[g + c], smem[(3 + c) * plane + i] = var[g + c];
        if constexpr (CROSS)
            for (int c = 0; c < 3; ++c) smem[(V + c) * plane + i] = values[g + c];
    }
    __syncthreads();

    // this thread's locations x of e (clamped image coordinates) and their terms that do not depend on the offset
    int xs[NE], ys[NE];
    float mx[NE][3], vx[NE][3], ax[NE][3], cx[NE][3];
#pragma unroll
    for (int k = 0; k < NE; ++k) {
        const int l = tid + k * kThreads;
        xs[k] = clampi(x0 - f + l % EW, W - 1), ys[k] = clampi(y0 - f + l / EW, H - 1);
        const int s = l < n_e ? (ys[k] - sy0) * SW + (xs[k] - sx0) : 0;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            mx[k][c] = smem[c * plane + s], vx[k][c] = smem[(3 + c) * plane + s];
            denoise_x_terms(vx[k][c], alpha, k2, &ax[k][c], &cx[k][c]);
        }
    }

    // output pixels (x0 + tx, y0 + ty + 8m), m = 0, 1; d = 0 has weight 1
    const int px = x0 + threadIdx.x;
    float wsum[2], acc[2][3];
#pragma unroll
    for (int m = 0; m < 2; ++m) {
        const int s = (y0 + threadIdx.y + kThreadsY * m - sy0) * SW + (px - sx0);
        wsum[m] = 1.0f;
#pragma unroll
        for (int c = 0; c < 3; ++c) acc[m][c] = smem[(V + c) * plane + s];
    }
    GuideAt gp[GUIDED ? 2 : 1];
    if constexpr (GUIDED) {
#pragma unroll
        for (int m = 0; m < 2; ++m) gp[m] = guide_at(gd, W, H, clampi(px, W - 1), clampi(y0 + threadIdx.y + kThreadsY * m, H - 1));
    }

    const int taps = 2 * f + 1;
    for (int dy = -r; dy <= r; ++dy) {
        if (y0 + dy > H - 1 || y0 + kTileY - 1 + dy < 0) continue;  // every candidate of the tile is outside the image
        for (int dx = -r; dx <= r; ++dx) {
            if ((dx | dy) == 0 || x0 + dx > W - 1 || x0 + kTileX - 1 + dx < 0) continue;
            // 1. e_d at this thread's locations
#pragma unroll
            for (int k = 0; k < NE; ++k) {
                const int l = tid + k * kThreads;
                if (NE * kThreads <= n_e || l < n_e) {
                    const int s = (clampi(ys[k] + dy, H - 1) - sy0) * SW + (clampi(xs[k] + dx, W - 1) - sx0);
                    float e = 0.0f;
#pragma unroll
                    for (int c = 0; c < 3; ++c)
                        e += denoise_term(mx[k][c], vx[k][c], ax[k][c], cx[k][c], smem[c * plane + s], smem[(3 + c) * plane + s], alpha, k2);
                    E[l] = e;
                }
            }
            __syncthreads();
            // 2. horizontal box sums
            for (int l = tid; l < kTileX * EH; l += kThreads) {
                const float* row = E + (l / kTileX) * EW + l % kTileX;
                float h = 0.0f;
                for (int a = 0; a < taps; ++a) h += row[a];
                Hs[l] = h;
            }
            __syncthreads();
            // 3. vertical box sums, weights, weighted means
#pragma unroll
            for (int m = 0; m < 2; ++m) {
                const int j = threadIdx.y + kThreadsY * m;
                const int qx = px + dx, qy = y0 + j + dy;
                if (qx < 0 || qx >= W || qy < 0 || qy >= H) continue;
                const float* col = Hs + j * kTileX + threadIdx.x;
                float D = 0.0f;
                for (int b = 0; b < taps; ++b) D += col[b * kTileX];
                float w = __expf(-fmaxf(D * inv_norm, 0.0f));
                if constexpr (GUIDED) w = fminf(w, guide_weight(gd, W, gp[m], qx, qy));
                const int s = (qy - sy0) * SW + (qx - sx0);
                wsum[m] += w;
#pragma unroll
                for (int c = 0; c < 3; ++c) acc[m][c] = fmaf(w, smem[(V + c) * plane + s], acc[m][c]);
            }
        }
    }
#pragma unroll
    for (int m = 0; m < 2; ++m) {
        const int py = y0 + threadIdx.y + kThreadsY * m;
        if (px >= W || py >= H) continue;
        const size_t g = 3 * ((size_t)py * W + px);
#pragma unroll
        for (int c = 0; c < 3; ++c) out[g + c] = __fdiv_rn(acc[m][c], wsum[m]);
    }
}

template <int NE>
__global__ void __launch_bounds__(kThreads) denoise_nlm_kernel(const float* __restrict__ mean, const float* __restrict__ var, int W, int H, int r, int f,
                                                               float k2, float alpha, float inv_norm, float* __restrict__ out) {
    nlm_body<NE, false>(mean, var, mean, W, H, r, f, k2, alpha, inv_norm, out, GuideIn{});
}

template <int NE>
__global__ void __launch_bounds__(kThreads) denoise_nlm_guided_kernel(const float* __restrict__ mean, const float* __restrict__ var, int W, int H, int r,
                                                                      int f, float k2, float alpha, float inv_norm, float* __restrict__ out, GuideIn g) {
    nlm_body<NE, true>(mean, var, mean, W, H, r, f, k2, alpha, inv_norm, out, g);
}

// The cross filter, both directions in one launch: blockIdx.z = 0 writes F_A (weights from B, values of A) into out_a,
// blockIdx.z = 1 writes F_B (weights from A, values of B) into out_b.
template <int NE, bool GUIDED>
__global__ void __launch_bounds__(kThreads) denoise_nlm_cross_kernel(const float* __restrict__ mean_a, const float* __restrict__ var_a,
                                                                     const float* __restrict__ mean_b, const float* __restrict__ var_b, int W, int H, int r,
                                                                     int f, float k2, float alpha, float inv_norm, float* __restrict__ out_a,
                                                                     float* __restrict__ out_b, GuideIn g) {
    const bool b = blockIdx.z != 0;
    nlm_body<NE, GUIDED, true>(b ? mean_a : mean_b, b ? var_a : var_b, b ? mean_b : mean_a, W, H, r, f, k2, alpha, inv_norm, b ? out_b : out_a, g);
}

// out = (F_A + F_B) / 2 and (err non-null) eps, the 3 x 3 mean of ((F_A - F_B) / 2)^2, per value of 3*W*H (dual_out, dual_error)
__global__ void dual_combine_kernel(const float* __restrict__ fa, const float* __restrict__ fb, int W, int H, float* __restrict__ out,
                                    float* __restrict__ err) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 3LL * W * H) return;
    out[i] = dual_out(fa[i], fb[i]);
    if (!err) return;
    const int c = (int)(i % 3);
    const long long p = i / 3;
    const int x = (int)(p % W), y = (int)(p / W);
    float a[9], b[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const size_t j = 3 * ((size_t)clampi(y + k / 3 - 1, H - 1) * W + clampi(x + k % 3 - 1, W - 1)) + c;
        a[k] = fa[j], b[k] = fb[j];
    }
    err[i] = dual_error(a, b);
}

// the sums of 3*W*H values over `counts` (per pixel) or `n` samples each -> mu, v (denoise_mean_var)
__global__ void denoise_convert_kernel(const AccumFx* __restrict__ s1, const AccumFx* __restrict__ s2, const int32_t* __restrict__ counts, uint32_t n,
                                       long long n_values, float* __restrict__ mean, float* __restrict__ var) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_values) return;
    denoise_mean_var(s1[i], s2[i], counts ? (uint32_t)counts[i / 3] : n, mean + i, var + i);
}

__global__ void denoise_tonemap_kernel(const float* __restrict__ x, int32_t* __restrict__ rgb, long long n_values) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_values) rgb[i] = to_rgb_f64((double)x[i]);
}

}  // namespace rtb

namespace {

template <int NE>
cudaError_t launch_nlm(const float* mean, const float* var, int W, int H, int r, int f, float k2, float alpha, float inv_norm, float* out,
                       const GuideIn* guide, cudaStream_t stream) {
    const size_t smem = smem_bytes(r, f);  // at most 116 KB (r = 15, f = 7); the guided filter reads the features through L1
    const void* kernel = guide ? (const void*)denoise_nlm_guided_kernel<NE> : (const void*)denoise_nlm_kernel<NE>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const dim3 grid((unsigned)((W + kTileX - 1) / kTileX), (unsigned)((H + kTileY - 1) / kTileY)), block(kTileX, kThreadsY);
    if (guide) denoise_nlm_guided_kernel<NE><<<grid, block, smem, stream>>>(mean, var, W, H, r, f, k2, alpha, inv_norm, out, *guide);
    else denoise_nlm_kernel<NE><<<grid, block, smem, stream>>>(mean, var, W, H, r, f, k2, alpha, inv_norm, out);
    return cudaGetLastError();
}

template <int NE>
cudaError_t launch_nlm_cross(const float* ma, const float* va, const float* mb, const float* vb, int W, int H, int r, int f, float k2, float alpha,
                             float inv_norm, float* fa, float* fb, const GuideIn* guide, cudaStream_t stream) {
    const size_t smem = smem_bytes(r, f, 9);  // at most 173 KB (r = 15, f = 7)
    const void* kernel = guide ? (const void*)denoise_nlm_cross_kernel<NE, true> : (const void*)denoise_nlm_cross_kernel<NE, false>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const dim3 grid((unsigned)((W + kTileX - 1) / kTileX), (unsigned)((H + kTileY - 1) / kTileY), 2), block(kTileX, kThreadsY);
    if (guide) denoise_nlm_cross_kernel<NE, true><<<grid, block, smem, stream>>>(ma, va, mb, vb, W, H, r, f, k2, alpha, inv_norm, fa, fb, *guide);
    else denoise_nlm_cross_kernel<NE, false><<<grid, block, smem, stream>>>(ma, va, mb, vb, W, H, r, f, k2, alpha, inv_norm, fa, fb, GuideIn{});
    return cudaGetLastError();
}

int check_denoise(const RtDenoise* opt, const char* who) {
    if (!opt) return set_error(RT_ERR_INVALID, "%s: null RtDenoise", who);
    if (opt->search_radius < 0 || opt->search_radius > RT_DENOISE_MAX_SEARCH_RADIUS || opt->patch_radius < 0 || opt->patch_radius > RT_DENOISE_MAX_PATCH_RADIUS)
        return set_error(RT_ERR_INVALID, "%s: search_radius must lie in [0, %d] and patch_radius in [0, %d]", who, RT_DENOISE_MAX_SEARCH_RADIUS,
                         RT_DENOISE_MAX_PATCH_RADIUS);
    if (!(opt->k > 0.0) || !(opt->alpha >= 0.0)) return set_error(RT_ERR_INVALID, "%s: k must be > 0 and alpha >= 0", who);
    return RT_OK;
}

int check_guide(const RtGuide* guide, bool render, const char* who) {
    if (!guide) return set_error(RT_ERR_INVALID, "%s: null RtGuide", who);
    if (!(guide->k_feature > 0.0) || !(guide->tau > 0.0) || std::isinf(guide->tau))
        return set_error(RT_ERR_INVALID, "%s: k_feature must be > 0 and tau finite and > 0", who);
    if (render && guide->feature_samples < 1) return set_error(RT_ERR_INVALID, "%s: feature_samples must be >= 1", who);
    return RT_OK;
}

// the filter on device buffers of the current device (arguments checked); guide: the feature-guided instance
int denoise(const float* mean, const float* var, int W, int H, const RtDenoise* opt, float* out, cudaStream_t stream, const GuideIn* guide = nullptr) {
    const int r = opt->search_radius, f = opt->patch_radius;
    const float k2 = (float)(opt->k * opt->k), alpha = (float)opt->alpha, inv_norm = (float)(1.0 / (3.0 * (2 * f + 1) * (2 * f + 1)));
    cudaError_t e;
    switch (locations_per_thread(f)) {
        case 2: e = launch_nlm<2>(mean, var, W, H, r, f, k2, alpha, inv_norm, out, guide, stream); break;
        case 3: e = launch_nlm<3>(mean, var, W, H, r, f, k2, alpha, inv_norm, out, guide, stream); break;
        case 4: e = launch_nlm<4>(mean, var, W, H, r, f, k2, alpha, inv_norm, out, guide, stream); break;
        case 5: e = launch_nlm<5>(mean, var, W, H, r, f, k2, alpha, inv_norm, out, guide, stream); break;
        default: e = launch_nlm<6>(mean, var, W, H, r, f, k2, alpha, inv_norm, out, guide, stream); break;
    }
    static_assert(locations_per_thread(0) == 2 && locations_per_thread(RT_DENOISE_MAX_PATCH_RADIUS) == 6, "denoise_nlm_kernel instances");
    if (e != cudaSuccess) return set_error(RT_ERR_CUDA, "denoise: %s", cudaGetErrorString(e));
    return RT_OK;
}

// the cross filter of the halves A and B (arguments checked): F_A into fa and F_B into fb (scratch, 3*W*H each), then out and
// (err non-null) eps; guide: the feature-guided instance
int denoise_cross(const float* ma, const float* va, const float* mb, const float* vb, int W, int H, const RtDenoise* opt, const GuideIn* guide, float* fa,
                  float* fb, float* out, float* err, cudaStream_t stream) {
    const int r = opt->search_radius, f = opt->patch_radius;
    const float k2 = (float)(opt->k * opt->k), alpha = (float)opt->alpha, inv_norm = (float)(1.0 / (3.0 * (2 * f + 1) * (2 * f + 1)));
    cudaError_t e;
    switch (locations_per_thread(f)) {
        case 2: e = launch_nlm_cross<2>(ma, va, mb, vb, W, H, r, f, k2, alpha, inv_norm, fa, fb, guide, stream); break;
        case 3: e = launch_nlm_cross<3>(ma, va, mb, vb, W, H, r, f, k2, alpha, inv_norm, fa, fb, guide, stream); break;
        case 4: e = launch_nlm_cross<4>(ma, va, mb, vb, W, H, r, f, k2, alpha, inv_norm, fa, fb, guide, stream); break;
        case 5: e = launch_nlm_cross<5>(ma, va, mb, vb, W, H, r, f, k2, alpha, inv_norm, fa, fb, guide, stream); break;
        default: e = launch_nlm_cross<6>(ma, va, mb, vb, W, H, r, f, k2, alpha, inv_norm, fa, fb, guide, stream); break;
    }
    if (e != cudaSuccess) return set_error(RT_ERR_CUDA, "denoise_cross: %s", cudaGetErrorString(e));
    const long long n_values = 3LL * W * H;
    dual_combine_kernel<<<(unsigned)((n_values + 255) / 256), 256, 0, stream>>>(fa, fb, W, H, out, err);
    if ((e = cudaGetLastError()) != cudaSuccess) return set_error(RT_ERR_CUDA, "denoise_cross: %s", cudaGetErrorString(e));
    return RT_OK;
}

bool overlaps(const float* a, const float* b, size_t n) { return a < b + n && b < a + n; }

GuideIn guide_in(const float* albedo, const float* albedo_var, const float* normal, const float* normal_var, const RtGuide* guide) {
    return GuideIn{albedo, albedo_var, normal, normal_var, (float)(3.0 * guide->k_feature * guide->k_feature), (float)guide->tau};
}

// device blocks of one denoised render, returned to the device cache on every exit
struct DenoiseBuffers {
    AccumFx *accum = nullptr, *moment2 = nullptr;
    int32_t *samples = nullptr, *rgb = nullptr;
    float *mean = nullptr, *var = nullptr, *out = nullptr;
    float* feat[4] = {nullptr, nullptr, nullptr, nullptr};  // albedo, albedo_var, normal, normal_var (guided)
    size_t n_pixels = 0;
    ~DenoiseBuffers() {
        cudaStreamSynchronize(0);
        const size_t n = n_pixels;
        rtb::cache_free(accum, 3 * n * sizeof(AccumFx)), rtb::cache_free(moment2, 3 * n * sizeof(AccumFx));
        rtb::cache_free(samples, n * sizeof(int32_t)), rtb::cache_free(rgb, 3 * n * sizeof(int32_t));
        rtb::cache_free(mean, 3 * n * sizeof(float)), rtb::cache_free(var, 3 * n * sizeof(float)), rtb::cache_free(out, 3 * n * sizeof(float));
        for (float* b : feat) rtb::cache_free(b, 3 * n * sizeof(float));
    }
};

// rt_render_denoised (guide == nullptr) and rt_render_denoised_guided
int render_denoised(const RtScene* scene_, const RtCamera* cam, const RtParams* params, const RtAdaptive* ad, const RtDenoise* opt, const RtGuide* guide,
                    int32_t* rgb, float* denoised_rgb, RtProgressFn cb, void* user, RtStats* stats, const char* who) {
    int rc = have_device();
    if (rc != RT_OK) return rc;
    if ((rc = validate_render(scene_, cam, params)) != RT_OK) return rc;
    if ((rc = check_denoise(opt, who)) != RT_OK) return rc;
    if (guide && (rc = check_guide(guide, true, who)) != RT_OK) return rc;
    if (ad) {
        if ((rc = check_adaptive(params, ad, who)) != RT_OK) return rc;
    } else {
        if (params->sample_begin != 0 || params->sample_count != 0)
            return set_error(RT_ERR_INVALID, "%s: sample_begin and sample_count must be 0 (the render owns the sample range)", who);
        if (params->samples_per_pixel < 2) return set_error(RT_ERR_INVALID, "%s: a uniform render needs samples_per_pixel >= 2 (a variance)", who);
    }
    if ((rc = check_pipeline(params)) != RT_OK) return rc;
    RtScene* scene = const_cast<RtScene*>(scene_);
    DeviceGuard g(scene->device);
    cudaStream_t stream = 0;
    const int W = params->width, H = params->height;
    const unsigned int npix = (unsigned int)W * (unsigned int)H;
    const size_t n_values = 3 * (size_t)npix;

    DenoiseBuffers b;
    b.n_pixels = npix;
    CU_TRY(rtb::cache_malloc((void**)&b.accum, n_values * sizeof(AccumFx)));
    CU_TRY(rtb::cache_malloc((void**)&b.moment2, n_values * sizeof(AccumFx)));
    if (ad) CU_TRY(rtb::cache_malloc((void**)&b.samples, npix * sizeof(int32_t)));
    CU_TRY(rtb::cache_malloc((void**)&b.rgb, n_values * sizeof(int32_t)));
    CU_TRY(rtb::cache_malloc((void**)&b.mean, n_values * sizeof(float)));
    CU_TRY(rtb::cache_malloc((void**)&b.var, n_values * sizeof(float)));
    CU_TRY(rtb::cache_malloc((void**)&b.out, n_values * sizeof(float)));
    if (guide)
        for (float*& f : b.feat) CU_TRY(rtb::cache_malloc((void**)&f, n_values * sizeof(float)));

    rtb::RowProgress rows{cb, user, H, 0};
    int launches = 0;
    uint64_t paths = 0;
    if (ad) {
        rc = adaptive_rounds(scene, cam, params, ad, b.accum, b.moment2, b.samples, stream, &rows, &launches, &paths);
        if (rc != RT_OK) return rc;
    } else {
        DCamera dc;
        make_camera(*cam, dc);
        CU_TRY(cudaMemsetAsync(scene->d_rays, 0, sizeof(unsigned long long), stream));
        CU_TRY(cudaEventRecord(scene->ev0, stream));
        CU_TRY(cudaMemsetAsync(b.accum, 0, n_values * sizeof(AccumFx), stream));
        CU_TRY(cudaMemsetAsync(b.moment2, 0, n_values * sizeof(AccumFx), stream));
        rc = launch_persist_moments(scene, dc, params, 0, params->samples_per_pixel, b.accum, b.moment2, nullptr, npix, stream, &launches);
        if (rc != RT_OK) return rc;
        paths = (uint64_t)npix * (uint64_t)params->samples_per_pixel;
    }
    if (guide) {
        RtParams fp = *params;
        fp.sample_begin = 0, fp.sample_count = guide->feature_samples;
        if ((rc = launch_features(scene, cam, &fp, b.feat[0], b.feat[1], b.feat[2], b.feat[3], stream)) != RT_OK) return rc;
        launches += 1;
    }
    const unsigned blocks = (unsigned)((n_values + 255) / 256);
    denoise_convert_kernel<<<blocks, 256, 0, stream>>>(b.accum, b.moment2, b.samples, (uint32_t)params->samples_per_pixel, (long long)n_values, b.mean,
                                                       b.var);
    CU_TRY(cudaGetLastError());
    if (guide) {
        const GuideIn gi = guide_in(b.feat[0], b.feat[1], b.feat[2], b.feat[3], guide);
        if ((rc = denoise(b.mean, b.var, W, H, opt, b.out, stream, &gi)) != RT_OK) return rc;
    } else if ((rc = denoise(b.mean, b.var, W, H, opt, b.out, stream)) != RT_OK) {
        return rc;
    }
    denoise_tonemap_kernel<<<blocks, 256, 0, stream>>>(b.out, b.rgb, (long long)n_values);
    CU_TRY(cudaGetLastError());
    launches += 3;
    CU_TRY(cudaEventRecord(scene->ev1, stream));
    if (rgb) CU_TRY(cudaMemcpyAsync(rgb, b.rgb, n_values * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    if (denoised_rgb) CU_TRY(cudaMemcpyAsync(denoised_rgb, b.out, n_values * sizeof(float), cudaMemcpyDeviceToHost, stream));
    CU_TRY(cudaStreamSynchronize(stream));
    rtb::row_progress(1, 1, &rows);  // every row of a uniform render; whatever rows the rounds did not cover
    if (stats) {
        std::memset(stats, 0, sizeof *stats);
        float ms = 0;
        CU_TRY(cudaEventElapsedTime(&ms, scene->ev0, scene->ev1));
        unsigned long long rays = 0;
        CU_TRY(cudaMemcpy(&rays, scene->d_rays, sizeof rays, cudaMemcpyDeviceToHost));
        stats->paths = paths, stats->rays = rays, stats->device_ms = ms;
        stats->kernel_launches = launches;
        stats->pipeline_used = RT_PIPELINE_PERSISTENT;
        stats->bvh_layout_used = persist_layout_used(scene, params);
    }
    return RT_OK;
}

// the active pixels after a dual round: (list non-null) the identity list of round 0 and the half count of each pixel
__global__ void dual_count_kernel(uint32_t* __restrict__ identity, unsigned int n_list, const uint32_t* __restrict__ list, int32_t half,
                                  int32_t* __restrict__ d_half) {
    const unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_list) return;
    if (identity) identity[i] = i;
    d_half[identity ? i : list[i]] = half;
}

// the active pixels after a dual round that brought each of them to n samples: whether they go on (filtered_pixel_done)
__global__ void dual_eval_kernel(const uint32_t* __restrict__ list, unsigned int n_list, uint32_t n, uint32_t n_max, double threshold,
                                 const float* __restrict__ out, const float* __restrict__ err, unsigned char* __restrict__ keep) {
    const unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_list) return;
    const size_t p = list[i];
    keep[i] = filtered_pixel_done(n, n_max, out + 3 * p, err + 3 * p, threshold) ? 0 : 1;
}

// device blocks of one dual render, returned to the device cache on every exit
struct DualBuffers {
    AccumFx* sums[4] = {nullptr, nullptr, nullptr, nullptr};  // S1 and S2 of A, S1 and S2 of B
    float* planes[8] = {};                                    // mu_A, v_A, mu_B, v_B, F_A, F_B, out, eps
    float* feat[4] = {nullptr, nullptr, nullptr, nullptr};   // albedo, albedo_var, normal, normal_var (guided)
    int32_t *half = nullptr, *rgb = nullptr;
    uint32_t *list_a = nullptr, *list_b = nullptr;
    unsigned char* keep = nullptr;
    int* n_sel = nullptr;
    void* temp = nullptr;
    size_t n_pixels = 0, temp_bytes = 0;
    ~DualBuffers() {
        cudaStreamSynchronize(0);
        const size_t n = n_pixels;
        for (AccumFx* b : sums) rtb::cache_free(b, 3 * n * sizeof(AccumFx));
        for (float* b : planes) rtb::cache_free(b, 3 * n * sizeof(float));
        for (float* b : feat) rtb::cache_free(b, 3 * n * sizeof(float));
        rtb::cache_free(half, n * sizeof(int32_t)), rtb::cache_free(rgb, 3 * n * sizeof(int32_t));
        rtb::cache_free(list_a, n * sizeof(uint32_t)), rtb::cache_free(list_b, n * sizeof(uint32_t));
        rtb::cache_free(keep, n), rtb::cache_free(n_sel, sizeof(int)), rtb::cache_free(temp, temp_bytes);
    }
};

int check_dual_counts(const RtParams* params, const RtAdaptive* ad, const char* who) {
    const int32_t spp = params->samples_per_pixel;
    if (spp < 4 || spp % 2 != 0) return set_error(RT_ERR_INVALID, "%s: samples_per_pixel must be even and >= 4 (two halves with a variance each)", who);
    if (ad && (ad->min_samples < 4 || ad->min_samples % 2 != 0))
        return set_error(RT_ERR_INVALID, "%s: min_samples must be even and >= 4 (two halves with a variance each)", who);
    return RT_OK;
}

// rt_render_denoised_dual: the rounds of adaptive_rounds' schedule (one round of samples_per_pixel for a uniform render), each
// rendering its two half ranges, converting both halves of every pixel, cross-filtering, combining and evaluating the active
// pixels with the filtered rule
int render_denoised_dual(const RtScene* scene_, const RtCamera* cam, const RtParams* params, const RtAdaptive* ad, const RtDenoise* opt,
                         const RtGuide* guide, int32_t* rgb, float* denoised_rgb, float* error_rgb, int32_t* samples, RtProgressFn cb, void* user,
                         RtStats* stats) {
    const char* who = "rt_render_denoised_dual";
    int rc = have_device();
    if (rc != RT_OK) return rc;
    if ((rc = validate_render(scene_, cam, params)) != RT_OK) return rc;
    if ((rc = check_denoise(opt, who)) != RT_OK) return rc;
    if (guide && (rc = check_guide(guide, true, who)) != RT_OK) return rc;
    if (ad) {
        if ((rc = check_adaptive(params, ad, who)) != RT_OK) return rc;
    } else if (params->sample_begin != 0 || params->sample_count != 0) {
        return set_error(RT_ERR_INVALID, "%s: sample_begin and sample_count must be 0 (the render owns the sample range)", who);
    }
    if ((rc = check_dual_counts(params, ad, who)) != RT_OK) return rc;
    if ((rc = check_pipeline(params)) != RT_OK) return rc;
    RtScene* scene = const_cast<RtScene*>(scene_);
    DeviceGuard g(scene->device);
    cudaStream_t stream = 0;
    const int W = params->width, H = params->height;
    const unsigned int npix = (unsigned int)W * (unsigned int)H;
    const size_t n_values = 3 * (size_t)npix;
    const uint32_t n_max = (uint32_t)params->samples_per_pixel, m = ad ? (uint32_t)ad->min_samples : n_max;
    const double threshold = ad ? ad->noise_threshold : 0.0;

    DualBuffers b;
    b.n_pixels = npix;
    for (AccumFx*& p : b.sums) CU_TRY(rtb::cache_malloc((void**)&p, n_values * sizeof(AccumFx)));
    for (float*& p : b.planes) CU_TRY(rtb::cache_malloc((void**)&p, n_values * sizeof(float)));
    if (guide)
        for (float*& p : b.feat) CU_TRY(rtb::cache_malloc((void**)&p, n_values * sizeof(float)));
    CU_TRY(rtb::cache_malloc((void**)&b.half, npix * sizeof(int32_t)));
    CU_TRY(rtb::cache_malloc((void**)&b.rgb, n_values * sizeof(int32_t)));
    CU_TRY(rtb::cache_malloc((void**)&b.list_a, npix * sizeof(uint32_t)));
    CU_TRY(rtb::cache_malloc((void**)&b.list_b, npix * sizeof(uint32_t)));
    CU_TRY(rtb::cache_malloc((void**)&b.keep, npix));
    CU_TRY(rtb::cache_malloc((void**)&b.n_sel, sizeof(int)));
    CU_TRY(cub::DeviceSelect::Flagged(nullptr, b.temp_bytes, b.list_a, b.keep, b.list_b, b.n_sel, (int)npix, stream));
    CU_TRY(rtb::cache_malloc(&b.temp, b.temp_bytes));
    float *mu_a = b.planes[0], *v_a = b.planes[1], *mu_b = b.planes[2], *v_b = b.planes[3], *out = b.planes[6], *err = b.planes[7];

    rtb::RowProgress rows{cb, user, H, 0};
    DCamera dc;
    make_camera(*cam, dc);
    CU_TRY(cudaMemsetAsync(scene->d_rays, 0, sizeof(unsigned long long), stream));
    CU_TRY(cudaEventRecord(scene->ev0, stream));
    int launches = 0;
    if (guide) {
        RtParams fp = *params;
        fp.sample_begin = 0, fp.sample_count = guide->feature_samples;
        if ((rc = launch_features(scene, cam, &fp, b.feat[0], b.feat[1], b.feat[2], b.feat[3], stream)) != RT_OK) return rc;
        launches += 1;
    }
    const GuideIn gi = guide ? guide_in(b.feat[0], b.feat[1], b.feat[2], b.feat[3], guide) : GuideIn{};
    for (AccumFx* p : b.sums) CU_TRY(cudaMemsetAsync(p, 0, n_values * sizeof(AccumFx), stream));
    const int n_rounds = adaptive_round_total(m, n_max);
    const unsigned blocks = (unsigned)((n_values + 255) / 256);
    uint64_t paths = 0;
    unsigned int n_list = npix;
    uint32_t n_done = 0;  // samples every active pixel holds
    for (int round = 0; n_list > 0u; ++round) {
        const uint32_t count = adaptive_round_count(n_done, m, n_max), h = count / 2;
        // round 0 covers every pixel: the list is the identity, which the render takes as a null list
        const uint32_t* list = round == 0 ? nullptr : b.list_a;
        rc = launch_persist_moments(scene, dc, params, (int)n_done, (int)h, b.sums[0], b.sums[1], list, n_list, stream, &launches);
        if (rc != RT_OK) return rc;
        rc = launch_persist_moments(scene, dc, params, (int)(n_done + h), (int)h, b.sums[2], b.sums[3], list, n_list, stream, &launches);
        if (rc != RT_OK) return rc;
        paths += (uint64_t)n_list * count;
        n_done += count;
        const unsigned list_blocks = (n_list + 255) / 256;
        dual_count_kernel<<<list_blocks, 256, 0, stream>>>(round == 0 ? b.list_a : nullptr, n_list, b.list_a, (int32_t)(n_done / 2), b.half);
        CU_TRY(cudaGetLastError());
        // every pixel: stopped pixels still feed their neighbours
        denoise_convert_kernel<<<blocks, 256, 0, stream>>>(b.sums[0], b.sums[1], b.half, 0, (long long)n_values, mu_a, v_a);
        CU_TRY(cudaGetLastError());
        denoise_convert_kernel<<<blocks, 256, 0, stream>>>(b.sums[2], b.sums[3], b.half, 0, (long long)n_values, mu_b, v_b);
        CU_TRY(cudaGetLastError());
        rc = denoise_cross(mu_a, v_a, mu_b, v_b, W, H, opt, guide ? &gi : nullptr, b.planes[4], b.planes[5], out, err, stream);
        if (rc != RT_OK) return rc;
        dual_eval_kernel<<<list_blocks, 256, 0, stream>>>(b.list_a, n_list, n_done, n_max, threshold, out, err, b.keep);
        CU_TRY(cudaGetLastError());
        launches += 6;
        int n_next = 0;
        if (n_done < n_max) {
            CU_TRY(cub::DeviceSelect::Flagged(b.temp, b.temp_bytes, b.list_a, b.keep, b.list_b, b.n_sel, (int)n_list, stream));
            CU_TRY(cudaMemcpyAsync(&n_next, b.n_sel, sizeof(int), cudaMemcpyDeviceToHost, stream));
            launches += 1;
        }
        CU_TRY(cudaStreamSynchronize(stream));
        std::swap(b.list_a, b.list_b);
        n_list = (unsigned int)n_next;
        rtb::row_progress(round + 1, n_rounds, &rows);
    }
    denoise_tonemap_kernel<<<blocks, 256, 0, stream>>>(out, b.rgb, (long long)n_values);
    CU_TRY(cudaGetLastError());
    launches += 1;
    CU_TRY(cudaEventRecord(scene->ev1, stream));
    if (rgb) CU_TRY(cudaMemcpyAsync(rgb, b.rgb, n_values * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    if (denoised_rgb) CU_TRY(cudaMemcpyAsync(denoised_rgb, out, n_values * sizeof(float), cudaMemcpyDeviceToHost, stream));
    if (error_rgb) CU_TRY(cudaMemcpyAsync(error_rgb, err, n_values * sizeof(float), cudaMemcpyDeviceToHost, stream));
    if (samples) CU_TRY(cudaMemcpyAsync(samples, b.half, npix * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    CU_TRY(cudaStreamSynchronize(stream));
    if (samples)
        for (size_t i = 0; i < npix; ++i) samples[i] *= 2;  // (the device holds the count of each half)
    rtb::row_progress(1, 1, &rows);  // whatever rows the rounds did not cover
    if (stats) {
        std::memset(stats, 0, sizeof *stats);
        float ms = 0;
        CU_TRY(cudaEventElapsedTime(&ms, scene->ev0, scene->ev1));
        unsigned long long rays = 0;
        CU_TRY(cudaMemcpy(&rays, scene->d_rays, sizeof rays, cudaMemcpyDeviceToHost));
        stats->paths = paths, stats->rays = rays, stats->device_ms = ms;
        stats->kernel_launches = launches;
        stats->pipeline_used = RT_PIPELINE_PERSISTENT;
        stats->bvh_layout_used = persist_layout_used(scene, params);
    }
    return RT_OK;
}

}  // namespace

extern "C" {

int rt_denoise_device(const float* d_mean_rgb, const float* d_var_rgb, int32_t width, int32_t height, const RtDenoise* opt, float* d_out_rgb, int device,
                      void* stream) {
    int rc = have_device();
    if (rc != RT_OK) return rc;
    if (!d_mean_rgb || !d_var_rgb || !d_out_rgb) return set_error(RT_ERR_INVALID, "rt_denoise_device: null buffer");
    if (width <= 0 || height <= 0 || height > RT_DENOISE_MAX_HEIGHT)
        return set_error(RT_ERR_INVALID, "rt_denoise_device: width must be > 0 and height in [1, %d]", RT_DENOISE_MAX_HEIGHT);
    if ((rc = check_denoise(opt, "rt_denoise_device")) != RT_OK) return rc;
    const size_t n_values = 3 * (size_t)width * (size_t)height;
    if (overlaps(d_out_rgb, d_mean_rgb, n_values) || overlaps(d_out_rgb, d_var_rgb, n_values))
        return set_error(RT_ERR_INVALID, "rt_denoise_device: d_out_rgb overlaps an input");
    if (device < 0) cudaGetDevice(&device);
    DeviceGuard g(device);
    return denoise(d_mean_rgb, d_var_rgb, width, height, opt, d_out_rgb, (cudaStream_t)stream);
}

int rt_denoise_guided_device(const float* d_mean_rgb, const float* d_var_rgb, const float* d_albedo, const float* d_albedo_var, const float* d_normal,
                             const float* d_normal_var, int32_t width, int32_t height, const RtDenoise* opt, const RtGuide* guide, float* d_out_rgb,
                             int device, void* stream) {
    int rc = have_device();
    if (rc != RT_OK) return rc;
    const float* in[6] = {d_mean_rgb, d_var_rgb, d_albedo, d_albedo_var, d_normal, d_normal_var};
    for (const float* p : in)
        if (!p) return set_error(RT_ERR_INVALID, "rt_denoise_guided_device: null buffer");
    if (!d_out_rgb) return set_error(RT_ERR_INVALID, "rt_denoise_guided_device: null buffer");
    if (width <= 0 || height <= 0 || height > RT_DENOISE_MAX_HEIGHT)
        return set_error(RT_ERR_INVALID, "rt_denoise_guided_device: width must be > 0 and height in [1, %d]", RT_DENOISE_MAX_HEIGHT);
    if ((rc = check_denoise(opt, "rt_denoise_guided_device")) != RT_OK) return rc;
    if ((rc = check_guide(guide, false, "rt_denoise_guided_device")) != RT_OK) return rc;
    const size_t n_values = 3 * (size_t)width * (size_t)height;
    for (const float* p : in)
        if (overlaps(d_out_rgb, p, n_values)) return set_error(RT_ERR_INVALID, "rt_denoise_guided_device: d_out_rgb overlaps an input");
    if (device < 0) cudaGetDevice(&device);
    DeviceGuard g(device);
    const GuideIn gi = guide_in(d_albedo, d_albedo_var, d_normal, d_normal_var, guide);
    return denoise(d_mean_rgb, d_var_rgb, width, height, opt, d_out_rgb, (cudaStream_t)stream, &gi);
}

int rt_render_denoised(const RtScene* scene, const RtCamera* cam, const RtParams* params, const RtAdaptive* ad, const RtDenoise* opt, int32_t* rgb,
                       float* denoised_rgb, RtProgressFn cb, void* user, RtStats* stats) {
    return render_denoised(scene, cam, params, ad, opt, nullptr, rgb, denoised_rgb, cb, user, stats, "rt_render_denoised");
}

int rt_denoise_cross_device(const float* d_mean_a, const float* d_var_a, const float* d_mean_b, const float* d_var_b, const float* d_albedo,
                            const float* d_albedo_var, const float* d_normal, const float* d_normal_var, int32_t width, int32_t height, const RtDenoise* opt,
                            const RtGuide* guide, float* d_out_rgb, float* d_err_rgb, int device, void* stream_) {
    const char* who = "rt_denoise_cross_device";
    int rc = have_device();
    if (rc != RT_OK) return rc;
    const float* in[8] = {d_mean_a, d_var_a, d_mean_b, d_var_b, d_albedo, d_albedo_var, d_normal, d_normal_var};
    for (int i = 0; i < 4; ++i)
        if (!in[i]) return set_error(RT_ERR_INVALID, "%s: null buffer", who);
    for (int i = 4; i < 8; ++i)
        if (!in[i] != !guide) return set_error(RT_ERR_INVALID, "%s: the four feature buffers must be given with a guide and NULL without one", who);
    if (!d_out_rgb) return set_error(RT_ERR_INVALID, "%s: null buffer", who);
    if (width <= 0 || height <= 0 || height > RT_DENOISE_MAX_HEIGHT)
        return set_error(RT_ERR_INVALID, "%s: width must be > 0 and height in [1, %d]", who, RT_DENOISE_MAX_HEIGHT);
    if ((rc = check_denoise(opt, who)) != RT_OK) return rc;
    if (guide && (rc = check_guide(guide, false, who)) != RT_OK) return rc;
    const size_t n_values = 3 * (size_t)width * (size_t)height;
    for (const float* p : in)
        if (p && (overlaps(d_out_rgb, p, n_values) || (d_err_rgb && overlaps(d_err_rgb, p, n_values))))
            return set_error(RT_ERR_INVALID, "%s: an output overlaps an input", who);
    if (d_err_rgb && overlaps(d_out_rgb, d_err_rgb, n_values)) return set_error(RT_ERR_INVALID, "%s: d_out_rgb overlaps d_err_rgb", who);
    if (device < 0) cudaGetDevice(&device);
    DeviceGuard g(device);
    cudaStream_t stream = (cudaStream_t)stream_;
    float* scratch = nullptr;  // F_A and F_B, stream-ordered so that the call stays asynchronous
    CU_TRY(cudaMallocAsync((void**)&scratch, 2 * n_values * sizeof(float), stream));
    const GuideIn gi = guide ? guide_in(d_albedo, d_albedo_var, d_normal, d_normal_var, guide) : GuideIn{};
    rc = denoise_cross(d_mean_a, d_var_a, d_mean_b, d_var_b, width, height, opt, guide ? &gi : nullptr, scratch, scratch + n_values, d_out_rgb, d_err_rgb,
                       stream);
    const cudaError_t e = cudaFreeAsync(scratch, stream);
    if (rc != RT_OK) return rc;
    if (e != cudaSuccess) return set_error(RT_ERR_CUDA, "%s: cudaFreeAsync: %s", who, cudaGetErrorString(e));
    return RT_OK;
}

int rt_render_denoised_dual(const RtScene* scene, const RtCamera* cam, const RtParams* params, const RtAdaptive* ad, const RtDenoise* opt,
                            const RtGuide* guide, int32_t* rgb, float* denoised_rgb, float* error_rgb, int32_t* samples, RtProgressFn cb, void* user,
                            RtStats* stats) {
    return render_denoised_dual(scene, cam, params, ad, opt, guide, rgb, denoised_rgb, error_rgb, samples, cb, user, stats);
}

int rt_render_denoised_guided(const RtScene* scene, const RtCamera* cam, const RtParams* params, const RtAdaptive* ad, const RtDenoise* opt,
                              const RtGuide* guide, int32_t* rgb, float* denoised_rgb, RtProgressFn cb, void* user, RtStats* stats) {
    if (!guide) {  // (render_denoised takes a null guide for the colour-only filter)
        const int rc = have_device();
        return rc != RT_OK ? rc : set_error(RT_ERR_INVALID, "rt_render_denoised_guided: null RtGuide");
    }
    return render_denoised(scene, cam, params, ad, opt, guide, rgb, denoised_rgb, cb, user, stats, "rt_render_denoised_guided");
}

}  // extern "C"
