// EXTENSION (no counterpart in the reference): per-pixel second moments and noise-threshold adaptive sampling.
//
// Both entry points run the moments family of the persistent kernel (rt_persist.cu: persist_moments_kernel), which adds
// moment2_fixed of every fixed-point sample beside the sample itself and takes its pixels from a list.  Every path owns its
// Philox counter (pixel, sample) and the sums are order-independent integers, so a pixel that receives samples [0, n) in
// several rounds holds exactly the sums of a uniform n-spp render: an adaptive image is reproducible bit for bit.
//
// Rounds (rt_render_adaptive) depend on the parameters alone: round 0 renders samples [0, m) of every pixel, each later
// round as many new samples as all earlier rounds together for the pixels still active, the last one capped at the
// maximum — so a pixel's count is always one of m, 2m, 4m, ..., max.  After each round adaptive_eval_kernel applies the
// stop rule (rt_device.cuh: adaptive_pixel_done) to the active pixels, cub::DeviceSelect::Flagged (stable) compacts the
// rest into the next list, and one host synchronisation reads its length.  adaptive_rounds runs this loop for every render
// of the family (rt_denoise.cu too) with the work of one round passed in; a uniform render is its single round, m = max.
//
// With a neighbourhood prior (rt_render_adaptive_prior; the definition is in include/rt_b200.h) the evaluation is two
// launches: prior_term_kernel updates the terms (N, d) of the pixels rendered this round, then prior_eval_kernel pools the
// window of every active pixel (one thread per pixel, the terms read through L1) and applies the prior rule.
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

int check_pipeline(const RtParams* p) {
    if (p->pipeline != RT_PIPELINE_AUTO && p->pipeline != RT_PIPELINE_PERSISTENT)
        return set_error(RT_ERR_UNSUPPORTED, "moments and adaptive sampling run on the persistent pipeline only (pipeline AUTO or PERSISTENT)");
    return RT_OK;
}

int check_sample_range(const RtParams* params, const RtAdaptive* ad, const char* who) {
    if (params->sample_begin != 0 || params->sample_count != 0)
        return set_error(RT_ERR_INVALID, "%s: sample_begin and sample_count must be 0 (the render owns the sample range)", who);
    if (!ad) return RT_OK;
    if (ad->min_samples < 2 || ad->min_samples > params->samples_per_pixel)
        return set_error(RT_ERR_INVALID, "%s: min_samples must lie in [2, samples_per_pixel]", who);
    if (!(ad->noise_threshold >= 0.0)) return set_error(RT_ERR_INVALID, "%s: noise_threshold must be >= 0", who);
    return RT_OK;
}

int check_prior(const RtPrior* prior, const char* who) {
    if (!prior) return set_error(RT_ERR_INVALID, "%s: null RtPrior", who);
    if (!std::isfinite(prior->prior_samples) || !(prior->prior_samples >= 0.0)) return set_error(RT_ERR_INVALID, "%s: prior_samples must be finite and >= 0", who);
    if (prior->radius < 1 || prior->radius > RT_PRIOR_MAX_RADIUS) return set_error(RT_ERR_INVALID, "%s: radius must lie in [1, %d]", who, RT_PRIOR_MAX_RADIUS);
    return RT_OK;
}

}  // namespace rtb

namespace {

__global__ void iota_kernel(uint32_t* __restrict__ list, unsigned int n) {
    const unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) list[i] = i;
}

// the active pixels after a round that brought each of them to n samples: their count, and whether they go on
__global__ void adaptive_eval_kernel(const uint32_t* __restrict__ list, unsigned int n_list, uint32_t n, uint32_t n_max, double threshold,
                                     const AccumFx* __restrict__ accum, const AccumFx* __restrict__ moment2, int32_t* __restrict__ samples,
                                     unsigned char* __restrict__ keep) {
    const unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_list) return;
    const uint32_t p = list[i];
    samples[p] = (int32_t)n;
    keep[i] = adaptive_pixel_done(n, n_max, accum + 3 * (size_t)p, moment2 + 3 * (size_t)p, threshold) ? 0 : 1;
}

// the active pixels after a round that brought each of them to n samples: their count and their terms (prior_term)
__global__ void prior_term_kernel(const uint32_t* __restrict__ list, unsigned int n_list, uint32_t n, const AccumFx* __restrict__ accum,
                                  const AccumFx* __restrict__ moment2, int32_t* __restrict__ samples, double* __restrict__ terms) {
    const unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_list) return;
    const uint32_t p = list[i];
    samples[p] = (int32_t)n;
    prior_term((const uint64_t*)accum + 3 * (size_t)p, (const uint64_t*)moment2 + 3 * (size_t)p, n, terms + 4 * (size_t)p);
}

// the active pixels after prior_term_kernel: the pool of each one's window, its posterior variances and the prior rule
__global__ void prior_eval_kernel(const uint32_t* __restrict__ list, unsigned int n_list, uint32_t n, uint32_t n_max, double threshold, int W,
                                  int H, int b, double n0, const AccumFx* __restrict__ accum, const double* __restrict__ terms,
                                  unsigned char* __restrict__ keep) {
    const unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_list) return;
    if (n >= n_max) {
        keep[i] = 0;
        return;
    }
    const uint32_t p = list[i];
    double sum[4], var[3];
    prior_pool((int)(p % (uint32_t)W), (int)(p / (uint32_t)W), W, H, b, [&](size_t q) { return terms + 4 * q; }, sum);
    const double* t = terms + 4 * (size_t)p;
#pragma unroll
    for (int c = 0; c < 3; ++c) var[c] = prior_posterior(t[c], t[3], sum[c], sum[3], n0);
    keep[i] = prior_pixel_done(n, n_max, (const uint64_t*)accum + 3 * (size_t)p, var, threshold) ? 0 : 1;
}

// every pixel tonemapped with its own sample count (to_rgb of raytrace.rs:59-68)
__global__ void tonemap_counts_kernel(const AccumFx* __restrict__ accum, const int32_t* __restrict__ samples, int32_t* __restrict__ rgb, int n_values) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_values) rgb[i] = to_rgb_f64((double)accum[i] * (1.0 / (RT_ACCUM_FIXED_ONE * (double)samples[i / 3])));
}

}  // namespace

namespace rtb {

int adaptive_rounds(unsigned int npix, uint32_t m, uint32_t n_max, cudaStream_t stream, RowProgress* rows, int* launches, uint64_t* paths,
                    const std::function<int()>& start, const std::function<int(const AdaptiveRound&)>& round) {
    DeviceBlocks b(stream);
    uint32_t *list, *next;
    unsigned char *keep, *temp;
    int* n_sel;
    size_t temp_bytes = 0;
    CU_TRY(b.alloc(&list, npix));
    CU_TRY(b.alloc(&next, npix));
    CU_TRY(b.alloc(&keep, npix));
    CU_TRY(b.alloc(&n_sel, 1));
    CU_TRY(cub::DeviceSelect::Flagged(nullptr, temp_bytes, list, keep, next, n_sel, (int)npix, stream));
    CU_TRY(b.alloc(&temp, temp_bytes));
    const int n_rounds = adaptive_round_total(m, n_max);  // the schedule depends on (m, max) alone: the logger is paced by rounds

    int rc = start();
    if (rc != RT_OK) return rc;
    iota_kernel<<<(npix + 255) / 256, 256, 0, stream>>>(list, npix);
    CU_TRY(cudaGetLastError());
    *launches += 1;
    unsigned int n_list = npix;
    uint32_t n_done = 0;  // samples every active pixel holds
    for (int r = 0; n_list > 0u; ++r) {
        const uint32_t count = adaptive_round_count(n_done, m, n_max);
        // round 0 covers every pixel: the list is the identity, which the render takes as a null list
        if ((rc = round(AdaptiveRound{n_done, count, list, r == 0 ? nullptr : list, n_list, keep})) != RT_OK) return rc;
        *paths += (uint64_t)n_list * count;
        n_done += count;
        int n_next = 0;
        if (n_done < n_max) {
            CU_TRY(cub::DeviceSelect::Flagged(temp, temp_bytes, list, keep, next, n_sel, (int)n_list, stream));
            CU_TRY(cudaMemcpyAsync(&n_next, n_sel, sizeof(int), cudaMemcpyDeviceToHost, stream));
            *launches += 1;
        }
        CU_TRY(cudaStreamSynchronize(stream));
        std::swap(list, next);
        n_list = (unsigned int)n_next;
        rtb::row_progress(r + 1, n_rounds, rows);
    }
    return RT_OK;
}

int moments_rounds(RtScene* scene, const RtCamera* cam, const RtParams* params, uint32_t m, double threshold, AccumFx* d_accum, AccumFx* d_moment2,
                   int32_t* d_samples, cudaStream_t stream, RowProgress* rows, int* launches, uint64_t* paths, const RtPrior* prior) {
    const unsigned int npix = (unsigned int)params->width * (unsigned int)params->height;
    const size_t n_values = 3 * (size_t)npix;
    const uint32_t n_max = (uint32_t)params->samples_per_pixel;
    DCamera dc;
    make_camera(*cam, dc);
    DeviceBlocks b(stream);
    double* terms = nullptr;  // (prior) N_r, N_g, N_b, d of every pixel
    if (prior) CU_TRY(b.alloc(&terms, 4 * (size_t)npix));
    const auto start = [&]() -> int {
        CU_TRY(cudaMemsetAsync(scene->d_rays, 0, sizeof(unsigned long long), stream));
        CU_TRY(cudaEventRecord(scene->ev0, stream));
        CU_TRY(cudaMemsetAsync(d_accum, 0, n_values * sizeof(AccumFx), stream));
        CU_TRY(cudaMemsetAsync(d_moment2, 0, n_values * sizeof(AccumFx), stream));
        return RT_OK;
    };
    const auto round = [&](const AdaptiveRound& r) -> int {
        const int rc = launch_persist_moments(scene, dc, params, (int)r.first, (int)r.count, d_accum, d_moment2, r.render_list, r.n_list, stream, launches);
        if (rc != RT_OK) return rc;
        const unsigned list_blocks = (r.n_list + 255) / 256;
        if (prior) {
            prior_term_kernel<<<list_blocks, 256, 0, stream>>>(r.list, r.n_list, r.first + r.count, d_accum, d_moment2, d_samples, terms);
            CU_TRY(cudaGetLastError());
            prior_eval_kernel<<<list_blocks, 256, 0, stream>>>(r.list, r.n_list, r.first + r.count, n_max, threshold, params->width, params->height,
                                                               prior->radius, prior->prior_samples, d_accum, terms, r.keep);
            CU_TRY(cudaGetLastError());
            *launches += 2;
            return RT_OK;
        }
        adaptive_eval_kernel<<<list_blocks, 256, 0, stream>>>(r.list, r.n_list, r.first + r.count, n_max, threshold, d_accum, d_moment2,
                                                              d_samples, r.keep);
        CU_TRY(cudaGetLastError());
        *launches += 1;
        return RT_OK;
    };
    return adaptive_rounds(npix, m, n_max, stream, rows, launches, paths, start, round);
}

int render_stats(const RtScene* scene, const RtParams* params, uint64_t paths, int launches, RtStats* stats) {
    if (!stats) return RT_OK;
    std::memset(stats, 0, sizeof *stats);
    CU_TRY(cudaEventSynchronize(scene->ev1));
    float ms = 0;
    CU_TRY(cudaEventElapsedTime(&ms, scene->ev0, scene->ev1));
    unsigned long long rays = 0;
    CU_TRY(cudaMemcpy(&rays, scene->d_rays, sizeof rays, cudaMemcpyDeviceToHost));
    stats->paths = paths, stats->rays = rays, stats->device_ms = ms;
    stats->kernel_launches = launches;
    stats->pipeline_used = RT_PIPELINE_PERSISTENT;
    stats->bvh_layout_used = persist_layout_used(scene, params);
    return RT_OK;
}

}  // namespace rtb

extern "C" {

int rt_render_moments_fixed_device(const RtScene* scene_, const RtCamera* cam, const RtParams* params, uint64_t* d_accum_fixed, uint64_t* d_moment2_fixed,
                                   void* stream_, RtStats* stats) {
    int rc = have_device();
    if (rc != RT_OK) return rc;
    if ((rc = validate_render(scene_, cam, params)) != RT_OK) return rc;
    if (!d_accum_fixed || !d_moment2_fixed) return set_error(RT_ERR_INVALID, "rt_render_moments_fixed_device: null accumulation buffer");
    if ((rc = check_pipeline(params)) != RT_OK) return rc;
    RtScene* scene = const_cast<RtScene*>(scene_);
    cudaStream_t stream = (cudaStream_t)stream_;
    DeviceGuard g(scene->device);
    const int begin = params->sample_begin;
    const int count = params->sample_count > 0 ? params->sample_count : params->samples_per_pixel - begin;
    if (count <= 0) return set_error(RT_ERR_INVALID, "render: empty sample range");
    DCamera dc;
    make_camera(*cam, dc);
    if (stats) {
        CU_TRY(cudaMemsetAsync(scene->d_rays, 0, sizeof(unsigned long long), stream));
        CU_TRY(cudaEventRecord(scene->ev0, stream));
    }
    int launches = 0;
    const unsigned int npix = (unsigned int)params->width * (unsigned int)params->height;
    rc = launch_persist_moments(scene, dc, params, begin, count, (AccumFx*)d_accum_fixed, (AccumFx*)d_moment2_fixed, nullptr, npix, stream, &launches);
    if (rc != RT_OK) return rc;
    if (stats) CU_TRY(cudaEventRecord(scene->ev1, stream));
    return render_stats(scene, params, (uint64_t)npix * count, launches, stats);
}

}  // extern "C"

namespace {

// rt_render_adaptive (prior == nullptr) and rt_render_adaptive_prior
int render_adaptive(const RtScene* scene_, const RtCamera* cam, const RtParams* params, const RtAdaptive* ad, const RtPrior* prior, int32_t* rgb,
                    int32_t* samples, uint64_t* accum_fixed, uint64_t* moment2_fixed, RtProgressFn cb, void* user, RtStats* stats, const char* who) {
    int rc = have_device();
    if (rc != RT_OK) return rc;
    if ((rc = validate_render(scene_, cam, params)) != RT_OK) return rc;
    if (!ad) return set_error(RT_ERR_INVALID, "%s: null RtAdaptive", who);
    if (prior && (rc = check_prior(prior, who)) != RT_OK) return rc;
    if ((rc = check_sample_range(params, ad, who)) != RT_OK) return rc;
    if ((rc = check_pipeline(params)) != RT_OK) return rc;
    RtScene* scene = const_cast<RtScene*>(scene_);
    DeviceGuard g(scene->device);
    cudaStream_t stream = 0;
    const unsigned int npix = (unsigned int)params->width * (unsigned int)params->height;
    const size_t n_values = 3 * (size_t)npix;

    DeviceBlocks b(stream);
    AccumFx *d_accum, *d_moment2;
    int32_t *d_samples, *d_rgb;
    CU_TRY(b.alloc(&d_accum, n_values));
    CU_TRY(b.alloc(&d_moment2, n_values));
    CU_TRY(b.alloc(&d_samples, npix));
    CU_TRY(b.alloc(&d_rgb, n_values));

    rtb::RowProgress rows{cb, user, params->height, 0};
    int launches = 0;
    uint64_t paths = 0;
    rc = moments_rounds(scene, cam, params, (uint32_t)ad->min_samples, ad->noise_threshold, d_accum, d_moment2, d_samples, stream, &rows, &launches, &paths,
                        prior);
    if (rc != RT_OK) return rc;
    tonemap_counts_kernel<<<(unsigned)((n_values + 255) / 256), 256, 0, stream>>>(d_accum, d_samples, d_rgb, (int)n_values);
    CU_TRY(cudaGetLastError());
    launches += 1;
    CU_TRY(cudaEventRecord(scene->ev1, stream));
    if (rgb) CU_TRY(cudaMemcpyAsync(rgb, d_rgb, n_values * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    if (samples) CU_TRY(cudaMemcpyAsync(samples, d_samples, npix * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    if (accum_fixed) CU_TRY(cudaMemcpyAsync(accum_fixed, d_accum, n_values * sizeof(AccumFx), cudaMemcpyDeviceToHost, stream));
    if (moment2_fixed) CU_TRY(cudaMemcpyAsync(moment2_fixed, d_moment2, n_values * sizeof(AccumFx), cudaMemcpyDeviceToHost, stream));
    CU_TRY(cudaStreamSynchronize(stream));
    rtb::row_progress(1, 1, &rows);  // whatever rows the rounds did not cover
    return render_stats(scene, params, paths, launches, stats);
}

}  // namespace

extern "C" {

int rt_render_adaptive(const RtScene* scene, const RtCamera* cam, const RtParams* params, const RtAdaptive* ad, int32_t* rgb, int32_t* samples,
                       uint64_t* accum_fixed, uint64_t* moment2_fixed, RtProgressFn cb, void* user, RtStats* stats) {
    return render_adaptive(scene, cam, params, ad, nullptr, rgb, samples, accum_fixed, moment2_fixed, cb, user, stats, "rt_render_adaptive");
}

int rt_render_adaptive_prior(const RtScene* scene, const RtCamera* cam, const RtParams* params, const RtAdaptive* ad, const RtPrior* prior, int32_t* rgb,
                             int32_t* samples, uint64_t* accum_fixed, uint64_t* moment2_fixed, RtProgressFn cb, void* user, RtStats* stats) {
    if (!prior) {  // (render_adaptive takes a null RtPrior for the rule without a prior)
        const int rc = have_device();
        return rc != RT_OK ? rc : set_error(RT_ERR_INVALID, "rt_render_adaptive_prior: null RtPrior");
    }
    return render_adaptive(scene, cam, params, ad, prior, rgb, samples, accum_fixed, moment2_fixed, cb, user, stats, "rt_render_adaptive_prior");
}

}  // extern "C"
