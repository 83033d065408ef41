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
// rest into the next list, and one host synchronisation reads its length.
#include <cuda_runtime.h>

#include <cub/device/device_select.cuh>

#include <algorithm>
#include <cmath>
#include <cstring>

#include "rt_device.cuh"
#include "scene_internal.h"

using namespace rtb;

namespace rtb {

int check_pipeline(const RtParams* p) {
    if (p->pipeline != RT_PIPELINE_AUTO && p->pipeline != RT_PIPELINE_PERSISTENT)
        return set_error(RT_ERR_UNSUPPORTED, "moments and adaptive sampling run on the persistent pipeline only (pipeline AUTO or PERSISTENT)");
    return RT_OK;
}

int check_adaptive(const RtParams* params, const RtAdaptive* ad, const char* who) {
    if (!ad) return set_error(RT_ERR_INVALID, "%s: null RtAdaptive", who);
    if (params->sample_begin != 0 || params->sample_count != 0)
        return set_error(RT_ERR_INVALID, "%s: sample_begin and sample_count must be 0 (the render owns the sample range)", who);
    if (ad->min_samples < 2 || ad->min_samples > params->samples_per_pixel)
        return set_error(RT_ERR_INVALID, "%s: min_samples must lie in [2, samples_per_pixel]", who);
    if (!(ad->noise_threshold >= 0.0)) return set_error(RT_ERR_INVALID, "%s: noise_threshold must be >= 0", who);
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

// every pixel tonemapped with its own sample count (to_rgb of raytrace.rs:59-68)
__global__ void tonemap_counts_kernel(const AccumFx* __restrict__ accum, const int32_t* __restrict__ samples, int32_t* __restrict__ rgb, int n_values) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_values) rgb[i] = to_rgb_f64((double)accum[i] * (1.0 / (RT_ACCUM_FIXED_ONE * (double)samples[i / 3])));
}

// device blocks of the rounds (lists, flags, selection scratch), returned to the device cache on every exit
struct RoundBuffers {
    uint32_t *list_a = nullptr, *list_b = nullptr;
    unsigned char* keep = nullptr;
    int* n_sel = nullptr;
    void* temp = nullptr;
    size_t n_pixels = 0, temp_bytes = 0;
    ~RoundBuffers() {
        cudaStreamSynchronize(0);  // (an error return may leave work in flight; the cache hands blocks on without a free)
        const size_t n = n_pixels;
        rtb::cache_free(list_a, n * sizeof(uint32_t)), rtb::cache_free(list_b, n * sizeof(uint32_t));
        rtb::cache_free(keep, n), rtb::cache_free(n_sel, sizeof(int)), rtb::cache_free(temp, temp_bytes);
    }
};

// the outputs of one adaptive render on the device
struct AdaptiveBuffers {
    AccumFx *accum = nullptr, *moment2 = nullptr;
    int32_t *samples = nullptr, *rgb = nullptr;
    size_t n_pixels = 0;
    ~AdaptiveBuffers() {
        cudaStreamSynchronize(0);
        const size_t n = n_pixels;
        rtb::cache_free(accum, 3 * n * sizeof(AccumFx)), rtb::cache_free(moment2, 3 * n * sizeof(AccumFx));
        rtb::cache_free(samples, n * sizeof(int32_t)), rtb::cache_free(rgb, 3 * n * sizeof(int32_t));
    }
};

}  // namespace

namespace rtb {

int adaptive_rounds(RtScene* scene, const RtCamera* cam, const RtParams* params, const RtAdaptive* ad, AccumFx* d_accum, AccumFx* d_moment2,
                    int32_t* d_samples, cudaStream_t stream, RowProgress* rows, int* launches_out, uint64_t* paths_out) {
    const unsigned int npix = (unsigned int)params->width * (unsigned int)params->height;
    const size_t n_values = 3 * (size_t)npix;
    const uint32_t n_max = (uint32_t)params->samples_per_pixel, m = (uint32_t)ad->min_samples;

    RoundBuffers b;
    b.n_pixels = npix;
    CU_TRY(rtb::cache_malloc((void**)&b.list_a, npix * sizeof(uint32_t)));
    CU_TRY(rtb::cache_malloc((void**)&b.list_b, npix * sizeof(uint32_t)));
    CU_TRY(rtb::cache_malloc((void**)&b.keep, npix));
    CU_TRY(rtb::cache_malloc((void**)&b.n_sel, sizeof(int)));
    CU_TRY(cub::DeviceSelect::Flagged(nullptr, b.temp_bytes, b.list_a, b.keep, b.list_b, b.n_sel, (int)npix, stream));
    CU_TRY(rtb::cache_malloc(&b.temp, b.temp_bytes));

    DCamera dc;
    make_camera(*cam, dc);
    const int n_rounds = adaptive_round_total(m, n_max);  // the schedule depends on (m, max) alone: the logger is paced by rounds

    CU_TRY(cudaMemsetAsync(scene->d_rays, 0, sizeof(unsigned long long), stream));
    CU_TRY(cudaEventRecord(scene->ev0, stream));
    CU_TRY(cudaMemsetAsync(d_accum, 0, n_values * sizeof(AccumFx), stream));
    CU_TRY(cudaMemsetAsync(d_moment2, 0, n_values * sizeof(AccumFx), stream));
    iota_kernel<<<(npix + 255) / 256, 256, 0, stream>>>(b.list_a, npix);
    CU_TRY(cudaGetLastError());
    int launches = 1;
    uint64_t paths = 0;
    unsigned int n_list = npix;
    uint32_t n_done = 0;  // samples every active pixel holds
    for (int round = 0; n_list > 0u; ++round) {
        const uint32_t count = adaptive_round_count(n_done, m, n_max);
        // round 0 covers every pixel: the list is the identity, which the kernel takes as a null list
        int rc = launch_persist_moments(scene, dc, params, (int)n_done, (int)count, d_accum, d_moment2, round == 0 ? nullptr : b.list_a, n_list, stream,
                                        &launches);
        if (rc != RT_OK) return rc;
        paths += (uint64_t)n_list * count;
        n_done += count;
        adaptive_eval_kernel<<<(n_list + 255) / 256, 256, 0, stream>>>(b.list_a, n_list, n_done, n_max, ad->noise_threshold, d_accum, d_moment2, d_samples,
                                                                       b.keep);
        CU_TRY(cudaGetLastError());
        launches += 1;
        int n_next = 0;
        if (n_done < n_max) {
            CU_TRY(cub::DeviceSelect::Flagged(b.temp, b.temp_bytes, b.list_a, b.keep, b.list_b, b.n_sel, (int)n_list, stream));
            CU_TRY(cudaMemcpyAsync(&n_next, b.n_sel, sizeof(int), cudaMemcpyDeviceToHost, stream));
            launches += 1;
        }
        CU_TRY(cudaStreamSynchronize(stream));
        std::swap(b.list_a, b.list_b);
        n_list = (unsigned int)n_next;
        rtb::row_progress(round + 1, n_rounds, rows);
    }
    *launches_out += launches, *paths_out += paths;
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
    if (stats) {
        std::memset(stats, 0, sizeof *stats);
        stats->paths = (uint64_t)npix * count;
        stats->kernel_launches = launches;
        stats->pipeline_used = RT_PIPELINE_PERSISTENT;
        stats->bvh_layout_used = persist_layout_used(scene, params);
        CU_TRY(cudaEventRecord(scene->ev1, stream));
        CU_TRY(cudaEventSynchronize(scene->ev1));
        float ms = 0;
        CU_TRY(cudaEventElapsedTime(&ms, scene->ev0, scene->ev1));
        unsigned long long rays = 0;
        CU_TRY(cudaMemcpy(&rays, scene->d_rays, sizeof rays, cudaMemcpyDeviceToHost));
        stats->rays = rays, stats->device_ms = ms;
    }
    return RT_OK;
}

int rt_render_adaptive(const RtScene* scene_, const RtCamera* cam, const RtParams* params, const RtAdaptive* ad, int32_t* rgb, int32_t* samples,
                       uint64_t* accum_fixed, uint64_t* moment2_fixed, RtProgressFn cb, void* user, RtStats* stats) {
    int rc = have_device();
    if (rc != RT_OK) return rc;
    if ((rc = validate_render(scene_, cam, params)) != RT_OK) return rc;
    if ((rc = check_adaptive(params, ad, "rt_render_adaptive")) != RT_OK) return rc;
    if ((rc = check_pipeline(params)) != RT_OK) return rc;
    RtScene* scene = const_cast<RtScene*>(scene_);
    DeviceGuard g(scene->device);
    cudaStream_t stream = 0;
    const unsigned int npix = (unsigned int)params->width * (unsigned int)params->height;
    const size_t n_values = 3 * (size_t)npix;

    AdaptiveBuffers b;
    b.n_pixels = npix;
    CU_TRY(rtb::cache_malloc((void**)&b.accum, n_values * sizeof(AccumFx)));
    CU_TRY(rtb::cache_malloc((void**)&b.moment2, n_values * sizeof(AccumFx)));
    CU_TRY(rtb::cache_malloc((void**)&b.samples, npix * sizeof(int32_t)));
    CU_TRY(rtb::cache_malloc((void**)&b.rgb, n_values * sizeof(int32_t)));

    rtb::RowProgress rows{cb, user, params->height, 0};
    int launches = 0;
    uint64_t paths = 0;
    rc = adaptive_rounds(scene, cam, params, ad, b.accum, b.moment2, b.samples, stream, &rows, &launches, &paths);
    if (rc != RT_OK) return rc;
    tonemap_counts_kernel<<<(unsigned)((n_values + 255) / 256), 256, 0, stream>>>(b.accum, b.samples, b.rgb, (int)n_values);
    CU_TRY(cudaGetLastError());
    launches += 1;
    CU_TRY(cudaEventRecord(scene->ev1, stream));
    if (rgb) CU_TRY(cudaMemcpyAsync(rgb, b.rgb, n_values * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    if (samples) CU_TRY(cudaMemcpyAsync(samples, b.samples, npix * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    if (accum_fixed) CU_TRY(cudaMemcpyAsync(accum_fixed, b.accum, n_values * sizeof(AccumFx), cudaMemcpyDeviceToHost, stream));
    if (moment2_fixed) CU_TRY(cudaMemcpyAsync(moment2_fixed, b.moment2, n_values * sizeof(AccumFx), cudaMemcpyDeviceToHost, stream));
    CU_TRY(cudaStreamSynchronize(stream));
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

}  // extern "C"
