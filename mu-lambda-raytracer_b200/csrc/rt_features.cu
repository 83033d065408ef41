// EXTENSION (no counterpart in the reference): the first-event albedo and normal features of the guided denoiser
// (rt_denoise_guided_device; the definition is in include/rt_b200.h).
//
// first_event_features_kernel: one thread owns one pixel (a warp covers an 8 x 4 tile, as item_to_pixel maps render items,
// so that the camera rays start coherent) and loops over samples [begin, begin + count) in ascending order.  Each sample
// rebuilds the first segment of the render's path for (pixel, sample) with the device functions and Philox draws of
// integrate_item / extend_and_shade: time and camera ray from draw 0, the medium event from draw 1, then the closest
// surface below it through the tree layout the persistent render uses.  The albedo and normal of that event go into f64
// sums (feature_accumulate); the pixel's mean and variance of the mean are rounded once to f32 (feature_mean_var).  No
// atomics: the output is reproducible bit for bit.  The render kernels are not touched.
#include <cuda_runtime.h>

#include <cstring>

#include "rt_denoise.cuh"
#include "rt_device.cuh"
#include "scene_internal.h"

using namespace rtb;

namespace rtb {  // kernels with stable names (profiles)

__global__ void __launch_bounds__(128) first_event_features_kernel(DSceneView S, DCamera cam, DRenderParams P, int wide, int begin, int count,
                                                                    float* __restrict__ albedo, float* __restrict__ albedo_var, float* __restrict__ normal,
                                                                    float* __restrict__ normal_var) {
    const long long item = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int px, py, chunk;
    if (!item_to_pixel(P, item, px, py, chunk)) return;
    PathRng rng;
    rng.pixel = (uint32_t)(py * P.width + px);
    rng.k0 = P.seed_lo, rng.k1 = P.seed_hi;
    double s1[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0}, s2[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};  // albedo rgb, normal xyz
    for (int k = 0; k < count; ++k) {
        rng.sample = (uint32_t)(begin + k), rng.draw = 0;
        const float time = time_of_flags(camera_time_flags(cam, rng));
        float u[4];
        rng_next4(rng, u);
        const Ray r = generate_camera_ray(cam, P, px, py, u);
        float t = RTB_INF;
        int medium = -1, prim, face;
        rng.draw = 1;
        if (S.n_media > 0) sample_media(S, r, RTB_T_MIN, rng, t, medium);
        if (wide) closest_hit4(S, r, RTB_T_MIN, t, -1, 0, t, prim, face, time);
        else closest_hit(S, r, RTB_T_MIN, t, -1, 0, t, prim, face, time);
        V3 a, n = v3(0.f, 0.f, 0.f);
        if (prim >= 0) {
            PrimRec Pr = load_prim(S.prims + prim);
            apply_motion(S, Pr, time);
            const DMaterial& M = S.mats[Pr.mat];
            Surface sf;
            surface_at(S, Pr, r, t, face, M.tex >= 0 && texture_needs_uv(S, M.tex), sf);
            n = sf.n;
            if (M.kind == MAT_DIELECTRIC) {
                a = v3(1.f, 1.f, 1.f);
            } else {
                a = material_color(S, M, sf);
                a = v3(fminf(fmaxf(a.x, 0.f), 1.f), fminf(fmaxf(a.y, 0.f), 1.f), fminf(fmaxf(a.z, 0.f), 1.f));
            }
        } else if (medium >= 0) {  // the isotropic material's colour at the event (volumes.rs:55-63: u = v = 0)
            Surface sf;
            sf.p = r.o + t * r.d, sf.n = v3(1.f, 0.f, 0.f), sf.u = 0.f, sf.v = 0.f, sf.front = true;
            a = material_color(S, S.mats[S.media[medium].mat], sf);
        } else {
            a = background_color(S, r);
        }
        feature_accumulate(s1 + 0, s2 + 0, a.x), feature_accumulate(s1 + 1, s2 + 1, a.y), feature_accumulate(s1 + 2, s2 + 2, a.z);
        feature_accumulate(s1 + 3, s2 + 3, n.x), feature_accumulate(s1 + 4, s2 + 4, n.y), feature_accumulate(s1 + 5, s2 + 5, n.z);
    }
    const size_t o = 3 * ((size_t)py * P.width + px);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        feature_mean_var(s1[c], s2[c], (uint32_t)count, albedo + o + c, albedo_var + o + c);
        feature_mean_var(s1[3 + c], s2[3 + c], (uint32_t)count, normal + o + c, normal_var + o + c);
    }
}

int launch_features(RtScene* s, const RtCamera* cam, const RtParams* p, float* albedo, float* albedo_var, float* normal, float* normal_var,
                    cudaStream_t stream) {
    if (p->bvh_layout != 0 && p->bvh_layout != 2 && p->bvh_layout != 4) return set_error(RT_ERR_INVALID, "render: bvh_layout must be 0 (auto), 2 or 4");
    const int begin = p->sample_begin, count = p->sample_count > 0 ? p->sample_count : p->samples_per_pixel - begin;
    if (count <= 0) return set_error(RT_ERR_INVALID, "render: empty sample range");
    DCamera dc;
    make_camera(*cam, dc);
    const DRenderParams P = device_params(p, begin, count, 1);
    const long long items = (long long)P.tiles_x * P.tiles_y * 32;
    const int wide = persist_layout_used(s, p) == 4 ? 1 : 0;
    first_event_features_kernel<<<(unsigned)((items + 127) / 128), 128, 0, stream>>>(s->view, dc, P, wide, begin, count, albedo, albedo_var, normal,
                                                                                      normal_var);
    CU_TRY(cudaGetLastError());
    return RT_OK;
}

}  // namespace rtb

extern "C" {

int rt_render_features_device(const RtScene* scene_, const RtCamera* cam, const RtParams* params, float* d_albedo, float* d_albedo_var, float* d_normal,
                              float* d_normal_var, void* stream_, RtStats* stats) {
    int rc = have_device();
    if (rc != RT_OK) return rc;
    if ((rc = validate_render(scene_, cam, params)) != RT_OK) return rc;
    float* out[4] = {d_albedo, d_albedo_var, d_normal, d_normal_var};
    const size_t n_values = 3 * (size_t)params->width * (size_t)params->height;
    for (int i = 0; i < 4; ++i) {
        if (!out[i]) return set_error(RT_ERR_INVALID, "rt_render_features_device: null buffer");
        for (int j = 0; j < i; ++j)
            if (out[i] < out[j] + n_values && out[j] < out[i] + n_values) return set_error(RT_ERR_INVALID, "rt_render_features_device: outputs overlap");
    }
    RtScene* scene = const_cast<RtScene*>(scene_);
    cudaStream_t stream = (cudaStream_t)stream_;
    DeviceGuard g(scene->device);
    if (stats) CU_TRY(cudaEventRecord(scene->ev0, stream));
    if ((rc = launch_features(scene, cam, params, d_albedo, d_albedo_var, d_normal, d_normal_var, stream)) != RT_OK) return rc;
    if (stats) {
        const int count = params->sample_count > 0 ? params->sample_count : params->samples_per_pixel - params->sample_begin;
        std::memset(stats, 0, sizeof *stats);
        stats->paths = stats->rays = (uint64_t)params->width * (uint64_t)params->height * (uint64_t)count;
        stats->kernel_launches = 1;
        stats->pipeline_used = RT_PIPELINE_PERSISTENT;
        stats->bvh_layout_used = persist_layout_used(scene, params);
        CU_TRY(cudaEventRecord(scene->ev1, stream));
        CU_TRY(cudaEventSynchronize(scene->ev1));
        float ms = 0;
        CU_TRY(cudaEventElapsedTime(&ms, scene->ev0, scene->ev1));
        stats->device_ms = ms;
    }
    return RT_OK;
}

}  // extern "C"
