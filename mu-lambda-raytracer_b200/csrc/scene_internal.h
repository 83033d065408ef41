// The opaque RtScene of include/rt_b200.h and helpers shared by the CUDA translation units (rt_api.cu, rt_wavefront.cu).
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <utility>
#include <vector>

#include "dev_cache.h"
#include "flatten.h"
#include "internal.h"
#include "rt_types.h"

#define CU_TRY(expr)                                                                                                \
    do {                                                                                                            \
        cudaError_t e_ = (expr);                                                                                    \
        if (e_ != cudaSuccess) return rtb::set_error(RT_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)

namespace rtb {

struct DeviceGuard {  // run on the scene's device, restore the caller's afterwards
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (dev != prev) cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        int cur = -1;
        cudaGetDevice(&cur);
        if (prev >= 0 && cur != prev) cudaSetDevice(prev);
    }
};

struct WavefrontState;  // rt_wavefront.cu
struct PersistState;    // rt_persist.cu

DRenderParams device_params(const RtParams* p, int first_sample, int spi, int chunks);
int persist_layout_used(const RtScene* s, const RtParams* p);
void persist_preload(const RtScene* s);

struct RowProgress {  // see rtb::row_progress (rt_api.cu)
    RtProgressFn cb;
    void* user;
    int rows, reported;
};
void row_progress(int done, int total, void* user);

}  // namespace rtb

struct RtScene {
    int device = 0;
    rtb::DSceneView view{};
    rtb::FlatScene flat;  // host copy (info + hit -> description node mapping)
    std::vector<std::pair<void*, size_t>> owned;  // (block, bytes): returned to the device cache on destruction
    std::vector<cudaArray_t> arrays;
    std::vector<std::pair<size_t, size_t>> array_extent;
    std::vector<cudaTextureObject_t> textures;
    int64_t device_bytes = 0;
    rtb::OwnedDesc* desc = nullptr;  // deep copy of the description (sub-tree queries of rt_intersect_batch)
    // scratch of rt_render (host-buffer entry point), grown on demand
    rtb::AccumFx* d_accum = nullptr;  // fixed-point radiance sums (rt_types.h)
    float* d_accum_f = nullptr;       // the same as floats, for callers that ask for them
    int32_t* d_rgb = nullptr;
    size_t scratch_values = 0;
    unsigned long long* d_rays = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    rtb::WavefrontState* wf = nullptr;  // global path pool + queues (RT_PIPELINE_WAVEFRONT), allocated on first use
    rtb::PersistState* ps = nullptr;    // counters of the persistent pipeline (RT_PIPELINE_PERSISTENT)
};

namespace rtb {
int lbvh_build(FlatScene& f, float* build_ms);  // rt_lbvh.cu: BVH over f.prim_bounds on the current device
int scene_scratch(RtScene* scene, size_t n_values);  // grow d_accum / d_accum_f / d_rgb to n_values
// samples [begin, begin + count) of every pixel ADDED into the fixed-point buffer d_accum (memory of scene's device)
int accumulate_fixed(const RtScene* scene, const RtCamera* cam, const RtParams* params, AccumFx* d_accum, cudaStream_t stream, RtProgressFn cb,
                     void* user, RtStats* stats, bool sync_for_stats);
// pipelines: samples [begin, begin+count) of every pixel, ADDED into d_accum; *launches counts kernel launches
int launch_megakernel(const RtScene* s, const DCamera& cam, const RtParams* p, int begin, int count, AccumFx* d_accum, cudaStream_t stream,
                      RtProgressFn cb, void* user, int* launches);
int launch_wavefront(RtScene* s, const DCamera& cam, const RtParams* p, int begin, int count, AccumFx* d_accum, cudaStream_t stream,
                     RtProgressFn cb, void* user, int* launches);
void free_wavefront(RtScene* s);
int launch_persist(RtScene* s, const DCamera& cam, const RtParams* p, int begin, int count, AccumFx* d_accum, cudaStream_t stream,
                   RtProgressFn cb, void* user, int* launches);
bool persist_supports(const RtScene* s, const RtParams* p);
void free_persist(RtScene* s);
// the moments family of the persistent kernel (EXTENSION): samples [begin, begin + count) of the n_list pixels of d_list
// (ascending pixel ids; nullptr with n_list = W*H: every pixel), radiance_fixed ADDED into d_accum and moment2_fixed into d_moment2
int launch_persist_moments(RtScene* s, const DCamera& cam, const RtParams* p, int begin, int count, AccumFx* d_accum, AccumFx* d_moment2,
                           const uint32_t* d_list, unsigned int n_list, cudaStream_t stream, int* launches);
int have_device();  // RT_OK, or RT_ERR_NO_DEVICE with the message set
int validate_render(const RtScene* scene, const RtCamera* cam, const RtParams* p);
// rt_adaptive.cu: RT_ERR_UNSUPPORTED unless the persistent pipeline; the checks of an RtAdaptive and the sample range
int check_pipeline(const RtParams* p);
int check_adaptive(const RtParams* params, const RtAdaptive* ad, const char* who);
// the rounds of rt_render_adaptive on a validated job: zeroes d_accum / d_moment2 (3*W*H) and leaves each pixel's sums and its
// count (d_samples, W*H) on the device; records scene->ev0 before the first launch, reports rows through `rows`, synchronises
// `stream` after every round.  Adds to *launches and *paths.
int adaptive_rounds(RtScene* scene, const RtCamera* cam, const RtParams* params, const RtAdaptive* ad, AccumFx* d_accum, AccumFx* d_moment2,
                    int32_t* d_samples, cudaStream_t stream, RowProgress* rows, int* launches, uint64_t* paths);
// the schedule of the rounds: the new samples of the round after every active pixel holds n_done (0 before round 0) of at
// most n_max, with min_samples m: m, then as many as all earlier rounds together, the last one capped at n_max
inline uint32_t adaptive_round_count(uint32_t n_done, uint32_t m, uint32_t n_max) { return n_done == 0 ? m : std::min(n_done, n_max - n_done); }
inline int adaptive_round_total(uint32_t m, uint32_t n_max) {
    int n_rounds = 0;
    for (uint32_t n = 0; n < n_max; n += adaptive_round_count(n, m, n_max)) n_rounds += 1;
    return n_rounds;
}
// rt_features.cu: the first-event features of samples [begin, begin + count) of the params' range (rt_render_features_device),
// 3*W*H floats each, on a validated job; one launch
int launch_features(RtScene* s, const RtCamera* cam, const RtParams* p, float* albedo, float* albedo_var, float* normal, float* normal_var,
                    cudaStream_t stream);
}  // namespace rtb
