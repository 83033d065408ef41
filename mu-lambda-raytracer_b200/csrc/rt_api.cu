// CUDA side of librt_b200: kernels + the extern "C" entry points of include/rt_b200.h that touch the device.
//
// The boundary replaced here is Renderer::new_with_rng + Renderer::render (src/raytrace.rs:151-186) as called by
// do_tracing (src/main.rs:147-157).  There is NO CPU fallback: without a CUDA device every entry point returns
// RT_ERR_NO_DEVICE.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "flatten.h"
#include "internal.h"
#include "rt_device.cuh"
#include "scene_internal.h"

using namespace rtb;

// ============================================================================ kernels

// Megakernel: one thread integrates `samples_per_item` consecutive samples of one pixel (regenerating paths in
// place), a warp covers an 8x4 pixel tile, and the per-thread sum is added to the accumulation buffer with three
// float reductions.  rays_out counts path segments (warp-aggregated).
__global__ void __launch_bounds__(128) render_items_kernel(DSceneView S, DCamera cam, DRenderParams P, long long n_items, int total_samples,
                                                           AccumFx* __restrict__ accum, unsigned long long* __restrict__ rays_out) {
    long long item = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t n_rays = 0;
    int px, py, chunk;
    if (item < n_items && item_to_pixel(P, item, px, py, chunk)) {
        int first = chunk * P.samples_per_item;
        int count = min(P.samples_per_item, total_samples - first);
        AccumFx sum[3];
        integrate_item(S, cam, P, px, py, P.sample_begin + first, count, sum, n_rays);
        AccumFx* dst = accum + 3 * ((size_t)py * P.width + px);
        atomicAdd(dst + 0, sum[0]);
        atomicAdd(dst + 1, sum[1]);
        atomicAdd(dst + 2, sum[2]);
    }
    // one counter update per warp
    for (int off = 16; off > 0; off >>= 1) n_rays += __shfl_down_sync(0xffffffffu, n_rays, off);
    if ((threadIdx.x & 31) == 0 && n_rays) atomicAdd(rays_out, (unsigned long long)n_rays);
}

__global__ void tonemap_kernel(const float* __restrict__ accum, int32_t* __restrict__ rgb, int n_values, double scale) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_values) rgb[i] = to_rgb_f64((double)accum[i] * scale);
}
// the same from fixed-point sums: scale = 2^-32 / samples_per_pixel
__global__ void tonemap_fixed_kernel(const AccumFx* __restrict__ accum, int32_t* __restrict__ rgb, int n_values, double scale) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_values) rgb[i] = to_rgb_f64((double)accum[i] * scale);
}
// fixed-point sums -> float sums (one rounding per value); add = 1 accumulates into `out`
__global__ void fixed_to_float_kernel(const AccumFx* __restrict__ accum, float* __restrict__ out, long long n_values, int add) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_values) return;
    float v = (float)((double)accum[i] * (1.0 / 4294967296.0));
    out[i] = add ? out[i] + v : v;
}

__global__ void intersect_kernel(DSceneView S, int mode, const float* __restrict__ rays, long long n, RtHit* __restrict__ out, float time) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float q[8];
    for (int k = 0; k < 8; ++k) q[k] = rays[8 * i + k];
    RtHit h;
    intersect_query(S, mode, q, h, time);
    out[i] = h;
}

__global__ void texture_kernel(DSceneView S, int tex, const float* __restrict__ uvp, long long n, float* __restrict__ rgb) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* q = uvp + 5 * i;
    V3 c = texture_value(S, tex, q[0], q[1], v3(q[2], q[3], q[4]));
    rgb[3 * i] = c.x, rgb[3 * i + 1] = c.y, rgb[3 * i + 2] = c.z;
}

__global__ void scatter_kernel(DSceneView S, const RtScatterIn* __restrict__ in, long long n, RtScatterOut* __restrict__ out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    RtScatterIn q = in[i];
    RtScatterOut o;
    scatter_query(S, q, o);
    out[i] = o;
}

__global__ void camera_kernel(DCamera cam, DRenderParams P, const int32_t* __restrict__ pixel, const int32_t* __restrict__ sample, long long n,
                              float* __restrict__ rays, float* __restrict__ us) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float r6[6], u4[4];
    camera_query(cam, P, pixel[i], sample[i], r6, u4);
    for (int k = 0; k < 6; ++k) rays[6 * i + k] = r6[k];
    for (int k = 0; k < 4; ++k) us[4 * i + k] = u4[k];
}

// ============================================================================ host-side scene object

namespace {

template <class T>
int upload(const std::vector<T>& v, T** out, std::vector<std::pair<void*, size_t>>& owned, int64_t& bytes) {
    *out = nullptr;
    size_t n = std::max<size_t>(v.size(), 1) * sizeof(T);  // never a null table
    void* p = nullptr;
    CU_TRY(rtb::cache_malloc(&p, n));
    owned.emplace_back(p, n);
    if (!v.empty()) CU_TRY(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    *out = (T*)p;
    bytes += (int64_t)n;
    return RT_OK;
}

}  // namespace


namespace rtb {

int have_device() {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return set_error(RT_ERR_NO_DEVICE, "no usable CUDA device (%s); librt_b200 has no CPU path", e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    return RT_OK;
}

}  // namespace rtb

namespace {

int upload_scene(RtScene* s) {
    FlatScene& f = s->flat;
    DSceneView& v = s->view;
    DNode* nodes;
    DNode4* nodes4;
    DPrim* prims;
    DBigSphere* big;
    DInstance* inst;
    DMaterial* mats;
    DTexture* texs;
    DMedium* media;
    DPrim* media_prims;
    float* pvec;
    float* moving;
    unsigned short* pperm;
    int rc;
    if ((rc = upload(f.nodes, &nodes, s->owned, s->device_bytes))) return rc;
    if ((rc = upload(f.nodes4, &nodes4, s->owned, s->device_bytes))) return rc;
    if ((rc = upload(f.prims, &prims, s->owned, s->device_bytes))) return rc;
    if ((rc = upload(f.big, &big, s->owned, s->device_bytes))) return rc;
    if ((rc = upload(f.inst, &inst, s->owned, s->device_bytes))) return rc;
    if ((rc = upload(f.mats, &mats, s->owned, s->device_bytes))) return rc;
    if ((rc = upload(f.texs, &texs, s->owned, s->device_bytes))) return rc;
    if ((rc = upload(f.media, &media, s->owned, s->device_bytes))) return rc;
    if ((rc = upload(f.media_prims, &media_prims, s->owned, s->device_bytes))) return rc;
    if ((rc = upload(f.perlin_vec, &pvec, s->owned, s->device_bytes))) return rc;
    if ((rc = upload(f.moving, &moving, s->owned, s->device_bytes))) return rc;
    if ((rc = upload(f.perlin_perm, &pperm, s->owned, s->device_bytes))) return rc;
    // image textures -> CUDA texture objects (RGBA8, point sampling, clamp, texel coordinates)
    std::vector<DImage> images;
    for (auto& im : f.images) {
        cudaChannelFormatDesc cd = cudaCreateChannelDesc<uchar4>();
        cudaArray_t arr = nullptr;
        CU_TRY(rtb::cache_malloc_array(&arr, &cd, im.width, im.height));
        s->arrays.push_back(arr);
        s->array_extent.emplace_back((size_t)im.width, (size_t)im.height);
        CU_TRY(cudaMemcpy2DToArray(arr, 0, 0, im.rgba.data(), (size_t)im.width * 4, (size_t)im.width * 4, im.height, cudaMemcpyHostToDevice));
        cudaResourceDesc rd{};
        rd.resType = cudaResourceTypeArray;
        rd.res.array.array = arr;
        cudaTextureDesc td{};
        td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
        td.filterMode = cudaFilterModePoint;
        td.readMode = cudaReadModeElementType;
        td.normalizedCoords = 0;
        cudaTextureObject_t tex = 0;
        CU_TRY(cudaCreateTextureObject(&tex, &rd, &td, nullptr));
        s->textures.push_back(tex);
        images.push_back(DImage{(unsigned long long)tex, im.width, im.height});
        s->device_bytes += (int64_t)im.width * im.height * 4;
    }
    DImage* dimages;
    if ((rc = upload(images, &dimages, s->owned, s->device_bytes))) return rc;
    v.nodes = nodes, v.nodes4 = f.nodes4.empty() ? nullptr : nodes4, v.n_nodes4 = (int)f.nodes4.size(), v.prims = prims, v.big = big, v.inst = inst, v.mats = mats, v.texs = texs, v.media = media, v.media_prims = media_prims;
    v.perlin_vec = pvec, v.perlin_perm = pperm, v.images = dimages, v.moving = moving;
    v.n_nodes = (int)f.nodes.size(), v.n_prims = (int)f.prims.size(), v.n_media = (int)f.media.size();
    v.n_perlin = (int)(f.perlin_vec.size() / (4 * RTB_PERLIN_POINTS));
    v.media_general = f.media.size() > 4 ? 1 : 0;
    for (const auto& m : f.media) v.media_general |= m.count > 1 ? 1 : 0;
    v.clear_media = f.clear_media;
    v.bg_kind = f.bg_kind;
    for (int k = 0; k < 3; ++k) v.bg_top[k] = f.bg_top[k], v.bg_bottom[k] = f.bg_bottom[k];
    return RT_OK;
}

void free_scene(RtScene* s) {
    if (!s) return;
    {
        DeviceGuard g(s->device);
        cudaDeviceSynchronize();  // cached blocks are handed to the next scene without a real free: nothing may still be using them
        for (auto t : s->textures) cudaDestroyTextureObject(t);
        for (size_t i = 0; i < s->arrays.size(); ++i) rtb::cache_free_array(s->arrays[i], s->array_extent[i].first, s->array_extent[i].second);
        for (auto& b : s->owned) rtb::cache_free(b.first, b.second);
        rtb::cache_free(s->d_accum, s->scratch_values * sizeof(AccumFx));
        rtb::cache_free(s->d_accum_f, s->scratch_values * sizeof(float));
        rtb::cache_free(s->d_rgb, s->scratch_values * sizeof(int32_t));
        rtb::cache_free(s->d_rays, sizeof(unsigned long long));
        if (s->ev0) cudaEventDestroy(s->ev0);
        if (s->ev1) cudaEventDestroy(s->ev1);
        free_wavefront(s);
        free_persist(s);
    }
    if (s->desc) rtb::free_desc(s->desc);
    delete s;
}

int create_scene(const RtSceneDesc* desc, int32_t root, bool build_bvh, int device, bool keep_desc, RtScene** out) {
    RtScene* s = new RtScene();
    std::string err;
    int rc = flatten_scene(desc, root, build_bvh ? BUILD_AUTO : BUILD_NONE, s->flat, err);
    if (rc != RT_OK) {
        delete s;
        return set_error(rc, "%s", err.c_str());
    }
    if (device < 0) cudaGetDevice(&device);
    s->device = device;
    DeviceGuard g(device);
    if (s->flat.needs_device_build) {  // large scene: linear BVH built on the GPU (rt_lbvh.cu); the host SAH sweep if that tree is too deep
        rc = rtb::lbvh_build(s->flat, &s->flat.device_build_ms);
        if (rc == RT_ERR_UNSUPPORTED) {
            s->flat = FlatScene();
            rc = flatten_scene(desc, root, BUILD_HOST, s->flat, err);
            if (rc != RT_OK) set_error(rc, "%s", err.c_str());
        }
        if (rc != RT_OK) {
            delete s;
            return rc;
        }
    }
    rc = upload_scene(s);
    if (rc == RT_OK && rtb::cache_malloc((void**)&s->d_rays, sizeof(unsigned long long)) != cudaSuccess) rc = set_error(RT_ERR_CUDA, "cudaMalloc failed");
    if (rc == RT_OK && (cudaEventCreate(&s->ev0) != cudaSuccess || cudaEventCreate(&s->ev1) != cudaSuccess)) rc = set_error(RT_ERR_CUDA, "cudaEventCreate failed");
    if (rc != RT_OK) {
        free_scene(s);
        return rc;
    }
    if (keep_desc) s->desc = rtb::clone_desc(desc);
    if (build_bvh) rtb::persist_preload(s);
    *out = s;
    return RT_OK;
}

}  // namespace

namespace rtb {

int validate_render(const RtScene* scene, const RtCamera* cam, const RtParams* p) {
    if (!scene || !cam || !p) return set_error(RT_ERR_INVALID, "render: null argument");
    if (p->width < 2 || p->height < 2) return set_error(RT_ERR_INVALID, "render: image must be at least 2x2 (u = (i+U)/(W-1))");
    if ((long long)p->width * p->height > (1ll << 31) / 3) return set_error(RT_ERR_INVALID, "render: image too large");
    if (p->samples_per_pixel <= 0 || p->max_depth < 0) return set_error(RT_ERR_INVALID, "render: samples_per_pixel must be > 0 and max_depth >= 0");
    if (p->sample_begin < 0 || p->sample_count < 0) return set_error(RT_ERR_INVALID, "render: negative sample range");
    // sample indices are int on the host (accumulate_fixed, the launch loops) and uint32 on the device
    if ((long long)p->sample_begin + p->sample_count > RT_MAX_SAMPLE_END) return set_error(RT_ERR_INVALID, "render: sample range ends beyond 2^31 - 1");
    if (p->pipeline < RT_PIPELINE_AUTO || p->pipeline > RT_PIPELINE_PERSISTENT) return set_error(RT_ERR_INVALID, "render: unknown pipeline");
    return RT_OK;
}

DRenderParams device_params(const RtParams* p, int first_sample, int spi, int chunks) {
    DRenderParams P{};
    P.width = p->width, P.height = p->height, P.max_depth = p->max_depth;
    P.sample_begin = first_sample, P.samples_per_item = spi, P.items_per_pixel = chunks;
    P.tiles_x = (p->width + 7) / 8, P.tiles_y = (p->height + 3) / 4;
    P.seed_lo = (uint32_t)p->seed, P.seed_hi = (uint32_t)(p->seed >> 32);
    P.inv_wm1 = 1.0f / ((float)p->width - 1.0f), P.inv_hm1 = 1.0f / ((float)p->height - 1.0f);
    P.inv_npix = 1.0 / ((double)p->width * (double)p->height);
    return P;
}

// the megakernel pipeline: samples [begin, begin+count) of every pixel, added into d_accum
int launch_megakernel(const RtScene* s, const DCamera& cam, const RtParams* p, int begin, int count, AccumFx* d_accum, cudaStream_t stream,
                      RtProgressFn cb, void* user, int* launches) {
    int spi = p->samples_per_item > 0 ? p->samples_per_item : 16;
    spi = std::min(spi, count);
    long long pixels_padded = (long long)((p->width + 7) / 8) * ((p->height + 3) / 4) * 32;
    // bound one launch to ~2^28 camera paths so that progress can be reported and no launch runs for seconds
    long long max_chunks = std::max<long long>(1, (1ll << 28) / (pixels_padded * spi));
    int done = 0;
    while (done < count) {
        int chunks_left = (count - done + spi - 1) / spi;
        int chunks = (int)std::min<long long>(chunks_left, max_chunks);
        int samples = std::min(count - done, chunks * spi);
        DRenderParams P = device_params(p, begin + done, spi, chunks);
        long long n_items = pixels_padded * chunks;
        unsigned blocks = (unsigned)((n_items + 127) / 128);
        render_items_kernel<<<blocks, 128, 0, stream>>>(s->view, cam, P, n_items, samples, d_accum, s->d_rays);
        CU_TRY(cudaGetLastError());
        *launches += 1;
        done += samples;
        if (cb) {
            CU_TRY(cudaStreamSynchronize(stream));
            cb(done, count, user);
        }
    }
    return RT_OK;
}
}  // namespace rtb

namespace {

// AUTO resolves to the pipeline measured fastest on B200 for this scene class (see DESIGN.md "Pipelines")
int pick_pipeline(const RtScene* s, const RtParams* p) {
    if (p->pipeline != RT_PIPELINE_AUTO) return p->pipeline;
    return persist_supports(s, p) ? RT_PIPELINE_PERSISTENT : RT_PIPELINE_MEGAKERNEL;  // measured fastest on C1-C4 (DESIGN.md section 5)
}

int run_pipeline(RtScene* s, const DCamera& cam, const RtParams* p, int begin, int count, AccumFx* d_accum, cudaStream_t stream, RtProgressFn cb,
                 void* user, int* launches, int* used) {
    *used = pick_pipeline(s, p);
    if (*used == RT_PIPELINE_WAVEFRONT) return launch_wavefront(s, cam, p, begin, count, d_accum, stream, cb, user, launches);
    if (*used == RT_PIPELINE_WAVEFRONT_SMEM)
        return set_error(RT_ERR_UNSUPPORTED, "RT_PIPELINE_WAVEFRONT_SMEM was a rejected experiment (tools/experiments/rt_warpfront.cu); the library no longer carries it");
    if (*used == RT_PIPELINE_PERSISTENT) return launch_persist(s, cam, p, begin, count, d_accum, stream, cb, user, launches);
    return launch_megakernel(s, cam, p, begin, count, d_accum, stream, cb, user, launches);
}

}  // namespace

// samples [begin, begin + count) of every pixel ADDED into the fixed-point buffer d_accum (device memory of scene's device)
int rtb::accumulate_fixed(const RtScene* scene, const RtCamera* cam, const RtParams* params, AccumFx* d_accum, cudaStream_t stream, RtProgressFn cb,
                            void* user, RtStats* stats, bool sync_for_stats) {
    int begin = params->sample_begin;
    int count = params->sample_count > 0 ? params->sample_count : params->samples_per_pixel - begin;
    if (count <= 0) return set_error(RT_ERR_INVALID, "render: empty sample range");
    DCamera dc;
    make_camera(*cam, dc);
    int launches = 0;
    if (stats) {
        CU_TRY(cudaMemsetAsync(scene->d_rays, 0, sizeof(unsigned long long), stream));
        CU_TRY(cudaEventRecord(scene->ev0, stream));
    }
    int used = 0;
    int rc = run_pipeline(const_cast<RtScene*>(scene), dc, params, begin, count, d_accum, stream, cb, user, &launches, &used);
    if (rc != RT_OK) return rc;
    if (stats) {
        std::memset(stats, 0, sizeof *stats);
        stats->paths = (uint64_t)params->width * params->height * count;
        stats->kernel_launches = launches;
        stats->pipeline_used = used;
        stats->bvh_layout_used = used == RT_PIPELINE_PERSISTENT ? persist_layout_used(scene, params) : 2;
        if (sync_for_stats) {
            CU_TRY(cudaEventRecord(scene->ev1, stream));
            CU_TRY(cudaEventSynchronize(scene->ev1));
            float ms = 0;
            CU_TRY(cudaEventElapsedTime(&ms, scene->ev0, scene->ev1));
            unsigned long long rays = 0;
            CU_TRY(cudaMemcpy(&rays, scene->d_rays, sizeof rays, cudaMemcpyDeviceToHost));
            stats->rays = rays;
            stats->device_ms = ms;
        }
    }
    return RT_OK;
}

static int ensure_scratch(RtScene* scene, size_t n_values) {
    if (scene->scratch_values >= n_values) return RT_OK;
    rtb::cache_free(scene->d_accum, scene->scratch_values * sizeof(AccumFx));
    rtb::cache_free(scene->d_accum_f, scene->scratch_values * sizeof(float));
    rtb::cache_free(scene->d_rgb, scene->scratch_values * sizeof(int32_t));
    scene->d_accum = nullptr, scene->d_accum_f = nullptr, scene->d_rgb = nullptr, scene->scratch_values = 0;
    CU_TRY(rtb::cache_malloc((void**)&scene->d_accum, n_values * sizeof(AccumFx)));
    CU_TRY(rtb::cache_malloc((void**)&scene->d_accum_f, n_values * sizeof(float)));
    CU_TRY(rtb::cache_malloc((void**)&scene->d_rgb, n_values * sizeof(int32_t)));
    scene->scratch_values = n_values;
    return RT_OK;
}
int rtb::scene_scratch(RtScene* scene, size_t n_values) { return ensure_scratch(scene, n_values); }

static int tonemap_args(const void* a, const void* b, int32_t n_pixels, int32_t spp, int* device) {
    if (!a || !b || n_pixels <= 0 || spp <= 0) return set_error(RT_ERR_INVALID, "rt_tonemap: bad argument");
    int rc = have_device();
    if (rc != RT_OK) return rc;
    if (*device < 0) cudaGetDevice(device);
    return RT_OK;
}

// Renderer::render's logger(j, H) is called once per row (raytrace.rs:182).  The pipelines report (samples done, samples
// total); this adapter turns that into one call per row index, in increasing j, on the calling thread.
void rtb::row_progress(int done, int total, void* user) {
    rtb::RowProgress* r = (rtb::RowProgress*)user;
    if (!r->cb) return;
    int upto = total > 0 ? (int)((long long)r->rows * done / total) : r->rows;
    while (r->reported < upto && r->reported < r->rows) r->cb(r->reported++, r->rows, r->user);
}

// ============================================================================ extern "C"

extern "C" {

int rt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int rt_scene_create(const RtSceneDesc* desc, int device, RtScene** out) {
    if (!desc || !out) return set_error(RT_ERR_INVALID, "rt_scene_create: null argument");
    *out = nullptr;
    int rc = have_device();
    if (rc != RT_OK) return rc;
    if (device >= rt_device_count()) return set_error(RT_ERR_INVALID, "rt_scene_create: device %d does not exist", device);
    return create_scene(desc, desc->root, true, device, true, out);
}

void rt_scene_destroy(RtScene* scene) { free_scene(scene); }

int rt_scene_info(const RtScene* scene, int32_t* n_prims, int32_t* n_bvh_nodes, int32_t* n_media, int64_t* device_bytes) {
    if (!scene) return set_error(RT_ERR_INVALID, "rt_scene_info: null scene");
    if (n_prims) *n_prims = (int32_t)scene->flat.prims.size();
    if (n_bvh_nodes) *n_bvh_nodes = (int32_t)scene->flat.nodes.size();
    if (n_media) *n_media = (int32_t)scene->flat.media.size();
    if (device_bytes) *device_bytes = scene->device_bytes;
    return RT_OK;
}

int rt_scene_build_info(const RtScene* scene, int32_t* built_on_device, float* build_ms, int32_t* depth) {
    if (!scene) return set_error(RT_ERR_INVALID, "rt_scene_build_info: null scene");
    if (built_on_device) *built_on_device = scene->flat.built_on_device ? 1 : 0;
    if (build_ms) *build_ms = scene->flat.device_build_ms;
    if (depth) *depth = scene->flat.bvh_depth;
    return RT_OK;
}

int rt_render_accumulate_fixed_device(const RtScene* scene, const RtCamera* cam, const RtParams* params, uint64_t* d_accum_fixed, void* stream_,
                                      RtStats* stats) {
    int rc = validate_render(scene, cam, params);
    if (rc != RT_OK) return rc;
    if (!d_accum_fixed) return set_error(RT_ERR_INVALID, "rt_render_accumulate_fixed_device: null accumulation buffer");
    DeviceGuard g(scene->device);
    return rtb::accumulate_fixed(scene, cam, params, (AccumFx*)d_accum_fixed, (cudaStream_t)stream_, nullptr, nullptr, stats, true);
}

int rt_render_accumulate_device(const RtScene* scene_, const RtCamera* cam, const RtParams* params, float* d_accum_rgb, void* stream_, RtStats* stats) {
    int rc = validate_render(scene_, cam, params);
    if (rc != RT_OK) return rc;
    if (!d_accum_rgb) return set_error(RT_ERR_INVALID, "rt_render_accumulate_device: null accumulation buffer");
    RtScene* scene = const_cast<RtScene*>(scene_);
    cudaStream_t stream = (cudaStream_t)stream_;
    DeviceGuard g(scene->device);
    // the pipelines sum in fixed point (scene scratch); the caller's float buffer receives the converted sums
    const size_t n_values = (size_t)3 * params->width * params->height;
    if ((rc = ensure_scratch(scene, n_values)) != RT_OK) return rc;
    CU_TRY(cudaMemsetAsync(scene->d_accum, 0, n_values * sizeof(AccumFx), stream));
    rc = rtb::accumulate_fixed(scene, cam, params, scene->d_accum, stream, nullptr, nullptr, stats, false);
    if (rc != RT_OK) return rc;
    fixed_to_float_kernel<<<(unsigned)((n_values + 255) / 256), 256, 0, stream>>>(scene->d_accum, d_accum_rgb, (long long)n_values, 1);
    CU_TRY(cudaGetLastError());
    if (stats) {
        stats->kernel_launches += 1;
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

int rt_tonemap_device(const float* d_accum_rgb, int32_t* d_rgb, int32_t n_pixels, int32_t samples_per_pixel, int device, void* stream_) {
    int rc = tonemap_args(d_accum_rgb, d_rgb, n_pixels, samples_per_pixel, &device);
    if (rc != RT_OK) return rc;
    DeviceGuard g(device);
    int n = 3 * n_pixels;
    tonemap_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream_>>>(d_accum_rgb, d_rgb, n, 1.0 / (double)samples_per_pixel);
    CU_TRY(cudaGetLastError());
    return RT_OK;
}

int rt_tonemap_fixed_device(const uint64_t* d_accum_fixed, int32_t* d_rgb, int32_t n_pixels, int32_t samples_per_pixel, int device, void* stream_) {
    int rc = tonemap_args(d_accum_fixed, d_rgb, n_pixels, samples_per_pixel, &device);
    if (rc != RT_OK) return rc;
    DeviceGuard g(device);
    int n = 3 * n_pixels;
    tonemap_fixed_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream_>>>((const AccumFx*)d_accum_fixed, d_rgb, n,
                                                                             1.0 / (RT_ACCUM_FIXED_ONE * (double)samples_per_pixel));
    CU_TRY(cudaGetLastError());
    return RT_OK;
}

int rt_accum_fixed_to_float_device(const uint64_t* d_accum_fixed, float* d_accum_rgb, int64_t n_values, int device, void* stream_) {
    if (!d_accum_fixed || !d_accum_rgb || n_values <= 0) return set_error(RT_ERR_INVALID, "rt_accum_fixed_to_float_device: bad argument");
    int rc = have_device();
    if (rc != RT_OK) return rc;
    if (device < 0) cudaGetDevice(&device);
    DeviceGuard g(device);
    fixed_to_float_kernel<<<(unsigned)((n_values + 255) / 256), 256, 0, (cudaStream_t)stream_>>>((const AccumFx*)d_accum_fixed, d_accum_rgb, (long long)n_values, 0);
    CU_TRY(cudaGetLastError());
    return RT_OK;
}

void rt_release_cached_memory(void) { rtb::cache_release_all(); }

int rt_render(const RtScene* scene_, const RtCamera* cam, const RtParams* params, float* accum_rgb, int32_t* rgb, RtProgressFn cb, void* user,
              RtStats* stats) {
    int rc = validate_render(scene_, cam, params);
    if (rc != RT_OK) return rc;
    RtScene* scene = const_cast<RtScene*>(scene_);  // scratch buffers are cached in the scene object
    DeviceGuard g(scene->device);
    size_t n_values = (size_t)3 * params->width * params->height;
    if ((rc = ensure_scratch(scene, n_values)) != RT_OK) return rc;
    cudaStream_t stream = 0;
    rtb::RowProgress rows{cb, user, params->height, 0};
    RtStats local;
    CU_TRY(cudaMemsetAsync(scene->d_rays, 0, sizeof(unsigned long long), stream));
    CU_TRY(cudaEventRecord(scene->ev0, stream));
    CU_TRY(cudaMemsetAsync(scene->d_accum, 0, n_values * sizeof(AccumFx), stream));
    {
        // stats are finalised below, after the tonemap: the timed region is render + tonemap
        int begin = params->sample_begin;
        int count = params->sample_count > 0 ? params->sample_count : params->samples_per_pixel - begin;
        if (count <= 0) return set_error(RT_ERR_INVALID, "render: empty sample range");
        DCamera dc;
        make_camera(*cam, dc);
        int launches = 0, used = 0;
        rc = run_pipeline(scene, dc, params, begin, count, scene->d_accum, stream, cb ? rtb::row_progress : nullptr, &rows, &launches, &used);
        if (rc != RT_OK) return rc;
        std::memset(&local, 0, sizeof local);
        local.paths = (uint64_t)params->width * params->height * count;
        local.kernel_launches = launches, local.pipeline_used = used;
        local.bvh_layout_used = used == RT_PIPELINE_PERSISTENT ? persist_layout_used(scene, params) : 2;
    }
    tonemap_fixed_kernel<<<(unsigned)((n_values + 255) / 256), 256, 0, stream>>>(scene->d_accum, scene->d_rgb, (int)n_values,
                                                                                1.0 / (RT_ACCUM_FIXED_ONE * (double)params->samples_per_pixel));
    CU_TRY(cudaGetLastError());
    local.kernel_launches += 1;
    CU_TRY(cudaEventRecord(scene->ev1, stream));
    if (accum_rgb) {
        fixed_to_float_kernel<<<(unsigned)((n_values + 255) / 256), 256, 0, stream>>>(scene->d_accum, scene->d_accum_f, (long long)n_values, 0);
        CU_TRY(cudaGetLastError());
        CU_TRY(cudaMemcpyAsync(accum_rgb, scene->d_accum_f, n_values * sizeof(float), cudaMemcpyDeviceToHost, stream));
    }
    if (rgb) CU_TRY(cudaMemcpyAsync(rgb, scene->d_rgb, n_values * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    CU_TRY(cudaStreamSynchronize(stream));
    rtb::row_progress(1, 1, &rows);  // whatever rows the pipeline's own reports did not cover
    if (stats) {
        float ms = 0;
        CU_TRY(cudaEventElapsedTime(&ms, scene->ev0, scene->ev1));
        unsigned long long rays = 0;
        CU_TRY(cudaMemcpy(&rays, scene->d_rays, sizeof rays, cudaMemcpyDeviceToHost));
        local.rays = rays, local.device_ms = ms;
        *stats = local;
    }
    return RT_OK;
}

int rt_intersect_batch(const RtScene* scene, int32_t node, const float* rays, int64_t n, RtHit* out) {
    return rt_intersect_batch_at(scene, node, 0.0f, rays, n, out);
}

int rt_intersect_batch_at(const RtScene* scene, int32_t node, float time, const float* rays, int64_t n, RtHit* out) {
    if (!scene || !rays || !out || n < 0) return set_error(RT_ERR_INVALID, "rt_intersect_batch: bad argument");
    if (n == 0) return RT_OK;
    DeviceGuard g(scene->device);
    const RtScene* target = scene;
    RtScene* sub = nullptr;
    int mode = node == -2 ? QUERY_BVH4 : QUERY_BVH;  // -2: the whole world through the 4-wide tree (binary tree if the scene has none)
    if (node >= 0 && scene->desc && node != scene->desc->d.root) {
        // a sub-tree: flatten it on its own (no outer transforms) and test it by brute force
        if (node >= scene->desc->d.n_nodes) return set_error(RT_ERR_INVALID, "rt_intersect_batch: node %d out of range", node);
        int rc = create_scene(&scene->desc->d, node, false, scene->device, false, &sub);
        if (rc != RT_OK) return rc;
        target = sub;
        mode = scene->desc->d.nodes[node].kind == RT_NODE_MEDIUM ? QUERY_MEDIUM : QUERY_LINEAR;
    } else if (node >= 0 && scene->desc && scene->desc->d.nodes[node].kind == RT_NODE_MEDIUM) {
        mode = QUERY_MEDIUM;  // the root itself is a medium: its clipped boundary interval, as documented in the header
    }
    float* d_rays = nullptr;
    RtHit* d_out = nullptr;
    int rc = RT_OK;
    do {
        if (cudaMalloc(&d_rays, (size_t)n * 8 * sizeof(float)) != cudaSuccess || cudaMalloc(&d_out, (size_t)n * sizeof(RtHit)) != cudaSuccess) {
            rc = set_error(RT_ERR_CUDA, "rt_intersect_batch: cudaMalloc failed");
            break;
        }
        if (cudaMemcpy(d_rays, rays, (size_t)n * 8 * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) {
            rc = set_error(RT_ERR_CUDA, "rt_intersect_batch: upload failed");
            break;
        }
        intersect_kernel<<<(unsigned)((n + 127) / 128), 128>>>(target->view, mode, d_rays, n, d_out, time);
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) {
            rc = set_error(RT_ERR_CUDA, "rt_intersect_batch: kernel failed: %s", cudaGetErrorString(e));
            break;
        }
        if (cudaMemcpy(out, d_out, (size_t)n * sizeof(RtHit), cudaMemcpyDeviceToHost) != cudaSuccess) {
            rc = set_error(RT_ERR_CUDA, "rt_intersect_batch: download failed");
            break;
        }
        // report description node ids instead of device primitive indices
        for (int64_t i = 0; i < n; ++i)
            if (out[i].prim >= 0) out[i].prim = target->flat.prim_node[out[i].prim];
    } while (0);
    cudaFree(d_rays);
    cudaFree(d_out);
    if (sub) free_scene(sub);
    return rc;
}

int rt_texture_value_batch(const RtScene* scene, int32_t texture, const float* uvp, int64_t n, float* out_rgb) {
    if (!scene || !uvp || !out_rgb || n < 0) return set_error(RT_ERR_INVALID, "rt_texture_value_batch: bad argument");
    if (texture < 0 || texture >= (int)scene->flat.texs.size()) return set_error(RT_ERR_INVALID, "rt_texture_value_batch: texture %d out of range", texture);
    if (n == 0) return RT_OK;
    DeviceGuard g(scene->device);
    float *d_in = nullptr, *d_out = nullptr;
    int rc = RT_OK;
    do {
        if (cudaMalloc(&d_in, (size_t)n * 5 * sizeof(float)) != cudaSuccess || cudaMalloc(&d_out, (size_t)n * 3 * sizeof(float)) != cudaSuccess) {
            rc = set_error(RT_ERR_CUDA, "rt_texture_value_batch: cudaMalloc failed");
            break;
        }
        cudaMemcpy(d_in, uvp, (size_t)n * 5 * sizeof(float), cudaMemcpyHostToDevice);
        texture_kernel<<<(unsigned)((n + 127) / 128), 128>>>(scene->view, texture, d_in, n, d_out);
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) {
            rc = set_error(RT_ERR_CUDA, "rt_texture_value_batch: kernel failed: %s", cudaGetErrorString(e));
            break;
        }
        cudaMemcpy(out_rgb, d_out, (size_t)n * 3 * sizeof(float), cudaMemcpyDeviceToHost);
    } while (0);
    cudaFree(d_in);
    cudaFree(d_out);
    return rc;
}

int rt_scatter_batch(const RtScene* scene, const RtScatterIn* in, int64_t n, RtScatterOut* out) {
    if (!scene || !in || !out || n < 0) return set_error(RT_ERR_INVALID, "rt_scatter_batch: bad argument");
    if (n == 0) return RT_OK;
    const int n_mats = (int)scene->flat.mats.size();
    for (int64_t i = 0; i < n; ++i)
        if (in[i].material < 0 || in[i].material >= n_mats) return set_error(RT_ERR_INVALID, "rt_scatter_batch: material %d out of range", in[i].material);
    DeviceGuard g(scene->device);
    RtScatterIn* d_in = nullptr;
    RtScatterOut* d_out = nullptr;
    int rc = RT_OK;
    do {
        if (cudaMalloc(&d_in, (size_t)n * sizeof(RtScatterIn)) != cudaSuccess || cudaMalloc(&d_out, (size_t)n * sizeof(RtScatterOut)) != cudaSuccess) {
            rc = set_error(RT_ERR_CUDA, "rt_scatter_batch: cudaMalloc failed");
            break;
        }
        cudaMemcpy(d_in, in, (size_t)n * sizeof(RtScatterIn), cudaMemcpyHostToDevice);
        scatter_kernel<<<(unsigned)((n + 127) / 128), 128>>>(scene->view, d_in, n, d_out);
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) {
            rc = set_error(RT_ERR_CUDA, "rt_scatter_batch: kernel failed: %s", cudaGetErrorString(e));
            break;
        }
        cudaMemcpy(out, d_out, (size_t)n * sizeof(RtScatterOut), cudaMemcpyDeviceToHost);
    } while (0);
    cudaFree(d_in);
    cudaFree(d_out);
    return rc;
}

int rt_generate_rays(const RtCamera* cam, const RtParams* params, const int32_t* pixel, const int32_t* sample, int64_t n, float* out_rays,
                     float* out_sample) {
    if (!cam || !params || !pixel || !sample || !out_rays || !out_sample || n < 0) return set_error(RT_ERR_INVALID, "rt_generate_rays: bad argument");
    if (params->width < 2 || params->height < 2) return set_error(RT_ERR_INVALID, "rt_generate_rays: image must be at least 2x2");
    int rc = have_device();
    if (rc != RT_OK) return rc;
    if (n == 0) return RT_OK;
    DCamera dc;
    make_camera(*cam, dc);
    DRenderParams P = device_params(params, 0, 1, 1);
    int32_t *d_px = nullptr, *d_s = nullptr;
    float *d_r = nullptr, *d_u = nullptr;
    do {
        if (cudaMalloc(&d_px, (size_t)n * 4) != cudaSuccess || cudaMalloc(&d_s, (size_t)n * 4) != cudaSuccess ||
            cudaMalloc(&d_r, (size_t)n * 24) != cudaSuccess || cudaMalloc(&d_u, (size_t)n * 16) != cudaSuccess) {
            rc = set_error(RT_ERR_CUDA, "rt_generate_rays: cudaMalloc failed");
            break;
        }
        cudaMemcpy(d_px, pixel, (size_t)n * 4, cudaMemcpyHostToDevice);
        cudaMemcpy(d_s, sample, (size_t)n * 4, cudaMemcpyHostToDevice);
        camera_kernel<<<(unsigned)((n + 127) / 128), 128>>>(dc, P, d_px, d_s, n, d_r, d_u);
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) {
            rc = set_error(RT_ERR_CUDA, "rt_generate_rays: kernel failed: %s", cudaGetErrorString(e));
            break;
        }
        cudaMemcpy(out_rays, d_r, (size_t)n * 24, cudaMemcpyDeviceToHost);
        cudaMemcpy(out_sample, d_u, (size_t)n * 16, cudaMemcpyDeviceToHost);
    } while (0);
    cudaFree(d_px), cudaFree(d_s), cudaFree(d_r), cudaFree(d_u);
    return rc;
}

}  // extern "C"
