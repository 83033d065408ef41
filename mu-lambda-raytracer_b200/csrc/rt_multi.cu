// rt_render_multi: the render loop sharded over several GPUs of ONE process (SURVEY §8e).
//
// The reference parallelises Renderer::render over image rows with rayon on one host (src/raytrace.rs:176-185).
// Here every (pixel, sample) path is independent and owns a Philox counter, so device g of G renders ALL pixels
// for the g-th contiguous slice of the sample range; the G fixed-point accumulation buffers (64-bit integers, so the sum
// is exact and the image identical to the one-GPU render) are summed onto the root device with ONE ncclReduce over
// NVLink and the root tonemaps (to_rgb, raytrace.rs:59-68).  No other exchange exists on this path.  (Under
// torch.distributed — one process per GPU — the same slicing is done by mu_lambda_raytracer_b200/distributed.py with
// rt_render_accumulate_fixed_device + dist.reduce.)
//
// NCCL is bound at run time (dlopen of libnccl.so.2): the library has no link-time dependency on it, and inside a
// process that already loaded a libnccl (PyTorch) the same copy is reused.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "scene_internal.h"

namespace {

// the handful of NCCL entry points used, declared locally so that no nccl.h is needed at build time
typedef struct ncclComm* ncclComm_t;
typedef int ncclResult_t;  // 0 = ncclSuccess
enum { kNcclUint64 = 5, kNcclFloat = 7, kNcclSum = 0 };  // ncclDataType_t / ncclRedOp_t values of nccl.h

struct Nccl {
    void* so = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    ncclResult_t (*Reduce)(const void*, void*, size_t, int, int, int, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    std::string error;
};

Nccl& nccl() {
    static Nccl n;
    static std::once_flag once;
    std::call_once(once, [] {
        for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
            n.so = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (n.so) break;
        }
        if (!n.so) {
            n.error = std::string("cannot load libnccl.so.2: ") + (dlerror() ? dlerror() : "not found");
            return;
        }
        auto sym = [&](const char* s) {
            void* p = dlsym(n.so, s);
            if (!p && n.error.empty()) n.error = std::string("libnccl lacks ") + s;
            return p;
        };
        n.CommInitAll = (decltype(n.CommInitAll))sym("ncclCommInitAll");
        n.CommDestroy = (decltype(n.CommDestroy))sym("ncclCommDestroy");
        n.GroupStart = (decltype(n.GroupStart))sym("ncclGroupStart");
        n.GroupEnd = (decltype(n.GroupEnd))sym("ncclGroupEnd");
        n.Reduce = (decltype(n.Reduce))sym("ncclReduce");
        n.GetErrorString = (decltype(n.GetErrorString))sym("ncclGetErrorString");
    });
    return n;
}

// communicators are cached per device list (creating them costs ~100 ms)
struct CommSet {
    std::vector<int> devices;
    std::vector<ncclComm_t> comms;
};
std::mutex g_comm_mutex;
std::vector<CommSet> g_comm_sets;

int get_comms(const std::vector<int>& devices, std::vector<ncclComm_t>& out) {
    std::lock_guard<std::mutex> lock(g_comm_mutex);
    rtb::DeviceGuard restore(devices[0]);  // the caller's current device comes back on every exit
    for (auto& cs : g_comm_sets)
        if (cs.devices == devices) {
            out = cs.comms;
            return RT_OK;
        }
    Nccl& n = nccl();
    if (!n.error.empty()) return rtb::set_error(RT_ERR_UNSUPPORTED, "rt_render_multi: %s", n.error.c_str());
    CommSet cs;
    cs.devices = devices;
    cs.comms.resize(devices.size());
    ncclResult_t r = n.CommInitAll(cs.comms.data(), (int)devices.size(), devices.data());
    if (r != 0) return rtb::set_error(RT_ERR_CUDA, "ncclCommInitAll failed: %s", n.GetErrorString(r));
    // NCCL connects its NVLink transports lazily inside the first collective (hundreds of ms): do that here, once,
    // as part of communicator set-up rather than inside the first render's timed region
    std::vector<float*> warm(devices.size(), nullptr);
    for (size_t g = 0; g < devices.size(); ++g) {
        cudaSetDevice(devices[g]);
        CU_TRY(cudaMalloc(&warm[g], 256 * sizeof(float)));
        CU_TRY(cudaMemset(warm[g], 0, 256 * sizeof(float)));
    }
    r = n.GroupStart();
    for (size_t g = 0; g < devices.size() && r == 0; ++g) {
        cudaSetDevice(devices[g]);
        r = n.Reduce(warm[g], warm[g], 256, kNcclFloat, kNcclSum, 0, cs.comms[g], 0);
    }
    ncclResult_t r2 = n.GroupEnd();
    for (size_t g = 0; g < devices.size(); ++g) {
        cudaSetDevice(devices[g]);
        cudaStreamSynchronize(0);
        cudaFree(warm[g]);
    }
    if (r != 0 || r2 != 0) return rtb::set_error(RT_ERR_CUDA, "ncclReduce (warm-up) failed: %s", n.GetErrorString(r != 0 ? r : r2));
    g_comm_sets.push_back(cs);
    out = cs.comms;
    return RT_OK;
}

}  // namespace

extern "C" {

void rt_sample_slice(int32_t sample_begin, int32_t sample_count, int32_t n_parts, int32_t part, int32_t* begin, int32_t* count) {
    if (n_parts < 1) n_parts = 1;
    if (part < 0) part = 0;
    if (part >= n_parts) part = n_parts - 1;
    int32_t base = sample_count / n_parts, extra = sample_count % n_parts;
    if (count) *count = base + (part < extra ? 1 : 0);
    if (begin) *begin = sample_begin + part * base + std::min(part, extra);
}

int rt_render_multi(RtScene* const* scenes, int32_t n_scenes, const RtCamera* cam, const RtParams* params, float* accum_rgb, int32_t* rgb,
                    RtProgressFn cb, void* user, RtStats* stats) {
    if (!scenes || n_scenes < 1 || !cam || !params) return rtb::set_error(RT_ERR_INVALID, "rt_render_multi: bad argument");
    for (int g = 0; g < n_scenes; ++g)
        if (!scenes[g]) return rtb::set_error(RT_ERR_INVALID, "rt_render_multi: scene %d is null", g);
    if (n_scenes == 1) return rt_render(scenes[0], cam, params, accum_rgb, rgb, cb, user, stats);
    std::vector<int> devices;
    for (int g = 0; g < n_scenes; ++g) {
        if (std::find(devices.begin(), devices.end(), scenes[g]->device) != devices.end())
            return rtb::set_error(RT_ERR_INVALID, "rt_render_multi: two scenes live on device %d", scenes[g]->device);
        devices.push_back(scenes[g]->device);
    }
    if (params->width < 2 || params->height < 2 || params->samples_per_pixel <= 0 || params->sample_begin < 0 || params->sample_count < 0)
        return rtb::set_error(RT_ERR_INVALID, "rt_render_multi: bad image size or sample range");
    if ((long long)params->sample_begin + params->sample_count > RT_MAX_SAMPLE_END)
        return rtb::set_error(RT_ERR_INVALID, "rt_render_multi: sample range ends beyond 2^31 - 1");
    int begin = params->sample_begin;
    int count = params->sample_count > 0 ? params->sample_count : params->samples_per_pixel - begin;
    if (count <= 0) return rtb::set_error(RT_ERR_INVALID, "render: empty sample range");
    rtb::DeviceGuard caller(devices[0]);  // whatever device the calling thread had current comes back on every exit
    std::vector<ncclComm_t> comms;
    int rc = get_comms(devices, comms);
    if (rc != RT_OK) return rc;

    const size_t n_values = (size_t)3 * params->width * params->height;
    // per-device accumulation buffers (the scene's scratch, grown on demand)
    for (int g = 0; g < n_scenes; ++g) {
        rtb::DeviceGuard guard(scenes[g]->device);
        if ((rc = rtb::scene_scratch(scenes[g], n_values)) != RT_OK) return rc;
    }
    RtScene* root = scenes[0];
    struct Events {  // destroyed on every exit
        cudaEvent_t t0 = nullptr, t1 = nullptr;
        ~Events() {
            if (t0) cudaEventDestroy(t0);
            if (t1) cudaEventDestroy(t1);
        }
    } ev;
    cudaEvent_t& t0 = ev.t0;
    cudaEvent_t& t1 = ev.t1;
    {
        rtb::DeviceGuard guard(root->device);
        CU_TRY(cudaEventCreate(&t0));
        CU_TRY(cudaEventCreate(&t1));
        CU_TRY(cudaEventRecord(t0, 0));
    }
    // one host thread per device: zero, render the slice.  The root's slice runs on the calling thread, which is the
    // only one allowed to invoke the logger: its progress paces the per-row reports (every device has the same work).
    std::vector<int> codes(n_scenes, RT_OK);
    std::vector<std::string> messages(n_scenes);
    std::vector<RtStats> part(n_scenes);
    std::vector<std::thread> threads;
    rtb::RowProgress rows{cb, user, params->height, 0};
    auto render_slice = [&](int g) {
        RtScene* s = scenes[g];
        cudaSetDevice(s->device);
        RtParams p = *params;
        rt_sample_slice(begin, count, n_scenes, g, &p.sample_begin, &p.sample_count);
        std::memset(&part[g], 0, sizeof(RtStats));
        cudaError_t e = cudaMemsetAsync(s->d_accum, 0, n_values * sizeof(rtb::AccumFx), 0);
        if (e != cudaSuccess) {
            codes[g] = RT_ERR_CUDA, messages[g] = cudaGetErrorString(e);
            return;
        }
        if (p.sample_count > 0) {
            codes[g] = rtb::accumulate_fixed(s, cam, &p, s->d_accum, 0, (g == 0 && cb) ? rtb::row_progress : nullptr, &rows, &part[g], true);
            if (codes[g] != RT_OK) messages[g] = rt_last_error();
        }
    };
    for (int g = 1; g < n_scenes; ++g) threads.emplace_back(render_slice, g);
    render_slice(0);
    for (auto& t : threads) t.join();
    for (int g = 0; g < n_scenes; ++g)
        if (codes[g] != RT_OK) return rtb::set_error(codes[g], "device %d: %s", devices[g], messages[g].c_str());
    // the one exchange step of the path: sum the accumulation buffers onto the root
    Nccl& n = nccl();
    ncclResult_t r = n.GroupStart();
    for (int g = 0; g < n_scenes && r == 0; ++g) {
        cudaSetDevice(devices[g]);
        r = n.Reduce(scenes[g]->d_accum, scenes[g]->d_accum, n_values, kNcclUint64, kNcclSum, 0, comms[g], 0);
    }
    ncclResult_t r2 = n.GroupEnd();
    if (r == 0) r = r2;
    if (r != 0) return rtb::set_error(RT_ERR_CUDA, "ncclReduce failed: %s", n.GetErrorString(r));
    for (int g = 1; g < n_scenes; ++g) {
        cudaSetDevice(devices[g]);
        CU_TRY(cudaStreamSynchronize(0));
    }
    rtb::DeviceGuard guard(root->device);
    rc = rt_tonemap_fixed_device((const uint64_t*)root->d_accum, root->d_rgb, params->width * params->height, params->samples_per_pixel, root->device, nullptr);
    if (rc != RT_OK) return rc;
    CU_TRY(cudaEventRecord(t1, 0));
    if (accum_rgb) {
        if ((rc = rt_accum_fixed_to_float_device((const uint64_t*)root->d_accum, root->d_accum_f, (int64_t)n_values, root->device, nullptr)) != RT_OK) return rc;
        CU_TRY(cudaMemcpyAsync(accum_rgb, root->d_accum_f, n_values * sizeof(float), cudaMemcpyDeviceToHost, 0));
    }
    if (rgb) CU_TRY(cudaMemcpyAsync(rgb, root->d_rgb, n_values * sizeof(int32_t), cudaMemcpyDeviceToHost, 0));
    CU_TRY(cudaStreamSynchronize(0));
    rtb::row_progress(1, 1, &rows);  // the rows the root's own progress reports did not cover
    if (stats) {
        float ms = 0;
        CU_TRY(cudaEventElapsedTime(&ms, t0, t1));
        std::memset(stats, 0, sizeof *stats);
        for (int g = 0; g < n_scenes; ++g) stats->paths += part[g].paths, stats->rays += part[g].rays, stats->kernel_launches += part[g].kernel_launches;
        stats->kernel_launches += 1;
        stats->device_ms = ms;  // root-device events around render + reduce + tonemap (every other device finishes before the reduce does)
        stats->pipeline_used = part[0].pipeline_used, stats->bvh_layout_used = part[0].bvh_layout_used;
    }
    return RT_OK;
}

}  // extern "C"
