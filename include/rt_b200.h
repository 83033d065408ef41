/*
 * rt_b200.h — C ABI of the B200-native path-tracing hot path.
 *
 * This is the drop-in boundary for the reference's render loop.  The reference
 * (mu-lambda/mu-lambda-raytracer, Rust) has no FFI; the seam this library
 * replaces is
 *
 *     Renderer::new_with_rng(camera, world, background, params, tracer, rng)
 *     Renderer::render(logger) -> Vec<Vec<RGB>>            src/raytrace.rs:151-186
 *
 * called from exactly one place, do_tracing (src/main.rs:147-157).  Because the
 * reference's world is an opaque Box<dyn Hittable> (src/worlds.rs:18,
 * src/hittable.rs:33-35), the host hands the library a *scene description*
 * (RtSceneDesc): the reference's object tree written down node for node in
 * construction order, all values f64 exactly as the Rust code holds them.
 *
 * Conventions: plain-old-data structs, caller-owned memory, `int` status
 * returns (0 = RT_OK), rt_last_error() for the message, no exceptions and no
 * callbacks from device threads.  There is NO CPU fallback: every compute
 * entry point returns RT_ERR_NO_DEVICE when no CUDA device is usable.
 */
#ifndef RT_B200_H
#define RT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_B200_ABI_VERSION 3

/* ---- status codes (replace the reference's unwrap()/panic!(), SURVEY §5) ---- */
enum {
    RT_OK = 0,
    RT_ERR_INVALID = 1,    /* bad argument / malformed description */
    RT_ERR_NO_DEVICE = 2,  /* no usable CUDA device: there is no CPU path */
    RT_ERR_CUDA = 3,       /* a CUDA call failed; see rt_last_error() */
    RT_ERR_UNSUPPORTED = 4 /* description uses a construct the device path cannot flatten */
};

/* ---- scene description: mirrors the reference's trait-object tree ---- */

/* node kinds: one per Hittable impl of the reference */
enum {
    RT_NODE_SPHERE = 1,    /* shapes.rs:26-82      f = cx,cy,cz,radius (radius may be negative) */
    RT_NODE_XYRECT = 2,    /* shapes.rs:92-108     f = x0,x1,y0,y1,z */
    RT_NODE_XZRECT = 3,    /* shapes.rs:117-133    f = x0,x1,z0,z1,y */
    RT_NODE_YZRECT = 4,    /* shapes.rs:142-158    f = y0,y1,z0,z1,x */
    RT_NODE_BLOCK = 5,     /* shapes.rs:166-198    f = p0x,p0y,p0z,p1x,p1y,p1z */
    RT_NODE_TRANSLATE = 6, /* transforms.rs:20-42  f = ox,oy,oz; child = wrapped node */
    RT_NODE_ROTATE = 7,    /* transforms.rs:51-142 axis = 0/1/2, f[0] = angle in degrees; child */
    RT_NODE_MEDIUM = 8,    /* volumes.rs:7-65      f[0] = density d; material = its Isotropic; child = boundary */
    RT_NODE_BVH = 9,       /* bhv.rs:85-101        children[first_child .. +child_count], insertion order */
    RT_NODE_LIST = 10,     /* hittable.rs:37-68    children[first_child .. +child_count], insertion order */
    /* EXTENSION — no counterpart in the reference (src/vec.rs:215-219: its Ray has no time).  The MovingSphere of "Ray
     * Tracing: The Next Week": f = c0x,c0y,c0z, c1x,c1y,c1z, radius; centre(time) = c0 + time * (c1 - c0) for the ray's
     * time in [0, 1] (RtCamera.time0/time1).  Parity is stated against the oracle's restatement of the BOOK. */
    RT_NODE_MOVING_SPHERE = 11
};

typedef struct RtNode {
    int32_t kind;
    int32_t material;    /* index into materials, -1 when the kind has none */
    int32_t first_child; /* TRANSLATE/ROTATE/MEDIUM: child node index; BVH/LIST: offset into children[] */
    int32_t child_count; /* BVH/LIST only */
    int32_t axis;        /* ROTATE only */
    int32_t reserved;
    double f[8];
} RtNode;

enum {
    RT_MAT_LAMBERTIAN = 1,    /* materials.rs:14-34   texture */
    RT_MAT_METAL = 2,         /* materials.rs:36-61   albedo, fuzz */
    RT_MAT_DIELECTRIC = 3,    /* materials.rs:70-106  ior */
    RT_MAT_DIFFUSE_LIGHT = 4, /* materials.rs:108-127 texture */
    RT_MAT_ISOTROPIC = 5      /* volumes.rs:67-83     texture */
};

typedef struct RtMaterial {
    int32_t kind;
    int32_t texture; /* index into textures, -1 when unused */
    double albedo[3];
    double fuzz;
    double ior;
} RtMaterial;

enum {
    RT_TEX_SOLID = 1,   /* textures.rs:8-26     color */
    RT_TEX_CHECKER = 2, /* textures.rs:28-49    odd, even = texture indices */
    RT_TEX_NOISE = 3,   /* textures.rs:151-167  perlin = table index, scale */
    RT_TEX_IMAGE = 4    /* image_texture.rs     image = image index */
};

typedef struct RtTexture {
    int32_t kind;
    int32_t a; /* CHECKER: odd texture; NOISE: perlin table; IMAGE: image */
    int32_t b; /* CHECKER: even texture */
    int32_t reserved;
    double color[3];
    double scale;
} RtTexture;

#define RT_PERLIN_POINTS 1024 /* textures.rs:51 */

typedef struct RtPerlin {
    double ranvec[RT_PERLIN_POINTS][3];
    int32_t perm_x[RT_PERLIN_POINTS];
    int32_t perm_y[RT_PERLIN_POINTS];
    int32_t perm_z[RT_PERLIN_POINTS];
} RtPerlin;

typedef struct RtImage {
    int32_t width, height;
    const uint8_t* rgb; /* width*height*3, row 0 = top of the file, as image::RgbImage */
} RtImage;

enum { RT_BG_BLACK = 0, RT_BG_GRADIENT = 1 }; /* raytrace.rs:12-48 */

typedef struct RtSceneDesc {
    int32_t root; /* node index of what World::build returned */
    int32_t background_kind;
    double background_top[3];    /* GradientBackground.top    (raytrace.rs:13) */
    double background_bottom[3]; /* GradientBackground.bottom (raytrace.rs:14) */
    int32_t n_nodes, n_children, n_materials, n_textures, n_perlins, n_images;
    const RtNode* nodes;
    const int32_t* children;
    const RtMaterial* materials;
    const RtTexture* textures;
    const RtPerlin* perlins;
    const RtImage* images;
} RtSceneDesc;

/* the seven inputs of Camera::new (camera.rs:15-23) */
typedef struct RtCamera {
    double lookfrom[3], lookat[3], vup[3];
    double vfov_deg;
    double aspect_ratio; /* the FLAG ratio, not W/H (main.rs:197) */
    double aperture;
    double focus_dist;
    /* EXTENSION (motion blur; the reference's camera has no shutter): every camera ray — and the whole path after it —
     * gets a time uniform in [time0, time1) within [0, 1], at which moving spheres are evaluated (resolution 2^-13).
     * time0 = time1 = 0 is the reference's behaviour. */
    double time0, time1;
} RtCamera;

/*
 * RT_PIPELINE_WAVEFRONT      generate / extend / shade as separate kernels over a pool of in-flight paths, with
 *                            per-material-class queues and ballot/prefix-sum compaction between the stages
 * RT_PIPELINE_WAVEFRONT_SMEM retired experiment (per-warp pools in shared memory, the slowest of the four in round 1;
 *                            source kept under tools/experiments/); selecting it returns RT_ERR_UNSUPPORTED
 * RT_PIPELINE_MEGAKERNEL     one thread per pixel x run of samples, no queues (the comparator north_star asks for)
 * RT_PIPELINE_PERSISTENT     the wavefront stages inside one resident kernel: two paths per lane (registers + shared
 *                            memory), warp ballots choose between the extend and the shade stage, no global queues
 * RT_PIPELINE_AUTO           the pipeline measured fastest on B200 for the scene
 */
enum { RT_PIPELINE_AUTO = 0, RT_PIPELINE_MEGAKERNEL = 1, RT_PIPELINE_WAVEFRONT = 2, RT_PIPELINE_WAVEFRONT_SMEM = 3 /* retired: RT_ERR_UNSUPPORTED */, RT_PIPELINE_PERSISTENT = 4 };

/* the largest end, sample_begin + sample_count, of a sample range: sample indices are 32-bit signed integers */
#define RT_MAX_SAMPLE_END 2147483647

/* RenderingParams (raytrace.rs:50-55) + max_depth (main.rs:72) + device-side knobs */
typedef struct RtParams {
    int32_t width, height;
    int32_t samples_per_pixel; /* spp of the WHOLE image (used by the tonemap divisor) */
    int32_t max_depth;
    uint64_t seed;             /* key of the Philox render streams */
    int32_t sample_begin;      /* this call renders samples [sample_begin, sample_begin+sample_count), which must end at or
                                  before RT_MAX_SAMPLE_END (RT_ERR_INVALID otherwise) */
    int32_t sample_count;      /* 0 = all of samples_per_pixel */
    int32_t pipeline;          /* RT_PIPELINE_* */
    int32_t device;            /* ignored: a scene lives on the device it was created on */
    int32_t samples_per_item;  /* tuning: consecutive samples one GPU thread integrates (0 = auto) */
    int32_t bvh_layout;        /* persistent pipeline: 0 = auto, 2 = binary 32-byte-node BVH, 4 = 4-wide 128-byte-node BVH */
} RtParams;

typedef struct RtScene RtScene; /* opaque: flattened scene resident on one device */

/* closest-hit record of the test entry point (mirrors hittable.rs:7-15) */
typedef struct RtHit {
    float t;
    float p[3];
    float normal[3];
    float u, v;
    int32_t front_face;
    int32_t material; /* index into desc.materials; -1 = miss */
    int32_t prim;     /* device primitive id, -1 = miss */
} RtHit;

/* counters of one render call (rays = path segments traced) */
typedef struct RtStats {
    uint64_t paths;
    uint64_t rays;
    double device_ms; /* CUDA-event time of the timed region */
    int32_t kernel_launches;
    int32_t pipeline_used;
    int32_t bvh_layout_used; /* 2 or 4 (RtParams.bvh_layout) */
    int32_t reserved;
} RtStats;

/*
 * The logger closure of Renderer::render (raytrace.rs:174,182): called exactly `total` = image-height times per
 * render, once for every row index j = 0 .. total-1 in increasing order, on the calling host thread, paced by the
 * device's progress (a row is reported when the matching share of the samples has been traced).
 */
typedef void (*RtProgressFn)(int row, int total, void* user);

/*
 * Accumulation.  Radiance sums are kept on the device as unsigned 64-bit FIXED-POINT integers with 32 fractional bits
 * (value = sum * RT_ACCUM_FIXED_ONE).  Integer addition is associative, so an image does not depend on the order in
 * which the device's reductions land nor on how the samples are split over calls or GPUs: one seed, one image, bit
 * for bit — as the reference's per-row PCG streams give it (raytrace.rs:179,197).  A sample is clamped to
 * [0, 2^20] before conversion (NaN counts as 0); the 64-bit sum holds at least 2^11 such extremes per pixel.
 * The float buffers of the entry points below are these sums converted once (round to nearest).
 */
#define RT_ACCUM_FIXED_ONE 4294967296.0

const char* rt_last_error(void);
int rt_abi_version(void);
int rt_device_count(void);

/* canonical SHA-256 of a description (values as f64, construction order) */
int rt_scene_hash(const RtSceneDesc* desc, uint8_t out[32]);

/* flatten + build the device BVH + upload.  Replaces World::build's result + World::background. */
int rt_scene_create(const RtSceneDesc* desc, int device, RtScene** out);
void rt_scene_destroy(RtScene* scene);
/*
 * Destroyed scenes hand their device blocks (tables, scratch images, texture arrays; at most 512 MB per device) to a
 * per-device free list instead of cudaFree, because freeing stalls for tens of milliseconds on this driver.  This call
 * returns all of it to the driver (all devices).  Safe at any time; live scenes are not touched.
 */
void rt_release_cached_memory(void);
int rt_scene_info(const RtScene* scene, int32_t* n_prims, int32_t* n_bvh_nodes, int32_t* n_media, int64_t* device_bytes);
/*
 * How the scene's BVH was built.  Scenes of RT_GPU_BUILD_MIN primitives or more (environment RT_BVH_GPU_MIN overrides)
 * get a linear BVH built ON THE GPU (Morton codes, radix sort, Karras' parallel hierarchy, bottom-up boxes; an extension:
 * the reference builds on the host, src/bhv.rs:122-145); smaller ones the host's SAH sweep plus the 4-wide collapse.
 *   built_on_device: 1 / 0;  build_ms: device time of the GPU build (0 for a host build);  depth: depth of the binary tree
 */
#define RT_GPU_BUILD_MIN 32768
int rt_scene_build_info(const RtScene* scene, int32_t* built_on_device, float* build_ms, int32_t* depth);

/*
 * Renderer::new_with_rng + render (raytrace.rs:151-186) with HOST buffers.
 *   accum_rgb: optional, 3*W*H floats, sum of sample radiance (not divided by spp)
 *   rgb:       optional, 3*W*H int32 in 0..=255 after to_rgb (raytrace.rs:59-68);
 *              row j = 0 is the BOTTOM row, exactly like the reference's Vec<Vec<RGB>>.
 * Blocking; cb is invoked on the calling host thread only.  Thread-compatible: different scenes may render from
 * different host threads at the same time, one scene serves one render call at a time (it owns scratch buffers).
 */
int rt_render(const RtScene* scene, const RtCamera* cam, const RtParams* params, float* accum_rgb,
              int32_t* rgb, RtProgressFn cb, void* user, RtStats* stats);

/*
 * Same work with DEVICE buffers (for sharded multi-GPU use: the caller owns the
 * accumulation buffer, reduces it across ranks, then tonemaps on the root).
 * d_accum_rgb: 3*W*H floats on scene's device, ADDED to (caller zeroes it).
 * stream: a cudaStream_t passed as void* (NULL = default stream).  Asynchronous
 * unless stats != NULL (then it synchronises to fill device_ms / rays).
 */
int rt_render_accumulate_device(const RtScene* scene, const RtCamera* cam, const RtParams* params,
                                float* d_accum_rgb, void* stream, RtStats* stats);
int rt_tonemap_device(const float* d_accum_rgb, int32_t* d_rgb, int32_t n_pixels, int32_t samples_per_pixel,
                      int device, void* stream);
/*
 * The same with the library's native fixed-point sums (3*W*H uint64 on the scene's device, ADDED to): what a sharded
 * render reduces across ranks with an integer sum — exact, so 1 GPU and N GPUs give identical images.
 */
int rt_render_accumulate_fixed_device(const RtScene* scene, const RtCamera* cam, const RtParams* params,
                                      uint64_t* d_accum_fixed, void* stream, RtStats* stats);
int rt_tonemap_fixed_device(const uint64_t* d_accum_fixed, int32_t* d_rgb, int32_t n_pixels, int32_t samples_per_pixel,
                            int device, void* stream);
int rt_accum_fixed_to_float_device(const uint64_t* d_accum_fixed, float* d_accum_rgb, int64_t n_values, int device,
                                   void* stream);

/*
 * EXTENSION (no counterpart in the reference): per-pixel second moments and noise-threshold adaptive sampling.
 *
 * Second moments are kept beside the radiance sums as unsigned 64-bit fixed-point sums of the SQUARED samples: every
 * sample q of the accumulation (in RT_ACCUM_FIXED_ONE units) adds (min(q, 2^44))^2 >> 40, i.e. radiance^2 in units of
 * 1 / RT_MOMENT2_FIXED_ONE, exactly.  A sample above 4096 is capped in the square; the sum holds 2^16 - 1 such extremes.
 * Both entry points run on the persistent pipeline only (RT_ERR_UNSUPPORTED for another pipeline).
 *
 * rt_render_moments_fixed_device: rt_render_accumulate_fixed_device plus d_moment2_fixed (3*W*H uint64 on the scene's
 * device, ADDED to).  Sums of disjoint sample ranges add up exactly, so it composes with sample slices.
 *
 * rt_render_adaptive: samples every pixel until its noise is below a threshold, at most params->samples_per_pixel (the
 * cap; sample_begin and sample_count must be 0).  Round 0 renders samples [0, min_samples) of every pixel (min_samples
 * >= 2); each later round doubles the count of the pixels still active, the last capped at the maximum, so a pixel's
 * count n is one of min_samples * 2^k or the cap, and its sums equal those of a uniform n-spp render bit for bit.  A pixel
 * stops when n reaches the cap or when every channel, with mean mu, sample variance s^2 and standard error se =
 * sqrt(s^2 / n), has se / (2 sqrt(max(mu, 2^-16))) <= noise_threshold (the error after the gamma-2 tonemap) or
 * mu - 3 se >= 1 (saturated).  Host buffers, each optional: rgb (3*W*H, every pixel tonemapped with its own count; row 0
 * at the bottom), samples (W*H counts), accum_fixed and moment2_fixed (3*W*H sums).  cb as in rt_render, paced by rounds.
 * stats->paths is the number of paths traced (the sum of the counts).
 */
#define RT_MOMENT2_FIXED_ONE 16777216.0
typedef struct RtAdaptive {
    double noise_threshold; /* >= 0; with 0 only pixels with a zero variance estimate (or saturated) stop early */
    int32_t min_samples;    /* >= 2 and <= samples_per_pixel */
    int32_t reserved;
} RtAdaptive;
int rt_render_moments_fixed_device(const RtScene* scene, const RtCamera* cam, const RtParams* params, uint64_t* d_accum_fixed,
                                   uint64_t* d_moment2_fixed, void* stream, RtStats* stats);
int rt_render_adaptive(const RtScene* scene, const RtCamera* cam, const RtParams* params, const RtAdaptive* adaptive,
                       int32_t* rgb, int32_t* samples, uint64_t* accum_fixed, uint64_t* moment2_fixed, RtProgressFn cb,
                       void* user, RtStats* stats);

/*
 * EXTENSION (no counterpart in the reference): a non-local-means denoiser guided by the per-pixel variance of the mean
 * (Rousselle, Knaus & Zwicker, "Adaptive Rendering with Non-Local Means Filtering", SIGGRAPH Asia 2012).
 *
 * Per pixel p and channel c, with mean mu and variance of the mean v (f32, [H][W][3]), for every offset d of the search
 * window [-r, r]^2 whose candidate q = p + d lies in the image, and y = clamp(x + d) (clamp = to the image):
 *   e_d(x) = sum_c [(mu_c(x) - mu_c(y))^2 - alpha (v_c(x) + min(v_c(x), v_c(y)))] / (1e-10 + k^2 (v_c(x) + v_c(y)))
 *   D(p, d) = mean of e_d(clamp(p + o)) over o in [-f, f]^2, / 3;   w = exp(-max(0, D)), and w = 1 for d = 0
 *   out_c(p) = sum_d w mu_c(q) / sum_d w   (one weight for the three channels)
 * The filter is biased: it trades noise for blur where patches look alike within their noise.
 *
 * rt_denoise_device: the filter on device buffers of `device` (3*W*H floats each; d_out_rgb must not overlap an input;
 * height at most RT_DENOISE_MAX_HEIGHT, the rows of 65 535 tiles of 16).
 * Deterministic: the same inputs give the same bits.  Asynchronous on `stream` (a cudaStream_t, NULL = default stream).
 *
 * rt_render_denoised: renders through the moments family of rt_render_moments_fixed_device — a uniform render of
 * samples_per_pixel (>= 2) when `adaptive` is NULL, else the rounds of rt_render_adaptive — then, per pixel with its own
 * count n, mu = S1 2^-32 / n and v = max(0, (S2 2^-24 - n mu^2) / (n - 1)) / n (f64, each rounded once to f32), denoises
 * and tonemaps the result with to_rgb.  Host buffers, each optional, row 0 at the bottom: rgb (3*W*H int32) and
 * denoised_rgb (3*W*H floats, the filtered means).  Persistent pipeline only; sample_begin and sample_count must be 0.
 * cb: called once per row index as in rt_render; an adaptive render paces it by rounds, a uniform one reports every row
 * when the render has finished (the moments family runs as one launch).  stats: paths traced, device_ms from the first render launch to the
 * end of the tonemap.
 */
#define RT_DENOISE_DEFAULT_SEARCH_RADIUS 10
#define RT_DENOISE_DEFAULT_PATCH_RADIUS 3
#define RT_DENOISE_DEFAULT_K 0.45
#define RT_DENOISE_DEFAULT_ALPHA 1.0
#define RT_DENOISE_MAX_SEARCH_RADIUS 15
#define RT_DENOISE_MAX_PATCH_RADIUS 7
#define RT_DENOISE_MAX_HEIGHT 1048560
typedef struct RtDenoise {
    double k;              /* strength, > 0 with (float)(k * k) finite (k^2 at most FLT_MAX): larger blurs more */
    double alpha;          /* variance cancellation, >= 0 with (float)alpha finite (at most FLT_MAX) */
    int32_t search_radius; /* r in [0, RT_DENOISE_MAX_SEARCH_RADIUS]; 0 returns the input */
    int32_t patch_radius;  /* f in [0, RT_DENOISE_MAX_PATCH_RADIUS] */
} RtDenoise;
int rt_denoise_device(const float* d_mean_rgb, const float* d_var_rgb, int32_t width, int32_t height, const RtDenoise* opt,
                      float* d_out_rgb, int device, void* stream);
int rt_render_denoised(const RtScene* scene, const RtCamera* cam, const RtParams* params, const RtAdaptive* adaptive,
                       const RtDenoise* opt, int32_t* rgb, float* denoised_rgb, RtProgressFn cb, void* user, RtStats* stats);

/*
 * EXTENSION: a feature-guided mode of the denoiser above.  The form follows Rousselle, Knaus & Zwicker, "Robust Denoising
 * using Feature and Color Information" (Pacific Graphics 2013); it was not checked against the paper's text.
 *
 * Features: the albedo and the normal at the FIRST EVENT of each path, which the render computes with the same Philox
 * draws (camera ray, then the medium event, then the closest surface below it through the render's tree layout):
 *   surface, Lambertian / metal / diffuse light: albedo = the material's colour (texture value or albedo), each channel
 *     clamped to [0, 1]; normal = the face-forwarded world normal (RtHit.normal)
 *   surface, dielectric: albedo (1, 1, 1); normal as above.  (Glass is a first event: what lies behind it is not guided.)
 *   medium event: albedo = the isotropic material's colour at the event; normal (0, 0, 0).  Media are not transparent.
 *   miss: albedo = the background colour of the ray; normal (0, 0, 0)
 * Per pixel and channel over n samples: the mean m and the variance of the mean s = max(0, (sum f^2 - n m^2) / (n - 1)) / n,
 * s = 0 for n = 1 (f64, each rounded once to f32).
 *
 * Guided filter: the weight of candidate q for pixel p becomes
 *   w(p, q) = min(w_colour(p, q), exp(-max(0, d_albedo(p, q))), exp(-max(0, d_normal(p, q))))
 * with w_colour the weight of rt_denoise_device, and per feature, with g_c(p)^2 the squared central-difference gradient of the
 * channel's mean at p (neighbours clamped to the image):
 *   g_c(p)^2 = ((m_c(x+1,y) - m_c(x-1,y)) / 2)^2 + ((m_c(x,y+1) - m_c(x,y-1)) / 2)^2
 *   d(p, q)  = (1/3) sum_c [(m_c(p) - m_c(q))^2 - (s_c(p) + min(s_c(p), s_c(q)))] / (k_feature^2 max(tau, s_c(p), g_c(p)^2))
 * Feature distances are per pixel, not per patch.  Where every feature weight is 1 (constant features of zero variance, or a
 * k_feature whose square exceeds the f32 range) the output is rt_denoise_device's bit for bit.  Radii and bounds are those of
 * RtDenoise: the features are read through the cache, not staged in shared memory.
 *
 * rt_render_features_device: the features of samples [sample_begin, sample_begin + count) of every pixel (count =
 * sample_count, or samples_per_pixel - sample_begin when 0) into four device buffers of 3*W*H floats on the scene's device,
 * [H][W][3], row 0 at the bottom; the outputs must not overlap.  Deterministic; asynchronous on `stream` unless stats is given
 * (device_ms of the pass).
 * rt_denoise_guided_device: rt_denoise_device with the four feature buffers; d_out_rgb must not overlap an input.
 * rt_render_denoised_guided: rt_render_denoised, plus the features of samples [0, guide->feature_samples) of the same seed and
 * the guided filter; stats->device_ms includes the feature pass.
 */
#define RT_GUIDE_DEFAULT_K_FEATURE 1.0 /* set by the sweep of DESIGN.md section 5f */
#define RT_GUIDE_DEFAULT_TAU 1e-2
#define RT_GUIDE_DEFAULT_FEATURE_SAMPLES 16
typedef struct RtGuide {
    double k_feature;        /* > 0: larger lets more across feature edges */
    double tau;              /* > 0 and finite: the floor of the feature's normalisation */
    /* The filter computes 1 / (3 k_feature^2 max(tau, s, g^2)) in f32 with subnormals flushed to zero, so (float)(3 k_feature^2),
     * (float)tau and their f32 product must each be at least FLT_MIN; (float)(3 k_feature^2) may be +inf (k_feature above about
     * 1.07e19: the feature is ignored).  Smaller values are RT_ERR_INVALID. */
    int32_t feature_samples; /* >= 1; used by rt_render_denoised_guided only */
    int32_t reserved;
} RtGuide;
int rt_render_features_device(const RtScene* scene, const RtCamera* cam, const RtParams* params, float* d_albedo,
                              float* d_albedo_var, float* d_normal, float* d_normal_var, void* stream, RtStats* stats);
int rt_denoise_guided_device(const float* d_mean_rgb, const float* d_var_rgb, const float* d_albedo, const float* d_albedo_var,
                             const float* d_normal, const float* d_normal_var, int32_t width, int32_t height,
                             const RtDenoise* opt, const RtGuide* guide, float* d_out_rgb, int device, void* stream);
int rt_render_denoised_guided(const RtScene* scene, const RtCamera* cam, const RtParams* params, const RtAdaptive* adaptive,
                              const RtDenoise* opt, const RtGuide* guide, int32_t* rgb, float* denoised_rgb, RtProgressFn cb,
                              void* user, RtStats* stats);

/*
 * EXTENSION: dual-buffer cross-filtered denoising with a per-pixel error estimate, and adaptive sampling driven by that
 * estimate.  The form follows Rousselle, Knaus & Zwicker, "Adaptive Rendering with Non-Local Means Filtering" (SIGGRAPH
 * Asia 2012); it was not checked against the paper's text.
 *
 * Split: a job renders in ranges of samples (one for a uniform render, one per round for an adaptive one).  A range
 * [b, b + c), c even, sends [b, b + c/2) to buffer A and [b + c/2, b + c) to buffer B; each holds the (S1, S2) sums of the
 * moments family.  samples_per_pixel and min_samples (adaptive) must be even and >= 4, so every count n of the schedule of
 * rt_render_adaptive is even and each half of a pixel holds n/2 >= 2 samples.  Per half, mu and v are those of
 * rt_render_denoised with n/2.
 * Cross filter: F_A is the filter of rt_denoise_device whose weights w(p, q) are computed from (mu_B, v_B), applied to
 * mu_A; F_B is the same with A and B swapped.  With a guide each weight is also bounded by the feature weight of
 * rt_denoise_guided_device (the same features for both halves).  out = (F_A + F_B) / 2 (f32).
 * Error estimate: per channel, eps_c(p) = the mean over the 3 x 3 neighbourhood of p (neighbours clamped to the image, in
 * row order from the bottom left) of ((F_A,c - F_B,c) / 2)^2, in f32 with every operation rounded on its own.  It estimates
 * the VARIANCE of out_c(p), not its bias.
 * Filtered stop rule: the rule of rt_render_adaptive on (out, eps) in place of (mu, se^2): per channel, in f64 with every
 * operation rounded on its own, e = sqrt(eps) / (2 sqrt(max(out, 2^-16))); a pixel stops when n reaches the cap or when
 * every channel has e <= noise_threshold or out - 3 sqrt(eps) >= 1.
 * Exact reductions: with A = B, F_A = F_B = the output of rt_denoise_device (rt_denoise_guided_device with a guide) bit
 * for bit, out equals it and eps = 0; swapping A and B gives the same out and eps bit for bit.
 *
 * rt_denoise_cross_device: the cross filter and the error estimate on device buffers of `device` (3*W*H floats each).
 * guide NULL: colour-only, and the four feature pointers must be NULL; else all four are given.  d_err_rgb is optional;
 * no output may overlap an input or the other output.  Asynchronous on `stream`.
 * rt_render_denoised_dual: renders the two halves through the moments family — uniformly when `adaptive` is NULL, else in
 * the rounds of rt_render_adaptive with the filtered stop rule (noise_threshold is its threshold) — cross-filters (guided
 * when `guide` is given: the features of samples [0, guide->feature_samples), computed once before the first round) and
 * tonemaps out with to_rgb.  In an adaptive render each round renders its half ranges for the active pixels, converts both
 * halves of every pixel, filters the whole image and evaluates the active pixels.  Host buffers, each optional, row 0 at the
 * bottom: rgb (3*W*H), denoised_rgb (out) and error_rgb (eps), 3*W*H floats each, samples (W*H counts).  Persistent
 * pipeline only; sample_begin and sample_count must be 0.  cb as in rt_render_denoised.  stats: paths = the sum of the
 * counts, device_ms from the first render launch (the feature pass) to the end of the tonemap.
 */
int rt_denoise_cross_device(const float* d_mean_a, const float* d_var_a, const float* d_mean_b, const float* d_var_b,
                            const float* d_albedo, const float* d_albedo_var, const float* d_normal, const float* d_normal_var,
                            int32_t width, int32_t height, const RtDenoise* opt, const RtGuide* guide, float* d_out_rgb,
                            float* d_err_rgb, int device, void* stream);
int rt_render_denoised_dual(const RtScene* scene, const RtCamera* cam, const RtParams* params, const RtAdaptive* adaptive,
                            const RtDenoise* opt, const RtGuide* guide, int32_t* rgb, float* denoised_rgb, float* error_rgb,
                            int32_t* samples, RtProgressFn cb, void* user, RtStats* stats);

/*
 * EXTENSION: per-pixel selection among three strengths of the cross filter by Stein's unbiased risk estimate (SURE), with a
 * bias-aware error estimate that drives adaptive sampling.  In the spirit of Li, Wu & Chuang, "SURE-based optimization for
 * adaptive sampling and reconstruction" (SIGGRAPH Asia 2012) and Rousselle, Knaus & Zwicker, "Robust Denoising using Feature
 * and Color Information" (Pacific Graphics 2013); the form was not checked against the papers' text.
 *
 * Inputs: those of rt_denoise_cross_device.  Candidates j = 0, 1, 2 with strengths s = (1, ratio^2, ratio^-2), computed in f64
 * and each rounded once to f32: s_1 = (float)(ratio * ratio), s_2 = (float)(1 / (ratio * ratio)).
 *   Weights: with D(p, q) the patch distance of rt_denoise_device, w_j(p, q) = exp(-s_j max(0, D(p, q))); with a guide,
 *   min(w_j, the feature weight of rt_denoise_guided_device).  w = 1 at d = 0; candidates outside the image are skipped.
 *   j = 0 is the cross filter; j = 1 blurs less (about k / ratio), j = 2 more (about k ratio).
 *   Filters: F_A,j takes its weights from (mu_B, v_B) and its values from mu_A, with weight sum W_A,j(p) = sum_q w_j(p, q) >= 1;
 *   F_B,j is the same with A and B swapped.  F_A,j is a linear smoother of mu_A whose derivative in mu_A(p) is 1 / W_A,j(p).
 *   Risk of one half, per channel (f32, every operation rounded on its own, in this order; W = 1 gives exactly v_A):
 *     R_A,j,c(p) = (F_A,j,c(p) - mu_A,c(p))^2 + v_A,c(p) (2 / W_A,j(p) - 1)
 *   an unbiased estimate of E[(F_A,j,c(p) - t_c(p))^2] (t the expected value) for independent pixels and an unbiased v; R_B is
 *   the same with A and B swapped.
 *   Risk of the output: s_hat_j,c(p) = (R_A,j,c + R_B,j,c) / 2, an estimate of an upper bound of E[(out_j - t)^2] with
 *   out_j = (F_A,j + F_B,j) / 2, since ((a + b) / 2)^2 <= (a^2 + b^2) / 2.
 *   Selection: S_j(p) = the mean over the (2b + 1)^2 window around p (b = smooth_radius; neighbours clamped to the image, in row
 *   order from the bottom left) of (s_hat_j,0 + s_hat_j,1) + s_hat_j,2, the sum and the division by (2b + 1)^2 in f32 with every
 *   operation rounded on its own; j*(p) = argmin_j S_j(p), ties to the smaller j.
 *   Outputs: out(p) = (F_A,j* + F_B,j*) / 2 as in rt_denoise_cross_device; err_c(p) = max(0, the window mean, in the same order,
 *   of s_hat_j*(p),c); choice(p) = j*(p).
 *   SURE stop rule: the filtered stop rule of rt_render_denoised_dual with (out, err) in place of (out, eps).
 * Exact reductions: ratio = 1 gives rt_denoise_cross_device's out bit for bit (colour-only and guided) and choice 0 everywhere;
 * r = 0 gives every W = 1, out = (mu_A + mu_B) / 2 and err the window mean of (v_A + v_B) / 2; swapping A and B gives the same
 * out, err and choice bit for bit.
 * Caveat: with a guide, the features come from samples [0, feature_samples), which overlap half A of the first range, so the
 * weights of F_A are not independent of A and the estimate is approximate in guided mode.
 *
 * RtSure: ratio >= 1, with (float)(ratio^2) finite and (float)(ratio^-2) at least FLT_MIN; smooth_radius in
 * [0, RT_SURE_MAX_SMOOTH_RADIUS].  Other values are RT_ERR_INVALID.
 * rt_denoise_sure_device: rt_denoise_cross_device with the selection: out and the optional err (3*W*H floats each) and choice
 * (W*H int32); no output may overlap an input or another output.  Deterministic; asynchronous on `stream`.  It allocates
 * 11 x 3*W*H floats of stream-ordered scratch (F and W of the three candidates in both directions, and s_hat), against
 * 2 x 3*W*H for rt_denoise_cross_device: about 1.9 GB at 3840 x 3840.  rt_render_denoised_sure holds the same scratch.
 * rt_render_denoised_sure: rt_render_denoised_dual with the SURE filter in place of the cross filter and the SURE stop rule in
 * adaptive renders; error_rgb receives err and choice (optional, W*H) the final choice of every pixel.
 */
#define RT_SURE_DEFAULT_RATIO 1.5         /* set by the sweep of DESIGN.md section 5h */
#define RT_SURE_DEFAULT_SMOOTH_RADIUS 5
#define RT_SURE_MAX_SMOOTH_RADIUS 7
typedef struct RtSure {
    double ratio;          /* >= 1: the strengths of the candidates are 1, ratio^2 and ratio^-2 */
    int32_t smooth_radius; /* b in [0, RT_SURE_MAX_SMOOTH_RADIUS]: the window of the selection is (2b + 1)^2 */
    int32_t reserved;
} RtSure;
int rt_denoise_sure_device(const float* d_mean_a, const float* d_var_a, const float* d_mean_b, const float* d_var_b,
                           const float* d_albedo, const float* d_albedo_var, const float* d_normal, const float* d_normal_var,
                           int32_t width, int32_t height, const RtDenoise* opt, const RtGuide* guide, const RtSure* sure,
                           float* d_out_rgb, float* d_err_rgb, int32_t* d_choice, int device, void* stream);
int rt_render_denoised_sure(const RtScene* scene, const RtCamera* cam, const RtParams* params, const RtAdaptive* adaptive,
                            const RtDenoise* opt, const RtGuide* guide, const RtSure* sure, int32_t* rgb, float* denoised_rgb,
                            float* error_rgb, int32_t* samples, int32_t* choice, RtProgressFn cb, void* user, RtStats* stats);

/*
 * EXTENSION: a neighbourhood prior on each pixel's per-sample variance (empirical Bayes), for the stop rules of
 * rt_render_adaptive and rt_render_denoised_sure.  A pixel whose first samples found no light has mu = 0 and s^2 = 0, so its
 * error estimate is 0 and it stops in round 0; the prior lends it the variance of the pixels around it.
 *
 * Term of a pixel q holding n_q >= 2 samples, per channel c, with mu as in the rule of rt_render_adaptive (f64, every
 * operation rounded on its own): N_q,c = max(0, S2 2^-24 - n_q mu^2) (that is (n_q - 1) s^2) and d_q = n_q - 1.  Stored as
 * four f64 per pixel (N_r, N_g, N_b, d).
 * Pool of p: the window is the (2b + 1)^2 square around p WITHOUT p; neighbours outside the image are skipped (not clamped).
 * sum N_c and sum d in f64 over the window in row order from the bottom left (dy = -b..b, then dx = -b..b), every addition
 * rounded on its own; P_c(p) = sum N_c / sum d (f64).  Every pixel takes part with its current sums: a stopped pixel keeps
 * feeding its neighbours.
 * Posterior per-sample variance, n0 = prior_samples (f64, every operation rounded on its own, in this form):
 *   s~^2_c = (N_p,c + n0 P_c) / ((n_p - 1) + n0)
 * and, when the window holds no pixel (a 1 x 1 image), s~^2_c = N_p,c / (n_p - 1) = s^2 (no prior).  n0 = 0 gives s^2 bit for
 * bit.  There is no prior on the mean.
 * Prior rule: the rule of rt_render_adaptive with s~^2 in place of s^2 (mu, the slope, the saturation test and the cap as
 * there).  A mu = 0 pixel with noisy neighbours keeps sampling; one whose neighbours are all noise-free still stops.
 * SURE prior rule (rt_render_denoised_sure_prior): the same pool and posterior per half, from the half's own sums with
 * n = n_p / 2 and the neighbours' sums of the same half: v~_A = s~^2_A / (n_p / 2) (f64, rounded once to f32), v~_B likewise.
 * s_hat'_j,c = (R'_A + R'_B) / 2 with R' the risk of rt_render_denoised_sure with v~ in place of v; err'_c(p) = max(0, the
 * window mean of s_hat'_j*(p),c) with j*(p), the window and the order of the selection.  The stop rule is the filtered rule on
 * (out, err').  out and the choice are those of rt_render_denoised_sure: the prior only decides which pixels go on.
 * Exact reductions: n0 = 0 at any radius gives rt_render_adaptive and rt_render_denoised_sure bit for bit (every output, the
 * counts and stats->paths); so does a window without pixels at any n0 in the per-pixel functions (an image of one pixel,
 * which the renders, at least 2 x 2, do not take).
 *
 * RtPrior: prior_samples finite and >= 0, radius in [1, RT_PRIOR_MAX_RADIUS]; other values, or a NULL RtPrior, are
 * RT_ERR_INVALID.
 * rt_render_adaptive_prior: rt_render_adaptive with the prior rule.  It holds 4 f64 of terms per pixel of scratch.
 * rt_render_denoised_sure_prior: rt_render_denoised_sure with the SURE prior rule; `adaptive` must be given (a uniform render
 * has no stop rule).  error_rgb receives err'.  It holds 8 f64 of terms and 6 f32 of v~ per pixel beside the scratch of
 * rt_render_denoised_sure.
 */
#define RT_PRIOR_DEFAULT_SAMPLES 16.0 /* set by the sweep of DESIGN.md section 5i */
#define RT_PRIOR_DEFAULT_RADIUS 7
#define RT_PRIOR_MAX_RADIUS 7
typedef struct RtPrior {
    double prior_samples; /* n0 >= 0 and finite: the weight of the neighbourhood's variance, in samples */
    int32_t radius;       /* b in [1, RT_PRIOR_MAX_RADIUS]: the window is (2b + 1)^2 without the pixel */
    int32_t reserved;
} RtPrior;
int rt_render_adaptive_prior(const RtScene* scene, const RtCamera* cam, const RtParams* params, const RtAdaptive* adaptive,
                             const RtPrior* prior, int32_t* rgb, int32_t* samples, uint64_t* accum_fixed, uint64_t* moment2_fixed,
                             RtProgressFn cb, void* user, RtStats* stats);
int rt_render_denoised_sure_prior(const RtScene* scene, const RtCamera* cam, const RtParams* params, const RtAdaptive* adaptive,
                                  const RtDenoise* opt, const RtGuide* guide, const RtSure* sure, const RtPrior* prior, int32_t* rgb,
                                  float* denoised_rgb, float* error_rgb, int32_t* samples, int32_t* choice, RtProgressFn cb,
                                  void* user, RtStats* stats);

/*
 * rt_render over several GPUs of one process (the reference's row-parallel rayon loop, raytrace.rs:176-185, becomes
 * sample slices): scenes[g] is the same description created on a distinct device; device g renders every pixel for
 * the g-th slice of the sample range (rt_sample_slice), the float accumulation buffers are summed onto scenes[0]'s
 * device with one ncclReduce, and that device tonemaps.  NCCL is bound at run time (dlopen libnccl.so.2);
 * RT_ERR_UNSUPPORTED if it cannot be loaded.  n_scenes == 1 is rt_render.  Buffers and callback as in rt_render.
 */
int rt_render_multi(RtScene* const* scenes, int32_t n_scenes, const RtCamera* cam, const RtParams* params, float* accum_rgb,
                    int32_t* rgb, RtProgressFn cb, void* user, RtStats* stats);
/* part `part` of `n_parts` of the sample range: contiguous, disjoint, covering, sizes differ by at most one */
void rt_sample_slice(int32_t sample_begin, int32_t sample_count, int32_t n_parts, int32_t part, int32_t* begin, int32_t* count);

/*
 * Hittable::hit for a batch of rays (test entry point, SURVEY §8c level 2).
 *   node: index of a node of the description the scene was created from; the
 *         closest hit of that subtree is returned (root = whole world, media excluded
 *         unless node is itself a MEDIUM, in which case `t` = entry and `u` = exit of
 *         the clipped boundary interval and no free-flight sampling is done).
 *         node = -1: the whole world through the binary BVH; node = -2: through the 4-wide BVH.
 *   rays: N x 8 floats: origin xyz, direction xyz (NOT normalised), t_min, t_max.
 */
int rt_intersect_batch(const RtScene* scene, int32_t node, const float* rays, int64_t n, RtHit* out);
/* the same with the rays at time `time` in [0, 1] (moving spheres; rt_intersect_batch is time 0) */
int rt_intersect_batch_at(const RtScene* scene, int32_t node, float time, const float* rays, int64_t n, RtHit* out);

/*
 * Material::scatter / Material::emit (materials.rs:7-11; impls :25-127, volumes.rs:77-83) for a batch of fixed hits
 * (test entry point, SURVEY §8c level 2 for the shade stage).  The caller supplies the hit record (p, the face-forwarded
 * normal, u, v, front_face as hittable.rs:7-15 holds them), the incoming ray and the four uniforms the device would draw
 * for this event: uniform[0..2] -> the in-ball sample of Lambertian / fuzzy Metal / Isotropic (z = 1 - 2 u0,
 * azimuth 2 pi u1, radius cbrt(u2): the direct sampler that replaces vec.rs:23-30's rejection loop), uniform[3] -> the
 * Dielectric's reflect-or-refract draw (materials.rs:98).
 *   scattered = 1: attenuation and the scattered ray's direction (its origin is p); emitted = 0
 *   scattered = 0: emitted = Material::emit (DiffuseLight: its texture, both faces; everything else 0)
 */
typedef struct RtScatterIn {
    float ray_origin[3], ray_dir[3];
    float p[3], normal[3];
    float u, v;
    int32_t front_face;
    int32_t material; /* index into desc.materials */
    float uniform[4];
} RtScatterIn;
typedef struct RtScatterOut {
    int32_t scattered;
    float attenuation[3];
    float dir[3];
    float emitted[3];
} RtScatterOut;
int rt_scatter_batch(const RtScene* scene, const RtScatterIn* in, int64_t n, RtScatterOut* out);

/*
 * Texture::value (textures.rs:4-6) for a batch (test entry point).
 *   texture: index into desc.textures; uvp: N x 5 floats (u, v, p.x, p.y, p.z); out: N x 3 floats.
 */
int rt_texture_value_batch(const RtScene* scene, int32_t texture, const float* uvp, int64_t n, float* out_rgb);

/*
 * Camera::get_ray + the pixel jitter of render_pixel (camera.rs:40-48, raytrace.rs:191-192) for a batch of
 * (pixel, sample) pairs (test entry point).  pixel = j*width + i with j = 0 the bottom row.
 *   out_rays:   N x 6 floats, origin xyz + direction xyz (not normalised)
 *   out_sample: N x 4 floats, the four uniforms used: jitter x, jitter y, lens disk x, lens disk y
 */
int rt_generate_rays(const RtCamera* cam, const RtParams* params, const int32_t* pixel, const int32_t* sample,
                     int64_t n, float* out_rays, float* out_sample);

/*
 * Measured ceilings of a device for the roofline the render kernels are quoted against (bench.py): dependent-FFMA
 * chains on every SM (scalar FFMA and packed FFMA2, 2 flops per multiply-add) and repeated reads of an L2-resident
 * 32 MB buffer; best of several CUDA-event-timed launches each.  Measurement aid; not on the render path.
 */
typedef struct RtPeaks {
    double fp32_ffma_tflops;        /* scalar FFMA chains */
    double fp32_ffma2_tflops;       /* packed FFMA2 chains (sm_100) */
    double fp32_theoretical_tflops; /* SMs x 128 lanes x 2 x the device's maximum SM clock */
    double l2_read_gbs;
    double sm_clock_mhz;            /* cudaDevAttrClockRate */
    int32_t sm_count;
    int32_t reserved;
} RtPeaks;
int rt_measure_peaks(int device, RtPeaks* out);

/* ---- host side above the ABI: worlds.rs restated against the description ---- */

typedef struct RtWorldInfo {
    double lookfrom[3], lookat[3];
    double vfov_deg;
    int32_t background_kind;
    int32_t needs_earthmap;
    int32_t uses_rng;
} RtWorldInfo;

int rt_world_count(void);
const char* rt_world_name(int index);
int rt_world_info(const char* name, RtWorldInfo* out);
/* World::build with rng = Pcg64::seed_from_u64(seed) (main.rs:185, rngator.rs:27-31).
 * earth_rgb may be NULL unless the world needs it.  *n_draws (optional) = next_u64 calls consumed. */
int rt_world_build(const char* name, uint64_t seed, const uint8_t* earth_rgb, int32_t earth_w, int32_t earth_h,
                   RtSceneDesc** out, uint64_t* n_draws);
void rt_scene_desc_free(RtSceneDesc* desc);

#ifdef __cplusplus
}
#endif
#endif /* RT_B200_H */
