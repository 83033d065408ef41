"""ctypes mirror of include/rt_b200.h — the C ABI of librt_b200.so.

Struct layouts follow the header field for field; `load()` opens the in-tree shared library and declares the
prototype of every exported entry point.  There is no Python or CPU fallback: if the library is missing,
`load()` raises, and every compute entry point of the library itself fails with RT_ERR_NO_DEVICE when no
CUDA device is usable.
"""
import ctypes as C
import os

RT_OK, RT_ERR_INVALID, RT_ERR_NO_DEVICE, RT_ERR_CUDA, RT_ERR_UNSUPPORTED = 0, 1, 2, 3, 4

RT_NODE_SPHERE, RT_NODE_XYRECT, RT_NODE_XZRECT, RT_NODE_YZRECT, RT_NODE_BLOCK = 1, 2, 3, 4, 5
RT_NODE_TRANSLATE, RT_NODE_ROTATE, RT_NODE_MEDIUM, RT_NODE_BVH, RT_NODE_LIST, RT_NODE_MOVING_SPHERE = 6, 7, 8, 9, 10, 11
RT_MAT_LAMBERTIAN, RT_MAT_METAL, RT_MAT_DIELECTRIC, RT_MAT_DIFFUSE_LIGHT, RT_MAT_ISOTROPIC = 1, 2, 3, 4, 5
RT_TEX_SOLID, RT_TEX_CHECKER, RT_TEX_NOISE, RT_TEX_IMAGE = 1, 2, 3, 4
RT_BG_BLACK, RT_BG_GRADIENT = 0, 1
RT_PIPELINE_AUTO, RT_PIPELINE_MEGAKERNEL, RT_PIPELINE_WAVEFRONT, RT_PIPELINE_WAVEFRONT_SMEM, RT_PIPELINE_PERSISTENT = 0, 1, 2, 3, 4
RT_PERLIN_POINTS = 1024


class RtNode(C.Structure):
    _fields_ = [("kind", C.c_int32), ("material", C.c_int32), ("first_child", C.c_int32), ("child_count", C.c_int32),
                ("axis", C.c_int32), ("reserved", C.c_int32), ("f", C.c_double * 8)]


class RtMaterial(C.Structure):
    _fields_ = [("kind", C.c_int32), ("texture", C.c_int32), ("albedo", C.c_double * 3), ("fuzz", C.c_double),
                ("ior", C.c_double)]


class RtTexture(C.Structure):
    _fields_ = [("kind", C.c_int32), ("a", C.c_int32), ("b", C.c_int32), ("reserved", C.c_int32),
                ("color", C.c_double * 3), ("scale", C.c_double)]


class RtPerlin(C.Structure):
    _fields_ = [("ranvec", (C.c_double * 3) * RT_PERLIN_POINTS), ("perm_x", C.c_int32 * RT_PERLIN_POINTS),
                ("perm_y", C.c_int32 * RT_PERLIN_POINTS), ("perm_z", C.c_int32 * RT_PERLIN_POINTS)]


class RtImage(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("rgb", C.POINTER(C.c_uint8))]


class RtSceneDesc(C.Structure):
    _fields_ = [("root", C.c_int32), ("background_kind", C.c_int32), ("background_top", C.c_double * 3),
                ("background_bottom", C.c_double * 3),
                ("n_nodes", C.c_int32), ("n_children", C.c_int32), ("n_materials", C.c_int32),
                ("n_textures", C.c_int32), ("n_perlins", C.c_int32), ("n_images", C.c_int32),
                ("nodes", C.POINTER(RtNode)), ("children", C.POINTER(C.c_int32)),
                ("materials", C.POINTER(RtMaterial)), ("textures", C.POINTER(RtTexture)),
                ("perlins", C.POINTER(RtPerlin)), ("images", C.POINTER(RtImage))]


class RtCamera(C.Structure):
    _fields_ = [("lookfrom", C.c_double * 3), ("lookat", C.c_double * 3), ("vup", C.c_double * 3),
                ("vfov_deg", C.c_double), ("aspect_ratio", C.c_double), ("aperture", C.c_double),
                ("focus_dist", C.c_double), ("time0", C.c_double), ("time1", C.c_double)]


class RtParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("samples_per_pixel", C.c_int32),
                ("max_depth", C.c_int32), ("seed", C.c_uint64), ("sample_begin", C.c_int32),
                ("sample_count", C.c_int32), ("pipeline", C.c_int32), ("device", C.c_int32),
                ("samples_per_item", C.c_int32), ("bvh_layout", C.c_int32)]


class RtHit(C.Structure):
    _fields_ = [("t", C.c_float), ("p", C.c_float * 3), ("normal", C.c_float * 3), ("u", C.c_float), ("v", C.c_float),
                ("front_face", C.c_int32), ("material", C.c_int32), ("prim", C.c_int32)]


class RtScatterIn(C.Structure):
    _fields_ = [("ray_origin", C.c_float * 3), ("ray_dir", C.c_float * 3), ("p", C.c_float * 3), ("normal", C.c_float * 3),
                ("u", C.c_float), ("v", C.c_float), ("front_face", C.c_int32), ("material", C.c_int32), ("uniform", C.c_float * 4)]


class RtScatterOut(C.Structure):
    _fields_ = [("scattered", C.c_int32), ("attenuation", C.c_float * 3), ("dir", C.c_float * 3), ("emitted", C.c_float * 3)]


class RtStats(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("rays", C.c_uint64), ("device_ms", C.c_double),
                ("kernel_launches", C.c_int32), ("pipeline_used", C.c_int32), ("bvh_layout_used", C.c_int32),
                ("reserved", C.c_int32)]


class RtPeaks(C.Structure):
    _fields_ = [("fp32_ffma_tflops", C.c_double), ("fp32_ffma2_tflops", C.c_double), ("fp32_theoretical_tflops", C.c_double),
                ("l2_read_gbs", C.c_double), ("sm_clock_mhz", C.c_double), ("sm_count", C.c_int32), ("reserved", C.c_int32)]


class RtAdaptive(C.Structure):  # EXTENSION: noise-threshold adaptive sampling (rt_render_adaptive)
    _fields_ = [("noise_threshold", C.c_double), ("min_samples", C.c_int32), ("reserved", C.c_int32)]


class RtDenoise(C.Structure):  # EXTENSION: variance-guided non-local-means denoiser (rt_denoise_device, rt_render_denoised)
    _fields_ = [("k", C.c_double), ("alpha", C.c_double), ("search_radius", C.c_int32), ("patch_radius", C.c_int32)]


RT_DENOISE_DEFAULT_SEARCH_RADIUS, RT_DENOISE_DEFAULT_PATCH_RADIUS, RT_DENOISE_DEFAULT_K, RT_DENOISE_DEFAULT_ALPHA = 10, 3, 0.45, 1.0
RT_DENOISE_MAX_SEARCH_RADIUS, RT_DENOISE_MAX_PATCH_RADIUS, RT_DENOISE_MAX_HEIGHT = 15, 7, 1048560


class RtGuide(C.Structure):  # EXTENSION: feature-guided denoising (rt_denoise_guided_device, rt_render_denoised_guided)
    _fields_ = [("k_feature", C.c_double), ("tau", C.c_double), ("feature_samples", C.c_int32), ("reserved", C.c_int32)]


RT_GUIDE_DEFAULT_K_FEATURE, RT_GUIDE_DEFAULT_TAU, RT_GUIDE_DEFAULT_FEATURE_SAMPLES = 1.0, 1e-2, 16


class RtWorldInfo(C.Structure):
    _fields_ = [("lookfrom", C.c_double * 3), ("lookat", C.c_double * 3), ("vfov_deg", C.c_double),
                ("background_kind", C.c_int32), ("needs_earthmap", C.c_int32), ("uses_rng", C.c_int32)]


RtProgressFn = C.CFUNCTYPE(None, C.c_int, C.c_int, C.c_void_p)

# every symbol include/rt_b200.h declares: name -> (restype, argtypes)
PROTOTYPES = {
    "rt_last_error": (C.c_char_p, []),
    "rt_abi_version": (C.c_int, []),
    "rt_device_count": (C.c_int, []),
    "rt_scene_hash": (C.c_int, [C.POINTER(RtSceneDesc), C.POINTER(C.c_uint8)]),
    "rt_scene_create": (C.c_int, [C.POINTER(RtSceneDesc), C.c_int, C.POINTER(C.c_void_p)]),
    "rt_scene_destroy": (None, [C.c_void_p]),
    "rt_scene_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                C.POINTER(C.c_int64)]),
    "rt_scene_build_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_float), C.POINTER(C.c_int32)]),
    "rt_render": (C.c_int, [C.c_void_p, C.POINTER(RtCamera), C.POINTER(RtParams), C.c_void_p, C.c_void_p,
                            RtProgressFn, C.c_void_p, C.POINTER(RtStats)]),
    "rt_render_accumulate_device": (C.c_int, [C.c_void_p, C.POINTER(RtCamera), C.POINTER(RtParams), C.c_void_p,
                                              C.c_void_p, C.POINTER(RtStats)]),
    "rt_render_multi": (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.POINTER(RtCamera), C.POINTER(RtParams), C.c_void_p,
                                  C.c_void_p, RtProgressFn, C.c_void_p, C.POINTER(RtStats)]),
    "rt_sample_slice": (None, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "rt_tonemap_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int, C.c_void_p]),
    "rt_render_accumulate_fixed_device": (C.c_int, [C.c_void_p, C.POINTER(RtCamera), C.POINTER(RtParams), C.c_void_p,
                                                    C.c_void_p, C.POINTER(RtStats)]),
    "rt_render_moments_fixed_device": (C.c_int, [C.c_void_p, C.POINTER(RtCamera), C.POINTER(RtParams), C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.POINTER(RtStats)]),
    "rt_render_adaptive": (C.c_int, [C.c_void_p, C.POINTER(RtCamera), C.POINTER(RtParams), C.POINTER(RtAdaptive), C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, RtProgressFn, C.c_void_p, C.POINTER(RtStats)]),
    "rt_denoise_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(RtDenoise), C.c_void_p, C.c_int, C.c_void_p]),
    "rt_render_denoised": (C.c_int, [C.c_void_p, C.POINTER(RtCamera), C.POINTER(RtParams), C.POINTER(RtAdaptive), C.POINTER(RtDenoise),
                                     C.c_void_p, C.c_void_p, RtProgressFn, C.c_void_p, C.POINTER(RtStats)]),
    "rt_render_features_device": (C.c_int, [C.c_void_p, C.POINTER(RtCamera), C.POINTER(RtParams), C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.POINTER(RtStats)]),
    "rt_denoise_guided_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                           C.POINTER(RtDenoise), C.POINTER(RtGuide), C.c_void_p, C.c_int, C.c_void_p]),
    "rt_render_denoised_guided": (C.c_int, [C.c_void_p, C.POINTER(RtCamera), C.POINTER(RtParams), C.POINTER(RtAdaptive),
                                            C.POINTER(RtDenoise), C.POINTER(RtGuide), C.c_void_p, C.c_void_p, RtProgressFn, C.c_void_p,
                                            C.POINTER(RtStats)]),
    "rt_denoise_cross_device": (C.c_int, [C.c_void_p] * 8 + [C.c_int32, C.c_int32, C.POINTER(RtDenoise), C.POINTER(RtGuide), C.c_void_p, C.c_void_p,
                                          C.c_int, C.c_void_p]),
    "rt_render_denoised_dual": (C.c_int, [C.c_void_p, C.POINTER(RtCamera), C.POINTER(RtParams), C.POINTER(RtAdaptive), C.POINTER(RtDenoise),
                                          C.POINTER(RtGuide), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, RtProgressFn, C.c_void_p,
                                          C.POINTER(RtStats)]),
    "rt_tonemap_fixed_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int, C.c_void_p]),
    "rt_accum_fixed_to_float_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "rt_release_cached_memory": (None, []),
    "rt_intersect_batch": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.POINTER(RtHit)]),
    "rt_intersect_batch_at": (C.c_int, [C.c_void_p, C.c_int32, C.c_float, C.c_void_p, C.c_int64, C.POINTER(RtHit)]),
    "rt_scatter_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "rt_texture_value_batch": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "rt_generate_rays": (C.c_int, [C.POINTER(RtCamera), C.POINTER(RtParams), C.c_void_p, C.c_void_p, C.c_int64,
                                   C.c_void_p, C.c_void_p]),
    "rt_measure_peaks": (C.c_int, [C.c_int, C.POINTER(RtPeaks)]),
    "rt_world_count": (C.c_int, []),
    "rt_world_name": (C.c_char_p, [C.c_int]),
    "rt_world_info": (C.c_int, [C.c_char_p, C.POINTER(RtWorldInfo)]),
    "rt_world_build": (C.c_int, [C.c_char_p, C.c_uint64, C.c_void_p, C.c_int32, C.c_int32,
                                 C.POINTER(C.POINTER(RtSceneDesc)), C.POINTER(C.c_uint64)]),
    "rt_scene_desc_free": (None, [C.POINTER(RtSceneDesc)]),
}

RT_ACCUM_FIXED_ONE = 4294967296.0
RT_MAX_SAMPLE_END = 2 ** 31 - 1  # the largest sample_begin + sample_count
RT_MOMENT2_FIXED_ONE = 16777216.0

_HERE = os.path.dirname(os.path.abspath(__file__))
# RT_B200_LIB: another build of the same library (A/B measurements of compile-time choices); never a different implementation
LIB_PATH = os.environ.get("RT_B200_LIB") or os.path.join(_HERE, "librt_b200.so")
_lib = None


def load():
    """Open librt_b200.so (built in-tree by build.py) and set the prototypes.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "There is no CPU or pure-Python fallback for the render path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError here = the library does not export what the header declares
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class RtError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"rt_b200 error {code}: {message}")
        self.code = code


def check(code):
    if code != RT_OK:
        raise RtError(code, load().rt_last_error().decode("utf-8", "replace"))
