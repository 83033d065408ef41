"""Host-side mirror of the reference's render interface over the C ABI (no compute happens in Python).

Reference surface being mirrored (names, argument meaning, error behaviour):
  worlds() / World{name, camera, background, build}      src/worlds.rs:14-19, :471-484
  Camera::new(lookfrom, lookat, vup, vfov, aspect, aperture, focus_dist)   src/camera.rs:15-38
  RenderingParams{samples_per_pixel, image_height, image_width}           src/raytrace.rs:50-55
  RecursiveRayTracer{max_depth}                                           src/raytrace.rs:74-76
  SeedableRngator::new(seed)                                              src/rngator.rs:17-25
  Renderer::new_with_rng(camera, world, background, params, tracer, rng).render(logger) -> rows of (r,g,b),
      row j = 0 is the BOTTOM row, logger(j, height) called `height` times   src/raytrace.rs:151-186
"""
import ctypes as C
import os

import numpy as np

from . import abi

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_EARTHMAP = os.path.join(_ROOT, "assets", "earthmap.ppm")


def load_earthmap(path=None):
    """Decoded RGB8 texels of the reference's earthmap.jpg (1024x512), shipped as a binary PPM so that every host
    sees the same bytes (jpeg decoders differ by +-1 LSB; SURVEY hard part 8).  Returns (H, W, 3) uint8."""
    path = path or os.environ.get("RT_EARTHMAP") or DEFAULT_EARTHMAP
    with open(path, "rb") as f:
        data = f.read()
    if data[:2] != b"P6":
        raise ValueError(f"{path}: expected a binary PPM (P6)")
    fields, pos = [], 2
    while len(fields) < 3:
        while data[pos:pos + 1].isspace():
            pos += 1
        if data[pos:pos + 1] == b"#":
            pos = data.index(b"\n", pos)
            continue
        end = pos
        while not data[end:end + 1].isspace():
            end += 1
        fields.append(int(data[pos:end]))
        pos = end
    w, h, maxval = fields
    if maxval != 255:
        raise ValueError("earthmap PPM must be 8-bit")
    return np.frombuffer(data, dtype=np.uint8, offset=pos + 1, count=w * h * 3).reshape(h, w, 3).copy()


def _stats_dict(stats):
    """Renderer.stats of the RtStats of one call"""
    return {"paths": stats.paths, "rays": stats.rays, "device_ms": stats.device_ms, "kernel_launches": stats.kernel_launches,
            "pipeline": stats.pipeline_used, "bvh_layout": stats.bvh_layout_used}


def _adaptive(noise_threshold, min_samples):
    """the RtAdaptive of an adaptive render, or None (a uniform render) when noise_threshold is None"""
    if noise_threshold is None:
        return None
    ad = abi.RtAdaptive()
    ad.noise_threshold, ad.min_samples = float(noise_threshold), int(min_samples)
    return ad


def _image_inputs(who, ins, subject="every input", plural=False):
    """the inputs of a denoise function, checked and made contiguous: torch tensors, float32 on one CUDA device, each of the
    shape [H, W, 3].  Errors read "<who>: <subject> must be ...", in the plural for a subject that names several inputs."""
    import torch
    a, s = ("", "s") if plural else ("a ", "")
    if not all(isinstance(t, torch.Tensor) for t in ins):
        raise TypeError(f"{who}: {subject} must be {a}torch tensor{s}")
    if any(t.dtype != torch.float32 or not t.is_cuda or t.device != ins[0].device for t in ins):
        raise ValueError(f"{who}: {subject} must be {a}float32 CUDA tensor{s} on one device")
    if ins[0].dim() != 3 or ins[0].shape[2] != 3 or any(t.shape != ins[0].shape for t in ins):
        raise ValueError(f"{who}: {subject} must have the shape [H, W, 3]")
    return [t.contiguous() for t in ins]


class GradientBackground:  # raytrace.rs:12-35
    kind = abi.RT_BG_GRADIENT


class BlackBackground:  # raytrace.rs:37-48
    kind = abi.RT_BG_BLACK


class RenderingParams:  # raytrace.rs:50-55
    def __init__(self, samples_per_pixel, image_height, image_width):
        self.samples_per_pixel = int(samples_per_pixel)
        self.image_height = int(image_height)
        self.image_width = int(image_width)


class RecursiveRayTracer:  # raytrace.rs:74-76
    def __init__(self, max_depth=50):
        self.max_depth = int(max_depth)


class SeedableRngator:  # rngator.rs:17-31 — on the device the seed keys the Philox render streams
    def __init__(self, seed):
        self.seed = int(seed) & 0xFFFFFFFFFFFFFFFF


class Camera:  # camera.rs:15-38: the seven inputs; the basis is derived inside the library in f64
    def __init__(self, lookfrom, lookat, vup, vfov, aspect_ratio, aperture, focus_dist, time0=0.0, time1=0.0):
        """time0/time1: shutter interval in [0, 1] of the motion-blur EXTENSION (the reference's camera has none: 0, 0)"""
        self.c = abi.RtCamera()
        for i in range(3):
            self.c.lookfrom[i], self.c.lookat[i], self.c.vup[i] = float(lookfrom[i]), float(lookat[i]), float(vup[i])
        self.c.vfov_deg, self.c.aspect_ratio = float(vfov), float(aspect_ratio)
        self.c.aperture, self.c.focus_dist = float(aperture), float(focus_dist)
        self.c.time0, self.c.time1 = float(time0), float(time1)


class SceneDescription:
    """What World::build produces here: the reference's object tree written down as an RtSceneDesc."""

    def __init__(self, ptr, n_draws=0, owned=True):
        self.ptr, self.n_draws, self._owned = ptr, n_draws, owned

    @property
    def desc(self):
        return self.ptr.contents

    def hash(self):
        out = (C.c_uint8 * 32)()
        abi.check(abi.load().rt_scene_hash(self.ptr, out))
        return bytes(out).hex()

    def __del__(self):
        try:
            if getattr(self, "_owned", False) and self.ptr:
                abi.load().rt_scene_desc_free(self.ptr)
                self.ptr = None
        except Exception:  # interpreter shutdown: the module globals may already be gone
            pass


class Scene:
    """A description flattened, BVH-built and resident on one GPU (rt_scene_create)."""

    def __init__(self, description, device=-1):
        self.description = description  # keep alive for sub-tree queries by the caller
        self.device = int(device)  # -1: the current device
        h = C.c_void_p()
        abi.check(abi.load().rt_scene_create(description.ptr, int(device), C.byref(h)))
        self.handle = h

    def info(self):
        a, b, c, d = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
        abi.check(abi.load().rt_scene_info(self.handle, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return {"prims": a.value, "bvh_nodes": b.value, "media": c.value, "device_bytes": d.value}

    def build_info(self):
        a, b, c = C.c_int32(), C.c_float(), C.c_int32()
        abi.check(abi.load().rt_scene_build_info(self.handle, C.byref(a), C.byref(b), C.byref(c)))
        return {"built_on_device": bool(a.value), "build_ms": b.value, "depth": c.value}

    def close(self):
        if self.handle:
            abi.load().rt_scene_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class World:  # worlds.rs:14-19
    def __init__(self, name):
        self._name = name
        self._info = abi.RtWorldInfo()
        abi.check(abi.load().rt_world_info(name.encode(), C.byref(self._info)))

    def name(self):
        return self._name

    def camera(self):
        return {"lookfrom": tuple(self._info.lookfrom), "lookat": tuple(self._info.lookat),
                "field_of_view": self._info.vfov_deg}

    def background(self):
        return GradientBackground() if self._info.background_kind == abi.RT_BG_GRADIENT else BlackBackground()

    def build(self, seed, earthmap=None):
        """World::build with rng = Pcg64::seed_from_u64(seed) (main.rs:185); returns a SceneDescription."""
        ptr, draws = C.POINTER(abi.RtSceneDesc)(), C.c_uint64()
        earth, ew, eh = None, 0, 0
        if self._info.needs_earthmap:
            img = load_earthmap() if earthmap is None else np.ascontiguousarray(earthmap, dtype=np.uint8)
            eh, ew = img.shape[:2]
            earth = img.ctypes.data_as(C.c_void_p)
            self._keep = img
        abi.check(abi.load().rt_world_build(self._name.encode(), int(seed) & 0xFFFFFFFFFFFFFFFF, earth, ew, eh,
                                            C.byref(ptr), C.byref(draws)))
        return SceneDescription(ptr, draws.value)


def worlds():  # worlds.rs:471-484, same order
    lib = abi.load()
    return [World(lib.rt_world_name(i).decode()) for i in range(lib.rt_world_count())]


class Renderer:  # raytrace.rs:137-198
    def __init__(self, camera, world, background, parameters, tracer, rng):
        if not isinstance(world, Scene):
            raise TypeError("world must be a Scene (a description resident on the GPU)")
        self.camera, self.world, self.background = camera, world, background
        self.parameters, self.tracer, self.rng = parameters, tracer, rng
        self.stats = None
        self.pipeline = abi.RT_PIPELINE_AUTO
        self.bvh_layout = 0  # 0 = auto, 2 = binary 32-byte-node BVH, 4 = 4-wide BVH (RtParams.bvh_layout)

    @classmethod
    def new_with_rng(cls, camera, world, background, parameters, tracer, rng):
        return cls(camera, world, background, parameters, tracer, rng)

    def _params(self):
        p = abi.RtParams()
        p.width, p.height = self.parameters.image_width, self.parameters.image_height
        p.samples_per_pixel, p.max_depth = self.parameters.samples_per_pixel, self.tracer.max_depth
        p.seed, p.sample_begin, p.sample_count = self.rng.seed, 0, 0
        p.pipeline, p.device, p.bvh_layout = self.pipeline, -1, self.bvh_layout
        return p

    def render_arrays(self, logger=None, want_accum=True):
        """One rt_render call with HOST buffers.  Returns (rgb int32 [H,W,3], accum float32 [H,W,3] or None);
        row 0 is the bottom row.  `logger(j, H)` is called on this thread once per row index, as Renderer::render does
        (raytrace.rs:182), paced by the device's progress."""
        p = self._params()
        h, w = p.height, p.width
        rgb = np.empty((h, w, 3), dtype=np.int32)
        accum = np.empty((h, w, 3), dtype=np.float32) if want_accum else None
        cb = abi.RtProgressFn(lambda row, total, user: logger(row, total)) if logger else abi.RtProgressFn()
        stats = abi.RtStats()
        abi.check(abi.load().rt_render(self.world.handle, C.byref(self.camera.c), C.byref(p),
                                       accum.ctypes.data_as(C.c_void_p) if want_accum else None,
                                       rgb.ctypes.data_as(C.c_void_p), cb, None, C.byref(stats)))
        self.stats = _stats_dict(stats)
        return rgb, accum

    def render_adaptive(self, noise_threshold, min_samples=16, logger=None):
        """EXTENSION: noise-threshold adaptive sampling (rt_render_adaptive).  Every pixel gets samples until the standard
        error of its tonemapped value is at most `noise_threshold` in every channel (or the channel saturates), at least
        `min_samples` and at most parameters.samples_per_pixel.  Returns (rgb int32 [H,W,3], samples int32 [H,W],
        accum_fixed uint64 [H,W,3], moment2_fixed uint64 [H,W,3]) with row 0 at the bottom; the sums are in
        1 / RT_ACCUM_FIXED_ONE and 1 / RT_MOMENT2_FIXED_ONE units.  logger(j, H) as in render_arrays, paced by rounds."""
        p = self._params()
        h, w = p.height, p.width
        rgb = np.empty((h, w, 3), dtype=np.int32)
        samples = np.empty((h, w), dtype=np.int32)
        accum = np.empty((h, w, 3), dtype=np.uint64)
        moment2 = np.empty((h, w, 3), dtype=np.uint64)
        ad = _adaptive(noise_threshold, min_samples)
        cb = abi.RtProgressFn(lambda row, total, user: logger(row, total)) if logger else abi.RtProgressFn()
        stats = abi.RtStats()
        abi.check(abi.load().rt_render_adaptive(self.world.handle, C.byref(self.camera.c), C.byref(p), C.byref(ad),
                                                rgb.ctypes.data, samples.ctypes.data, accum.ctypes.data, moment2.ctypes.data,
                                                cb, None, C.byref(stats)))
        self.stats = _stats_dict(stats)
        return rgb, samples, accum, moment2

    def render_denoised(self, noise_threshold=None, min_samples=16, logger=None, guide=None, **denoise_options):
        """EXTENSION: a render through the moments family, then the variance-guided non-local-means filter (rt_render_denoised).
        noise_threshold None: a uniform render of parameters.samples_per_pixel (>= 2); else adaptive sampling as in
        render_adaptive.  denoise_options: search_radius, patch_radius, k, alpha (see `denoise`).  guide: None, or a dict of
        k_feature, tau and feature_samples (each optional; defaults RT_GUIDE_DEFAULT_*) for the feature-guided filter
        (rt_render_denoised_guided, see `denoise_guided`).  Returns (rgb int32 [H,W,3], to_rgb of the filtered means;
        denoised float32 [H,W,3], the filtered means), row 0 at the bottom."""
        p = self._params()
        h, w = p.height, p.width
        rgb = np.empty((h, w, 3), dtype=np.int32)
        out = np.empty((h, w, 3), dtype=np.float32)
        ad = _adaptive(noise_threshold, min_samples)
        cb = abi.RtProgressFn(lambda row, total, user: logger(row, total)) if logger else abi.RtProgressFn()
        stats = abi.RtStats()
        if guide is None:
            abi.check(abi.load().rt_render_denoised(self.world.handle, C.byref(self.camera.c), C.byref(p), C.byref(ad) if ad else None,
                                                    C.byref(denoise_options_struct(**denoise_options)), rgb.ctypes.data, out.ctypes.data,
                                                    cb, None, C.byref(stats)))
        else:
            abi.check(abi.load().rt_render_denoised_guided(self.world.handle, C.byref(self.camera.c), C.byref(p),
                                                           C.byref(ad) if ad else None, C.byref(denoise_options_struct(**denoise_options)),
                                                           C.byref(guide_struct(**guide)), rgb.ctypes.data, out.ctypes.data, cb, None,
                                                           C.byref(stats)))
        self.stats = _stats_dict(stats)
        return rgb, out

    def render_denoised_dual(self, noise_threshold=None, min_samples=16, logger=None, guide=None, **denoise_options):
        """EXTENSION: dual-buffer cross-filtered denoising with a per-pixel error estimate (rt_render_denoised_dual; the definition
        is in include/rt_b200.h).  Each range of samples is split into two halves; each half is filtered with weights from the
        other, and the two results give the output and an estimate of its variance.  noise_threshold None: a uniform render of
        parameters.samples_per_pixel (even, >= 4); else adaptive sampling whose stop rule judges the FILTERED value and its error
        estimate, with min_samples (even, >= 4).  guide and denoise_options as in render_denoised.  Returns (rgb int32 [H,W,3];
        denoised float32 [H,W,3], the filtered means; error float32 [H,W,3], the error estimate eps (a variance); samples int32
        [H,W], each pixel's count), row 0 at the bottom.  logger(j, H) as in render_adaptive."""
        p = self._params()
        h, w = p.height, p.width
        rgb = np.empty((h, w, 3), dtype=np.int32)
        out = np.empty((h, w, 3), dtype=np.float32)
        err = np.empty((h, w, 3), dtype=np.float32)
        samples = np.empty((h, w), dtype=np.int32)
        ad = _adaptive(noise_threshold, min_samples)
        cb = abi.RtProgressFn(lambda row, total, user: logger(row, total)) if logger else abi.RtProgressFn()
        stats = abi.RtStats()
        abi.check(abi.load().rt_render_denoised_dual(self.world.handle, C.byref(self.camera.c), C.byref(p), C.byref(ad) if ad else None,
                                                     C.byref(denoise_options_struct(**denoise_options)),
                                                     C.byref(guide_struct(**guide)) if guide is not None else None, rgb.ctypes.data,
                                                     out.ctypes.data, err.ctypes.data, samples.ctypes.data, cb, None, C.byref(stats)))
        self.stats = _stats_dict(stats)
        return rgb, out, err, samples

    def render_features(self, feature_samples=abi.RT_GUIDE_DEFAULT_FEATURE_SAMPLES):
        """EXTENSION: the first-event features of samples [0, feature_samples) of every pixel (rt_render_features_device; the
        definition is in include/rt_b200.h).  Returns numpy float32 (albedo, albedo_var, normal, normal_var), each [H, W, 3]
        with row 0 at the bottom: per channel the mean over the samples and the variance of that mean."""
        import torch
        p = self._params()
        p.sample_begin, p.sample_count = 0, int(feature_samples)
        dev = torch.device("cuda", self.world.device) if self.world.device >= 0 else torch.device("cuda")
        bufs = [torch.empty((p.height, p.width, 3), dtype=torch.float32, device=dev) for _ in range(4)]
        stats = abi.RtStats()
        abi.check(abi.load().rt_render_features_device(self.world.handle, C.byref(self.camera.c), C.byref(p),
                                                           *[b.data_ptr() for b in bufs], None, C.byref(stats)))
        self.stats = _stats_dict(stats)
        return tuple(b.cpu().numpy() for b in bufs)

    def render(self, logger=None):
        """Renderer::render: H rows of W (r, g, b) tuples, row j = 0 at the BOTTOM; logger(j, H) called H times."""
        rgb, _ = self.render_arrays(logger, want_accum=False)
        return [[tuple(int(c) for c in px) for px in row] for row in rgb]


def denoise_options_struct(search_radius=abi.RT_DENOISE_DEFAULT_SEARCH_RADIUS, patch_radius=abi.RT_DENOISE_DEFAULT_PATCH_RADIUS,
                           k=abi.RT_DENOISE_DEFAULT_K, alpha=abi.RT_DENOISE_DEFAULT_ALPHA):
    """the RtDenoise of the keyword arguments (defaults: the header's RT_DENOISE_DEFAULT_*)"""
    opt = abi.RtDenoise()
    opt.search_radius, opt.patch_radius, opt.k, opt.alpha = int(search_radius), int(patch_radius), float(k), float(alpha)
    return opt


def denoise(mean, var, search_radius=abi.RT_DENOISE_DEFAULT_SEARCH_RADIUS, patch_radius=abi.RT_DENOISE_DEFAULT_PATCH_RADIUS,
            k=abi.RT_DENOISE_DEFAULT_K, alpha=abi.RT_DENOISE_DEFAULT_ALPHA):
    """EXTENSION: the variance-guided non-local-means filter (rt_denoise_device) of a mean image and the variance of each mean,
    both contiguous CUDA float32 tensors [H, W, 3] on one device.  search_radius r: the window of candidates [-r, r]^2;
    patch_radius f: patches of (2f + 1)^2 pixels; k > 0: strength; alpha >= 0: how much of the variance the patch distance
    cancels.  The kernel computes in f32, so k^2 and alpha must be at most FLT_MAX (about 3.4e38).  Returns a new tensor [H, W, 3], computed on the tensors' device and ordered on its current stream."""
    import torch
    mean, var = _image_inputs("denoise", (mean, var), "mean and var", plural=True)
    out = torch.empty_like(mean)
    stream = torch.cuda.current_stream(mean.device).cuda_stream
    abi.check(abi.load().rt_denoise_device(mean.data_ptr(), var.data_ptr(), mean.shape[1], mean.shape[0],
                                           C.byref(denoise_options_struct(search_radius, patch_radius, k, alpha)), out.data_ptr(),
                                           mean.device.index, stream))
    return out


def guide_struct(k_feature=abi.RT_GUIDE_DEFAULT_K_FEATURE, tau=abi.RT_GUIDE_DEFAULT_TAU, feature_samples=abi.RT_GUIDE_DEFAULT_FEATURE_SAMPLES):
    """the RtGuide of the keyword arguments (defaults: the header's RT_GUIDE_DEFAULT_*)"""
    g = abi.RtGuide()
    g.k_feature, g.tau, g.feature_samples = float(k_feature), float(tau), int(feature_samples)
    return g


def denoise_guided(mean, var, albedo, albedo_var, normal, normal_var, k_feature=abi.RT_GUIDE_DEFAULT_K_FEATURE,
                   tau=abi.RT_GUIDE_DEFAULT_TAU, **options):
    """EXTENSION: the feature-guided non-local-means filter (rt_denoise_guided_device): `denoise` whose weights are also bounded by
    the first-event albedo and normal features (Renderer.render_features; the definition is in include/rt_b200.h).  All six
    inputs are contiguous CUDA float32 tensors [H, W, 3] on one device.  k_feature > 0: larger lets more across feature edges;
    tau > 0: the floor of a feature's normalisation.  The kernel forms 1 / (3 k_feature^2 tau) in f32 without subnormals, so
    3 k_feature^2, tau and their product must each be at least FLT_MIN (about 1.18e-38); 3 k_feature^2 beyond the f32 range
    ignores the feature.  options: search_radius, patch_radius, k, alpha as in `denoise`.  Returns a
    new tensor [H, W, 3], computed on the tensors' device and ordered on its current stream."""
    import torch
    ins = _image_inputs("denoise_guided", (mean, var, albedo, albedo_var, normal, normal_var))
    out = torch.empty_like(ins[0])
    stream = torch.cuda.current_stream(mean.device).cuda_stream
    abi.check(abi.load().rt_denoise_guided_device(*[t.data_ptr() for t in ins], mean.shape[1], mean.shape[0],
                                                  C.byref(denoise_options_struct(**options)), C.byref(guide_struct(k_feature, tau)),
                                                  out.data_ptr(), mean.device.index, stream))
    return out


def denoise_cross(mean_a, var_a, mean_b, var_b, features=None, k_feature=abi.RT_GUIDE_DEFAULT_K_FEATURE, tau=abi.RT_GUIDE_DEFAULT_TAU,
                  **options):
    """EXTENSION: the dual-buffer cross filter (rt_denoise_cross_device; the definition is in include/rt_b200.h) of two
    independent halves of a render, each a mean image and the variance of each mean.  Half A is filtered with weights computed
    from B and B with weights from A.  features: None (colour-only), or (albedo, albedo_var, normal, normal_var) as in
    `denoise_guided`, with k_feature and tau.  options: search_radius, patch_radius, k, alpha as in `denoise`.  Every input is
    a contiguous CUDA float32 tensor [H, W, 3] on one device.  Returns new tensors (out, err): the mean of the two filtered
    halves and the error estimate eps (an estimate of out's variance), computed on the tensors' device and ordered on its
    current stream."""
    import torch
    ins = (mean_a, var_a, mean_b, var_b) + (tuple(features) if features is not None else ())
    if features is not None and len(ins) != 8:
        raise ValueError("denoise_cross: features must be (albedo, albedo_var, normal, normal_var)")
    ins = _image_inputs("denoise_cross", ins)
    ptrs = [t.data_ptr() for t in ins] + [None] * (8 - len(ins))
    out, err = torch.empty_like(ins[0]), torch.empty_like(ins[0])
    stream = torch.cuda.current_stream(mean_a.device).cuda_stream
    guide = C.byref(guide_struct(k_feature, tau)) if features is not None else None
    abi.check(abi.load().rt_denoise_cross_device(*ptrs, mean_a.shape[1], mean_a.shape[0], C.byref(denoise_options_struct(**options)), guide,
                                                 out.data_ptr(), err.data_ptr(), mean_a.device.index, stream))
    return out, err


def to_ppm(rgb):
    """main.rs:144,175-179: 'P3\\nW H\\n255' then one 'r g b' line per pixel, rows in reverse j (top row first)."""
    h, w = rgb.shape[:2]
    lines = ["P3", f"{w} {h}", "255"]
    for j in range(h - 1, -1, -1):
        lines.extend(f"{int(r)} {int(g)} {int(b)}" for r, g, b in rgb[j])
    return "\n".join(lines) + "\n"
