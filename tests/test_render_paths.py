"""The render kernels path by path against an f64 path tracer that follows the same Philox streams (path_reference.py).

Every pixel's fixed-point sum must equal the sum of exactly the right paths, in every pipeline, kernel instance and entry
point: a path dropped or traced twice at a launch or reservation boundary, a wrong Philox counter or a wrong pixel of a
pixel list moves a pixel's sum by a whole path, far beyond the per-path tolerance.

A pixel passes when |GPU sum - reference sum| <= paths x TOL_PATH (in 2^-32 units), or when one of its paths is "fragile":
it came within MARGIN (relative) of a branch threshold, where the f32 device may legitimately take the other branch.
Fragile pixels are excluded and must stay few.

Tolerances.  Worst per-path error measured on an NVIDIA B200 (1000 W power limit) over this file's GPU tests: 1.53e-6 in
the persistent, wavefront and megakernel pipelines (at 128 x 72), 1.34e-6 in the moments family, 1.5e-7 in the other
persistent variants and the wavefront at 4096 slots, 8.9e-8 in the adaptive render, 3.9e-9 in the launch-split cases (whose
paths are short).  TOL_PATH is 4x the worst.  The host build (tests/emul) differs from the reference by at most 3.2e-6 on
the CPU guards' views; its contraction differs from the device's.  At MARGIN = 1e-5 at most 0.1 % of paths were fragile;
fragile pixels were at most 0.4 % at 8 samples or fewer, 0.9 % in the adaptive render (up to 64 samples) and 2.6 % at 2048
samples per pixel.  The whole file runs in under 10 s on the GPU.
"""
import ctypes as C
import functools

import numpy as np
import pytest

import path_reference as R
import render_path_cases as K
import support as S
from mu_lambda_raytracer_b200 import abi
from mu_lambda_raytracer_b200 import renderer as rt

TOL_PATH = 6.2e-6  # 4x the worst per-path error measured on a B200 (module docstring)
MARGIN = 1e-5  # a path whose margin is below this is fragile
FRAGILE_PATHS = 1e-3  # at most this share of paths may be fragile


def fragile_pixel_bound(count):
    """the largest share of pixels that may hold a fragile path and be excluded: it grows with the paths per pixel (measured
    at most 0.94 % at 64 samples or fewer and 2.6 % at 2048, module docstring)"""
    return 0.01 if count <= 64 else 0.03
SEED = 0x5EED0000_00000042
END = abi.RT_MAX_SAMPLE_END


# ------------------------------------------------------------------------------------------------------------------ CPU
def _emul_scene(b):
    return S.EmulScene(C.pointer(b.desc))


def test_philox_known_answers_and_host_build():
    """Random123's known answers (kat_vectors, philox4x32_10) and the host build's philox4x32_10, bit for bit"""
    kat = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
           ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for ctr, key, want in kat:
        assert tuple(int(x) for x in R.philox(*ctr, *key)) == want
    rng = np.random.default_rng(1)
    ctr = rng.integers(0, 2 ** 32, size=(2000, 4), dtype=np.uint64)
    key = rng.integers(0, 2 ** 32, size=2, dtype=np.uint64)
    got = np.stack(R.philox(ctr[:, 0], ctr[:, 1], ctr[:, 2], ctr[:, 3], int(key[0]), int(key[1])), axis=1)
    L = S.emul()
    k = key.astype(np.uint32)
    for i in range(0, 2000, 7):
        c = ctr[i].astype(np.uint32)
        out = np.zeros(4, dtype=np.uint32)
        L.emul_philox(c.ctypes.data, k.ctypes.data, out.ctypes.data)
        assert got[i].tolist() == out.tolist()


def test_u32_to_unit_is_exact():
    """truncation to the 24 leading bits, x 2^-32: exactly the f32 value __uint2float_rz(x) * 2^-32 (the host build)"""
    x = np.concatenate([np.arange(0, 70000), (1 << np.arange(32)), (1 << np.arange(1, 33)) - 1,
                        np.random.default_rng(2).integers(0, 2 ** 32, 100000)]).astype(np.uint64)
    u = R.u32_to_unit(x)
    assert u.max() < 1.0 and u.min() == 0.0
    assert np.array_equal(u.astype(np.float32).astype(np.float64), u)  # an f32 value
    trunc = np.array([(int(v) >> max(int(v).bit_length() - 24, 0)) << max(int(v).bit_length() - 24, 0) for v in x[::50]], dtype=np.float64)
    assert np.array_equal(u[::50], trunc * 2.0 ** -32)
    assert R.u32_to_unit(np.array([0xFFFFFFFF], np.uint64))[0] == (2 ** 24 - 1) * 2.0 ** -24


@pytest.mark.parametrize("aperture", [0.0, 0.25])
def test_camera_rays_match_host_build(aperture):
    W, H = 37, 23
    cam = S.make_camera((1, 2, 9), (0.5, 1, 0), 35.0, W / H, aperture=aperture)
    p = abi.RtParams()
    p.width, p.height, p.samples_per_pixel, p.seed = W, H, 1, SEED
    rng = np.random.default_rng(3)
    pixel = rng.integers(0, W * H, 4000).astype(np.int32)
    sample = rng.integers(0, 2 ** 31 - 1, 4000).astype(np.int32)
    rays = np.zeros((4000, 6), np.float32)
    us = np.zeros((4000, 4), np.float32)
    S.emul().emul_generate_rays(C.byref(cam.c), C.byref(p), pixel.ctypes.data, sample.ctypes.data, 4000, rays.ctypes.data, us.ctypes.data)
    u = R.uniforms(pixel, sample, 0, 0, SEED)
    assert np.array_equal(u, us.astype(np.float64))
    o, d = R.camera_rays(R.device_camera(cam.c), W, H, pixel.astype(np.int64), u)
    assert np.abs(o - rays[:, :3]).max() <= 1e-6 * np.abs(o).max()
    assert (np.abs(d - rays[:, 3:]) <= 1e-6 * np.abs(d).max(axis=1, keepdims=True)).all()


def test_fixed_point_restatements():
    x = np.array([0.0, 2.0 ** -33, 2.0 ** -32, 1.5 * 2.0 ** -32, 0.3, 1.0, 4096.0, 8192.0, 2.0 ** 20, 2.0 ** 21, np.nan, -1.0], np.float32)
    q = R.radiance_fixed(x)
    assert q.tolist() == [0, 1, 1, 2, int(np.float32(0.3).astype(np.float64) * 2 ** 32), 2 ** 32, 2 ** 44, 2 ** 45, 2 ** 52, 2 ** 52, 0, 0]
    assert R.moment2_fixed(2 ** 32) == 2 ** 24 and R.moment2_fixed(2 ** 45) == 2 ** 48 and R.moment2_fixed(3) == 0


@pytest.mark.parametrize("name", list(K.MATRIX))
def test_scene_features_select_the_intended_instance(name):
    """the feature bits the flattener reports are the ones the scene is meant to have, and they pick the intended instance;
    the medium scenes' media are clear (the chain phase has work) and the general scene has more than four media"""
    fn, bits, inst = K.MATRIX[name]
    b, _ = fn()
    es = _emul_scene(b)
    assert es.features == bits, (bin(es.features), bin(bits))
    assert K.instance_of(es.features, es.n_media) == inst
    if name in ("boxes", "final", "all"):
        assert es.n_media == 1 and es.clear_media == 1
    assert (es.n_media > 4) == (name == "general")


@pytest.mark.parametrize("variant", ["spheres", "boxes", "final", "all", "general"])
def test_exact_scenes_select_the_intended_instance(variant):
    b, _ = K.exact_scene(1.0, variant)
    es = _emul_scene(b)
    assert K.instance_of(es.features, es.n_media) == variant


@functools.lru_cache(maxsize=None)
def _host_paths(name, W, H, begins):
    """per-path radiance of the host build (emul_render, one sample per call) and of the reference"""
    fn = K.MATRIX[name][0]
    b, view = fn()
    es = _emul_scene(b)
    cam = K.camera(view, W, H)
    sc = R.Scene(b)
    host, ref, rays = [], [], 0
    for s in begins:
        acc, r = es.render(cam, W, H, 1, max_depth=50, seed=SEED, sample_begin=s, fixed=True)
        host.append(acc.reshape(-1, 3).astype(np.float64) * 2.0 ** -32)
        ref.append(R.trace(sc, cam, W, H, np.arange(W * H), np.full(W * H, s), SEED, 50))
        rays += r
    return host, ref, rays


@pytest.mark.parametrize("name", list(K.MATRIX))
def test_reference_matches_host_build_path_by_path(name):
    """every robust path of the reference equals the host build's path within the per-path tolerance, and so does the ray
    count; fragile paths are rare"""
    host, ref, rays = _host_paths(name, 48, 32, (0, 7, 1000, END - 1))
    err = np.concatenate([np.abs(h - r.radiance).max(axis=1) for h, r in zip(host, ref)])
    margin = np.concatenate([r.margin for r in ref])
    robust = margin >= MARGIN
    assert 1.0 - robust.mean() <= FRAGILE_PATHS
    assert err[robust].max() <= TOL_PATH, err[robust].max()
    segs = sum(int(r.segments.sum()) for r in ref)
    assert abs(rays - segs) <= 50 * int((~robust).sum()), (rays, segs)


@pytest.mark.parametrize("view", ["floor", "matrix"])
@pytest.mark.parametrize("name", list(K.MATRIX))
def test_reference_detects_a_dropped_duplicated_or_shifted_sample(name, view):
    """Detection power.  A pixel holds samples [7, 9).  Three edits of that sum: drop sample 8, count sample 7 twice, or hold
    [8, 10) instead (every sample shifted by one).  Each must move the pixel by at least 50 pixel tolerances (50 x 2 x
    TOL_PATH) on most robust pixels, so one path scheduled wrongly cannot hide in the tolerance.
    "matrix": the view and size the GPU tests check each scene at.  Pixels that see a light or the sky directly hold
    near-equal neighbouring samples there, so a shift moves at least 90 % of the pixels; a drop or a duplicate moves 95 %.
    "floor": a view down on the lit floor, where no pixel sees the sky or a light: every edit moves 95 %."""
    b, matrix_view = K.MATRIX[name][0]()
    if view == "matrix":
        W, H = 33, 17
        cam = K.camera(matrix_view, W, H)
    else:
        W, H = 24, 16
        cam = S.make_camera((0, 2.5, 6), (0, 0, 0), 30.0, W / H)
    sc = R.Scene(b)
    r7, r8, r9 = (R.trace(sc, cam, W, H, np.arange(W * H), np.full(W * H, k), SEED, 50) for k in (7, 8, 9))
    robust = (r7.margin >= MARGIN) & (r8.margin >= MARGIN) & (r9.margin >= MARGIN)
    edits = {"drop": (r8.radiance, 0.95), "duplicate": (r7.radiance, 0.95),
             "shift": (r9.radiance - r7.radiance, 0.90 if view == "matrix" else 0.95)}
    for what, (moved, share) in edits.items():
        far = np.abs(moved).max(axis=1) >= 50 * 2 * TOL_PATH
        assert far[robust].mean() >= share, (what, far[robust].mean())


# ------------------------------------------------------------------------------------------------------------------ GPU
# kernel variants: (pipeline, samples_per_item, bvh_layout, environment)
VARIANTS = {
    "persistent": (abi.RT_PIPELINE_PERSISTENT, 0, 0, {}),
    "generic": (abi.RT_PIPELINE_PERSISTENT, 0, 0, {"RT_PS_FEAT": "0"}),
    "variant1": (abi.RT_PIPELINE_PERSISTENT, 0, 0, {"RT_PS_VARIANT": "1"}),
    "binary": (abi.RT_PIPELINE_PERSISTENT, 0, 2, {}),
    "chain": (abi.RT_PIPELINE_PERSISTENT, 0, 0, {"RT_PS_CHAIN": "1"}),
    "chainq": (abi.RT_PIPELINE_PERSISTENT, 0, 0, {"RT_PS_CHAINQ": "1", "RT_PS_CHAINQ_LOG2_PATHS": "14", "RT_PS_CHAINQ_LOG2_CAP": "8"}),
    "gpu_bvh": (abi.RT_PIPELINE_PERSISTENT, 0, 0, {"RT_BVH_GPU_MIN": "2"}),
    "wavefront": (abi.RT_PIPELINE_WAVEFRONT, 0, 0, {}),
    "wavefront4096": (abi.RT_PIPELINE_WAVEFRONT, 0, 0, {"RT_WF_SLOTS": "4096"}),
    "mega": (abi.RT_PIPELINE_MEGAKERNEL, 0, 0, {}),
    "mega1": (abi.RT_PIPELINE_MEGAKERNEL, 1, 0, {}),
    "mega3": (abi.RT_PIPELINE_MEGAKERNEL, 3, 0, {}),
}
PIPELINES = ["persistent", "wavefront", "mega"]


def _cheap_scene():
    """paths of one to three segments: a lit Lambertian floor and a light under a gradient sky"""
    b = S.DescBuilder()
    items = [b.rect(abi.RT_NODE_XZRECT, -50, 50, -50, 50, 0.0, K._lam(b, 0.5, 0.6, 0.7)),
             b.sphere((0, 1, -3), 1.0, K._light(b, 2.0))]
    b.finish(b.group(abi.RT_NODE_LIST, items), background=abi.RT_BG_GRADIENT)
    return b, dict(lookfrom=(0, 1.5, 4), lookat=(0, 0.5, 0), vfov=60.0)


SCENES = dict({k: v[0] for k, v in K.MATRIX.items()}, cheap=_cheap_scene)


def _params(W, H, begin, count, depth=50, variant="persistent"):
    pipeline, spi, layout, _ = VARIANTS[variant]
    p = abi.RtParams()
    p.width, p.height, p.samples_per_pixel, p.max_depth, p.seed = W, H, min(begin + count, END), depth, SEED
    p.sample_begin, p.sample_count, p.pipeline, p.device, p.samples_per_item, p.bvh_layout = begin, count, pipeline, -1, spi, layout
    return p


def _scene(b, variant, monkeypatch):
    for k, v in VARIANTS[variant][3].items():
        monkeypatch.setenv(k, v)
    return rt.Scene(rt.SceneDescription(C.pointer(b.desc), owned=False))


def _accum(scene, cam, p):
    import torch
    s1 = torch.zeros(p.height, p.width, 3, dtype=torch.int64, device="cuda")
    st = abi.RtStats()
    abi.check(abi.load().rt_render_accumulate_fixed_device(scene.handle, C.byref(cam.c), C.byref(p), s1.data_ptr(), None, C.byref(st)))
    torch.cuda.synchronize()
    return s1.cpu().numpy().view(np.uint64).reshape(-1, 3), st


def _moments(scene, cam, p):
    import torch
    s1 = torch.zeros(p.height, p.width, 3, dtype=torch.int64, device="cuda")
    s2 = torch.zeros(p.height, p.width, 3, dtype=torch.int64, device="cuda")
    st = abi.RtStats()
    abi.check(abi.load().rt_render_moments_fixed_device(scene.handle, C.byref(cam.c), C.byref(p), s1.data_ptr(), s2.data_ptr(), None, C.byref(st)))
    torch.cuda.synchronize()
    return s1.cpu().numpy().view(np.uint64).reshape(-1, 3), s2.cpu().numpy().view(np.uint64).reshape(-1, 3), st


@functools.lru_cache(maxsize=None)
def _reference(name, W, H, begin, count, depth, pixels=None):
    """the reference's paths of samples [begin, begin + count) of `pixels` (all when None): radiance [n, count, 3],
    segments and margins [n, count]"""
    b, view = SCENES[name]()
    pix = np.arange(W * H) if pixels is None else np.asarray(pixels)
    P, Sm = np.meshgrid(pix, np.arange(begin, begin + count), indexing="ij")
    res = R.trace(R.Scene(b), K.camera(view, W, H), W, H, P.ravel(), Sm.ravel(), SEED, depth)
    n = len(pix)
    return res.radiance.reshape(n, count, 3), res.segments.reshape(n, count), res.margin.reshape(n, count)


def _check(label, gpu, rays, name, W, H, begin, count, depth, pixels=None):
    """gpu: fixed-point sums [n, 3] of the pixels; rays: stats.rays (None: not checked).  Returns the worst error per path."""
    rad, segs, margin = _reference(name, W, H, begin, count, depth, pixels)
    fragile = (margin < MARGIN).any(axis=1)
    ref = rad.sum(axis=1) * 2.0 ** 32
    err = np.abs(gpu.astype(np.float64) - ref).max(axis=1) * 2.0 ** -32 / count
    bad = ~fragile & (err > TOL_PATH)
    worst = float(err[~fragile].max()) if (~fragile).any() else 0.0
    print(f"MEASURE {label}: worst per-path error {worst:.3e}, fragile pixels {fragile.mean():.2e}, fragile paths {(margin < MARGIN).mean():.2e}")
    assert not bad.any(), (label, np.flatnonzero(bad)[:10], err[bad][:10])
    assert (margin < MARGIN).mean() <= FRAGILE_PATHS
    assert fragile.mean() <= fragile_pixel_bound(count), (label, fragile.mean())
    if rays is not None:
        allowance = int(depth * (margin < MARGIN).sum())
        assert abs(int(rays) - int(segs.sum())) <= allowance, (label, int(rays), int(segs.sum()))
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("name", list(K.MATRIX))
def test_every_instance_sums_the_right_paths(name, variant, monkeypatch):
    """every kernel the library can dispatch to, on every scene of the matrix, at 33 x 17 and samples [7, 13)"""
    if variant in ("chain", "chainq") and name == "spheres":
        pytest.skip("no clear medium: the variant is not taken")
    if variant == "chainq" and name == "general":
        pytest.skip("the chain queues serve the fast media sampler only (want_chain_queues)")
    b, view = K.MATRIX[name][0]()
    scene = _scene(b, variant, monkeypatch)
    W, H, begin, count = 33, 17, 7, 6
    cam = K.camera(view, W, H)
    gpu, st = _accum(scene, cam, _params(W, H, begin, count, variant=variant))
    _check(f"{variant}/{name}", gpu, st.rays, name, W, H, begin, count, 50)
    _assert_variant_taken(variant, name, scene, st)
    scene.close()


def _assert_variant_taken(variant, name, scene, st):
    """what the library reports of the variant it ran.  The feature instance, RT_PS_FEAT, RT_PS_VARIANT, RT_PS_CHAIN,
    RT_WF_SLOTS and samples_per_item leave no trace in the stats; for those the condition the host code selects them on is
    checked where it depends on the scene (the chain phase needs a clear medium, test_scene_features_select_the_intended_instance)."""
    assert st.pipeline_used == VARIANTS[variant][0]
    if variant == "binary":
        assert st.bvh_layout_used == 2
    elif variant == "persistent":
        assert st.bvh_layout_used == 4
    assert scene.build_info()["built_on_device"] == (variant == "gpu_bvh")
    if variant == "chainq":  # per launch: reset + persistent kernel + chain reset + chain kernel, then drain rounds of 4
        assert st.kernel_launches >= 4 and st.kernel_launches % 2 == 0, st.kernel_launches
    elif st.pipeline_used == abi.RT_PIPELINE_PERSISTENT:
        assert st.kernel_launches == 2


@pytest.mark.gpu
@pytest.mark.parametrize("variant", PIPELINES)
@pytest.mark.parametrize("W,H", [(2, 2), (3, 5), (2, 257), (257, 2), (33, 17), (128, 72)])
def test_image_shapes(W, H, variant, monkeypatch):
    """fewer pixels than a warp (one reservation wraps the image several times), one-pixel-wide strips, a frame"""
    b, view = K.MATRIX["final"][0]()
    scene = _scene(b, variant, monkeypatch)
    cam = K.camera(view, W, H)
    count = 64 if W * H < 32 else 8
    gpu, st = _accum(scene, cam, _params(W, H, 0, count, variant=variant))
    _check(f"shape {W}x{H}/{variant}", gpu, st.rays, "final", W, H, 0, count, 50)
    scene.close()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", PIPELINES)
@pytest.mark.parametrize("depth", [0, 1, 2, 50])
def test_max_depth(depth, variant, monkeypatch):
    b, view = K.MATRIX["boxes"][0]()
    scene = _scene(b, variant, monkeypatch)
    W, H, count = 33, 17, 8
    cam = K.camera(view, W, H)
    gpu, st = _accum(scene, cam, _params(W, H, 0, count, depth=depth, variant=variant))
    if depth == 0:
        assert not gpu.any() and st.rays == 0
    _check(f"depth {depth}/{variant}", gpu, st.rays, "boxes", W, H, 0, count, depth)
    scene.close()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", PIPELINES + ["moments"])
@pytest.mark.parametrize("begin,count", [(0, 5), (7, 5), (END - 5, 5)])
def test_sample_ranges(begin, count, variant, monkeypatch):
    """sample_begin 0 and 7, and a range that ends exactly at 2^31 - 1, on every pipeline and the moments family"""
    b, view = K.MATRIX["spheres"][0]()
    scene = _scene(b, "persistent" if variant == "moments" else variant, monkeypatch)
    W, H = 33, 17
    cam = K.camera(view, W, H)
    if variant == "moments":
        gpu, _, st = _moments(scene, cam, _params(W, H, begin, count))
    else:
        gpu, st = _accum(scene, cam, _params(W, H, begin, count, variant=variant))
    _check(f"range {begin}+{count}/{variant}", gpu, st.rays, "spheres", W, H, begin, count, 50)
    scene.close()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", PIPELINES + ["moments"])
def test_one_path_per_pixel(variant, monkeypatch):
    """sample_count = 1 at several sample_begin values: every pixel holds exactly one path, so a wrong counter cannot hide in
    a sum over samples"""
    b, view = K.MATRIX["final"][0]()
    scene = _scene(b, "persistent" if variant == "moments" else variant, monkeypatch)
    W, H = 48, 32
    cam = K.camera(view, W, H)
    for begin in (0, 1, 31, 4097, END - 1):
        if variant == "moments":
            gpu, _, st = _moments(scene, cam, _params(W, H, begin, 1))
        else:
            gpu, st = _accum(scene, cam, _params(W, H, begin, 1, variant=variant))
        _check(f"one path at {begin}/{variant}", gpu, st.rays, "final", W, H, begin, 1, 50)
    scene.close()


MOMENTS_FAMILY = {"spheres": ("spheres", 0), "boxes": ("boxes", 0), "final": ("final", 0), "all": ("all", 0),
                  "wide-general": ("general", 0), "binary": ("final", 2), "binary-general": ("general", 2)}


@pytest.mark.gpu
@pytest.mark.parametrize("member", list(MOMENTS_FAMILY))
def test_moments_family(member, monkeypatch):
    """S1 against the reference, S2 against the sum of moment2_fixed of the reference's samples"""
    name, layout = MOMENTS_FAMILY[member]
    b, view = K.MATRIX[name][0]()
    scene = _scene(b, "persistent", monkeypatch)
    W, H, begin, count = 33, 17, 3, 6
    cam = K.camera(view, W, H)
    p = _params(W, H, begin, count)
    p.bvh_layout = layout
    s1, s2, st = _moments(scene, cam, p)
    assert st.bvh_layout_used == (layout or 4)
    _check(f"moments {member}", s1, st.rays, name, W, H, begin, count, 50)
    _check_moment2(f"moments {member}", s2, name, W, H, begin, count)
    scene.close()


@pytest.mark.gpu
def test_adaptive_render_sums_the_first_n_samples(monkeypatch):
    """rt_render_adaptive: each pixel's sums are the reference's over [0, n_i), n_i from the returned counts; the threshold
    stops pixels in several rounds, so the later rounds launch over pixel lists"""
    b, view = K.MATRIX["final"][0]()
    scene = _scene(b, "persistent", monkeypatch)
    W, H, cap, m = 40, 24, 64, 4
    cam = K.camera(view, W, H)
    r = rt.Renderer.new_with_rng(cam, scene, abi.RT_BG_GRADIENT, rt.RenderingParams(cap, H, W), rt.RecursiveRayTracer(50), rt.SeedableRngator(SEED))
    _, n, s1, s2 = r.render_adaptive(0.02, m)
    n, s1 = n.ravel(), s1.reshape(-1, 3)
    assert len(np.unique(n)) >= 3, np.unique(n)
    rad, _, margin = _reference("final", W, H, 0, cap, 50)
    take = np.arange(cap)[None, :] < n[:, None]
    ref = (rad * take[:, :, None]).sum(axis=1) * 2.0 ** 32
    fragile = ((margin < MARGIN) & take).any(axis=1)
    err = np.abs(s1.astype(np.float64) - ref).max(axis=1) * 2.0 ** -32 / n
    print(f"MEASURE adaptive: worst per-path error {err[~fragile].max():.3e}, fragile pixels {fragile.mean():.2e}")
    assert not (~fragile & (err > TOL_PATH)).any()
    assert fragile.mean() <= fragile_pixel_bound(cap)
    assert r.stats["paths"] == int(n.sum())
    scene.close()


@pytest.mark.gpu
def test_multi_gpu_sums_the_right_paths():
    n_dev = abi.load().rt_device_count()
    if n_dev < 2:
        pytest.skip("needs two GPUs")
    b, view = K.MATRIX["final"][0]()
    scenes = [rt.Scene(rt.SceneDescription(C.pointer(b.desc), owned=False), device=g) for g in range(2)]
    W, H, count = 33, 17, 9
    cam = K.camera(view, W, H)
    p = _params(W, H, 3, count)
    arr = (C.c_void_p * 2)(*[s.handle.value for s in scenes])
    accum = np.zeros((H, W, 3), np.float32)
    rgb = np.zeros((H, W, 3), np.int32)
    st = abi.RtStats()
    abi.check(abi.load().rt_render_multi(arr, 2, C.byref(cam.c), C.byref(p), accum.ctypes.data, rgb.ctypes.data, abi.RtProgressFn(), None, C.byref(st)))
    rad, _, margin = _reference("final", W, H, 3, count, 50)
    fragile = (margin < MARGIN).any(axis=1)
    ref = rad.sum(axis=1)
    err = np.abs(accum.reshape(-1, 3).astype(np.float64) - ref).max(axis=1) / count
    assert not (~fragile & (err > TOL_PATH + 1e-6 * np.abs(ref).max(axis=1))).any()
    assert fragile.mean() <= fragile_pixel_bound(count)
    for s in scenes:
        s.close()


# ---- launch splits, checked on sampled pixels.  Path numbers are sample-major (path = sample * npix + pixel), and every
# launch holds whole samples, so every launch boundary falls at pixel 0: the sampled pixels are the first and last few, the
# middle ones, and a seeded random set.
def _sampled_pixels(npix, n_random=24):
    pix = set(range(4)) | set(range(npix - 4, npix)) | set(range(npix // 2 - 3, npix // 2 + 4))
    pix.update(np.random.default_rng(5).integers(0, npix, n_random).tolist())
    return tuple(sorted(pix))


def _check_moment2(label, s2, name, W, H, begin, count, pixels=None):
    """S2 against the sum of moment2_fixed of the reference's samples, on the pixels without a fragile path"""
    rad, _, margin = _reference(name, W, H, begin, count, 50, pixels)
    robust = (margin >= MARGIN).all(axis=1)
    x = rad * 2.0 ** 32
    want2 = (np.minimum(x, 2.0 ** 44) ** 2 * 2.0 ** -40).sum(axis=1)
    allow = (2.0 * np.minimum(x, 2.0 ** 44) * TOL_PATH * 2.0 ** 32 * 2.0 ** -40 + 2.0).sum(axis=1) + 2.0 ** 24 * TOL_PATH ** 2 * count
    bad = robust[:, None] & (np.abs(s2.astype(np.float64) - want2) > allow)
    assert not bad.any(), (label, np.argwhere(bad)[:5])


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["persistent_callback", "persistent_2^33", "persistent_2^33+1", "mega", "moments_2^33+1"])
def test_launch_splits(case, monkeypatch):
    """Every split of a render into launches, with the launch count asserted.  The moments family splits at 2^33 / n_list
    samples per launch; rt_render_moments_fixed_device renders over the whole image (n_list = npix), and so does round 0 of
    an adaptive render.  A later adaptive round with a short pixel list splits only when n_list x its sample count exceeds
    2^33 paths, which no test can afford, so the split of the moments launch loop is checked at n_list = npix."""
    b, view = _cheap_scene()
    variant = "mega" if case == "mega" else "persistent"
    scene = _scene(b, variant, monkeypatch)
    if case == "persistent_callback":  # 2^29 / npix = 512 samples per launch: 512 + 512 + 76
        W = H = 1024
        spp, launches = 1100, 3 * 2 + 1
    elif "2^33" in case:  # 2^33 / npix = 2048 samples per launch; 2048 reaches the largest path number, 2^33 - 1
        W = H = 2048
        spp = 2048 if case == "persistent_2^33" else 2049
        launches = 2 if spp == 2048 else 4
    else:  # 2^28 / (2^20 padded pixels x 16 samples per item) = 16 items, 256 samples per launch: 256 + 256 + 88
        W = H = 1024
        spp, launches = 600, 3
    cam = K.camera(view, W, H)
    pixels = _sampled_pixels(W * H)
    if case == "persistent_callback":
        rows = []
        r = rt.Renderer.new_with_rng(cam, scene, abi.RT_BG_GRADIENT, rt.RenderingParams(spp, H, W), rt.RecursiveRayTracer(50), rt.SeedableRngator(SEED))
        r.pipeline = abi.RT_PIPELINE_PERSISTENT
        _, accum = r.render_arrays(logger=lambda j, n: rows.append(j))
        assert rows == list(range(H)) and r.stats["kernel_launches"] == launches
        sums = accum.reshape(-1, 3)[list(pixels)].astype(np.float64) * 2.0 ** 32
        rad, _, margin = _reference("cheap", W, H, 0, spp, 50, pixels)
        fragile = (margin < MARGIN).any(axis=1)
        ref = rad.sum(axis=1) * 2.0 ** 32
        err = np.abs(sums - ref).max(axis=1) * 2.0 ** -32
        ok = err <= spp * TOL_PATH + 2.0 ** -24 * np.abs(ref * 2.0 ** -32).max(axis=1)  # + the float32 rounding of the sum
        assert (ok | fragile).all()
        assert fragile.mean() <= fragile_pixel_bound(spp)
    elif case.startswith("moments"):
        s1, s2, st = _moments(scene, cam, _params(W, H, 0, spp))
        assert st.kernel_launches == launches, st.kernel_launches
        _check(case, s1[list(pixels)], None, "cheap", W, H, 0, spp, 50, pixels)
        _check_moment2(case, s2[list(pixels)], "cheap", W, H, 0, spp, pixels)
    else:
        gpu, st = _accum(scene, cam, _params(W, H, 0, spp, variant=variant))
        assert st.kernel_launches == launches, st.kernel_launches
        _check(case, gpu[list(pixels)], None, "cheap", W, H, 0, spp, 50, pixels)
    scene.close()


# ---- exact-valued accounting: every path's radiance is exactly E
def _exact_sums(variant, E, W, H, begin, count, monkeypatch):
    """a kernel variant on the spheres-only exact scene, or the default persistent pipeline on the exact scene that selects
    the instance `variant`"""
    kernel, content = (variant, "spheres") if variant in VARIANTS else ("persistent", variant)
    b, view = K.exact_scene(E, content)
    scene = _scene(b, kernel, monkeypatch)
    out = _accum(scene, K.camera(view, W, H), _params(W, H, begin, count, variant=kernel))
    scene.close()
    return out


EXACT_VARIANTS = [v for v in VARIANTS if v not in ("chain", "chainq")] + ["boxes", "final", "all", "general"]


@pytest.mark.gpu
@pytest.mark.parametrize("variant", EXACT_VARIANTS)
@pytest.mark.parametrize("W,H,begin,count", [(3, 5, 0, 37), (33, 17, 7, 11), (2, 257, END - 13, 13)])
def test_exact_accounting(variant, W, H, begin, count, monkeypatch):
    """every path ends on a light of emission E: every pixel sum is exactly count * q(E), one ray per path"""
    E = 0.8125
    q = int(R.radiance_fixed(np.float32(E)))
    gpu, st = _exact_sums(variant, E, W, H, begin, count, monkeypatch)
    assert (gpu == np.uint64(count * q)).all(), np.unique(gpu)
    assert st.rays == W * H * count and st.paths == W * H * count


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["spheres", "boxes", "final", "all", "general", "binary"])
def test_exact_accounting_moments(variant, monkeypatch):
    E = 1.5
    q = int(R.radiance_fixed(np.float32(E)))
    b, view = K.exact_scene(E, variant if variant != "binary" else "final")
    scene = _scene(b, "persistent", monkeypatch)
    W, H, begin, count = 33, 17, 5, 19
    cam = K.camera(view, W, H)
    p = _params(W, H, begin, count)
    p.bvh_layout = 2 if variant == "binary" else 0
    s1, s2, st = _moments(scene, cam, p)
    assert (s1 == np.uint64(count * q)).all() and (s2 == np.uint64(count * R.moment2_fixed(q))).all()
    assert st.rays == W * H * count
    scene.close()


@pytest.mark.gpu
def test_clamp_sums_to_2_63_and_tonemaps_to_255(monkeypatch):
    """E = 2^21 is clamped to 2^20 per sample: 2048 samples sum to exactly 2^63; the byte is 255"""
    b, view = K.exact_scene(2.0 ** 21, "spheres")
    scene = _scene(b, "persistent", monkeypatch)
    cam = K.camera(view, 2, 2)
    gpu, _ = _accum(scene, cam, _params(2, 2, 0, 2048))
    assert (gpu == np.uint64(2 ** 63)).all()
    r = rt.Renderer.new_with_rng(cam, scene, abi.RT_BG_GRADIENT, rt.RenderingParams(2048, 2, 2), rt.RecursiveRayTracer(50), rt.SeedableRngator(SEED))
    rgb, _ = r.render_arrays()
    assert (rgb == 255).all()
    scene.close()


@pytest.mark.gpu
def test_second_moment_cap(monkeypatch):
    """E = 8192 is capped in the square: each sample adds 2^48, and 2^16 - 1 samples sum to exactly 2^64 - 2^48"""
    b, view = K.exact_scene(8192.0, "spheres")
    scene = _scene(b, "persistent", monkeypatch)
    cam = K.camera(view, 2, 2)
    s1, s2, _ = _moments(scene, cam, _params(2, 2, 0, 2 ** 16 - 1))
    assert (s2 == np.uint64(2 ** 64 - 2 ** 48)).all() and (s1 == np.uint64((2 ** 16 - 1) * 2 ** 45)).all()
    scene.close()


@pytest.mark.gpu
def test_sample_range_beyond_2_31_is_rejected(monkeypatch):
    """a range that ends at 2^31 - 1 renders; one sample more is RT_ERR_INVALID on every entry point"""
    import torch
    b, view = K.exact_scene(1.0, "spheres")
    scene = _scene(b, "persistent", monkeypatch)
    cam = K.camera(view, 4, 4)
    lib = abi.load()
    buf = torch.zeros(4, 4, 3, dtype=torch.int64, device="cuda")
    buf2 = torch.zeros(4, 4, 3, dtype=torch.int64, device="cuda")
    for begin, count, rc in [(END - 4, 4, abi.RT_OK), (END - 4, 5, abi.RT_ERR_INVALID), (END, 1, abi.RT_ERR_INVALID)]:
        for variant in PIPELINES:
            p = _params(4, 4, begin, count, variant=variant)
            p.samples_per_pixel = 1
            assert lib.rt_render_accumulate_fixed_device(scene.handle, C.byref(cam.c), C.byref(p), buf.data_ptr(), None, None) == rc
            assert lib.rt_render(scene.handle, C.byref(cam.c), C.byref(p), None, None, abi.RtProgressFn(), None, None) == rc
        p = _params(4, 4, begin, count)
        p.samples_per_pixel = 1
        assert lib.rt_render_moments_fixed_device(scene.handle, C.byref(cam.c), C.byref(p), buf.data_ptr(), buf2.data_ptr(), None, None) == rc
        arr = (C.c_void_p * 1)(scene.handle.value)
        assert lib.rt_render_multi(arr, 1, C.byref(cam.c), C.byref(p), None, None, abi.RtProgressFn(), None, None) == rc
    torch.cuda.synchronize()
    scene.close()
