"""The variance-guided non-local-means denoiser (an EXTENSION: the reference has no denoiser).

CPU part: the conversion from fixed-point sums to (mean, variance of the mean) and one channel's term of the patch distance,
run through the host build of rt_denoise.cuh, against numpy restatements; the struct size, the entry points and the CLI
without a device.  GPU part: rt_denoise_device against a numpy restatement of the definition in include/rt_b200.h, its
properties, the glue of rt_render_denoised bit for bit, argument validation and a quality guard."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import mu_lambda_raytracer_b200 as rt
from mu_lambda_raytracer_b200 import abi
import support as S

CLI = os.path.join(S.ROOT, "mu-lambda-raytracer_b200", "rt_main")
EPS = 1e-10


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    """tests/emul/denoise_emul.cpp: the per-pixel functions of rt_denoise.cuh built for the host"""
    path = str(tmp_path_factory.mktemp("denoise_emul") / "libdenoise_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-w", "-shared", "-o", path, os.path.join(S.ROOT, "tests", "emul", "denoise_emul.cpp")])
    L = C.CDLL(path)
    L.emul_denoise_mean_var.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.emul_denoise_term.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_float, C.c_void_p]
    L.emul_sizeof_rt_denoise.restype = C.c_int64
    return L


def mean_var_ref(s1, s2, n):
    """mu = S1 2^-32 / n and v = max(0, (S2 2^-24 - n mu^2) / (n - 1)) / n in f64, one rounding per operation, then f32.
    s1, s2: uint64 [..., 3]; n: counts broadcastable to [..., 1]"""
    dn = np.asarray(n, np.float64)
    mu = s1.astype(np.float64) * 2.0 ** -32 / dn
    m2 = s2.astype(np.float64) * 2.0 ** -24
    var = np.maximum((m2 - dn * (mu * mu)) / (dn - 1.0), 0.0)
    return mu.astype(np.float32), (var / dn).astype(np.float32)


def term_ref(mu_x, v_x, mu_y, v_y, k, alpha):
    """one channel of e_d(x) in f64"""
    mu_x, v_x, mu_y, v_y = (np.asarray(a, np.float64) for a in (mu_x, v_x, mu_y, v_y))
    return ((mu_x - mu_y) ** 2 - alpha * (v_x + np.minimum(v_x, v_y))) / (EPS + k * k * (v_x + v_y))


def nlm_ref(mu, v, r, f, k, alpha):
    """the definition of include/rt_b200.h in f64: a loop over the offsets d, e_d on the whole image with y = clamp(x + d),
    the patch mean as a box filter over the image padded in edge mode (= e at clamp(p + o)), candidates outside skipped"""
    from numpy.lib.stride_tricks import sliding_window_view
    mu, v = mu.astype(np.float64), v.astype(np.float64)
    H, W, _ = mu.shape
    yy, xx = np.mgrid[0:H, 0:W]
    wsum, acc = np.ones((H, W)), mu.copy()
    for dy in range(-r, r + 1):
        for dx in range(-r, r + 1):
            if dx == 0 and dy == 0:
                continue
            ys, xs = np.clip(yy + dy, 0, H - 1), np.clip(xx + dx, 0, W - 1)
            e = term_ref(mu, v, mu[ys, xs], v[ys, xs], k, alpha).sum(axis=2)
            D = sliding_window_view(np.pad(e, f, mode="edge"), (2 * f + 1, 2 * f + 1)).mean(axis=(2, 3)) / 3.0
            w = np.exp(-np.maximum(D, 0.0)) * ((yy + dy >= 0) & (yy + dy < H) & (xx + dx >= 0) & (xx + dx < W))
            wsum += w
            acc += w[..., None] * mu[ys, xs]
    return acc / wsum[..., None]


def nlm_ref_pixels(mu, v, pixels, r, f, k, alpha):
    """the same definition for a list of pixels (y, x) only, vectorised over offsets and patch positions"""
    mu, v = mu.astype(np.float64), v.astype(np.float64)
    H, W, _ = mu.shape
    d = np.arange(-r, r + 1)
    dy, dx = [a.ravel() for a in np.meshgrid(d, d, indexing="ij")]
    o = np.arange(-f, f + 1)
    oy, ox = [a.ravel() for a in np.meshgrid(o, o, indexing="ij")]
    out = []
    for py, px in pixels:
        xy, xx = np.clip(py + oy, 0, H - 1), np.clip(px + ox, 0, W - 1)  # x = clamp(p + o)
        yy, yx = np.clip(xy[None, :] + dy[:, None], 0, H - 1), np.clip(xx[None, :] + dx[:, None], 0, W - 1)
        e = term_ref(mu[xy, xx][None], v[xy, xx][None], mu[yy, yx], v[yy, yx], k, alpha).sum(axis=2)  # [offsets, patch]
        w = np.exp(-np.maximum(e.mean(axis=1) / 3.0, 0.0))
        w[(dy == 0) & (dx == 0)] = 1.0
        inside = (py + dy >= 0) & (py + dy < H) & (px + dx >= 0) & (px + dx < W)
        w, qy, qx = w[inside], (py + dy)[inside], (px + dx)[inside]
        out.append((w[:, None] * mu[qy, qx]).sum(axis=0) / w.sum())
    return np.array(out)


def synthetic(H, W, seed):
    """edges plus noise; the variance spread over seven decades, and zero on a fifth of the pixels"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    base = np.where(xx < W // 2, 0.2, 0.9)[..., None] * np.array([1.0, 0.7, 0.4]) + np.where(yy < H // 3, 0.3, 0.0)[..., None]
    base = base + 0.05 * ((xx + yy) % 7 == 0)[..., None]
    v = 10.0 ** rng.uniform(-8, -1, (H, W, 3))
    v[rng.random((H, W)) < 0.2] = 0.0
    mu = np.maximum(base + rng.standard_normal((H, W, 3)) * np.sqrt(v), 0.0)
    return mu.astype(np.float32), v.astype(np.float32)


# ------------------------------------------------------------------------------------------------------------------ CPU
def test_mean_var_conversion_matches_numpy_bit_for_bit(emul):
    rng = np.random.default_rng(3)
    N = 300_000
    n = rng.choice([2, 3, 16, 64, 1000, 20000], N).astype(np.uint32)
    mu = rng.choice([0.0, 1e-7, 0.01, 0.5, 3.0, 40.0], N) * rng.uniform(0.5, 1.5, N)
    s1 = np.round(mu * n * 2.0 ** 32).astype(np.uint64)
    rel = rng.choice([0.0, 1e-13, 1e-3, 1.0, 30.0], N)
    s2 = np.round(mu * mu * (1.0 + rel) * n * 2.0 ** 24).astype(np.uint64)
    s2[: N // 8] = np.floor(s1[: N // 8].astype(np.float64) ** 2 * 2.0 ** -40 / n[: N // 8]).astype(np.uint64)  # S2 < n mu^2
    s2[N // 8: N // 4] = 0
    s1[-1000:], s2[-1000:] = 0, 0  # mu = 0
    got_mu, got_v = np.zeros(N, np.float32), np.zeros(N, np.float32)
    emul.emul_denoise_mean_var(s1.ctypes.data, s2.ctypes.data, n.ctypes.data, N, got_mu.ctypes.data, got_v.ctypes.data)
    want_mu, want_v = mean_var_ref(s1, s2, n)
    assert np.array_equal(got_mu.view(np.uint32), want_mu.view(np.uint32))
    assert np.array_equal(got_v.view(np.uint32), want_v.view(np.uint32))
    assert (want_v == 0).mean() > 0.2 and (want_v > 0).mean() > 0.3  # both sides of the clamp are exercised


def test_patch_term_matches_numpy(emul):
    rng = np.random.default_rng(4)
    N = 200_000
    mu_x, mu_y = (rng.choice([0.0, 0.01, 0.5, 2.0], N) * rng.uniform(0.5, 1.5, N)).astype(np.float32), np.zeros(N, np.float32)
    mu_y[:] = np.where(rng.random(N) < 0.3, mu_x, mu_x + rng.standard_normal(N).astype(np.float32) * 0.05)
    v_x = (10.0 ** rng.uniform(-9, 0, N) * (rng.random(N) > 0.1)).astype(np.float32)
    v_y = (10.0 ** rng.uniform(-9, 0, N) * (rng.random(N) > 0.1)).astype(np.float32)
    for k, alpha in ((0.45, 1.0), (0.45, 0.0), (1.0, 4.0), (0.2, 0.5)):
        k2 = np.float32(k * k)
        got = np.zeros(N, np.float32)
        emul.emul_denoise_term(mu_x.ctypes.data, v_x.ctypes.data, mu_y.ctypes.data, v_y.ctypes.data, N, float(alpha), float(k2), got.ctypes.data)
        want = term_ref(mu_x, v_x, mu_y, v_y, np.sqrt(np.float64(k2)), alpha)
        # f32 tolerance: a few ulps of the largest term of the numerator over the denominator
        d = mu_x.astype(np.float64) - mu_y
        scale = (d * d + alpha * (v_x + np.minimum(v_x, v_y))) / (EPS + k2 * (v_x.astype(np.float64) + v_y))
        assert np.all(np.abs(got - want) <= 1e-6 * scale + 1e-30), (k, alpha)


def test_pixel_restatement_matches_image_restatement():
    """the per-pixel restatement (used on the 3840 x 2160 input) is the image restatement"""
    mu, v = synthetic(23, 37, 5)
    for r, f in ((0, 1), (2, 0), (3, 1), (10, 3)):
        full = nlm_ref(mu, v, r, f, 0.45, 1.0)
        pix = [(0, 0), (22, 36), (11, 18), (0, 36), (5, 2)]
        assert np.allclose(nlm_ref_pixels(mu, v, pix, r, f, 0.45, 1.0), full[tuple(np.array(pix).T)], rtol=1e-12, atol=0)


def test_rt_denoise_struct_size_matches_header(emul):
    assert C.sizeof(abi.RtDenoise) == emul.emul_sizeof_rt_denoise() == 24


def test_entry_points_without_a_device():
    lib = abi.load()
    if lib.rt_device_count() > 0:
        pytest.skip("a CUDA device is present")
    p, opt = abi.RtParams(), rt.renderer.denoise_options_struct()
    assert lib.rt_denoise_device(None, None, 0, 0, C.byref(opt), None, -1, None) == abi.RT_ERR_NO_DEVICE
    assert lib.rt_render_denoised(None, None, C.byref(p), None, C.byref(opt), None, None, abi.RtProgressFn(), None, None) == abi.RT_ERR_NO_DEVICE
    assert b"no CPU path" in lib.rt_last_error()


def test_cli_rejects_denoise_on_several_gpus():
    r = subprocess.run([CLI, "--world=cornell_smoke", "--denoise", "--gpus=2"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120)
    assert r.returncode == 1 and "--denoise" in r.stderr and r.stdout == ""


# ------------------------------------------------------------------------------------------------------------------ GPU
def _denoise_np(mu, v, **kw):
    import torch
    out = rt.denoise(torch.from_numpy(mu).cuda(), torch.from_numpy(v).cuda(), **kw)
    torch.cuda.synchronize()
    return out.cpu().numpy()


# Largest |device - restatement| / (|restatement| + 1e-3), f32 kernel against the f64 restatement.  Measured on an NVIDIA B200
# (1000 W): 0 (1x1), 1.1e-7 (2x3), 1.9e-6 (23x37), 2.6e-6 (48x64) over every (r, f, k, alpha) case, 4.8e-7 over the sampled
# pixels of 3840x2160.  The bound is four times the largest of these; a wrong tap, a wrong clamp or a skipped candidate moves
# the output by far more (the weights of the synthetic edges are of order 1).
REL_TOL = 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(1, 1), (2, 3), (23, 37), (48, 64)])
def test_denoise_matches_numpy_restatement(H, W):
    """every (r, f) of {0, 1, 3, 10} x {0, 1, 3} (r = 10 is larger than the small images), and two strengths"""
    mu, v = synthetic(H, W, H * 1000 + W)
    worst = 0.0
    for r in (0, 1, 3, 10):
        for f in (0, 1, 3):
            for k, alpha in ((0.45, 1.0), (1.0, 0.0)):
                got = _denoise_np(mu, v, search_radius=r, patch_radius=f, k=k, alpha=alpha)
                want = nlm_ref(mu, v, r, f, k, alpha)
                err = np.abs(got - want) / (np.abs(want) + 1e-3)
                worst = max(worst, float(err.max()))
                assert err.max() < REL_TOL, (r, f, k, alpha, float(err.max()))
    print(f"denoise vs restatement {H}x{W}: worst relative error {worst:.3g}")


@pytest.mark.gpu
def test_denoise_large_image_sampled_pixels():
    """3840 x 2160 with the defaults: 200 sampled pixels (borders and corners included) against the per-pixel restatement"""
    H, W = 2160, 3840
    mu, v = synthetic(H, W, 11)
    got = _denoise_np(mu, v)
    rng = np.random.default_rng(12)
    pix = [(0, 0), (H - 1, W - 1), (0, W - 1), (H - 1, 0), (H // 2, W // 2 - 1)] + list(zip(rng.integers(0, H, 195), rng.integers(0, W, 195)))
    want = nlm_ref_pixels(mu, v, pix, 10, 3, 0.45, 1.0)
    err = np.abs(got[tuple(np.array(pix).T)] - want) / (np.abs(want) + 1e-3)
    print(f"denoise 3840x2160 sampled: worst relative error {err.max():.3g}")
    assert err.max() < REL_TOL


@pytest.mark.gpu
def test_denoise_properties():
    mu, v = synthetic(100, 130, 21)
    # r = 0: the input, bit for bit (whatever f)
    for f in (0, 3, 7):
        assert np.array_equal(_denoise_np(mu, v, search_radius=0, patch_radius=f).view(np.uint32), mu.view(np.uint32))
    # a constant image: the constant, to f32 rounding.  The bound is that of two f32 sums of up to 31^2 positive terms;
    # measured on an NVIDIA B200: 7.2e-6 with and without variance (0.3 is not a binary fraction, so even unit weights round)
    c = np.broadcast_to(np.array([0.3, 0.5, 3.0], np.float32), mu.shape).copy()
    for var in (np.zeros_like(v), v):
        out = _denoise_np(c, var, search_radius=15, patch_radius=7)
        print("constant image: largest relative deviation", float(np.abs(out / c - 1).max()))
        assert np.allclose(out, c, rtol=31 * 31 * 2.0 ** -24, atol=0), float(np.abs(out / c - 1).max())
    # two calls: the same bits
    a, b = _denoise_np(mu, v), _denoise_np(mu, v)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.gpu
def test_denoise_rejects_bad_arguments():
    import torch
    lib = abi.load()
    mu = torch.zeros(8, 8, 3, device="cuda")
    var = torch.zeros_like(mu)
    out = torch.zeros_like(mu)

    def call(m=mu.data_ptr(), v=var.data_ptr(), o=out.data_ptr(), W=8, H=8, **kw):
        return lib.rt_denoise_device(m, v, W, H, C.byref(rt.renderer.denoise_options_struct(**kw)), o, -1, None)

    assert call() == abi.RT_OK
    for bad in (dict(m=None), dict(v=None), dict(o=None), dict(W=0), dict(H=-1), dict(search_radius=-1), dict(search_radius=16),
                dict(patch_radius=-1), dict(patch_radius=8), dict(k=0.0), dict(k=-1.0), dict(k=float("nan")), dict(alpha=-0.1),
                dict(alpha=float("nan")), dict(o=mu.data_ptr()), dict(o=var.data_ptr() + 4 * 3 * 8 * 7), dict(H=abi.RT_DENOISE_MAX_HEIGHT + 1, W=1)):
        assert call(**bad) == abi.RT_ERR_INVALID, bad
    assert lib.rt_denoise_device(mu.data_ptr(), var.data_ptr(), 8, 8, None, out.data_ptr(), -1, None) == abi.RT_ERR_INVALID
    with pytest.raises(ValueError):
        rt.denoise(mu.double(), var.double())


# ------------------------------------------------------------------------------------------------------------ the glue
def _setup(name, aspect=1.0):
    world = rt.World(name)
    scene = rt.Scene(world.build(42))
    info = world.camera()
    cam = S.make_camera(info["lookfrom"], info["lookat"], info["field_of_view"], aspect)
    return world, scene, cam


def _params(W, H, spp, seed=42, begin=0, count=0, pipeline=abi.RT_PIPELINE_AUTO):
    p = abi.RtParams()
    p.width, p.height, p.samples_per_pixel, p.max_depth, p.seed = W, H, spp, 50, seed
    p.sample_begin, p.sample_count, p.pipeline, p.device = begin, count, pipeline, -1
    return p


def _renderer(world, scene, cam, W, H, spp, seed=42):
    return rt.Renderer.new_with_rng(cam, scene, world.background(), rt.RenderingParams(spp, H, W), rt.RecursiveRayTracer(50), rt.SeedableRngator(seed))


def _moments(scene, cam, W, H, spp, seed=42):
    import torch
    s1 = torch.zeros(H, W, 3, dtype=torch.int64, device="cuda")
    s2 = torch.zeros_like(s1)
    abi.check(abi.load().rt_render_moments_fixed_device(scene.handle, C.byref(cam.c), C.byref(_params(W, H, spp, seed)), s1.data_ptr(), s2.data_ptr(),
                                                        None, None))
    torch.cuda.synchronize()
    return s1.cpu().numpy().view(np.uint64), s2.cpu().numpy().view(np.uint64)


def to_rgb_ref(mean):
    x = np.clip(np.sqrt(mean), 0.0, 0.99999999)
    return (255.999 * x).astype(np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_smoke", "final_scene"])
def test_render_denoised_uniform_is_the_chain(name):
    """rt_render_denoised(adaptive = NULL) = rt_render_moments_fixed_device, the numpy conversion, rt_denoise_device, to_rgb"""
    world, scene, cam = _setup(name)
    W, H, spp = 72, 56, 24
    rows = []
    r = _renderer(world, scene, cam, W, H, spp)
    rgb, den = r.render_denoised(logger=lambda j, total: rows.append((j, total)), search_radius=5, patch_radius=2)
    assert rows == [(j, H) for j in range(H)]
    s1, s2 = _moments(scene, cam, W, H, spp)
    mu, v = mean_var_ref(s1, s2, spp)
    want = _denoise_np(mu, v, search_radius=5, patch_radius=2)
    assert np.array_equal(den.view(np.uint32), want.view(np.uint32))
    assert np.array_equal(rgb, to_rgb_ref(den.astype(np.float64)))
    assert r.stats["paths"] == W * H * spp and r.stats["device_ms"] > 0
    scene.close()


@pytest.mark.gpu
def test_render_denoised_adaptive_is_the_chain():
    """with an RtAdaptive: the same chain fed from rt_render_adaptive's sums and per-pixel counts"""
    world, scene, cam = _setup("cornell_smoke")
    W = H = 64
    r = _renderer(world, scene, cam, W, H, 128)
    rgb, den = r.render_denoised(0.02, 8)
    st = r.stats
    _, n, s1, s2 = _renderer(world, scene, cam, W, H, 128).render_adaptive(0.02, 8)
    assert len(np.unique(n)) >= 3 and st["paths"] == int(n.sum())
    mu, v = mean_var_ref(s1, s2, n[..., None])
    want = _denoise_np(mu, v)
    assert np.array_equal(den.view(np.uint32), want.view(np.uint32))
    assert np.array_equal(rgb, to_rgb_ref(den.astype(np.float64)))
    scene.close()


@pytest.mark.gpu
@pytest.mark.parametrize("adaptive", [False, True])
def test_cli_denoise_ppm_matches_the_library(adaptive):
    args = ["--world=cornell_smoke", "--seed=42", "--aspect_ratio=1:1", "--image_width=48", "--samples_per_pixel=32", "--denoise", "--stats"]
    if adaptive:
        args += ["--noise_threshold=0.02", "--min_samples=8"]
    r = subprocess.run([CLI, *args], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert "Done!" in r.stderr and '"mean_spp": ' in r.stderr
    world, scene, cam = _setup("cornell_smoke")
    rd = _renderer(world, scene, cam, 48, 48, 32)
    rgb, _ = rd.render_denoised(0.02 if adaptive else None, 8)
    assert rt.to_ppm(rgb) == r.stdout
    assert f'"paths": {rd.stats["paths"]},' in r.stderr
    scene.close()


@pytest.mark.gpu
def test_render_denoised_rejects_bad_arguments():
    world, scene, cam = _setup("cornell_smoke")
    lib = abi.load()

    def call(p, ad=None, **kw):
        return lib.rt_render_denoised(scene.handle, C.byref(cam.c), C.byref(p), C.byref(ad) if ad else None,
                                      C.byref(rt.renderer.denoise_options_struct(**kw)), None, None, abi.RtProgressFn(), None, None)

    def adaptive(t=0.01, m=4):
        ad = abi.RtAdaptive()
        ad.noise_threshold, ad.min_samples = t, m
        return ad

    assert call(_params(16, 16, 1)) == abi.RT_ERR_INVALID  # a uniform render needs two samples for a variance
    assert call(_params(16, 16, 8, begin=2)) == abi.RT_ERR_INVALID
    assert call(_params(16, 16, 8, count=4)) == abi.RT_ERR_INVALID
    assert call(_params(16, 16, 8, count=4), adaptive()) == abi.RT_ERR_INVALID
    assert call(_params(16, 16, 8), adaptive(m=1)) == abi.RT_ERR_INVALID
    assert call(_params(16, 16, 8), adaptive(t=float("nan"))) == abi.RT_ERR_INVALID
    assert call(_params(16, 16, 8), k=0.0) == abi.RT_ERR_INVALID
    assert call(_params(16, 16, 8), search_radius=16) == abi.RT_ERR_INVALID
    assert lib.rt_render_denoised(scene.handle, C.byref(cam.c), C.byref(_params(16, 16, 8)), None, None, None, None, abi.RtProgressFn(), None,
                                  None) == abi.RT_ERR_INVALID
    for pipeline in (abi.RT_PIPELINE_MEGAKERNEL, abi.RT_PIPELINE_WAVEFRONT):
        assert call(_params(16, 16, 8, pipeline=pipeline)) == abi.RT_ERR_UNSUPPORTED
        assert call(_params(16, 16, 8, pipeline=pipeline), adaptive()) == abi.RT_ERR_UNSUPPORTED
    assert call(_params(16, 16, 8)) == abi.RT_OK and call(_params(16, 16, 8), adaptive()) == abi.RT_OK
    scene.close()


# Measured on an NVIDIA B200 (1000 W): the largest per-channel shift of the frame-mean radiance is 1.21 %; see the docstring.
MEAN_SHIFT_BOUND = 0.015
# Measured: the denoised display RMSE is 0.34 of the noisy one's.
RMSE_RATIO_BOUND = 0.45


@pytest.mark.gpu
def test_denoiser_is_useful():
    """cornell_smoke 128^2 at 64 spp against a 4096-spp uniform ground truth on another seed: the display RMSE (gamma 2,
    clamped) of the denoised image is below the noisy one's, and the filter moves each channel's frame-mean radiance by less
    than MEAN_SHIFT_BOUND (relative).  Measured on an NVIDIA B200 (1000 W): display RMSE 0.1027 noisy, 0.0354 denoised
    (ratio 0.34; bound RMSE_RATIO_BOUND = 0.45); frame-mean shift 1.21 %, 1.19 %, 1.16 % (r, g, b; all darker; bound 1.5 %).
    The sums are integers and the filter is deterministic, so these values repeat exactly on the same build; the margins
    leave room for a change of the filter's arithmetic, not for a different filter."""
    world, scene, cam = _setup("cornell_smoke")
    W = H = 128
    r = _renderer(world, scene, cam, W, H, 64)
    _, den = r.render_denoised()
    s1, s2 = _moments(scene, cam, W, H, 64)
    noisy, _ = mean_var_ref(s1, s2, 64)
    g1, _ = _moments(scene, cam, W, H, 4096, seed=7)
    gt = g1.astype(np.float64) * 2.0 ** -32 / 4096
    disp = lambda x: np.sqrt(np.clip(x.astype(np.float64), 0.0, 1.0))  # noqa: E731
    rmse_noisy = float(np.sqrt(np.mean((disp(noisy) - disp(gt)) ** 2)))
    rmse_den = float(np.sqrt(np.mean((disp(den) - disp(gt)) ** 2)))
    shift = np.abs(den.astype(np.float64).mean(axis=(0, 1)) / noisy.astype(np.float64).mean(axis=(0, 1)) - 1.0)
    print("useful: display rmse noisy", rmse_noisy, "denoised", rmse_den, "frame-mean shift", shift.tolist())
    assert rmse_den < RMSE_RATIO_BOUND * rmse_noisy, (rmse_den, rmse_noisy)
    assert shift.max() < MEAN_SHIFT_BOUND, shift
    scene.close()
