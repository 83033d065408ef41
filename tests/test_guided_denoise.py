"""The first-event feature pass and the feature-guided mode of the non-local-means denoiser (an EXTENSION).

CPU part: the feature mean / variance conversion (bit for bit) and the feature distance of rt_denoise.cuh's host build
against numpy restatements; the struct size, the entry points and the CLI without a device.  GPU part: the feature pass
against a host-side rebuild of each path's first event, the guided filter against a numpy restatement of the definition in
include/rt_b200.h, its reduction to the colour-only filter, the glue of rt_render_denoised_guided bit for bit, argument
validation and quality guards."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import mu_lambda_raytracer_b200 as rt
from mu_lambda_raytracer_b200 import abi
import support as S
import test_denoise as TD

CLI = os.path.join(S.ROOT, "mu-lambda-raytracer_b200", "rt_main")


@pytest.fixture(scope="module")
def guide_emul(tmp_path_factory):
    """tests/emul/guide_emul.cpp: the feature functions of rt_denoise.cuh built for the host"""
    path = str(tmp_path_factory.mktemp("guide_emul") / "libguide_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-w", "-shared", "-o", path, os.path.join(S.ROOT, "tests", "emul", "guide_emul.cpp")])
    L = C.CDLL(path)
    L.emul_feature_mean_var.argtypes = [C.c_void_p, C.c_int64, C.c_uint32, C.c_void_p, C.c_void_p]
    L.emul_guide_distance.argtypes = [C.c_void_p] * 6 + [C.c_int64, C.c_float, C.c_float, C.c_void_p]
    L.emul_sizeof_rt_guide.restype = C.c_int64
    return L


def feature_mean_var_ref(f):
    """f: float32 [..., n] samples in ascending order -> (mean, variance of the mean) in f64, one rounding per operation, f32"""
    n = f.shape[-1]
    s1, s2 = np.zeros(f.shape[:-1]), np.zeros(f.shape[:-1])
    for k in range(n):
        x = f[..., k].astype(np.float64)
        s1, s2 = s1 + x, s2 + x * x
    mu = s1 / n
    var = np.maximum((s2 - n * (mu * mu)) / (n - 1.0), 0.0) if n > 1 else np.zeros_like(mu)
    return mu.astype(np.float32), (var / n).astype(np.float32)


def gradient2(m):
    """g_c(p)^2 of the header: central differences with clamped neighbours, f64"""
    m = m.astype(np.float64)
    H, W, _ = m.shape
    xs, ys = np.arange(W), np.arange(H)
    gx = (m[:, np.minimum(xs + 1, W - 1)] - m[:, np.maximum(xs - 1, 0)]) / 2
    gy = (m[np.minimum(ys + 1, H - 1)] - m[np.maximum(ys - 1, 0)]) / 2
    return gx * gx + gy * gy


def distance_ref(m_p, s_p, g2_p, m_q, s_q, kf, tau):
    """d(p, q) of one feature in f64 (arrays [..., 3])"""
    m_p, s_p, g2_p, m_q, s_q = (np.asarray(a, np.float64) for a in (m_p, s_p, g2_p, m_q, s_q))
    num = (m_p - m_q) ** 2 - (s_p + np.minimum(s_p, s_q))
    return (num / (kf * kf * np.maximum(np.maximum(tau, s_p), g2_p))).sum(axis=-1) / 3.0


def guided_ref(mu, v, feats, r, f, k, alpha, kf, tau):
    """the guided definition of include/rt_b200.h in f64 over the whole image (TD.nlm_ref plus the feature weights)"""
    from numpy.lib.stride_tricks import sliding_window_view
    mu, v = mu.astype(np.float64), v.astype(np.float64)
    (ma, sa, mn, sn) = feats
    g2 = [gradient2(ma), gradient2(mn)]
    H, W, _ = mu.shape
    yy, xx = np.mgrid[0:H, 0:W]
    wsum, acc = np.ones((H, W)), mu.copy()
    for dy in range(-r, r + 1):
        for dx in range(-r, r + 1):
            if dx == 0 and dy == 0:
                continue
            ys, xs = np.clip(yy + dy, 0, H - 1), np.clip(xx + dx, 0, W - 1)
            e = TD.term_ref(mu, v, mu[ys, xs], v[ys, xs], k, alpha).sum(axis=2)
            D = sliding_window_view(np.pad(e, f, mode="edge"), (2 * f + 1, 2 * f + 1)).mean(axis=(2, 3)) / 3.0
            w = np.exp(-np.maximum(D, 0.0))
            for (m, s), g in zip(((ma, sa), (mn, sn)), g2):
                w = np.minimum(w, np.exp(-np.maximum(distance_ref(m, s, g, m[ys, xs], s[ys, xs], kf, tau), 0.0)))
            w = w * ((yy + dy >= 0) & (yy + dy < H) & (xx + dx >= 0) & (xx + dx < W))
            wsum += w
            acc += w[..., None] * mu[ys, xs]
    return acc / wsum[..., None]


def guided_ref_pixels(mu, v, feats, pixels, r, f, k, alpha, kf, tau):
    """the same for a list of pixels (y, x) only"""
    mu, v = mu.astype(np.float64), v.astype(np.float64)
    (ma, sa, mn, sn) = feats
    H, W, _ = mu.shape
    d = np.arange(-r, r + 1)
    dy, dx = [a.ravel() for a in np.meshgrid(d, d, indexing="ij")]
    o = np.arange(-f, f + 1)
    oy, ox = [a.ravel() for a in np.meshgrid(o, o, indexing="ij")]
    out = []
    for py, px in pixels:
        xy, xx = np.clip(py + oy, 0, H - 1), np.clip(px + ox, 0, W - 1)
        yy, yx = np.clip(xy[None, :] + dy[:, None], 0, H - 1), np.clip(xx[None, :] + dx[:, None], 0, W - 1)
        e = TD.term_ref(mu[xy, xx][None], v[xy, xx][None], mu[yy, yx], v[yy, yx], k, alpha).sum(axis=2)
        w = np.exp(-np.maximum(e.mean(axis=1) / 3.0, 0.0))
        inside = (py + dy >= 0) & (py + dy < H) & (px + dx >= 0) & (px + dx < W)
        qy, qx = np.clip(py + dy, 0, H - 1), np.clip(px + dx, 0, W - 1)
        for m, s in ((ma, sa), (mn, sn)):
            mm = m.astype(np.float64)
            gx = (mm[py, min(px + 1, W - 1)] - mm[py, max(px - 1, 0)]) / 2
            gy = (mm[min(py + 1, H - 1), px] - mm[max(py - 1, 0), px]) / 2
            w = np.minimum(w, np.exp(-np.maximum(distance_ref(m[py, px], s[py, px], gx * gx + gy * gy, m[qy, qx], s[qy, qx], kf, tau), 0.0)))
        w[(dy == 0) & (dx == 0)] = 1.0
        w, qy, qx = w[inside], qy[inside], qx[inside]
        out.append((w[:, None] * mu[qy, qx]).sum(axis=0) / w.sum())
    return np.array(out)


def synthetic_features(H, W, seed):
    """albedo with a vertical edge, normals with a horizontal one, both noisy with per-pixel variances (some zero)"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    ma = np.where(xx < W // 3, 0.2, 0.8)[..., None] * np.array([1.0, 0.5, 0.25])
    mn = np.where(yy < H // 2, 1.0, 0.0)[..., None] * np.array([0.0, 1.0, 0.0]) + np.where(yy < H // 2, 0.0, 1.0)[..., None] * np.array([1.0, 0.0, 0.0])
    sa = 10.0 ** rng.uniform(-7, -2, (H, W, 3)) * (rng.random((H, W, 1)) > 0.3)
    sn = 10.0 ** rng.uniform(-7, -2, (H, W, 3)) * (rng.random((H, W, 1)) > 0.3)
    ma = ma + rng.standard_normal((H, W, 3)) * np.sqrt(sa)
    mn = mn + rng.standard_normal((H, W, 3)) * np.sqrt(sn)
    return tuple(a.astype(np.float32) for a in (ma, sa, mn, sn))


# ------------------------------------------------------------------------------------------------------------------ CPU
def test_feature_mean_var_matches_numpy_bit_for_bit(guide_emul):
    rng = np.random.default_rng(31)
    for n in (1, 2, 3, 16, 64):
        N = 50_000
        base = rng.choice([0.0, 0.3, 1.0, -0.7], (N, 1))
        f = (base + rng.choice([0.0, 1e-4, 0.1], (N, 1)) * rng.standard_normal((N, n))).astype(np.float32)
        f[: N // 10] = base[: N // 10]  # constant samples: the variance clamps to 0
        mu, v = np.zeros(N, np.float32), np.zeros(N, np.float32)
        guide_emul.emul_feature_mean_var(np.ascontiguousarray(f).ctypes.data, N, n, mu.ctypes.data, v.ctypes.data)
        want_mu, want_v = feature_mean_var_ref(f)
        assert np.array_equal(mu.view(np.uint32), want_mu.view(np.uint32)), n
        assert np.array_equal(v.view(np.uint32), want_v.view(np.uint32)), n
        if n > 1:
            assert (want_v > 0).mean() > 0.3
        else:
            assert not want_v.any()


def test_feature_distance_matches_numpy(guide_emul):
    rng = np.random.default_rng(32)
    N = 100_000
    m_p = rng.uniform(-1, 1, (N, 3)).astype(np.float32)
    m_q = np.where(rng.random((N, 1)) < 0.3, m_p, m_p + 0.1 * rng.standard_normal((N, 3))).astype(np.float32)
    s_p = (10.0 ** rng.uniform(-8, -1, (N, 3)) * (rng.random((N, 3)) > 0.2)).astype(np.float32)
    s_q = (10.0 ** rng.uniform(-8, -1, (N, 3)) * (rng.random((N, 3)) > 0.2)).astype(np.float32)
    gx = (rng.standard_normal((N, 3)) * 10.0 ** rng.uniform(-4, 0, (N, 1))).astype(np.float32)
    gy = (rng.standard_normal((N, 3)) * 10.0 ** rng.uniform(-4, 0, (N, 1))).astype(np.float32)
    for kf, tau in ((0.6, 1e-3), (0.3, 1e-4), (2.0, 1e-2)):
        got = np.zeros(N, np.float32)
        guide_emul.emul_guide_distance(*[a.ctypes.data for a in (m_p, s_p, m_q, s_q, gx, gy)], N, float(np.float32(3 * kf * kf)), float(np.float32(tau)), got.ctypes.data)
        g2 = gx.astype(np.float64) ** 2 + gy.astype(np.float64) ** 2
        want = distance_ref(m_p, s_p, g2, m_q, s_q, kf, np.float32(tau))
        # f32 tolerance: a few ulps of the sum of the absolute terms
        num = np.abs((m_p.astype(np.float64) - m_q) ** 2) + 2 * s_p
        scale = (num / (kf * kf * np.maximum(np.maximum(np.float32(tau), s_p), g2))).sum(axis=1) / 3.0
        assert np.all(np.abs(got - want) <= 2e-6 * scale + 1e-30), (kf, tau)
    # a k_feature whose square exceeds the f32 range: every distance is 0
    got = np.ones(N, np.float32)
    guide_emul.emul_guide_distance(*[a.ctypes.data for a in (m_p, s_p, m_q, s_q, gx, gy)], N, float("inf"), 1e-3, got.ctypes.data)
    assert not got.any()


def test_guided_pixel_restatement_matches_image_restatement():
    mu, v = TD.synthetic(23, 37, 5)
    feats = synthetic_features(23, 37, 6)
    for r, f in ((0, 1), (2, 0), (3, 1), (10, 3)):
        full = guided_ref(mu, v, feats, r, f, 0.45, 1.0, 0.6, 1e-3)
        pix = [(0, 0), (22, 36), (11, 18), (0, 36), (5, 2)]
        assert np.allclose(guided_ref_pixels(mu, v, feats, pix, r, f, 0.45, 1.0, 0.6, 1e-3), full[tuple(np.array(pix).T)], rtol=1e-12, atol=0)


def test_rt_guide_struct_size_matches_header(guide_emul):
    assert C.sizeof(abi.RtGuide) == guide_emul.emul_sizeof_rt_guide() == 24


def test_guided_entry_points_without_a_device():
    lib = abi.load()
    if lib.rt_device_count() > 0:
        pytest.skip("a CUDA device is present")
    p, opt, g = abi.RtParams(), rt.renderer.denoise_options_struct(), rt.renderer.guide_struct()
    assert lib.rt_render_features_device(None, None, C.byref(p), None, None, None, None, None, None) == abi.RT_ERR_NO_DEVICE
    assert lib.rt_denoise_guided_device(None, None, None, None, None, None, 0, 0, C.byref(opt), C.byref(g), None, -1, None) == abi.RT_ERR_NO_DEVICE
    assert lib.rt_render_denoised_guided(None, None, C.byref(p), None, C.byref(opt), C.byref(g), None, None, abi.RtProgressFn(), None,
                                         None) == abi.RT_ERR_NO_DEVICE
    assert b"no CPU path" in lib.rt_last_error()


def test_cli_rejects_denoise_guided_on_several_gpus():
    r = subprocess.run([CLI, "--world=cornell_smoke", "--denoise_guided", "--gpus=2"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                       timeout=120)
    assert r.returncode == 1 and "--denoise_guided" in r.stderr and r.stdout == ""


# ------------------------------------------------------------------------------------------------------------------ GPU
def _features(scene, cam, W, H, n, seed=42, begin=0, layout=0):
    """rt_render_features_device -> numpy (albedo, albedo_var, normal, normal_var), and the layout it used"""
    import torch
    bufs = [torch.full((H, W, 3), float("nan"), device="cuda") for _ in range(4)]
    p = TD._params(W, H, begin + n, seed, begin, n)
    p.bvh_layout = layout
    st = abi.RtStats()
    abi.check(abi.load().rt_render_features_device(scene.handle, C.byref(cam.c), C.byref(p), *[b.data_ptr() for b in bufs], None, C.byref(st)))
    torch.cuda.synchronize()
    return tuple(b.cpu().numpy() for b in bufs), st.bvh_layout_used


def _rebuild_first_events(world, scene, cam, W, H, n, layout, seed=42):
    """per (pixel, sample) on the host side: rt_generate_rays, rt_intersect_batch over the world (t_min = 0.001) through the
    layout, then the albedo from the description or rt_texture_value_batch.  Returns albedo, normal [H, W, n, 3], prim and
    whether the hit is textured [H, W, n]"""
    lib = abi.load()
    npix = W * H
    pixel = np.repeat(np.arange(npix, dtype=np.int32), n)
    sample = np.tile(np.arange(n, dtype=np.int32), npix)
    rays6 = np.zeros((len(pixel), 6), np.float32)
    us = np.zeros((len(pixel), 4), np.float32)
    abi.check(lib.rt_generate_rays(C.byref(cam.c), C.byref(TD._params(W, H, n, seed)), pixel.ctypes.data, sample.ctypes.data, len(pixel),
                                   rays6.ctypes.data, us.ctypes.data))
    rays = np.zeros((len(pixel), 8), np.float32)
    rays[:, :6], rays[:, 6], rays[:, 7] = rays6, 0.001, np.inf
    hits = (abi.RtHit * len(pixel))()
    abi.check(lib.rt_intersect_batch(scene.handle, -2 if layout == 4 else -1, rays.ctypes.data, len(pixel), hits))
    d = scene.description.desc
    albedo, normal = np.zeros((len(pixel), 3), np.float32), np.zeros((len(pixel), 3), np.float32)
    prim = np.array([h.prim for h in hits])
    textured = np.array([h.prim >= 0 and d.materials[h.material].texture >= 0 for h in hits])
    bg = (np.array(d.background_bottom[:]), np.array(d.background_top[:]))
    for i, h in enumerate(hits):
        if h.prim < 0:
            if d.background_kind == abi.RT_BG_GRADIENT:
                dd = rays6[i, 3:].astype(np.float64)
                t = 0.5 * (dd[1] / np.linalg.norm(dd) + 1.0)
                albedo[i] = (1 - t) * bg[0] + t * bg[1]
            continue
        normal[i] = h.normal[:]
        m = d.materials[h.material]
        if m.kind == abi.RT_MAT_DIELECTRIC:
            albedo[i] = 1.0
        elif m.texture < 0:
            albedo[i] = np.clip(np.array(m.albedo[:]), 0, 1)
        else:
            uvp = np.array([[h.u, h.v, *h.p[:]]], np.float32)
            c = np.zeros(3, np.float32)
            abi.check(lib.rt_texture_value_batch(scene.handle, m.texture, uvp.ctypes.data, 1, c.ctypes.data))
            albedo[i] = np.clip(c, 0, 1)
    return albedo.reshape(H, W, n, 3), normal.reshape(H, W, n, 3), prim.reshape(H, W, n), textured.reshape(H, W, n)


# The checker and Perlin-noise textures are steep functions of the hit point, and the feature kernel and the test entry points
# compute p = o + t d in kernels of their own (one FMA contraction may differ): measured on an NVIDIA B200 (1000 W), textured
# albedos of two_spheres and simple_light differ by up to 3.9e-5; untextured albedos and normals agree within 1e-5.
TEXTURE_TOL = 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["two_spheres", "earth", "cornell_box", "simple_light"])
def test_features_are_the_first_events(name):
    """media-free worlds: every (pixel, sample) rebuilt on the host side matches the pass (values within 1e-5), and the numpy
    mean and variance of the rebuilt samples match the pass's buffers"""
    world, scene, cam = TD._setup(name)
    W, H, n = 40, 30, 4
    (fa, fva, fn, fvn), layout = _features(scene, cam, W, H, n)
    albedo, normal, prim, textured = _rebuild_first_events(world, scene, cam, W, H, n, layout)
    assert (prim >= 0).mean() > 0.2
    # one sample at a time: the first event of sample s alone
    for s in range(n):
        (a1, va1, n1, vn1), _ = _features(scene, cam, W, H, 1, begin=s)
        assert not va1.any() and not vn1.any()
        err = np.abs(a1 - albedo[:, :, s]).max(axis=2)
        assert err[~textured[:, :, s]].max(initial=0) <= 1e-5, (name, s)
        assert err[textured[:, :, s]].max(initial=0) <= TEXTURE_TOL, (name, s, float(err.max()))
        assert np.abs(n1 - normal[:, :, s]).max() <= 1e-5, (name, s)
        assert np.array_equal(np.abs(n1).sum(axis=2) > 0, prim[:, :, s] >= 0)
    want = [feature_mean_var_ref(np.moveaxis(x, 2, 3)) for x in (albedo, normal)]
    for got, w in zip((fa, fva, fn, fvn), (want[0][0], want[0][1], want[1][0], want[1][1])):
        assert np.allclose(got, w, rtol=1e-5, atol=TEXTURE_TOL)
    scene.close()


@pytest.mark.gpu
def test_features_with_media():
    """cornell_smoke, one sample: every normal is 0 or a unit vector, every albedo a (clamped) material colour; two calls give
    the same bits, and the render layouts agree on the events"""
    world, scene, cam = TD._setup("cornell_smoke")
    W = H = 48
    (a, va, nrm, vn), layout = _features(scene, cam, W, H, 1)
    length = np.linalg.norm(nrm.astype(np.float64), axis=2)
    assert np.all((length == 0) | (np.abs(length - 1) < 1e-5))
    d = scene.description.desc
    colours = [d.materials[i].albedo[:] for i in range(d.n_materials)] + [d.textures[i].color[:] for i in range(d.n_textures)]
    colours = np.clip(np.array(colours + [[1.0, 1.0, 1.0], [0.0, 0.0, 0.0]]), 0, 1)
    dist = np.abs(a.reshape(-1, 1, 3).astype(np.float64) - colours[None]).max(axis=2).min(axis=1)
    assert dist.max() < 1e-6
    assert (length == 0).mean() > 0.05  # medium events (or misses) occur
    (a2, va2, n2, vn2), _ = _features(scene, cam, W, H, 1)
    for x, y in ((a, a2), (va, va2), (nrm, n2), (vn, vn2)):
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32))
    (a16, va16, n16, vn16), _ = _features(scene, cam, W, H, 16)
    assert np.isfinite(a16).all() and (va16 >= 0).all() and (vn16 > 0).any()
    scene.close()


def _guided_np(mu, v, feats, **kw):
    import torch
    t = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (mu, v, *feats)]
    out = rt.denoise_guided(*t, **kw)
    torch.cuda.synchronize()
    return out.cpu().numpy()


# Largest |device - restatement| / (|restatement| + 1e-3), f32 kernel against the f64 restatement.  Measured on an NVIDIA B200
# (1000 W): 0 (1x1), 1.3e-7 (2x3), 2.2e-6 (23x37), 3.5e-6 (48x64) over every case, 6.6e-7 over the sampled pixels of
# 3840x2160.  The bound is about thirty times the largest; a wrong feature tap or a wrong gradient moves the output by far
# more: the synthetic feature edges change weights of order 1.
GUIDED_REL_TOL = 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(1, 1), (2, 3), (23, 37), (48, 64)])
def test_guided_matches_numpy_restatement(H, W):
    mu, v = TD.synthetic(H, W, H * 1000 + W)
    feats = synthetic_features(H, W, H * 7 + W)
    worst = 0.0
    for r in (0, 1, 3, 10):
        for f in (0, 1, 3):
            for k, alpha, kf, tau in ((0.45, 1.0, 0.6, 1e-3), (1.0, 0.0, 0.3, 1e-4)):
                got = _guided_np(mu, v, feats, search_radius=r, patch_radius=f, k=k, alpha=alpha, k_feature=kf, tau=tau)
                want = guided_ref(mu, v, feats, r, f, k, alpha, kf, np.float32(tau))
                err = np.abs(got - want) / (np.abs(want) + 1e-3)
                worst = max(worst, float(err.max()))
                assert err.max() < GUIDED_REL_TOL, (r, f, k, alpha, kf, tau, float(err.max()))
    print(f"guided vs restatement {H}x{W}: worst relative error {worst:.3g}")


@pytest.mark.gpu
def test_guided_large_image_sampled_pixels():
    H, W = 2160, 3840
    mu, v = TD.synthetic(H, W, 11)
    feats = synthetic_features(H, W, 13)
    got = _guided_np(mu, v, feats, k_feature=0.6, tau=1e-3)
    rng = np.random.default_rng(12)
    pix = [(0, 0), (H - 1, W - 1), (0, W - 1), (H - 1, 0), (H // 2, W // 3)] + list(zip(rng.integers(0, H, 195), rng.integers(0, W, 195)))
    want = guided_ref_pixels(mu, v, feats, pix, 10, 3, 0.45, 1.0, 0.6, np.float32(1e-3))
    err = np.abs(got[tuple(np.array(pix).T)] - want) / (np.abs(want) + 1e-3)
    print(f"guided 3840x2160 sampled: worst relative error {err.max():.3g}")
    assert err.max() < GUIDED_REL_TOL


@pytest.mark.gpu
def test_guided_reduces_to_the_colour_filter():
    """constant features of zero variance, or k_feature = 1e30: the colour-only filter's output bit for bit"""
    mu, v = TD.synthetic(70, 90, 41)
    zero = np.zeros_like(mu)
    const = (np.full_like(mu, 0.5), zero, np.broadcast_to(np.array([0, 1, 0], np.float32), mu.shape).copy(), zero)
    feats = synthetic_features(70, 90, 42)
    for r, f in ((10, 3), (3, 0), (15, 7)):
        want = TD._denoise_np(mu, v, search_radius=r, patch_radius=f)
        for fe, kf in ((const, 0.6), (feats, 1e30)):
            got = _guided_np(mu, v, fe, search_radius=r, patch_radius=f, k_feature=kf)
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (r, f, kf)


@pytest.mark.gpu
def test_feature_edge_stops_averaging():
    """an albedo edge of zero variance between x = 39 and 40: changing the colour left of it does not change the output right of
    it.  Exceptions, by the definition: the one column whose gradient straddles the edge (x = 40: g^2 = 0.09 lets a weight of
    exp(-11) across), and with patches (f > 0) the colour weights of right-side candidates whose patches reach across, so
    that only x >= 40 + r + f is untouched.  Elsewhere k_feature 0.6 and tau 1e-3 give d = 1000, a weight of exactly 0 in f32."""
    H, W = 48, 96
    mu, v = TD.synthetic(H, W, 51)
    v[:] = np.maximum(v, 1e-3)  # strong colour noise: the colour filter alone would average across
    xx = np.arange(W)[None, :, None]
    albedo = np.where(xx < 40, 0.2, 0.8).astype(np.float32) * np.ones((H, W, 3), np.float32)
    zero = np.zeros_like(mu)
    feats = (albedo, zero, np.broadcast_to(np.array([0, 0, 1], np.float32), mu.shape).copy(), zero)
    mu2 = mu.copy()
    mu2[:, :40] += 0.3
    for f, first in ((0, 41), (3, 40 + 10 + 3)):
        a = _guided_np(mu, v, feats, patch_radius=f, k_feature=0.6, tau=1e-3)
        b = _guided_np(mu2, v, feats, patch_radius=f, k_feature=0.6, tau=1e-3)
        assert np.array_equal(a[:, first:].view(np.uint32), b[:, first:].view(np.uint32)), f
        assert not np.array_equal(a[:, :40], b[:, :40])
        c = TD._denoise_np(mu2, v, patch_radius=f)  # (the colour-only filter does mix across it)
        assert not np.array_equal(c[:, 40:], TD._denoise_np(mu, v, patch_radius=f)[:, 40:])


@pytest.mark.gpu
def test_denoise_guided_rejects_bad_arguments():
    import torch
    lib = abi.load()
    t = [torch.zeros(8, 8, 3, device="cuda") for _ in range(7)]
    ptr = [x.data_ptr() for x in t]

    def call(bufs=None, o=ptr[6], W=8, H=8, guide=None, **kw):
        g = rt.renderer.guide_struct(**(guide or {}))
        b = list(ptr[:6]) if bufs is None else bufs
        return lib.rt_denoise_guided_device(*b, W, H, C.byref(rt.renderer.denoise_options_struct(**kw)), C.byref(g), o, -1, None)

    assert call() == abi.RT_OK
    for i in range(6):
        assert call(bufs=ptr[:i] + [None] + ptr[i + 1:6]) == abi.RT_ERR_INVALID, i
        assert call(o=ptr[i]) == abi.RT_ERR_INVALID, i
    for bad in (dict(o=None), dict(W=0), dict(H=-1), dict(search_radius=16), dict(patch_radius=8), dict(k=0.0),
                dict(guide=dict(k_feature=0.0)), dict(guide=dict(k_feature=float("nan"))), dict(guide=dict(tau=0.0)),
                dict(guide=dict(tau=-1.0)), dict(guide=dict(tau=float("inf"))), dict(H=abi.RT_DENOISE_MAX_HEIGHT + 1, W=1)):
        assert call(**bad) == abi.RT_ERR_INVALID, bad
    assert lib.rt_denoise_guided_device(*ptr[:6], 8, 8, C.byref(rt.renderer.denoise_options_struct()), None, ptr[6], -1, None) == abi.RT_ERR_INVALID
    assert call(guide=dict(feature_samples=0)) == abi.RT_OK  # (feature_samples is the render's)
    with pytest.raises(ValueError):
        rt.denoise_guided(*[x.double() for x in t[:6]])


@pytest.mark.gpu
def test_render_features_rejects_bad_arguments():
    import torch
    world, scene, cam = TD._setup("cornell_smoke")
    lib = abi.load()
    t = [torch.zeros(16, 16, 3, device="cuda") for _ in range(4)]
    ptr = [x.data_ptr() for x in t]

    def call(p, bufs=ptr):
        return lib.rt_render_features_device(scene.handle, C.byref(cam.c), C.byref(p), *bufs, None, None)

    assert call(TD._params(16, 16, 4)) == abi.RT_OK
    for i in range(4):
        assert call(TD._params(16, 16, 4), ptr[:i] + [None] + ptr[i + 1:]) == abi.RT_ERR_INVALID
    assert call(TD._params(16, 16, 4), [ptr[0], ptr[0] + 4, ptr[2], ptr[3]]) == abi.RT_ERR_INVALID
    assert call(TD._params(16, 16, 4, begin=4)) == abi.RT_ERR_INVALID  # empty range
    assert call(TD._params(1, 16, 4)) == abi.RT_ERR_INVALID
    p = TD._params(16, 16, 4)
    p.bvh_layout = 3
    assert call(p) == abi.RT_ERR_INVALID
    assert lib.rt_render_features_device(scene.handle, None, C.byref(TD._params(16, 16, 4)), *ptr, None, None) == abi.RT_ERR_INVALID
    scene.close()


# ------------------------------------------------------------------------------------------------------------ the glue
GUIDE = dict(k_feature=0.6, tau=1e-3, feature_samples=8)  # (not the defaults: those run in the adaptive and CLI cases)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_smoke", "final_scene"])
def test_render_denoised_guided_uniform_is_the_chain(name):
    """features, moments, the numpy conversion, rt_denoise_guided_device, to_rgb"""
    world, scene, cam = TD._setup(name)
    W, H, spp = 72, 56, 24
    rows = []
    r = TD._renderer(world, scene, cam, W, H, spp)
    rgb, den = r.render_denoised(logger=lambda j, total: rows.append((j, total)), guide=GUIDE, search_radius=5, patch_radius=2)
    assert rows == [(j, H) for j in range(H)]
    assert r.stats["paths"] == W * H * spp and r.stats["device_ms"] > 0
    feats, _ = _features(scene, cam, W, H, GUIDE["feature_samples"])
    assert np.array_equal(np.stack(r.render_features(GUIDE["feature_samples"])).view(np.uint32), np.stack(feats).view(np.uint32))
    s1, s2 = TD._moments(scene, cam, W, H, spp)
    mu, v = TD.mean_var_ref(s1, s2, spp)
    want = _guided_np(mu, v, feats, search_radius=5, patch_radius=2, k_feature=GUIDE["k_feature"], tau=GUIDE["tau"])
    assert np.array_equal(den.view(np.uint32), want.view(np.uint32))
    assert np.array_equal(rgb, TD.to_rgb_ref(den.astype(np.float64)))
    # without `guide`: the colour-only entry point
    rgb0, den0 = TD._renderer(world, scene, cam, W, H, spp).render_denoised(search_radius=5, patch_radius=2)
    assert np.array_equal(den0.view(np.uint32), TD._denoise_np(mu, v, search_radius=5, patch_radius=2).view(np.uint32))
    scene.close()


@pytest.mark.gpu
def test_render_denoised_guided_adaptive_is_the_chain():
    world, scene, cam = TD._setup("cornell_smoke")
    W = H = 64
    r = TD._renderer(world, scene, cam, W, H, 128)
    rgb, den = r.render_denoised(0.02, 8, guide={})
    _, n, s1, s2 = TD._renderer(world, scene, cam, W, H, 128).render_adaptive(0.02, 8)
    assert len(np.unique(n)) >= 3 and r.stats["paths"] == int(n.sum())
    mu, v = TD.mean_var_ref(s1, s2, n[..., None])
    feats, _ = _features(scene, cam, W, H, abi.RT_GUIDE_DEFAULT_FEATURE_SAMPLES)
    want = _guided_np(mu, v, feats)
    assert np.array_equal(den.view(np.uint32), want.view(np.uint32))
    assert np.array_equal(rgb, TD.to_rgb_ref(den.astype(np.float64)))
    scene.close()


@pytest.mark.gpu
@pytest.mark.parametrize("adaptive", [False, True])
def test_cli_denoise_guided_ppm_matches_the_library(adaptive):
    args = ["--world=cornell_smoke", "--seed=42", "--aspect_ratio=1:1", "--image_width=48", "--samples_per_pixel=32", "--denoise_guided", "--stats"]
    if adaptive:
        args += ["--noise_threshold=0.02", "--min_samples=8"]
    r = subprocess.run([CLI, *args], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert "Done!" in r.stderr and '"mean_spp": ' in r.stderr
    world, scene, cam = TD._setup("cornell_smoke")
    rd = TD._renderer(world, scene, cam, 48, 48, 32)
    rgb, _ = rd.render_denoised(0.02 if adaptive else None, 8, guide={})
    assert rt.to_ppm(rgb) == r.stdout
    assert f'"paths": {rd.stats["paths"]},' in r.stderr
    rgb0, _ = TD._renderer(world, scene, cam, 48, 48, 32).render_denoised(0.02 if adaptive else None, 8)
    assert rt.to_ppm(rgb0) != r.stdout  # the guided filter is a different filter
    scene.close()


@pytest.mark.gpu
def test_render_denoised_guided_rejects_bad_arguments():
    world, scene, cam = TD._setup("cornell_smoke")
    lib = abi.load()

    def call(p, ad=None, guide=None, **kw):
        return lib.rt_render_denoised_guided(scene.handle, C.byref(cam.c), C.byref(p), C.byref(ad) if ad else None,
                                             C.byref(rt.renderer.denoise_options_struct(**kw)), C.byref(rt.renderer.guide_struct(**(guide or {}))),
                                             None, None, abi.RtProgressFn(), None, None)

    assert call(_p := TD._params(16, 16, 8)) == abi.RT_OK
    assert call(TD._params(16, 16, 1)) == abi.RT_ERR_INVALID
    assert call(TD._params(16, 16, 8, begin=2)) == abi.RT_ERR_INVALID
    assert call(TD._params(16, 16, 8), k=0.0) == abi.RT_ERR_INVALID
    for g in (dict(feature_samples=0), dict(feature_samples=-3), dict(k_feature=0.0), dict(tau=0.0), dict(tau=float("nan"))):
        assert call(_p, guide=g) == abi.RT_ERR_INVALID, g
    assert lib.rt_render_denoised_guided(scene.handle, C.byref(cam.c), C.byref(_p), None, C.byref(rt.renderer.denoise_options_struct()), None, None,
                                         None, abi.RtProgressFn(), None, None) == abi.RT_ERR_INVALID
    for pipeline in (abi.RT_PIPELINE_MEGAKERNEL, abi.RT_PIPELINE_WAVEFRONT):
        assert call(TD._params(16, 16, 8, pipeline=pipeline)) == abi.RT_ERR_UNSUPPORTED
    scene.close()


# ---------------------------------------------------------------------------------------------------------- quality guards
def _disc_error(name, W, H, spp, gt_spp):
    """display error of colour-only and guided denoising of one render against a high-spp ground truth on another seed"""
    world, scene, cam = TD._setup(name)
    r = TD._renderer(world, scene, cam, W, H, spp)
    _, col = r.render_denoised()
    _, gui = r.render_denoised(guide={})
    g1, _ = TD._moments(scene, cam, W, H, gt_spp, seed=7)
    gt = g1.astype(np.float64) * 2.0 ** -32 / gt_spp
    s1, s2 = TD._moments(scene, cam, W, H, spp)
    noisy, _ = TD.mean_var_ref(s1, s2, spp)
    disp = lambda x: np.sqrt(np.clip(x.astype(np.float64), 0.0, 1.0))  # noqa: E731
    err = {k: np.abs(disp(x) - disp(gt)).mean(axis=2) for k, x in (("noisy", noisy), ("colour", col), ("guided", gui))}
    scene.close()
    return world, cam, err


# Measured on an NVIDIA B200 (1000 W) with the default RtGuide: noise sphere 0.0390 guided against 0.0470 colour-only (ratio
# 0.83; 0.133 noisy); cornell_smoke 0.0212 against 0.0235 (ratio 0.90; 0.070 noisy).  The sums are integers and the filters
# deterministic, so these repeat exactly on the same build; the margins leave room for a change of the arithmetic.
NOISE_SPHERE_RATIO_BOUND = 0.9
SMOKE_RATIO_BOUND = 1.05


@pytest.mark.gpu
def test_guided_helps_on_the_noise_sphere():
    """final_scene 256^2 at 64 spp against 2048 spp: inside the Perlin-noise sphere's disc (2 287 pixels) the guided filter's
    mean display error is below NOISE_SPHERE_RATIO_BOUND times the colour-only filter's.  (At 128^2, with the earlier
    k_feature 0.6 and tau 1e-3, the guided filter was worse there: 0.090 against 0.054.)"""
    import sys
    sys.path.insert(0, os.path.join(S.ROOT, "tools"))
    import denoise_bench as DB
    world, cam, err = _disc_error("final_scene", 256, 256, 64, 2048)
    mask = DB.sphere_disc(world, *DB.TEXTURED_SPHERES["final_scene"]["noise_sphere"], 256, 256)
    col, gui = float(err["colour"][mask].mean()), float(err["guided"][mask].mean())
    print("noise sphere: mean display error colour", col, "guided", gui, "noisy", float(err["noisy"][mask].mean()), "pixels", int(mask.sum()))
    assert gui < NOISE_SPHERE_RATIO_BOUND * col, (gui, col)


@pytest.mark.gpu
def test_guided_no_worse_on_cornell_smoke():
    """cornell_smoke 128^2 at 64 spp against 4096 spp (media: normals are 0 at medium events): the guided filter's mean display
    error is at most SMOKE_RATIO_BOUND times the colour-only filter's"""
    _, _, err = _disc_error("cornell_smoke", 128, 128, 64, 4096)
    col, gui = float(err["colour"].mean()), float(err["guided"].mean())
    print("cornell_smoke: mean display error colour", col, "guided", gui, "noisy", float(err["noisy"].mean()))
    assert gui <= SMOKE_RATIO_BOUND * col, (gui, col)
