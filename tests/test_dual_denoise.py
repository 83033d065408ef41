"""Dual-buffer cross-filtered denoising with a per-pixel error estimate, and adaptive sampling driven by it (an EXTENSION).

CPU part: the combination (out, eps) and the filtered stop rule of rt_denoise.cuh's host build against numpy restatements,
the entry points and the CLI without a device.  GPU part: the exactness of the split, the cross filter against a numpy
restatement of the definition in include/rt_b200.h, its exact reductions and swap symmetry, the glue of
rt_render_denoised_dual bit for bit (uniform, adaptive through a Python replay of the rounds, the CLI), argument validation
and quality guards."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import mu_lambda_raytracer_b200 as rt
from mu_lambda_raytracer_b200 import abi
import support as S
import test_denoise as TD
import test_guided_denoise as TG

CLI = os.path.join(S.ROOT, "mu-lambda-raytracer_b200", "rt_main")


@pytest.fixture(scope="module")
def dual_emul(tmp_path_factory):
    """tests/emul/dual_emul.cpp: the dual-buffer functions of rt_denoise.cuh built for the host"""
    path = str(tmp_path_factory.mktemp("dual_emul") / "libdual_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-w", "-ffp-contract=off", "-shared", "-o", path,
                           os.path.join(S.ROOT, "tests", "emul", "dual_emul.cpp")])
    L = C.CDLL(path)
    L.emul_dual.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.emul_filtered_pixel_done.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_void_p]
    return L


def dual_out_ref(fa, fb):
    """(F_A + F_B) / 2 in f32"""
    return ((np.float32(fa) + np.float32(fb)) * np.float32(0.5)).astype(np.float32)


def dual_error_ref(fa9, fb9):
    """eps from F_A, F_B at the nine neighbours ([..., 9], f32): the mean of ((F_A - F_B) / 2)^2, one f32 rounding per operation
    in neighbour order"""
    s = np.zeros(fa9.shape[:-1], np.float32)
    for k in range(9):
        d = (fa9[..., k] - fb9[..., k]) * np.float32(0.5)
        s = s + d * d
    return (s / np.float32(9.0)).astype(np.float32)


def filtered_done_ref(n, n_max, out, eps, t):
    """the filtered stop rule of include/rt_b200.h in f64, one rounding per operation; out, eps [..., 3]"""
    o = np.asarray(out, np.float32).astype(np.float64)
    se = np.sqrt(np.asarray(eps, np.float32).astype(np.float64))
    e = se / (2.0 * np.sqrt(np.maximum(o, 2.0 ** -16)))
    return (np.asarray(n) >= n_max) | ((e <= t) | (o - 3.0 * se >= 1.0)).all(axis=-1)


def box3_ref(x):
    """the mean over the 3 x 3 neighbourhood, neighbours clamped (f64, [H, W, 3])"""
    from numpy.lib.stride_tricks import sliding_window_view
    return sliding_window_view(np.pad(x, ((1, 1), (1, 1), (0, 0)), mode="edge"), (3, 3), axis=(0, 1)).mean(axis=(-2, -1))


def cross_ref(mu_w, v_w, mu_val, r, f, k, alpha, feats=None, kf=1.0, tau=1e-2):
    """the filter of include/rt_b200.h in f64 with the weights computed from (mu_w, v_w) (and the features) and the values
    of mu_val"""
    from numpy.lib.stride_tricks import sliding_window_view
    mu_w, v_w, mu_val = mu_w.astype(np.float64), v_w.astype(np.float64), mu_val.astype(np.float64)
    H, W, _ = mu_w.shape
    yy, xx = np.mgrid[0:H, 0:W]
    wsum, acc = np.ones((H, W)), mu_val.copy()
    g2 = [TG.gradient2(feats[0]), TG.gradient2(feats[2])] if feats is not None else None
    for dy in range(-r, r + 1):
        for dx in range(-r, r + 1):
            if dx == 0 and dy == 0:
                continue
            ys, xs = np.clip(yy + dy, 0, H - 1), np.clip(xx + dx, 0, W - 1)
            e = TD.term_ref(mu_w, v_w, mu_w[ys, xs], v_w[ys, xs], k, alpha).sum(axis=2)
            D = sliding_window_view(np.pad(e, f, mode="edge"), (2 * f + 1, 2 * f + 1)).mean(axis=(2, 3)) / 3.0
            w = np.exp(-np.maximum(D, 0.0))
            if feats is not None:
                for (m, s), g in zip(((feats[0], feats[1]), (feats[2], feats[3])), g2):
                    w = np.minimum(w, np.exp(-np.maximum(TG.distance_ref(m, s, g, m[ys, xs], s[ys, xs], kf, tau), 0.0)))
            w = w * ((yy + dy >= 0) & (yy + dy < H) & (xx + dx >= 0) & (xx + dx < W))
            wsum += w
            acc += w[..., None] * mu_val[ys, xs]
    return acc / wsum[..., None]


def dual_ref(mu_a, v_a, mu_b, v_b, r, f, k, alpha, feats=None, kf=1.0, tau=1e-2):
    """(F_A, F_B, out, eps) of the definition in f64"""
    fa = cross_ref(mu_b, v_b, mu_a, r, f, k, alpha, feats, kf, tau)
    fb = cross_ref(mu_a, v_a, mu_b, r, f, k, alpha, feats, kf, tau)
    return fa, fb, (fa + fb) / 2, box3_ref(((fa - fb) / 2) ** 2)


def cross_ref_pixels(mu_w, v_w, mu_val, pixels, r, f, k, alpha, feats=None, kf=1.0, tau=1e-2):
    """cross_ref for a list of pixels (y, x) only (TG.guided_ref_pixels with weights and values from different buffers)"""
    mu_w, v_w, mu_val = mu_w.astype(np.float64), v_w.astype(np.float64), mu_val.astype(np.float64)
    H, W, _ = mu_w.shape
    d = np.arange(-r, r + 1)
    dy, dx = [a.ravel() for a in np.meshgrid(d, d, indexing="ij")]
    o = np.arange(-f, f + 1)
    oy, ox = [a.ravel() for a in np.meshgrid(o, o, indexing="ij")]
    out = []
    for py, px in pixels:
        xy, xx = np.clip(py + oy, 0, H - 1), np.clip(px + ox, 0, W - 1)
        yy, yx = np.clip(xy[None, :] + dy[:, None], 0, H - 1), np.clip(xx[None, :] + dx[:, None], 0, W - 1)
        e = TD.term_ref(mu_w[xy, xx][None], v_w[xy, xx][None], mu_w[yy, yx], v_w[yy, yx], k, alpha).sum(axis=2)
        w = np.exp(-np.maximum(e.mean(axis=1) / 3.0, 0.0))
        inside = (py + dy >= 0) & (py + dy < H) & (px + dx >= 0) & (px + dx < W)
        qy, qx = np.clip(py + dy, 0, H - 1), np.clip(px + dx, 0, W - 1)
        if feats is not None:
            for m, s in ((feats[0], feats[1]), (feats[2], feats[3])):
                mm = m.astype(np.float64)
                gx = (mm[py, min(px + 1, W - 1)] - mm[py, max(px - 1, 0)]) / 2
                gy = (mm[min(py + 1, H - 1), px] - mm[max(py - 1, 0), px]) / 2
                w = np.minimum(w, np.exp(-np.maximum(TG.distance_ref(m[py, px], s[py, px], gx * gx + gy * gy, m[qy, qx], s[qy, qx], kf, tau), 0.0)))
        w[(dy == 0) & (dx == 0)] = 1.0
        w, qy, qx = w[inside], qy[inside], qx[inside]
        out.append((w[:, None] * mu_val[qy, qx]).sum(axis=0) / w.sum())
    return np.array(out)


def display(mean):
    """the displayed value of a radiance: gamma 2 of the clamped mean"""
    return np.sqrt(np.clip(np.asarray(mean, np.float64), 0.0, 1.0))


def synthetic_halves(H, W, seed):
    """two independent halves of one noisy image: the same edges, their own noise and variances"""
    mu_a, v_a = TD.synthetic(H, W, seed)
    mu_b, v_b = TD.synthetic(H, W, seed + 1)
    return mu_a, v_a, mu_b, v_b


# ------------------------------------------------------------------------------------------------------------------ CPU
def test_out_and_error_match_numpy_bit_for_bit(dual_emul):
    rng = np.random.default_rng(61)
    N = 200_000
    fa = (rng.choice([0.0, 1e-6, 0.02, 0.5, 3.0], (N, 1)) * rng.uniform(0.5, 1.5, (N, 9))).astype(np.float32)
    fb = np.where(rng.random((N, 9)) < 0.2, fa, fa * (1 + rng.choice([1e-7, 1e-3, 0.1], (N, 1)) * rng.standard_normal((N, 9)))).astype(np.float32)
    out, eps = np.zeros(N, np.float32), np.zeros(N, np.float32)
    dual_emul.emul_dual(fa.ctypes.data, fb.ctypes.data, N, out.ctypes.data, eps.ctypes.data)
    assert np.array_equal(out.view(np.uint32), dual_out_ref(fa[:, 4], fb[:, 4]).view(np.uint32))
    assert np.array_equal(eps.view(np.uint32), dual_error_ref(fa, fb).view(np.uint32))
    # A = B: out is the input and eps is 0; swapping A and B changes nothing
    dual_emul.emul_dual(fa.ctypes.data, fa.ctypes.data, N, out.ctypes.data, eps.ctypes.data)
    assert np.array_equal(out.view(np.uint32), fa[:, 4].view(np.uint32)) and not eps.any()
    o2, e2 = np.zeros(N, np.float32), np.zeros(N, np.float32)
    dual_emul.emul_dual(fa.ctypes.data, fb.ctypes.data, N, out.ctypes.data, eps.ctypes.data)
    dual_emul.emul_dual(fb.ctypes.data, fa.ctypes.data, N, o2.ctypes.data, e2.ctypes.data)
    assert np.array_equal(out.view(np.uint32), o2.view(np.uint32)) and np.array_equal(eps.view(np.uint32), e2.view(np.uint32))


def test_filtered_stop_rule_matches_numpy(dual_emul):
    rng = np.random.default_rng(62)
    N = 300_000
    n_max = 1024
    n = rng.choice([16, 32, 64, 512, 1024], N).astype(np.uint32)
    out = (rng.choice([0.0, 1e-6, 0.01, 0.3, 1.0, 5.0], (N, 1)) * rng.uniform(0.5, 1.5, (N, 3))).astype(np.float32)
    eps = (rng.choice([0.0, 1e-10, 1e-6, 1e-4, 1e-2, 1.0], (N, 1)) * rng.uniform(0.5, 1.5, (N, 3))).astype(np.float32)
    # exactly at the threshold t = 1/4: out = 1/4 gives e = sqrt(eps) = sqrt(1/16); and exactly saturated: out - 3 sqrt(eps) = 1
    out[:1000], eps[:1000] = 0.25, 0.0625
    out[1000:2000], eps[1000:2000] = 4.0, 1.0
    out[2000:3000], eps[2000:3000] = np.nextafter(np.float32(4.0), np.float32(0.0)), 1.0  # just below saturation
    for t in (0.0, 0.25, 0.01, 0.5):
        got = np.zeros(N, np.uint8)
        dual_emul.emul_filtered_pixel_done(n.ctypes.data, n_max, out.ctypes.data, eps.ctypes.data, N, t, got.ctypes.data)
        want = filtered_done_ref(n, n_max, out, eps, t)
        assert np.array_equal(got.astype(bool), want), t
        assert want[n == n_max].all() and 0 < want[n < n_max].mean() < 1
    assert filtered_done_ref(16, n_max, out[:1000], eps[:1000], 0.25).all() and not filtered_done_ref(16, n_max, out[:1], eps[:1], 0.2499).any()
    assert filtered_done_ref(16, n_max, out[1000:1001], eps[1000:1001], 0.0).all()
    assert not filtered_done_ref(16, n_max, out[2000:2001], eps[2000:2001], 0.0).any()


def test_dual_entry_points_without_a_device():
    lib = abi.load()
    if lib.rt_device_count() > 0:
        pytest.skip("a CUDA device is present")
    p, opt = abi.RtParams(), rt.renderer.denoise_options_struct()
    assert lib.rt_denoise_cross_device(*[None] * 8, 0, 0, C.byref(opt), None, None, None, -1, None) == abi.RT_ERR_NO_DEVICE
    assert lib.rt_render_denoised_dual(None, None, C.byref(p), None, C.byref(opt), None, None, None, None, None, abi.RtProgressFn(), None,
                                       None) == abi.RT_ERR_NO_DEVICE
    assert b"no CPU path" in lib.rt_last_error()


@pytest.mark.parametrize("extra", [["--gpus=2"], ["--samples_per_pixel=31"], ["--min_samples=7", "--noise_threshold=0.02"]])
def test_cli_rejects_denoise_dual_arguments(extra):
    r = subprocess.run([CLI, "--world=cornell_smoke", "--denoise_dual", *extra], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120)
    assert r.returncode == 1 and "--denoise_dual" in r.stderr and r.stdout == ""


# ------------------------------------------------------------------------------------------------------------------ GPU
def _moments_range(scene, cam, W, H, begin, count, seed=42):
    import torch
    s1 = torch.zeros(H, W, 3, dtype=torch.int64, device="cuda")
    s2 = torch.zeros_like(s1)
    abi.check(abi.load().rt_render_moments_fixed_device(scene.handle, C.byref(cam.c), C.byref(TD._params(W, H, begin + count, seed, begin, count)),
                                                        s1.data_ptr(), s2.data_ptr(), None, None))
    torch.cuda.synchronize()
    return s1.cpu().numpy().view(np.uint64), s2.cpu().numpy().view(np.uint64)


def _cross_np(mu_a, v_a, mu_b, v_b, feats=None, **kw):
    import torch
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    out, err = rt.denoise_cross(t(mu_a), t(v_a), t(mu_b), t(v_b), features=None if feats is None else [t(x) for x in feats], **kw)
    torch.cuda.synchronize()
    return out.cpu().numpy(), err.cpu().numpy()


def _check_against_ref(got_out, got_err, fa, fb, out, eps, tol):
    """out: relative to |out| + 1e-3; eps through its square root, whose error is at most that of F_A and F_B in the
    neighbourhood: |sqrt(got) - sqrt(want)| <= tol (max |F| over the 3 x 3 neighbourhood + 1e-3)"""
    from scipy.ndimage import maximum_filter
    e_out = np.abs(got_out - out) / (np.abs(out) + 1e-3)
    scale = maximum_filter(np.maximum(np.abs(fa), np.abs(fb)), size=(3, 3, 1), mode="nearest") + 1e-3
    e_err = np.abs(np.sqrt(got_err.astype(np.float64)) - np.sqrt(eps)) / scale
    return float(e_out.max()), float(e_err.max())


# Largest |device - restatement| / (|restatement| + 1e-3) of out, and the scaled error of sqrt(eps) (_check_against_ref), f32
# kernel against the f64 restatement; the cross filter runs the arithmetic of the colour-only and guided filters, whose
# measured errors are quoted in test_denoise.py and test_guided_denoise.py (at most 3.5e-6).  A weight taken from the wrong
# buffer or a value from the wrong half moves the output by far more: the two synthetic halves differ by their noise.
DUAL_REL_TOL = 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(1, 1), (3, 5), (23, 37), (48, 64)])
def test_cross_matches_numpy_restatement(H, W):
    mu_a, v_a, mu_b, v_b = synthetic_halves(H, W, H * 1000 + W)
    feats = TG.synthetic_features(H, W, H * 7 + W)
    worst = [0.0, 0.0]
    for r, f in ((0, 0), (1, 1), (3, 0), (10, 3)):
        for guided in (False, True):
            kw = dict(search_radius=r, patch_radius=f, k=0.45, alpha=1.0)
            g = dict(feats=feats, k_feature=0.6, tau=1e-3) if guided else {}
            got_out, got_err = _cross_np(mu_a, v_a, mu_b, v_b, **g, **kw)
            fa, fb, out, eps = dual_ref(mu_a, v_a, mu_b, v_b, r, f, 0.45, 1.0, feats if guided else None, 0.6, np.float32(1e-3))
            e = _check_against_ref(got_out, got_err, fa, fb, out, eps, DUAL_REL_TOL)
            worst = [max(a, b) for a, b in zip(worst, e)]
            assert e[0] < DUAL_REL_TOL and e[1] < DUAL_REL_TOL, (r, f, guided, e)
            if r > 0 and H * W > 1:
                assert np.abs(fa - fb).max() > 1e-3  # (the halves differ: a value from the wrong half would show)
    print(f"cross vs restatement {H}x{W}: worst out {worst[0]:.3g}, worst sqrt(eps) {worst[1]:.3g}")


@pytest.mark.gpu
@pytest.mark.parametrize("guided", [False, True])
def test_cross_large_image_sampled_pixels(guided):
    H, W = 2160, 3840
    mu_a, v_a, mu_b, v_b = synthetic_halves(H, W, 71)
    feats = TG.synthetic_features(H, W, 73) if guided else None
    g = dict(feats=feats, k_feature=0.6, tau=1e-3) if guided else {}
    got_out, got_err = _cross_np(mu_a, v_a, mu_b, v_b, **g)
    rng = np.random.default_rng(72)
    pix = [(0, 0), (H - 1, W - 1), (0, W - 1), (H - 1, 0)] + list(zip(rng.integers(0, H, 36), rng.integers(0, W, 36)))
    # F_A and F_B at the 3 x 3 neighbourhood of every sampled pixel, in the neighbour order of the definition
    nb = [(min(max(y + dy, 0), H - 1), min(max(x + dx, 0), W - 1)) for y, x in pix for dy in (-1, 0, 1) for dx in (-1, 0, 1)]
    kw = (10, 3, 0.45, 1.0, feats, 0.6, np.float32(1e-3))
    fa = cross_ref_pixels(mu_b, v_b, mu_a, nb, *kw).reshape(len(pix), 9, 3)
    fb = cross_ref_pixels(mu_a, v_a, mu_b, nb, *kw).reshape(len(pix), 9, 3)
    out, eps = (fa[:, 4] + fb[:, 4]) / 2, (((fa - fb) / 2) ** 2).mean(axis=1)
    idx = tuple(np.array(pix).T)
    e_out = np.abs(got_out[idx] - out) / (np.abs(out) + 1e-3)
    e_err = np.abs(np.sqrt(got_err[idx].astype(np.float64)) - np.sqrt(eps)) / (np.maximum(np.abs(fa), np.abs(fb)).max(axis=1) + 1e-3)
    print(f"cross 3840x2160 sampled (guided {guided}): worst out {e_out.max():.3g}, worst sqrt(eps) {e_err.max():.3g}")
    assert e_out.max() < DUAL_REL_TOL and e_err.max() < DUAL_REL_TOL


@pytest.mark.gpu
def test_cross_exact_reductions_and_swap_symmetry():
    """A = B: out is rt_denoise_device's (rt_denoise_guided_device's) output bit for bit and eps = 0; A and B swapped: the same
    out and eps bit for bit"""
    H, W = 70, 90
    mu_a, v_a, mu_b, v_b = synthetic_halves(H, W, 81)
    feats = TG.synthetic_features(H, W, 82)
    for r, f in ((10, 3), (3, 0), (15, 7)):
        kw = dict(search_radius=r, patch_radius=f)
        out, err = _cross_np(mu_a, v_a, mu_a, v_a, **kw)
        assert np.array_equal(out.view(np.uint32), TD._denoise_np(mu_a, v_a, **kw).view(np.uint32)) and not err.any(), (r, f)
        g = dict(k_feature=0.6, tau=1e-3)
        out, err = _cross_np(mu_a, v_a, mu_a, v_a, feats=feats, **g, **kw)
        assert np.array_equal(out.view(np.uint32), TG._guided_np(mu_a, v_a, feats, **g, **kw).view(np.uint32)) and not err.any(), (r, f)
        for fe in (None, feats):
            o1, e1 = _cross_np(mu_a, v_a, mu_b, v_b, feats=fe, **kw)
            o2, e2 = _cross_np(mu_b, v_b, mu_a, v_a, feats=fe, **kw)
            assert np.array_equal(o1.view(np.uint32), o2.view(np.uint32)) and np.array_equal(e1.view(np.uint32), e2.view(np.uint32))
            assert (e1 > 0).mean() > 0.5


@pytest.mark.gpu
def test_denoise_cross_rejects_bad_arguments():
    import torch
    lib = abi.load()
    t = [torch.zeros(8, 8, 3, device="cuda") for _ in range(10)]
    ptr = [x.data_ptr() for x in t]
    opt = C.byref(rt.renderer.denoise_options_struct())

    def call(bufs=None, feats=(None,) * 4, guide=None, o=ptr[8], e=ptr[9], W=8, H=8):
        b = list(ptr[:4]) if bufs is None else bufs
        g = C.byref(rt.renderer.guide_struct(**guide)) if guide is not None else None
        return lib.rt_denoise_cross_device(*b, *feats, W, H, opt, g, o, e, -1, None)

    assert call() == abi.RT_OK and call(e=None) == abi.RT_OK
    assert call(feats=ptr[4:8], guide={}) == abi.RT_OK
    for i in range(4):
        assert call(bufs=ptr[:i] + [None] + ptr[i + 1:4]) == abi.RT_ERR_INVALID, i
        assert call(o=ptr[i]) == abi.RT_ERR_INVALID and call(e=ptr[i]) == abi.RT_ERR_INVALID, i
        # guide and features all or none
        assert call(feats=ptr[4:8][:i] + [None] + ptr[4:8][i + 1:], guide={}) == abi.RT_ERR_INVALID, i
        assert call(feats=[ptr[4 + i] if j == i else None for j in range(4)]) == abi.RT_ERR_INVALID, i
        assert call(feats=ptr[4:8], guide={}, o=ptr[4 + i]) == abi.RT_ERR_INVALID, i
    assert call(feats=ptr[4:8]) == abi.RT_ERR_INVALID and call(guide={}) == abi.RT_ERR_INVALID
    for bad in (dict(o=None), dict(e=ptr[8]), dict(o=ptr[9] + 4 * 3 * 8 * 7), dict(W=0), dict(H=-1), dict(H=abi.RT_DENOISE_MAX_HEIGHT + 1, W=1),
                dict(feats=ptr[4:8], guide=dict(tau=0.0))):
        assert call(**bad) == abi.RT_ERR_INVALID, bad
    assert lib.rt_denoise_cross_device(*ptr[:4], *(None,) * 4, 8, 8, None, None, ptr[8], ptr[9], -1, None) == abi.RT_ERR_INVALID
    with pytest.raises(ValueError):
        rt.denoise_cross(*[x.double() for x in t[:4]])


# ------------------------------------------------------------------------------------------------------------ the glue
GUIDE = dict(k_feature=0.6, tau=1e-3, feature_samples=8)


@pytest.mark.gpu
def test_split_is_exact():
    """the moments of [0, n/2) plus those of [n/2, n) are the moments of [0, n) bit for bit"""
    world, scene, cam = TD._setup("cornell_smoke")
    W, H, n = 40, 30, 24
    a, b = _moments_range(scene, cam, W, H, 0, n // 2), _moments_range(scene, cam, W, H, n // 2, n // 2)
    s1, s2 = TD._moments(scene, cam, W, H, n)
    assert np.array_equal(a[0] + b[0], s1) and np.array_equal(a[1] + b[1], s2)
    assert not np.array_equal(a[0], b[0])
    scene.close()


@pytest.mark.gpu
@pytest.mark.parametrize("guided", [False, True])
def test_render_denoised_dual_uniform_is_the_chain(guided):
    """two moments renders of the halves, the numpy conversion with n/2, rt_denoise_cross_device, to_rgb"""
    world, scene, cam = TD._setup("cornell_smoke")
    W, H, spp = 72, 56, 24
    rows = []
    r = TD._renderer(world, scene, cam, W, H, spp)
    rgb, den, err, n = r.render_denoised_dual(logger=lambda j, total: rows.append((j, total)), guide=GUIDE if guided else None, search_radius=5,
                                              patch_radius=2)
    assert rows == [(j, H) for j in range(H)]
    assert r.stats["paths"] == W * H * spp and r.stats["device_ms"] > 0 and (n == spp).all()
    a, b = _moments_range(scene, cam, W, H, 0, spp // 2), _moments_range(scene, cam, W, H, spp // 2, spp // 2)
    mu_a, v_a = TD.mean_var_ref(*a, spp // 2)
    mu_b, v_b = TD.mean_var_ref(*b, spp // 2)
    feats = TG._features(scene, cam, W, H, GUIDE["feature_samples"])[0] if guided else None
    g = dict(k_feature=GUIDE["k_feature"], tau=GUIDE["tau"]) if guided else {}
    want, want_err = _cross_np(mu_a, v_a, mu_b, v_b, feats=feats, search_radius=5, patch_radius=2, **g)
    assert np.array_equal(den.view(np.uint32), want.view(np.uint32)) and np.array_equal(err.view(np.uint32), want_err.view(np.uint32))
    assert np.array_equal(rgb, TD.to_rgb_ref(den.astype(np.float64)))
    scene.close()


def _replay(world, scene, cam, W, H, cap, t, m, feats=None, guide=None):
    """the rounds of rt_render_denoised_dual in Python: each round renders its half ranges for every pixel, adds them to the
    active pixels only, converts, calls rt_denoise_cross_device and applies the restated rule to the active pixels"""
    sums = [np.zeros((H, W, 3), np.uint64) for _ in range(4)]
    half = np.zeros((H, W), np.int64)
    active = np.ones((H, W), bool)
    n_done = 0
    while active.any():
        count = m if n_done == 0 else min(n_done, cap - n_done)
        h = count // 2
        for j, begin in ((0, n_done), (2, n_done + h)):
            s1, s2 = _moments_range(scene, cam, W, H, begin, h)
            sums[j][active] += s1[active]
            sums[j + 1][active] += s2[active]
        n_done += count
        half[active] = n_done // 2
        mu_a, v_a = TD.mean_var_ref(sums[0], sums[1], half[..., None])
        mu_b, v_b = TD.mean_var_ref(sums[2], sums[3], half[..., None])
        out, err = _cross_np(mu_a, v_a, mu_b, v_b, feats=feats, **(guide or {}))
        idx = np.nonzero(active)
        active[idx] = ~filtered_done_ref(n_done, cap, out[idx], err[idx], t)
    return 2 * half, out, err


@pytest.mark.gpu
@pytest.mark.parametrize("guided", [False, True])
def test_render_denoised_dual_adaptive_is_the_replay(guided):
    world, scene, cam = TD._setup("cornell_smoke")
    W = H = 64
    r = TD._renderer(world, scene, cam, W, H, 128)
    rows = []
    rgb, den, err, n = r.render_denoised_dual(0.02, 8, logger=lambda j, total: rows.append((j, total)), guide={} if guided else None)
    assert sorted(rows) == [(j, H) for j in range(H)]
    feats = TG._features(scene, cam, W, H, abi.RT_GUIDE_DEFAULT_FEATURE_SAMPLES)[0] if guided else None
    n_ref, out_ref, err_ref = _replay(world, scene, cam, W, H, 128, 0.02, 8, feats)
    assert len(np.unique(n)) >= 3 and r.stats["paths"] == int(n.sum())
    assert np.array_equal(n, n_ref)
    assert np.array_equal(den.view(np.uint32), out_ref.view(np.uint32)) and np.array_equal(err.view(np.uint32), err_ref.view(np.uint32))
    assert np.array_equal(rgb, TD.to_rgb_ref(den.astype(np.float64)))
    scene.close()


@pytest.mark.gpu
@pytest.mark.parametrize("adaptive", [False, True])
def test_cli_denoise_dual_ppm_matches_the_library(adaptive):
    args = ["--world=cornell_smoke", "--seed=42", "--aspect_ratio=1:1", "--image_width=48", "--samples_per_pixel=32", "--denoise_dual", "--stats"]
    if adaptive:
        args += ["--noise_threshold=0.02", "--min_samples=8", "--denoise_guided"]
    r = subprocess.run([CLI, *args], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert "Done!" in r.stderr and '"mean_spp": ' in r.stderr
    world, scene, cam = TD._setup("cornell_smoke")
    rd = TD._renderer(world, scene, cam, 48, 48, 32)
    rgb, _, _, n = rd.render_denoised_dual(0.02 if adaptive else None, 8, guide={} if adaptive else None)
    assert rt.to_ppm(rgb) == r.stdout
    assert f'"paths": {rd.stats["paths"]},' in r.stderr and f'"mean_spp": {n.mean():.3f}' in r.stderr
    scene.close()


@pytest.mark.gpu
def test_render_denoised_dual_rejects_bad_arguments():
    world, scene, cam = TD._setup("cornell_smoke")
    lib = abi.load()

    def call(p, ad=None, guide=None, **kw):
        g = C.byref(rt.renderer.guide_struct(**guide)) if guide is not None else None
        return lib.rt_render_denoised_dual(scene.handle, C.byref(cam.c), C.byref(p), C.byref(ad) if ad else None,
                                           C.byref(rt.renderer.denoise_options_struct(**kw)), g, None, None, None, None, abi.RtProgressFn(), None, None)

    def adaptive(t=0.01, m=4):
        ad = abi.RtAdaptive()
        ad.noise_threshold, ad.min_samples = t, m
        return ad

    assert call(TD._params(16, 16, 8)) == abi.RT_OK and call(TD._params(16, 16, 8), adaptive()) == abi.RT_OK
    assert call(TD._params(16, 16, 4), guide={}) == abi.RT_OK and call(TD._params(16, 16, 12), adaptive(m=6)) == abi.RT_OK
    for spp in (2, 3, 7, 9):
        assert call(TD._params(16, 16, spp)) == abi.RT_ERR_INVALID, spp
    for m in (2, 3, 5):
        assert call(TD._params(16, 16, 8), adaptive(m=m)) == abi.RT_ERR_INVALID, m
    assert call(TD._params(16, 16, 9), adaptive(m=4)) == abi.RT_ERR_INVALID  # an odd cap
    assert call(TD._params(16, 16, 8, begin=2)) == abi.RT_ERR_INVALID
    assert call(TD._params(16, 16, 8, count=4), adaptive()) == abi.RT_ERR_INVALID
    assert call(TD._params(16, 16, 8), adaptive(t=float("nan"))) == abi.RT_ERR_INVALID
    assert call(TD._params(16, 16, 8), k=0.0) == abi.RT_ERR_INVALID
    assert call(TD._params(16, 16, 8), guide=dict(feature_samples=0)) == abi.RT_ERR_INVALID
    assert lib.rt_render_denoised_dual(scene.handle, C.byref(cam.c), C.byref(TD._params(16, 16, 8)), None, None, None, None, None, None, None,
                                       abi.RtProgressFn(), None, None) == abi.RT_ERR_INVALID
    for pipeline in (abi.RT_PIPELINE_MEGAKERNEL, abi.RT_PIPELINE_WAVEFRONT):
        assert call(TD._params(16, 16, 8, pipeline=pipeline)) == abi.RT_ERR_UNSUPPORTED
        assert call(TD._params(16, 16, 8, pipeline=pipeline), adaptive()) == abi.RT_ERR_UNSUPPORTED
    scene.close()


# ---------------------------------------------------------------------------------------------------------- quality guards
# These bound measurements (DESIGN.md section 5g); the goals the dual filter was built for are missed there, and the bounds guard
# the measured behaviour, they are not quality claims.  Measured on an NVIDIA B200 (1000 W); the sums are integers and the filters
# deterministic, so the values repeat exactly on the same build, and the margins leave room for a change of the arithmetic.
def _ground_truth(scene, cam, W, H, spp=4096):
    g1, _ = TD._moments(scene, cam, W, H, spp, seed=7)
    return g1.astype(np.float64) * 2.0 ** -32 / spp


# The goal was a smaller shift than the colour-only filter's; measured |shift|: dual 2.20 %, 2.20 %, 2.08 % (r, g, b) against
# colour-only 1.21 %, 1.19 %, 1.16 %.
DUAL_SHIFT_BOUND = 0.03


@pytest.mark.gpu
def test_dual_filter_frame_mean_shift():
    """cornell_smoke 128^2 at 64 spp: the shift of each channel's frame-mean radiance against the noisy image.  The dual filter
    shifts it more than the colour-only filter (the weights from one half select candidates by that half's noise, which is skewed
    low; DESIGN.md section 5g), below DUAL_SHIFT_BOUND."""
    world, scene, cam = TD._setup("cornell_smoke")
    W = H = 128
    _, col = TD._renderer(world, scene, cam, W, H, 64).render_denoised()
    _, dual, _, _ = TD._renderer(world, scene, cam, W, H, 64).render_denoised_dual()
    s1, s2 = TD._moments(scene, cam, W, H, 64)
    noisy, _ = TD.mean_var_ref(s1, s2, 64)
    shift = lambda x: x.astype(np.float64).mean(axis=(0, 1)) / noisy.astype(np.float64).mean(axis=(0, 1)) - 1.0  # noqa: E731
    print("frame-mean shift: colour", shift(col).tolist(), "dual", shift(dual).tolist())
    assert np.abs(shift(dual)).max() < DUAL_SHIFT_BOUND, shift(dual)
    scene.close()


# The mean of (out - gt)^2 / eps over the channels with eps > 0, cornell_smoke 128^2 at 64 spp: measured 26.6 (0.58 % of the
# pixels have eps = 0).  eps estimates the variance of out only, and the filter's bias dominates its error: eps is about 27 times
# too small as an estimate of the squared error.
CALIBRATION_BAND = (10.0, 60.0)


@pytest.mark.gpu
def test_error_estimate_calibration():
    world, scene, cam = TD._setup("cornell_smoke")
    W = H = 128
    _, out, eps, _ = TD._renderer(world, scene, cam, W, H, 64).render_denoised_dual()
    gt = _ground_truth(scene, cam, W, H)
    pos = eps > 0
    ratio = float((((out.astype(np.float64) - gt) ** 2)[pos] / eps[pos]).mean())
    print("calibration: mean (out - gt)^2 / eps", ratio, "share eps = 0", float((~pos).mean()))
    assert CALIBRATION_BAND[0] < ratio < CALIBRATION_BAND[1], ratio
    scene.close()


# The goal was a smaller early-stop tail than the rule of rt_render_adaptive; measured: 54.7 % of the 58.5 % of pixels stopped
# before the cap for the filtered rule (mean spp 461), against 51.8 % of 30.5 % for the section 5d rule.
TAIL_SHARE_BOUND = 0.65


@pytest.mark.gpu
def test_filtered_rule_early_stop_tail():
    """cornell_smoke 128^2, cap 1024, t = 0.01, min_samples 16: among the pixels stopped before the cap, the share whose display
    error exceeds 3 t, for the filtered rule judged on the dual filter's output; below TAIL_SHARE_BOUND."""
    world, scene, cam = TD._setup("cornell_smoke")
    W = H = 128
    t = 0.01
    gt = display(_ground_truth(scene, cam, W, H))
    _, out, _, n = TD._renderer(world, scene, cam, W, H, 1024).render_denoised_dual(t, 16)
    _, n0, s1, _ = TD._renderer(world, scene, cam, W, H, 1024).render_adaptive(t, 16)
    share = lambda x, cnt: float((np.abs(display(x) - gt).max(axis=2)[cnt < 1024] > 3 * t).mean())  # noqa: E731
    dual, plain = share(out, n), share(s1.astype(np.float64) * 2.0 ** -32 / n0[..., None], n0)
    print("early-stop tail: filtered rule", dual, "stopped", float((n < 1024).mean()), "mean spp", float(n.mean()), "; section 5d rule", plain,
          "stopped", float((n0 < 1024).mean()), "mean spp", float(n0.mean()))
    assert (n < 1024).mean() > 0.2 and dual < TAIL_SHARE_BOUND, (dual, plain)
    scene.close()
