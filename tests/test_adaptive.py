"""Per-pixel second moments and noise-threshold adaptive sampling (an EXTENSION: the reference renders a fixed count).

CPU part: the exact integer square (moment2_fixed) and the f64 stop rule (adaptive_pixel_done) of rt_device.cuh, run through
the host build of the header, against Python restatements; the entry points and the CLI without a device.  GPU part: the
moments family of the persistent kernel against single-sample renders and the product instance, the calibration of the
variance estimate, and adaptive renders against uniform renders of the same counts, bit for bit."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import mu_lambda_raytracer_b200 as rt
from mu_lambda_raytracer_b200 import abi
import support as S

CLI = os.path.join(S.ROOT, "mu-lambda-raytracer_b200", "rt_main")


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    """tests/emul/adaptive_emul.cpp: moment2_fixed and adaptive_pixel_done of rt_device.cuh built for the host"""
    path = str(tmp_path_factory.mktemp("adaptive_emul") / "libadaptive_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-w", "-shared", "-o", path, os.path.join(S.ROOT, "tests", "emul", "adaptive_emul.cpp")])
    L = C.CDLL(path)
    L.emul_moment2_fixed.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
    L.emul_adaptive_done.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_void_p]
    return L


def moment2_ref(q):
    """(min(q, 2^44))^2 >> 40 with Python integers"""
    return [min(int(x), 1 << 44) ** 2 >> 40 for x in np.asarray(q).ravel()]


def stop_ref(n, n_max, s1, s2, threshold):
    """the stop rule in numpy (f64, one rounding per operation): n [N], s1 / s2 [N, 3] fixed-point sums -> done [N]"""
    dn = np.asarray(n, np.float64)[:, None]
    mu = s1.astype(np.float64) * 2.0 ** -32 / dn
    m2 = s2.astype(np.float64) * 2.0 ** -24
    var = np.maximum((m2 - dn * (mu * mu)) / (dn - 1.0), 0.0)
    se = np.sqrt(var / dn)
    e = se / (2.0 * np.sqrt(np.maximum(mu, 2.0 ** -16)))
    ok = (e <= threshold) | (mu - 3.0 * se >= 1.0)
    return (np.asarray(n) >= n_max) | ok.all(axis=1)


def to_rgb_ref(mean):
    """to_rgb (raytrace.rs:59-68) in f64"""
    x = np.clip(np.sqrt(mean), 0.0, 0.99999999)
    return (255.999 * x).astype(np.int32)


def test_moment2_fixed_is_the_exact_capped_square(emul):
    rng = np.random.default_rng(1)
    q = np.array([0, 1, 2, (1 << 20) - 1, 1 << 32, (1 << 44) - 1, 1 << 44, (1 << 44) + 1, 1 << 52, (1 << 64) - 1] +
                 list(rng.integers(0, 1 << 46, 5000, dtype=np.uint64)) + list(rng.integers(0, 1 << 34, 5000, dtype=np.uint64)), dtype=np.uint64)
    out = np.zeros_like(q)
    emul.emul_moment2_fixed(q.ctypes.data, len(q), out.ctypes.data)
    assert [int(x) for x in out] == moment2_ref(q)
    assert int(out[6]) == int(out[7]) == int(out[8]) == 1 << 48  # a sample above 4096 is capped in the square


def test_stop_rule_matches_numpy(emul):
    rng = np.random.default_rng(2)
    N, n_max = 200_000, 1024
    n = rng.choice([2, 4, 16, 64, 256, 1024], N).astype(np.uint32)
    mu = rng.choice([0.0, 1e-6, 0.01, 0.3, 0.9, 1.5, 40.0], (N, 3)) * rng.uniform(0.5, 1.5, (N, 3))
    s1 = np.round(mu * n[:, None] * 2.0 ** 32).astype(np.uint64)
    rel = rng.choice([0.0, 1e-12, 0.01, 1.0, 10.0], (N, 3))  # 0 and 1e-12: S2 at or just below n mu^2 (rounding)
    s2 = np.round((mu * mu * (1.0 + rel) * n[:, None]) * 2.0 ** 24).astype(np.uint64)
    s2[: N // 8] = np.floor(s1[: N // 8].astype(np.float64) ** 2 * 2.0 ** -40 / n[: N // 8, None]).astype(np.uint64)  # S2 < n mu^2
    s1[-100:], s2[-100:] = 0, 0  # mu = 0
    for t in (0.0, 1e-3, 0.01, 0.05, 1e9):
        got = np.zeros(N, np.uint8)
        emul.emul_adaptive_done(n.ctypes.data, n_max, s1.ctypes.data, s2.ctypes.data, N, t, got.ctypes.data)
        want = stop_ref(n, n_max, s1, s2, t)
        assert np.array_equal(got.astype(bool), want), (t, np.flatnonzero(got.astype(bool) != want)[:5])
        assert want[n == n_max].all()
        if 0.0 < t < 1.0:
            assert 0.05 < want[n < n_max].mean() < 0.95, t  # the random cases exercise both outcomes
    # saturated channels: mean far above 1 stops even with threshold 0, a mean near 1 with a large error does not
    sat = stop_ref(np.array([16, 16]), 1024, np.array([[40 * 16 << 32] * 3, [16 << 32] * 3], np.uint64),
                   np.array([[(2 * 40 * 40 * 16) << 24] * 3, [(16 * 4) << 24] * 3], np.uint64), 0.0)
    assert sat.tolist() == [True, False]


def test_entry_points_without_a_device():
    lib = abi.load()
    if lib.rt_device_count() > 0:
        pytest.skip("a CUDA device is present")
    p, ad = abi.RtParams(), abi.RtAdaptive()
    assert lib.rt_render_moments_fixed_device(None, None, C.byref(p), None, None, None, None) == abi.RT_ERR_NO_DEVICE
    assert lib.rt_render_adaptive(None, None, C.byref(p), C.byref(ad), None, None, None, None, abi.RtProgressFn(), None, None) == abi.RT_ERR_NO_DEVICE
    assert b"no CPU path" in lib.rt_last_error()


def test_cli_rejects_noise_threshold_on_several_gpus():
    r = subprocess.run([CLI, "--world=cornell_smoke", "--noise_threshold=0.01", "--gpus=2"], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       text=True, timeout=120)
    assert r.returncode == 1 and "--noise_threshold" in r.stderr and r.stdout == ""


# ------------------------------------------------------------------------------------------------------------------ GPU
def _setup(name, aspect=1.0):
    world = rt.World(name)
    scene = rt.Scene(world.build(42))
    info = world.camera()
    cam = S.make_camera(info["lookfrom"], info["lookat"], info["field_of_view"], aspect)
    return world, scene, cam


def _params(W, H, spp, seed=42, begin=0, count=0, pipeline=abi.RT_PIPELINE_AUTO, layout=0):
    p = abi.RtParams()
    p.width, p.height, p.samples_per_pixel, p.max_depth, p.seed = W, H, spp, 50, seed
    p.sample_begin, p.sample_count, p.pipeline, p.device, p.bvh_layout = begin, count, pipeline, -1, layout
    return p


def _moments(scene, cam, W, H, begin, count, seed=42, layout=0):
    """uniform moments render of samples [begin, begin + count): (S1, S2, stats) as uint64 [H, W, 3]"""
    import torch
    s1 = torch.zeros(H, W, 3, dtype=torch.int64, device="cuda")
    s2 = torch.zeros(H, W, 3, dtype=torch.int64, device="cuda")
    st = abi.RtStats()
    abi.check(abi.load().rt_render_moments_fixed_device(scene.handle, C.byref(cam.c), C.byref(_params(W, H, begin + count, seed, begin, count, layout=layout)),
                                                        s1.data_ptr(), s2.data_ptr(), None, C.byref(st)))
    torch.cuda.synchronize()
    return s1.cpu().numpy().view(np.uint64), s2.cpu().numpy().view(np.uint64), st


def _accum_fixed(scene, cam, W, H, begin, count, seed=42):
    import torch
    s1 = torch.zeros(H, W, 3, dtype=torch.int64, device="cuda")
    st = abi.RtStats()
    abi.check(abi.load().rt_render_accumulate_fixed_device(scene.handle, C.byref(cam.c), C.byref(_params(W, H, begin + count, seed, begin, count)),
                                                           s1.data_ptr(), None, C.byref(st)))
    torch.cuda.synchronize()
    return s1.cpu().numpy().view(np.uint64), st


def _adaptive(world, scene, cam, W, H, cap, t, m, seed=42, logger=None):
    r = rt.Renderer.new_with_rng(cam, scene, world.background(), rt.RenderingParams(cap, H, W), rt.RecursiveRayTracer(50), rt.SeedableRngator(seed))
    out = r.render_adaptive(t, m, logger)
    return out + (r.stats,)


@pytest.mark.gpu
@pytest.mark.parametrize("name,layout", [("cornell_smoke", 0), ("final_scene", 0), ("final_scene", 2)])
def test_moments_are_exact_sums_of_squares(name, layout):
    """S2 of a k-sample render is, integer for integer, the sum over s < k of moment2_fixed of the single-sample sums of
    [s, s + 1) — the square of every path's own fixed-point sample — and any split of the range adds up to the same S1, S2
    (also through the binary-tree instances, layout 2)"""
    world, scene, cam = _setup(name)
    W = H = 96
    k = 12
    s1, s2, st = _moments(scene, cam, W, H, 0, k, layout=layout)
    want1, want2 = np.zeros(W * H * 3, dtype=object), np.zeros(W * H * 3, dtype=object)
    for s in range(k):
        q, q2, _ = _moments(scene, cam, W, H, s, 1, layout=layout)
        want1 += np.array([int(x) for x in q.ravel()], dtype=object)
        want2 += np.array(moment2_ref(q), dtype=object)
    assert [int(x) for x in s1.ravel()] == list(want1)
    assert [int(x) for x in s2.ravel()] == list(want2)
    a1, a2, _ = _moments(scene, cam, W, H, 0, 5, layout=layout)
    b1, b2, _ = _moments(scene, cam, W, H, 5, 7, layout=layout)
    assert np.array_equal(a1 + b1, s1) and np.array_equal(a2 + b2, s2)
    assert st.paths == W * H * k and st.bvh_layout_used == (layout or 4) and (s2 > 0).mean() > 0.2
    scene.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["random", "cornell_smoke", "final_scene", "earth"])
def test_moments_family_traces_the_product_paths(name):
    """the moments instance against the product instance (rt_render_accumulate_fixed_device) on the same job: the relation of
    test_feature_instances_trace_the_generic_instance_paths (FMA contraction differs between kernels)"""
    aspect = 1.5 if name in ("random", "earth") else 1.0
    world, scene, cam = _setup(name, aspect)
    W, spp = 128, 32
    H = int(W / aspect)
    m1, _, st_m = _moments(scene, cam, W, H, 0, spp)
    a1, st_a = _accum_fixed(scene, cam, W, H, 0, spp)
    a0, a1f = a1.astype(np.float64), m1.astype(np.float64)
    assert st_m.paths == st_a.paths and abs(int(st_m.rays) - int(st_a.rays)) <= 1e-3 * st_a.rays
    close = np.isclose(a0, a1f, rtol=1e-4, atol=1e-4 * a0.mean()).all(axis=2)
    assert close.mean() > 0.99, close.mean()
    assert abs(a0.mean() - a1f.mean()) < 1e-3 * a0.mean()
    scene.close()


def _mean_se(s1, s2, n):
    mu = s1.astype(np.float64) * 2.0 ** -32 / n
    var = np.maximum((s2.astype(np.float64) * 2.0 ** -24 - n * mu * mu) / (n - 1), 0.0)
    return mu, var / n


@pytest.mark.gpu
def test_variance_estimate_is_calibrated():
    """two disjoint halves [0, 64) and [64, 128): the pixel mean of (mu_a - mu_b)^2 / (se_a^2 + se_b^2) is near 1 when the
    standard errors are right.  Measured on a B200: 1.001, over the 84 % of pixel channels with a non-zero estimate."""
    world, scene, cam = _setup("cornell_smoke")
    W = H = 96
    a1, a2, _ = _moments(scene, cam, W, H, 0, 64)
    b1, b2, _ = _moments(scene, cam, W, H, 64, 64)
    mu_a, v_a = _mean_se(a1, a2, 64)
    mu_b, v_b = _mean_se(b1, b2, 64)
    ok = (v_a + v_b) > 0
    z = (mu_a - mu_b)[ok] ** 2 / (v_a + v_b)[ok]
    print("calibration:", z.mean(), ok.mean())
    assert ok.mean() > 0.5 and 0.9 < z.mean() < 1.1, (z.mean(), ok.mean())
    scene.close()


@pytest.mark.gpu
def test_adaptive_render_is_a_prefix_of_uniform_renders():
    """every pixel's sums are those of a uniform moments render at its own count, every count is in the round set
    {m, 2m, 4m, ..., max}, the stop rule said "go on" at every earlier round and "stop" at the last, and rgb is to_rgb of
    the pixel's own mean"""
    world, scene, cam = _setup("cornell_smoke")
    W = H = 64
    cap, m, t = 96, 6, 0.02
    rows = []
    rgb, n, s1, s2, stats = _adaptive(world, scene, cam, W, H, cap, t, m, logger=lambda j, total: rows.append((j, total)))
    assert rows == [(j, H) for j in range(H)]
    assert stats["paths"] == int(n.sum())
    rounds = [6, 12, 24, 48, 96]
    assert set(np.unique(n)) <= set(rounds) and len(np.unique(n)) >= 3, np.unique(n, return_counts=True)
    assert stop_ref(n.ravel(), cap, s1.reshape(-1, 3), s2.reshape(-1, 3), t).all()
    for c in rounds:
        u1, u2, _ = _moments(scene, cam, W, H, 0, c)
        at = n == c
        assert np.array_equal(s1[at], u1[at]) and np.array_equal(s2[at], u2[at]), c
        later = n > c  # these went on after round c
        assert not stop_ref(np.full(later.sum(), c), cap, u1[later], u2[later], t).any(), c
    assert np.array_equal(rgb, to_rgb_ref(s1.astype(np.float64) * (1.0 / (abi.RT_ACCUM_FIXED_ONE * n[..., None].astype(np.float64)))))
    scene.close()


@pytest.mark.gpu
def test_adaptive_edge_cases():
    world, scene, cam = _setup("final_scene")
    W = H = 48
    # threshold 0 with min == max: the uniform moments render, and rt_render's image
    rgb, n, s1, s2, stats = _adaptive(world, scene, cam, W, H, 16, 0.0, 16)
    u1, u2, _ = _moments(scene, cam, W, H, 0, 16)
    assert (n == 16).all() and np.array_equal(s1, u1) and np.array_equal(s2, u2)
    r = rt.Renderer.new_with_rng(cam, scene, world.background(), rt.RenderingParams(16, H, W), rt.RecursiveRayTracer(50), rt.SeedableRngator(42))
    assert np.array_equal(r.render_arrays()[0], rgb)
    # threshold 0: a pixel stops before the cap only with a zero variance estimate (or saturated) in every channel
    _, n0, a0, b0, _ = _adaptive(world, scene, cam, W, H, 32, 0.0, 4)
    assert (n0 == 32).any() and stop_ref(n0.ravel(), 32, a0.reshape(-1, 3), b0.reshape(-1, 3), 0.0).all()
    # a huge threshold stops every pixel after round 0
    _, n1, _, _, st1 = _adaptive(world, scene, cam, W, H, 512, 1e9, 8)
    assert (n1 == 8).all() and st1["paths"] == W * H * 8
    # two runs: identical outputs
    a = _adaptive(world, scene, cam, W, H, 128, 0.03, 8)
    b = _adaptive(world, scene, cam, W, H, 128, 0.03, 8)
    for x, y in zip(a[:4], b[:4]):
        assert np.array_equal(x, y)
    assert a[4]["rays"] == b[4]["rays"] and a[4]["paths"] == int(a[1].sum())
    assert stop_ref(a[1].ravel(), 128, a[2].reshape(-1, 3), a[3].reshape(-1, 3), 0.03).all()
    scene.close()


@pytest.mark.gpu
def test_adaptive_rejects_bad_arguments():
    world, scene, cam = _setup("cornell_smoke")
    lib = abi.load()

    def call(p, t=0.01, m=4):
        ad = abi.RtAdaptive()
        ad.noise_threshold, ad.min_samples = t, m
        return lib.rt_render_adaptive(scene.handle, C.byref(cam.c), C.byref(p), C.byref(ad), None, None, None, None, abi.RtProgressFn(), None, None)

    assert call(_params(16, 16, 8), m=1) == abi.RT_ERR_INVALID
    assert call(_params(16, 16, 8), m=9) == abi.RT_ERR_INVALID
    assert call(_params(16, 16, 8), t=-0.1) == abi.RT_ERR_INVALID
    assert call(_params(16, 16, 8), t=float("nan")) == abi.RT_ERR_INVALID
    assert call(_params(16, 16, 8, begin=2)) == abi.RT_ERR_INVALID
    assert call(_params(16, 16, 8, count=4)) == abi.RT_ERR_INVALID
    for pipeline in (abi.RT_PIPELINE_MEGAKERNEL, abi.RT_PIPELINE_WAVEFRONT):
        assert call(_params(16, 16, 8, pipeline=pipeline)) == abi.RT_ERR_UNSUPPORTED
        assert lib.rt_render_moments_fixed_device(scene.handle, C.byref(cam.c), C.byref(_params(16, 16, 8, pipeline=pipeline)), 1, 1, None, None) == abi.RT_ERR_UNSUPPORTED
    assert call(_params(16, 16, 8)) == abi.RT_OK
    scene.close()


@pytest.mark.gpu
def test_cli_adaptive_ppm_matches_the_library():
    args = ["--world=cornell_smoke", "--seed=42", "--aspect_ratio=1:1", "--image_width=48", "--samples_per_pixel=64", "--noise_threshold=0.02",
            "--min_samples=8", "--stats"]
    r = subprocess.run([CLI, *args], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert "Done!" in r.stderr and '"mean_spp": ' in r.stderr
    world, scene, cam = _setup("cornell_smoke")
    rgb, n, _, _, stats = _adaptive(world, scene, cam, 48, 48, 64, 0.02, 8)
    assert rt.to_ppm(rgb) == r.stdout
    assert f'"paths": {stats["paths"]},' in r.stderr and 8 < n.mean() < 64
    scene.close()


@pytest.mark.gpu
def test_stop_rule_is_useful():
    """cornell_smoke 128^2, cap 1024, threshold t = 0.01, against a 4096-spp uniform ground truth: among the pixels that
    stopped before the cap, the share whose display error (any channel, after the gamma-2 tonemap) exceeds 3 t.  Measured on
    a B200: 30 % of the pixels stop, and 52 % of those are off by more than 3 t.  The rule cannot see what the first
    min_samples samples missed: a pixel whose 16 paths all found no light has mean 0 and variance estimate 0, and stops.
    The bound guards that measurement (DESIGN.md section 5d); it is not a quality claim."""
    world, scene, cam = _setup("cornell_smoke")
    W = H = 128
    t = 0.01
    rgb, n, s1, s2, stats = _adaptive(world, scene, cam, W, H, 1024, t, 16)
    g1, _, _ = _moments(scene, cam, W, H, 0, 4096, seed=7)
    disp = lambda s, c: np.sqrt(np.clip(s.astype(np.float64) * 2.0 ** -32 / c, 0.0, 1.0))
    err = np.abs(disp(s1, n[..., None]) - disp(g1, 4096)).max(axis=2)
    stopped = n < 1024
    bad = (err[stopped] > 3 * t).mean()
    print("useful: stopped", stopped.mean(), "bad", bad, "mean spp", n.mean())
    assert stopped.mean() > 0.2 and bad < 0.6, (stopped.mean(), bad)
    scene.close()
