#!/usr/bin/env python
"""What the variance-guided non-local-means denoiser costs and what it buys, on C3 (cornell_smoke 600^2) and C4 (final_scene
800^2).  Prints one JSON line; needs a CUDA device.  Reuses the jobs, ground truths and error measure of adaptive_bench.py.

(a) kernel time of rt_denoise_device: CUDA events over many launches after a warm-up, on synthetic inputs at 600^2, 800^2
    and 3840^2 with the defaults, plus an r / f sweep at 800^2.  The operation count is the arithmetic of the definition per
    pixel and offset of the window: 27 for e (three channels), 2 (2f + 1) for the two box sums, 7 for the weight and the
    weighted sums; the tile halos and the skipped offset d = 0 are not counted.  600^2 and 800^2 inputs (mean and variance,
    4 and 7.7 MB) fit the 126 MB L2; 3840^2 (354 MB) does not.
(b) quality at 16 / 64 / 256 spp: display error (largest channel after the gamma-2 tonemap) at the 50th / 95th / 99th
    percentiles against adaptive_bench's ground truths (C3 8 000 spp, C4 20 000 spp, seed 7), noisy and denoised, and the
    frame-mean radiance per channel of both.
(c) equal time: the uniform spp, rendered through the product path (rt_render_accumulate_fixed_device, what a user who does
    not denoise runs), whose device time equals that of the denoised render (render + filter); rendered and measured.
(d) adaptive sampling (threshold 0.01, min_samples 16, adaptive_bench's cap) with and without the filter.
(e) a sweep of k and alpha (and r, f) at 64 spp.
(f) where the filter hurts: the display error inside the image discs of final_scene's textured spheres (the earth-mapped
    and the Perlin-noise sphere, worlds.rs:386-468), noisy and denoised at 64 spp.

usage: python tools/denoise_bench.py [--out FILE] [--quick]"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import mu_lambda_raytracer_b200 as rt  # noqa: E402
from mu_lambda_raytracer_b200 import abi  # noqa: E402
import adaptive_bench as AB  # noqa: E402

DEFAULTS = dict(search_radius=abi.RT_DENOISE_DEFAULT_SEARCH_RADIUS, patch_radius=abi.RT_DENOISE_DEFAULT_PATCH_RADIUS, k=abi.RT_DENOISE_DEFAULT_K,
                alpha=abi.RT_DENOISE_DEFAULT_ALPHA)
SPPS = [16, 64, 256]
THRESHOLD = 0.01
# final_scene's textured spheres (centre, radius): the earth-mapped and the Perlin-noise sphere
TEXTURED_SPHERES = {"final_scene": {"earth_sphere": ((400.0, 200.0, 400.0), 100.0), "noise_sphere": ((220.0, 280.0, 300.0), 80.0)}}


def op_count(W, H, r, f):
    return float(W) * H * ((2 * r + 1) ** 2 - 1) * (27 + 2 * (2 * f + 1) + 7)


def time_kernel(mean, var, out, opt, min_seconds=0.3):
    """ms per launch of rt_denoise_device: events around n launches after 3 warm-up launches, n chosen for >= min_seconds"""
    import torch
    lib = abi.load()
    H, W = mean.shape[:2]

    def launch():
        abi.check(lib.rt_denoise_device(mean.data_ptr(), var.data_ptr(), W, H, C.byref(opt), out.data_ptr(), -1, None))

    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    launch()
    b.record()
    b.synchronize()
    n = int(min(500, max(5, min_seconds * 1e3 / max(a.elapsed_time(b), 1e-3))))
    a.record()
    for _ in range(n):
        launch()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n, n


def synthetic(H, W, seed=1):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    mean = torch.rand(H, W, 3, device="cuda", generator=g)
    var = torch.rand(H, W, 3, device="cuda", generator=g) * 1e-2
    return mean, var


def sphere_disc(world, centre, radius, W, H, shrink=0.9):
    """pixels [H, W] (row 0 at the bottom) within shrink x the projected radius of a sphere's image, through the world's camera"""
    info = world.camera()
    eye, at = np.array(info["lookfrom"], np.float64), np.array(info["lookat"], np.float64)
    w = (eye - at) / np.linalg.norm(eye - at)
    u = np.cross([0.0, 1.0, 0.0], w)
    u /= np.linalg.norm(u)
    v = np.cross(w, u)
    d = np.array(centre) - eye
    z = -d @ w
    t = np.tan(np.radians(info["field_of_view"]) / 2)
    ci, cj = ((d @ u) / (z * t) + 1) / 2 * (W - 1), ((d @ v) / (z * t) + 1) / 2 * (H - 1)
    rad = radius / z / t * (H - 1) / 2 * shrink
    jj, ii = np.mgrid[0:H, 0:W]
    return (ii - ci) ** 2 + (jj - cj) ** 2 <= rad * rad


def kernel_times(quick):
    import torch
    sizes = [(96, 96)] if quick else [(600, 600), (800, 800), (3840, 3840)]
    sweep = [(5, 2), (7, 3), (10, 2), (10, 5), (15, 3), (15, 7)]
    rows = []
    for (H, W) in sizes:
        mean, var = synthetic(H, W)
        out = torch.empty_like(mean)
        for r, f in [(DEFAULTS["search_radius"], DEFAULTS["patch_radius"])] + (sweep if (H, W) == sizes[min(1, len(sizes) - 1)] else []):
            opt = rt.renderer.denoise_options_struct(**dict(DEFAULTS, search_radius=r, patch_radius=f))
            ms, n = time_kernel(mean, var, out, opt)
            ops = op_count(W, H, r, f)
            rows.append({"width": W, "height": H, "search_radius": r, "patch_radius": f, "ms": ms, "launches": n, "gops": ops * 1e-9,
                         "gops_per_s": ops / (ms * 1e-3) * 1e-9})
        del mean, var, out
        torch.cuda.empty_cache()
    return rows


def quality(key, world_name, size, cap, gt_spp, quick):
    import torch
    if quick:
        size, cap, gt_spp = 96, 64, 256
    world, scene, cam = AB.setup(world_name)
    W = H = size
    s1 = torch.zeros(H, W, 3, dtype=torch.int64, device="cuda")
    s2 = torch.zeros_like(s1)
    AB.render_uniform(scene, cam, s1, s2, gt_spp, seed=7)
    gt = AB.display(s1.cpu().numpy().view(np.uint64).astype(np.float64) * 2.0 ** -32 / gt_spp)

    def renderer(spp):
        return rt.Renderer.new_with_rng(cam, scene, world.background(), rt.RenderingParams(spp, H, W), rt.RecursiveRayTracer(50), rt.SeedableRngator(42))

    def noisy(spp):
        """mean and variance of the mean of a uniform moments render, as the library converts them (f32), and its device ms"""
        st = AB.render_uniform(scene, cam, s1, s2, spp)
        a, b = s1.cpu().numpy().view(np.uint64), s2.cpu().numpy().view(np.uint64)
        mu = a.astype(np.float64) * 2.0 ** -32 / spp
        var = np.maximum((b.astype(np.float64) * 2.0 ** -24 - spp * (mu * mu)) / (spp - 1.0), 0.0) / spp
        return mu.astype(np.float32), var.astype(np.float32), st.device_ms

    frame_mean = lambda x: [float(c) for c in np.asarray(x, np.float64).mean(axis=(0, 1))]  # noqa: E731
    renderer(16).render_denoised()  # warm-up: modules, grid sizing
    runs = []
    for spp in SPPS:
        mu, var, ms_noisy = noisy(spp)
        r = renderer(spp)
        _, den = r.render_denoised()
        ms_den = r.stats["device_ms"]
        # (c) the product path at the spp of the same device time (its time is linear in spp), rendered and measured
        ms_prod = AB.render_uniform(scene, cam, s1, s2, spp, moments=False).device_ms
        spp_eq = max(2, int(round(spp * ms_den / ms_prod)))
        ms_eq = AB.render_uniform(scene, cam, s1, s2, spp_eq, moments=False).device_ms
        mu_eq = s1.cpu().numpy().view(np.uint64).astype(np.float64) * 2.0 ** -32 / spp_eq
        runs.append({"spp": spp, "noisy": {"device_ms": ms_noisy, "product_device_ms": ms_prod, "err_p50_p95_p99": AB.display_errors(mu, gt),
                                           "frame_mean": frame_mean(mu)},
                     "denoised": {"device_ms": ms_den, "err_p50_p95_p99": AB.display_errors(den, gt), "frame_mean": frame_mean(den)},
                     "product_same_time": {"spp": spp_eq, "device_ms": ms_eq, "err_p50_p95_p99": AB.display_errors(mu_eq, gt)}})
    # (d) adaptive, with and without the filter
    ra = renderer(cap)
    _, n, acc, _ = ra.render_adaptive(THRESHOLD, 16)
    ms_ad = ra.stats["device_ms"]
    rd = renderer(cap)
    _, den_ad = rd.render_denoised(THRESHOLD, 16)
    adaptive = {"threshold": THRESHOLD, "min_samples": 16, "cap": cap, "mean_spp": float(n.mean()),
                "adaptive": {"device_ms": ms_ad, "err_p50_p95_p99": AB.display_errors(acc.astype(np.float64) * 2.0 ** -32 / n[..., None], gt)},
                "adaptive_denoised": {"device_ms": rd.stats["device_ms"], "err_p50_p95_p99": AB.display_errors(den_ad, gt)}}
    # (e) parameters at 64 spp
    mu, var, _ = noisy(64)
    tm, tv = torch.from_numpy(mu).cuda(), torch.from_numpy(var).cuda()
    # (f) the textured spheres
    den64 = rt.denoise(tm, tv).cpu().numpy()
    regions = {}
    for name, (centre, radius) in TEXTURED_SPHERES.get(world_name, {}).items():
        m = sphere_disc(world, centre, radius, W, H)
        e_noisy, e_den = (np.abs(AB.display(x) - gt).max(axis=2)[m] for x in (mu, den64))
        regions[name] = {"pixels": int(m.sum()), "noisy_mean_p95": [float(e_noisy.mean()), float(np.percentile(e_noisy, 95))],
                         "denoised_mean_p95": [float(e_den.mean()), float(np.percentile(e_den, 95))],
                         "share_worse": float((e_den > e_noisy).mean())}
    e_all = [np.abs(AB.display(x) - gt).max(axis=2) for x in (mu, den64)]
    regions["whole_image"] = {"pixels": int(W * H), "noisy_mean_p95": [float(e_all[0].mean()), float(np.percentile(e_all[0], 95))],
                              "denoised_mean_p95": [float(e_all[1].mean()), float(np.percentile(e_all[1], 95))],
                              "share_worse": float((e_all[1] > e_all[0]).mean())}
    sweep = []
    grid = [dict(DEFAULTS, k=k, alpha=a) for k in (0.3, 0.45, 0.7, 1.0) for a in (0.5, 1.0, 2.0, 4.0)]
    grid += [dict(DEFAULTS, search_radius=r, patch_radius=f) for r, f in ((5, 2), (7, 3), (10, 1), (10, 2), (15, 3))]
    for opt in grid:
        den = rt.denoise(tm, tv, **opt).cpu().numpy()
        sweep.append(dict(opt, err_p50_p95_p99=AB.display_errors(den, gt), rmse=float(np.sqrt(np.mean((AB.display(den) - gt) ** 2)))))
    scene.close()
    return {"world": world_name, "size": size, "ground_truth_spp": gt_spp, "spp_runs": runs, "adaptive": adaptive, "sweep_64spp": sweep,
            "regions_64spp": regions}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    if abi.load().rt_device_count() < 1:
        raise SystemExit("denoise_bench needs a CUDA device")
    name, power = AB.gpu_info()
    result = {"gpu": name, "power_limit": power, "defaults": DEFAULTS, "kernel": kernel_times(args.quick), "configs": {}}
    for key, world_name, size, cap, _, gt_spp, _ in AB.CONFIGS:
        result["configs"][key] = quality(key, world_name, size, cap, gt_spp, args.quick)
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
