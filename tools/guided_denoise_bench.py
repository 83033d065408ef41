#!/usr/bin/env python
"""What the feature-guided mode of the denoiser costs and what it buys, against the colour-only filter, on C3 (cornell_smoke
600^2) and C4 (final_scene 800^2).  Prints one JSON line; needs a CUDA device.  Reuses the jobs, ground truths and error
measure of adaptive_bench.py and the timing, inputs and sphere discs of denoise_bench.py.

(a) the feature pass (rt_render_features_device) on C4 at 800^2 for 4 / 16 / 64 feature samples: device ms (CUDA events),
    best of three after a warm-up.
(b) kernel time of rt_denoise_guided_device against rt_denoise_device on the same synthetic inputs (features: a copy of the
    colour planes) at the sizes and radii of denoise_bench (a).
(c) quality at 16 / 64 / 256 spp: display error percentiles of noisy, colour-only and guided (rt_render_denoised_guided, default
    RtGuide), the frame-mean radiance of each, and the product path at the device time of the guided render.
(d) the textured-sphere discs of final_scene and the whole frame at 64 spp: mean / p95 display error and the share of pixels
    worse than noisy, colour-only and guided.
(e) at 64 spp: k_feature x tau, and feature_samples.

usage: python tools/guided_denoise_bench.py [--out FILE] [--quick]"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import denoise_bench as DB  # noqa: E402  (puts the repository and tests/ on sys.path)
import adaptive_bench as AB  # noqa: E402
import mu_lambda_raytracer_b200 as rt  # noqa: E402
from mu_lambda_raytracer_b200 import abi  # noqa: E402

GUIDE = dict(k_feature=abi.RT_GUIDE_DEFAULT_K_FEATURE, tau=abi.RT_GUIDE_DEFAULT_TAU, feature_samples=abi.RT_GUIDE_DEFAULT_FEATURE_SAMPLES)


def feature_times(quick):
    world, scene, cam = AB.setup("final_scene")
    W = H = 96 if quick else 800
    rd = rt.Renderer.new_with_rng(cam, scene, world.background(), rt.RenderingParams(4, H, W), rt.RecursiveRayTracer(50), rt.SeedableRngator(42))
    rd.render_features(4)  # warm-up
    rows = []
    for n in (4, 16, 64):
        ms = []
        for _ in range(3):
            rd.render_features(n)
            ms.append(rd.stats["device_ms"])
        rows.append({"width": W, "height": H, "feature_samples": n, "device_ms": min(ms)})
    scene.close()
    return rows


def time_guided(mean, var, feats, out, opt, guide, min_seconds=0.3):
    """ms per launch of rt_denoise_guided_device, as denoise_bench.time_kernel times rt_denoise_device"""
    import torch
    lib = abi.load()
    H, W = mean.shape[:2]
    ptrs = [t.data_ptr() for t in (mean, var, *feats)]

    def launch():
        abi.check(lib.rt_denoise_guided_device(*ptrs, W, H, C.byref(opt), C.byref(guide), out.data_ptr(), -1, None))

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


def kernel_times(quick):
    import torch
    sizes = [(96, 96)] if quick else [(600, 600), (800, 800), (3840, 3840)]
    sweep = [(5, 2), (7, 3), (10, 2), (10, 5), (15, 3), (15, 7)]
    guide = rt.renderer.guide_struct()
    rows = []
    for (H, W) in sizes:
        mean, var = DB.synthetic(H, W)
        feats = (mean.clone(), var.clone(), mean.clone(), var.clone())
        out = torch.empty_like(mean)
        for r, f in [(DB.DEFAULTS["search_radius"], DB.DEFAULTS["patch_radius"])] + (sweep if (H, W) == sizes[min(1, len(sizes) - 1)] else []):
            opt = rt.renderer.denoise_options_struct(**dict(DB.DEFAULTS, search_radius=r, patch_radius=f))
            ms_c, _ = DB.time_kernel(mean, var, out, opt)
            ms_g, n = time_guided(mean, var, feats, out, opt, guide)
            rows.append({"width": W, "height": H, "search_radius": r, "patch_radius": f, "colour_ms": ms_c, "guided_ms": ms_g, "ratio": ms_g / ms_c,
                         "launches": n})
        del mean, var, feats, out
        torch.cuda.empty_cache()
    return rows


def regions(world, world_name, W, H, gt, noisy, outs):
    """(d): per textured sphere and the whole frame, mean / p95 display error and the share of pixels worse than noisy"""
    err = {k: np.abs(AB.display(x) - gt).max(axis=2) for k, x in dict(outs, noisy=noisy).items()}
    masks = {name: DB.sphere_disc(world, c, rad, W, H) for name, (c, rad) in DB.TEXTURED_SPHERES.get(world_name, {}).items()}
    masks["whole_image"] = np.ones((H, W), bool)
    res = {}
    for name, m in masks.items():
        res[name] = {"pixels": int(m.sum())}
        for k, e in err.items():
            res[name][k] = {"mean": float(e[m].mean()), "p95": float(np.percentile(e[m], 95))}
            if k != "noisy":
                res[name][k]["share_worse"] = float((e[m] > err["noisy"][m]).mean())
    return res


def quality(world_name, size, gt_spp, quick):
    import torch
    if quick:
        size, gt_spp = 96, 256
    world, scene, cam = AB.setup(world_name)
    W = H = size
    s1 = torch.zeros(H, W, 3, dtype=torch.int64, device="cuda")
    s2 = torch.zeros_like(s1)
    AB.render_uniform(scene, cam, s1, s2, gt_spp, seed=7)
    gt = AB.display(s1.cpu().numpy().view(np.uint64).astype(np.float64) * 2.0 ** -32 / gt_spp)

    def renderer(spp):
        return rt.Renderer.new_with_rng(cam, scene, world.background(), rt.RenderingParams(spp, H, W), rt.RecursiveRayTracer(50), rt.SeedableRngator(42))

    def noisy(spp):
        st = AB.render_uniform(scene, cam, s1, s2, spp)
        a, b = s1.cpu().numpy().view(np.uint64), s2.cpu().numpy().view(np.uint64)
        mu = a.astype(np.float64) * 2.0 ** -32 / spp
        var = np.maximum((b.astype(np.float64) * 2.0 ** -24 - spp * (mu * mu)) / (spp - 1.0), 0.0) / spp
        return mu.astype(np.float32), var.astype(np.float32), st.device_ms

    frame_mean = lambda x: [float(c) for c in np.asarray(x, np.float64).mean(axis=(0, 1))]  # noqa: E731
    renderer(16).render_denoised(guide={})  # warm-up
    renderer(16).render_denoised()
    runs = []
    for spp in DB.SPPS:
        mu, _, ms_noisy = noisy(spp)
        rc = renderer(spp)
        _, col = rc.render_denoised()
        rg = renderer(spp)
        _, gui = rg.render_denoised(guide={})
        ms_prod = AB.render_uniform(scene, cam, s1, s2, spp, moments=False).device_ms
        spp_eq = max(2, int(round(spp * rg.stats["device_ms"] / ms_prod)))
        ms_eq = AB.render_uniform(scene, cam, s1, s2, spp_eq, moments=False).device_ms
        mu_eq = s1.cpu().numpy().view(np.uint64).astype(np.float64) * 2.0 ** -32 / spp_eq
        runs.append({"spp": spp,
                     "noisy": {"device_ms": ms_noisy, "err_p50_p95_p99": AB.display_errors(mu, gt), "frame_mean": frame_mean(mu)},
                     "colour": {"device_ms": rc.stats["device_ms"], "err_p50_p95_p99": AB.display_errors(col, gt), "frame_mean": frame_mean(col)},
                     "guided": {"device_ms": rg.stats["device_ms"], "err_p50_p95_p99": AB.display_errors(gui, gt), "frame_mean": frame_mean(gui)},
                     "product_same_time_as_guided": {"spp": spp_eq, "device_ms": ms_eq, "err_p50_p95_p99": AB.display_errors(mu_eq, gt)}})
    # (d) and (e) at 64 spp: the filters on one render's mean and variance, the features of the same seed
    mu, var, _ = noisy(64)
    tm, tv = torch.from_numpy(mu).cuda(), torch.from_numpy(var).cuda()
    rd = renderer(64)
    feats = {n: [torch.from_numpy(x).cuda() for x in rd.render_features(n)] for n in (4, 16, 64)}
    col = rt.denoise(tm, tv).cpu().numpy()
    gui = rt.denoise_guided(tm, tv, *feats[GUIDE["feature_samples"]]).cpu().numpy()
    reg = regions(world, world_name, W, H, gt, mu, {"colour": col, "guided": gui})

    def score(den):
        e = np.abs(AB.display(den) - gt).max(axis=2)
        out = {"err_p50_p95_p99": AB.display_errors(den, gt), "mean": float(e.mean())}
        for name, (c, rad) in DB.TEXTURED_SPHERES.get(world_name, {}).items():
            out[name + "_mean"] = float(e[DB.sphere_disc(world, c, rad, W, H)].mean())
        return out

    sweep = []
    for kf in (0.3, 0.6, 1.0, 2.0):
        for tau in (1e-4, 1e-3, 1e-2):
            sweep.append(dict(k_feature=kf, tau=tau, feature_samples=GUIDE["feature_samples"],
                              **score(rt.denoise_guided(tm, tv, *feats[GUIDE["feature_samples"]], k_feature=kf, tau=tau).cpu().numpy())))
    for n in (4, 64):
        sweep.append(dict(k_feature=GUIDE["k_feature"], tau=GUIDE["tau"], feature_samples=n, **score(rt.denoise_guided(tm, tv, *feats[n]).cpu().numpy())))
    sweep.append(dict(colour_only=True, **score(col)))
    scene.close()
    return {"world": world_name, "size": size, "ground_truth_spp": gt_spp, "spp_runs": runs, "regions_64spp": reg, "sweep_64spp": sweep}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    if abi.load().rt_device_count() < 1:
        raise SystemExit("guided_denoise_bench needs a CUDA device")
    name, power = AB.gpu_info()
    result = {"gpu": name, "power_limit": power, "guide_defaults": GUIDE, "denoise_defaults": DB.DEFAULTS, "feature_pass": feature_times(args.quick),
              "kernel": kernel_times(args.quick), "configs": {}}
    for key, world_name, size, _, _, gt_spp, _ in AB.CONFIGS:
        result["configs"][key] = quality(world_name, size, gt_spp, args.quick)
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
