#!/usr/bin/env python
"""What dual-buffer cross filtering costs and what it buys, against the colour-only and guided filters, on C3 (cornell_smoke 600^2)
and C4 (final_scene 800^2).  Prints one JSON line; needs a CUDA device.  Reuses the jobs, ground truths (seed 7) and display-error
measure of adaptive_bench.py, the timing, synthetic inputs and sphere discs of denoise_bench.py and guided_denoise_bench.py.

(a) kernel time: the cross kernel (both directions, torch.profiler) and the whole rt_denoise_cross_device call (CUDA events)
    against rt_denoise_device and rt_denoise_guided_device, at the sizes and radii of denoise_bench (a).
(b) -Xptxas -v of the cross instances, and the blocks per SM they allow at the default radii (from registers and shared memory).
(c) quality at 16 / 64 / 256 spp: noisy, colour-only, guided, dual, dual guided, and the product path at the device time of the
    dual render: display error percentiles, the noise sphere's mean error (C4), the frame-mean shift per channel against the
    noisy image of the same samples and against the ground truth, and the calibration of eps.
(d) filter-driven adaptive sampling (min_samples 16, thresholds 0.02 / 0.01 / 0.005) against a uniform dual render at the same
    device time: mean spp, device ms, the share of it in per-round filtering (rounds x one conversion and filter of the image,
    timed apart), percentiles, and the share of early-stopped pixels off by more than 3 t.
(e) a k sweep of the dual filter at 64 spp.

usage: python tools/dual_denoise_bench.py [--out FILE] [--quick]"""
import argparse
import ctypes as C
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import denoise_bench as DB  # noqa: E402  (puts the repository and tests/ on sys.path)
import adaptive_bench as AB  # noqa: E402
import guided_denoise_bench as GB  # noqa: E402
import mu_lambda_raytracer_b200 as rt  # noqa: E402
from mu_lambda_raytracer_b200 import abi  # noqa: E402

THRESHOLDS = [0.02, 0.01, 0.005]
MIN_SAMPLES = 16


def cross_call(mean, var, out, err, opt, feats=None, guide=None):
    lib = abi.load()
    H, W = mean.shape[:2]
    f = [t.data_ptr() for t in feats] if feats is not None else [None] * 4
    mb, vb = mean.flip(0), var.flip(0)  # a second half: the same statistics, other values

    def launch():
        abi.check(lib.rt_denoise_cross_device(mean.data_ptr(), var.data_ptr(), mb.data_ptr(), vb.data_ptr(), *f, W, H, C.byref(opt),
                                              C.byref(guide) if guide is not None else None, out.data_ptr(), err.data_ptr(), -1, None))
    return launch, (mb, vb)


def time_call(launch, min_seconds=0.3):
    import torch
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    launch()
    b.record()
    b.synchronize()
    n = int(min(300, max(5, min_seconds * 1e3 / max(a.elapsed_time(b), 1e-3))))
    a.record()
    for _ in range(n):
        launch()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n, n


def kernel_ms(launch, name, n=20):
    """device ms per launch of the kernels whose name contains `name` (torch.profiler, a run of its own)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    launch()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            launch()
        torch.cuda.synchronize()
    total = sum(e.device_time_total for e in prof.key_averages() if name in e.key)
    return total / n * 1e-3


def kernel_times(quick):
    import torch
    sizes = [(96, 96)] if quick else [(600, 600), (800, 800), (3840, 3840)]
    sweep = [(5, 2), (7, 3), (10, 2), (10, 5), (15, 3), (15, 7)]
    guide = rt.renderer.guide_struct()
    rows = []
    for (H, W) in sizes:
        mean, var = DB.synthetic(H, W)
        feats = (mean.clone(), var.clone(), mean.clone(), var.clone())
        out, err = torch.empty_like(mean), torch.empty_like(mean)
        for r, f in [(DB.DEFAULTS["search_radius"], DB.DEFAULTS["patch_radius"])] + (sweep if (H, W) == sizes[min(1, len(sizes) - 1)] else []):
            opt = rt.renderer.denoise_options_struct(**dict(DB.DEFAULTS, search_radius=r, patch_radius=f))
            ms_c, _ = DB.time_kernel(mean, var, out, opt)
            ms_g, _ = GB.time_guided(mean, var, feats, out, opt, guide)
            lc, keep_c = cross_call(mean, var, out, err, opt)
            lg, keep_g = cross_call(mean, var, out, err, opt, feats, guide)
            row = {"width": W, "height": H, "search_radius": r, "patch_radius": f, "colour_ms": ms_c, "guided_ms": ms_g,
                   "cross_kernel_ms": kernel_ms(lc, "denoise_nlm_cross_kernel"), "cross_guided_kernel_ms": kernel_ms(lg, "denoise_nlm_cross_kernel"),
                   "cross_call_ms": time_call(lc)[0], "cross_guided_call_ms": time_call(lg)[0]}
            row["cross_over_colour"] = row["cross_kernel_ms"] / ms_c
            row["cross_guided_over_guided"] = row["cross_guided_kernel_ms"] / ms_g
            rows.append(row)
            del keep_c, keep_g
        del mean, var, feats, out, err
        torch.cuda.empty_cache()
    return rows


def ptxas_cross():
    """registers and spills of the cross instances, and blocks per SM at the default radii (256 threads; 64 K registers and
    228 KB of shared memory per SM, 1 KB of it reserved per block)"""
    log = os.path.join(ROOT, "mu-lambda-raytracer_b200", "build", "rt_denoise.cu.ptxas.log")
    if not os.path.exists(log):
        return None
    lines = open(log).read().split("\n")
    r, f = DB.DEFAULTS["search_radius"], DB.DEFAULTS["patch_radius"]
    R = r + f
    smem = 4 * (9 * (32 + 2 * R) * (16 + 2 * R) + (32 + 2 * f) * (16 + 2 * f) + 32 * (16 + 2 * f))
    ne_default = ((32 + 2 * f) * (16 + 2 * f) + 255) // 256
    rows = []
    for i, line in enumerate(lines):
        m = re.search(r"Compiling entry function '(\S*(denoise_nlm_cross_kernel)ILi(\d)ELb(\d)E\S*)'", line)
        if not m:
            continue
        block = " ".join(lines[i:i + 5])
        regs = int(re.search(r"Used (\d+) registers", block).group(1))
        spill = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", block)
        row = {"kernel": m.group(2), "locations_per_thread": int(m.group(3)), "guided": m.group(4) == "1", "registers": regs,
               "spill_stores": int(spill.group(1)), "spill_loads": int(spill.group(2))}
        if int(m.group(3)) == ne_default:
            by_regs = 65536 // (((regs + 7) // 8 * 8) * 256)
            row["blocks_per_sm_default_radii"] = min(by_regs, 228 * 1024 // (smem + 1024))
            row["smem_bytes_default_radii"] = smem
        rows.append(row)
    return rows


def shift(x, ref):
    return [float(c) for c in np.asarray(x, np.float64).mean(axis=(0, 1)) / np.asarray(ref, np.float64).mean(axis=(0, 1)) - 1.0]


def calibration(out, eps, gt_mean):
    pos = eps > 0
    return {"mean_sq_err_over_eps": float((((out.astype(np.float64) - gt_mean) ** 2)[pos] / eps[pos]).mean()), "share_eps_zero": float((~pos).mean())}


def quality(key, world_name, size, cap, gt_spp, quick):
    import torch
    if quick:
        size, gt_spp, cap = 96, 256, 256
    world, scene, cam = AB.setup(world_name)
    W = H = size
    s1 = torch.zeros(H, W, 3, dtype=torch.int64, device="cuda")
    s2 = torch.zeros_like(s1)
    AB.render_uniform(scene, cam, s1, s2, gt_spp, seed=7)
    gt_mean = s1.cpu().numpy().view(np.uint64).astype(np.float64) * 2.0 ** -32 / gt_spp
    gt = AB.display(gt_mean)
    sphere = DB.sphere_disc(world, *DB.TEXTURED_SPHERES[world_name]["noise_sphere"], W, H) if world_name in DB.TEXTURED_SPHERES else None

    def renderer(spp):
        return rt.Renderer.new_with_rng(cam, scene, world.background(), rt.RenderingParams(spp, H, W), rt.RecursiveRayTracer(50), rt.SeedableRngator(42))

    def errors(x, ref=None):
        e = np.abs(AB.display(x) - gt).max(axis=2)
        res = {"err_p50_p95_p99": [float(np.percentile(e, q)) for q in (50, 95, 99)], "shift_vs_gt": shift(x, gt_mean)}
        if ref is not None:
            res["shift_vs_noisy"] = shift(x, ref)
        if sphere is not None:
            res["noise_sphere_mean"] = float(e[sphere].mean())
        return res

    renderer(16).render_denoised_dual()  # warm-up
    renderer(16).render_denoised_dual(guide={})
    runs = []
    for spp in DB.SPPS:
        AB.render_uniform(scene, cam, s1, s2, spp)
        noisy = s1.cpu().numpy().view(np.uint64).astype(np.float64) * 2.0 ** -32 / spp
        row = {"spp": spp, "noisy": errors(noisy)}
        for name, call in (("colour", lambda r: r.render_denoised()), ("guided", lambda r: r.render_denoised(guide={})),
                           ("dual", lambda r: r.render_denoised_dual()), ("dual_guided", lambda r: r.render_denoised_dual(guide={}))):
            rd = renderer(spp)
            res = call(rd)
            row[name] = dict(errors(res[1], noisy), device_ms=rd.stats["device_ms"])
            if name.startswith("dual"):
                row[name]["calibration"] = calibration(res[1], res[2], gt_mean)
        ms_prod = AB.render_uniform(scene, cam, s1, s2, spp, moments=False).device_ms
        spp_eq = max(2, int(round(spp * row["dual"]["device_ms"] / ms_prod)))
        ms_eq = AB.render_uniform(scene, cam, s1, s2, spp_eq, moments=False).device_ms
        row["product_same_time_as_dual"] = dict(errors(s1.cpu().numpy().view(np.uint64).astype(np.float64) * 2.0 ** -32 / spp_eq), spp=spp_eq, device_ms=ms_eq)
        runs.append(row)

    # (d) the filter's cost per round at this size: one conversion pair and cross filter, timed through the Python entry point
    mu = torch.rand(H, W, 3, device="cuda")
    va = torch.rand(H, W, 3, device="cuda") * 1e-2
    launch, keep = cross_call(mu, va, torch.empty_like(mu), torch.empty_like(mu), rt.renderer.denoise_options_struct())
    filter_ms = time_call(launch)[0]
    del keep

    def uniform_dual_ms(spp):
        rd = renderer(spp)
        rd.render_denoised_dual()
        return rd.stats["device_ms"]
    t_lo, t_hi = uniform_dual_ms(64), uniform_dual_ms(256)
    per_spp = (t_hi - t_lo) / 192.0
    adaptive = []
    for t in THRESHOLDS:
        rd = rt.Renderer.new_with_rng(cam, scene, world.background(), rt.RenderingParams(cap, H, W), rt.RecursiveRayTracer(50), rt.SeedableRngator(42))
        _, out, eps, n = rd.render_denoised_dual(t, MIN_SAMPLES)
        ms = rd.stats["device_ms"]
        rounds = 1
        c = MIN_SAMPLES
        while c < int(n.max()):
            c += min(c, cap - c)
            rounds += 1
        e = np.abs(AB.display(out) - gt).max(axis=2)
        stopped = n < cap
        spp_eq = max(4, 2 * int(round(max(0.0, (ms - t_lo) / per_spp + 64) / 2)))
        ru = renderer(spp_eq)
        _, out_u, _, _ = ru.render_denoised_dual()
        adaptive.append({"threshold": t, "mean_spp": float(n.mean()), "device_ms": ms, "rounds": rounds, "filter_ms_per_round": filter_ms,
                         "filter_share": rounds * filter_ms / ms, "stopped_share": float(stopped.mean()),
                         "tail_share_over_3t": float((e[stopped] > 3 * t).mean()) if stopped.any() else None,
                         "adaptive": errors(out), "uniform_same_time": dict(errors(out_u), spp=spp_eq, device_ms=ru.stats["device_ms"]),
                         "calibration": calibration(out, eps, gt_mean)})
    # (e) the strength k of the dual filter at 64 spp
    sweep = []
    for k in (0.3, 0.45, 0.6, 0.9):
        AB.render_uniform(scene, cam, s1, s2, 64)
        noisy = s1.cpu().numpy().view(np.uint64).astype(np.float64) * 2.0 ** -32 / 64
        _, out, eps, _ = renderer(64).render_denoised_dual(k=k)
        sweep.append(dict(k=k, **errors(out, noisy), calibration=calibration(out, eps, gt_mean)))
    scene.close()
    return {"world": world_name, "size": size, "cap": cap, "ground_truth_spp": gt_spp, "spp_runs": runs, "adaptive": adaptive, "k_sweep_64spp": sweep,
            "uniform_dual_ms_64_256": [t_lo, t_hi]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    if abi.load().rt_device_count() < 1:
        raise SystemExit("dual_denoise_bench needs a CUDA device")
    name, power = AB.gpu_info()
    result = {"gpu": name, "power_limit": power, "denoise_defaults": DB.DEFAULTS, "kernel": kernel_times(args.quick), "ptxas": ptxas_cross(), "configs": {}}
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
