#!/usr/bin/env python
"""What SURE selection among three cross-filter strengths costs and what it buys, against the dual-buffer cross filter, on C3
(cornell_smoke 600^2) and C4 (final_scene 800^2).  Prints one JSON line; needs a CUDA device.  Reuses the jobs, ground truths
(seed 7), timing and display-error measure of dual_denoise_bench.py.

(a) kernel time: the SURE candidates kernel (both directions, torch.profiler) and the whole rt_denoise_sure_device call (CUDA
    events) against the cross kernel and rt_denoise_cross_device, at the sizes and radii of dual_denoise_bench (a).
(b) -Xptxas -v of the SURE instances, and the blocks per SM they allow at the default radii (from registers and shared memory).
(c) quality at 16 / 64 / 256 spp: colour-only, dual, dual guided, SURE and SURE guided: display error percentiles, the noise
    sphere's mean error (C4), the frame-mean shift, the share of each choice, and the calibration sum (out - gt)^2 / sum err
    (for dual: the same with eps).
(d) SURE-driven adaptive sampling (min_samples 16, thresholds 0.02 / 0.01 / 0.005) against a uniform SURE render of the same
    device time, and the share of early-stopped pixels off by more than 3 t.
(e) a sweep of ratio x smooth_radius of the SURE filter at 64 spp.

usage: python tools/sure_denoise_bench.py [--out FILE] [--quick]"""
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
import dual_denoise_bench as DD  # noqa: E402
import mu_lambda_raytracer_b200 as rt  # noqa: E402
from mu_lambda_raytracer_b200 import abi  # noqa: E402

THRESHOLDS = [0.02, 0.01, 0.005]
MIN_SAMPLES = 16


def sure_call(mean, var, out, err, choice, opt, feats=None, guide=None):
    lib = abi.load()
    H, W = mean.shape[:2]
    f = [t.data_ptr() for t in feats] if feats is not None else [None] * 4
    mb, vb = mean.flip(0), var.flip(0)  # a second half: the same statistics, other values
    sure = rt.renderer.sure_struct()

    def launch():
        abi.check(lib.rt_denoise_sure_device(mean.data_ptr(), var.data_ptr(), mb.data_ptr(), vb.data_ptr(), *f, W, H, C.byref(opt),
                                             C.byref(guide) if guide is not None else None, C.byref(sure), out.data_ptr(), err.data_ptr(),
                                             choice.data_ptr(), -1, None))
    return launch, (mb, vb, sure)


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
        choice = torch.empty(H, W, dtype=torch.int32, device="cuda")
        for r, f in [(DB.DEFAULTS["search_radius"], DB.DEFAULTS["patch_radius"])] + (sweep if (H, W) == sizes[min(1, len(sizes) - 1)] else []):
            opt = rt.renderer.denoise_options_struct(**dict(DB.DEFAULTS, search_radius=r, patch_radius=f))
            row = {"width": W, "height": H, "search_radius": r, "patch_radius": f}
            for guided in (False, True):
                g = "_guided" if guided else ""
                fe, gd = (feats, guide) if guided else (None, None)
                lc, keep_c = DD.cross_call(mean, var, out, err, opt, fe, gd)
                ls, keep_s = sure_call(mean, var, out, err, choice, opt, fe, gd)
                row[f"cross{g}_kernel_ms"] = DD.kernel_ms(lc, "denoise_nlm_cross_kernel")
                row[f"sure{g}_kernel_ms"] = DD.kernel_ms(ls, "denoise_nlm_sure_kernel")
                row[f"sure{g}_risk_select_ms"] = DD.kernel_ms(ls, "sure_risk_kernel") + DD.kernel_ms(ls, "sure_select_kernel")
                row[f"cross{g}_call_ms"] = DD.time_call(lc)[0]
                row[f"sure{g}_call_ms"] = DD.time_call(ls)[0]
                row[f"sure{g}_kernel_over_cross"] = row[f"sure{g}_kernel_ms"] / row[f"cross{g}_kernel_ms"]
                row[f"sure{g}_call_over_cross"] = row[f"sure{g}_call_ms"] / row[f"cross{g}_call_ms"]
                del keep_c, keep_s
            rows.append(row)
        del mean, var, feats, out, err, choice
        torch.cuda.empty_cache()
    return rows


def ptxas_sure():
    """registers and spills of the SURE instances, and blocks per SM at the default radii (256 threads; 64 K registers and
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
        m = re.search(r"Compiling entry function '(\S*(denoise_nlm_sure_kernel|denoise_nlm_cross_kernel)ILi(\d)ELb(\d)E\S*)'", line)
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


def calibration(out, err, gt_mean):
    """sum (out - gt)^2 / sum err"""
    return float(((out.astype(np.float64) - gt_mean) ** 2).sum() / max(float(err.astype(np.float64).sum()), 1e-300))


def quality(world_name, size, cap, gt_spp, quick):
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
        res = {"err_p50_p95_p99": [float(np.percentile(e, q)) for q in (50, 95, 99)], "shift_vs_gt": DD.shift(x, gt_mean)}
        if ref is not None:
            res["shift_vs_noisy"] = DD.shift(x, ref)
        if sphere is not None:
            res["noise_sphere_mean"] = float(e[sphere].mean())
        return res

    renderer(16).render_denoised_sure()  # warm-up
    renderer(16).render_denoised_sure(guide={})
    runs = []
    for spp in DB.SPPS:
        AB.render_uniform(scene, cam, s1, s2, spp)
        noisy = s1.cpu().numpy().view(np.uint64).astype(np.float64) * 2.0 ** -32 / spp
        row = {"spp": spp, "noisy": errors(noisy)}
        for name, call in (("colour", lambda r: r.render_denoised()), ("dual", lambda r: r.render_denoised_dual()),
                           ("dual_guided", lambda r: r.render_denoised_dual(guide={})), ("sure", lambda r: r.render_denoised_sure()),
                           ("sure_guided", lambda r: r.render_denoised_sure(guide={}))):
            rd = renderer(spp)
            res = call(rd)
            row[name] = dict(errors(res[1], noisy), device_ms=rd.stats["device_ms"])
            if name != "colour":
                row[name]["calibration"] = calibration(res[1], res[2], gt_mean)
            if name.startswith("sure"):
                row[name]["choice_shares"] = [float((res[4] == j).mean()) for j in range(3)]
        runs.append(row)

    def uniform_sure_ms(spp):
        rd = renderer(spp)
        rd.render_denoised_sure()
        return rd.stats["device_ms"]
    t_lo, t_hi = uniform_sure_ms(64), uniform_sure_ms(256)
    per_spp = (t_hi - t_lo) / 192.0
    adaptive = []
    for t in THRESHOLDS:
        rd = rt.Renderer.new_with_rng(cam, scene, world.background(), rt.RenderingParams(cap, H, W), rt.RecursiveRayTracer(50), rt.SeedableRngator(42))
        _, out, err, n, choice = rd.render_denoised_sure(t, MIN_SAMPLES)
        ms = rd.stats["device_ms"]
        e = np.abs(AB.display(out) - gt).max(axis=2)
        stopped = n < cap
        spp_eq = max(4, 2 * int(round(max(0.0, (ms - t_lo) / per_spp + 64) / 2)))
        ru = renderer(spp_eq)
        _, out_u, _, _, _ = ru.render_denoised_sure()
        adaptive.append({"threshold": t, "mean_spp": float(n.mean()), "device_ms": ms, "stopped_share": float(stopped.mean()),
                         "tail_share_over_3t": float((e[stopped] > 3 * t).mean()) if stopped.any() else None,
                         "adaptive": errors(out), "uniform_same_time": dict(errors(out_u), spp=spp_eq, device_ms=ru.stats["device_ms"]),
                         "calibration": calibration(out, err, gt_mean)})
    sweep = []
    AB.render_uniform(scene, cam, s1, s2, 64)
    noisy = s1.cpu().numpy().view(np.uint64).astype(np.float64) * 2.0 ** -32 / 64
    for ratio in (1.5, 2.0, 3.0):
        for b in (1, 2, 3, 5):
            _, out, err, _, choice = renderer(64).render_denoised_sure(ratio=ratio, smooth_radius=b)
            sweep.append(dict(ratio=ratio, smooth_radius=b, **errors(out, noisy), calibration=calibration(out, err, gt_mean),
                              choice_shares=[float((choice == j).mean()) for j in range(3)]))
    scene.close()
    return {"world": world_name, "size": size, "cap": cap, "ground_truth_spp": gt_spp, "spp_runs": runs, "adaptive": adaptive,
            "sweep_64spp": sweep, "uniform_sure_ms_64_256": [t_lo, t_hi]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    if abi.load().rt_device_count() < 1:
        raise SystemExit("sure_denoise_bench needs a CUDA device")
    name, power = AB.gpu_info()
    result = {"gpu": name, "power_limit": power, "denoise_defaults": DB.DEFAULTS,
              "sure_defaults": {"ratio": abi.RT_SURE_DEFAULT_RATIO, "smooth_radius": abi.RT_SURE_DEFAULT_SMOOTH_RADIUS},
              "kernel": kernel_times(args.quick), "ptxas": ptxas_sure(), "configs": {}}
    for key, world_name, size, cap, _, gt_spp, _ in AB.CONFIGS:
        result["configs"][key] = quality(world_name, size, cap, gt_spp, args.quick)
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
