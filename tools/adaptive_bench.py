#!/usr/bin/env python
"""What per-pixel moments cost and what noise-threshold adaptive sampling buys, on C3 (cornell_smoke 600^2, cap 1000 spp)
and C4 (final_scene 800^2, cap 10 000 spp).  Prints one JSON line; needs a CUDA device.

(a) the moments family (rt_render_moments_fixed_device) against the product instance (rt_render_accumulate_fixed_device) on
    the same uniform job, alternated in one run, best of `--reps`; the registers / spills of both instances from the
    build's `-Xptxas -v` log.
(b) for each threshold: device time, mean spp and the 50/95/99th percentile of the display error (largest channel, after
    the gamma-2 tonemap) against a uniform ground truth of `gt_spp` samples with another seed — and the same for a uniform
    render at the adaptive render's mean spp.

usage: python tools/adaptive_bench.py [--out FILE] [--reps N] [--quick]"""
import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import mu_lambda_raytracer_b200 as rt  # noqa: E402
from mu_lambda_raytracer_b200 import abi  # noqa: E402

# name, world, size, cap, spp of the uniform job of (a), ground-truth spp, thresholds
CONFIGS = [("C3", "cornell_smoke", 600, 1000, 1000, 8000, [0.02, 0.01, 0.005]),
           ("C4", "final_scene", 800, 10000, 2000, 20000, [0.02, 0.01, 0.005])]
INSTANCES = {"C3": ("persist_kernelILb0ELb1ELi0ELi768ELi0ELi0ELi2ELb0ELj103ELb0E", "persist_moments_kernelILb1ELi768ELi0ELj103E"),
             "C4": ("persist_kernelILb0ELb1ELi0ELi768ELi0ELi0ELi2ELb0ELj1845ELb0E", "persist_moments_kernelILb1ELi768ELi0ELj1845E")}


def ptxas_usage(substr):
    log = os.path.join(ROOT, "mu-lambda-raytracer_b200", "build", "rt_persist.cu.ptxas.log")
    if not os.path.exists(log):
        return None
    lines = open(log).read().split("\n")
    for i, l in enumerate(lines):
        if "Compiling entry function" in l and substr in l:
            spill = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", lines[i + 2] if "Function properties" in lines[i + 1] else lines[i + 1])
            regs = next(re.search(r"Used (\d+) registers", x).group(1) for x in lines[i:i + 6] if "Used" in x)
            return {"registers": int(regs), "spill_stores": int(spill.group(1)), "spill_loads": int(spill.group(2))}
    return None


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True)
    name, power = [x.strip() for x in q.stdout.strip().split("\n")[0].split(",")]
    return name, power


def setup(world_name):
    """(world, scene, camera) of a square job of the world at its own camera"""
    import support as S
    world = rt.World(world_name)
    scene = rt.Scene(world.build(42))
    info = world.camera()
    return world, scene, S.make_camera(info["lookfrom"], info["lookat"], info["field_of_view"], 1.0)


def params(W, H, spp, seed=42, begin=0, count=0):
    p = abi.RtParams()
    p.width, p.height, p.samples_per_pixel, p.max_depth, p.seed = W, H, spp, 50, seed
    p.sample_begin, p.sample_count, p.pipeline, p.device = begin, count, abi.RT_PIPELINE_AUTO, -1
    return p


def render_uniform(scene, cam, s1, s2, spp, seed=42, moments=True):
    """a uniform render of spp samples into the zeroed device sums s1, s2 (int64 tensors [H, W, 3]); returns RtStats"""
    import torch
    H, W = s1.shape[:2]
    lib = abi.load()
    s1.zero_(), s2.zero_()
    st = abi.RtStats()
    if moments:
        abi.check(lib.rt_render_moments_fixed_device(scene.handle, C.byref(cam.c), C.byref(params(W, H, spp, seed)), s1.data_ptr(), s2.data_ptr(), None,
                                                     C.byref(st)))
    else:
        abi.check(lib.rt_render_accumulate_fixed_device(scene.handle, C.byref(cam.c), C.byref(params(W, H, spp, seed)), s1.data_ptr(), None, C.byref(st)))
    torch.cuda.synchronize()
    return st


def display(mean):
    """the displayed value of a radiance: gamma 2 of the clamped mean"""
    return np.sqrt(np.clip(np.asarray(mean, np.float64), 0.0, 1.0))


def display_errors(mean, gt):
    """50th / 95th / 99th percentile over the pixels of the largest channel's display error against gt = display(truth)"""
    e = np.abs(display(mean) - gt).max(axis=2)
    return [float(np.percentile(e, q)) for q in (50, 95, 99)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    import torch
    lib = abi.load()
    if lib.rt_device_count() < 1:
        raise SystemExit("adaptive_bench needs a CUDA device")
    name, power = gpu_info()
    result = {"gpu": name, "power_limit": power, "configs": {}}
    for key, world_name, size, cap, job_spp, gt_spp, thresholds in CONFIGS:
        if args.quick:
            size, cap, job_spp, gt_spp = 96, 64, 32, 256
        world, scene, cam = setup(world_name)
        W = H = size
        s1 = torch.zeros(H, W, 3, dtype=torch.int64, device="cuda")
        s2 = torch.zeros_like(s1)

        def uniform(spp, seed=42, moments=True):
            return render_uniform(scene, cam, s1, s2, spp, seed, moments)

        # (a) cost of the family on a uniform job
        uniform(min(job_spp, 16)), uniform(min(job_spp, 16), moments=False)  # warm-up: module load, grid sizing
        rates = {"moments": [], "product": []}
        for _ in range(args.reps):
            for k, mom in (("product", False), ("moments", True)):
                st = uniform(job_spp, moments=mom)
                rates[k].append(st.paths / (st.device_ms * 1e3))
        prod_inst, mom_inst = INSTANCES[key]
        cost = {"spp": job_spp, "mpaths_per_s_product": rates["product"], "mpaths_per_s_moments": rates["moments"],
                "moments_over_product_best": max(rates["moments"]) / max(rates["product"]),
                "ptxas_product": ptxas_usage(prod_inst), "ptxas_moments": ptxas_usage(mom_inst)}
        # (b) what adaptivity buys
        uniform(gt_spp, seed=7)
        gt = display(s1.cpu().numpy().view(np.uint64).astype(np.float64) * 2.0 ** -32 / gt_spp)

        def errors(acc, n):
            return display_errors(acc.astype(np.float64) * 2.0 ** -32 / n, gt)

        runs = []
        for t in thresholds:
            r = rt.Renderer.new_with_rng(cam, scene, world.background(), rt.RenderingParams(cap, H, W), rt.RecursiveRayTracer(50), rt.SeedableRngator(42))
            _, n, acc, _ = r.render_adaptive(t, 16)
            ad = {"threshold": t, "device_ms": r.stats["device_ms"], "mean_spp": float(n.mean()), "at_cap": float((n == cap).mean()),
                  "err_p50_p95_p99": errors(acc, n[..., None].astype(np.float64))}
            spp_u = max(2, int(round(n.mean())))
            st = uniform(spp_u)
            un = {"spp": spp_u, "device_ms": st.device_ms, "err_p50_p95_p99": errors(s1.cpu().numpy().view(np.uint64), float(spp_u))}
            runs.append({"adaptive": ad, "uniform_same_mean_spp": un})
        st = uniform(cap)
        full = {"spp": cap, "device_ms": st.device_ms, "err_p50_p95_p99": errors(s1.cpu().numpy().view(np.uint64), float(cap))}
        result["configs"][key] = {"world": world_name, "size": size, "cap": cap, "ground_truth_spp": gt_spp, "cost": cost, "thresholds": runs,
                                  "uniform_at_cap": full}
        scene.close()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
