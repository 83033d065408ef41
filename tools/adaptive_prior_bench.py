#!/usr/bin/env python
"""What the neighbourhood variance prior of the stop rules costs and what it buys, on C3 (cornell_smoke 600^2, cap 1000) and C4
(final_scene 800^2, cap 10 000).  Prints one JSON line; needs a CUDA device.  Reuses the jobs, ground truths (seed 7), timing
and display-error measure of adaptive_bench.py and sure_denoise_bench.py.

(a) sweep: prior_samples n0 in {4, 16, 64} x radius b in {1, 3, 5, 7} of the plain prior rule at t = 0.01, min_samples 16, on C3
    and C4 (device time, mean spp, display-error percentiles, the early-stop tail), and the early-stop tail of each on
    cornell_smoke 128^2 (cap 1024, 4096-spp ground truth, as test_adaptive_prior.test_prior_rule_is_useful).  The defaults are
    the point of least max over the two scenes of p95 * sqrt(device_ms): for Monte Carlo noise at a fixed cost per path, error
    times the square root of time is constant, so a lower value is a better use of device time.
(b) the plain prior rule (default prior) at t = 0.02 / 0.01 / 0.005 against a uniform render of the same device time, and the
    rule without a prior, with p50 / p95 / p99 and the mean spp.
(c) the SURE prior rule against a uniform SURE render of the same device time, on the jobs of sure_denoise_bench (d).
(d) the early-stop tail on cornell_smoke 128^2 at t = 0.01 for both rules, with and without the prior.
(e) cost: per-round kernel time by kind (render, evaluation, compaction, other) and the remainder of device time (gaps:
    synchronisation and launch), from torch.profiler, for the plain rule with and without the prior on C3 and C4 and on
    cornell_smoke 3840^2; the scratch bytes the prior adds.

usage: python tools/adaptive_prior_bench.py [--out FILE] [--quick]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import adaptive_bench as AB  # noqa: E402  (puts the repository and tests/ on sys.path)
import mu_lambda_raytracer_b200 as rt  # noqa: E402
from mu_lambda_raytracer_b200 import abi  # noqa: E402

THRESHOLDS = [0.02, 0.01, 0.005]
MIN_SAMPLES = 16
SWEEP_N0 = [4.0, 16.0, 64.0]
SWEEP_B = [1, 3, 5, 7]


def renderer(world, scene, cam, W, H, spp):
    return rt.Renderer.new_with_rng(cam, scene, world.background(), rt.RenderingParams(spp, H, W), rt.RecursiveRayTracer(50), rt.SeedableRngator(42))


def ground_truth(scene, cam, W, H, spp):
    import torch
    s1 = torch.zeros(H, W, 3, dtype=torch.int64, device="cuda")
    s2 = torch.zeros_like(s1)
    AB.render_uniform(scene, cam, s1, s2, spp, seed=7)
    return AB.display(s1.cpu().numpy().view(np.uint64).astype(np.float64) * 2.0 ** -32 / spp)


def display_error(mean, gt):
    return np.abs(AB.display(mean) - gt).max(axis=2)


def summary(mean, gt, n, cap, t, ms):
    e = display_error(mean, gt)
    stopped = n < cap
    return {"device_ms": ms, "mean_spp": float(n.mean()), "err_p50_p95_p99": [float(np.percentile(e, q)) for q in (50, 95, 99)],
            "stopped_share": float(stopped.mean()), "tail_share_over_3t": float((e[stopped] > 3 * t).mean()) if stopped.any() else None}


def plain(world, scene, cam, W, H, cap, t, prior, reps=1):
    """the mean and counts of an adaptive render, and its least device time over reps runs (the outputs repeat bit for bit)"""
    rd = renderer(world, scene, cam, W, H, cap)
    ms = []
    for _ in range(reps):
        _, n, acc, _ = rd.render_adaptive(t, MIN_SAMPLES, prior=prior)
        ms.append(rd.stats["device_ms"])
    return acc.astype(np.float64) * 2.0 ** -32 / n[..., None], n, min(ms)


def sure(world, scene, cam, W, H, cap, t, prior):
    rd = renderer(world, scene, cam, W, H, cap)
    _, out, _, n, _ = rd.render_denoised_sure(t, MIN_SAMPLES, prior=prior)
    return out, n, rd.stats["device_ms"]


def tail_128(world, scene, cam, gt, rule, prior, t=0.01):
    mean, n, ms = rule(world, scene, cam, 128, 128, 1024, t, prior)
    return summary(mean, gt, n, 1024, t, ms)


def uniform_same_time(world, scene, cam, W, H, ms, per_spp, gt):
    """a uniform moments render whose device time matches ms (spp from the measured time per spp)"""
    import torch
    spp = max(2, int(round(ms / per_spp)))
    s1 = torch.zeros(H, W, 3, dtype=torch.int64, device="cuda")
    s2 = torch.zeros_like(s1)
    st = AB.render_uniform(scene, cam, s1, s2, spp)
    e = display_error(s1.cpu().numpy().view(np.uint64).astype(np.float64) * 2.0 ** -32 / spp, gt)
    return {"spp": spp, "device_ms": st.device_ms, "err_p50_p95_p99": [float(np.percentile(e, q)) for q in (50, 95, 99)]}


def breakdown(world, scene, cam, W, H, cap, t, prior):
    """kernel time by kind over one adaptive render (torch.profiler), and the rest of device time"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    rd = renderer(world, scene, cam, W, H, cap)
    rd.render_adaptive(t, MIN_SAMPLES, prior=prior)  # warm-up
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        rd.render_adaptive(t, MIN_SAMPLES, prior=prior)
        torch.cuda.synchronize()
    kinds = {"render": 0.0, "evaluation": 0.0, "compaction": 0.0, "other": 0.0}
    copies_ms = 0.0  # the device-to-host copies of the results, after the timed window
    prior_eval_us = []
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name, us = ev.name, ev.device_time
        if "memcpy" in name.lower():
            copies_ms += us / 1e3
            continue
        if "memset" in name.lower():
            k = "other"
        elif "persist_moments" in name:
            k = "render"
        elif "prior_eval" in name or "prior_term" in name or "adaptive_eval" in name:
            k = "evaluation"
            if "prior_eval" in name or "prior_term" in name:
                prior_eval_us.append(us)
        elif "DeviceSelect" in name or "cub" in name.lower():
            k = "compaction"
        else:
            k = "other"
        kinds[k] += us / 1e3
    # device_ms of a run without the profiler
    _, n, _, _ = rd.render_adaptive(t, MIN_SAMPLES, prior=prior)
    ms = rd.stats["device_ms"]
    n_rounds = 0
    n_done = 0
    while n_done < cap:
        n_done += MIN_SAMPLES if n_done == 0 else min(n_done, cap - n_done)
        n_rounds += 1
    busy = sum(kinds.values())
    return {"width": W, "height": H, "cap": cap, "threshold": t, "prior": prior, "device_ms": ms, "paths": int(n.astype(np.int64).sum()),
            "render_mpaths_per_s": float(n.astype(np.int64).sum()) / (kinds["render"] * 1e3), "rounds_max": n_rounds, "kernel_ms": kinds,
            "copies_ms_untimed": copies_ms, "gaps_ms": ms - busy, "evaluation_share": kinds["evaluation"] / ms,
            "prior_kernels": {"launches": len(prior_eval_us), "total_ms": sum(prior_eval_us) / 1e3}}


def config(key, world_name, size, cap, gt_spp, quick):
    if quick:
        size, cap, gt_spp = 96, 256, 256
    world, scene, cam = AB.setup(world_name)
    W = H = size
    gt = ground_truth(scene, cam, W, H, gt_spp)
    plain(world, scene, cam, W, H, min(cap, 64), 0.01, {})  # warm-up
    res = {"world": world_name, "size": size, "cap": cap, "ground_truth_spp": gt_spp}
    sweep = []
    for n0 in SWEEP_N0:
        for b in SWEEP_B:
            mean, n, ms = plain(world, scene, cam, W, H, cap, 0.01, dict(radius=b, prior_samples=n0))
            row = dict(prior_samples=n0, radius=b, **summary(mean, gt, n, cap, 0.01, ms))
            row["p95_sqrt_ms"] = row["err_p50_p95_p99"][1] * float(np.sqrt(ms))
            sweep.append(row)
    res["sweep_t001"] = sweep
    # uniform time per spp from two uniform renders
    import torch
    s1 = torch.zeros(H, W, 3, dtype=torch.int64, device="cuda")
    s2 = torch.zeros_like(s1)
    lo, hi = (64, 256) if not quick else (16, 64)
    t_lo, t_hi = AB.render_uniform(scene, cam, s1, s2, lo).device_ms, AB.render_uniform(scene, cam, s1, s2, hi).device_ms
    per_spp = t_hi / hi
    res["uniform_ms"] = {str(lo): t_lo, str(hi): t_hi, "uniform_mpaths_per_s": W * H * hi / (t_hi * 1e3)}
    runs = []
    for t in THRESHOLDS:
        row = {"threshold": t}
        for name, prior in (("prior_default", {}), ("no_prior", None)):
            mean, n, ms = plain(world, scene, cam, W, H, cap, t, prior, reps=2)
            row[name] = summary(mean, gt, n, cap, t, ms)
            row[name]["uniform_same_time"] = uniform_same_time(world, scene, cam, W, H, ms, per_spp, gt)
        runs.append(row)
    res["plain_vs_uniform"] = runs

    def uniform_sure(spp):
        rd = renderer(world, scene, cam, W, H, spp)
        _, out, _, _, _ = rd.render_denoised_sure()
        return out, rd.stats["device_ms"]
    _, s_lo = uniform_sure(64)
    _, s_hi = uniform_sure(256)
    per_spp_sure = (s_hi - s_lo) / 192.0
    sruns = []
    for t in THRESHOLDS:
        row = {"threshold": t}
        for name, prior in (("prior_default", {}), ("no_prior", None)):
            out, n, ms = sure(world, scene, cam, W, H, cap, t, prior)
            row[name] = summary(out, gt, n, cap, t, ms)
            spp_eq = max(4, 2 * int(round(max(0.0, (ms - s_lo) / per_spp_sure + 64) / 2)))
            out_u, ms_u = uniform_sure(spp_eq)
            e = display_error(out_u, gt)
            row[name]["uniform_sure_same_time"] = {"spp": spp_eq, "device_ms": ms_u, "err_p50_p95_p99": [float(np.percentile(e, q)) for q in (50, 95, 99)]}
        sruns.append(row)
    res["sure_vs_uniform_sure"] = sruns
    res["breakdown"] = [breakdown(world, scene, cam, W, H, cap, 0.01, p) for p in ({}, None)]
    scene.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    if abi.load().rt_device_count() < 1:
        raise SystemExit("adaptive_prior_bench needs a CUDA device")
    name, power = AB.gpu_info()
    result = {"gpu": name, "power_limit": power, "defaults": {"prior_samples": abi.RT_PRIOR_DEFAULT_SAMPLES, "radius": abi.RT_PRIOR_DEFAULT_RADIUS},
              "scratch_bytes_per_pixel": {"plain": 4 * 8, "sure": 8 * 8 + 6 * 4}, "configs": {}}
    # (d) and the 128^2 tail of every sweep point
    world, scene, cam = AB.setup("cornell_smoke")
    gt = ground_truth(scene, cam, 128, 128, 4096)
    tails = {"plain_no_prior": tail_128(world, scene, cam, gt, plain, None), "plain_prior_default": tail_128(world, scene, cam, gt, plain, {}),
             "sure_no_prior": tail_128(world, scene, cam, gt, sure, None), "sure_prior_default": tail_128(world, scene, cam, gt, sure, {}),
             "plain_sweep": [dict(prior_samples=n0, radius=b, **tail_128(world, scene, cam, gt, plain, dict(radius=b, prior_samples=n0)))
                             for n0 in SWEEP_N0 for b in SWEEP_B],
             "sure_sweep": [dict(prior_samples=n0, radius=b, **tail_128(world, scene, cam, gt, sure, dict(radius=b, prior_samples=n0)))
                            for n0 in SWEEP_N0 for b in SWEEP_B]}
    result["tail_cornell_smoke_128"] = tails
    size = 512 if args.quick else 3840
    result["breakdown_cornell_smoke_%d" % size] = [breakdown(world, scene, cam, size, size, 64, 0.01, p) for p in ({}, None)]
    scene.close()
    for key, world_name, size, cap, _, gt_spp, _ in AB.CONFIGS:
        result["configs"][key] = config(key, world_name, size, cap, gt_spp, args.quick)
        sys.stderr.write(f"{key} done\n")
    # the sweep's choice
    score = {}
    for key, c in result["configs"].items():
        for row in c["sweep_t001"]:
            k = (row["prior_samples"], row["radius"])
            score[k] = max(score.get(k, 0.0), row["p95_sqrt_ms"])
    best = min(score, key=score.get)
    result["sweep_choice"] = {"prior_samples": best[0], "radius": best[1], "max_p95_sqrt_ms": score[best]}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
