#!/usr/bin/env python
"""Headline benchmark: Mpaths/s (camera paths per second) on final_scene 800x800, seed 42 (BASELINE.json C4).

  python bench.py --gpus N --steps K --warmup W            this repo's CUDA path (one rank per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W    the reference algorithm on the host CPU cores

A "step" is one pass of the hot path over the FIXED job the reference's README quotes (src/raytrace.rs:172-186 renders
one whole image): the full 800x800 frame at 10 000 samples per pixel = 6.4 G camera paths (`--c5`: 3840x3840 at 4096 spp).
With N GPUs the job's sample range is split into N slices (rt_sample_slice), so per-GPU work shrinks as N grows:
STRONG scaling.  Inside the timed region of every step: the slice render on every rank, the one exchange step of the
path (an exact integer reduce of the fixed-point accumulation buffers onto rank 0 over NCCL) and the tonemap.  Every step
renders the same samples, so every step — at every N — must produce the same image; its checksum is part of the line.

The reference is a Rust program and there is no Rust toolchain in this image, so the reference arm times the oracle —
the C++ f64 restatement of the reference's algorithm (oracle/) — on all host cores, on a bounded sample of the same job.

`--dump-outputs DIR` writes what the last timed step computed (see dump_outputs) as DIR/<name>.npy.  The job is fixed
by the arguments and seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes as C
import glob
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

SEED, MAX_DEPTH = 42, 50
WORKLOADS = {  # BASELINE.json configs[3] (the metric's config) and configs[4]
    "c4": {"world": "final_scene", "width": 800, "height": 800, "aspect": 1.0, "job_spp": 10000},
    "c5": {"world": "final_scene", "width": 3840, "height": 3840, "aspect": 1.0, "job_spp": 4096},
}


def baseline_metric():
    """the headline metric exactly as BASELINE.json words it (unit: Mpaths/s = million camera paths per second)"""
    try:
        with open(os.path.join(ROOT, "BASELINE.json")) as f:
            return json.load(f)["metric"]
    except Exception:
        return "Mpaths/s on final_scene 800x800 (device-timed) vs host-CPU reference"


# Algorithmic work of the REFERENCE's traversal per camera path on C4 (SURVEY §8d): counted by the oracle's
# instrumentation.  At N = 1 the counters of THIS run's CPU-baseline leg are used; this frozen copy (tests/golden/
# algo_work.py at 16 spp, BASELINE.md section 4) is the fallback for runs that skip that leg (N > 1, --cpu-spp 0).
ALGO_FROZEN = {"rays": 4.159, "aabb": 66.59, "sphere": 42.99, "rect": 60.77, "xform": 8.318, "medium": 8.318,
               "lambertian": 0.878, "metal": 0.0312, "dielectric": 0.315, "isotropic": 1.963, "perlin": 0.0682, "image": 0.0695,
               "background": 0.886}


def algo_flops_per_path(a):
    """flops = 27 aabb + 45 sphere + 15 rect + 12 xform + 40 medium + shade terms (SURVEY §8d)"""
    geometry = 27 * a["aabb"] + 45 * a["sphere"] + 15 * a["rect"] + 12 * a["xform"] + 40 * a["medium"]
    shade = (40 * a["lambertian"] + 60 * a["metal"] + 80 * a["dielectric"] + 25 * a["isotropic"] + 1400 * a["perlin"]
             + 55 * a["image"] + 20 * a["background"])
    return geometry + shade


def algo_bytes_per_path(a):
    """32 B per node / primitive record the reference's traversal touches (+ 48 B per medium test)"""
    return 32 * (a["aabb"] + a["sphere"] + a["rect"]) + 48 * a["medium"]


def profiled_traffic():
    """DRAM and L2 bytes per camera path of the dominant kernel, from the newest committed ncu --set full capture
    (profiles/r*_persist_traffic.json, written by tools/ncu_traffic.py with the commit it was taken at)"""
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_persist_traffic.json")))
    if not files:
        return None
    try:
        with open(files[-1]) as f:
            d = json.load(f)
        d["file"] = os.path.relpath(files[-1], ROOT)
        return d
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(s) > 3 + k and s[3 + k].lower().startswith("active") for s in self.samples)]
        power = [float(s[2]) for s in self.samples if s[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "power_w_max": max(power) if power else None, "samples": len(self.samples), "reasons": reasons}


def driver_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "MEASURED_PEAKS.json"
    except Exception:
        return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback of B200_PROFILING.md"


def cpu_reference_run(wl, spp, steps, warmup, threads=0):
    """Times the oracle (reference algorithm, f64, PCG64 row streams, row-parallel) on the full frame at `spp` samples
    per step.  Returns (Mpaths/s, ms per step, cores, per-path counters of the reference's traversal)."""
    import support as S
    ow = S.OracleWorld(wl["world"], SEED)
    cam = S.make_camera(ow.lookfrom, ow.lookat, ow.vfov, wl["aspect"])
    cores = threads or S.oracle().orc_hardware_threads()
    for w in range(warmup):
        ow.render(cam.c, wl["width"], wl["height"], 1, MAX_DEPTH, render_seed=SEED + 100000 * (w + 1), threads=cores, rows=(0, max(8, wl["height"] // 10)))
    secs, total = 0.0, np.zeros(16, dtype=np.float64)
    for k in range(steps):
        _, _, counters, s = ow.render(cam.c, wl["width"], wl["height"], spp, MAX_DEPTH, render_seed=SEED + 1000 * k, threads=cores)
        secs += s
        total += counters.astype(np.float64)
    per_path = {name: total[i] / max(total[0], 1.0) for i, name in enumerate(S.COUNTER_NAMES)}
    return total[0] / secs / 1e6, 1e3 * secs / steps, cores, per_path


DUMP_SAMPLE_PIXELS = 1 << 20  # 44 B per sampled pixel in the three files: 44 MB, under the 64 MB a dump may take


def dump_outputs(out_dir, rgb, accum):
    """Writes what the timed path hands its caller (distributed.render_sharded on rank 0) as float .npy files:
    rgb.npy, the tonemapped 8-bit image as float32, and accum.npy, the radiance sums per pixel and channel as float64
    (the int64 fixed-point sums times 2^-32: exact while a sum stays below 2^21).  Both are [H, W, 3] with row 0 at the
    bottom.  An image of more than DUMP_SAMPLE_PIXELS pixels is reduced to the same fixed, seeded sample of pixels in both
    files ([n, 3]), and pixel.npy holds the row-major index of each sampled pixel."""
    from mu_lambda_raytracer_b200 import abi
    H, W = rgb.shape[:2]
    out = {"rgb": rgb.cpu().numpy().astype(np.float32),
           "accum": accum.cpu().numpy().astype(np.float64) / abi.RT_ACCUM_FIXED_ONE}
    if H * W > DUMP_SAMPLE_PIXELS:
        pixel = np.sort(np.random.default_rng(SEED).choice(H * W, DUMP_SAMPLE_PIXELS, replace=False))
        out = {name: a.reshape(H * W, 3)[pixel] for name, a in out.items()}
        out["pixel"] = pixel.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_name(wl):
    return f"{'C5' if wl['width'] == 3840 else 'C4'} {wl['world']} {wl['width']}x{wl['height']} seed {SEED} max_depth {MAX_DEPTH}"


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    spp = args.ref_spp
    value, ms, cores, per_path = cpu_reference_run(wl, spp, args.steps, args.warmup)
    npix = wl["width"] * wl["height"]
    sample = (f"full {wl['width']}x{wl['height']} frame at {spp} spp per step ({npix * spp} camera paths; the job is {wl['job_spp']} spp: "
              f"cost is linear in spp, raytrace.rs:190-195), max_depth {MAX_DEPTH}")
    line = {
        "impl": "reference", "metric": baseline_metric(), "value": value, "unit": "Mpaths/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload_name(wl), "job_spp": wl["job_spp"], "spp_per_step": spp,
                   "note": "reference = C++ f64 restatement of the Rust renderer (oracle/); no Rust toolchain in this image"},
        "cpu_baseline": {"value": value, "unit": "Mpaths/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "rays_per_path": per_path["rays"], "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def run_b200(args, wl):
    import torch
    import mu_lambda_raytracer_b200 as rt
    from mu_lambda_raytracer_b200 import abi, distributed

    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the render path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world_size > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        host_group = dist.new_group(backend="gloo")  # host-side waits that keep the GPUs free (an NCCL barrier spins a kernel on them)
    lib = abi.load()
    dev = torch.device("cuda", local_rank)
    W, H = wl["width"], wl["height"]
    job_spp = args.spp if args.spp > 0 else wl["job_spp"]
    paths_per_step = W * H * job_spp

    peaks = None
    if rank == 0:  # the ceilings the roofline is quoted against, measured on this device in this run
        pk = abi.RtPeaks()
        abi.check(lib.rt_measure_peaks(local_rank, C.byref(pk)))
        peaks = {k: getattr(pk, k) for k, _ in abi.RtPeaks._fields_ if k != "reserved"}

    world = rt.World(wl["world"])
    desc = world.build(SEED)
    scene = rt.Scene(desc, device=local_rank)
    info = world.camera()
    focus = float(np.linalg.norm(np.asarray(info["lookat"]) - np.asarray(info["lookfrom"])))
    cam = rt.Camera(info["lookfrom"], info["lookat"], (0, 1, 0), info["field_of_view"], wl["aspect"], 0.0, focus)
    pipeline = {"auto": abi.RT_PIPELINE_AUTO, "megakernel": abi.RT_PIPELINE_MEGAKERNEL, "wavefront": abi.RT_PIPELINE_WAVEFRONT,
                "persistent": abi.RT_PIPELINE_PERSISTENT}[args.pipeline]

    accum = torch.zeros(H, W, 3, dtype=torch.int64, device=dev)  # fixed-point radiance sums (2^-32 units)
    rgb = torch.zeros(H, W, 3, dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stream = torch.cuda.current_stream()

    def step(i, stats=None, sc=None):
        """the product's sharded render (distributed.render_sharded): slice render -> exact int64 reduce -> tonemap on rank 0"""
        flush.fill_(i & 0xFF)  # L2 flush between steps
        return distributed.render_sharded(sc or scene, cam, W, H, job_spp, MAX_DEPTH, SEED, accum, rgb, first_sample=0, pipeline=pipeline,
                                          stream=stream, stats=stats)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    warm_stats = abi.RtStats()
    for w in range(args.warmup):
        step(1000 + w, stats=warm_stats if w == 0 else None)
    barrier()
    checksum0 = int(rgb.sum().item()) if rank == 0 else 0
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(args.steps):
        begin, count = step(k)
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.summary() if sampler else None
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = paths_per_step * args.steps / (ms_total / 1e3) / 1e6
    checksum = int(rgb.sum().item()) if rank == 0 else 0
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, rgb, accum)

    # ---- this rank's render region alone (CUDA events recorded by the library on the launching stream around the kernels of
    # the pipeline; no flush / reduce / tonemap): the numerator of the roofline figure
    st = abi.RtStats()
    torch.cuda.synchronize()
    step(2000, stats=st)
    barrier()
    render_ms, slice_paths = st.device_ms, int(st.paths)
    rays_per_path = st.rays / max(st.paths, 1)
    pipeline_used = {abi.RT_PIPELINE_MEGAKERNEL: "megakernel", abi.RT_PIPELINE_WAVEFRONT: "wavefront",
                     abi.RT_PIPELINE_PERSISTENT: "persistent"}.get(st.pipeline_used, str(st.pipeline_used))
    kernels = {"megakernel": "render_items_kernel", "wavefront": "wf_extend_kernel + wf_shade_kernel (one pair per round)",
               "persistent": "persist_kernel"}.get(pipeline_used, "?")
    launches_per_step = int(st.kernel_launches) + (1 if rank == 0 else 0)  # + tonemap (the L2 flush and the reduce are library kernels)

    # ---- end to end through the public host API with HOST buffers: scene upload + render + readback, every step
    e2e = None
    if args.e2e_steps > 0:
        scene_bytes = scene.info()["device_bytes"]
        host_rgb = torch.empty(H, W, 3, dtype=torch.int32).pin_memory()
        t0 = 0.0
        for k in range(-1, args.e2e_steps):  # k = -1: one untimed warm-up step (first-use allocations of the library)
            if k == 0:
                barrier()
                t0 = time.perf_counter()
            sc = rt.Scene(desc, device=local_rank)  # rt_scene_create: flatten + BVH build + H2D upload of the scene
            if dist is None:
                # one GPU: the reference-facing call itself, Renderer::render with HOST buffers (rt_render)
                p = abi.RtParams()
                p.width, p.height, p.samples_per_pixel, p.max_depth, p.seed, p.pipeline, p.device = W, H, job_spp, MAX_DEPTH, SEED, pipeline, -1
                abi.check(lib.rt_render(sc.handle, C.byref(cam.c), C.byref(p), None, host_rgb.data_ptr(), abi.RtProgressFn(), None, None))
            else:
                step(3000 + k, sc=sc)
                if rank == 0:
                    host_rgb.copy_(rgb, non_blocking=True)
                torch.cuda.synchronize()
            sc.close()
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": paths_per_step * args.e2e_steps / float(tt.item()) / 1e6, "unit": "Mpaths/s",
               "h2d_bytes_per_step": int(scene_bytes) * world_size, "d2h_bytes_per_step": int(host_rgb.numel() * 4),
               "api": ("rt_scene_create [flatten+BVH+upload] -> rt_render(host rgb buffer) -> rt_scene_destroy" if dist is None else
                       "rt_scene_create -> distributed.render_sharded [rt_render_accumulate_fixed_device -> ncclReduce(int64 sum) -> "
                       "rt_tonemap_fixed_device] -> pinned host rgb -> rt_scene_destroy"),
               "steps": args.e2e_steps, "checksum_matches": (int(host_rgb.sum().item()) == checksum) if rank == 0 else None}

    # ---- the same job through the ONE-process host of the same scheme (rt_render_multi: what `rt_main --gpus N` calls)
    multi = None
    if dist is not None and args.multi_steps > 0:
        barrier()
        if rank == 0:
            scenes = [scene] + [rt.Scene(desc, device=g) for g in range(world_size) if g != local_rank]
            arr = (C.c_void_p * len(scenes))(*[s.handle for s in scenes])
            p = abi.RtParams()
            p.width, p.height, p.samples_per_pixel, p.max_depth, p.seed, p.pipeline, p.device = W, H, job_spp, MAX_DEPTH, SEED, pipeline, -1
            host_rgb2 = np.empty((H, W, 3), np.int32)
            best, ms2 = None, abi.RtStats()
            for k in range(-1, args.multi_steps):
                t0 = time.perf_counter()
                abi.check(lib.rt_render_multi(arr, len(scenes), C.byref(cam.c), C.byref(p), None, host_rgb2.ctypes.data, abi.RtProgressFn(), None, C.byref(ms2)))
                dt = time.perf_counter() - t0
                if k >= 0:
                    best = dt if best is None else min(best, dt)
            multi = {"value": paths_per_step / best / 1e6, "unit": "Mpaths/s", "wall_ms_per_step": 1e3 * best, "device_ms_last_step": ms2.device_ms,
                     "api": "rt_render_multi(host rgb buffer): one process, one host thread per device, ncclReduce(uint64 sum), tonemap, D2H",
                     "checksum_matches": int(host_rgb2.sum()) == checksum}
            for s in scenes[1:]:
                s.close()
        dist.barrier(group=host_group)  # the other ranks wait here on the host: their GPUs belong to rank 0's threads meanwhile
        barrier()

    cpu, algo, algo_source = None, ALGO_FROZEN, "frozen (tests/golden/algo_work.py, BASELINE.md section 4)"
    if rank == 0 and world_size == 1 and args.cpu_spp > 0:
        v, ms, cores, per_path = cpu_reference_run(wl, args.cpu_spp, 1, 1)
        cpu = {"value": v, "unit": "Mpaths/s", "cores": cores, "kind": "port",
               "sample": f"full {W}x{H} frame at {args.cpu_spp} spp ({W * H * args.cpu_spp} paths, {ms / 1e3:.1f} s), C++ f64 restatement of the reference (no Rust toolchain)",
               "rays_per_path": per_path["rays"]}
        if wl["world"] == "final_scene":
            algo, algo_source = per_path, f"oracle instrumentation of this run's cpu_baseline leg ({args.cpu_spp} spp)"

    if rank == 0:
        drv, drv_how = driver_peaks()
        flops_pp, bytes_pp = algo_flops_per_path(algo), algo_bytes_per_path(algo)
        achieved = flops_pp * slice_paths / (render_ms / 1e3) / 1e12
        fp32_peak = max(peaks["fp32_ffma_tflops"], peaks["fp32_ffma2_tflops"])
        prof = profiled_traffic()
        traffic = prof["dram_bytes_per_path"] * slice_paths if prof else None
        l2 = None
        if prof and prof.get("l2_bytes_per_path"):
            l2_gbs = prof["l2_bytes_per_path"] * slice_paths / (render_ms / 1e3) / 1e9
            l2 = {"achieved_gbs": l2_gbs, "peak_gbs": peaks["l2_read_gbs"], "frac": l2_gbs / peaks["l2_read_gbs"],
                  "note": "achieved = lts sectors x 32 B per path of the committed ncu capture x paths per launch / live kernel time"}
        accum_bytes = 3 * 8 * slice_paths  # one 64-bit RED per channel per terminated path (upper bound)
        line = {
            "metric": baseline_metric(), "value": value, "unit": "Mpaths/s", "n_gpus": world_size, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": workload_name(wl), "job_spp": job_spp, "paths_per_step": paths_per_step,
                       "spp_per_gpu_per_step": count, "pipeline": pipeline_used, "bvh_layout": int(st.bvh_layout_used),
                       "parallelism": f"sample-slices x{world_size} (rt_sample_slice) + ncclReduce(sum) of the int64 fixed-point accumulation buffer",
                       "l2": "256 MB flush write between steps (inside the timed region)"},
            "clocks": clocks,
            "e2e": e2e,
            "render_multi": multi,
            "image_checksum": checksum, "image_checksum_stable": checksum == checksum0,
            "gpu_launches": launches_per_step * args.steps,
            "roofline": {"bound": "fp32", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s", "frac": achieved / fp32_peak,
                         "peak_theoretical": peaks["fp32_theoretical_tflops"], "frac_of_theoretical": achieved / peaks["fp32_theoretical_tflops"],
                         "peak_source": "measured in this run on this device by rt_measure_peaks: dependent-FFMA chains on every SM "
                                        f"(scalar {peaks['fp32_ffma_tflops']:.1f}, packed FFMA2 {peaks['fp32_ffma2_tflops']:.1f} TFLOP/s); "
                                        f"theoretical = {peaks['sm_count']} SMs x 128 lanes x 2 x {peaks['sm_clock_mhz']:.0f} MHz",
                         "traffic": traffic,
                         "traffic_note": (f"bytes per launch = dram bytes per path of {prof['file']} (ncu --set full, commit {prof.get('commit', '?')}) "
                                          "x paths per launch" if prof else "no committed ncu capture"),
                         "l2": l2,
                         "kernel": kernels, "kernel_ms": render_ms, "kernel_launches": int(st.kernel_launches),
                         "paths_per_kernel_ms": slice_paths,
                         "algorithmic_flops_per_path": flops_pp, "algorithmic_bytes_per_path": bytes_pp, "algorithmic_source": algo_source,
                         "hbm": {"achieved_gbs": accum_bytes / (render_ms / 1e3) / 1e9, "peak_gbs": drv.get("hbm_gbs"), "peak_source": drv_how,
                                 "note": "algorithmic HBM bytes = accumulation-buffer REDs only; the scene (~120 KB + 2 MB texture) is L1/L2 resident"}},
            "cpu_baseline": cpu,
            "rays_per_path": rays_per_path, "mrays_per_s": value * rays_per_path,
        }
        print(json.dumps(line), flush=True)
    scene.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--c5", action="store_true", help="the C5 job (final_scene 3840x3840, 4096 spp) instead of C4")
    ap.add_argument("--spp", type=int, default=0, help="samples per pixel of the job rendered per step (0 = the config's: 10 000 for C4)")
    ap.add_argument("--pipeline", default="auto", choices=["auto", "megakernel", "wavefront", "persistent"])
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--multi-steps", type=int, default=2, help="N > 1: timed steps of the one-process rt_render_multi leg (0 = skip)")
    ap.add_argument("--cpu-spp", type=int, default=128, help="spp of the bounded CPU-baseline sample (0 = skip)")
    ap.add_argument("--ref-spp", type=int, default=32, help="spp per step of --impl reference")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    wl = WORKLOADS["c5" if args.c5 else "c4"]
    if args.impl == "reference":
        return run_reference(args, wl)
    return run_b200(args, wl)


if __name__ == "__main__":
    sys.exit(main())
