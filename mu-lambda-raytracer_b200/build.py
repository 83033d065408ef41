"""In-tree build of librt_b200.so (CUDA kernels + C ABI) for sm_100a with nvcc; no JIT cache, no torch headers.

`python -m mu_lambda_raytracer_b200.build` or `__graft_entry__.build()`.  nvcc cross-compiles without a GPU.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "librt_b200.so")
CLI = os.path.join(HERE, "rt_main")

# Device math flags.  The product is built WITHOUT --use_fast_math: FTZ and the approximate division / square root are
# kept (IEEE versions cost 30 %: the node and primitive tests divide), the libm names (sinf in the checker and marble
# textures, acosf, atan2f) stay accurate, and the two hot approximations — MUFU sine/cosine in the in-ball/in-disk
# samplers, MUFU log/pow in the free-flight and radius draws — are explicit intrinsics in rt_device.cuh.  Measured on C4
# (profiles/r2_fastmath_ab.txt).  RT_BUILD_FLAVOR=fast|precise|floatred builds librt_b200_<flavor>.so beside the product
# for that A/B (abi.py: RT_B200_LIB selects it).
MATH = ["-ftz=true", "-prec-div=false", "-prec-sqrt=false"]
FLAVORS = {"": MATH, "fast": ["--use_fast_math"], "precise": [],
           "exp": MATH + ["-DRTB_PS_EXPERIMENTS"],  # + the rejected kernel placements of rt_persist.cu (tools/experiments/)
           "floatred": MATH + ["-DRTB_AB_FLOAT_RED"],
           "nonoise": MATH + ["-DRTB_AB_NO_NOISE"]}
FLAVOR = os.environ.get("RT_BUILD_FLAVOR", "")
if FLAVOR:
    OUT = os.path.join(HERE, "librt_b200_%s.so" % FLAVOR)
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17"] + FLAVORS[FLAVOR] + [
    "-Xcompiler", "-fPIC,-O3,-Wall,-Wno-unused-function"]
# host translation units restate f64 arithmetic of the reference: no FMA contraction there
CXX_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-Wall"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _run(cmd):
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("build failed: %s\n%s" % (" ".join(cmd), r.stdout))
    return r.stdout


def build(force=False, verbose=False):
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "rt_b200.h"))
    objs = []
    bdir = os.path.join(HERE, "build" + ("_" + FLAVOR if FLAVOR else ""))
    os.makedirs(bdir, exist_ok=True)
    for src in ("worlds.cpp", "scene_hash.cpp", "flatten.cpp"):  # pure host code: g++
        s = os.path.join(CSRC, src)
        o = os.path.join(bdir, src + ".o")
        if force or _newer(o, [s] + headers):
            out = _run(["g++"] + CXX_FLAGS + ["-c", s, "-o", o])
            if verbose and out:
                print(out)
        objs.append(o)
    for src in ("rt_api.cu", "rt_wavefront.cu", "rt_persist.cu", "rt_multi.cu", "rt_peaks.cu", "rt_lbvh.cu", "dev_cache.cu", "rt_adaptive.cu", "rt_denoise.cu", "rt_features.cu"):
        cu = os.path.join(CSRC, src)
        cuo = os.path.join(bdir, src + ".o")
        if force or _newer(cuo, [cu] + headers):
            out = _run([_nvcc()] + NVCC_FLAGS + ["-Xptxas", "-v", "-c", cu, "-o", cuo])
            with open(os.path.join(bdir, src + ".ptxas.log"), "w") as f:
                f.write(out)
            if verbose:
                print(out)
        objs.append(cuo)
    if force or _newer(OUT, objs):
        _run([_nvcc(), "-shared", "-o", OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static", "-ldl", "-lpthread"])
    main_src = os.path.join(CSRC, "main.cpp")
    if not FLAVOR and os.path.exists(main_src) and (force or _newer(CLI, [main_src, OUT] + headers)):
        _run(["g++"] + CXX_FLAGS + [main_src, "-o", CLI, "-L" + HERE, "-lrt_b200", "-Wl,-rpath,$ORIGIN"])
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
