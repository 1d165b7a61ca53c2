"""Build libgpsg_sm100.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python gps-gaussian_b200/build.py [--force] [--verbose]

Output: gps-gaussian_b200/lib/libgpsg_sm100.so (git-ignored; travels to the GPU box with gpurun).
raster_preprocess.cu is compiled with -fmad=false (see its header): the fp32 op order that decides
radii / tile rectangles must not be FMA-contracted.  point_splat.cu likewise: the stage-1 preview's pixel and
inverse depth are replayed bit for bit by the CPU oracle.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libgpsg_sm100.so")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
          "--expt-relaxed-constexpr", "-Xptxas", "-v"]
SOURCES = {
    "gpsg_capi.cu": [],
    "raster_preprocess.cu": ["-fmad=false"],
    "raster_binning.cu": [],
    "raster_render.cu": [],
    "raster_backward.cu": [],
    "corr.cu": [],
    "corr_tc.cu": [],
    "sh.cu": [],
    "unproject.cu": [],
    "loss.cu": [],
    "point_splat.cu": ["-fmad=false"],
}


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _deps(src):
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(os.path.dirname(HERE), "include", "gpsg.h"))
    return [src, os.path.abspath(__file__)] + hdrs


def _stale(dst, deps):
    if not os.path.exists(dst):
        return True
    t = os.path.getmtime(dst)
    return any(os.path.getmtime(d) > t for d in deps)


def _compile(name, extra, force, verbose):
    src = os.path.join(CSRC, name)
    obj = os.path.join(OBJ, name.replace(".cu", ".o"))
    if not force and not _stale(obj, _deps(src)):
        return obj, ""
    cmd = [_nvcc()] + ARCH + COMMON + extra + ["-c", src, "-o", obj]
    p = subprocess.run(cmd, capture_output=True, text=True)
    log = " ".join(cmd) + "\n" + p.stdout + p.stderr
    if p.returncode != 0:
        raise RuntimeError(log)
    with open(obj + ".log", "w") as f:
        f.write(log)
    if verbose:
        print(log)
    return obj, log


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(LIBDIR, exist_ok=True)
    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        res = list(ex.map(lambda kv: _compile(kv[0], kv[1], force, verbose), SOURCES.items()))
    objs = [r[0] for r in res]
    if force or _stale(LIB, objs):
        cmd = [_nvcc()] + ARCH + ["-shared", "-o", LIB] + objs + ["-Xcompiler", "-fvisibility=hidden", "-cudart",
                                                                  "static"]
        p = subprocess.run(cmd, capture_output=True, text=True)
        if p.returncode != 0:
            raise RuntimeError(" ".join(cmd) + "\n" + p.stdout + p.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
