"""Build the CPU oracle shared libraries (test infrastructure, not product).

    python oracle/build.py [--reference DIR]   # builds oracle/_build/liboracle_{f32,f64}.so

The reference's rasterizer source (graphdeco-inria/diff-gaussian-rasterization) and
sampler source (princeton-vl/RAFT-Stereo/sampler) are not part of the GPS-Gaussian tree,
so nothing of the reference compiles from its own sources (it is pure Python; see
DESIGN.md "Oracle").  The GPS-Gaussian checkout (`--reference DIR`, else the
GPSG_REFERENCE_DIR environment variable, else REF_DEFAULT when it holds one) is staged
unmodified into the git-ignored `oracle/_ref/`, where the C3/C5 harness
(gps_gaussian_b200/harness.py) runs the reference's own model and scripts against the
drop-ins.  Without a checkout nothing is staged and those tests skip.
"""
import os
import shutil
import stat
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_build")
REF_STAGED = os.path.join(HERE, "_ref")
REF_DEFAULT = "/root/reference"          # where the build environment mounts the GPS-Gaussian checkout (read-only)
SRCS = ["gpsg_oracle.c", "corr_oracle.c", "taichi_splat_oracle.c"]


def _newer(dst, srcs):
    if not os.path.exists(dst):
        return True
    t = os.path.getmtime(dst)
    return any(os.path.getmtime(s) > t for s in srcs)


def build(force=False, verbose=False):
    os.makedirs(OUT, exist_ok=True)
    srcs = [os.path.join(HERE, s) for s in SRCS if os.path.exists(os.path.join(HERE, s))]
    outs = {}
    for tag, defs in (("f32", []), ("f64", ["-DORACLE_F64"])):
        dst = os.path.join(OUT, f"liboracle_{tag}.so")
        outs[tag] = dst
        if not force and not _newer(dst, srcs + [os.path.abspath(__file__)]):
            continue
        # -ffp-contract=off: no FMA contraction, so fp32 results follow the written op order
        cmd = ["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-fopenmp", "-ffp-contract=off", "-fno-fast-math",
               "-Wall", "-Wno-unused-function"] + defs + srcs + ["-lm", "-o", dst]
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)
    stage_reference(reference_dir())
    return outs


def reference_dir():
    """GPSG_REFERENCE_DIR if set, else REF_DEFAULT if it holds a GPS-Gaussian tree, else None."""
    env = os.environ.get("GPSG_REFERENCE_DIR")
    if env:
        return env
    return REF_DEFAULT if os.path.isfile(os.path.join(REF_DEFAULT, "train_stage2.py")) else None


def stage_reference(src, force=False):
    """Copy the reference tree `src` to oracle/_ref (once, or again with `force`). Returns the staged path, or None when
    `src` is not given and nothing was staged before."""
    marker = os.path.join(REF_STAGED, "train_stage2.py")
    if src and (force or not os.path.exists(marker)):
        if not os.path.exists(os.path.join(src, "train_stage2.py")):
            raise FileNotFoundError(f"{src} is not a GPS-Gaussian tree (no train_stage2.py)")
        if os.path.isdir(REF_STAGED):
            shutil.rmtree(REF_STAGED)
        shutil.copytree(src, REF_STAGED, ignore=shutil.ignore_patterns(".git", "__pycache__", "*.pyc"))
        make_writable(REF_STAGED)
    return REF_STAGED if os.path.exists(marker) else None


def make_writable(path):
    """Add owner write permission throughout a copied tree (a read-only checkout keeps its modes through copytree, and
    the copy must stay removable and, for the harness's working copies, writable)."""
    for d, _, files in os.walk(path):
        for p in [d] + [os.path.join(d, f) for f in files]:
            if not os.path.islink(p):
                os.chmod(p, os.stat(p).st_mode | stat.S_IWUSR)


if __name__ == "__main__":
    ref = sys.argv[sys.argv.index("--reference") + 1] if "--reference" in sys.argv else None
    print(build(force="--force" in sys.argv, verbose=True), stage_reference(ref, force=ref is not None))
