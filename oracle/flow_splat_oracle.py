"""ctypes front-end of oracle/flow_splat_oracle.c: the stage-1 validation preview (reference lib/TaichiRender.py:26-60,
TaichiRenderBatch.flow2render) restated on the CPU in the op order of csrc/point_splat.cu.

TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/ and tools/ may import this module.

    python oracle/flow_splat_oracle.py        # builds oracle/_build/libflow_splat_{f32,f64}.so (also done by build())
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(_HERE, "_build")
SRC = os.path.join(_HERE, "flow_splat_oracle.c")
_LIBS = {}


def build(force=False):
    """gcc, -ffp-contract=off like the other oracle libraries: fp32 results follow the written op order."""
    os.makedirs(OUT, exist_ok=True)
    deps = [SRC, os.path.join(_HERE, "oracle_real.h"), os.path.abspath(__file__)]
    outs = {}
    for tag, defs in (("f32", []), ("f64", ["-DORACLE_F64"])):
        dst = os.path.join(OUT, f"libflow_splat_{tag}.so")
        outs[tag] = dst
        if not force and os.path.exists(dst) and all(os.path.getmtime(d) <= os.path.getmtime(dst) for d in deps):
            continue
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-Wall"]
                              + defs + [SRC, "-lm", "-o", dst])
    return outs


def _lib(tag):
    if tag not in _LIBS:
        path = os.path.join(OUT, f"libflow_splat_{tag}.so")
        if not os.path.exists(path):
            build()
        _LIBS[tag] = C.CDLL(path)
    return _LIBS[tag]


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _real(dtype):
    assert dtype in ("f32", "f64")
    return np.float32 if dtype == "f32" else np.float64


def splat_seq(pts, mask, res, bs=None, dtype="f32"):
    """The sequential splat of all views in order onto one state (lib/TaichiRender.py:53-57): pts[V,B,N,6],
    mask[V,B,N]; only samples b < bs.  Returns (depth[B,res,res], color[B,3,res,res], winner[B,res,res] = v*N + i,
    -1 where no point landed)."""
    r = _real(dtype)
    pts = np.ascontiguousarray(pts, r)
    V, B, N = pts.shape[0], pts.shape[1], pts.shape[2]
    mask = np.ascontiguousarray(np.asarray(mask, r).reshape(V, B, N))
    bs = B if bs is None else int(bs)
    depth = np.zeros((B, res, res), r)
    color = np.full((B, 3, res, res), -1.0, r)
    winner = np.full((B, res, res), -1, np.int32)
    getattr(_lib(dtype), f"oracle_splat_seq_{dtype}")(C.c_int(B), C.c_int(bs), C.c_int(V), C.c_int(N), C.c_int(res),
                                                       _p(pts), _p(mask), _p(depth), _p(color), _p(winner))
    return depth, color, winner


def flow2render_points(views, calib, dtype="f32"):
    """Per-point chain of TaichiRenderBatch.flow2render (lib/TaichiRender.py:26-52) in the sm_100a kernel's op order.
    `views`: two dicts (lmain, rmain) of numpy arrays flow_pred[B,1,S,S], mask[B,C,S,S], intr[B,3,3], extr[B,>=3,4],
    ref_intr[B,3,3], Tf_x[B], img[B,3,S,S]; calib[B,3,4].  Returns (pts[2,B,S*S,6], valid[2,B,S*S])."""
    r = _real(dtype)
    f0 = np.asarray(views[0]["flow_pred"])
    B, S = f0.shape[0], f0.shape[-1]
    st = lambda key, fn: np.ascontiguousarray(np.stack([fn(np.asarray(v[key])) for v in views]), r)
    flow = st("flow_pred", lambda a: a.reshape(B, S * S))
    mask = st("mask", lambda a: a[:, 0].reshape(B, S * S))
    intr, ref_intr = st("intr", lambda a: a.reshape(B, 9)), st("ref_intr", lambda a: a.reshape(B, 9))
    extr = st("extr", lambda a: a[:, :3, :].reshape(B, 12))
    tfx = st("Tf_x", lambda a: a.reshape(B))
    img = st("img", lambda a: a.reshape(B, 3, S * S))
    cal = np.ascontiguousarray(np.asarray(calib, r).reshape(B, 12))
    pts = np.zeros((2, B, S * S, 6), r)
    valid = np.zeros((2, B, S * S), r)
    getattr(_lib(dtype), f"oracle_flow2render_points_{dtype}")(C.c_int(B), C.c_int(S), _p(flow), _p(mask), _p(intr),
                                                                _p(extr), _p(ref_intr), _p(tfx), _p(img), _p(cal),
                                                                _p(pts), _p(valid))
    return pts, valid


def flow2render(views, calib, bs, res, dtype="f32"):
    """The whole preview: flow2render_points then splat_seq.  Returns dict(pts, valid, depth[B,res,res],
    color[B,3,res,res], winner[B,res,res])."""
    pts, valid = flow2render_points(views, calib, dtype)
    depth, color, winner = splat_seq(pts, valid, res, bs, dtype)
    return dict(pts=pts, valid=valid, depth=depth, color=color, winner=winner)


if __name__ == "__main__":
    print(build(force=True))
