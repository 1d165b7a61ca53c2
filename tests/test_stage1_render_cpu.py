"""Stage-1 validation preview (reference lib/TaichiRender.py, TaichiRenderBatch.flow2render) on the CPU: the fused oracle
chain against the reference's own torch prep (golden), the packed-key z-buffer reading against the sequential splat, the
lib.TaichiRender substitution of the GPSG_PATCH hook, and the C ABI's exports / argument checks."""
import ctypes as C
import importlib.util
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle.flow_splat_oracle import flow2render, splat_seq

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = np.load(os.path.join(os.path.dirname(__file__), "golden", "stage1_render_golden.npz"))
KEYS = ("flow_pred", "mask", "intr", "extr", "ref_intr", "Tf_x", "img")

# Near-decision margins of the preview (cf. the rasterizer's margin accounting, DESIGN.md section 2).  The fused chain
# (csrc/point_splat.cu == oracle_flow2render_points, fixed fp32 op order) and the reference's torch prep (linspace pixel
# grid, bmm) round differently.  Measured on the golden batch (res 96, B 2): max |dx|, |dy| = 1.5e-5 px and
# max |d inv| = 1.2e-7.  A pixel may legitimately differ between the two when a point touching it has x or y within
# EPS_XY of an integer (the trunc / clamp boundary), or when its two largest candidate inverse depths are within EPS_INV.
EPS_XY = 1e-4        # >= 4 x 1.5e-5 px
EPS_INV = 1e-6       # >= 4 x 1.2e-7


def golden_views():
    return [{k: G[f"{v}_{k}"] for k in KEYS} for v in ("lmain", "rmain")]


def f2i_sat(a):
    """float -> int32 like CUDA's cvt.rzi.s32.f32 (truncate, saturate, NaN -> 0)."""
    a = np.asarray(a, np.float64)
    return np.where(np.isnan(a), 0, np.clip(np.trunc(np.nan_to_num(a)), -2.0 ** 31, 2.0 ** 31 - 1)).astype(np.int64)


def near_decision_pixels(pts, mask, res, bs):
    """pts[2,B,N,6] (x, y, inv, rgb), mask[2,B,N] of one chain -> bool[B,res,res]: pixels touched by a point near a
    decision (x / y within EPS_XY of an integer, or the top two candidate inverse depths within EPS_INV)."""
    B = pts.shape[1]
    near = np.zeros((B, res, res), bool)
    pix = lambda a: np.clip(f2i_sat(a), 0, res - 1)
    for b in range(bs):
        p = pts[:, b][mask[:, b] > 0.5].astype(np.float64)
        p = p[p[:, 2] >= 0]                                   # only these can draw
        x, y, inv = p[:, 0], p[:, 1], p[:, 2]
        close = (np.abs(x - np.round(x)) <= EPS_XY) | (np.abs(y - np.round(y)) <= EPS_XY)
        for xi, yi in zip(x[close], y[close]):
            near[b, pix(yi - EPS_XY):pix(yi + EPS_XY) + 1, pix(xi - EPS_XY):pix(xi + EPS_XY) + 1] = True
        key = pix(y) * res + pix(x)
        o = np.lexsort((inv, key))
        k, v = key[o], inv[o]
        same = k[1:] == k[:-1]
        last = np.r_[k[1:] != k[:-1], True]                   # last of its pixel group = the max
        tie = same & last[1:] & (v[1:] - v[:-1] <= EPS_INV)
        near[b].reshape(-1)[k[1:][tie]] = True
    return near


def test_fused_oracle_matches_reference_prep_golden():
    res, bs = int(G["res"]), int(G["bs"])
    o = flow2render(golden_views(), G["novel_calib"], bs, res)
    m = G["ref_mask"] > 0
    assert np.array_equal(o["valid"] > 0.5, m)
    d = np.abs(o["pts"][m].astype(np.float64) - G["ref_pts_valid"])
    print(f"fused chain vs reference prep: max |dx| {d[:, 0].max():.2e} |dy| {d[:, 1].max():.2e} |dinv| {d[:, 2].max():.2e}")
    assert d[:, 0].max() * 4 <= EPS_XY and d[:, 1].max() * 4 <= EPS_XY and d[:, 2].max() * 4 <= EPS_INV
    assert d[:, 3:].max() == 0                                # raw colours, copied
    ref_pts = np.zeros_like(o["pts"])
    ref_pts[m] = G["ref_pts_valid"]
    near = near_decision_pixels(o["pts"], o["valid"], res, bs) | near_decision_pixels(ref_pts, G["ref_mask"], res, bs)
    diff = (o["color"] != G["ref_color"]).any(1)
    print(f"golden image: {int((G['ref_winner'] >= 0).sum())} covered pixels, {int(near.sum())} near a decision, "
          f"{int(diff.sum())} differ ({int((diff & near).sum())} of them near)")
    assert not (diff & ~near).any()
    assert (G["ref_winner"][bs:] == -1).all() and (o["color"][bs:] == -1).all()     # samples >= bs stay background


def packed_key_splat(pts, mask, res, bs):
    """numpy restatement of csrc/point_splat.cu: key = bits(inv) << 32 | (v*N + i + 1), one max per pixel."""
    V, B, N = mask.shape
    zbuf = np.zeros((B, res * res), np.uint64)
    for b in range(bs):
        for v in range(V):
            p = pts[v, b].astype(np.float32)
            inv = p[:, 2]
            with np.errstate(invalid="ignore"):
                draw = (mask[v, b] >= 0.5) & (inv >= 0)
            i = np.nonzero(draw)[0]
            ix, iy = np.clip(f2i_sat(p[i, 0]), 0, res - 1), np.clip(f2i_sat(p[i, 1]), 0, res - 1)
            bits = (inv[i].view(np.uint32) & np.uint32(0x7FFFFFFF)).astype(np.uint64)
            key = (bits << np.uint64(32)) | (np.uint64(v * N) + i.astype(np.uint64) + np.uint64(1))
            np.maximum.at(zbuf[b], iy * res + ix, key)
    zbuf = zbuf.reshape(B, res, res)
    win = (zbuf & np.uint64(0xFFFFFFFF)).astype(np.int64) - 1
    inv = (zbuf >> np.uint64(32)).astype(np.uint32).view(np.float32)
    color = np.full((B, 3, res, res), -1.0, np.float32)
    flat = pts.transpose(1, 0, 2, 3).reshape(B, V * N, 6)
    for b in range(B):
        w = win[b] >= 0
        color[b][:, w] = flat[b][win[b][w], 3:].T
    return color, inv, win


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_packed_key_max_equals_sequential_splat(seed):
    rng = np.random.default_rng(seed)
    V, B, N, res, bs = 2, 3, 4000, 16, 2
    pts = np.zeros((V, B, N, 6), np.float32)
    pts[..., 0] = rng.uniform(-6, res + 6, (V, B, N))                  # off-screen points clamp onto the border
    pts[..., 1] = rng.uniform(-6, res + 6, (V, B, N))
    pts[..., 2] = rng.choice(np.float32([0.0, -0.0, 0.25, 0.5, 0.5, 0.75, 1.0, 1.0]), (V, B, N))   # ties everywhere
    special = rng.uniform(size=(V, B, N))
    pts[..., 2][special < 0.03] = -rng.uniform(0.1, 2, int((special < 0.03).sum()))           # behind the camera
    pts[..., 2][(special >= 0.03) & (special < 0.05)] = np.nan
    pts[..., 2][(special >= 0.05) & (special < 0.06)] = np.inf
    pts[..., 2][(special >= 0.06) & (special < 0.07)] = -np.inf
    pts[..., 0][(special >= 0.07) & (special < 0.08)] = np.nan                                 # NaN pixel -> 0
    pts[..., 1][(special >= 0.08) & (special < 0.09)] = 3e9                                    # saturates
    pts[..., 3:] = rng.uniform(-1, 1, (V, B, N, 3))
    mask = (rng.uniform(size=(V, B, N)) > 0.2).astype(np.float32)
    depth, color, win = splat_seq(pts, mask, res, bs)
    kc, kinv, kwin = packed_key_splat(pts, mask, res, bs)
    assert np.array_equal(win, kwin)
    assert np.array_equal(color.view(np.uint32), kc.view(np.uint32))
    assert np.array_equal(depth.view(np.uint32), kinv.view(np.uint32))
    assert (win[bs:] == -1).all() and (win[:bs] >= 0).mean() > 0.9
    # the scenario exercises ties across views: some winners come from view 1 over an equal view-0 inverse depth
    assert (win[:bs] >= N).any() and (win[:bs][win[:bs] >= 0] < N).any()


def _run(code):
    env = dict(os.environ)
    env.pop("GPSG_PATCH", None)
    env["PYTHONPATH"] = ""
    return subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=300)


@pytest.mark.skipif(importlib.util.find_spec("taichi") is not None, reason="taichi is installed")
def test_patch_substitutes_lib_taichirender():
    from gps_gaussian_b200 import harness
    ref = harness.staged_reference()
    if ref is None:
        pytest.skip("oracle/_ref not staged")
    code = f"""
import sys
sys.path[:0] = [{ref!r}, {ROOT!r}]
def attempt():
    try:
        from lib.TaichiRender import TaichiRenderBatch
        return TaichiRenderBatch.__module__
    except ModuleNotFoundError as e:
        return "missing:" + e.name
print("before", attempt())
from gps_gaussian_b200 import patch
patch.install()
print("installed", attempt())
import lib.TaichiRender
print("hasattr", hasattr(lib.TaichiRender, "TaichiRenderBatch"), len(lib.TaichiRender.TaichiRenderBatch(1, 8).__dict__))
patch.uninstall()
print("after", attempt())
"""
    p = _run(code)
    assert p.returncode == 0, p.stderr[-3000:]
    lines = dict(line.split(" ", 1) for line in p.stdout.strip().splitlines())
    assert lines["before"] == "missing:taichi"
    assert lines["installed"] == "gps_gaussian_b200.TaichiRender"
    assert lines["hasattr"].startswith("True")
    assert lines["after"] == "missing:taichi"


def test_flow2render_exports_and_rejects_bad_arguments():
    from gps_gaussian_b200 import _lib
    for name in ("gpsg_flow2render", "gpsg_flow2render_workspace_bytes"):
        assert name in _lib.EXPORTED and hasattr(_lib.lib, name)
    assert _lib.lib.gpsg_flow2render_workspace_bytes(2, 1024) == 2 * 1024 * 1024 * 8
    pp = (C.c_void_p * 2)(8, 8)
    strides = (C.c_int64 * 2)(1024 * 1024, 1024 * 1024)

    def call(B=2, bs=1, S=1024, res=1024, ws=2 * 1024 * 1024 * 8):
        return _lib.lib.gpsg_flow2render(0, None, B, bs, S, res, pp, pp, strides, pp, pp, 3, pp, pp, pp, C.c_void_p(8),
                                         C.c_void_p(8), ws, C.c_void_p(8), None)
    # all of these are refused before any CUDA call (no device needed)
    assert call(S=512) == -1                 # source maps must be res x res
    assert call(bs=3) == -1                  # bs <= B
    assert call(S=46341, res=46341) == -1    # 2*S^2 + 1 >= 2^32
    assert call(ws=16) == -1                 # workspace too small
    assert "workspace" in _lib.lib.gpsg_last_error().decode()


def test_splat_seq_of_one_view_equals_the_taichi_baseline_oracle():
    """oracle_splat_seq with one view and bs = B is oracle/taichi_splat_oracle.c's splat on finite, in-range points."""
    from oracle.raster_oracle import taichi_splat
    rng = np.random.default_rng(3)
    B, N, res = 2, 3000, 12
    pts = np.zeros((B, N, 6), np.float32)
    pts[..., :2] = rng.uniform(-3, res + 3, (B, N, 2))
    pts[..., 2] = rng.choice(np.float32([0.1, 0.2, 0.3, 0.3]), (B, N))
    pts[..., 3:] = rng.uniform(-1, 1, (B, N, 3))
    mask = (rng.uniform(size=(B, N)) > 0.3).astype(np.float32)
    d0, c0 = taichi_splat(pts, mask, res)
    d1, c1, _ = splat_seq(pts[None], mask[None], res)
    assert np.array_equal(d0[:, 0], d1) and np.array_equal(c0, c1)
