"""Mirror of reference lib/TaichiRender.py -- `TaichiRenderBatch(bs, res).flow2render(data)`, the stage-1 validation
preview (train_stage1.py:52, 98-105), without Taichi.

Upstream projects both source views' point clouds into the novel camera with torch (two boolean-mask `index_put`s per
view, each a host sync, plus [B,S^2,6] temporaries and a `cat`) and splats them with a Taichi kernel whose colour write
races with its `atomic_max`.  Here one sm_100a kernel does flow -> depth -> point -> novel pixel + inverse depth and a
64-bit packed-key atomicMax z-buffer, and a second one resolves the colours (`gpsg_flow2render`, csrc/point_splat.cu):
no host synchronisation, and a deterministic image -- the sequential reading of upstream's kernel (views l then r,
pixels in order; the last point among those with the largest inverse depth wins).

Kept from upstream on purpose: off-screen points are clamped onto the border pixels, colours are the raw img values in
[-1, 1] on a -1 background, and only the first `bs` samples are rendered (the others stay -1).
This module does not import taichi.
"""
import ctypes as C

import torch

from . import _lib

_VIEWS = ('lmain', 'rmain')


def _f32(t, dev):
    return t.detach().to(device=dev, dtype=torch.float32).contiguous()


def _ptrs(ts):
    return (C.c_void_p * 2)(*[t.data_ptr() for t in ts])


def flow2render_maps(data, bs, res, novel_calib=None, with_inv_depth=False, out=None):
    """The preview of `data` (source views data['lmain'] / data['rmain'] with flow_pred, mask, intr, extr, ref_intr, Tf_x,
    img; novel camera data['novel_view']['intr'] / ['extr'], or `novel_calib` [B,3,4] = K E).  Returns (color[B,3,res,res],
    inv_depth[B,res,res] or None, zbuf[B,res,res] int64 -- the packed winner keys: inverse-depth bits << 32 |
    view*S^2 + pixel + 1, 0 = no point).  `out`: optional (color, inv_depth or None, zbuf) contiguous tensors to fill."""
    v0 = data[_VIEWS[0]]
    dev = v0['flow_pred'].device
    if dev.type != 'cuda':
        raise RuntimeError("flow2render (gpsg_sm100): the source maps must be CUDA tensors")
    if novel_calib is None:
        novel_calib = torch.matmul(data['novel_view']['intr'], data['novel_view']['extr'])   # as upstream (:27)
    calib = _f32(novel_calib, dev)
    B = int(calib.shape[0])
    if tuple(calib.shape) != (B, 3, 4):
        raise ValueError(f"flow2render: novel calib must be [B,3,4], got {tuple(calib.shape)}")
    S = int(v0['flow_pred'].shape[-1])
    if S != res:
        raise ValueError(f"flow2render: source maps are {S}x{S} but res = {res}")
    if not 0 <= bs <= B:
        raise ValueError(f"flow2render: bs = {bs} exceeds the batch ({B})")
    if 2 * S * S + 1 >= 2 ** 32:
        raise ValueError(f"flow2render: {S}x{S} maps exceed the 32-bit point id of the z-buffer key")
    flow, mask, intr, extr, ref_intr, tfx, img = [], [], [], [], [], [], []
    for name in _VIEWS:
        d = data[name]
        f = _f32(d['flow_pred'], dev)
        m = _f32(d['mask'], dev)
        if tuple(f.shape) != (B, 1, S, S) or m.dim() != 4 or tuple(m.shape[-2:]) != (S, S) or m.shape[0] != B:
            raise ValueError(f"flow2render: {name} flow_pred / mask must be [B,1,S,S] / [B,C,S,S]")
        e = d['extr']
        if e.dim() != 3 or e.shape[0] != B or e.shape[-1] != 4 or e.shape[-2] < 3:
            raise ValueError(f"flow2render: {name} extr must be [B,3|4,4]")
        e = _f32(e[:, :3, :], dev)
        i = _f32(d['img'], dev)
        if tuple(i.shape) != (B, 3, S, S):
            raise ValueError(f"flow2render: {name} img must be [B,3,S,S]")
        flow.append(f); mask.append(m); extr.append(e); img.append(i)
        intr.append(_f32(d['intr'], dev).reshape(B, 9)); ref_intr.append(_f32(d['ref_intr'], dev).reshape(B, 9))
        tfx.append(_f32(d['Tf_x'], dev).reshape(B))
    if out is not None:
        color, inv, zbuf = out
        for t, shape, dt in ((color, (B, 3, res, res), torch.float32), (inv, (B, res, res), torch.float32),
                             (zbuf, (B, res, res), torch.int64)):
            if t is not None and (tuple(t.shape) != shape or t.dtype != dt or not t.is_contiguous() or t.device != dev):
                raise ValueError(f"flow2render: out tensor must be a contiguous {dt} {shape} on {dev}")
    else:
        color = torch.empty((B, 3, res, res), dtype=torch.float32, device=dev)
        inv = torch.empty((B, res, res), dtype=torch.float32, device=dev) if with_inv_depth else None
        zbuf = torch.empty((B, res, res), dtype=torch.int64, device=dev)
    strides = (C.c_int64 * 2)(*[int(m.stride(0)) for m in mask])
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    with torch.cuda.device(dev):
        rc = _lib.lib.gpsg_flow2render(idx, C.c_void_p(torch.cuda.current_stream(dev).cuda_stream), B, int(bs), S, int(res),
                                       _ptrs(flow), _ptrs(mask), strides, _ptrs(intr), _ptrs(extr), 3,
                                       _ptrs(ref_intr), _ptrs(tfx), _ptrs(img), C.c_void_p(calib.data_ptr()),
                                       C.c_void_p(zbuf.data_ptr()), zbuf.numel() * 8, C.c_void_p(color.data_ptr()),
                                       C.c_void_p(inv.data_ptr()) if inv is not None else None)
    _lib.check(rc, "gpsg_flow2render")
    return color, inv, zbuf


class TaichiRenderBatch:
    """Same constructor and `flow2render(data)` as reference lib/TaichiRender.py:8-60."""

    def __init__(self, bs, res):
        self.bs = int(bs)
        self.res = int(res)

    def flow2render(self, data):
        """Writes data['novel_view']['img_pred'] ([B,3,res,res] fp32 on the maps' device) and returns data."""
        color, _, _ = flow2render_maps(data, self.bs, self.res)
        data['novel_view']['img_pred'] = color
        return data
