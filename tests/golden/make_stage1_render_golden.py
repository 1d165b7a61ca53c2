"""Generate tests/golden/stage1_render_golden.npz from the REFERENCE's own TaichiRenderBatch.flow2render.

Run in the build container (needs the reference checkout):  python tests/golden/make_stage1_render_golden.py [REF_DIR]
taichi is not installable, so a minimal stub goes into sys.modules for this generator only (ti.init / ti.cuda /
ti.data_oriented / ti.kernel as no-ops or identity decorators, ti.Vector.field, ti.types.ndarray, ti.i32) before
lib/TaichiRender.py is imported; the instance's Taichi kernel `render_respective_color` is replaced by a recorder.
`flow2render` (lib/TaichiRender.py:26-60) then runs verbatim on CPU float32 tensors of a seeded synthetic stage-1 batch
(synth.stage1_batch: two ring cameras, capsule inverse depth turned into flow; the novel intr/extr come from the same
scipy Slerp calls as lib/utils.py:57-84, whose final `.cuda()` is left out).  Stored: the inputs, the reference's
per-view masks as handed to the kernel (taichi_mask_list), their points where the mask is set
(taichi_pts_list[mask]) and the image the sequential splat oracle makes of those points."""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from gps_gaussian_b200 import synth  # noqa: E402
from oracle.flow_splat_oracle import splat_seq  # noqa: E402

B, RES, BS = 2, 96, 1            # train_stage1.py:52 builds TaichiRenderBatch(bs=1, ...); its val batch is 2


def taichi_stub():
    ti = types.ModuleType("taichi")
    ti.cuda, ti.i32 = "cuda", "i32"
    ti.init = lambda *a, **k: None
    ti.data_oriented = ti.kernel = lambda f: f
    ti.Vector = types.SimpleNamespace(field=lambda **k: types.SimpleNamespace(**k))
    ti.types = types.SimpleNamespace(ndarray=lambda *a, **k: None)
    return ti


def main():
    ref = sys.argv[1] if len(sys.argv) > 1 else "/root/reference"
    sys.modules["taichi"] = taichi_stub()
    sys.path.insert(0, ref)
    from lib.TaichiRender import TaichiRenderBatch
    d = synth.stage1_batch(RES, B, seed=2024)
    data = {v: {k: torch.from_numpy(a) for k, a in d[v].items()} for v in ("lmain", "rmain", "novel_view")}
    rec = []
    r = TaichiRenderBatch(BS, RES)
    r.render_respective_color = lambda pts, mask, depth, color: rec.append((pts.clone(), mask.clone()))
    r.flow2render(data)
    pts = np.stack([p.numpy() for p, _ in rec])          # [2,B,S*S,6]
    mask = np.stack([m.numpy()[..., 0] for _, m in rec])  # [2,B,S*S]
    depth, color, winner = splat_seq(pts, mask, RES, BS)
    out = {f"{v}_{k}": a for v in ("lmain", "rmain") for k, a in d[v].items()}
    out.update(novel_intr=d["novel_view"]["intr"], novel_extr=d["novel_view"]["extr"],
               novel_calib=torch.matmul(data["novel_view"]["intr"], data["novel_view"]["extr"]).numpy(),
               ref_pts_valid=pts[mask > 0.5], ref_mask=mask.astype(np.uint8), ref_color=color, ref_depth=depth,
               ref_winner=winner,
               bs=np.int32(BS), res=np.int32(RES))
    np.savez_compressed(os.path.join(HERE, "stage1_render_golden.npz"), **out)
    print("wrote stage1_render_golden.npz", pts.shape, int(mask.sum()), int((winner >= 0).sum()))


if __name__ == "__main__":
    main()
