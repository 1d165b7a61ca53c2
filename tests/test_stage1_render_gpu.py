"""Stage-1 validation preview on the B200 (csrc/point_splat.cu via gps_gaussian_b200.TaichiRender) and the stage-1 ->
stage-2 chain of the unmodified reference scripts under GPSG_PATCH=1."""
import glob
import math
import os
import sys
import types

import numpy as np
import pytest
import torch

from gps_gaussian_b200 import harness, synth
from gps_gaussian_b200.TaichiRender import TaichiRenderBatch, flow2render_maps
from oracle.flow_splat_oracle import flow2render as oracle_flow2render, splat_seq
from test_stage1_render_cpu import near_decision_pixels

pytestmark = pytest.mark.gpu
VIEWS = ("lmain", "rmain")
needs_ref = pytest.mark.skipif(harness.staged_reference() is None, reason="oracle/_ref not staged")


def to_device(d):
    return {v: {k: torch.from_numpy(a).cuda() for k, a in d[v].items()} for v in VIEWS + ("novel_view",)}


def run_device(data, bs, res, calib=None):
    """flow2render into NaN-poisoned outputs; returns numpy (color, inv_depth, winner = key low word - 1) and the calib."""
    if calib is None:
        calib = torch.matmul(data["novel_view"]["intr"], data["novel_view"]["extr"])
    B = int(calib.shape[0])
    out = (torch.full((B, 3, res, res), float("nan"), device="cuda"), torch.full((B, res, res), float("nan"), device="cuda"),
           torch.full((B, res, res), -7, dtype=torch.int64, device="cuda"))
    color, inv, zbuf = flow2render_maps(data, bs, res, novel_calib=calib, with_inv_depth=True, out=out)
    torch.cuda.synchronize()
    win = (zbuf.cpu().numpy() & 0xFFFFFFFF) - 1
    return color.cpu().numpy(), inv.cpu().numpy(), win, calib.cpu().numpy()


def check_bitexact(data, bs, res, calib=None):
    color, inv, win, cal = run_device(data, bs, res, calib)
    views = [{k: t.cpu().numpy() for k, t in data[v].items()} for v in VIEWS]
    o = oracle_flow2render(views, cal, bs, res)
    assert np.array_equal(win, o["winner"]), int((win != o["winner"]).sum())
    assert np.array_equal(color.view(np.uint32), o["color"].view(np.uint32)), int((color != o["color"]).sum())
    assert np.array_equal(inv.view(np.uint32), o["depth"].view(np.uint32))
    return color, win, o


@pytest.mark.parametrize("res,B,bs", [(256, 1, 1), (256, 2, 1), (256, 2, 2), (1024, 1, 1), (1024, 2, 1), (1024, 2, 2)])
def test_device_bitexact_vs_fused_oracle(res, B, bs):
    data = to_device(synth.stage1_batch(res, B, seed=res + B))
    color, win, o = check_bitexact(data, bs, res)
    covered = (win[:bs] >= 0).mean()
    print(f"res {res} B {B} bs {bs}: {covered:.1%} of the rendered samples' pixels covered")
    assert covered > 0.05 and (win[bs:] == -1).all() and (color[bs:] == -1).all()


def _edge(kind, res=256):
    d = synth.stage1_batch(res, 2, seed=7)
    data = to_device(d)
    calib = torch.matmul(data["novel_view"]["intr"], data["novel_view"]["extr"])
    if kind == "offscreen":                         # x += 2 res, y -= 2 res: every point clamps onto pixel (0, res-1)
        calib[:, 0, :] += 2.0 * res * calib[:, 2, :]
        calib[:, 1, :] -= 2.0 * res * calib[:, 2, :]
    elif kind == "behind":                          # every point behind the novel camera: inv < 0 never draws
        calib = -calib
    elif kind == "ties":                            # z == 4 for every point: exact inv ties within and across views
        calib[:, 2, :3] = 0.0
        calib[:, 2, 3] = 4.0
        calib[:, :2, :] *= 0.25
    elif kind == "nonfinite":
        for v, val in zip(VIEWS, (float("nan"), float("inf"))):
            f = data[v]["flow_pred"].view(-1)
            f[::7] = val
            f[3::11] = -float("inf")
    elif kind == "nomask":
        for v in VIEWS:
            data[v]["mask"].zero_()
    return data, calib.contiguous()


@pytest.mark.parametrize("kind", ["offscreen", "behind", "ties", "nonfinite", "nomask"])
def test_device_bitexact_edge_scenes(kind):
    res = 256
    data, calib = _edge(kind, res)
    color, win, o = check_bitexact(data, 2, res, calib)
    hit = win >= 0
    if kind == "offscreen":
        assert hit[:, 0, res - 1].all() and int(hit.sum()) == 2     # the border pile-up
    elif kind in ("behind", "nomask"):
        assert not hit.any() and (color == -1).all()
    elif kind == "ties":
        assert (win[hit] >= res * res).any()                      # on ties the later view wins
    print(f"{kind}: {int(hit.sum())} pixels hit")


def _taichi_stub():
    ti = types.ModuleType("taichi")
    ti.cuda, ti.i32 = "cuda", "i32"
    ti.init = lambda *a, **k: None
    ti.data_oriented = ti.kernel = lambda f: f
    ti.Vector = types.SimpleNamespace(field=lambda **k: types.SimpleNamespace(**k))
    ti.types = types.SimpleNamespace(ndarray=lambda *a, **k: None)
    return ti


@needs_ref
@pytest.mark.parametrize("res", [256, 1024])
def test_device_vs_reference_prep_on_gpu(res):
    """The reference's own flow2render prep (lib/TaichiRender.py:26-52) on CUDA tensors under a test-local taichi stub,
    then the sequential splat of its points, against the device image (near-decision accounting of the CPU test)."""
    harness.add_reference_to_path()
    saved = {k: sys.modules.pop(k) for k in ("taichi", "lib.TaichiRender") if k in sys.modules}
    sys.modules["taichi"] = _taichi_stub()
    try:
        import lib.TaichiRender as ref_mod
        assert ref_mod.__file__.startswith(harness.REF_STAGED)
        bs = 1
        data = to_device(synth.stage1_batch(res, 2, seed=99))
        rec = []
        r = ref_mod.TaichiRenderBatch(bs, res)
        r.render_respective_color = lambda pts, mask, depth, color: rec.append((pts.cpu().numpy(), mask.cpu().numpy()[..., 0]))
        r.flow2render({v: dict(data[v]) for v in data})
    finally:
        for k in ("taichi", "lib.TaichiRender"):
            sys.modules.pop(k, None)
        sys.modules.update(saved)
    pts, mask = np.stack([p for p, _ in rec]), np.stack([m for _, m in rec])
    _, ref_color, _ = splat_seq(pts, mask, res, bs)
    color, _, win, _ = run_device(data, bs, res)
    ours = oracle_flow2render([{k: t.cpu().numpy() for k, t in data[v].items()} for v in VIEWS],
                              torch.matmul(data["novel_view"]["intr"], data["novel_view"]["extr"]).cpu().numpy(), bs, res)
    assert np.array_equal(ours["valid"] > 0.5, mask > 0.5)
    near = near_decision_pixels(pts, mask, res, bs) | near_decision_pixels(ours["pts"], ours["valid"], res, bs)
    diff = (color != ref_color).any(1)
    print(f"res {res}: {int((win >= 0).sum())} covered, {int(near.sum())} near a decision, {int(diff.sum())} differ "
          f"({int((diff & near).sum())} of them near)")
    assert not (diff & ~near).any()


def test_two_calls_bit_identical_and_sync_free():
    res = 1024
    data = to_device(synth.stage1_batch(res, 2, seed=5))
    r = TaichiRenderBatch(2, res)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        a = r.flow2render(data)["novel_view"]["img_pred"].clone()
        b = r.flow2render(data)["novel_view"]["img_pred"].clone()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert a.shape == (2, 3, res, res) and a.dtype == torch.float32 and a.is_cuda
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    assert float((a > -1).float().mean()) > 0.05


# ---- the unmodified reference scripts ---------------------------------------------------------------------------------
RES1 = 256


@pytest.fixture(scope="module")
def dataset(tmp_path_factory):
    from gps_gaussian_b200 import synth_dataset
    root = str(tmp_path_factory.mktemp("s1data"))
    synth_dataset.write_dataset(root, n_train=2, n_val=2, res=RES1, hr=True)       # train_stage1.py:37 needs >= 2 val
    return root


@pytest.fixture(scope="module")
def stage1_run(dataset, tmp_path_factory):
    work = harness.make_workdir(str(tmp_path_factory.mktemp("s1") / "work"), dataset, src_res=RES1, num_steps=3,
                                batch_size=2, stage1=dict(src_res=RES1, num_steps=3, batch_size=2, eval_freq=1))
    p = harness.run_script(work, "train_stage1.py", patch=True, timeout=1500)
    return work, p


@needs_ref
def test_train_stage1_runs_unmodified_with_patch(stage1_run):
    work, p = stage1_run
    for name in ("train_stage1.py", "lib/TaichiRender.py", "core/corr.py", "lib/network.py"):
        with open(os.path.join(work, name), "rb") as a, open(os.path.join(harness.REF_STAGED, name), "rb") as b:
            assert a.read() == b.read()
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-6000:]
    assert "FINISHED TRAINING" in p.stdout
    ckpts = glob.glob(os.path.join(work, "experiments", "*", "ckpt", "*_final.pth"))
    assert len(ckpts) == 1
    sd = torch.load(ckpts[0], map_location="cpu")
    assert sd["total_steps"] == 3 and all(bool(torch.isfinite(v).all()) for v in sd["network"].values() if v.is_floating_point())
    import cv2
    shows = sorted(glob.glob(os.path.join(work, "experiments", "*", "show", "*.jpg")))
    assert [os.path.basename(f) for f in shows] == ["1.jpg", "2.jpg"]              # eval at steps 1 and 2
    for f in shows:
        im = cv2.imread(f)
        assert im.shape == (RES1, RES1, 3) and int(im.max()) > 0, (im.shape, im.max())


@needs_ref
def test_stage2_starts_from_the_stage1_checkpoint(stage1_run, dataset):
    work, p = stage1_run
    assert p.returncode == 0
    ckpt = glob.glob(os.path.join(work, "experiments", "*", "ckpt", "*_final.pth"))[0]
    with open(os.path.join(work, "config", "stage2.yaml"), "w") as f:
        f.write(harness.stage2_yaml(dataset, src_res=RES1, num_steps=3, batch_size=2, stage1_ckpt=ckpt))
    q = harness.run_script(work, "train_stage2.py", patch=True, timeout=1500)
    assert q.returncode == 0, q.stdout[-3000:] + q.stderr[-6000:]
    assert "Using checkpoint from stage1" in q.stderr and "FINISHED TRAINING" in q.stdout
    f2 = glob.glob(os.path.join(work, "experiments", "GPS-GS_stage2*", "ckpt", "*_final.pth"))
    assert len(f2) == 1
    sd = torch.load(f2[0], map_location="cpu")
    assert sd["total_steps"] == 3 and all(bool(torch.isfinite(v).all()) for v in sd["network"].values() if v.is_floating_point())
    # what train_stage2.py:50-52 loads: its own Trainer.load_ckpt (strict=False) on the stage-2 model
    cfg = harness.load_cfg(dataset, src_res=RES1, stage1_ckpt=ckpt)
    import train_stage2
    from lib.network import RtStereoHumanModel
    holder = types.SimpleNamespace(model=RtStereoHumanModel(cfg, with_gs_render=True).cuda())
    train_stage2.Trainer.load_ckpt(holder, cfg.stage1_ckpt, load_optimizer=False, strict=False)
    s1 = torch.load(ckpt, map_location="cpu")["network"]
    loaded = holder.model.state_dict()
    assert set(s1) <= set(loaded) and len(loaded) > len(s1)                    # + the Gaussian-parameter heads
    assert all(torch.equal(s1[k], loaded[k].cpu()) for k in s1)


@needs_ref
def test_stage1_fp32_flow_reg_cuda_equals_reg(dataset):
    """Stage-1 model (mixed_precision False): 'reg_cuda' through the patched fp32 FFMA volume build + fused lookup vs
    the reference's pure-PyTorch 'reg', after val_iters GRU iterations."""
    import tempfile
    import yaml
    from gps_gaussian_b200 import patch
    harness.add_reference_to_path()
    from torch.utils.data import default_collate
    flows = {}
    for corr in ("reg", "reg_cuda"):
        if corr == "reg_cuda":
            patch.install()
        try:
            from config.stereo_human_config import ConfigStereoHuman
            from lib.human_loader import StereoHumanDataset
            from lib.network import RtStereoHumanModel
            y = yaml.safe_load(harness.stage1_yaml(dataset, src_res=RES1))
            y["raft"]["corr_implementation"] = corr
            assert y["raft"]["mixed_precision"] is False
            c = ConfigStereoHuman()
            with tempfile.NamedTemporaryFile("w", suffix=".yaml", delete=False) as f:
                f.write(yaml.safe_dump(y))
            c.load(f.name)
            os.unlink(f.name)
            cfg = c.get_cfg()
            torch.manual_seed(1314)
            model = RtStereoHumanModel(cfg, with_gs_render=False).cuda().eval()
            ds = StereoHumanDataset(cfg.dataset, phase='val')
            data = default_collate([ds[0], ds[1]])
            for v in VIEWS:
                for k in data[v]:
                    data[v][k] = data[v][k].cuda()
            with torch.no_grad():
                data, _, _ = model(data, is_train=False)
            flows[corr] = torch.cat([data["lmain"]["flow_pred"], data["rmain"]["flow_pred"]]).float()
        finally:
            patch.uninstall()
    a, b = flows["reg"], flows["reg_cuda"]
    err, mag = float((a - b).abs().max()), float(a.abs().max())
    print(f"stage-1 fp32 flow after val_iters: max|reg|={mag:.3f}px, max|reg - reg_cuda|={err:.3e}px")
    assert math.isfinite(err) and err < 5e-3 * max(1.0, mag), (err, mag)
