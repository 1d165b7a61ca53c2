"""BASELINE config C3 on hardware: the reference's OWN stage-2 model, loader and optimisation step against the drop-ins.

Only `gps-gaussian_b200/dropin` (-> `diff_gaussian_rasterization`, `corr_sampler`, `yacs`) and the staged, unmodified
reference tree `oracle/_ref` (git-ignored; staged by `build()`, see oracle/build.py) are put on `sys.path`.  The
repository does not carry the reference's sources, so these tests skip where nothing was staged.  Checked, per VERDICT r1 "next round" item 1:
  (a) train_stage2.py:57-89 executed statement for statement (AMP + GradScaler): finite loss, finite gradients on every
      parameter, the scaler does not skip the step;
  (b) `img_pred` equals the CPU-oracle render of the Gaussians the network produced, within the rasterizer parity bound;
  (c) the disparity ("flow") after 3 GRU iterations through `corr_implementation='reg_cuda'` (CorrBlockFast1D -> our
      `corr_sampler`) equals the same model through 'reg' (the reference's pure-PyTorch CorrBlock1D, core/corr.py:110-156);
  (d) `train_stage2.py` itself runs 3 steps as a subprocess and `test_view_interp.py` renders novel views from the
      checkpoint it wrote -- with and without the GPSG_PATCH=1 import hook;
  (e) the hook's fused paths (tcgen05 volume build + fused lookup, fused map ingest) give the same step as the plain
      drop-ins.
"""
import glob
import math
import os

import numpy as np
import pytest
import torch

from gps_gaussian_b200 import harness

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(harness.staged_reference() is None,
                                 reason="oracle/_ref not staged (python oracle/build.py --reference <GPS-Gaussian checkout>)")]

RES = 512


@pytest.fixture(scope="module")
def dataset(tmp_path_factory):
    from gps_gaussian_b200 import synth_dataset
    root = str(tmp_path_factory.mktemp("c3data"))
    synth_dataset.write_dataset(root, n_train=2, n_val=1, res=RES, hr=True)
    return root


def _state(dataset, corr="reg_cuda", seed=1314):
    cfg = harness.load_cfg(dataset, src_res=RES, num_steps=3, batch_size=2, corr_implementation=corr)
    return harness.C3State(cfg, seed=seed)


def _gather_gaussians(data, i):
    """The reference's gather (lib/GaussianRender.py:14-33) of sample i, as numpy for the oracle."""
    parts = {k: [] for k in ("xyz", "rgb", "rot", "scale", "op")}
    for view in ("lmain", "rmain"):
        d = data[view]
        valid = d["pts_valid"][i]
        parts["xyz"].append(d["xyz"][i][valid])
        parts["rgb"].append(d["img"][i].permute(1, 2, 0).reshape(-1, 3)[valid])
        parts["rot"].append(d["rot_maps"][i].permute(1, 2, 0).reshape(-1, 4)[valid])
        parts["scale"].append(d["scale_maps"][i].permute(1, 2, 0).reshape(-1, 3)[valid])
        parts["op"].append(d["opacity_maps"][i].permute(1, 2, 0).reshape(-1, 1)[valid])
    cat = lambda k: torch.cat(parts[k], 0).detach().float().cpu().numpy()
    nv = data["novel_view"]
    return dict(means3D=cat("xyz"), colors=cat("rgb") * np.float32(0.5) + np.float32(0.5), rots=cat("rot"),
                scales=cat("scale"), opacity=cat("op"), H=int(nv["height"][i]), W=int(nv["width"][i]),
                tanfovx=math.tan(float(nv["FovX"][i]) * 0.5), tanfovy=math.tan(float(nv["FovY"][i]) * 0.5),
                view=nv["world_view_transform"][i].float().cpu().numpy().reshape(16),
                proj=nv["full_proj_transform"][i].float().cpu().numpy().reshape(16),
                campos=nv["camera_center"][i].float().cpu().numpy(), bg=np.zeros(3, np.float32))


def test_c3_step_against_dropins_finite_and_matches_oracle(dataset):
    from helpers import oracle_forward
    st = _state(dataset)
    assert sum(p.numel() for p in st.model.parameters()) == 5_144_408            # BASELINE.md: 20.6 MB of fp32 grads
    import diff_gaussian_rasterization, corr_sampler
    assert "gps-gaussian_b200" in diff_gaussian_rasterization.__file__ and "gps-gaussian_b200" in corr_sampler.__file__
    import lib.GaussianRender as ref_render
    assert ref_render.__file__.startswith(harness.REF_STAGED)                     # the reference's own pts2render is what runs
    data = st.batch(0)
    assert not data["novel_view"]["world_view_transform"].is_cuda                 # host camera tensors, as upstream
    out = harness.c3_step(st, data)
    # (a)
    assert math.isfinite(float(out["loss"])) and math.isfinite(float(out["flow_loss"])) and math.isfinite(float(out["l1"]))
    assert math.isfinite(float(out["grad_norm"])), "non-finite gradient norm after unscale_"
    # n_gru_layers == 1 (config/stereo_human_config.py:38): the 1/16 and 1/32 GRUs and their context heads exist but are
    # never called, upstream as here -- every other parameter must have received a finite gradient
    n_none = [n for n, p in st.model.named_parameters() if p.grad is None]
    assert all(("gru16" in n or "gru32" in n or "outputs16" in n or "outputs32" in n or "layer4" in n or "layer5" in n)
               for n in n_none), [n for n in n_none][:8]
    with_grad = [p for p in st.model.parameters() if p.grad is not None]
    assert sum(p.numel() for p in with_grad) > 2_000_000
    assert all(bool(torch.isfinite(p.grad).all()) for p in with_grad)
    assert out["scale_after"] >= out["scale_before"], "GradScaler skipped the step (inf/nan gradients)"
    # gradients reached the Gaussian-parameter heads and the stereo update block through the rasterizer / sampler
    gp = st.model.gs_parm_regresser
    for head in (gp.rot_head, gp.scale_head, gp.opacity_head):
        assert float(sum(p.grad.abs().sum() for p in head.parameters())) > 0
    assert float(sum(p.grad.abs().sum() for p in st.model.raft_stereo.update_module.parameters() if p.grad is not None)) > 0
    # (b)
    img_pred = out["data"]["novel_view"]["img_pred"]
    assert tuple(img_pred.shape) == (2, 3, 2 * RES, 2 * RES)
    for i in range(2):
        sc = _gather_gaussians(out["data"], i)
        assert sc["means3D"].shape[0] > 50_000 and np.isfinite(sc["means3D"]).all()
        _, ref = oracle_forward(sc, "f32", nthreads=os.cpu_count() or 8)
        assert ref["num_rendered"] > sc["means3D"].shape[0] // 2                  # the plane of Gaussians is in view
        d = np.abs(img_pred[i].detach().cpu().numpy() - ref["color"]).max(0)
        frac = float((d > 1e-4).mean())
        print(f"C3 sample {i}: P={sc['means3D'].shape[0]} N={ref['num_rendered']} max|d|={d.max():.3e} frac>1e-4={frac:.2e}")
        assert frac < 5e-4 and d.max() < 1e-2, (frac, d.max())


def test_c3_flow_reg_cuda_equals_reg(dataset):
    """Same seed => same weights; same batch; only the correlation implementation differs."""
    flows = {}
    for corr in ("reg", "reg_cuda"):
        st = _state(dataset, corr=corr)
        data = st.batch(0)
        with torch.no_grad():
            data, flow_loss, _ = st.model(data, is_train=True)
        flows[corr] = (torch.cat([data["lmain"]["flow_pred"], data["rmain"]["flow_pred"]]).float(), float(flow_loss))
        del st
    a, b = flows["reg"][0], flows["reg_cuda"][0]
    err = float((a - b).abs().max())
    mag = float(a.abs().max())
    print(f"flow after 3 iters: max|reg|={mag:.3f}px, max|reg - reg_cuda|={err:.3e}px, flow_loss {flows['reg'][1]:.4f} vs {flows['reg_cuda'][1]:.4f}")
    # fp16 volume (half ulp 2^-11 relative on correlations of O(1..10)) fed through 3 GRU iterations and x8 upsampling
    assert err < 5e-3 * max(1.0, mag), (err, mag)                       # measured on B200: 1.5e-3 px on a 3.9 px field
    assert abs(flows["reg"][1] - flows["reg_cuda"][1]) < 1e-2 * max(1.0, abs(flows["reg"][1]))


def test_c3_patched_fast_paths_give_the_same_step(dataset):
    """GPSG_PATCH route (fused tcgen05 volume build + fused 4-level lookup + fused map ingest) vs the plain drop-ins."""
    from gps_gaussian_b200 import patch
    res = {}
    for mode in ("plain", "patched"):
        if mode == "patched":
            patch.install()
        try:
            st = _state(dataset)
            import core.corr, core.raft_stereo_human, lib.GaussianRender
            want = "gps_gaussian_b200" if mode == "patched" else "core.corr"
            assert core.raft_stereo_human.CorrBlockFast1D.__module__.startswith(want)
            assert lib.GaussianRender.pts2render.__module__.startswith("gps_gaussian_b200" if mode == "patched" else "lib.")
            out = harness.c3_step(st, st.batch(0), pts2render=lib.GaussianRender.pts2render)
            grads = torch.cat([p.grad.reshape(-1) for p in st.model.parameters() if p.grad is not None]).double()
            res[mode] = (out["data"]["novel_view"]["img_pred"].detach().clone(), float(out["loss"]), grads,
                         out["scale_after"] >= out["scale_before"])
        finally:
            patch.uninstall()
    (ia, la, ga, oka), (ib, lb, gb, okb) = res["plain"], res["patched"]
    assert oka and okb
    d = (ia - ib).abs()
    cos = float((ga * gb).sum() / (ga.norm() * gb.norm()))
    print(f"patched vs plain: loss {la:.6f} vs {lb:.6f}; img max|d|={float(d.max()):.3e} frac>1e-4={float((d > 1e-4).float().mean()):.2e}; "
          f"grad cosine {cos:.6f}, |g| {float(ga.norm()):.4e} vs {float(gb.norm()):.4e}")
    assert abs(la - lb) < 2e-3 * max(1.0, abs(la))
    assert float((d > 1e-3).float().mean()) < 1e-3
    assert cos > 0.99


@pytest.mark.parametrize("patched", [False, True])
def test_reference_scripts_run_unmodified(dataset, tmp_path, patched):
    """(d): `python train_stage2.py` (3 steps, batch 2, AMP) then `python test_view_interp.py` on the checkpoint it
    saved, cwd = a working copy of oracle/_ref whose only change is config/stage2.yaml's data_root / num_steps."""
    work = harness.make_workdir(str(tmp_path / "work"), dataset, src_res=RES, num_steps=3, batch_size=2)
    for name in ("train_stage2.py", "test_view_interp.py", "lib/GaussianRender.py", "core/corr.py"):
        with open(os.path.join(work, name), "rb") as a, open(os.path.join(harness.REF_STAGED, name), "rb") as b:
            assert a.read() == b.read()
    p = harness.run_script(work, "train_stage2.py", patch=patched, timeout=1500)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-6000:]
    assert "FINISHED TRAINING" in p.stdout
    ckpts = glob.glob(os.path.join(work, "experiments", "*", "ckpt", "*_final.pth"))
    assert len(ckpts) == 1
    sd = torch.load(ckpts[0], map_location="cpu")
    assert sd["total_steps"] == 3 and all(bool(torch.isfinite(v).all()) for v in sd["network"].values() if v.is_floating_point())
    q = harness.run_script(work, "test_view_interp.py", ["--test_data_root", os.path.join(dataset, "val"), "--ckpt_path",
                                                          ckpts[0], "--novel_view_nums", "3"], patch=patched, timeout=900)
    assert q.returncode == 0, q.stdout[-3000:] + q.stderr[-6000:]
    imgs = sorted(glob.glob(os.path.join(work, "interp_out", "*.jpg")))
    assert len(imgs) == 3
    import cv2
    for f in imgs:
        im = cv2.imread(f)
        assert im.shape == (2 * RES, 2 * RES, 3) and im.mean() > 1.0              # something was rendered
