"""Harness items of SURVEY.md 8f-4 on the CPU: the `yacs` stand-in loads the reference's stage-2 config
(tests/golden/stage2.yaml), the synthetic dataset writer produces the files the reference's own `StereoHumanDataset` read
into flow whose unprojection lands on the analytic surface (tests/golden/loader_golden.npz, recorded by
tests/golden/make_loader_golden.py), and the GPSG_PATCH hook rebinds the reference's entry points (on stand-in modules
with the reference's module and attribute names).  Building the reference's model needs its sources, staged into
oracle/_ref by `build()` (oracle/build.py); that test skips where nothing was staged."""
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DROPIN = os.path.join(ROOT, "gps-gaussian_b200", "dropin")
GOLDEN = os.path.join(ROOT, "tests", "golden")

# stand-ins for the reference modules the hook targets: same module names, same import of CorrBlockFast1D into
# core.raft_stereo_human (core/raft_stereo_human.py:6), same public names
STANDIN = {
    "core/__init__.py": "",
    "core/corr.py": "class CorrSampler:\n    pass\n\n\nclass CorrBlock1D:\n    pass\n\n\nclass CorrBlockFast1D:\n    pass\n",
    "core/raft_stereo_human.py": "from core.corr import CorrBlock1D, CorrBlockFast1D\n",
    "lib/__init__.py": "",
    "lib/GaussianRender.py": "def pts2render(data, bg_color):\n    return data\n",
}


@pytest.fixture
def standin_tree(tmp_path):
    for name, code in STANDIN.items():
        os.makedirs(os.path.dirname(os.path.join(tmp_path, name)), exist_ok=True)
        with open(os.path.join(tmp_path, name), "w") as f:
            f.write(code)
    return str(tmp_path)


def test_yacs_standin_loads_the_reference_config():
    if DROPIN not in sys.path:
        sys.path.insert(0, DROPIN)
    import yacs.config
    assert yacs.config.__file__.startswith(DROPIN)                  # ours, not an installed yacs
    from yacs.config import CfgNode as CN
    c = CN()                                                        # the defaults the reference's ConfigStereoHuman sets
    for k, v in (("name", ""), ("stage1_ckpt", None), ("restore_ckpt", None), ("lr", 0.0), ("wdecay", 0.0),
                 ("batch_size", 0), ("num_steps", 0)):
        setattr(c, k, v)
    c.dataset = CN()
    for k in ("source_id", "train_novel_id", "val_novel_id", "src_res", "use_hr_img", "use_processed_data"):
        setattr(c.dataset, k, None)
    c.dataset.data_root, c.dataset.znear, c.dataset.zfar = "", 0.01, 100.0
    c.raft = CN()
    c.raft.mixed_precision, c.raft.train_iters, c.raft.val_iters = None, 0, 0
    c.raft.corr_implementation, c.raft.encoder_dims, c.raft.hidden_dims = "reg_cuda", [64, 96, 128], [128] * 3
    c.gsnet = CN()
    c.gsnet.encoder_dims = c.gsnet.decoder_dims = c.gsnet.parm_head_dim = None
    c.record = CN()
    c.record.ckpt_path = c.record.show_path = None
    c.record.loss_freq = c.record.eval_freq = 0
    c.defrost()                                                     # ConfigStereoHuman.load
    c.merge_from_file(os.path.join(GOLDEN, "stage2.yaml"))
    c.freeze()
    cfg = c.clone()                                                 # ConfigStereoHuman.get_cfg
    assert cfg.batch_size == 2 and cfg.restore_ckpt is None and abs(cfg.wdecay - 1e-5) < 1e-12      # 'None' / '1e-5' decoded
    assert cfg.raft.mixed_precision is True and cfg.raft.hidden_dims == [96, 96, 96] and cfg.dataset.use_hr_img is True
    assert cfg.raft.corr_implementation == "reg_cuda" and cfg.dataset.znear == 0.01                 # defaults survive
    with pytest.raises(AttributeError):
        cfg.exp_name = "x"                                                                          # frozen after load
    cfg.defrost()
    cfg.exp_name = "x"
    cfg.record.ckpt_path = "p"                                                                      # train_stage2.py:192-199
    cfg.freeze()
    import json
    assert json.loads(json.dumps(cfg))["record"]["ckpt_path"] == "p"                                # lib/train_recoder.py:24
    with pytest.raises(KeyError):
        cfg.clone().merge_from_list(["no.such.key", 1])


def test_synthetic_dataset_is_read_by_the_reference_loader(tmp_path):
    """What the reference's loader returned for the files the writer wrote (golden), and that the writer still writes
    those files."""
    import cv2
    from gps_gaussian_b200 import synth_dataset
    from oracle import unproject_oracle
    G = np.load(os.path.join(GOLDEN, "loader_golden.npz"))
    res = 96
    names = synth_dataset.write_dataset(str(tmp_path), n_train=2, n_val=1, res=res, hr=True)
    assert names["train"] == list(G["train_names"]) == list(G["sample_list"])
    for vid in (0, 1):                                              # what the loader consumed to make flow / calibration
        assert np.array_equal(cv2.imread(os.path.join(str(tmp_path), "train", "depth", names["train"][0], f"{vid}.png"), -1),
                              G[f"written_depth_{vid}"])
        for m in ("intrinsic", "extrinsic"):
            got = np.load(os.path.join(str(tmp_path), "train", "parm", names["train"][0], f"{vid}_{m}.npy"))
            assert np.allclose(got, G[f"written_{m}_{vid}"], rtol=0, atol=1e-12)
    item = {v: {k: G[f"{v}_{k}"] for k in ("img", "mask", "flow", "valid", "intr", "extr", "ref_intr", "Tf_x")}
            for v in ("lmain", "rmain")}
    for v in ("lmain", "rmain"):
        d = item[v]
        assert tuple(d["img"].shape) == (3, res, res) and tuple(d["mask"].shape) == (3, res, res)
        assert tuple(d["flow"].shape) == (1, res, res) and tuple(d["valid"].shape) == (1, res, res)
        assert float(d["valid"].mean()) > 0.1 and -1.0 <= float(d["img"].min()) and float(d["img"].max()) <= 1.0
    assert tuple(G["novel_img_shape"]) == (3, 2 * res, 2 * res) and int(G["novel_width"]) == 2 * res   # _hr image of view 3
    # flow (reference rectification + stereo_pts2flow) -> depth -> points (our oracle of flow2depth + depth2pc):
    # every valid point must lie on the capsule that was rendered (radius of sample 0, axis x = z = 0).
    radii = np.random.default_rng(synth_dataset.synth.SEED)
    r0 = 0.425 * float(radii.uniform(0.9, 1.05))
    for v in ("lmain", "rmain"):
        d = item[v]
        flow = d["flow"][None].astype(np.float64)
        valid = d["valid"][None].astype(np.float64)
        depth, xyz, pv = unproject_oracle.unproject(flow, np.repeat(valid, 3, 1), d["intr"][None].astype(np.float64),
                                                    d["extr"][None].astype(np.float64), d["ref_intr"][None].astype(np.float64),
                                                    d["Tf_x"].reshape(1).astype(np.float64))
        pts = xyz[0][pv[0]]
        mid = pts[(pts[:, 1] > r0 + 0.05) & (pts[:, 1] < 1.8 - r0 - 0.05)]            # cylinder part of the capsule
        assert mid.shape[0] > 200
        rad = np.sqrt(mid[:, 0] ** 2 + mid[:, 2] ** 2)
        assert abs(np.median(rad) - r0) < 0.01 and np.percentile(np.abs(rad - r0), 90) < 0.03, (np.median(rad), r0)
    # the test-time path (test_view_interp.py): original calibration for get_novel_calib
    assert tuple(G["test_lmain_intr_ori_shape"]) == (3, 3) and tuple(G["test_rmain_extr_ori_shape"]) == (3, 4)
    assert int(G["test_novel_height"]) == 2 * res


def test_import_hook_rebinds_the_reference_entry_points(standin_tree, tmp_path):
    """GPSG_PATCH=1 + dropin/ on PYTHONPATH: `sitecustomize` installs the post-import hook, the reference's own
    `from core.corr import CorrBlockFast1D` / `from lib.GaussianRender import pts2render` resolve to the fused paths;
    without the variable nothing is touched."""
    code = ("import core.raft_stereo_human as r, core.corr as c\n"
            "from lib.GaussianRender import pts2render\n"
            "print(r.CorrBlockFast1D.__module__, c.CorrSampler.__module__, pts2render.__module__)\n")
    out = {}
    for flag in ("0", "1"):
        env = dict(os.environ, PYTHONPATH=os.pathsep.join([DROPIN, standin_tree]), GPSG_PATCH=flag)
        p = subprocess.run([sys.executable, "-c", code], env=env, cwd=str(tmp_path), capture_output=True, text=True)
        assert p.returncode == 0, p.stderr[-2000:]
        out[flag] = p.stdout.split()
    assert out["0"] == ["core.corr", "core.corr", "lib.GaussianRender"]
    assert out["1"] == ["gps_gaussian_b200.corr", "gps_gaussian_b200.corr", "gps_gaussian_b200.GaussianRender"]


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "train_stage2.py")),
                    reason="oracle/_ref not staged (python oracle/build.py --reference <GPS-Gaussian checkout>)")
def test_c3_harness_builds_the_reference_model_and_batch_on_cpu(tmp_path):
    """Plumbing of gps_gaussian_b200.harness without a GPU: staged tree, config, the reference's loader + model (the
    pure-PyTorch 'reg' correlation path), one forward.  The GPU half is tests/test_c3_gpu.py."""
    from gps_gaussian_b200 import harness, synth_dataset
    assert harness.staged_reference() is not None
    root = str(tmp_path / "data")
    synth_dataset.write_dataset(root, n_train=2, n_val=1, res=128, hr=True)
    cfg = harness.load_cfg(root, src_res=128, num_steps=3, batch_size=2, corr_implementation="reg")
    assert cfg.stage1_ckpt is None and cfg.num_steps == 3 and cfg.dataset.data_root == root
    st = harness.C3State(cfg, device="cpu")
    data = st.batch(0)
    assert tuple(data["lmain"]["img"].shape) == (2, 3, 128, 128) and tuple(data["novel_view"]["img"].shape) == (2, 3, 256, 256)
    data, flow_loss, metrics = st.model(data, is_train=True)
    assert tuple(data["lmain"]["xyz"].shape) == (2, 128 * 128, 3) and data["rmain"]["pts_valid"].dtype == torch.bool
    assert bool(torch.isfinite(flow_loss)) and "train_epe" in metrics


@pytest.fixture
def standin_modules(standin_tree, monkeypatch):
    """The stand-ins importable in this process; `core` / `lib` modules imported before come back afterwards."""
    names = ("core", "core.corr", "core.raft_stereo_human", "lib", "lib.GaussianRender")
    saved = {m: sys.modules.pop(m) for m in names if m in sys.modules}
    monkeypatch.syspath_prepend(standin_tree)
    yield
    for m in names:
        sys.modules.pop(m, None)
    sys.modules.update(saved)


def test_patch_install_and_uninstall_in_process(standin_modules):
    """`patch.install()` rebinds modules that are ALREADY imported (incl. the `from core.corr import ...` copy held by
    core.raft_stereo_human); `patch.uninstall()` puts the reference's own objects back."""
    from gps_gaussian_b200 import patch
    import core.corr
    import core.raft_stereo_human
    import lib.GaussianRender
    orig = (core.corr.CorrBlockFast1D, core.corr.CorrSampler, core.raft_stereo_human.CorrBlockFast1D, lib.GaussianRender.pts2render)
    assert all(o.__module__ in ("core.corr", "lib.GaussianRender") for o in orig)
    patch.install()
    try:
        assert patch.active()
        assert core.corr.CorrBlockFast1D.__module__ == "gps_gaussian_b200.corr"
        assert core.raft_stereo_human.CorrBlockFast1D is core.corr.CorrBlockFast1D
        assert lib.GaussianRender.pts2render.__module__ == "gps_gaussian_b200.GaussianRender"
        patch.install()                                                   # idempotent
    finally:
        patch.uninstall()
    assert not patch.active()
    assert (core.corr.CorrBlockFast1D, core.corr.CorrSampler, core.raft_stereo_human.CorrBlockFast1D,
            lib.GaussianRender.pts2render) == orig
