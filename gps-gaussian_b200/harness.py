"""Run the UNMODIFIED reference scripts and model against the drop-ins (BASELINE config C3; VERDICT r1 item N1).

The reference tree is staged, byte for byte, into the git-ignored `oracle/_ref/` by `oracle/build.py` when it finds a
GPS-Gaussian checkout (`--reference DIR`, GPSG_REFERENCE_DIR, or its default location); it is never committed and
nothing in the product imports it.  Everything here is harness: it builds the reference's own `RtStereoHumanModel`, feeds it the synthetic
dataset through the reference's own `StereoHumanDataset`, and executes the optimisation step of the reference's
train_stage2.py:57-89 -- with `gps-gaussian_b200/dropin` providing `diff_gaussian_rasterization`,
`corr_sampler` and `yacs`.  Used by tests/test_c3_gpu.py and bench.py's `train_c3` block.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
DROPIN = os.path.join(HERE, "dropin")
REF_STAGED = os.path.join(ROOT, "oracle", "_ref")
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from oracle.build import make_writable  # noqa: E402


def staged_reference():
    return REF_STAGED if os.path.exists(os.path.join(REF_STAGED, "train_stage2.py")) else None


def add_reference_to_path():
    """dropin first (so `diff_gaussian_rasterization`, `corr_sampler`, `yacs` resolve to ours), then the staged tree."""
    ref = staged_reference()
    if ref is None:
        raise FileNotFoundError("oracle/_ref is not staged: run python oracle/build.py --reference <GPS-Gaussian checkout>")
    for p in (ref, DROPIN, ROOT):
        if p in sys.path:
            sys.path.remove(p)
        sys.path.insert(0, p)
    return ref


def stage2_yaml(data_root, src_res=512, num_steps=3, batch_size=2, corr_implementation=None, use_processed_data=True):
    """The reference's own config/stage2.yaml with only the user-facing knobs changed (data_root and stage1_ckpt are
    placeholders upstream: 'PATH/TO/...')."""
    import yaml
    with open(os.path.join(staged_reference(), "config", "stage2.yaml")) as f:
        y = yaml.safe_load(f)
    y["stage1_ckpt"] = "None"
    y["num_steps"] = int(num_steps)
    y["batch_size"] = int(batch_size)
    y["dataset"]["src_res"] = int(src_res)
    y["dataset"]["data_root"] = str(data_root)
    y["dataset"]["use_processed_data"] = bool(use_processed_data)
    if corr_implementation is not None:
        y["raft"]["corr_implementation"] = corr_implementation
    return yaml.safe_dump(y, sort_keys=False)


def make_workdir(path, data_root, **cfg):
    """A working copy of the staged tree (the scripts resolve 'config/stage2.yaml', 'core', 'lib', ... relative to the
    cwd and write experiments/ into it) with our config/stage2.yaml in place of the placeholder one."""
    ref = staged_reference()
    if ref is None:
        raise FileNotFoundError("oracle/_ref is not staged")
    if os.path.isdir(path):
        shutil.rmtree(path)
    shutil.copytree(ref, path)
    make_writable(path)
    with open(os.path.join(path, "config", "stage2.yaml"), "w") as f:
        f.write(stage2_yaml(data_root, **cfg))
    return path


def script_env(patch=False, extra=None):
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([DROPIN] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    env["GPSG_PATCH"] = "1" if patch else "0"
    env.setdefault("CUDA_VISIBLE_DEVICES", "0")
    if extra:
        env.update(extra)
    return env


def run_script(workdir, script, args=(), patch=False, timeout=900):
    """python <script> in the working copy with only dropin/ on PYTHONPATH. Returns CompletedProcess."""
    return subprocess.run([sys.executable, script] + list(args), cwd=workdir, env=script_env(patch), text=True,
                          capture_output=True, timeout=timeout)


# ----------------------------------------------------------------------------------------------------------------
# in-process: the reference's own model, loader and optimisation step
# ----------------------------------------------------------------------------------------------------------------

def load_cfg(data_root, **kw):
    add_reference_to_path()
    import tempfile
    from config.stereo_human_config import ConfigStereoHuman
    c = ConfigStereoHuman()
    with tempfile.NamedTemporaryFile("w", suffix=".yaml", delete=False) as f:
        f.write(stage2_yaml(data_root, **kw))
    try:
        c.load(f.name)
    finally:
        os.unlink(f.name)
    return c.get_cfg()


class C3State:
    """What train_stage2.py's Trainer.__init__ builds (:28-55), minus logger / val set / checkpoint I/O."""

    def __init__(self, cfg, seed=1314, device="cuda"):
        import numpy as np
        import torch
        import torch.optim as optim
        from torch.cuda.amp import GradScaler
        from lib.human_loader import StereoHumanDataset
        from lib.network import RtStereoHumanModel
        torch.manual_seed(seed)                                                     # train_stage2.py:206-207
        np.random.seed(seed)
        self.cfg = cfg
        self.device = device
        self.model = RtStereoHumanModel(cfg, with_gs_render=True)
        self.train_set = StereoHumanDataset(cfg.dataset, phase='train')
        self.optimizer = optim.AdamW(self.model.parameters(), lr=cfg.lr, weight_decay=cfg.wdecay, eps=1e-8)
        self.scheduler = optim.lr_scheduler.OneCycleLR(self.optimizer, cfg.lr, cfg.num_steps + 100, pct_start=0.01,
                                                       cycle_momentum=False, anneal_strategy='linear')
        self.model.to(device)
        self.model.train()
        self.model.raft_stereo.freeze_bn()
        self.scaler = GradScaler(enabled=cfg.raft.mixed_precision)

    def batch(self, first=0):
        """`batch_size` samples collated like the reference DataLoader does (pin_memory=True), source views moved to the
        GPU like Trainer.fetch_data (:143-146); the novel-view camera tensors stay on the host, as upstream."""
        import torch
        from torch.utils.data import default_collate
        items = [self.train_set[first + k] for k in range(self.cfg.batch_size)]
        data = default_collate(items)
        if self.device != "cpu":
            for k, v in data['novel_view'].items():
                if torch.is_tensor(v):
                    data['novel_view'][k] = v.pin_memory()
        for view in ('lmain', 'rmain'):
            for item in data[view].keys():
                data[view][item] = data[view][item].to(self.device)
        return data


def c3_step(st, data, pts2render=None, timers=None, allreduce=None):
    """One optimisation step, statement for statement train_stage2.py:57-89 (logging / checkpointing left out).
    `timers`: optional dict that receives CUDA-event stage times in ms (nets / render_fwd / loss / backward / optim).
    `allreduce`: optional callable(params) run between backward and unscale_ (data-parallel C5, train_stage2.py:83-85)."""
    import torch
    from lib.loss import l1_loss, ssim
    if pts2render is None:
        from lib.GaussianRender import pts2render
    ev = []

    def mark(name):
        if timers is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            ev.append((name, e))

    mark("start")
    st.optimizer.zero_grad()
    data, flow_loss, metrics = st.model(data, is_train=True)                         # :62
    mark("nets_fwd")
    data = pts2render(data, bg_color=st.cfg.dataset.bg_color)                         # :64
    mark("render_fwd")
    render_novel = data['novel_view']['img_pred']
    gt_novel = data['novel_view']['img'].to(render_novel.device)
    Ll1 = l1_loss(render_novel, gt_novel)
    Lssim = 1.0 - ssim(render_novel, gt_novel)
    loss = 1.0 * flow_loss + 0.8 * Ll1 + 0.2 * Lssim                                  # :70-72
    mark("loss_fwd")
    st.scaler.scale(loss).backward()                                                  # :83
    mark("backward")
    if allreduce is not None:
        allreduce(st.model.parameters())
        mark("allreduce")
    st.scaler.unscale_(st.optimizer)                                                  # :84
    gnorm = torch.nn.utils.clip_grad_norm_(st.model.parameters(), 1.0)                # :85
    scale_before = st.scaler.get_scale() if st.scaler.is_enabled() else 1.0
    st.scaler.step(st.optimizer)                                                      # :87
    st.scheduler.step()
    st.scaler.update()                                                                # :89
    mark("optim")
    out = {"loss": loss.detach(), "flow_loss": flow_loss.detach(), "l1": Ll1.detach(), "ssim_loss": Lssim.detach(),
           "grad_norm": gnorm.detach() if torch.is_tensor(gnorm) else gnorm, "scale_before": scale_before,
           "scale_after": st.scaler.get_scale() if st.scaler.is_enabled() else 1.0, "metrics": metrics, "data": data}
    if timers is not None:
        torch.cuda.synchronize()
        for (_, a), (name, b) in zip(ev[:-1], ev[1:]):
            timers[name] = timers.get(name, 0.0) + a.elapsed_time(b)
    return out
