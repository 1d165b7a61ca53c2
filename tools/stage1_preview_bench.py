"""Time the stage-1 validation preview (TaichiRenderBatch.flow2render) at train_stage1.py's eval shape: res 1024, a val
batch of 2, bs = 1 (train_stage1.py:36, 52).

    python tools/stage1_preview_bench.py [--res 1024] [--out profiles/stage1_preview_bench.json]

ours:      gps_gaussian_b200.TaichiRender (csrc/point_splat.cu: one memset + two kernels)
reference: the staged reference's own lib/TaichiRender.py (oracle/_ref) under a minimal taichi stub, its Taichi kernel
           replaced by a no-op -- i.e. the torch prep alone (flow2depth, depth2pc, perspective, boolean-mask index_put,
           cat), which is a lower bound on upstream's time.
Each is warmed up, then timed with CUDA events over >= 1 s of back-to-back calls; the host synchronisations of one call
are counted with torch.cuda.set_sync_debug_mode("warn").  The GPU name and power limit are recorded beside the numbers.
The preview runs once per eval_freq training steps, so this is a record, not a gate.
"""
import argparse
import json
import os
import subprocess
import sys
import types
import warnings

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gps_gaussian_b200 import harness, synth  # noqa: E402
from gps_gaussian_b200.TaichiRender import TaichiRenderBatch  # noqa: E402


def _taichi_stub():
    ti = types.ModuleType("taichi")
    ti.cuda, ti.i32 = "cuda", "i32"
    ti.init = lambda *a, **k: None
    ti.data_oriented = ti.kernel = lambda f: f
    ti.Vector = types.SimpleNamespace(field=lambda **k: types.SimpleNamespace(**k))
    ti.types = types.SimpleNamespace(ndarray=lambda *a, **k: None)
    return ti


def _time(fn, min_s=1.0, warmup=10):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    n, total = 8, 0.0
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        b.synchronize()
        total = a.elapsed_time(b) / 1e3
        if total >= min_s:
            return total / n * 1e3, n, total
        n = int(n * max(2.0, 1.2 * min_s / max(total, 1e-6)))


def _syncs(fn):
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("warn")
    try:
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            fn()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    return sum("synchroniz" in str(x.message) for x in w)


def _gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, _, power = q.stdout.strip().partition(",")
    return dict(gpu=name.strip() or torch.cuda.get_device_name(0), power_limit=power.strip() or "unknown")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, default=1024)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "stage1_preview_bench.json"))
    args = ap.parse_args()
    res, B, bs = args.res, 2, 1
    d = synth.stage1_batch(res, B, seed=1314)
    data = {v: {k: torch.from_numpy(a).cuda() for k, a in d[v].items()} for v in ("lmain", "rmain", "novel_view")}
    ours = TaichiRenderBatch(bs, res)
    result = dict(_gpu(), shape=dict(res=res, B=B, bs=bs), torch=torch.__version__)
    ms, n, tot = _time(lambda: ours.flow2render(data))
    result["ours"] = dict(ms_per_call=ms, calls=n, seconds=tot, host_syncs=_syncs(lambda: ours.flow2render(data)))
    if harness.staged_reference() is not None:
        harness.add_reference_to_path()
        sys.modules["taichi"] = _taichi_stub()
        sys.modules.pop("lib.TaichiRender", None)
        import lib.TaichiRender as ref_mod
        ref = ref_mod.TaichiRenderBatch(bs, res)
        ref.render_respective_color = lambda *a: None
        fn = lambda: ref.flow2render({v: dict(data[v]) for v in data})
        ms, n, tot = _time(fn)
        result["reference_prep_only"] = dict(ms_per_call=ms, calls=n, seconds=tot, host_syncs=_syncs(fn))
        result["speedup_vs_reference_prep"] = result["reference_prep_only"]["ms_per_call"] / result["ours"]["ms_per_call"]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
