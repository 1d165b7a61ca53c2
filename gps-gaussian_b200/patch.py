"""Opt-in route for the B200 fast paths on the UNMODIFIED reference scripts (VERDICT r1 "missing" item 3).

With only `dropin/` on PYTHONPATH the reference's own Python still runs around the two drop-in extensions:
core/corr.py:53-61 builds the volume with einsum -> cuBLAS + `/sqrt(D)` + three `avg_pool2d` and looks it up with four
sampler launches + `cat` (:44-51); lib/GaussianRender.py:14-33 does ten boolean-mask gathers per sample before `render`.
`GPSG_PATCH=1` (read by `dropin/sitecustomize.py`, which Python imports at start-up when `dropin/` is on PYTHONPATH)
installs a post-import hook that, right after the reference executes those two modules, rebinds

    core.corr.CorrBlockFast1D, core.corr.CorrSampler   -> gps_gaussian_b200.corr   (fused tcgen05 build, fused lookup)
    lib.GaussianRender.pts2render                      -> gps_gaussian_b200.GaussianRender.pts2render (fused map ingest)

so `from core.corr import CorrBlockFast1D` (core/raft_stereo_human.py:6) and `from lib.GaussianRender import pts2render`
(train_stage2.py:15, test_view_interp.py:15) pick ours up.  Same names, signatures and results (tests/test_c3_gpu.py runs
the stage-2 step both ways).  `install()` / `uninstall()` do the same for modules that are already imported.

lib.TaichiRender (train_stage1.py:16) cannot be patched after it executes: it imports `taichi` and calls
`ti.init(ti.cuda)` at import time, and taichi is not installable here.  It is SUBSTITUTED instead: while the hook is
installed, `import lib.TaichiRender` yields a module whose `TaichiRenderBatch` is gps_gaussian_b200.TaichiRender's (the
sm_100a preview splat), without running the reference file.  A real lib.TaichiRender that is already imported (taichi
present) gets its attribute rebound like the other targets.  `uninstall()` drops the substitute from sys.modules, so the
next import runs the reference module again (and fails again without taichi).
"""
import importlib.abc
import importlib.machinery
import sys

_ORIG = {}            # (module name, attribute) -> original object


def _set(mod, attr, new):
    key = (mod.__name__, attr)
    if key not in _ORIG:
        _ORIG[key] = getattr(mod, attr, None)
    setattr(mod, attr, new)


def _patch_corr(mod):
    from gps_gaussian_b200 import corr as ours
    _set(mod, "CorrBlockFast1D", ours.CorrBlockFast1D)
    _set(mod, "CorrSampler", ours.CorrSampler)
    user = sys.modules.get("core.raft_stereo_human")          # `from core.corr import ...` copies the binding
    if user is not None and hasattr(user, "CorrBlockFast1D"):
        _set(user, "CorrBlockFast1D", ours.CorrBlockFast1D)


def _patch_render(mod):
    from gps_gaussian_b200 import GaussianRender as ours
    _set(mod, "pts2render", ours.pts2render)


def _patch_taichi(mod):
    from gps_gaussian_b200 import TaichiRender as ours
    _set(mod, "TaichiRenderBatch", ours.TaichiRenderBatch)


_TARGETS = {"core.corr": _patch_corr, "lib.GaussianRender": _patch_render, "lib.TaichiRender": _patch_taichi}
_SUBSTITUTE = {"lib.TaichiRender"}       # never executed: the hook builds the module from ours
_MARK = "__gpsg_substitute__"


class _SubstituteLoader(importlib.abc.Loader):
    def __init__(self, hook):
        self._hook = hook

    def create_module(self, spec):
        return None                      # default module object

    def exec_module(self, module):
        setattr(module, _MARK, True)
        self._hook(module)


class _PatchingLoader(importlib.abc.Loader):
    def __init__(self, inner, hook):
        self._inner, self._hook = inner, hook

    def create_module(self, spec):
        return self._inner.create_module(spec)

    def exec_module(self, module):
        self._inner.exec_module(module)
        self._hook(module)


class _Finder(importlib.abc.MetaPathFinder):
    def find_spec(self, name, path=None, target=None):
        hook = _TARGETS.get(name)
        if hook is None:
            return None
        if name in _SUBSTITUTE:
            return importlib.machinery.ModuleSpec(name, _SubstituteLoader(hook), origin="gps_gaussian_b200 substitute")
        for finder in sys.meta_path:
            if finder is self or not hasattr(finder, "find_spec"):
                continue
            spec = finder.find_spec(name, path, target)
            if spec is not None and spec.loader is not None:
                spec.loader = _PatchingLoader(spec.loader, hook)
                return spec
        return None


_FINDER = _Finder()


def install():
    """Hook future imports and patch what is already imported. Idempotent."""
    if _FINDER not in sys.meta_path:
        sys.meta_path.insert(0, _FINDER)
    for name, hook in _TARGETS.items():
        if name in sys.modules:
            hook(sys.modules[name])


def uninstall():
    if _FINDER in sys.meta_path:
        sys.meta_path.remove(_FINDER)
    for (modname, attr), orig in list(_ORIG.items()):
        mod = sys.modules.get(modname)
        if mod is not None and orig is not None and not getattr(mod, _MARK, False):
            setattr(mod, attr, orig)
    _ORIG.clear()
    for name in _SUBSTITUTE:
        mod = sys.modules.get(name)
        if mod is not None and getattr(mod, _MARK, False):
            del sys.modules[name]
            parent, _, child = name.rpartition(".")
            if getattr(sys.modules.get(parent), child, None) is mod:
                delattr(sys.modules[parent], child)


def active():
    return _FINDER in sys.meta_path
