"""ctypes binding of libgpsg_sm100.so (the C ABI declared in include/gpsg.h).

There is NO fallback: if the shared library is missing this module raises at import time --
a product path that silently ran on the CPU oracle or on eager PyTorch would void every parity
claim.  Build it with `python gps-gaussian_b200/build.py` (or `__graft_entry__.build()`).
"""
import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libgpsg_sm100.so")


class GpsgError(RuntimeError):
    pass


class RasterSettings(C.Structure):
    """GpsgRasterSettings (include/gpsg.h) == the 12 fields of GaussianRasterizationSettings."""
    _fields_ = [("image_height", C.c_int32), ("image_width", C.c_int32), ("tanfovx", C.c_float),
                ("tanfovy", C.c_float), ("bg", C.c_float * 3), ("scale_modifier", C.c_float),
                ("viewmatrix", C.c_float * 16), ("projmatrix", C.c_float * 16), ("sh_degree", C.c_int32),
                ("campos", C.c_float * 3), ("prefiltered", C.c_int32), ("debug", C.c_int32)]


class GeomView(C.Structure):
    _fields_ = [("depths", C.c_void_p), ("means2D", C.c_void_p), ("conic_opacity", C.c_void_p),
                ("tiles_touched", C.c_void_p), ("point_offsets", C.c_void_p)]


class BinningView(C.Structure):
    _fields_ = [("point_list_keys", C.c_void_p), ("point_list", C.c_void_p)]


class ImageView(C.Structure):
    _fields_ = [("final_T", C.c_void_p), ("n_contrib", C.c_void_p), ("ranges", C.c_void_p)]


ALLOC_FN = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_size_t)

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: the CUDA extension is not built. Run `python gps-gaussian_b200/build.py` "
        "(nvcc, sm_100a). There is deliberately no CPU / PyTorch fallback.")

lib = C.CDLL(LIB_PATH)

_vp, _i, _i64, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_size_t
lib.gpsg_last_error.restype = C.c_char_p
lib.gpsg_last_error.argtypes = []
lib.gpsg_version.restype = _i
lib.gpsg_rasterize_forward.restype = _i
lib.gpsg_rasterize_forward.argtypes = [C.POINTER(RasterSettings), _i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                       _vp, _vp, ALLOC_FN, _vp, ALLOC_FN, _vp, ALLOC_FN, _vp, C.POINTER(C.c_int32)]
lib.gpsg_rasterize_backward_workspace_bytes.restype = _sz
lib.gpsg_rasterize_backward_workspace_bytes.argtypes = [_i]
lib.gpsg_rasterize_backward.restype = _i
lib.gpsg_rasterize_backward.argtypes = [C.POINTER(RasterSettings), _i, _vp, _i, _i, C.c_int32] + [_vp] * 21
lib.gpsg_mark_visible.restype = _i
lib.gpsg_mark_visible.argtypes = [_i, _vp, _i, _vp, C.POINTER(C.c_float), _vp]
lib.gpsg_geom_view.restype = _i
lib.gpsg_geom_view.argtypes = [_vp, _i, C.POINTER(GeomView)]
lib.gpsg_binning_view.restype = _i
lib.gpsg_binning_view.argtypes = [_vp, _i64, C.POINTER(BinningView)]
lib.gpsg_image_view.restype = _i
lib.gpsg_image_view.argtypes = [_vp, _i, _i, C.POINTER(ImageView)]
lib.gpsg_corr_sampler_forward.restype = _i
lib.gpsg_corr_sampler_forward.argtypes = [_i, _vp, _i, _i, _i, _i, _i, _vp, _i64, _i64, _i64, _vp, _i64, _i, _vp]
lib.gpsg_corr_sampler_backward.restype = _i
lib.gpsg_corr_sampler_backward.argtypes = [_i, _vp, _i, _i, _i, _i, _i, _vp, _i64, _vp, _i, _vp]

lib.gpsg_raster_geom_bytes.restype = _sz
lib.gpsg_raster_geom_bytes.argtypes = [_i]
lib.gpsg_raster_binning_bytes.restype = _sz
lib.gpsg_raster_binning_bytes.argtypes = [_i64]
lib.gpsg_raster_image_bytes.restype = _sz
lib.gpsg_raster_image_bytes.argtypes = [_i, _i]
lib.gpsg_raster_status_ptr.restype = _vp
lib.gpsg_raster_status_ptr.argtypes = [_vp, _i, _i]
lib.gpsg_rasterize_forward_planned.restype = _i
lib.gpsg_rasterize_forward_planned.argtypes = [C.POINTER(RasterSettings), _i, _vp, _i] + [_vp] * 10 + [_i64, _vp, _vp]
_pp = C.POINTER(C.c_void_p)
lib.gpsg_rasterize_forward_maps.restype = _i
lib.gpsg_rasterize_forward_maps.argtypes = [C.POINTER(RasterSettings), _i, _vp, _i, _pp, _pp, _pp, _pp, _pp, _pp, _vp, _vp,
                                            ALLOC_FN, _vp, ALLOC_FN, _vp, ALLOC_FN, _vp, C.POINTER(C.c_int32)]
lib.gpsg_rasterize_forward_maps_planned.restype = _i
lib.gpsg_rasterize_forward_maps_planned.argtypes = [C.POINTER(RasterSettings), _i, _vp, _i, _pp, _pp, _pp, _pp, _pp, _pp, _vp, _vp,
                                                    _vp, _vp, _i64, _vp, _vp]
lib.gpsg_rasterize_forward_maps_begin.restype = _i
lib.gpsg_rasterize_forward_maps_begin.argtypes = [C.POINTER(RasterSettings), _i, _vp, _i, _pp, _pp, _pp, _pp, _pp, _pp, _vp,
                                                  ALLOC_FN, _vp, ALLOC_FN, _vp, _vp]
lib.gpsg_rasterize_forward_maps_finish.restype = _i
lib.gpsg_rasterize_forward_maps_finish.argtypes = [C.POINTER(RasterSettings), _i, _vp, _i, _pp, _pp, _pp, _pp, _pp, _pp, _vp, _vp,
                                                   _vp, _vp, ALLOC_FN, _vp, _vp, C.POINTER(C.c_int32)]
lib.gpsg_rasterize_backward_maps_workspace_bytes.restype = _sz
lib.gpsg_rasterize_backward_maps_workspace_bytes.argtypes = [_i]
lib.gpsg_rasterize_backward_maps.restype = _i
lib.gpsg_rasterize_backward_maps.argtypes = [C.POINTER(RasterSettings), _i, _vp, _i, C.c_int32, _pp, _pp, _pp, _pp, _pp, _pp,
                                             _vp, _vp, _vp, _vp, _vp, _pp, _pp, _pp, _pp, _pp, _vp]
lib.gpsg_corr_build_pyramid.restype = _i
lib.gpsg_corr_build_pyramid.argtypes = [_i, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, C.POINTER(C.c_void_p), _i]
lib.gpsg_corr_build_backward.restype = _i
lib.gpsg_corr_build_backward.argtypes = [_i, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]
lib.gpsg_corr_lookup_pyramid_forward.restype = _i
lib.gpsg_corr_lookup_pyramid_forward.argtypes = [_i, _vp, _i, _i, _i, _i, C.POINTER(C.c_void_p), C.POINTER(C.c_int32), _i,
                                                 _vp, _i64, _i, _vp]
lib.gpsg_corr_lookup_pyramid_backward.restype = _i
lib.gpsg_corr_lookup_pyramid_backward.argtypes = [_i, _vp, _i, _i, _i, _i, C.POINTER(C.c_void_p), C.POINTER(C.c_int32), _i,
                                                  _vp, _i64, _i, _vp]
lib.gpsg_unproject_forward.restype = _i
lib.gpsg_unproject_forward.argtypes = [_i, _vp, _i, _i, _vp, _vp, _i64, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]
lib.gpsg_unproject_backward.restype = _i
lib.gpsg_unproject_backward.argtypes = [_i, _vp, _i, _i, _vp, _vp, _i64, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]
lib.gpsg_flow2render_workspace_bytes.restype = _sz
lib.gpsg_flow2render_workspace_bytes.argtypes = [_i, _i]
lib.gpsg_flow2render.restype = _i
lib.gpsg_flow2render.argtypes = [_i, _vp, _i, _i, _i, _i, _pp, _pp, C.POINTER(C.c_int64), _pp, _pp, _i, _pp, _pp, _pp, _vp,
                                 _vp, _sz, _vp, _vp]
lib.gpsg_l1_ssim_workspace_bytes.restype = _sz
lib.gpsg_l1_ssim_workspace_bytes.argtypes = [_i, _i, _i]
lib.gpsg_l1_ssim_forward.restype = _i
lib.gpsg_l1_ssim_forward.argtypes = [_i, _vp, _i, _i, _i, _vp, _vp, C.c_float, C.c_float, _vp, _vp, _vp]
lib.gpsg_l1_ssim_backward.restype = _i
lib.gpsg_l1_ssim_backward.argtypes = [_i, _vp, _i, _i, _i, _vp, _vp, _vp, C.c_float, C.c_float, _vp, _vp]
lib.gpsg_profile_enable.restype = _i
lib.gpsg_profile_enable.argtypes = [_i]
lib.gpsg_profile_read.restype = _i
lib.gpsg_profile_read.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_int32), _i]
lib.gpsg_profile_stage_name.restype = C.c_char_p
lib.gpsg_profile_stage_name.argtypes = [_i]

EXPORTED = ["gpsg_last_error", "gpsg_version", "gpsg_rasterize_forward", "gpsg_rasterize_backward_workspace_bytes",
            "gpsg_rasterize_backward", "gpsg_mark_visible", "gpsg_geom_view", "gpsg_binning_view", "gpsg_image_view",
            "gpsg_corr_sampler_forward", "gpsg_corr_sampler_backward", "gpsg_corr_build_pyramid", "gpsg_corr_build_backward",
            "gpsg_corr_lookup_pyramid_forward", "gpsg_corr_lookup_pyramid_backward", "gpsg_raster_geom_bytes",
            "gpsg_raster_binning_bytes", "gpsg_raster_image_bytes", "gpsg_raster_status_ptr",
            "gpsg_rasterize_forward_planned", "gpsg_rasterize_forward_maps", "gpsg_rasterize_forward_maps_planned", "gpsg_rasterize_forward_maps_begin", "gpsg_rasterize_forward_maps_finish",
            "gpsg_rasterize_backward_maps_workspace_bytes",
            "gpsg_rasterize_backward_maps", "gpsg_unproject_forward", "gpsg_unproject_backward", "gpsg_flow2render_workspace_bytes",
            "gpsg_flow2render", "gpsg_l1_ssim_workspace_bytes", "gpsg_l1_ssim_forward",
            "gpsg_l1_ssim_backward", "gpsg_set_corr_build", "gpsg_profile_enable",
            "gpsg_profile_read",
            "gpsg_profile_stage_name"]


def check(rc, what):
    if rc != 0:
        msg = lib.gpsg_last_error()
        raise GpsgError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")


# ---- torch-backed scratch allocator for the gpsg_alloc_fn callbacks ---------------------------
_tls = threading.local()


def _alloc_trampoline(user, nbytes):
    import torch
    try:
        t = torch.empty(int(nbytes), dtype=torch.uint8, device=_tls.device)
        _tls.bufs[int(user or 0)] = t
        return t.data_ptr()
    except Exception:  # never let an exception cross the C boundary
        return None


ALLOC_CB = ALLOC_FN(_alloc_trampoline)


def begin_alloc(device):
    _tls.device = device
    _tls.bufs = {}


def end_alloc():
    bufs = _tls.bufs
    _tls.bufs = {}
    return bufs


lib.gpsg_set_corr_build.restype = _i
lib.gpsg_set_corr_build.argtypes = [_i]


def set_corr_build(kind="tcgen05"):
    """'tcgen05' (default: tensor-core kernels for fp16 volumes when the shape fits) or 'ffma'."""
    check(lib.gpsg_set_corr_build(1 if kind == "ffma" else 0), "gpsg_set_corr_build")


def profile_enable(on=True):
    """True / 1: CUDA events around every stage + launch counts; 2: launch counts only; False: off."""
    check(lib.gpsg_profile_enable(2 if on == 2 else (1 if on else 0)), "gpsg_profile_enable")


def profile_read():
    """{stage: dict(ms=total, calls=n, launches=k)} since the last read (synchronises)."""
    cap = 32
    ms, calls, launches = (C.c_float * cap)(), (C.c_int32 * cap)(), (C.c_int32 * cap)()
    n = lib.gpsg_profile_read(ms, calls, launches, cap)
    if n < 0:
        check(n, "gpsg_profile_read")
    return {lib.gpsg_profile_stage_name(i).decode(): dict(ms=float(ms[i]), calls=int(calls[i]), launches=int(launches[i]))
            for i in range(n)}
