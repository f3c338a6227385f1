"""ctypes prototypes of include/hidegs_geometry.h (same shared library as the rasterizer)."""
import ctypes

from . import _lib

EXPORTED_SYMBOLS = (
    "hg_geometry_all_map", "hg_geometry_all_map_backward", "hg_activate_params", "hg_activate_params_backward", "hg_prologue_backward", "hg_depth_normal", "hg_depth_normal_backward",
    "hg_normal_consistency_workspace_bytes", "hg_normal_consistency_loss", "hg_adam_step", "hg_densification_stats", "hg_expand_to_size_workspace_bytes", "hg_expand_to_size",
    "hg_interpolation_weights", "hg_hier_interpolate", "hg_hier_interpolate_backward",
    "hg_dist2_knn3_workspace_bytes", "hg_dist2_knn3", "hg_densify_workspace_bytes", "hg_densify_plan", "hg_densify_apply",
    "hg_reset_opacity",
)


class Intrinsics(ctypes.Structure):
    """struct hg_intrinsics."""
    _fields_ = [("fx", ctypes.c_float), ("fy", ctypes.c_float), ("cx", ctypes.c_float), ("cy", ctypes.c_float)]


_ready = False


def lib():
    global _ready
    L = _lib.lib()
    if _ready:
        return L
    vp, i32, i64, sz, f32, ci = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t, ctypes.c_float, ctypes.c_int
    f64 = ctypes.c_double
    p64 = ctypes.POINTER(i64)
    proto = {
        "hg_geometry_all_map": (ci, [vp, vp, vp, vp, vp, i64, vp, vp]),
        "hg_geometry_all_map_backward": (ci, [vp, vp, vp, vp, vp, i64, vp, vp, vp, vp]),
        "hg_activate_params": (ci, [vp, vp, vp, i64, vp, vp, vp, vp]),
        "hg_activate_params_backward": (ci, [vp, vp, vp, i64, i32, vp, vp, vp, vp, vp, f32, vp, vp, vp, vp, vp, vp]),
        "hg_prologue_backward": (ci, [vp, vp, vp, vp, i64, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, f32, vp, vp, vp, vp,
                                      vp, vp]),
        "hg_depth_normal": (ci, [vp, vp, i32, i32, Intrinsics, vp, vp]),
        "hg_depth_normal_backward": (ci, [vp, vp, vp, i32, i32, Intrinsics, vp, vp]),
        "hg_normal_consistency_workspace_bytes": (sz, [i32, i32]),
        "hg_normal_consistency_loss": (ci, [vp, vp, vp, i32, i32, Intrinsics, f32, vp, vp, vp, vp, vp]),
        "hg_adam_step": (ci, [vp, vp, vp, vp, i64, i32, vp, vp, i64, f64, f64, f64, f64, i32, f32, i32, f64, vp]),
        "hg_densification_stats": (ci, [vp, vp, i64, vp, vp, vp, vp]),
        "hg_expand_to_size_workspace_bytes": (sz, [i32]),
        "hg_expand_to_size": (ci, [vp, vp, i32, f32, vp, i32, vp, vp, vp, vp, vp, ctypes.POINTER(i32), vp]),
        "hg_interpolation_weights": (ci, [vp, i32, f32, vp, vp, f32, f32, f32, vp, vp, vp]),
        "hg_hier_interpolate": (ci, [vp, vp, vp, vp, vp, i64, i32, vp, vp, vp, i64, i64, vp, vp, vp, vp, vp, vp]),
        "hg_hier_interpolate_backward": (ci, [vp, i64, i32, vp, vp, vp, i64, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
        "hg_dist2_knn3_workspace_bytes": (sz, [i64]),
        "hg_dist2_knn3": (ci, [vp, i64, vp, vp, vp]),
        "hg_densify_workspace_bytes": (sz, [i64]),
        "hg_densify_plan": (ci, [vp, p64, i64, vp, i32, f64, f64, f64, f64, f64, vp, p64, p64, p64, p64, vp]),
        "hg_densify_apply": (ci, [vp, vp, vp, p64, i64, vp, vp, vp, p64, i64, vp, ctypes.c_uint64, vp, vp]),
        "hg_reset_opacity": (ci, [vp, vp, vp, i64, vp]),
    }
    for name, (res, args) in proto.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _ready = True
    return L
