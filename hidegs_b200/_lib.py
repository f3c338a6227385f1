"""ctypes binding of the C-ABI declared in include/hidegs_raster.h.

The product path has no CPU fallback: if libhidegs_b200.so is missing this
module raises at first use instead of silently routing elsewhere.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhidegs_b200.so")

c_float_p = ctypes.c_void_p  # raw device pointers travel as integers
ALLOC_FN = ctypes.CFUNCTYPE(ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t)
# hg_chunk_fn(chunk_ctx, chunk, slot_begin, slot_end, stream)
CHUNK_FN = ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p)


class RasterInputs(ctypes.Structure):
    """struct hg_raster_inputs (include/hidegs_raster.h)."""
    _fields_ = [
        ("P", ctypes.c_int32), ("N", ctypes.c_int32), ("D", ctypes.c_int32), ("M", ctypes.c_int32),
        ("W", ctypes.c_int32), ("H", ctypes.c_int32),
        ("tan_fovx", ctypes.c_float), ("tan_fovy", ctypes.c_float), ("scale_modifier", ctypes.c_float),
        ("prefiltered", ctypes.c_int32), ("render_geo", ctypes.c_int32), ("debug", ctypes.c_int32),
        ("background", ctypes.c_void_p), ("viewmatrix", ctypes.c_void_p), ("projmatrix", ctypes.c_void_p),
        ("campos", ctypes.c_void_p),
        ("indices", ctypes.c_void_p), ("parent_indices", ctypes.c_void_p), ("ts", ctypes.c_void_p),
        ("kids", ctypes.c_void_p),
        ("means3D", ctypes.c_void_p), ("shs", ctypes.c_void_p), ("colors_precomp", ctypes.c_void_p),
        ("all_map", ctypes.c_void_p), ("opacities", ctypes.c_void_p), ("scales", ctypes.c_void_p),
        ("rotations", ctypes.c_void_p), ("cov3D_precomp", ctypes.c_void_p),
    ]


class RasterLayout(ctypes.Structure):
    """struct hg_raster_layout (include/hidegs_raster.h)."""
    _fields_ = [(n, ctypes.c_size_t) for n in (
        "geom_bytes", "depths", "tiles_touched", "point_offsets", "rects", "cov3D", "clamped", "records",
        "tiles", "ctr_stride", "tile_ctr", "tile_lists", "bin_header",
        "image_bytes", "final_T", "n_contrib", "ranges",
        "binning_bytes", "vals", "pairs")]


# Every symbol include/hidegs_raster.h declares (checked by the CPU test-suite).
EXPORTED_SYMBOLS = (
    "hg_raster_layout_query", "hg_raster_forward", "hg_raster_backward_accum_bytes", "hg_raster_backward",
    "hg_raster_backward_chunked", "hg_raster_backward_pose",
    "hg_mark_visible", "hg_raster_debug_keys", "hg_launch_count", "hg_reset_launch_count", "hg_last_error", "hg_version",
    "hg_profile_enable", "hg_profile_collect",
)

STAGES = ("preprocess_fwd", "scan", "binning", "blend_fwd", "accum_zero", "blend_bwd", "preprocess_bwd")

_lib = None


def lib():
    """Load (once) and return the shared library; raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "hidegs_b200: %s is missing. Build it with `python -m hidegs_b200.build` "
            "(there is no CPU or PyTorch fallback for the rasterizer)." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, sz = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t
    L.hg_raster_layout_query.argtypes = [i32, i32, i32, i64, ctypes.POINTER(RasterLayout)]
    L.hg_raster_layout_query.restype = ctypes.c_int
    L.hg_raster_forward.argtypes = [ctypes.POINTER(RasterInputs), ALLOC_FN, vp, ALLOC_FN, vp, ALLOC_FN, vp,
                                    vp, vp, vp, vp, vp, vp, ctypes.POINTER(i32), vp]
    L.hg_raster_forward.restype = ctypes.c_int
    L.hg_raster_backward_accum_bytes.argtypes = [i32]
    L.hg_raster_backward_accum_bytes.restype = sz
    L.hg_raster_backward.argtypes = [ctypes.POINTER(RasterInputs), i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                     vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.hg_raster_backward.restype = ctypes.c_int
    L.hg_raster_backward_chunked.argtypes = L.hg_raster_backward.argtypes[:-1] + [i32, CHUNK_FN, vp, vp, ctypes.c_float, vp, i32, vp]
    L.hg_raster_backward_chunked.restype = ctypes.c_int
    L.hg_raster_backward_pose.argtypes = L.hg_raster_backward_chunked.argtypes[:-1] + [vp, vp]
    L.hg_raster_backward_pose.restype = ctypes.c_int
    L.hg_raster_debug_keys.argtypes = [i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp]
    L.hg_raster_debug_keys.restype = ctypes.c_int
    L.hg_mark_visible.argtypes = [i32, vp, vp, vp, vp, vp]
    L.hg_mark_visible.restype = ctypes.c_int
    L.hg_launch_count.argtypes = []
    L.hg_launch_count.restype = i64
    L.hg_reset_launch_count.argtypes = []
    L.hg_reset_launch_count.restype = None
    L.hg_last_error.argtypes = []
    L.hg_last_error.restype = ctypes.c_char_p
    L.hg_version.argtypes = []
    L.hg_version.restype = ctypes.c_char_p
    L.hg_profile_enable.argtypes = [ctypes.c_int]
    L.hg_profile_enable.restype = None
    L.hg_profile_collect.argtypes = [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64), ctypes.c_int]
    L.hg_profile_collect.restype = ctypes.c_int
    _lib = L
    return L


def check(status, what):
    """Status code -> RuntimeError, mirroring AT_ERROR / CHECK_CUDA of the reference."""
    if status != 0:
        msg = lib().hg_last_error().decode("utf-8", "replace")
        raise RuntimeError("%s failed (status %d): %s" % (what, status, msg))


def layout(P, W, H, R=0):
    out = RasterLayout()
    check(lib().hg_raster_layout_query(P, W, H, R, ctypes.byref(out)), "hg_raster_layout_query")
    return out


def profile_enable(on):
    lib().hg_profile_enable(1 if on else 0)


def profile_collect():
    """{stage: (total_ms, launches)} since the last collect."""
    n = len(STAGES)
    ms = (ctypes.c_double * n)()
    cnt = (ctypes.c_int64 * n)()
    check(lib().hg_profile_collect(ms, cnt, n), "hg_profile_collect")
    return {STAGES[i]: (ms[i], cnt[i]) for i in range(n)}
