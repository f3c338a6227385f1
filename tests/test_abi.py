"""CPU checks of the drop-in boundary: the C-ABI library loads, exports every
symbol include/hidegs_raster.h declares, and rejects bad arguments before any
CUDA work (mirrors the reference's AT_ERROR / Exception paths,
rasterize_points.cu:64-66, diff_gaussian_rasterization/__init__.py:198-202)."""
import ctypes
import os
import re

import pytest
import torch

from hidegs_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols(path):
    text = open(path).read()
    return sorted(set(re.findall(r"HG_API[^;(]*?\b(hg_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = _lib.lib()
    names = []
    for h in sorted(os.listdir(os.path.join(ROOT, "include"))):
        if h.endswith(".h"):
            names += header_symbols(os.path.join(ROOT, "include", h))
    assert "hg_raster_forward" in names and "hg_raster_backward" in names
    for n in names:
        assert hasattr(lib, n), "symbol %s declared in include/ but not exported" % n
    assert set(_lib.EXPORTED_SYMBOLS) <= set(names)
    assert b"sm_100a" in lib.hg_version()


def test_layout_query_is_consistent():
    L = _lib.layout(1000, 1920, 1080, 5000)
    offs = [L.depths, L.tiles_touched, L.point_offsets, L.rects, L.cov3D, L.clamped, L.records, L.tile_ctr, L.tile_lists,
            L.bin_header]
    assert offs == sorted(offs) and all(o % 256 == 0 for o in offs)
    assert L.records - L.clamped >= 1000 and L.tile_ctr >= L.records + 64 * 1000
    assert L.tiles == 120 * 68 and L.tile_lists - L.tile_ctr >= 4 * L.ctr_stride * L.tiles
    assert L.bin_header - L.tile_lists >= 12 * L.tiles and L.geom_bytes >= L.bin_header + 64
    assert L.ranges + 8 * 120 * 68 <= L.image_bytes
    # the sorted list comes first in the binning block (all the backward reads), the bucketed pairs behind it
    assert L.vals == 0 and L.pairs >= 4 * 5000 and L.binning_bytes >= L.pairs + 8 * 5000
    # binning layout only depends on R, geometry layout on P and the tile grid
    L2 = _lib.layout(1000, 1920, 1080, 0)
    assert L2.records == L.records and L2.pairs == 0


def test_layout_query_rejects_bad_sizes():
    out = _lib.RasterLayout()
    assert _lib.lib().hg_raster_layout_query(-1, 16, 16, 0, ctypes.byref(out)) == 1
    assert _lib.lib().hg_raster_layout_query(1, 0, 16, 0, ctypes.byref(out)) == 1
    assert b"bad argument" in _lib.lib().hg_last_error()


def _dummy_alloc():
    return _lib.ALLOC_FN(lambda ctx, n: None)


def test_forward_validates_before_touching_the_gpu():
    lib = _lib.lib()
    s = _lib.RasterInputs()
    s.P, s.N, s.W, s.H = 4, 4, 32, 32
    cb = _dummy_alloc()
    r = ctypes.c_int32(0)
    # mandatory pointers missing
    rc = lib.hg_raster_forward(ctypes.byref(s), cb, None, cb, None, cb, None, 1, None, 1, 1, 1, 1, ctypes.byref(r), None)
    assert rc == 1 and b"mandatory" in lib.hg_last_error()
    # both SH and precomputed colours (fake non-null pointers are never dereferenced)
    for f in ("means3D", "opacities", "background", "viewmatrix", "projmatrix", "campos", "shs", "colors_precomp"):
        setattr(s, f, 256)
    s.M, s.D = 16, 3
    rc = lib.hg_raster_forward(ctypes.byref(s), cb, None, cb, None, cb, None, 1, None, 1, 1, 1, 1, ctypes.byref(r), None)
    assert rc == 1 and b"excatly one of either SHs" in lib.hg_last_error()
    s.colors_precomp = None
    rc = lib.hg_raster_forward(ctypes.byref(s), cb, None, cb, None, cb, None, 1, None, 1, 1, 1, 1, ctypes.byref(r), None)
    assert rc == 1 and b"scale/rotation pair" in lib.hg_last_error()
    s.scales, s.rotations = 256, 256
    s.D = 4  # degree 4 does not fit 16 coefficients
    rc = lib.hg_raster_forward(ctypes.byref(s), cb, None, cb, None, cb, None, 1, None, 1, 1, 1, 1, ctypes.byref(r), None)
    assert rc == 1 and b"SH degree" in lib.hg_last_error()
    # rotations are read as float4: a pointer off a 16-byte boundary is refused (one float into a row, or 8 bytes)
    s.D = 3
    for bad in (260, 264):
        s.rotations = bad
        rc = lib.hg_raster_forward(ctypes.byref(s), cb, None, cb, None, cb, None, 1, None, 1, 1, 1, 1, ctypes.byref(r),
                                   None)
        assert rc == 1 and b"rotations must be 16-byte aligned" in lib.hg_last_error()


def test_backward_validates_before_touching_the_gpu():
    lib = _lib.lib()
    s = _lib.RasterInputs()
    s.P, s.N, s.W, s.H = 4, 4, 32, 32
    bwd = lambda: lib.hg_raster_backward(ctypes.byref(s), 0, *([None] * 21), None)  # noqa: E731
    # every pointer is checked before the first CUDA call (fake non-null pointers are never dereferenced)
    assert bwd() == 1 and b"mandatory pointer" in lib.hg_last_error()
    for f in ("means3D", "opacities", "background", "viewmatrix", "projmatrix", "campos", "shs", "scales"):
        setattr(s, f, 256)
    s.M, s.D = 16, 3
    assert bwd() == 1 and b"scale/rotation pair" in lib.hg_last_error()
    s.rotations = 260
    assert bwd() == 1 and b"rotations must be 16-byte aligned" in lib.hg_last_error()
    # the same arguments with an aligned rotations pointer pass validate() and stop at the missing outputs
    s.rotations = 272
    assert bwd() == 1 and b"hg_raster_backward: a mandatory pointer is NULL" in lib.hg_last_error()
    s.rotations = 264
    rc = lib.hg_raster_backward_chunked(ctypes.byref(s), 0, *([None] * 21), 1, _lib.CHUNK_FN(0), None, None, 0.0, None,
                                        0, None)
    assert rc == 1 and b"rotations must be 16-byte aligned" in lib.hg_last_error()


def test_python_api_surface_matches_reference():
    import diff_gaussian_rasterization as d
    assert d.GaussianRasterizationSettings._fields == (
        "image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier", "viewmatrix", "projmatrix",
        "sh_degree", "campos", "prefiltered", "debug", "render_indices", "parent_indices", "interpolation_weights",
        "num_node_kids", "do_depth", "render_geo")
    assert hasattr(d._C, "rasterize_gaussians") and hasattr(d._C, "rasterize_gaussians_backward")
    rs = d.GaussianRasterizationSettings(*([None] * 18))
    r = d.GaussianRasterizer(rs)
    x = torch.zeros(2, 3)
    with pytest.raises(Exception, match="excatly one of either SHs"):
        r(means3D=x, means2D=x, opacities=x[:, :1])
    with pytest.raises(Exception, match="scale/rotation pair"):
        r(means3D=x, means2D=x, opacities=x[:, :1], shs=torch.zeros(2, 16, 3))


def test_no_cpu_fallback():
    """The product path must fail loudly on CPU tensors instead of falling back."""
    import diff_gaussian_rasterization as d
    e_i, e_f = torch.empty(0, dtype=torch.int32), torch.empty(0)
    with pytest.raises(RuntimeError, match="no CPU path"):
        d._C.rasterize_gaussians(torch.zeros(3), e_i, e_i, e_f, e_i, torch.zeros(2, 3), e_f, e_f, torch.zeros(2, 1),
                                 torch.ones(2, 3), torch.ones(2, 4), 1.0, e_f, torch.eye(4), torch.eye(4), 1.0, 1.0,
                                 16, 16, torch.zeros(2, 16, 3), 3, torch.zeros(3), False, True, False, True)


def test_product_package_never_imports_the_oracle():
    """Nothing under hidegs_b200/ may reference oracle/ (the oracle is test infrastructure)."""
    pkg = os.path.join(ROOT, "hidegs_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert "raster_oracle" not in text and "from oracle" not in text and "import oracle" not in text, f


def test_install_routes_reference_imports():
    """hidegs_b200.install(): the reference's import lines resolve to the drop-ins."""
    import importlib
    import sys
    import hidegs_b200
    saved = {k: sys.modules.get(k) for k in ("diff_gaussian_rasterization", "diff_gaussian_rasterization._C", "simple_knn",
                                            "simple_knn._C")}
    try:
        done = hidegs_b200.install(patch_reference_modules=False)
        assert "simple_knn._C" in done
        from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer, _C  # noqa: F401
        from simple_knn._C import distCUDA2
        assert _C is importlib.import_module("hidegs_b200.diff_gaussian_rasterization._C")
        assert distCUDA2 is importlib.import_module("hidegs_b200.simple_knn._C").distCUDA2
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_drop_in_signatures_match_reference():
    """Same parameter names / defaults as the reference's Python functions (SURVEY.md §8(b))."""
    import inspect
    from hidegs_b200 import gaussian_renderer as gr, loss_utils as lu
    from hidegs_b200.frequency_regularization import frequency_regularization_pyramid_scale as f
    assert list(inspect.signature(gr.render).parameters) == [
        "viewpoint_camera", "pc", "pipe", "bg_color", "scaling_modifier", "override_color", "indices", "use_trained_exp",
        "return_plane", "return_depth_normal"]
    assert list(inspect.signature(gr.render_post).parameters) == [
        "viewpoint_camera", "pc", "pipe", "bg_color", "scaling_modifier", "override_color", "render_indices",
        "parent_indices", "interpolation_weights", "num_node_kids", "interp_python", "use_trained_exp"]
    assert list(inspect.signature(gr.render_normal).parameters) == ["viewpoint_cam", "depth", "offset", "normal", "scale"]
    names = list(inspect.signature(f).parameters)
    assert names[:15] == [
        "rendered_image", "gt_image", "gaussians", "scene", "viewpoint_cam", "visibility_filter", "iteration", "lambda_freq",
        "lambda_scale", "num_levels", "high_freq_thresh", "save_results", "save_dir", "warmup_iterations", "debug"]
    # one optional trailing extension (per-camera ground-truth cache), inert by default
    assert names[15:] == ["gt_cache"] and inspect.signature(f).parameters["gt_cache"].default is None
    sig = inspect.signature(f).parameters
    assert (sig["lambda_freq"].default, sig["lambda_scale"].default, sig["num_levels"].default,
            sig["high_freq_thresh"].default, sig["warmup_iterations"].default) == (0.001, 0.005, 3, 0.2, 1000)
    assert list(inspect.signature(lu.ssim).parameters) == ["img1", "img2", "window_size", "size_average"]
    assert list(inspect.signature(lu.get_img_grad_weight).parameters) == ["img", "beta"]
    assert list(inspect.signature(lu.lncc).parameters) == ["ref", "nea"]


def test_torch_extension_surface_and_no_cpu_path():
    """The rasterizer's `_C` is the thin torch C++ extension (csrc_ext/raster_ext.cpp) over the C-ABI: same operator
    names as the reference's pybind module (ext.cpp:15-18) + mark_visible, no module-level mutable state in the Python
    shim, CPU tensors rejected (no fallback)."""
    import inspect
    import pytest
    import torch
    from hidegs_b200.diff_gaussian_rasterization import _C
    for name in ("rasterize_gaussians", "rasterize_gaussians_backward", "mark_visible", "sh_sink_supported"):
        assert callable(getattr(_C, name)), name
    assert type(_C.rasterize_gaussians).__name__ == "builtin_function_or_method"  # bound straight from the extension
    assert _C._hgC.__file__.endswith(".so") and "hidegs_b200" in _C._hgC.__file__
    src = inspect.getsource(_C)
    assert "global " not in src and "ctypes" not in src
    e_i, e_f = torch.empty(0, dtype=torch.int32), torch.empty(0)
    with pytest.raises(RuntimeError, match="no CPU path"):
        _C.rasterize_gaussians(torch.zeros(3), e_i, e_i, e_f, e_i, torch.zeros(4, 3), e_f, e_f, torch.zeros(4, 1),
                               torch.ones(4, 3), torch.ones(4, 4), 1.0, e_f, torch.eye(4), torch.eye(4), 1.0, 1.0, 16, 16,
                               torch.zeros(4, 16, 3), 3, torch.zeros(3), False, True, False, True)
    with pytest.raises(RuntimeError, match="num_points, 3"):
        _C.rasterize_gaussians(torch.zeros(3), e_i, e_i, e_f, e_i, torch.zeros(4, 2), e_f, e_f, torch.zeros(4, 1),
                               torch.ones(4, 3), torch.ones(4, 4), 1.0, e_f, torch.eye(4), torch.eye(4), 1.0, 1.0, 16, 16,
                               torch.zeros(4, 16, 3), 3, torch.zeros(3), False, True, False, True)
