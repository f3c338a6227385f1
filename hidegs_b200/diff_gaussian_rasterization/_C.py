"""`_C` operator module of the drop-in rasterizer package.

Same operator names, argument order and return tuples as the reference's pybind module
(submodules/hierarchy-rasterizer/ext.cpp:15-18, rasterize_points.h:18-80).  The operators live in the thin torch C++
extension `_hgC` (hidegs_b200/csrc_ext/raster_ext.cpp: shape checks, output / scratch tensors, the current CUDA stream,
status -> exception) over the C-ABI of include/hidegs_raster.h; this module only re-exports them and unpacks the
optional per-call extensions of the backward.  There is no module-level state and no fallback: if the extension is not
built, importing this module fails.
"""
import importlib
import os

import torch  # noqa: F401  (torch's shared libraries must be loaded before the extension)

_HERE = os.path.dirname(os.path.abspath(__file__))
try:
    _hgC = importlib.import_module(__package__ + "._hgC")
except ImportError as e:  # pragma: no cover
    raise ImportError("hidegs_b200: the rasterizer's torch extension (%s/_hgC*.so) is missing or does not load: %s.  "
                      "Build it with `python -m hidegs_b200.build` (there is no CPU or PyTorch fallback)." % (_HERE, e))

rasterize_gaussians = _hgC.rasterize_gaussians
mark_visible = _hgC.mark_visible
sh_sink_supported = _hgC.sh_sink_supported


def rasterize_gaussians_backward(*args, sh_sink=None, grad_arena=None, chunk_hook=None, sh_factor=None,
                                 skip_culled_rows=False, pose_workspace=None):
    """RasterizeGaussiansBackwardCUDA (rasterize_points.cu:149-279), positional arguments as in the reference.

    Per-call extensions (keyword only; nothing is remembered between calls):
      sh_sink    `(tensor [N, M, 3], beta)`: the SH gradient is accumulated into the tensor (sink = beta * sink + grad)
                 and the returned dL_dsh is None (needs `sh_sink_supported`)
      grad_arena flat fp32 tensor the gradients are written into instead of a fresh allocation (the returned gradients
                 are views of it; e.g. multicast symmetric memory for the in-fabric gradient exchange)
      chunk_hook `(n_chunks, fn)`: the per-Gaussian part is issued in `n_chunks` slot ranges and
                 `fn(chunk, slot_begin, slot_end)` is called right after each range has been queued on the current
                 stream (rows slot_begin..slot_end-1 of every gradient are final once that kernel completes)
      sh_factor  flat fp32 tensor of >= 3 N + 3 elements: instead of the [N, M, 3] SH gradient rows the call writes the
                 three clamp-masked colour gradients per Gaussian (the rows are their outer product with the SH basis
                 at the view direction) followed by the camera centre; dL_dsh is returned as None
                 (parallel.FactoredExchange ships these 12 bytes per Gaussian instead of 192)
      skip_culled_rows  the gradient rows of culled Gaussians (radii <= 0) are left UNWRITTEN instead of zero-filled:
                 only for a consumer that masks by `radii` (the trainer's fused prologue backward)
      pose_workspace  tensor of >= hg_camera_pose_workspace_bytes(N) bytes: the call also sums the camera side of the
                 gradient there (hg_raster_backward_pose; the camera pose refinement of the training step)."""
    sink, beta = sh_sink if sh_sink is not None else (None, 0.0)
    n_chunks, fn = chunk_hook if chunk_hook is not None else (0, None)
    return _hgC.rasterize_gaussians_backward(*args, sh_sink=sink, sh_beta=float(beta), grad_arena=grad_arena,
                                             n_chunks=int(n_chunks), chunk_hook=fn, sh_factor=sh_factor,
                                             skip_culled_rows=bool(skip_culled_rows), pose_workspace=pose_workspace)
