"""Drop-in for the reference's `diff_gaussian_rasterization` package.

Public surface kept identical to
submodules/hierarchy-rasterizer/diff_gaussian_rasterization/__init__.py:
`GaussianRasterizationSettings` (18 fields, :157-175), `GaussianRasterizer`
(:178-230), `rasterize_gaussians` (:17-40) and the `_C` operator module.
The autograd function saves the same tensors and returns the same gradient
tuple as `_RasterizeGaussians` (:42-155); the compute is the B200 library.
"""
from typing import NamedTuple

import torch
import torch.nn as nn

from . import _C


def rasterize_gaussians(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                        all_maps, raster_settings):
    return _RasterizeGaussians.apply(means3D, means2D, sh, colors_precomp, opacities, scales, rotations,
                                     cov3Ds_precomp, all_maps, raster_settings)


class _RasterizeGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, all_maps,
                raster_settings):
        rs = raster_settings
        args = (rs.bg, rs.render_indices, rs.parent_indices, rs.interpolation_weights, rs.num_node_kids, means3D,
                colors_precomp, all_maps, opacities, scales, rotations, rs.scale_modifier, cov3Ds_precomp,
                rs.viewmatrix, rs.projmatrix, rs.tanfovx, rs.tanfovy, rs.image_height, rs.image_width, sh,
                rs.sh_degree, rs.campos, rs.prefiltered, rs.render_geo, rs.debug, rs.do_depth)
        (num_rendered, color, radii, out_observe, out_all_map, out_plane_depth, geomBuffer, binningBuffer, imgBuffer,
         invdepths) = _C.rasterize_gaussians(*args)
        ctx.raster_settings = rs
        ctx.num_rendered = num_rendered
        # extension: an SH tensor may carry `_hg_grad_sink = callable -> (tensor, beta)`; its gradient is then
        # accumulated there by the backward kernel and autograd sees None (hidegs_b200.trainer uses it to skip the
        # AccumulateGrad pass over the largest parameter block)
        sink = getattr(sh, "_hg_grad_sink", None)
        ctx.sh_sink = sink if sink is not None and _C.sh_sink_supported(sh, rs.render_indices, rs.parent_indices) else None
        # extension: `means3D._hg_grad_arena = flat fp32 tensor` makes the backward of THIS call write its gradients
        # into that caller-owned arena (e.g. multicast symmetric memory of the data-parallel exchange)
        ctx.grad_arena = getattr(means3D, "_hg_grad_arena", None)
        # extension: `sh._hg_grad_factor = flat fp32 tensor (>= 3 N + 3)` makes the backward of THIS call write the
        # three colour-gradient factors per Gaussian there instead of the SH rows (parallel.FactoredExchange); autograd
        # sees None for the SH gradient
        factor = getattr(sh, "_hg_grad_factor", None)
        ctx.sh_factor = (factor if factor is not None and ctx.sh_sink is None
                         and _C.sh_sink_supported(sh, rs.render_indices, rs.parent_indices) else None)
        ctx.save_for_backward(out_all_map, colors_precomp, all_maps, means3D, scales, rotations, cov3Ds_precomp,
                              radii, sh, opacities, geomBuffer, binningBuffer, imgBuffer)
        ctx.mark_non_differentiable(radii, out_observe)
        return color, radii, out_observe, out_all_map, out_plane_depth, invdepths

    @staticmethod
    def backward(ctx, grad_out_color, _radii, _observe, grad_out_all_map, grad_out_plane_depth, grad_out_depth):
        rs = ctx.raster_settings
        (all_map_pixels, colors_precomp, all_maps, means3D, scales, rotations, cov3Ds_precomp, radii, sh, opacities,
         geomBuffer, binningBuffer, imgBuffer) = ctx.saved_tensors
        H, W = rs.image_height, rs.image_width
        dev = means3D.device
        # autograd hands None for outputs that did not take part in the loss.
        if grad_out_color is None:
            grad_out_color = torch.zeros((3, H, W), dtype=torch.float32, device=dev)
        if grad_out_all_map is None:
            grad_out_all_map = torch.zeros((5, H, W), dtype=torch.float32, device=dev)
        if grad_out_plane_depth is None:
            grad_out_plane_depth = torch.zeros((1, H, W), dtype=torch.float32, device=dev)
        if grad_out_depth is None:
            # the inverse depth took no part in the loss: "absent" (empty) instead of a zero image — the backward then
            # runs its no-depth-gradient kernels (a zero upstream gradient contributes exactly nothing)
            grad_out_depth = torch.empty((0, H, W), dtype=torch.float32, device=dev)
        args = (rs.bg, all_map_pixels, rs.render_indices, rs.parent_indices, rs.interpolation_weights,
                rs.num_node_kids, means3D, radii, colors_precomp, all_maps, opacities, scales, rotations,
                rs.scale_modifier, cov3Ds_precomp, rs.viewmatrix, rs.projmatrix, rs.tanfovx, rs.tanfovy,
                grad_out_color, grad_out_all_map, grad_out_plane_depth, grad_out_depth, sh, rs.sh_degree, rs.campos,
                geomBuffer, ctx.num_rendered, binningBuffer, imgBuffer, rs.render_geo, rs.debug)
        (grad_means2D, grad_colors_precomp, grad_opacities, grad_means3D, grad_cov3Ds_precomp, grad_sh, grad_scales,
         grad_rotations, grad_all_map) = _C.rasterize_gaussians_backward(
            *args, sh_sink=ctx.sh_sink() if ctx.sh_sink is not None else None, grad_arena=ctx.grad_arena,
            sh_factor=ctx.sh_factor, skip_culled_rows=getattr(ctx, "skip_culled_rows", False),
            pose_workspace=getattr(ctx, "pose_workspace", None))
        return (grad_means3D, grad_means2D, grad_sh, grad_colors_precomp, grad_opacities, grad_scales,
                grad_rotations, grad_cov3Ds_precomp, grad_all_map, None)


class GaussianRasterizationSettings(NamedTuple):
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool
    debug: bool
    render_indices: torch.Tensor
    parent_indices: torch.Tensor
    interpolation_weights: torch.Tensor
    num_node_kids: torch.Tensor
    do_depth: bool
    render_geo: bool


class GaussianRasterizer(nn.Module):
    def __init__(self, raster_settings):
        super().__init__()
        self.raster_settings = raster_settings

    def markVisible(self, positions):
        with torch.no_grad():
            rs = self.raster_settings
            return _C.mark_visible(positions, rs.viewmatrix, rs.projmatrix)

    def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None,
                cov3D_precomp=None, all_map=None):
        rs = self.raster_settings
        if (shs is None and colors_precomp is None) or (shs is not None and colors_precomp is not None):
            raise Exception('Please provide excatly one of either SHs or precomputed colors!')
        if ((scales is None or rotations is None) and cov3D_precomp is None) or \
                ((scales is not None or rotations is not None) and cov3D_precomp is not None):
            raise Exception('Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!')
        empty = torch.Tensor([])
        shs = empty if shs is None else shs
        colors_precomp = empty if colors_precomp is None else colors_precomp
        scales = empty if scales is None else scales
        rotations = empty if rotations is None else rotations
        cov3D_precomp = empty if cov3D_precomp is None else cov3D_precomp
        all_map = empty if all_map is None else all_map
        return rasterize_gaussians(means3D, means2D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp,
                                   all_map, rs)
