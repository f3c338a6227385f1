"""View-sharded training step of HiDeGS on the B200 hot path (SURVEY.md §3.1, §8(e), BASELINE.json configs[3] / [4]).

The reference ships no train.py (README.md:175); the step below is the one its pieces compose into
(gaussian_renderer.render -> l1 / ssim / frequency_regularization_pyramid_scale / single-view normal term ->
backward -> OurAdam step), with the weights of arguments/__init__.py:100-135:

    loss = (1 - lambda_dssim) * l1_loss(image, gt) + lambda_dssim * (1 - ssim(image, gt))
         + frequency_regularization_pyramid_scale(image, gt, gaussians, scene, cam, visibility_filter, iteration)[0]
         + single_view_weight * mean((1 - get_img_grad_weight(gt)).clamp(0, 1) ** 2 * |depth_normal - rendered_normal|.sum(0))

Data parallelism: Gaussians are replicated, the views of a step are split `views[rank::world]`, every rank accumulates
the gradients of its views in ONE flat fp32 arena (59 floats per Gaussian: xyz 3 | features 48 | opacity 1 | scaling 3 |
rotation 4, SoA by group), the arena is all-reduced once per step (NCCL over NVLink) and the fused Adam kernel consumes
it with grad_scale = 1 / views.  Parameters live in a matching flat arena, so the optimiser is 6 launches per step.

A view runs without autograd (`ViewShardedTrainer.view_step_direct`: the forward / backward bodies of the same Functions
on a hand-written tape).  Everything per Gaussian is sparse in the view: the rasterizer's backward leaves the gradient rows
of culled Gaussians unwritten (HG_BWD_SKIP_CULLED_ROWS) and ONE kernel (`hg_prologue_backward`) takes the rendered rows
from the rasterizer's gradients to the raw-parameter arena (all_map backward, scale-regulariser gradient, activation
chain rule, accumulation); the activations themselves are computed once per optimiser step.
"""
import ctypes
import math

import torch
import torch.distributed as dist

from . import gaussian_renderer as gr
from . import loss_utils as lu
from ._geometry_lib import lib as _G
from . import _lib
from . import parallel
from .frequency_regularization import (GroundTruthCache, _FreqLoss, _FreqTotal, _ScaleReg, detect_true_high_frequency_regions,
                                       frequency_regularization_pyramid_scale)
from .diff_gaussian_rasterization import _RasterizeGaussians

GROUPS = (("xyz", 3), ("features", 48), ("opacity", 1), ("scaling", 3), ("rotation", 4))


class PipelineParams:
    """arguments/__init__.py PipelineParams defaults."""
    convert_SHs_python = False
    compute_cov3D_python = False
    debug = False


class OptimizationParams:
    """The entries of arguments/__init__.py:83-135 the training step reads."""
    position_lr_init = 0.00016
    feature_lr = 0.0025
    opacity_lr = 0.05
    scaling_lr = 0.005
    rotation_lr = 0.001
    lambda_dssim = 0.2
    single_view_weight = 0.015
    lambda_freq = 0.001
    lambda_scale = 0.005
    freq_warmup_iterations = 1000
    # adaptive density control (ViewShardedTrainer(densify=True)); intervals count optimiser steps.  The reference ships
    # no train.py, so these are not read from it: intervals, percent_dense and min_opacity are graphdeco 3DGS's
    # (arguments/__init__.py, train.py), the gradient threshold is hierarchical-3DGS's, whose statistic is the same
    # running maximum of the screen-space gradient norm this build accumulates (not a mean)
    densify_from_iter = 500
    densify_until_iter = 15_000
    densification_interval = 100
    opacity_reset_interval = 3000
    densify_grad_threshold = 0.015
    percent_dense = 0.01
    min_opacity = 0.005
    # per-image exposure (ViewShardedTrainer(train_exposure=True)): Adam with eps 1e-8 over the whole table, lr
    # get_expon_lr_func(exposure_lr_init, exposure_lr_final, exposure_lr_delay_steps, exposure_lr_delay_mult,
    # max_steps=iterations) at the trainer's iteration.  The reference ships no train.py; these are hierarchical-3DGS's
    # arguments/__init__.py values as recalled, not read from or checked against a reference tree
    exposure_lr_init = 0.01
    exposure_lr_final = 0.0001
    exposure_lr_delay_steps = 5000
    exposure_lr_delay_mult = 0.001
    iterations = 30_000
    # monocular inverse-depth supervision (ViewShardedTrainer(depth_regularization=True)): weight
    # get_expon_lr_func(depth_l1_weight_init, depth_l1_weight_final, max_steps=iterations) at the trainer's iteration;
    # graphdeco 3DGS's arguments/__init__.py values as recalled, not checked against a reference tree
    depth_l1_weight_init = 1.0
    depth_l1_weight_final = 0.01
    # camera pose refinement (ViewShardedTrainer(train_poses=True)): Adam with eps 1e-8 over the whole [n, 8] table at
    # constant rates, the translation one multiplied by spatial_lr_scale as position_lr_init is.  Nothing upstream
    # defines these: they are this build's choice (translation in scene units, rotation in radians, per step)
    pose_lr_translation = 0.0001
    pose_lr_rotation = 0.0001
    # 3DGS-MCMC densification (ViewShardedTrainer(mcmc=True); DESIGN.md §3 "MCMC densification"): refine (relocate,
    # then grow) every mcmc_refine_interval steps in (mcmc_refine_from_iter, mcmc_refine_until_iter), position noise
    # every step.  The 3DGS-MCMC paper's and gsplat MCMCStrategy's values as recalled, not checked against a reference
    mcmc_refine_from_iter = 500
    mcmc_refine_until_iter = 25_000
    mcmc_refine_interval = 100
    mcmc_min_opacity = 0.005
    mcmc_grow_factor = 1.05
    mcmc_noise_lr = 5e5
    mcmc_opacity_reg = 0.01
    mcmc_scale_reg = 0.01
    # the position learning-rate schedule of graphdeco 3DGS (xyz_scheduler_args), used in MCMC mode only:
    # get_expon_lr_func(position_lr_init * s, position_lr_final * s, lr_delay_mult=position_lr_delay_mult,
    # max_steps=position_lr_max_steps), s = spatial_lr_scale.  Without MCMC the xyz rate stays position_lr_init * s
    position_lr_final = 0.0000016
    position_lr_delay_mult = 0.01
    position_lr_max_steps = 30_000


class _ActivateParams(torch.autograd.Function):
    """get_scaling / get_rotation / get_opacity of the model (exp / normalize / sigmoid) in ONE kernel, and — in the
    backward — their chain rule fused with the accumulation of all five parameter gradients into the flat gradient
    arena (dst = beta * dst + grad).  Replaces ~6 elementwise launches forward and ~25 backward (activation backward +
    autograd's AccumulateGrad of five leaves) per view.  The leaves receive no autograd gradient (None): their `.grad`
    are views of the arena this Function writes."""

    @staticmethod
    def forward(ctx, xyz, features, opacity_raw, scaling_raw, rotation_raw, owner):
        N = xyz.size(0)
        dev = xyz.device
        act = torch.empty(N * 8, dtype=torch.float32, device=dev)  # rotation first: float4 rows stay 16-byte aligned
        rotation, scaling, opacity = act[:4 * N].view(N, 4), act[4 * N:7 * N].view(N, 3), act[7 * N:].view(N, 1)
        with torch.cuda.device(dev):
            rc = _G().hg_activate_params(scaling_raw.data_ptr(), rotation_raw.data_ptr(), opacity_raw.data_ptr(), N,
                                         scaling.data_ptr(), rotation.data_ptr(), opacity.data_ptr(),
                                         torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, "activate_params")
        ctx.owner = owner
        ctx.set_materialize_grads(False)  # a missing gradient stays None (the SH gradient may arrive through the sink)
        return xyz.view_as(xyz), features.view_as(features), opacity, scaling, rotation

    @staticmethod
    def backward(ctx, g_xyz, g_feat, g_op, g_sc, g_rot):
        p = ctx.owner
        N = p.N

        def ptr(t):
            return t.contiguous().data_ptr() if t is not None else None
        if g_feat is None and not p._sink_used:  # no feature gradient at all in this view: accumulate zeros
            g_feat = torch.zeros((N, 16, 3), dtype=torch.float32, device=p.param_arena.device) if not p._grad_dirty else None
        missing = [i for i, t in enumerate((g_xyz, g_op, g_sc, g_rot)) if t is None]
        if missing:  # (rare: an output that took no part in the loss)
            z = lambda w: torch.zeros((N, w), dtype=torch.float32, device=p.param_arena.device)  # noqa: E731
            g_xyz = z(3) if g_xyz is None else g_xyz
            g_op = z(1) if g_op is None else g_op
            g_sc = z(3) if g_sc is None else g_sc
            g_rot = z(4) if g_rot is None else g_rot
        if g_feat is not None and p._sink_used:
            # the features were ALSO used outside the rasterizer in this view: that gradient comes on top of what the
            # rasterizer's backward has just accumulated through the sink (never with beta = 0)
            p.grad_arena[p.slices["features"]].add_(g_feat.reshape(-1))
            g_feat = None
        keep = [t.contiguous() if t is not None else None for t in (g_xyz, g_feat, g_op, g_sc, g_rot)]
        d = {k: p.grad_arena[p.slices[k]] for k in ("xyz", "features", "opacity", "scaling", "rotation")}
        with torch.cuda.device(p.param_arena.device):
            rc = _G().hg_activate_params_backward(
                p._scaling.data_ptr(), p._rotation.data_ptr(), p._opacity.data_ptr(), N, 48,
                ptr(keep[0]), ptr(keep[1]), ptr(keep[2]), ptr(keep[3]), ptr(keep[4]), 1.0 if p._grad_dirty else 0.0,
                d["xyz"].data_ptr(), d["features"].data_ptr(), d["opacity"].data_ptr(), d["scaling"].data_ptr(),
                d["rotation"].data_ptr(), torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, "activate_params_backward")
        p._grad_dirty = True
        p._sink_used = False
        return None, None, None, None, None, None


def morton_order(xyz):
    """Permutation that sorts points along a 30-bit Morton (Z-order) curve: 10 bits per axis, all axes quantised with the
    SAME scale (the largest extent), so a thin slab interleaves mostly its two long axes."""
    xyz = xyz.detach().float().cpu()
    lo = xyz.min(0).values
    extent = float((xyz.max(0).values - lo).max().clamp_min(1e-30))
    q = ((xyz - lo) / extent * 1023.0).long().clamp_(0, 1023)

    def spread(v):  # insert two zero bits between the 10 bits of v
        v = (v | (v << 16)) & 0x030000FF
        v = (v | (v << 8)) & 0x0300F00F
        v = (v | (v << 4)) & 0x030C30C3
        return (v | (v << 2)) & 0x09249249
    code = spread(q[:, 0]) | (spread(q[:, 1]) << 1) | (spread(q[:, 2]) << 2)
    return torch.argsort(code, stable=True)


def arena_layout(N):
    """({group: first float}, total floats) of the parameter / gradient / moment arenas of N Gaussians: the GROUPS in
    order, every group starting on a multiple of 4 floats (16 bytes) — the fused kernels move rotation / feature rows
    as float4 and the in-fabric exchange works on 16-byte units, for ANY Gaussian count (pad floats stay zero)."""
    starts, total = {}, 0
    for name, w in GROUPS:
        starts[name] = total
        total += (N * w + 3) // 4 * 4
    return starts, total


def densify_arenas(param_arena, exp_avg, exp_avg_sq, N, accum, max_grad, min_opacity, extent, max_screen_size=None,
                   seed=0, samples=None, percent_dense=0.01, skybox_points=0):
    """graphdeco 3DGS densify_and_clone + densify_and_split + prune over flat arenas of N rows (arena_layout; DESIGN.md
    §3 "Densify and prune"): returns (new parameter arena, new exp_avg, new exp_avg_sq, counts) with counts =
    dict(kept, cloned, split, pruned, n): original rows kept, rows cloned, rows split, rows pruned (originals, clones
    and children), n = N'.  `accum` [N] fp32: the max-form screen-space gradient
    statistic.  Children are drawn from Philox4x32-10 keyed by `seed` (the same bits on every rank), or taken from
    `samples` [2 |split|, 3] (torch.normal(0, stds.repeat(2, 1)) of the reference).  One host synchronisation.
    Raises ValueError when nothing would be left (N' = 0)."""
    dev = param_arena.device
    L = _G()
    st = torch.cuda.current_stream(dev).cuda_stream
    ws = torch.empty(int(L.hg_densify_workspace_bytes(N)), dtype=torch.uint8, device=dev)
    starts, _total = arena_layout(N)
    off = (ctypes.c_int64 * 5)(*[starts[n] for n, _ in GROUPS])
    kept, cloned, split, new_n = (ctypes.c_int64() for _ in range(4))
    accum = accum.contiguous()
    with torch.cuda.device(dev):
        rc = L.hg_densify_plan(param_arena.data_ptr(), off, N, accum.data_ptr(), int(skybox_points), float(max_grad),
                               float(min_opacity), float(extent), float(max_screen_size or 0.0), float(percent_dense),
                               ws.data_ptr(), ctypes.byref(kept), ctypes.byref(cloned), ctypes.byref(split),
                               ctypes.byref(new_n), st)
    _lib.check(rc, "densify_plan")
    n2 = new_n.value
    counts = dict(kept=kept.value, cloned=cloned.value, split=split.value, pruned=N + cloned.value + split.value - n2,
                  n=n2)
    if n2 == 0:
        raise ValueError("densify_and_prune would leave no Gaussians (%s)" % counts)
    starts2, total2 = arena_layout(n2)
    off2 = (ctypes.c_int64 * 5)(*[starts2[n] for n, _ in GROUPS])
    # every float of the new arenas (pads included) is written by the kernel
    new = [torch.empty(total2, dtype=torch.float32, device=dev) for _ in range(3)]
    if samples is not None:
        samples = samples.to(device=dev, dtype=torch.float32).contiguous()
        if tuple(samples.shape) != (2 * split.value, 3):
            raise ValueError("samples must be [2 * %d, 3], got %s" % (split.value, tuple(samples.shape)))
    with torch.cuda.device(dev):
        rc = L.hg_densify_apply(param_arena.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), off, N,
                                new[0].data_ptr(), new[1].data_ptr(), new[2].data_ptr(), off2, n2,
                                samples.data_ptr() if samples is not None and samples.numel() else None,
                                int(seed) & 0xFFFFFFFFFFFFFFFF, ws.data_ptr(), st)
    _lib.check(rc, "densify_apply")
    return new[0], new[1], new[2], counts


# ---- 3DGS-MCMC densification (DESIGN.md §3 "MCMC densification"; include/hidegs_geometry.h hg_mcmc_*) ------------------
def mcmc_refines(it, opt):
    """Whether step `it` refines (relocate, then grow) after its optimiser update: refine_from < it < refine_until and
    it a multiple of refine_interval."""
    return opt.mcmc_refine_from_iter < it < opt.mcmc_refine_until_iter and it % opt.mcmc_refine_interval == 0


def mcmc_grow_target(N, cap_max, grow_factor):
    """Row count after a growth of N rows: min(cap_max, int(grow_factor * N)); N itself when that is not larger."""
    return max(N, min(int(cap_max), int(grow_factor * N)))


def mcmc_workspace(N, dev):
    """A zero-filled workspace of the hg_mcmc_* entries for N rows (the regulariser's counter starts at zero)."""
    return torch.zeros(int(_G().hg_mcmc_workspace_bytes(N)), dtype=torch.uint8, device=dev)


def _offsets(N):
    starts, _total = arena_layout(N)
    return (ctypes.c_int64 * 5)(*[starts[n] for n, _ in GROUPS])


def _sources(sources, n, N, dev):
    """Injected draws as int64 device rows in [0, N) (checked on the host: a test path, it may synchronise)."""
    s = torch.as_tensor(sources).to(device=dev, dtype=torch.int64).contiguous().view(-1)
    if n is not None and s.numel() != n:
        raise ValueError("sources must hold %d rows, got %d" % (n, s.numel()))
    if s.numel() and (int(s.min()) < 0 or int(s.max()) >= N):
        raise ValueError("sources must be rows in [0, %d)" % N)
    return s


def mcmc_regularizer(param_arena, grad_arena, N, opacity_reg, scale_reg, grad_mult=1.0, loss_mult=0.0, loss=None,
                     workspace=None, skybox_points=0):
    """Reg = opacity_reg mean(o) + scale_reg mean(s) over the N rows: adds grad_mult dReg into the opacity and scaling
    rows of `grad_arena`, adds loss_mult Reg onto the device scalar `loss` (may be None) and returns Reg as a device
    scalar (None, and no launch, when both weights are 0).  `workspace`: mcmc_workspace(N) (allocated when None)."""
    if opacity_reg == 0.0 and scale_reg == 0.0:
        return None
    dev = param_arena.device
    ws = mcmc_workspace(N, dev) if workspace is None else workspace
    value = torch.empty((), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        rc = _G().hg_mcmc_regularizer(param_arena.data_ptr(), grad_arena.data_ptr(), _offsets(N), N, int(skybox_points),
                                      float(opacity_reg), float(scale_reg), float(grad_mult), float(loss_mult),
                                      value.data_ptr(), loss.data_ptr() if loss is not None else None, ws.data_ptr(),
                                      torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(rc, "mcmc_regularizer")
    return value


def mcmc_inject_noise(param_arena, N, scale, seed=0, normals=None, skybox_points=0):
    """gsplat's inject_noise_to_position in place: xyz += scale sigma(100 ((1 - o) - 0.995)) (R diag(s^2) R^T) z with
    scale = lr_xyz(it) * noise_lr; z from Philox4x32-10 keyed by `seed`, or `normals` [N, 3]."""
    dev = param_arena.device
    if normals is not None:
        normals = normals.to(device=dev, dtype=torch.float32).contiguous()
        if tuple(normals.shape) != (N, 3):
            raise ValueError("normals must be [%d, 3], got %s" % (N, tuple(normals.shape)))
    with torch.cuda.device(dev):
        rc = _G().hg_mcmc_inject_noise(param_arena.data_ptr(), _offsets(N), N, int(skybox_points), float(scale),
                                       normals.data_ptr() if normals is not None else None,
                                       int(seed) & 0xFFFFFFFFFFFFFFFF, torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(rc, "mcmc_inject_noise")


def mcmc_relocate_arenas(param_arena, exp_avg, exp_avg_sq, N, min_opacity=0.005, seed=0, sources=None,
                         skybox_points=0, workspace=None):
    """Relocate the dead rows (o <= min_opacity) of N-row arenas onto live ones drawn with probability o, in place
    (DESIGN.md §3 "MCMC densification").  Returns (param_arena, exp_avg, exp_avg_sq, counts) with counts =
    dict(dead=, alive=) as int64 device scalars: nothing is read back.  Draws from Philox4x32-10 keyed by `seed`, or
    `sources` (the source row of each dead row in row order; checked on the host)."""
    dev = param_arena.device
    ws = mcmc_workspace(N, dev) if workspace is None else workspace
    src = _sources(sources, None, N, dev) if sources is not None else None
    out = torch.empty(2, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        rc = _G().hg_mcmc_relocate(param_arena.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), _offsets(N), N,
                                   int(skybox_points), float(min_opacity),
                                   src.data_ptr() if src is not None and src.numel() else None,
                                   src.numel() if src is not None else 0, int(seed) & 0xFFFFFFFFFFFFFFFF,
                                   out.data_ptr(), ws.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(rc, "mcmc_relocate")
    return param_arena, exp_avg, exp_avg_sq, dict(dead=out[0], alive=out[1])


def mcmc_grow_arenas(param_arena, exp_avg, exp_avg_sq, N, n_target, min_opacity=0.005, seed=0, sources=None,
                     skybox_points=0, workspace=None):
    """Grow N-row arenas to `n_target` rows (N < n_target <= 2 N): n_target - N draws over all rows with probability
    o (Philox4x32-10 keyed by `seed`, or `sources` [n_target - N]); the drawn rows take (o', s') and zero moments, and
    their copies are appended in draw order with zero moments.  Returns (new parameter arena, new exp_avg, new
    exp_avg_sq, counts = dict(added=, n=)) with host ints; n_target <= N returns the arenas unchanged."""
    n_target = int(n_target)
    if n_target <= N:
        return param_arena, exp_avg, exp_avg_sq, dict(added=0, n=N)
    if n_target > 2 * N:
        raise ValueError("mcmc_grow_arenas: n_target %d exceeds 2 N = %d" % (n_target, 2 * N))
    dev = param_arena.device
    ws = mcmc_workspace(N, dev) if workspace is None else workspace
    src = _sources(sources, n_target - N, N, dev) if sources is not None else None
    _starts, total = arena_layout(n_target)
    new = [torch.empty(total, dtype=torch.float32, device=dev) for _ in range(3)]  # every float written by the kernels
    with torch.cuda.device(dev):
        rc = _G().hg_mcmc_grow(param_arena.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), _offsets(N), N,
                               new[0].data_ptr(), new[1].data_ptr(), new[2].data_ptr(), _offsets(n_target), n_target,
                               int(skybox_points), float(min_opacity), src.data_ptr() if src is not None else None,
                               int(seed) & 0xFFFFFFFFFFFFFFFF, ws.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(rc, "mcmc_grow")
    return new[0], new[1], new[2], dict(added=n_target - N, n=n_target)


def cameras_extent(cameras):
    """Scene extent of the densification thresholds: 1.1 x the largest distance of a camera centre from their mean
    (the radius of the reference's getNerfppNorm)."""
    c = torch.stack([torch.as_tensor(cam.camera_center, dtype=torch.float64).reshape(3).cpu() for cam in cameras])
    return float(torch.linalg.norm(c - c.mean(0), dim=1).max()) * 1.1


class GaussianParams:
    """Trainable Gaussians in the reference's parameterisation (scene/gaussian_model.py:60-140): raw leaves
    `_xyz`, `_features` (N,16,3), `_opacity` (logit), `_scaling` (log), `_rotation` (un-normalised quaternion) and the
    activated accessors render() reads.  All leaves are views into one flat parameter arena; their `.grad` are views
    into one flat gradient arena of the same layout."""

    def __init__(self, xyz, features, opacity_logit, scaling_log, rotation, sh_degree=3):
        N = xyz.size(0)
        starts, total = arena_layout(N)
        param_arena = torch.zeros(total, dtype=torch.float32, device=xyz.device)
        src = dict(xyz=xyz, features=features.reshape(N, -1), opacity=opacity_logit, scaling=scaling_log, rotation=rotation)
        for name, w in GROUPS:
            param_arena[starts[name]:starts[name] + N * w].view(N, w).copy_(src[name].reshape(N, w))
        self._attach(param_arena, N)
        self.active_sh_degree = self.max_sh_degree = sh_degree
        self.skybox_points = 0
        self.order = None
        # fused activations (CUDA only): one kernel per view forward, one backward that also accumulates into the arena
        self.fused = xyz.is_cuda
        self._act = None          # (xyz, features, opacity, scaling, rotation) of the current view
        self._grad_dirty = False  # False: the next fused backward overwrites the arena (no zero fill needed)
        self.sh_sink = self.fused  # SH gradient accumulated by the rasterizer's own backward kernel
        self._sink_used = False
        self.exposure_mapping = None  # per-image exposure: setup_exposures
        self._exposure = self.exposure_grad = None
        self.camera_pose_mapping = None  # per-image camera pose correction: setup_camera_poses
        self._camera_pose = self.camera_pose_grad = None

    def setup_exposures(self, image_names, exposures=None):
        """Per-image exposure table of the reference's GaussianModel (`_exposure`, `exposure_mapping`; applied by
        render(..., use_trained_exp=True), DESIGN.md §3 "Per-image exposure"): row i is the [3, 4] affine of
        image_names[i], eye(3, 4) to start with, or exposures[name] (a load_exposures dict, which must cover every
        name).  The leaf `_exposure` [n, 3, 4] has its `.grad` aliasing `exposure_grad`, as the arena leaves alias the
        gradient arena.  The table is per image, not per Gaussian: densify_and_prune and resize leave it alone."""
        names = list(image_names)
        if len(set(names)) != len(names):
            raise ValueError("setup_exposures: duplicate image names")
        dev = self.param_arena.device
        table = torch.eye(3, 4, dtype=torch.float32).repeat(len(names), 1, 1)
        if exposures is not None:
            missing = [n for n in names if n not in exposures]
            if missing:
                raise ValueError("setup_exposures: no exposure for %s" % missing[:5])
            for i, n in enumerate(names):
                table[i] = torch.as_tensor(exposures[n], dtype=torch.float32).cpu().reshape(3, 4)
        self.exposure_mapping = {n: i for i, n in enumerate(names)}
        self._exposure = table.to(dev).requires_grad_(True)
        self.exposure_grad = torch.zeros_like(self._exposure, requires_grad=False)
        self._exposure.grad = self.exposure_grad

    def exposure_index(self, image_name):
        """Row of `image_name` in the exposure table; ValueError if there is no table or no such image."""
        if self.exposure_mapping is None:
            raise ValueError("no exposure table: call setup_exposures(image_names) first")
        try:
            return self.exposure_mapping[image_name]
        except KeyError:
            raise ValueError("no exposure for image %r" % (image_name,)) from None

    def get_exposure_from_name(self, image_name):
        """GaussianModel.get_exposure_from_name: the [3, 4] exposure of `image_name` (a differentiable view of the
        table), as render(..., use_trained_exp=True) reads it."""
        return self._exposure[self.exposure_index(image_name)]

    def save_exposures(self, path):
        """exposure.json of the table (ply_io.save_exposures, rows in mapping order)."""
        from . import ply_io
        names = sorted(self.exposure_mapping, key=self.exposure_mapping.get)
        ply_io.save_exposures(path, self._exposure, names)

    def setup_camera_poses(self, image_names, poses=None):
        """Per-image camera pose corrections (DESIGN.md §3 "Camera pose refinement"): row i of the leaf `_camera_pose`
        [n, 8] is xi = (rho 3, phi 3, 2 zero pads) of image_names[i], applied in the camera frame (p_cam' = Exp(phi)
        p_cam + rho); zero to start with, or poses[name] (a ply_io.load_camera_poses dict, which must cover every name).
        Its `.grad` aliases `camera_pose_grad`.  The table is per image, not per Gaussian: densify_and_prune and resize
        leave it alone."""
        from . import camera_pose as cp
        names = list(image_names)
        if len(set(names)) != len(names):
            raise ValueError("setup_camera_poses: duplicate image names")
        table = torch.zeros((len(names), cp.ROW), dtype=torch.float32)
        if poses is not None:
            missing = [n for n in names if n not in poses]
            if missing:
                raise ValueError("setup_camera_poses: no pose for %s" % missing[:5])
            for i, n in enumerate(names):
                xi = torch.as_tensor(poses[n], dtype=torch.float32).cpu().reshape(-1)
                if xi.numel() != 6:
                    raise ValueError("setup_camera_poses: the pose of %r has %d numbers, expected 6" % (n, xi.numel()))
                table[i, :6] = xi
        self.camera_pose_mapping = {n: i for i, n in enumerate(names)}
        self._camera_pose = table.to(self.param_arena.device).requires_grad_(True)
        self.camera_pose_grad = torch.zeros_like(self._camera_pose, requires_grad=False)
        self._camera_pose.grad = self.camera_pose_grad

    def camera_pose_index(self, image_name):
        """Row of `image_name` in the camera pose table; ValueError if there is no table or no such image."""
        if self.camera_pose_mapping is None:
            raise ValueError("no camera pose table: call setup_camera_poses(image_names) first")
        try:
            return self.camera_pose_mapping[image_name]
        except KeyError:
            raise ValueError("no camera pose for image %r" % (image_name,)) from None

    def _corrected_matrices(self, k, viewmatrix, projmatrix, campos):
        """[36] device buffer: viewmatrix' | projmatrix' | campos' | 0 of row k (hg_camera_pose_apply, no host read)."""
        dev = self.param_arena.device
        out = torch.empty(36, dtype=torch.float32, device=dev)
        vm, pm, cp_ = (t.to(device=dev, dtype=torch.float32).contiguous() for t in (viewmatrix, projmatrix, campos))
        with torch.cuda.device(dev):
            rc = _G().hg_camera_pose_apply(vm.data_ptr(), pm.data_ptr(), cp_.data_ptr(), self._camera_pose.data_ptr(),
                                           self._camera_pose.size(0), k, out.data_ptr(),
                                           torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, "camera_pose_apply")
        return out

    def corrected_camera(self, cam):
        """A shallow copy of `cam` whose world_view_transform / full_proj_transform / camera_center (CUDA tensors) carry
        the correction of its image, for render() and evaluation; intrinsics and image size are the camera's."""
        import copy
        if not self.fused:
            raise ValueError("corrected_camera needs CUDA parameters")
        buf = self._corrected_matrices(self.camera_pose_index(cam.image_name), cam.world_view_transform,
                                       cam.full_proj_transform, cam.camera_center)
        out = copy.copy(cam)
        out.world_view_transform = buf[:16].view(4, 4)
        out.full_proj_transform = buf[16:32].view(4, 4)
        out.camera_center = buf[32:35]
        return out

    def save_camera_poses(self, path, cameras):
        """camera_poses.json (ply_io.save_camera_poses): xi of every image of the table, and the corrected
        world-to-camera matrix of those among `cameras` (float64 on the host, camera_pose.corrected_w2c)."""
        from . import camera_pose as cp
        from . import ply_io
        names = sorted(self.camera_pose_mapping, key=self.camera_pose_mapping.get)
        table = self._camera_pose.detach().double().cpu().numpy()
        w2c = {}
        for cam in cameras:
            k = self.camera_pose_index(cam.image_name)
            w2c[cam.image_name] = cp.corrected_w2c(cam.world_view_transform.detach().double().cpu().numpy(), table[k, :6])
        ply_io.save_camera_poses(path, self._camera_pose, names, w2c)

    def _attach(self, param_arena, N):
        """Adopt `param_arena` (arena_layout(N)) with a fresh gradient arena of the same layout, the leaves and their
        `.grad` views.  The constructor and `resize` both come through here.  Where the gradient arena is multicast
        symmetric memory its allocation is collective: every rank calls this with the same N."""
        dev = param_arena.device
        starts, total = arena_layout(N)
        self.N = N
        self.param_arena = param_arena
        # the gradient arena is born where the per-step exchange wants it: multicast symmetric memory when the ranks
        # share an NVSwitch (in-fabric all-reduce kernel), a plain tensor otherwise (NCCL / gloo all-reduce)
        self.exchange = None
        if dist.is_initialized() and dist.get_world_size() > 1 and dev.type == "cuda":
            self.grad_arena, self.exchange = parallel.make_exchange_arena(total, dev)
        else:
            self.grad_arena = torch.zeros(total, dtype=torch.float32, device=dev)
        self.leaves, self.slices = {}, {}
        for name, w in GROUPS:
            sl = slice(starts[name], starts[name] + N * w)
            self.slices[name] = sl
            shape = (N, 16, 3) if name == "features" else (N, w)
            leaf = self.param_arena[sl].view(shape).requires_grad_(True)
            leaf.grad = self.grad_arena[sl].view(shape)
            self.leaves[name] = leaf
        self._xyz, self._features = self.leaves["xyz"], self.leaves["features"]
        self._opacity, self._scaling, self._rotation = self.leaves["opacity"], self.leaves["scaling"], self.leaves["rotation"]

    def resize(self, param_arena, N):
        """Adopt a parameter arena of N rows (densify_and_prune): new gradient arena, leaves and `.grad` views.  The
        rows are no longer along the Morton curve of `from_scene(spatial_order=True)`: `.order` becomes None."""
        self._attach(param_arena, N)
        self.order = None
        self._act = None
        self._grad_dirty = False
        self._sink_used = False

    @classmethod
    def from_scene(cls, scene, device, spatial_order=False):
        """From a synthetic scene dict (hidegs_b200.synthetic.make_scene): activated values -> raw leaves.

        `spatial_order`: store the Gaussians along a Morton curve (`morton_order`).  A camera sees a compact region of
        the scene, so with a spatially coherent layout the visible set of a view is a few contiguous index ranges:
        whole warps of the per-Gaussian kernels are culled or live together, the sparse Adam touches whole sectors, and
        the blend kernels' record gathers stay local in L2.  The permutation is kept in `.order` (row i of the model is
        row order[i] of the input); rendering and training are invariant to it."""
        op = scene["opacity"].clamp(1e-6, 1 - 1e-6)
        t = [scene["means3D"], scene["shs"], torch.log(op / (1 - op)), torch.log(scene["scales"]), scene["rotations"]]
        order = None
        if spatial_order:
            order = morton_order(scene["means3D"])
            t = [x[order] for x in t]
        out = cls(*[x.to(device) for x in t])
        out.order = order
        return out

    def _activated(self, i):
        if self._act is None:
            self._act = _ActivateParams.apply(self._xyz, self._features, self._opacity, self._scaling, self._rotation, self)
            if self.sh_sink:  # the rasterizer backward accumulates dL/dSH straight into the gradient arena
                self._act[1]._hg_grad_sink = self._sh_sink_now
        return self._act[i]

    def _sh_sink_now(self):
        """(sink tensor, beta) at the time the rasterizer backward of the current view runs."""
        self._sink_used = True
        return self.grad_arena[self.slices["features"]].view(self.N, 16, 3), (1.0 if self._grad_dirty else 0.0)

    def begin_view(self):
        """Fresh activation node for the next forward/backward (one autograd graph per view)."""
        self._act = None

    get_xyz = property(lambda s: s._activated(0) if s.fused else s._xyz)
    get_features = property(lambda s: s._activated(1) if s.fused else s._features)
    get_opacity = property(lambda s: s._activated(2) if s.fused else torch.sigmoid(s._opacity))
    get_scaling = property(lambda s: s._activated(3) if s.fused else torch.exp(s._scaling))
    get_rotation = property(lambda s: s._activated(4) if s.fused else torch.nn.functional.normalize(s._rotation))

    def zero_grad(self):
        self._act = None
        if self.fused:
            self._grad_dirty = False  # the first backward of the step overwrites the arena: no memset
        else:
            self.grad_arena.zero_()
        for name, leaf in self.leaves.items():  # autograd may have replaced .grad; point it back at the arena
            shape = leaf.shape
            leaf.grad = self.grad_arena[self.slices[name]].view(shape)


class ArenaAdam:
    """Fused Adam over the parameter arena (scene/OurAdam.py semantics, one launch per parameter group; the SH
    block takes two: DC at feature_lr, the rest at feature_lr / 20, as GaussianModel.training_setup does)."""

    def __init__(self, params: GaussianParams, opt=OptimizationParams, spatial_lr_scale=1.0, eps=1e-15):
        self.p = params
        self.exp_avg = torch.zeros_like(params.param_arena)
        self.exp_avg_sq = torch.zeros_like(params.param_arena)
        self.lr = dict(xyz=opt.position_lr_init * spatial_lr_scale, features=opt.feature_lr, opacity=opt.opacity_lr,
                       scaling=opt.scaling_lr, rotation=opt.rotation_lr)
        self.spatial_lr_scale = spatial_lr_scale
        self.eps, self.step_count = eps, 0

    def resize(self, exp_avg, exp_avg_sq):
        """Adopt moment arenas of the parameters' new size (densify_and_prune); the step count carries on, as
        cat_tensors_to_optimizer keeps state["step"]."""
        self.exp_avg, self.exp_avg_sq = exp_avg, exp_avg_sq

    @torch.no_grad()
    def step(self, grad_scale=1.0, visible_mask=None):
        self.step_count += 1
        p = self.p
        p._act = None  # the activated copies are stale after the update
        st = torch.cuda.current_stream().cuda_stream
        mask = None
        if visible_mask is not None:
            vm = visible_mask.contiguous()
            self._mask_keepalive = vm = vm.view(torch.uint8) if vm.dtype == torch.bool else vm
            mask = vm.data_ptr()
        with torch.cuda.device(p.param_arena.device):
            for name, w in GROUPS:
                sl = p.slices[name]
                base = sl.start * 4
                if name == "features":
                    # rows of 48 floats: [dc(3) | rest(45)]: two learning rates in one pass
                    rc = self._launch(base, p.N, 48, mask, self.lr["features"] / 20.0, grad_scale, st, 3, self.lr["features"])
                    _lib.check(rc, "adam_step")
                    continue
                rc = self._launch(base, p.N, w, mask, self.lr[name], grad_scale, st)
                _lib.check(rc, "adam_step")

    def _launch(self, byte_off, rows, width, mask, lr, grad_scale, st, head_cols=0, head_lr=0.0):
        p = self.p
        return _G().hg_adam_step(p.param_arena.data_ptr() + byte_off, p.grad_arena.data_ptr() + byte_off,
                                 self.exp_avg.data_ptr() + byte_off, self.exp_avg_sq.data_ptr() + byte_off, rows, width,
                                 mask, None, 0, lr, 0.9, 0.999, self.eps, self.step_count, grad_scale, head_cols, head_lr, st)


def balance_views(costs, world, speeds=None):
    """Shard `len(costs)` views over `world` ranks with equal counts and near-equal time.  `costs[i]`: predicted cost
    of view i (its device time or num_rendered from an earlier visit).  `speeds[r]` (optional): time multiplier of rank
    r — the GPUs of one box do not run at exactly the same pace (power / thermal headroom, host placement) — so that the
    time of a rank is speeds[r] * (sum of its views' costs) and a slower rank is handed lighter views.
    Start: the better of views[rank::world] and longest-processing-time-first with a per-rank capacity; then pairwise
    swaps between the slowest rank and the others while they lower the larger of the two times.  Returns one sorted
    index list per rank; every rank computes the same assignment from the same table."""
    n = len(costs)
    c = [float(x) for x in costs]
    s = [1.0] * world if speeds is None else [float(x) for x in speeds]
    room = [n // world + (1 if r < n % world else 0) for r in range(world)]
    lpt = [[] for _ in range(world)]
    load = [0.0] * world
    for i in sorted(range(n), key=lambda k: (-c[k], k)):
        r = min((q for q in range(world) if len(lpt[q]) < room[q]), key=lambda q: (load[q] + s[q] * c[i], q))
        lpt[r].append(i)
        load[r] += s[r] * c[i]
    strided = [list(range(n))[r::world] for r in range(world)]
    total = lambda sh: [s[r] * sum(c[i] for i in x) for r, x in enumerate(sh)]  # noqa: E731
    out = lpt if max(total(lpt)) <= max(total(strided)) else strided
    load = total(out)
    for _ in range(4 * n):
        h = max(range(world), key=lambda q: (load[q], -q))
        best = None
        for r in range(world):
            if r == h:
                continue
            for a_ in out[h]:
                for b_ in out[r]:
                    d = c[a_] - c[b_]
                    if d <= 0:
                        continue
                    worst = max(load[h] - s[h] * d, load[r] + s[r] * d)
                    if worst < load[h] and (best is None or worst < best[0]):
                        best = (worst, r, a_, b_)
        if best is None:
            break
        _w, r, a_, b_ = best
        out[h][out[h].index(a_)] = b_
        out[r][out[r].index(b_)] = a_
        load[h] -= s[h] * (c[a_] - c[b_])
        load[r] += s[r] * (c[a_] - c[b_])
    return [sorted(x) for x in out]


class ViewShardedTrainer:
    train_exposure = False  # (class defaults: also read by trainers assembled without __init__)
    depth_regularization = False
    train_poses = False
    mcmc = False

    def __init__(self, params: GaussianParams, background, opt=OptimizationParams, pipe=PipelineParams, group=None,
                 sparse_adam=True, densification_stats=False, cache_ground_truth=False, start_iteration=0, densify=False,
                 scene_extent=None, train_exposure=False, depth_regularization=False, train_poses=False, mcmc=False,
                 mcmc_cap_max=None):
        """`densify`: run the adaptive density control schedule of the OptimizationParams densify_* fields inside
        `step()` (off by default); it needs `scene_extent` (`cameras_extent(cameras)`) and turns the densification
        statistics on.
        `train_exposure`: render every view through the exposure of its `cam.image_name` and learn the table (off by
        default); it needs `params.setup_exposures(image_names)` first.  Every step zeroes the exposure gradient table,
        sums it over the ranks and steps it with its own Adam (eps 1e-8, dense over the whole table, the lr schedule of
        the OptimizationParams exposure_* fields).
        `depth_regularization`: add graphdeco's masked inverse-depth L1, w(it) mean |(invdepth - cam.invdepthmap) *
        cam.depth_mask|, to the loss of every view whose camera carries a reliable prior (ply_io.attach_depth_prior;
        DESIGN.md §3 "Depth regularisation"), with w(it) the schedule of the OptimizationParams depth_l1_weight_*
        fields (off by default).  A view without a reliable prior, or a step with w(it) = 0, runs as it does with the
        flag off.
        `train_poses`: render every view through the pose correction of its `cam.image_name` and learn the table (off
        by default; DESIGN.md §3 "Camera pose refinement"); it needs `params.setup_camera_poses(image_names)` first and
        the direct executor (not HG_TRAINER_DIRECT=0: the autograd path has no camera gradient).  Every step zeroes the
        pose gradient table, sums it over the ranks and steps it with its own Adam (eps 1e-8, dense over the whole
        table, the constant rates OptimizationParams.pose_lr_translation x spatial_lr_scale and pose_lr_rotation).
        `mcmc`: 3DGS-MCMC densification instead of adaptive density control (off by default; DESIGN.md §3 "MCMC
        densification"): the opacity / scale regulariser in every step, relocation of dead Gaussians and growth by
        mcmc_grow_factor up to `mcmc_cap_max` Gaussians on the schedule of the OptimizationParams mcmc_* fields, position
        noise after every optimiser update, and graphdeco's position learning-rate schedule.  It needs CUDA parameters
        without skybox points and mcmc_cap_max >= params.N, and excludes `densify`.  The model's size never exceeds
        mcmc_cap_max; nothing of it reads back to the host, and every rank computes the same bits (the arenas are
        identical after the exchange and the Adam step, and every kernel is deterministic in its inputs and seed)."""
        import os
        if mcmc:  # (refusals before anything changes)
            if densify:
                raise ValueError("mcmc=True and densify=True are two densification strategies: choose one")
            if params.skybox_points:
                raise ValueError("mcmc=True: models with skybox points are not supported")
            if mcmc_cap_max is None or int(mcmc_cap_max) < params.N:
                raise ValueError("mcmc=True needs mcmc_cap_max >= params.N = %d, got %r" % (params.N, mcmc_cap_max))
            if not 1.0 <= float(opt.mcmc_grow_factor) <= 2.0:
                raise ValueError("mcmc_grow_factor must be in [1, 2], got %r" % (opt.mcmc_grow_factor,))
            if not params.fused:
                raise ValueError("mcmc=True needs CUDA parameters")
        self.params, self.bg, self.opt, self.pipe, self.group = params, background, opt, pipe, group
        if densify and scene_extent is None:
            raise ValueError("densify=True needs scene_extent (cameras_extent(cameras))")
        self.train_poses = bool(train_poses)
        if self.train_poses:
            if params._camera_pose is None:
                raise ValueError("train_poses=True needs params.setup_camera_poses(image_names)")
            if not params.fused:
                raise ValueError("train_poses=True needs CUDA parameters")
            if os.environ.get("HG_TRAINER_DIRECT", "1") == "0":
                raise ValueError("train_poses=True needs the direct executor: the autograd path (HG_TRAINER_DIRECT=0) "
                                 "forms no camera gradient")
            self.pose_exp_avg = torch.zeros_like(params._camera_pose, requires_grad=False)
            self.pose_exp_avg_sq = torch.zeros_like(params._camera_pose, requires_grad=False)
            self.pose_step_count = 0
            self._pose_ws = None
        self.train_exposure = bool(train_exposure)
        if self.train_exposure:
            if params._exposure is None:
                raise ValueError("train_exposure=True needs params.setup_exposures(image_names)")
            if not params.fused:
                raise ValueError("train_exposure=True needs CUDA parameters")
            from .optim import get_expon_lr_func
            self.exposure_lr = get_expon_lr_func(opt.exposure_lr_init, opt.exposure_lr_final, opt.exposure_lr_delay_steps,
                                                 opt.exposure_lr_delay_mult, max_steps=opt.iterations)
            self.exposure_exp_avg = torch.zeros_like(params._exposure, requires_grad=False)
            self.exposure_exp_avg_sq = torch.zeros_like(params._exposure, requires_grad=False)
            self.exposure_step_count = 0
            self._exposure_ws = None
        self.depth_regularization = bool(depth_regularization)
        if self.depth_regularization:
            from .optim import get_expon_lr_func
            self.depth_l1_weight = get_expon_lr_func(opt.depth_l1_weight_init, opt.depth_l1_weight_final,
                                                     max_steps=opt.iterations)
            self._depth_ws = None
        self.densify, self.scene_extent = densify, scene_extent
        densification_stats = densification_stats or densify
        self.adam = ArenaAdam(params, opt)
        self.mcmc = bool(mcmc)
        if self.mcmc:
            from .optim import get_expon_lr_func
            sc = self.adam.spatial_lr_scale
            self.mcmc_cap_max = int(mcmc_cap_max)
            self.xyz_lr = get_expon_lr_func(opt.position_lr_init * sc, opt.position_lr_final * sc,
                                            lr_delay_mult=opt.position_lr_delay_mult,
                                            max_steps=opt.position_lr_max_steps)
            self._mcmc_ws = mcmc_workspace(params.N, params.param_arena.device)
        # the reference steps its optimiser on the rows that were visible (`optimizer.step(relevant)`, OurAdam.py:106)
        self.sparse_adam = sparse_adam and params.param_arena.is_cuda
        self.visible = torch.zeros(params.N, dtype=torch.uint8, device=params.param_arena.device)
        # per-camera cache of everything derived from the ground-truth image alone (frequency-loss spectra, high-frequency
        # mask, edge-aware weight of the normal term); keyed by the camera object, built at the camera's first visit
        self.cache_ground_truth = cache_ground_truth
        self._gt_cache = {}
        self.densification_stats = densification_stats and params.param_arena.is_cuda
        if self.densification_stats:  # GaussianModel.training_setup (scene/gaussian_model.py:282-294)
            self._zero_densification_stats()
        self._opacity_resets = 0
        # the frequency / scale regulariser switches on at opt.freq_warmup_iterations, as the reference's
        # frequency_regularization_pyramid_scale(iteration, warmup_iterations=1000) does; `start_iteration` resumes a run
        self.iteration = int(start_iteration)
        # autograd-free executor of a view (view_step_direct); HG_TRAINER_DIRECT=0 keeps the autograd path
        self.direct = params.fused and os.environ.get("HG_TRAINER_DIRECT", "1") != "0"
        self._one = None
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0

    def view_loss(self, cam, gt, iteration, gt_ready=None):
        """Forward of one view: returns (loss tensor, render package).  `gt_ready`: CUDA event after which `gt` holds
        the image (an upload running on a copy stream while the view renders)."""
        o = self.opt
        self.params.begin_view()
        exp = self.train_exposure
        if exp:
            self.params.exposure_index(cam.image_name)  # (ValueError before any work for an unknown image)
        pkg = gr._render_impl(cam, self.params, self.pipe, self.bg, use_trained_exp=exp,
                              _visibility_as_mask=self.params.param_arena.is_cuda)
        if gt_ready is not None:
            torch.cuda.current_stream().wait_event(gt_ready)
        image = pkg["render"]
        loss = (1.0 - o.lambda_dssim) * lu.l1_loss(image, gt) + o.lambda_dssim * (1.0 - lu.ssim(image, gt))
        cache = None
        if self.cache_ground_truth and iteration >= o.freq_warmup_iterations:
            cache = self._gt_cache.get(id(cam))
            if cache is None:
                cache = self._gt_cache[id(cam)] = (cam, GroundTruthCache(gt), (1.0 - lu.get_img_grad_weight(gt)).clamp(0, 1) ** 2)
        freq, _mask, _info = frequency_regularization_pyramid_scale(
            image, gt, self.params, None, cam, pkg["visibility_filter"], iteration, lambda_freq=o.lambda_freq,
            lambda_scale=o.lambda_scale, warmup_iterations=o.freq_warmup_iterations,
            gt_cache=cache[1] if cache is not None else None)
        loss = loss + freq
        if o.single_view_weight > 0:
            image_weight = cache[2] if cache is not None else (1.0 - lu.get_img_grad_weight(gt)).clamp(0, 1) ** 2
            loss = loss + gr.normal_consistency_loss(pkg["plane_depth"], pkg["out_all_map"], cam, image_weight,
                                                     o.single_view_weight)
        depth = self._depth_term(cam, iteration)
        if depth is not None:  # + w(it) * Ll1depth, added last
            mono, mask, w = depth
            depth_l1 = lu.inverse_depth_l1(pkg["depth"], mono, mask)
            loss = loss + w * depth_l1
            pkg["depth_l1"] = depth_l1.detach()
        return loss, pkg

    # ------------------------------------------------------------------------------------------------------------------
    # The same view without autograd.  The training step is host bound (2.2 ms of host time per view against ~1.7 ms of
    # kernels: tools/train_cpu_profile.py), and most of that host time is autograd's — nine custom Functions applied and
    # walked back, ~40 glue ops recorded and differentiated.  The graph of a view is FIXED, so it is executed here as a
    # straight sequence: the forward and backward BODIES of the very same Functions (one implementation, one set of
    # kernels) run on a hand-written tape, the loss weights are folded into the three image-gradient terms, and nothing
    # is recorded.  tests/test_trainer_gpu.py holds it to the autograd path (same gradient arena, same loss).
    class _Tape:
        """What an autograd.Function body expects of `ctx`."""

        def __init__(self, *needs):
            self.needs_input_grad = needs
            self.saved_tensors = ()

        def save_for_backward(self, *tensors):
            self.saved_tensors = tensors

        def mark_non_differentiable(self, *_a):
            pass

        def set_materialize_grads(self, _v):
            pass

    def view_step_direct(self, cam, gt, iteration, gt_ready=None):
        """Forward AND backward of one view (gradients accumulated into the arena), without autograd.  Returns
        (loss value tensor, dict with "visibility_filter" (mask), "radii", "means2D_grad" — defined on the rendered rows
        only: the rasterizer's backward does not write the rows of culled Gaussians here); with train_exposure also
        "render", the exposed, clamped image the losses saw; with the depth term on this view also "depth_l1", the
        unweighted masked inverse-depth L1 (device scalar); with train_poses also "pose_grad", this view's contribution
        (dL/drho, dL/dphi) to its camera's row of the pose gradient table (device, 6 floats)."""
        o, p, T = self.opt, self.params, self._Tape
        dev = p.param_arena.device
        depth = self._depth_term(cam, iteration)  # (mono, mask, w) or None: the view runs as with the flag off
        exp_off = None  # byte offset of this camera's exposure row in the table / its gradient table
        if self.train_exposure:
            exp_off = 48 * p.exposure_index(cam.image_name)
        pose_k = p.camera_pose_index(cam.image_name) if self.train_poses else None
        with torch.no_grad():
            # ---- forward
            # the activated parameters are the same for every view of one optimiser step: step() keeps them
            act = getattr(self, "_step_activations", None)
            if act is None:
                tA = T(True, True, True, True, True, False)
                act = _ActivateParams.forward(tA, p._xyz, p._features, p._opacity, p._scaling, p._rotation, p)
                if getattr(self, "_in_step", False):
                    self._step_activations = act
            xyz, feat, opacity, scaling, rotation = act
            e_i = torch.empty(0, dtype=torch.int32, device=dev)
            e_f = torch.empty(0, dtype=torch.float32, device=dev)
            rs = gr._raster_settings(cam, p, self.pipe, self.bg, 1.0, True, True, e_i, e_i, e_f, e_i)
            pose_ws = None
            if pose_k is not None:  # the corrected camera, formed on the device: every kernel below reads it
                cbuf = p._corrected_matrices(pose_k, rs.viewmatrix, rs.projmatrix, rs.campos)
                rs = rs._replace(viewmatrix=cbuf[:16].view(4, 4), projmatrix=cbuf[16:32].view(4, 4), campos=cbuf[32:35])
                pose_ws = self._pose_workspace(p.N, dev)
            tM = T(True, False, True, False, False)
            all_map_in = gr._AllMap.forward(tM, xyz, scaling, rotation, rs.viewmatrix, rs.campos)
            if p.sh_sink:
                feat._hg_grad_sink = p._sh_sink_now
            tR = T(True, True, True, False, True, True, True, False, True, False)
            color, radii, _observe, out_all_map, plane_depth, _inv = _RasterizeGaussians.forward(
                tR, xyz, xyz, feat, e_f, opacity, scaling, rotation, e_f, all_map_in, rs)
            if exp_off is None:
                image = color.clamp(0, 1)
            else:  # clamp(color through the camera's exposure, 0, 1): hg_exposure_apply
                image = torch.empty_like(color)
                with torch.cuda.device(dev):
                    rc = lu._L().hg_exposure_apply(color.data_ptr(), p._exposure.data_ptr() + exp_off, color.size(1),
                                                   color.size(2), image.data_ptr(), torch.cuda.current_stream().cuda_stream)
                _lib.check(rc, "exposure_apply")
            if gt_ready is not None:
                torch.cuda.current_stream().wait_event(gt_ready)
            tL, tS = T(False, False, False), T(True, False, False)  # (the L1 gradient is formed in the combine kernel)
            l1 = lu._PixelLoss.forward(tL, image, gt, False)
            ss = lu._SSIM.forward(tS, image, gt, True)
            visible = radii > 0
            cache = None
            freq_on = iteration >= o.freq_warmup_iterations
            if self.cache_ground_truth and freq_on:
                cache = self._gt_cache.get(id(cam))
                if cache is None:
                    cache = self._gt_cache[id(cam)] = (cam, GroundTruthCache(gt),
                                                       (1.0 - lu.get_img_grad_weight(gt)).clamp(0, 1) ** 2)
            tF = tSc = tT = None
            reg_total = normal_term = None
            if freq_on:  # frequency_regularization_pyramid_scale (same arithmetic, same order)
                freq_loss = scale_loss = None
                count = cache[1].count if cache is not None else None
                if o.lambda_freq > 0:
                    tF = T(True, False, False, False, False)
                    if cache is not None:
                        freq_loss, _stats = _FreqLoss.forward(tF, image, gt, 3, cache[1].state)
                    else:  # the high-frequency mask of this ground truth rides the same launches
                        freq_loss, _stats, _mask, count = _FreqLoss.forward(tF, image, gt, 3, None, 0.2)
                if o.lambda_scale > 0:
                    if count is None:
                        count = detect_true_high_frequency_regions(gt)[1]
                    tSc = T(True, False)
                    scale_loss = _ScaleReg.forward(tSc, scaling, visible)
                if freq_loss is not None or scale_loss is not None:
                    tT = T(freq_loss is not None, scale_loss is not None, False, False, False)
                    reg_total = _FreqTotal.forward(tT, freq_loss, scale_loss, count, o.lambda_freq, o.lambda_scale)
            tN = None
            if o.single_view_weight > 0:
                image_weight = cache[2] if cache is not None else (1.0 - lu.get_img_grad_weight(gt)).clamp(0, 1) ** 2
                tN = T(True, True, False, False, False)
                normal_term = gr._NormalConsistency.forward(tN, plane_depth, out_all_map, image_weight,
                                                            gr.camera_intrinsics(cam), o.single_view_weight)
            # (1 - l) L1 + l (1 - SSIM) + regulariser total + normal term: one launch for the scalar bookkeeping
            loss = torch.empty((), dtype=torch.float32, device=dev)
            with torch.cuda.device(dev):
                rc = lu._L().hg_training_loss_value(
                    l1.data_ptr(), ss.data_ptr(), reg_total.data_ptr() if reg_total is not None else None,
                    normal_term.data_ptr() if normal_term is not None else None, float(o.lambda_dssim), loss.data_ptr(),
                    torch.cuda.current_stream().cuda_stream)
            _lib.check(rc, "training_loss_value")
            g_inv = depth_l1 = None
            if depth is not None:  # + w(it) mean |(invdepth - mono) * mask| onto `loss`, and its gradient, in one pass
                mono, mask, w = depth
                g_inv = torch.empty_like(_inv)
                depth_l1 = torch.empty((), dtype=torch.float32, device=dev)
                lu._invdepth_l1_launch(_inv, mono, mask, w, g_inv, depth_l1, loss,
                                       self._depth_workspace(_inv.size(-2), _inv.size(-1), dev))
            # ---- backward (upstream gradient of the loss = 1)
            # dL/dcolor = [0 <= color <= 1] ((1 - l) dL1 - l dSSIM + gate lf dfreq) in ONE pass over the image
            if self._one is None:
                self._one = torch.ones((), dtype=torch.float32, device=dev)
            g_color = lu._SSIM.backward(tS, self._one)[0]
            # d(lambda_freq * clamp gate * freq_loss) / d image: the scalar rides the regulariser's last backward kernel
            g_freq = _FreqLoss.backward(tF, tT.partials[1])[0] if tF is not None else None
            if exp_off is None:
                with torch.cuda.device(dev):
                    rc = lu._L().hg_training_image_grad(
                        color.data_ptr(), gt.data_ptr(), g_color.data_ptr(), g_freq.data_ptr() if g_freq is not None else None,
                        color.numel(), 1.0 - o.lambda_dssim, -o.lambda_dssim,
                        self._one.data_ptr() if g_freq is not None else None, g_color.data_ptr(),
                        torch.cuda.current_stream().cuda_stream)
                _lib.check(rc, "training_image_grad")
            else:  # the same gradient through the exposure, + this view's 12 exposure sums into the camera's row
                H, W = color.size(1), color.size(2)
                ws = self._exposure_workspace(H, W, dev)
                with torch.cuda.device(dev):
                    rc = lu._L().hg_training_image_grad_exposure(
                        color.data_ptr(), p._exposure.data_ptr() + exp_off, gt.data_ptr(), g_color.data_ptr(),
                        g_freq.data_ptr() if g_freq is not None else None, H, W, 1.0 - o.lambda_dssim, -o.lambda_dssim,
                        self._one.data_ptr() if g_freq is not None else None, g_color.data_ptr(),
                        p.exposure_grad.data_ptr() + exp_off, ws.data_ptr(), torch.cuda.current_stream().cuda_stream)
                _lib.check(rc, "training_image_grad_exposure")
            g_pd = tN.gd.reshape(plane_depth.shape) if tN is not None else None
            g_am = tN.gam if tN is not None else None
            # with the SH sink the rasterizer's backward leaves the gradient rows of culled Gaussians unwritten: the
            # fused prologue backward below looks at `radii` first (a UAV view culls ~80 % of the slab).  Without the
            # sink the SH gradient comes back as a dense tensor that the prologue backward adds to the arena row for
            # row, so every row of it (culled Gaussians, inactive SH bands) must be written
            tR.skip_culled_rows = tR.sh_sink is not None
            tR.pose_workspace = pose_ws  # (None: the plain backward)
            (g_xyz, g_means2D, g_sh, _gc, g_op, g_sc, g_rot, _gcov, g_all_map_in, _n) = _RasterizeGaussians.backward(
                tR, g_color, None, None, g_am, g_pd, g_inv)
            # all_map backward + scale-regulariser gradient + activation chain rule + accumulation into the arena: one
            # kernel over the rendered rows (hg_prologue_backward)
            self._prologue_backward(p, radii, rs, g_xyz, g_sh, g_op, g_sc, g_rot, g_all_map_in,
                                    tSc.grad if tSc is not None else None, tT.partials[2] if tSc is not None else None,
                                    pose_ws)
            pose_grad = None
            if pose_k is not None:  # both partial sets -> dL/dxi of this view, added onto the camera's gradient row
                pose_grad = torch.empty(6, dtype=torch.float32, device=dev)
                with torch.cuda.device(dev):
                    rc = _G().hg_camera_pose_grad_finish(
                        p._camera_pose.data_ptr(), p._camera_pose.size(0), pose_k, p.N, pose_ws.data_ptr(),
                        p.camera_pose_grad.data_ptr(), pose_grad.data_ptr(), torch.cuda.current_stream().cuda_stream)
                _lib.check(rc, "camera_pose_grad_finish")
        out = {"visibility_filter": visible, "radii": radii, "means2D_grad": g_means2D,
               "num_rendered": int(tR.num_rendered)}
        if pose_grad is not None:
            out["pose_grad"] = pose_grad
        if exp_off is not None:
            out["render"] = image
        if depth_l1 is not None:
            out["depth_l1"] = depth_l1
        return loss, out

    @staticmethod
    def _prologue_backward(p, radii, rs, g_xyz, g_feat, g_op, g_sc, g_rot, g_all_map, g_sc_extra, extra_scale,
                           pose_ws=None):
        """Gradients w.r.t. the activated parameters (+ dL/dall_map, + the scale regulariser's gradient) -> the raw
        parameters' rows of the gradient arena, dst = beta * dst + grad, rows with radii <= 0 skipped.  `pose_ws`: also
        sum the camera side of the all_map gradient there (hg_prologue_backward_pose)."""
        N = p.N
        if g_feat is not None and p._sink_used:  # (features also used outside the rasterizer: on top of the sink)
            p.grad_arena[p.slices["features"]].add_(g_feat.reshape(-1))
            g_feat = None
        if g_feat is None and not p._sink_used and not p._grad_dirty:  # no feature gradient at all in the first view
            g_feat = torch.zeros((N, 16, 3), dtype=torch.float32, device=p.param_arena.device)
        ptr = lambda t: t.contiguous().data_ptr() if t is not None else None  # noqa: E731
        d = {k: p.grad_arena[p.slices[k]] for k in ("xyz", "features", "opacity", "scaling", "rotation")}
        args = (p._scaling.data_ptr(), p._rotation.data_ptr(), p._opacity.data_ptr(), p._xyz.data_ptr(), N, 48,
                radii.data_ptr(), rs.viewmatrix.contiguous().data_ptr(), rs.campos.contiguous().data_ptr(),
                ptr(g_xyz), ptr(g_feat), ptr(g_op), ptr(g_sc), ptr(g_rot), ptr(g_all_map), ptr(g_sc_extra),
                ptr(extra_scale), 1.0 if p._grad_dirty else 0.0, d["xyz"].data_ptr(), d["features"].data_ptr(),
                d["opacity"].data_ptr(), d["scaling"].data_ptr(), d["rotation"].data_ptr())
        with torch.cuda.device(p.param_arena.device):
            st = torch.cuda.current_stream().cuda_stream
            if pose_ws is None:
                rc = _G().hg_prologue_backward(*args, st)
            else:
                rc = _G().hg_prologue_backward_pose(*args, pose_ws.data_ptr(), st)
        _lib.check(rc, "prologue_backward")
        p._grad_dirty = True
        p._sink_used = False

    def last_view_ms(self):
        """Device time of every view of the last step (needs `self.time_views = True` during that step; synchronises).
        The cost table for `balance_views` when the same views come round again: time is not exactly proportional to
        num_rendered (losses and per-Gaussian kernels are per view, list lengths matter)."""
        marks = getattr(self, "_view_marks", None)
        if not marks:
            return []
        marks[-1].synchronize()
        return [marks[i].elapsed_time(marks[i + 1]) for i in range(len(marks) - 1)]

    def step(self, views, total_views=None):
        """One optimiser step over this rank's `views` = [(camera, gt_image[, gt_ready_event]), ...]; returns the summed
        loss tensor."""
        if self.train_exposure:
            for view in views:  # an image without an exposure raises before the step has changed anything
                self.params.exposure_index(view[0].image_name)
        if self.depth_regularization:
            for view in views:  # a prior the step cannot use raises before the step has changed anything
                self._depth_prior(view[0])
        if self.train_poses:
            for view in views:  # an image without a pose raises before the step has changed anything
                self.params.camera_pose_index(view[0].image_name)
        self.iteration += 1
        timing = getattr(self, "timing", None)  # optional list: (start, views done, step done) CUDA events per step
        if timing is not None:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record()
        self.params.zero_grad()
        if self.train_exposure:
            p = self.params
            p.exposure_grad.zero_()  # (n x 48 bytes; the views add their sums into it)
            p._exposure.grad = p.exposure_grad
        if self.train_poses:
            p = self.params
            p.camera_pose_grad.zero_()  # (n x 32 bytes; the views add their gradients into it)
            p._camera_pose.grad = p.camera_pose_grad
        total = None
        self.last_view_costs = []
        # optional (`self.time_views = True`): one CUDA event per view boundary, read back by last_view_ms()
        marks = [torch.cuda.Event(enable_timing=True)] if getattr(self, "time_views", False) else None
        if marks is not None:
            marks[0].record()
        if self.sparse_adam:
            self.visible.zero_()
        self._in_step, self._step_activations = True, None
        for view in views:
            cam, gt = view[0], view[1]
            if getattr(self, "direct", False):
                loss, pkg = self.view_step_direct(cam, gt, self.iteration, view[2] if len(view) > 2 else None)
            else:
                loss, pkg = self.view_loss(cam, gt, self.iteration, view[2] if len(view) > 2 else None)
                loss.backward()
            total = loss.detach() if total is None else total + loss.detach()
            if self.sparse_adam:
                vf = pkg["visibility_filter"]
                if vf.dtype == torch.bool:  # mask form (no host sync): union by bitwise or
                    self.visible.bitwise_or_(vf.view(torch.uint8))
                else:
                    self.visible.index_fill_(0, vf, 1)
            if self.densification_stats:
                self._add_densification_stats(pkg)
            self.last_view_costs.append(pkg.get("num_rendered", 0) if isinstance(pkg, dict) else 0)
            if marks is not None:
                marks.append(torch.cuda.Event(enable_timing=True))
                marks[-1].record()
        self._view_marks = marks
        self._in_step, self._step_activations = False, None  # the optimiser is about to change the parameters
        if timing is not None:
            ev[1].record()
        self.params.begin_view()
        if self.params.fused and not self.params._grad_dirty:  # no view produced a gradient
            self.params.grad_arena.zero_()
        n_views = len(views)
        if self.world > 1:
            if self.params.exchange is not None:  # ONE kernel: multimem.ld_reduce + multimem.st through the NVSwitch
                self.params.exchange.all_reduce_()
            else:
                dist.all_reduce(self.params.grad_arena, op=dist.ReduceOp.SUM, group=self.group)
            if self.sparse_adam:  # union of the ranks' visible sets
                dist.all_reduce(self.visible, op=dist.ReduceOp.MAX, group=self.group)
            if self.train_exposure:
                dist.all_reduce(self.params.exposure_grad, op=dist.ReduceOp.SUM, group=self.group)
            if self.train_poses:
                dist.all_reduce(self.params.camera_pose_grad, op=dist.ReduceOp.SUM, group=self.group)
            if total_views is not None:
                n_views = total_views
            else:  # ranks may hold uneven shards of views[rank::world]: count what was really rendered
                cnt = torch.tensor([float(n_views)], device=self.params.grad_arena.device)
                dist.all_reduce(cnt, op=dist.ReduceOp.SUM, group=self.group)
                n_views = int(round(float(cnt.item())))
        if self.mcmc:  # the same arena on every rank after the exchange: the regulariser adds the same bits everywhere
            p, o = self.params, self.opt
            self.adam.lr["xyz"] = float(self.xyz_lr(self.iteration))
            if total is None:
                total = torch.zeros((), dtype=torch.float32, device=p.param_arena.device)
            mcmc_regularizer(p.param_arena, p.grad_arena, p.N, o.mcmc_opacity_reg, o.mcmc_scale_reg,
                             grad_mult=float(max(n_views, 1)), loss_mult=float(len(views)), loss=total,
                             workspace=self._mcmc_ws)
        self.adam.step(grad_scale=1.0 / max(n_views, 1), visible_mask=self.visible if self.sparse_adam else None)
        if self.train_exposure:
            self._exposure_adam_step(1.0 / max(n_views, 1))
        if self.train_poses:
            self._pose_adam_step(1.0 / max(n_views, 1))
        if getattr(self, "densify", False):
            self._density_schedule()
        if self.mcmc:
            self._mcmc_schedule()
        if timing is not None:
            ev[2].record()
            timing.append(ev)
        return total

    def _depth_prior(self, cam):
        """(invdepthmap, depth_mask or None) of the camera when it carries a reliable prior, else None.  ValueError
        for a prior this trainer cannot use: not a float32 [1, H, W] tensor at the camera's resolution on the
        parameters' device."""
        mono = getattr(cam, "invdepthmap", None)
        if mono is None or not getattr(cam, "depth_reliable", True):
            return None
        mask = getattr(cam, "depth_mask", None)
        shape = (1, int(cam.image_height), int(cam.image_width))
        dev = self.params.param_arena.device
        for what, t in (("invdepthmap", mono), ("depth_mask", mask)):
            if t is None:
                continue
            if not isinstance(t, torch.Tensor) or t.dtype != torch.float32 or tuple(t.shape) != shape:
                raise ValueError("camera %r: %s must be a float32 tensor of shape %s, got %s"
                                 % (getattr(cam, "image_name", None), what, shape,
                                    (t.dtype, tuple(t.shape)) if isinstance(t, torch.Tensor) else type(t)))
            if t.device != dev:
                raise ValueError("camera %r: %s is on %s, the parameters on %s"
                                 % (getattr(cam, "image_name", None), what, t.device, dev))
        return mono.contiguous(), mask.contiguous() if mask is not None else None

    def _depth_term(self, cam, iteration):
        """(mono, mask, w(iteration)) when the depth term applies to this view, else None."""
        if not self.depth_regularization:
            return None
        prior = self._depth_prior(cam)
        if prior is None:
            return None
        w = float(self.depth_l1_weight(iteration))
        return prior + (w,) if w != 0.0 else None

    def _depth_workspace(self, H, W, dev):
        """Workspace of hg_invdepth_l1, zero-filled once and grown when a larger image comes (the kernel leaves its
        counter at zero again after every call)."""
        need = int(lu._L().hg_invdepth_l1_workspace_bytes(H, W))
        if self._depth_ws is None or self._depth_ws.numel() < need:
            self._depth_ws = torch.zeros(need, dtype=torch.uint8, device=dev)
        return self._depth_ws

    def _exposure_workspace(self, H, W, dev):
        """Workspace of hg_training_image_grad_exposure, zero-filled once and grown when a larger image comes (the kernel
        leaves its counter at zero again after every call)."""
        need = int(lu._L().hg_exposure_grad_workspace_bytes(H, W))
        if self._exposure_ws is None or self._exposure_ws.numel() < need:
            self._exposure_ws = torch.zeros(need, dtype=torch.uint8, device=dev)
        return self._exposure_ws

    @torch.no_grad()
    def _exposure_adam_step(self, grad_scale):
        """hierarchical-3DGS's exposure_optimizer (torch.optim.Adam([_exposure]), eps 1e-8) with its lr set from
        exposure_scheduler_args(iteration): dense over the whole table (rows of images not in the step keep moving on
        their moments), its own step count, the gradient scaled by 1 / views as the Gaussians' is."""
        p = self.params
        if self.exposure_exp_avg.shape != p._exposure.shape:
            raise RuntimeError("the exposure table was replaced after the trainer was built (setup_exposures)")
        self.exposure_step_count += 1
        n = p._exposure.size(0)
        with torch.cuda.device(p.param_arena.device):
            rc = _G().hg_adam_step(p._exposure.data_ptr(), p.exposure_grad.data_ptr(), self.exposure_exp_avg.data_ptr(),
                                   self.exposure_exp_avg_sq.data_ptr(), n, 12, None, None, 0,
                                   float(self.exposure_lr(self.iteration)), 0.9, 0.999, 1e-8, self.exposure_step_count,
                                   float(grad_scale), 0, 0.0, torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, "adam_step")

    def _pose_workspace(self, N, dev):
        """Partial sums of the pose variants of the backward (hg_camera_pose_workspace_bytes(N)), grown with N; every
        byte the finish reads is written by the view's two kernels first."""
        need = int(_G().hg_camera_pose_workspace_bytes(N))
        if self._pose_ws is None or self._pose_ws.numel() < need:
            self._pose_ws = torch.empty(need, dtype=torch.uint8, device=dev)
        return self._pose_ws

    @torch.no_grad()
    def _pose_adam_step(self, grad_scale):
        """Adam over the whole pose table (torch.optim.Adam semantics, eps 1e-8, its own step count, the gradient
        scaled by 1 / views as the Gaussians' is): rho (the 3 head columns) at pose_lr_translation x spatial_lr_scale,
        phi at pose_lr_rotation; the pad columns have zero gradient and stay zero.  One launch."""
        p = self.params
        if self.pose_exp_avg.shape != p._camera_pose.shape:
            raise RuntimeError("the camera pose table was replaced after the trainer was built (setup_camera_poses)")
        self.pose_step_count += 1
        lr_t = float(self.opt.pose_lr_translation) * float(getattr(self.adam, "spatial_lr_scale", 1.0))
        with torch.cuda.device(p.param_arena.device):
            rc = _G().hg_adam_step(p._camera_pose.data_ptr(), p.camera_pose_grad.data_ptr(), self.pose_exp_avg.data_ptr(),
                                   self.pose_exp_avg_sq.data_ptr(), p._camera_pose.size(0), p._camera_pose.size(1), None,
                                   None, 0, float(self.opt.pose_lr_rotation), 0.9, 0.999, 1e-8, self.pose_step_count,
                                   float(grad_scale), 3, lr_t, torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, "adam_step")

    def _zero_densification_stats(self):
        dev, N = self.params.param_arena.device, self.params.N
        self.xyz_gradient_accum = torch.zeros((N, 1), device=dev)
        self.denom = torch.zeros((N, 1), device=dev)
        self.max_radii2D = torch.zeros(N, device=dev)

    @torch.no_grad()
    def densify_and_prune(self, max_grad, min_opacity, extent, max_screen_size=None, seed=None):
        """GaussianModel.densify_and_prune of graphdeco 3DGS over the arenas (DESIGN.md §3 "Densify and prune"): clone
        the small Gaussians whose gradient statistic reaches `max_grad`, split the large ones in two, prune the
        transparent ones (and, with `max_screen_size`, the ones larger than 0.1 `extent` in world space).  With several
        ranks the statistics are combined first (gradient and radius by MAX, visit count by SUM), so every rank makes
        the same decisions and draws the same children: the arenas stay bit-identical.  `seed` keys the split draws
        (default: the iteration).  Returns the counts of `densify_arenas` (cloned, split, pruned, n = N', ...); raises ValueError, leaving the model as
        it was, if no Gaussian would be left."""
        if not self.densification_stats:
            raise RuntimeError("densify_and_prune needs ViewShardedTrainer(densification_stats=True)")
        p = self.params
        if self.world > 1:
            dist.all_reduce(self.xyz_gradient_accum, op=dist.ReduceOp.MAX, group=self.group)
            dist.all_reduce(self.max_radii2D, op=dist.ReduceOp.MAX, group=self.group)
            dist.all_reduce(self.denom, op=dist.ReduceOp.SUM, group=self.group)
        new_p, new_m, new_v, counts = densify_arenas(
            p.param_arena, self.adam.exp_avg, self.adam.exp_avg_sq, p.N, self.xyz_gradient_accum.view(-1), max_grad,
            min_opacity, extent, max_screen_size, self.iteration if seed is None else seed,
            percent_dense=getattr(self.opt, "percent_dense", 0.01), skybox_points=p.skybox_points)
        p.resize(new_p, counts["n"])
        self.adam.resize(new_m, new_v)
        self.visible = torch.zeros(p.N, dtype=torch.uint8, device=new_p.device)
        self._zero_densification_stats()
        self._step_activations = None
        return counts

    @torch.no_grad()
    def reset_opacity(self):
        """GaussianModel.reset_opacity: opacity = min(opacity, 0.01) (through the logit), with that group's Adam moments
        zeroed (replace_tensor_to_optimizer); every other float of the arenas is left as it is."""
        p = self.params
        sl = p.slices["opacity"]
        with torch.cuda.device(p.param_arena.device):
            rc = _G().hg_reset_opacity(p.param_arena[sl].data_ptr(), self.adam.exp_avg[sl].data_ptr(),
                                       self.adam.exp_avg_sq[sl].data_ptr(), p.N, torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, "reset_opacity")
        p._act = None

    def _density_schedule(self):
        """graphdeco's train.py schedule, after the optimiser step of step `it`: densify every densification_interval
        steps in (densify_from_iter, densify_until_iter), with the size threshold 20 once the opacity has been reset;
        reset the opacity every opacity_reset_interval steps before densify_until_iter."""
        o, it = self.opt, self.iteration
        if it >= o.densify_until_iter:
            return
        if it > o.densify_from_iter and it % o.densification_interval == 0:
            self.densify_and_prune(o.densify_grad_threshold, o.min_opacity, self.scene_extent,
                                   20 if it > o.opacity_reset_interval else None)
        if it % o.opacity_reset_interval == 0:
            self.reset_opacity()

    def _require_mcmc(self, what):
        if not self.mcmc:
            raise RuntimeError("%s needs ViewShardedTrainer(mcmc=True, mcmc_cap_max=...)" % what)

    @torch.no_grad()
    def relocate_dead(self, seed=None):
        """3DGS-MCMC relocation in place: every dead Gaussian (opacity <= mcmc_min_opacity) becomes a copy of a live one
        drawn with probability proportional to its opacity, and the sources' opacity and scale are corrected (DESIGN.md
        §3 "MCMC densification").  The moments of sources and destinations are zeroed.  `seed` keys the draws (default:
        the iteration).  Returns dict(dead=, alive=) as int64 device scalars: nothing is read back."""
        self._require_mcmc("relocate_dead")
        p = self.params
        counts = mcmc_relocate_arenas(p.param_arena, self.adam.exp_avg, self.adam.exp_avg_sq, p.N,
                                      self.opt.mcmc_min_opacity, self.iteration if seed is None else seed,
                                      skybox_points=p.skybox_points, workspace=self._mcmc_ws)[3]
        p._act = None
        self._step_activations = None
        return counts

    @torch.no_grad()
    def grow(self, seed=None):
        """3DGS-MCMC growth: N' = min(mcmc_cap_max, int(mcmc_grow_factor N)) Gaussians, the new ones copies of rows drawn
        with probability proportional to opacity (sources and copies share the corrected opacity and scale; their
        moments start at zero).  Goes through GaussianParams.resize / ArenaAdam.resize, which re-create the gradient
        exchange (collectively across ranks); the visibility mask and the densification statistics start afresh.
        `seed` keys the draws (default: the iteration).  Returns dict(added=, n=) with host ints computed from N alone:
        nothing is read back.  At the cap nothing changes."""
        self._require_mcmc("grow")
        p = self.params
        n_target = mcmc_grow_target(p.N, self.mcmc_cap_max, self.opt.mcmc_grow_factor)
        if n_target <= p.N:
            return dict(added=0, n=p.N)
        new_p, new_m, new_v, counts = mcmc_grow_arenas(
            p.param_arena, self.adam.exp_avg, self.adam.exp_avg_sq, p.N, n_target, self.opt.mcmc_min_opacity,
            self.iteration if seed is None else seed, skybox_points=p.skybox_points, workspace=self._mcmc_ws)
        p.resize(new_p, counts["n"])
        self.adam.resize(new_m, new_v)
        self.visible = torch.zeros(p.N, dtype=torch.uint8, device=new_p.device)
        if self.densification_stats:
            self._zero_densification_stats()
        self._mcmc_ws = mcmc_workspace(p.N, new_p.device)
        self._step_activations = None
        return counts

    @torch.no_grad()
    def _mcmc_schedule(self):
        """gsplat MCMCStrategy.step_post_backward after the optimiser step of step `it`: relocate then grow when
        mcmc_refines(it), then position noise at lr_xyz(it) * mcmc_noise_lr on every step (past the refinement window
        too), keyed by the iteration."""
        it = self.iteration
        if mcmc_refines(it, self.opt):
            self.relocate_dead()
            self.grow()
        p = self.params
        mcmc_inject_noise(p.param_arena, p.N, self.adam.lr["xyz"] * self.opt.mcmc_noise_lr, seed=it,
                          skybox_points=p.skybox_points)
        p._act = None

    def _add_densification_stats(self, pkg):
        g = pkg["means2D_grad"] if "means2D_grad" in pkg else pkg["viewspace_points"].grad
        if g is None:
            return
        N = self.params.N
        if pkg["visibility_filter"].dtype == torch.bool:  # mask form: radii is already per Gaussian (0 where culled)
            radii_full = pkg["radii"].to(torch.int32).contiguous()
        else:
            radii_full = torch.zeros(N, dtype=torch.int32, device=g.device)
            radii_full[pkg["visibility_filter"]] = pkg["radii"]
        with torch.cuda.device(g.device):
            rc = _G().hg_densification_stats(g.contiguous().data_ptr(), radii_full.data_ptr(), N,
                                             self.xyz_gradient_accum.data_ptr(), self.denom.data_ptr(),
                                             self.max_radii2D.data_ptr(), torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, "densification_stats")
