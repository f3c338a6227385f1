"""GPU: the view-sharded training step (hidegs_b200/trainer.py): gradient arena == sum of per-view autograd gradients,
arena Adam == the reference optimiser's arithmetic per parameter group, loss goes down on a fixed view."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _setup(dev, n=30_000, W=320, H=208):
    from hidegs_b200 import synthetic as syn, trainer as tr
    sc = syn.make_scene(n, seed=2, log_scale_mean=math.log(0.01 * 1920.0 / W))
    cams = [syn.default_camera(W, H, eye=(dx, 0.0, -5.0)).to(dev) for dx in (0.0, 0.3)]
    g = torch.Generator().manual_seed(4)
    gts = [torch.nn.functional.avg_pool2d(torch.rand(1, 3, H, W, generator=g), 5, stride=1, padding=2)[0].clamp(0, 1).to(dev)
           for _ in cams]
    return sc, cams, gts, tr


def test_gradient_arena_accumulates_views(cuda_device):
    dev = cuda_device
    sc, cams, gts, tr = _setup(dev)
    params = tr.GaussianParams.from_scene(sc, dev)
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev))
    params.zero_grad()
    for cam, gt in zip(cams, gts):
        loss, _ = trainer.view_loss(cam, gt, 2000)
        loss.backward()
    arena = params.grad_arena.clone()
    # the leaves' .grad must still alias the arena
    for name, leaf in params.leaves.items():
        assert leaf.grad.data_ptr() == params.grad_arena[params.slices[name]].data_ptr(), name
    # independent evaluation: fresh parameters, one view at a time, gradients summed by hand
    total = torch.zeros_like(arena)
    for cam, gt in zip(cams, gts):
        p2 = tr.GaussianParams.from_scene(sc, dev)
        t2 = tr.ViewShardedTrainer(p2, torch.zeros(3, device=dev))
        loss, _ = t2.view_loss(cam, gt, 2000)
        loss.backward()
        total += p2.grad_arena
    err = (arena - total).abs().max().item()
    # two evaluations of the same view differ by the order of the backward blend's float atomics (~1e-6 relative)
    assert err <= 1e-5 * total.abs().max().item() + 1e-12, err
    assert arena.abs().max().item() > 0


def test_arena_adam_matches_per_group_reference_adam(cuda_device):
    from hidegs_b200.optim import Adam
    dev = cuda_device
    sc, cams, gts, tr = _setup(dev, n=5000)
    params = tr.GaussianParams.from_scene(sc, dev)
    adam = tr.ArenaAdam(params)
    o = tr.OptimizationParams
    # reference layout: separate tensors per group, features split in dc / rest with lr / 20 (gaussian_model.py training_setup)
    ref = {k: v.detach().clone() for k, v in params.leaves.items()}
    f_dc = torch.nn.Parameter(ref["features"][:, :1].contiguous())
    f_rest = torch.nn.Parameter(ref["features"][:, 1:].contiguous())
    leaves = {k: torch.nn.Parameter(ref[k]) for k in ("xyz", "opacity", "scaling", "rotation")}
    opt = Adam([{"params": [leaves["xyz"]], "lr": o.position_lr_init}, {"params": [f_dc], "lr": o.feature_lr},
                {"params": [f_rest], "lr": o.feature_lr / 20.0}, {"params": [leaves["opacity"]], "lr": o.opacity_lr},
                {"params": [leaves["scaling"]], "lr": o.scaling_lr}, {"params": [leaves["rotation"]], "lr": o.rotation_lr}],
               lr=0.0, eps=1e-15)
    g = torch.Generator().manual_seed(8)
    for s in range(3):
        grads = torch.randn(params.grad_arena.numel(), generator=g).to(dev) * 0.01
        params.grad_arena.copy_(grads)
        for k in leaves:
            leaves[k].grad = params.leaves[k].grad.clone() * 0.5
        f_dc.grad = params.leaves["features"].grad[:, :1].contiguous() * 0.5
        f_rest.grad = params.leaves["features"].grad[:, 1:].contiguous() * 0.5
        adam.step(grad_scale=0.5)
        opt.step()
    for k in leaves:
        a, b = params.leaves[k].detach(), leaves[k].detach()
        assert (a - b).abs().max().item() <= 1e-6 * b.abs().max().item(), k
    a = params.leaves["features"].detach()
    assert (a[:, :1] - f_dc.detach()).abs().max().item() <= 2e-6 * f_dc.abs().max().item()
    assert (a[:, 1:] - f_rest.detach()).abs().max().item() <= 1e-6 * f_rest.abs().max().item()


def test_training_reduces_loss(cuda_device):
    dev = cuda_device
    sc, cams, gts, tr = _setup(dev)
    params = tr.GaussianParams.from_scene(sc, dev)
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), start_iteration=1500)  # past the warm-up
    views = list(zip(cams, gts))
    losses = [float(trainer.step(views).item()) for _ in range(12)]
    assert np.isfinite(losses).all()
    assert losses[-1] < losses[0], losses


def test_sparse_arena_adam_and_densification_stats(cuda_device):
    """Rows outside the visibility mask keep parameters AND moments (OurAdam.step(relevant)); densification statistics
    follow GaussianModel.add_densification_stats (max of the screen-space gradient norm, denom += 1) and the
    max_radii2D update of the training loop."""
    from hidegs_b200._geometry_lib import lib as G
    dev = cuda_device
    sc, cams, gts, tr = _setup(dev, n=5000)
    params = tr.GaussianParams.from_scene(sc, dev)
    adam = tr.ArenaAdam(params)
    before = params.param_arena.clone()
    g = torch.Generator().manual_seed(3)
    params.grad_arena.copy_(torch.randn(params.grad_arena.numel(), generator=g).to(dev) * 0.01)
    mask = (torch.rand(params.N, generator=g) < 0.3).to(dev)
    adam.step(visible_mask=mask)
    for name, w in tr.GROUPS:
        sl = params.slices[name]
        a, b = params.param_arena[sl].view(params.N, w), before[sl].view(params.N, w)
        assert torch.equal(a[~mask], b[~mask]), name
        assert not adam.exp_avg[sl].view(params.N, w)[~mask].any()
        assert (a[mask] != b[mask]).any()
    # reference arithmetic on the masked rows (dense torch Adam on a copy restricted to the rows)
    sl = params.slices["xyz"]
    ref = torch.nn.Parameter(before[sl].view(params.N, 3)[mask].clone())
    ref.grad = params.grad_arena[sl].view(params.N, 3)[mask].clone()
    torch.optim.Adam([ref], lr=tr.OptimizationParams.position_lr_init, eps=1e-15).step()
    got = params.param_arena[sl].view(params.N, 3)[mask]
    assert (got - ref.detach()).abs().max().item() <= 1e-6 * ref.abs().max().item()
    # densification statistics
    N = 1000
    grad = torch.randn(N, 3, generator=g).to(dev)
    radii = torch.randint(-1, 30, (N,), generator=g, dtype=torch.int32).to(dev)
    accum = torch.rand(N, 1, generator=g).to(dev) * 0.5
    denom = torch.zeros(N, 1, device=dev)
    maxr = torch.full((N,), 5.0, device=dev)
    a0, m0 = accum.clone(), maxr.clone()
    rc = G().hg_densification_stats(grad.data_ptr(), radii.data_ptr(), N, accum.data_ptr(), denom.data_ptr(), maxr.data_ptr(),
                                    torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    f = radii > 0
    want = a0.clone()
    want[f] = torch.max(torch.norm(grad[f, :2], dim=-1, keepdim=True), a0[f])   # gaussian_model.py:764
    assert torch.allclose(accum, want, rtol=1e-6, atol=0)
    assert torch.equal(denom[:, 0], f.float())
    wr = m0.clone()
    wr[f] = torch.max(m0[f], radii[f].float())
    assert torch.equal(maxr, wr)


def test_sh_sink_matches_the_autograd_path(cuda_device):
    """The SH gradient accumulated by the rasterizer's backward kernel (sink) equals what autograd + AccumulateGrad
    produce, over two views, also when the features are used outside the rasterizer as well."""
    dev = cuda_device
    sc, cams, gts, tr = _setup(dev)
    arenas = {}
    for use_sink in (True, False):
        params = tr.GaussianParams.from_scene(sc, dev)
        params.sh_sink = use_sink
        trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev))
        params.zero_grad()
        for cam, gt in zip(cams, gts):
            loss, _ = trainer.view_loss(cam, gt, 2000)
            loss = loss + 1e-3 * (params.get_features ** 2).sum()  # a second consumer of the same features tensor
            loss.backward()
        arenas[use_sink] = params.grad_arena.clone()
    a, b = arenas[True], arenas[False]
    err = (a - b).abs().max().item()
    assert err <= 1e-5 * b.abs().max().item() + 1e-12, err
    sl = tr.GaussianParams.from_scene(sc, dev).slices["features"]
    assert b[sl].abs().max().item() > 0


@pytest.mark.parametrize("cache_gt", [False, True])
def test_direct_view_executor_matches_autograd(cuda_device, cache_gt):
    """The autograd-free executor of a view (ViewShardedTrainer.view_step_direct) runs the same kernels in the same
    order as the autograd path: same loss value, same gradient arena (up to the blend's float-atomic order), same
    visibility set and means2D gradient, over two accumulated views; then whole optimiser steps agree too."""
    dev = cuda_device
    sc, cams, gts, tr = _setup(dev)
    out = {}
    for direct in (True, False):
        params = tr.GaussianParams.from_scene(sc, dev)
        trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), cache_ground_truth=cache_gt,
                                        densification_stats=True)
        trainer.direct = direct
        params.zero_grad()
        losses, vis, g2d = [], [], []
        for cam, gt in zip(cams, gts):
            if direct:
                loss, pkg = trainer.view_step_direct(cam, gt, 2000)
                g2d.append(pkg["means2D_grad"].clone())
            else:
                loss, pkg = trainer.view_loss(cam, gt, 2000)
                loss.backward()
                g2d.append(pkg["viewspace_points"].grad.clone())
            losses.append(float(loss.detach()))
            vis.append(pkg["visibility_filter"].clone())
        out[direct] = (params.grad_arena.clone(), losses, vis, g2d)
    a, b = out[True], out[False]
    assert all(abs(x - y) <= 1e-6 * abs(y) + 1e-9 for x, y in zip(a[1], b[1])), (a[1], b[1])
    err = (a[0] - b[0]).abs().max().item()
    assert err <= 1e-5 * b[0].abs().max().item() + 1e-12, err
    assert all(torch.equal(x, y) for x, y in zip(a[2], b[2]))
    for x, y, v in zip(a[3], b[3], a[2]):
        # (the executor's rasterizer backward leaves the rows of culled Gaussians unwritten — HG_BWD_SKIP_CULLED_ROWS:
        # every consumer masks by radii — so only the rendered rows are defined; the autograd path holds zeros there)
        assert float(y[~v].abs().max()) == 0.0
        assert (x[v] - y[v]).abs().max().item() <= 1e-5 * y.abs().max().item() + 1e-12
    # three full steps (Adam included): parameters stay together
    arenas = {}
    for direct in (True, False):
        params = tr.GaussianParams.from_scene(sc, dev)
        trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), cache_ground_truth=cache_gt,
                                        start_iteration=1500)
        trainer.direct = direct
        for _ in range(3):
            trainer.step(list(zip(cams, gts)))
        arenas[direct] = params.param_arena.clone()
    # (Adam divides by sqrt(v) with eps = 1e-15: where a gradient is at the blend's atomic-order noise level the update
    # of a single element may differ by ~lr, so the bulk is compared tightly and the tail loosely)
    diff = (arenas[True] - arenas[False]).abs()
    assert float((diff > 1e-3).float().mean()) <= 1e-3 and float(diff.median()) <= 1e-6, \
        (float((diff > 1e-3).float().mean()), float(diff.median()), float(diff.max()))


def test_gaussian_count_not_multiple_of_four(cuda_device):
    """The arenas pad every parameter group to 16 bytes: a step with N = 4k + 1 Gaussians runs on the fused path and
    matches the autograd path."""
    dev = cuda_device
    sc, cams, gts, tr = _setup(dev, n=30_001)
    arenas = {}
    for direct in (True, False):
        params = tr.GaussianParams.from_scene(sc, dev)
        assert params.fused and all(params.slices[n].start % 4 == 0 for n, _ in tr.GROUPS)
        trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), start_iteration=1500)
        trainer.direct = direct
        trainer.step(list(zip(cams, gts)))
        arenas[direct] = (params.grad_arena.clone(), params.param_arena.clone())
    err = (arenas[True][0] - arenas[False][0]).abs().max().item()
    # (two evaluations of the SAME path differ by ~1.6e-5 of the largest entry here: float-atomic order of the blend)
    assert err <= 1e-4 * arenas[False][0].abs().max().item() + 1e-12, err
    assert torch.isfinite(arenas[True][1]).all()
