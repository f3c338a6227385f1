"""GPU: monocular inverse-depth supervision (DESIGN.md §3 "Depth regularisation").  The kernel against torch, the
training step's direct executor against its autograd path, the step against the composition on the CPU rasterizer
oracle with the depth term added, the step without a usable prior against the step with the flag off, and the term
pulling a perturbed scene's depth towards the prior."""
import math

import pytest
import torch

from test_step_oracle_gpu import _EXPOSURES, OracleRaster, _oracle_view, _scene, _torch_adam, _views

pytestmark = pytest.mark.gpu


def _L():
    from hidegs_b200._losses_lib import lib
    return lib()


def _inputs(dev, H, W, seed):
    """inverse depth, a prior off by a mixed-sign residual (exactly equal at every 5th pixel), a mask with zeros,
    ones and fractions."""
    g = torch.Generator().manual_seed(seed)
    inv = torch.rand(1, H, W, generator=g) * 0.5 + 0.05
    mono = inv + 0.05 * torch.randn(1, H, W, generator=g)
    flat_inv, flat_mono = inv.view(-1), mono.view(-1)
    flat_mono[::5] = flat_inv[::5]
    mask = torch.rand(1, H, W, generator=g)
    mask[mask < 0.25] = 0.0
    mask[mask > 0.9] = 1.0
    return inv.to(dev), mono.to(dev), mask.to(dev)


def _run(inv, mono, mask, w, ws=None, loss=None):
    H, W = inv.shape[-2:]
    if ws is None:
        ws = torch.zeros(int(_L().hg_invdepth_l1_workspace_bytes(H, W)), dtype=torch.uint8, device=inv.device)
    grad = torch.empty_like(inv)
    value = torch.empty((), dtype=torch.float32, device=inv.device)
    rc = _L().hg_invdepth_l1(inv.data_ptr(), mono.data_ptr(), mask.data_ptr() if mask is not None else None, H, W, w,
                             grad.data_ptr(), value.data_ptr(), loss.data_ptr() if loss is not None else None,
                             ws.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert rc == 0, _L().hg_last_error()
    return grad, value


def _misaligned(t):
    """The same values in a view at storage offset 1 (4 bytes past a 16-byte boundary)."""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    return v


@pytest.mark.parametrize("HW", [(1, 1), (7, 13), (208, 320), (1080, 1920)])
@pytest.mark.parametrize("masked", [False, True])
def test_invdepth_l1_kernel_matches_torch(cuda_device, HW, masked):
    dev = cuda_device
    H, W = HW
    inv, mono, mask = _inputs(dev, H, W, seed=H * 7 + W)
    if not masked:
        mask = None
    w = 0.37
    grad, value = _run(inv, mono, mask, w)
    # value: 1e-6 relative of float64
    d64 = inv.double() - mono.double()
    if mask is not None:
        d64 = d64 * mask.double()
    want = float(d64.abs().mean())
    assert abs(float(value) - want) <= 1e-6 * want + 1e-30, (float(value), want)
    # gradient: the fp32 torch autograd formulation, within 1 ulp element by element, and the same sign pattern
    x = inv.clone().requires_grad_(True)
    d = (x - mono) * mask if mask is not None else x - mono
    (w * torch.abs(d).mean()).backward()
    ref = x.grad
    ulp = torch.nextafter(ref.abs(), torch.full_like(ref, math.inf)) - ref.abs()
    assert bool(((grad - ref).abs() <= ulp).all()), float((grad - ref).abs().max())
    assert torch.equal(torch.signbit(grad), torch.signbit(ref))
    zero = d.detach() == 0
    if mask is not None:
        zero |= mask == 0
    assert bool(zero.any()) and bool((grad[zero] == 0).all()) and not bool(torch.signbit(grad[zero]).any())
    assert bool((grad[~zero] != 0).all())
    # deterministic: a second call gives the same bits
    grad2, value2 = _run(inv, mono, mask, w)
    assert torch.equal(value2.view(torch.int32), value.view(torch.int32)) and torch.equal(grad2, grad)
    # loss_inout: += w * value, as torch's `loss + w * value` in fp32
    loss = torch.tensor(0.3125, device=dev)
    _g, v3 = _run(inv, mono, mask, w, loss=loss)
    assert float(loss) == float(torch.tensor(0.3125, device=dev) + torch.tensor(w, device=dev) * v3)
    _run(inv, mono, mask, w, loss=loss)
    assert float(loss) == float((torch.tensor(0.3125, device=dev) + torch.tensor(w, device=dev) * v3)
                                + torch.tensor(w, device=dev) * v3)
    # a workspace used at a larger size serves this one; misaligned views take the scalar path to the same result
    big = torch.zeros(int(_L().hg_invdepth_l1_workspace_bytes(1080, 1920)), dtype=torch.uint8, device=dev)
    bi, bm, bk = _inputs(dev, 1080, 1920, seed=99)
    _run(bi, bm, bk, 1.0, ws=big)
    grad4, value4 = _run(inv, mono, mask, w, ws=big)
    assert torch.equal(value4.view(torch.int32), value.view(torch.int32)) and torch.equal(grad4, grad)
    mi, mm = _misaligned(inv), _misaligned(mono)
    mk = _misaligned(mask) if mask is not None else None
    H, W = inv.shape[-2:]
    ws = torch.zeros(int(_L().hg_invdepth_l1_workspace_bytes(H, W)), dtype=torch.uint8, device=dev)
    mg = _misaligned(torch.zeros_like(inv))
    value5 = torch.empty((), dtype=torch.float32, device=dev)
    assert _L().hg_invdepth_l1(mi.data_ptr(), mm.data_ptr(), mk.data_ptr() if mk is not None else None, H, W, w,
                               mg.data_ptr(), value5.data_ptr(), None, ws.data_ptr(),
                               torch.cuda.current_stream().cuda_stream) == 0
    assert torch.equal(value5.view(torch.int32), value.view(torch.int32)) and torch.equal(mg, grad)
    # the autograd wrapper: the unweighted value, the kernel's gradient scaled by the upstream scalar
    from hidegs_b200 import loss_utils as lu
    y = inv.clone().requires_grad_(True)
    v = lu.inverse_depth_l1(y, mono, mask)
    assert torch.equal(v.detach().view(torch.int32), value.view(torch.int32))
    (w * v).backward()
    assert bool(((y.grad - ref).abs() <= 2 * ulp).all())


# ---------------------------------------------------------------------------------------------------------------------
# trainer
def _prior_maps(dev, sc, cams, sigma=0.08, seed=7):
    """Inverse depth of each camera rendered from a copy of the scene with its z positions perturbed (so the residual
    against the unperturbed scene's inverse depth is non-zero and of mixed sign)."""
    from hidegs_b200 import gaussian_renderer as gr, trainer as tr
    g = torch.Generator().manual_seed(seed)
    moved = dict(sc)
    moved["means3D"] = sc["means3D"].clone()
    moved["means3D"][:, 2] += sigma * torch.randn(sc["means3D"].size(0), generator=g)
    params = tr.GaussianParams.from_scene(moved, dev)
    with torch.no_grad():
        return [gr.render(c, params, tr.PipelineParams, torch.zeros(3, device=dev))["depth"].detach().clone()
                for c in cams]


def _fraction_mask(dev, H, W, seed=3):
    g = torch.Generator().manual_seed(seed)
    m = torch.rand(1, H, W, generator=g)
    m[m < 0.2] = 0.0
    return m.to(dev)


def _attach(cams, maps, dev, unreliable=()):
    """Reliable priors with a fractional mask on even cameras and without one on odd cameras; cameras in `unreliable`
    get depth_params whose scale is 100x the median (graphdeco's reliability test fails)."""
    from hidegs_b200.ply_io import attach_depth_prior
    for k, (c, m) in enumerate(zip(cams, maps)):
        H, W = m.shape[-2:]
        dp = dict(scale=100.0, offset=0.0, med_scale=1.0) if k in unreliable else None
        attach_depth_prior(c, m, dp, mask=_fraction_mask(dev, H, W, seed=k) if k % 2 == 0 else None)


def _setup(dev, n=30_000, W=320, H=208, ncams=3):
    from hidegs_b200 import synthetic as syn
    sc = syn.make_scene(n, seed=2, log_scale_mean=math.log(0.01 * 1920.0 / W))
    cams = []
    for k in range(ncams):
        c = syn.default_camera(W, H, eye=(0.3 * k - 0.3, 0.1 * k, -5.0)).to(dev)
        c.image_name = "img_%d" % k
        cams.append(c)
    g = torch.Generator().manual_seed(4)
    gts = [torch.nn.functional.avg_pool2d(torch.rand(1, 3, H, W, generator=g), 5, stride=1, padding=2)[0].clamp(0, 1).to(dev)
           for _ in cams]
    return sc, cams, gts


@pytest.mark.parametrize("cache_gt", [False, True])
def test_direct_executor_matches_autograd_with_depth(cuda_device, cache_gt):
    """view_step_direct against view_loss().backward() with the term on: same loss, depth value, visibility and
    gradient arena (the tolerance of test_direct_view_executor_matches_autograd); camera 2's prior is unreliable."""
    from hidegs_b200 import trainer as tr
    dev = cuda_device
    sc, cams, gts = _setup(dev)
    _attach(cams, _prior_maps(dev, sc, cams), dev, unreliable=(2,))
    out = {}
    for direct, depth in ((True, True), (False, True), (True, False)):
        params = tr.GaussianParams.from_scene(sc, dev)
        trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), cache_ground_truth=cache_gt,
                                        depth_regularization=depth)
        trainer.direct = direct
        params.zero_grad()
        losses, vis, dl = [], [], []
        for cam, gt in zip(cams, gts):
            if direct:
                loss, pkg = trainer.view_step_direct(cam, gt, 2000)
            else:
                loss, pkg = trainer.view_loss(cam, gt, 2000)
                loss.backward()
            losses.append(float(loss.detach()))
            vis.append(pkg["visibility_filter"].clone())
            dl.append(float(pkg["depth_l1"]) if "depth_l1" in pkg else None)
        out[(direct, depth)] = (params.grad_arena.clone(), losses, vis, dl)
    a, b, off = out[(True, True)], out[(False, True)], out[(True, False)]
    assert all(abs(x - y) <= 1e-6 * abs(y) + 1e-9 for x, y in zip(a[1], b[1])), (a[1], b[1])
    err = (a[0] - b[0]).abs().max().item()
    assert err <= 1e-5 * b[0].abs().max().item() + 1e-12, err
    assert all(torch.equal(x, y) for x, y in zip(a[2], b[2]))
    assert a[3][2] is None and b[3][2] is None  # the unreliable prior adds no term
    assert all(abs(x - y) <= 1e-6 * abs(y) for x, y in zip(a[3][:2], b[3][:2])), (a[3], b[3])
    # the premise: the term took part (weight w(2000) of the default schedule)
    from hidegs_b200.optim import get_expon_lr_func
    O = tr.OptimizationParams
    w = get_expon_lr_func(O.depth_l1_weight_init, O.depth_l1_weight_final, max_steps=O.iterations)(2000)
    for k in range(2):
        assert abs((a[1][k] - off[1][k]) - w * a[3][k]) <= 1e-5 * abs(a[1][k]), (a[1][k], off[1][k], a[3][k])
    assert a[1][2] == off[1][2]
    assert float((a[0] - off[0]).abs().max()) > 1e-3 * float(off[0].abs().max())


class _InjectGrad(torch.autograd.Function):
    """Identity on `color`; its backward also hands `g_inv` to `inv`, so the rasterizer's backward receives the depth
    term's gradient together with the image gradients."""

    @staticmethod
    def forward(ctx, color, inv, g_inv):
        ctx.g_inv = g_inv
        return color.clone()

    @staticmethod
    def backward(ctx, g):
        return g, ctx.g_inv, None


def _depth_oracle_raster(prior, record):
    """OracleRaster with the depth term: the oracle's inverse depth `_inv`, w * torch.abs((inv - mono) * mask).mean()
    on the host (torch CPU autograd), its value into `record`, its gradient back through the oracle's backward."""
    def raster(fa, *inputs):
        color, radii, obs, am, pd, inv = OracleRaster.apply(fa, *inputs)
        if prior is not None:
            mono, mask, w = prior
            inv_h = inv.detach().cpu().requires_grad_(True)
            d = inv_h - mono.cpu()
            if mask is not None:
                d = d * mask.cpu()
            value = torch.abs(d).mean()
            (w * value).backward()
            record.update(value=float(value.detach()), weighted=float(w * value.detach()))
            color = _InjectGrad.apply(color, inv, inv_h.grad.to(inv.device))
        return color, radii, obs, am, pd, inv
    return raster


@pytest.mark.parametrize("exposure", [False, True], ids=["plain", "exposure"])
def test_step_with_depth_vs_oracle(cuda_device, exposure):
    """One step over two views (a reliable prior with a fractional mask, and an unreliable prior) against the
    composition on the CPU oracle with the depth term: loss 1e-3, exact visibility sets, gradient arena 1e-3
    element-wise and 1e-4 relative L2 (single_view_weight = 0), the parameters after Adam; with train_exposure also
    the exposure gradient."""
    import raster_utils as ru
    from hidegs_b200 import trainer as tr
    dev = cuda_device
    sc = _scene()
    names = ["img_a", "img_b"]
    views = _views(dev, ((0.0, 0.0, -5.0), (0.3, 0.0, -5.0)), names=names)
    cams = [c for c, _ in views]
    maps = _prior_maps(dev, sc, cams, sigma=0.5)
    _attach(cams, maps, dev, unreliable=(1,))
    d0 = ((cams[0].invdepthmap - _prior_maps(dev, sc, cams[:1], sigma=0.0)[0]) * cams[0].depth_mask)
    assert bool((d0 > 0).any()) and bool((d0 < 0).any())  # the premise: a mixed-sign residual
    assert cams[0].depth_reliable and not cams[1].depth_reliable
    iteration = 2000
    opt = type("ImageTerms", (tr.OptimizationParams,), dict(single_view_weight=0.0))
    exposures = {k: torch.tensor(v, device=dev) for k, v in _EXPOSURES.items()} if exposure else None
    params = tr.GaussianParams.from_scene(sc, dev)
    if exposures is not None:
        params.setup_exposures(list(exposures), exposures=exposures)
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), opt=opt, start_iteration=iteration - 1,
                                    train_exposure=exposure, depth_regularization=True)
    names_g = [n for n, _ in tr.GROUPS]
    raw = {k: v.detach().clone() for k, v in params.leaves.items()}
    table = params._exposure.detach().clone() if exposure else None
    seen = []
    run_view = trainer.view_step_direct

    def recording(*a):
        loss, pkg = run_view(*a)
        seen.append((float(loss), pkg["visibility_filter"].clone(), pkg.get("depth_l1")))
        return loss, pkg
    trainer.view_step_direct = recording
    got_loss = float(trainer.step(views))
    assert seen[0][2] is not None and seen[1][2] is None
    w = float(trainer.depth_l1_weight(iteration))
    leaves = {k: v.clone().requires_grad_(True) for k, v in raw.items()}
    table_h = table.cpu().requires_grad_(True) if table is not None else None
    want_loss, vis = 0.0, []
    for (cam, gt), (view_loss, view_vis, view_dl) in zip(views, seen):
        prior = trainer._depth_prior(cam)
        record = {}
        e = table_h[params.exposure_index(cam.image_name)] if table_h is not None else None
        loss, visible, _info = _oracle_view(leaves, cam, gt, torch.zeros(3, device=dev), dev, iteration, opt,
                                            _depth_oracle_raster(prior + (w,) if prior is not None else None, record),
                                            3, e)
        loss += record.get("weighted", 0.0)
        if view_dl is not None:
            assert abs(float(view_dl) - record["value"]) <= 1e-3 * record["value"], (float(view_dl), record)
            assert record["weighted"] > 0.01 * loss, record  # the premise: the term is a visible part of the loss
        assert torch.equal(view_vis, visible)
        assert abs(view_loss - loss) <= 1e-3 * abs(loss), (view_loss, loss)
        want_loss += loss
        vis.append(visible)
    assert abs(got_loss - want_loss) <= 1e-3 * abs(want_loss), (got_loss, want_loss)
    ours = [params.grad_arena[params.slices[n]].view(raw[n].shape) for n in names_g]
    theirs = [leaves[n].grad for n in names_g]
    ru.assert_grads_close(ours, theirs, names=names_g, what="composed step with the depth term", l2_tol=1e-4)
    # Adam on the union of the visible rows, gradients scaled by 1 / views
    scale = 0.5
    rows = torch.stack(vis).any(0)
    lrs = dict(xyz=opt.position_lr_init, opacity=opt.opacity_lr, scaling=opt.scaling_lr, rotation=opt.rotation_lr)
    for n, g in zip(names_g, theirs):
        g = g * scale
        if n == "features":
            stepped = torch.cat([_torch_adam(raw[n][:, :1], g[:, :1], opt.feature_lr, 1e-15),
                                 _torch_adam(raw[n][:, 1:], g[:, 1:], opt.feature_lr / 20.0, 1e-15)], 1)
        else:
            stepped = _torch_adam(raw[n], g, lrs[n], 1e-15)
        want = torch.where(rows.view(-1, *([1] * (stepped.dim() - 1))), stepped, raw[n])
        got = params.leaves[n].detach()
        assert torch.equal(got[~rows], raw[n][~rows]), n
        diff = (got - want).abs()
        lr = opt.feature_lr if n == "features" else lrs[n]
        assert float((diff > 0.05 * lr).float().mean()) <= 2e-3, (n, float(diff.max()))
        assert float(diff.max()) <= 2.0 * lr * 1.0001 + 1e-12, (n, float(diff.max()))
    if exposure:
        ru.assert_grads_close([params.exposure_grad.clone()], [table_h.grad.to(dev)], names=("exposure",),
                              what="composed step with the depth term, exposure gradient")


@pytest.mark.parametrize("case", ["no_prior", "unreliable", "zero_weight"])
def test_no_usable_prior_runs_the_plain_step(cuda_device, case, monkeypatch):
    """With depth_regularization=True, views without a prior, views with unreliable priors, and a step with w(it) = 0
    run the code the flag-off step runs: the depth kernel is never launched and the rasterizer's backward gets no
    inverse-depth gradient (so it keeps its no-depth kernels).  Loss and visibility are bit-identical to the flag-off
    step; the gradient arena and the parameters agree to the blend backward's float-atomic order, which differs from
    run to run of the same step."""
    from hidegs_b200 import loss_utils as lu, trainer as tr
    from hidegs_b200.diff_gaussian_rasterization import _RasterizeGaussians
    dev = cuda_device
    sc, cams, gts = _setup(dev, ncams=2)
    if case != "no_prior":
        _attach(cams, _prior_maps(dev, sc, cams), dev, unreliable=(0, 1) if case == "unreliable" else ())

    class ZeroWeight(tr.OptimizationParams):
        depth_l1_weight_init = depth_l1_weight_final = 0.0
    launches, depth_grads = [], []
    real_launch, real_bwd = lu._invdepth_l1_launch, _RasterizeGaussians.backward
    monkeypatch.setattr(lu, "_invdepth_l1_launch", lambda *a: launches.append(1) or real_launch(*a))
    monkeypatch.setattr(_RasterizeGaussians, "backward",
                        staticmethod(lambda ctx, *g: depth_grads.append(g[-1]) or real_bwd(ctx, *g)))
    res = {}
    for on in (False, True):
        params = tr.GaussianParams.from_scene(sc, dev)
        trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), start_iteration=1500,
                                        opt=ZeroWeight if case == "zero_weight" else tr.OptimizationParams,
                                        depth_regularization=on)
        vis = []
        run_view = trainer.view_step_direct

        def recording(*a):
            loss, pkg = run_view(*a)
            assert "depth_l1" not in pkg
            vis.append(pkg["visibility_filter"].clone())
            return loss, pkg
        trainer.view_step_direct = recording
        loss = trainer.step(list(zip(cams, gts)))
        res[on] = (loss.clone(), params.grad_arena.clone(), params.param_arena.clone(), vis)
    assert not launches and len(depth_grads) == 4 and all(g is None for g in depth_grads)
    (l0, g0, p0, v0), (l1, g1, p1, v1) = res[False], res[True]
    assert torch.equal(l0.view(torch.int32), l1.view(torch.int32))
    assert all(torch.equal(a, b) for a, b in zip(v0, v1))
    assert float((g1 - g0).abs().max()) <= 1e-5 * float(g0.abs().max())
    diff = (p1 - p0).abs()
    assert float((diff > 1e-3).float().mean()) <= 1e-3 and float(diff.median()) <= 1e-6


def test_depth_term_pulls_depth_towards_the_prior(cuda_device):
    """Start from the scene with its z positions perturbed; ground truth images and priors come from the unperturbed
    scene.  After the same steps, the rendered inverse depth's masked L1 to the priors has fallen further with the
    term than without it."""
    from hidegs_b200 import gaussian_renderer as gr, synthetic as syn, trainer as tr
    dev = cuda_device
    W, H = 240, 160
    sc = syn.make_scene(30_000, seed=2, log_scale_mean=math.log(0.01 * 1920.0 / W))
    cams = []
    for k in range(4):
        c = syn.default_camera(W, H, eye=(0.4 * (k % 2) - 0.2, 0.3 * (k // 2) - 0.15, -5.0)).to(dev)
        c.image_name = "v%d" % k
        cams.append(c)
    truth = tr.GaussianParams.from_scene(sc, dev)
    with torch.no_grad():
        outs = [gr.render(c, truth, tr.PipelineParams, torch.zeros(3, device=dev)) for c in cams]
    gts = [o["render"].detach().contiguous() for o in outs]
    _attach(cams, [o["depth"].detach().clone() for o in outs], dev)
    g = torch.Generator().manual_seed(5)
    moved = dict(sc)
    moved["means3D"] = sc["means3D"].clone()
    moved["means3D"][:, 2] += 0.15 * torch.randn(sc["means3D"].size(0), generator=g)

    class Opt(tr.OptimizationParams):
        position_lr_init = 2e-3

    def depth_error(params):
        with torch.no_grad():
            total = 0.0
            for c in cams:
                inv = gr.render(c, params, tr.PipelineParams, torch.zeros(3, device=dev))["depth"]
                d = inv - c.invdepthmap
                total += float((d * c.depth_mask).abs().mean() if c.depth_mask is not None else d.abs().mean())
            return total / len(cams)
    err = {}
    for on in (False, True):
        params = tr.GaussianParams.from_scene(moved, dev)
        e0 = depth_error(params)
        trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), opt=Opt, depth_regularization=on)
        views = list(zip(cams, gts))
        for _ in range(100):
            trainer.step(views)
        err[on] = (e0, depth_error(params))
    print("depth L1 to the priors: start %.6g; after 100 steps without the term %.6g, with it %.6g"
          % (err[True][0], err[False][1], err[True][1]))
    # measured on an NVIDIA B200 (power limit 1000 W): start 7.44e-3; after 100 steps 3.77e-3 without the term and
    # 7.29e-4 with it
    assert err[True][0] == err[False][0]
    assert err[True][1] < err[False][1] and err[True][1] < err[True][0]
