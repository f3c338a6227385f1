"""GPU: per-image exposure in the training step — hg_exposure_apply / hg_training_image_grad_exposure against float64
torch, the identity fast path against hg_training_image_grad and the plain trainer, the autograd-free executor against
the autograd path (render(..., use_trained_exp=True)), the exposure Adam against torch.optim.Adam, a run that recovers
known exposures, the public interfaces, and two or more ranks (tools/exposure_probe.py --check)."""
import copy
import json
import math
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------------
# kernels
def _L():
    from hidegs_b200 import loss_utils as lu
    return lu._L()


def _f32(x):
    return x.to(torch.float32).to(torch.float64)


def _exposed_f32(c, E):
    """The kernels' fma chain, each fma rounded once to fp32 (a product of two fp32 is exact in fp64)."""
    c = c.double()
    E = E.double()
    out = []
    for ch in range(3):
        x = _f32(c[2] * E[2, ch] + E[ch, 3])
        x = _f32(c[1] * E[1, ch] + x)
        out.append(_f32(c[0] * E[0, ch] + x))
    return torch.stack(out)


def _inputs(dev, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    n = 3 * H * W
    color = torch.rand(3, H, W, generator=g) * 1.2 - 0.1
    E = torch.eye(3, 4) + 0.1 * torch.randn(3, 4, generator=g)
    # channel 0 passes colour 0 straight through (column 0 = e_0, no offset), so pixels exactly on 0 and 1 exist
    E[:, 0] = torch.tensor([1.0, 0.0, 0.0])
    E[0, 3] = 0.0
    flat = color[0].view(-1)
    flat[::7] = 0.0
    flat[3::11] = 1.0
    gt = torch.rand(3, H, W, generator=g)
    gt[0].view(-1)[::13] = color[0].view(-1)[::13].clamp(0, 1)  # d == 0: zero L1 sign
    gs = torch.randn(3, H, W, generator=g) / n
    gf = torch.randn(3, H, W, generator=g) / n
    return [t.to(dev).contiguous() for t in (color, E, gt, gs, gf)]


def _run_grad(color, E, gt, gs, gf, wf, eg, ws, out=None, w_l1=0.8, w_ssim=-0.2):
    H, W = color.shape[1:]
    out = torch.empty_like(color) if out is None else out
    ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
    rc = _L().hg_training_image_grad_exposure(color.data_ptr(), E.data_ptr(), gt.data_ptr(), ptr(gs), ptr(gf), H, W,
                                              w_l1, w_ssim, ptr(wf), out.data_ptr(), eg.data_ptr(), ws.data_ptr(),
                                              torch.cuda.current_stream().cuda_stream)
    assert rc == 0, _L().hg_last_error()
    return out


def _ws(H, W, dev):
    return torch.zeros(int(_L().hg_exposure_grad_workspace_bytes(H, W)), dtype=torch.uint8, device=dev)


@pytest.mark.parametrize("terms", ["ssim+freq", "none", "ssim"])
@pytest.mark.parametrize("HW", [(37, 53), (151, 203)])
def test_exposure_kernels_match_float64(cuda_device, terms, HW):
    dev = cuda_device
    H, W = HW
    color, E, gt, gs, gf = _inputs(dev, H, W, seed=H + W)
    if terms == "none":
        gs = gf = None
    elif terms == "ssim":
        gf = None
    wf = torch.tensor(0.37, device=dev) if gf is not None else None
    n = 3 * H * W
    # image
    img = torch.empty_like(color)
    rc = _L().hg_exposure_apply(color.data_ptr(), E.data_ptr(), H, W, img.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    c64, E64 = color.double(), E.double()
    e64 = torch.einsum("chw,cd->dhw", c64, E64[:, :3]) + E64[:, 3, None, None]
    assert (img.double() - e64.clamp(0, 1)).abs().max().item() <= 1e-6
    e32 = _exposed_f32(color, E)
    assert torch.equal(img.double(), e32.clamp(0, 1))
    outside = float(((e32 < 0) | (e32 > 1)).double().mean())
    assert 0.1 <= outside <= 0.3, outside
    assert bool((e32[0] == 0).any()) and bool((e32[0] == 1).any())
    # gradient
    eg = torch.zeros(3, 4, device=dev)
    ws = _ws(H, W, dev)
    out = _run_grad(color, E, gt, gs, gf, wf, eg, ws)
    gate = (e32 >= 0) & (e32 <= 1)
    d = (e32.clamp(0, 1).float() - gt).double()  # the sign of the fp32 difference, as the kernel forms it
    g = torch.sign(d) * (0.8 / n)
    mag = g.abs()  # size of the terms (a sum of terms of either sign is held to their size, not to the result's)
    if gs is not None:
        g = g - 0.2 * gs.double()
        mag = mag + 0.2 * gs.double().abs()
    if gf is not None:
        g = g + 0.37 * gf.double()
        mag = mag + 0.37 * gf.double().abs()
    ge = torch.where(gate, g, torch.zeros_like(g))
    mag = torch.where(gate, mag, torch.zeros_like(mag))
    ref = torch.einsum("cd,dhw->chw", E64[:, :3], ge)
    scale = torch.einsum("cd,dhw->chw", E64[:, :3].abs(), mag)
    # The fp32 kernel rounds every term of a sum whose terms have either sign, so its error is a fraction of the terms'
    # size, not of the result's: held to 1e-6 of the terms' size everywhere, and to 1e-6 of the result itself where
    # the terms do not cancel (|ref| at least half their size)
    err_out = (out.double() - ref).abs()
    assert bool((err_out <= 1e-6 * scale + 1e-30).all())
    plain = ref.abs() >= 0.5 * scale
    assert bool(plain.any()) and bool((err_out[plain] <= 1e-6 * ref.abs()[plain]).all())
    assert bool((out[:, ~gate.any(0)] == 0).all())  # a pixel with all three gates shut has no gradient
    ref_eg = torch.zeros(3, 4, dtype=torch.float64, device=dev)
    sabs = torch.zeros(3, 4, dtype=torch.float64, device=dev)
    for c in range(3):
        for ch in range(3):
            ref_eg[c, ch] = (c64[c] * ge[ch]).sum()
            sabs[c, ch] = (c64[c].abs() * mag[ch]).sum()
        ref_eg[c, 3] = ge[c].sum()
        sabs[c, 3] = mag[c].sum()
    # the same for the exposure sums: 1e-6 of the terms' size everywhere (entries that nearly cancel), plain 1e-5
    # relative where the sum is at least a tenth of its terms' size
    err = (eg.double() - ref_eg).abs()
    assert bool((err <= 1e-5 * ref_eg.abs() + 1e-6 * sabs).all()), (err, ref_eg)
    plain = ref_eg.abs() >= 0.1 * sabs
    assert bool(plain.any()) and bool((err[plain] <= 1e-5 * ref_eg.abs()[plain]).all()), (err, ref_eg)
    # deterministic, and added onto what is there
    eg2 = torch.zeros(3, 4, device=dev)
    _run_grad(color, E, gt, gs, gf, wf, eg2, ws)
    assert torch.equal(eg.view(torch.int32), eg2.view(torch.int32))
    _run_grad(color, E, gt, gs, gf, wf, eg2, ws)
    assert torch.equal(eg2, 2 * eg)
    # out may alias g_ssim (the trainer's use)
    if gs is not None:
        alias = gs.clone()
        eg3 = torch.zeros(3, 4, device=dev)
        _run_grad(color, E, gt, alias, gf, wf, eg3, ws, out=alias)
        assert torch.equal(alias.view(torch.int32), out.view(torch.int32)) and torch.equal(eg3, eg)


def test_identity_exposure_is_bitwise_the_plain_gradient(cuda_device):
    dev = cuda_device
    H, W = 121, 167
    color, _E, gt, gs, gf = _inputs(dev, H, W, seed=5)
    E = torch.eye(3, 4, device=dev)
    wf = torch.tensor(0.37, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    img = torch.empty_like(color)
    assert _L().hg_exposure_apply(color.data_ptr(), E.data_ptr(), H, W, img.data_ptr(), st) == 0
    assert torch.equal(img, color.clamp(0, 1))
    for with_terms in (True, False):
        a_s, a_f = (gs, gf) if with_terms else (None, None)
        ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
        plain = torch.empty_like(color)
        assert _L().hg_training_image_grad(color.data_ptr(), gt.data_ptr(), ptr(a_s), ptr(a_f), color.numel(), 0.8, -0.2,
                                           ptr(wf) if a_f is not None else None, plain.data_ptr(), st) == 0
        eg = torch.zeros(12, device=dev)
        out = _run_grad(color, E, gt, a_s, a_f, wf if a_f is not None else None, eg, _ws(H, W, dev))
        assert torch.equal(out.view(torch.int32), plain.view(torch.int32))


# ---------------------------------------------------------------------------------------------------------------------
# trainer
def _setup(dev, n=30_000, W=320, H=208, names=("img_a", "img_b", "img_c")):
    from hidegs_b200 import synthetic as syn, trainer as tr
    sc = syn.make_scene(n, seed=2, log_scale_mean=math.log(0.01 * 1920.0 / W))
    cams = []
    for k, name in enumerate(names):
        c = syn.default_camera(W, H, eye=(0.3 * k - 0.3, 0.1 * k, -5.0)).to(dev)
        c.image_name = name
        cams.append(c)
    g = torch.Generator().manual_seed(4)
    gts = [torch.nn.functional.avg_pool2d(torch.rand(1, 3, H, W, generator=g), 5, stride=1, padding=2)[0].clamp(0, 1).to(dev)
           for _ in cams]
    return sc, cams, gts, tr


def _exposures(names, seed, dev):
    g = torch.Generator().manual_seed(seed)
    return {n: (torch.eye(3, 4) + 0.05 * torch.randn(3, 4, generator=g)).to(dev) for n in names}


def test_identity_exposure_step_matches_plain_step(cuda_device):
    dev = cuda_device
    sc, cams, gts, tr = _setup(dev)
    res = {}
    for on in (False, True):
        params = tr.GaussianParams.from_scene(sc, dev)
        if on:
            params.setup_exposures([c.image_name for c in cams] + ["unused"])
        trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), start_iteration=1500, train_exposure=on)
        loss = trainer.step(list(zip(cams, gts)))
        res[on] = (float(loss), params.param_arena.clone(), params)
    (l0, a0, _), (l1, a1, p1) = res[False], res[True]
    assert abs(l1 - l0) <= 1e-6 * abs(l0)
    diff = (a1 - a0).abs()
    assert float((diff > 1e-3).float().mean()) <= 1e-3 and float(diff.median()) <= 1e-6
    # only the exposure table moved: the rendered images' rows, not the unused one
    moved = (p1._exposure.detach() - torch.eye(3, 4, device=dev)).abs().amax(dim=(1, 2))
    assert bool((moved[:3] > 0).all()) and float(moved[3]) == 0.0


@pytest.mark.parametrize("cache_gt", [False, True])
def test_direct_executor_matches_autograd_with_exposure(cuda_device, cache_gt):
    dev = cuda_device
    sc, cams, gts, tr = _setup(dev)
    names = [c.image_name for c in cams]
    table = _exposures(names + ["never_rendered"], seed=9, dev=dev)
    seq = [0, 1, 0]  # camera a twice; camera c is in the table but not rendered
    out = {}
    for direct in (True, False):
        params = tr.GaussianParams.from_scene(sc, dev)
        params.setup_exposures(names + ["never_rendered"], exposures=table)
        trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), cache_ground_truth=cache_gt,
                                        train_exposure=True)
        trainer.direct = direct
        params.zero_grad()
        params.exposure_grad.zero_()
        losses, vis, rows = [], [], []
        for i in seq:
            before = params.exposure_grad.clone()
            if direct:
                loss, pkg = trainer.view_step_direct(cams[i], gts[i], 2000)
            else:
                loss, pkg = trainer.view_loss(cams[i], gts[i], 2000)
                loss.backward()
            losses.append(float(loss.detach()))
            vis.append(pkg["visibility_filter"].clone())
            rows.append(params.exposure_grad - before)
        out[direct] = (params.grad_arena.clone(), losses, vis, params.exposure_grad.clone(), rows)
    a, b = out[True], out[False]
    assert all(abs(x - y) <= 1e-6 * abs(y) + 1e-9 for x, y in zip(a[1], b[1])), (a[1], b[1])
    err = (a[0] - b[0]).abs().max().item()
    assert err <= 1e-5 * b[0].abs().max().item() + 1e-12, err
    assert all(torch.equal(x, y) for x, y in zip(a[2], b[2]))
    ea, eb = a[3], b[3]
    assert (ea - eb).abs().max().item() <= 1e-5 * eb.abs().max().item(), (ea, eb)
    # the repeated camera's row is the sum of its two views; rows of cameras not rendered stay zero
    for t in (ea, eb):
        assert float(t[2].abs().max()) == 0.0 and float(t[3].abs().max()) == 0.0
    ra = a[4]
    assert (ea[0] - (ra[0][0] + ra[2][0])).abs().max().item() <= 1e-6 * ea[0].abs().max().item()
    assert float(ea[0].abs().max()) > 0 and float(ea[1].abs().max()) > 0


def test_exposure_adam_matches_torch_adam(cuda_device):
    from hidegs_b200.optim import get_expon_lr_func
    dev = cuda_device
    sc, cams, gts, tr = _setup(dev)
    names = [c.image_name for c in cams]
    params = tr.GaussianParams.from_scene(sc, dev)
    params.setup_exposures(names + ["never_rendered"], exposures=_exposures(names + ["never_rendered"], 3, dev))
    start = 4990  # steps inside and past the end of the lr delay ramp
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), train_exposure=True, start_iteration=start)
    leaf = torch.nn.Parameter(params._exposure.detach().clone())
    o = tr.OptimizationParams
    lr = get_expon_lr_func(o.exposure_lr_init, o.exposure_lr_final, o.exposure_lr_delay_steps, o.exposure_lr_delay_mult,
                           max_steps=o.iterations)
    ref = torch.optim.Adam([leaf], lr=0.0, eps=1e-8)
    steps = [[0, 1, 2], [0, 1], [0], [0, 0], [2]]  # rows b and c get no gradient in later steps
    for k, ids in enumerate(steps):
        trainer.step([(cams[i], gts[i]) for i in ids])
        g = params.exposure_grad.clone()
        if k >= 2:
            assert float(g[1].abs().max()) == 0.0
        leaf.grad = g * (1.0 / len(ids))
        for pg in ref.param_groups:
            pg["lr"] = lr(start + k + 1)
        ref.step()
    got = params._exposure.detach()
    err = (got - leaf.detach()).abs()
    assert bool((err <= 1e-6 * leaf.detach().abs() + 1e-9).all()), float(err.max())
    # dense: row b kept moving in the steps it was not rendered in; the never-rendered row never moved
    assert trainer.exposure_step_count == len(steps)
    assert torch.equal(got[3], _exposures(names + ["never_rendered"], 3, dev)["never_rendered"])


def test_exposure_training_recovers_known_exposures(cuda_device):
    from hidegs_b200 import gaussian_renderer as gr
    dev = cuda_device
    sc, cams, _gts, tr = _setup(dev, W=240, H=160, names=("v0", "v1", "v2", "v3"))
    g = torch.Generator().manual_seed(21)
    truth = {}
    for c in cams:
        E = torch.zeros(3, 4)
        E[:, :3] = torch.diag(torch.empty(3).uniform_(0.7, 1.3, generator=g))
        E[:, 3] = torch.empty(3).uniform_(-0.05, 0.05, generator=g)
        truth[c.image_name] = E.to(dev)
    params = tr.GaussianParams.from_scene(sc, dev)
    params.setup_exposures([c.image_name for c in cams], exposures=truth)
    with torch.no_grad():  # ground truth: the scene rendered through the true exposures
        gts = [gr.render(c, params, tr.PipelineParams, torch.zeros(3, device=dev), use_trained_exp=True)["render"]
               .contiguous() for c in cams]
    params.setup_exposures([c.image_name for c in cams])  # start from eye(3, 4)

    class Opt(tr.OptimizationParams):
        position_lr_init = feature_lr = opacity_lr = scaling_lr = rotation_lr = 0.0
        exposure_lr_init, exposure_lr_final, exposure_lr_delay_steps = 0.02, 0.001, 0
        iterations = 300

    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), opt=Opt, train_exposure=True)
    arena0 = params.param_arena.clone()
    T = torch.stack([truth[c.image_name] for c in cams])
    d0 = float((params._exposure.detach() - T).norm())
    views = list(zip(cams, gts))
    losses = [float(trainer.step(views)) for _ in range(300)]
    d1 = float((params._exposure.detach() - T).norm())
    assert d1 <= d0 / 5, (d0, d1)
    assert sum(losses[-10:]) < sum(losses[:10])
    assert torch.equal(params.param_arena, arena0)  # Gaussian learning rates 0


def test_exposure_interfaces(cuda_device, tmp_path):
    from hidegs_b200 import gaussian_renderer as gr, ply_io
    dev = cuda_device
    sc, cams, gts, tr = _setup(dev)
    names = [c.image_name for c in cams]
    params = tr.GaussianParams.from_scene(sc, dev)
    params.setup_exposures(names, exposures=_exposures(names, 5, dev))
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), train_exposure=True, start_iteration=6000,
                                    densification_stats=True)
    for _ in range(2):
        trainer.step(list(zip(cams, gts)))
    # render(use_trained_exp=True) on the trainer's model == the executor's exposed image
    for c, gt in zip(cams, gts):
        with torch.no_grad():
            ref = gr.render(c, params, tr.PipelineParams, torch.zeros(3, device=dev), use_trained_exp=True)["render"]
        params.zero_grad()
        _loss, pkg = trainer.view_step_direct(c, gt, 6000)
        assert (pkg["render"] - ref).abs().max().item() <= 1e-6
    # exposure.json round trip
    path = str(tmp_path / "exposure.json")
    params.save_exposures(path)
    q = tr.GaussianParams.from_scene(sc, dev)
    q.setup_exposures(names, exposures=ply_io.load_exposures(path, device=dev))
    assert torch.equal(q._exposure.detach(), params._exposure.detach())
    # densify / prune leave the table alone
    before = params._exposure.detach().clone()
    trainer.densify_and_prune(0.0002, 0.005, 1.0)
    assert torch.equal(params._exposure.detach(), before) and params._exposure.grad is params.exposure_grad
    trainer.step(list(zip(cams, gts)))
    # an image without an exposure, on either path
    stranger = copy.copy(cams[0])
    stranger.image_name = "not_in_the_table"
    for direct in (True, False):
        trainer.direct = direct
        with pytest.raises(ValueError):
            trainer.step([(stranger, gts[0])])
    # train_exposure without a table
    with pytest.raises(ValueError):
        tr.ViewShardedTrainer(tr.GaussianParams.from_scene(sc, dev), torch.zeros(3, device=dev), train_exposure=True)


def test_exposure_multi_gpu_ranks_stay_identical(cuda_device):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    world = torch.cuda.device_count()
    env = dict(os.environ, PYTHONPATH=ROOT)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr",
           "127.0.0.1", "--master-port", "29543", os.path.join(ROOT, "tools", "exposure_probe.py"), "--check"]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    out = json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])
    assert out["world"] == world
    assert out["ranks_identical"] and out["equals_single_process"], out
    assert out["table_moved"] > 0, out
