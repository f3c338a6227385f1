"""Camera pose refinement in the training step (ViewShardedTrainer(train_poses=True), DESIGN.md §3 "Camera pose
refinement"): the pose gradient against identities that move the Gaussians instead of the camera, against float64
autograd off zero and against finite differences; determinism; the zero-lr step; recovery of perturbed cameras;
several ranks; the interfaces."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

NAMES = ("img_a", "img_b", "img_c")


def _setup(dev, n=30_000, W=320, H=208, sh_degree=3, zero_high_bands=False, seed=2):
    from hidegs_b200 import synthetic as syn, trainer as tr
    sc = syn.make_scene(n, seed=seed, log_scale_mean=math.log(0.01 * 1920.0 / W))
    if zero_high_bands:
        sc["shs"][:, 1:] = 0.0
    cams = []
    for k, name in enumerate(NAMES):
        c = syn.default_camera(W, H, eye=(0.3 * k - 0.3, 0.1 * k, -5.0)).to(dev)
        c.image_name = name
        cams.append(c)
    g = torch.Generator().manual_seed(4)
    gts = [torch.nn.functional.avg_pool2d(torch.rand(1, 3, H, W, generator=g), 5, stride=1, padding=2)[0].clamp(0, 1)
           .to(dev) for _ in cams]
    params = tr.GaussianParams.from_scene(sc, dev)
    params.active_sh_degree = sh_degree
    params.setup_camera_poses(NAMES)
    return params, cams, gts, tr


def _R(cam):
    """World-to-camera rotation (column convention) of a camera's row-vector viewmatrix."""
    return cam.world_view_transform.detach().double().cpu()[:3, :3].T


def _xyz_grad(p):
    return p.grad_arena[p.slices["xyz"]].view(p.N, 3).double().cpu()


def _quat_torque(q, gq):
    """dL/domega of q -> Exp(omega) (x) q (world-axis rotation of the orientation), for the gradient gq of the raw
    quaternions q (real first), to first order: q + 0.5 [0, omega] (x) q, differentiated in float64."""
    w = torch.zeros(3, dtype=torch.float64, requires_grad=True)
    r, x, y, z = q.unbind(1)
    a, b, c = 0.5 * w[0], 0.5 * w[1], 0.5 * w[2]
    # Hamilton product [0, a, b, c] (x) [r, x, y, z]
    dq = torch.stack([-a * x - b * y - c * z, a * r + b * z - c * y, -a * z + b * r + c * x, a * y - b * x + c * r], 1)
    (dq * gq).sum().backward()
    return w.grad


def _identity_sides(p, cam, campos):
    """(R sum dL/dx, R sum [(x - c) x dL/dx + torque(q, dL/dq)]) of the view in the arena, float64."""
    R = _R(cam)
    gx = _xyz_grad(p)
    x = p._xyz.detach().double().cpu()
    gq = p.grad_arena[p.slices["rotation"]].view(p.N, 4).double().cpu()
    q = p._rotation.detach().double().cpu()
    c = campos.detach().double().cpu().reshape(1, 3)
    trans = R @ gx.sum(0)
    rot = R @ (torch.linalg.cross(x - c, gx, dim=1).sum(0) + _quat_torque(q, gq))
    return trans, rot


def _rel(a, b):
    return float(torch.linalg.norm(a - b) / torch.linalg.norm(b))


def _depth_prior(cam, dev, seed=7):
    g = torch.Generator().manual_seed(seed)
    H, W = int(cam.image_height), int(cam.image_width)
    cam.invdepthmap = (0.15 + 0.1 * torch.rand(1, H, W, generator=g)).to(dev)
    cam.depth_mask = (torch.rand(1, H, W, generator=g) > 0.2).float().to(dev)
    cam.depth_reliable = True


def test_translation_identity_every_term_on(cuda_device):
    """Moving the camera by rho = moving every Gaussian by R^T rho (SH view directions included), so at SH degree 3
    with the normal, frequency, depth and exposure terms on: dL/drho = R sum_i dL/dx_i."""
    dev = cuda_device
    p, cams, gts, tr = _setup(dev)
    p.setup_exposures(NAMES)
    with torch.no_grad():
        p._exposure += 0.03 * torch.randn(p._exposure.shape, generator=torch.Generator().manual_seed(3)).to(dev)
    cam = cams[1]
    _depth_prior(cam, dev)
    t = tr.ViewShardedTrainer(p, torch.zeros(3, device=dev), start_iteration=1500, train_poses=True, train_exposure=True,
                              depth_regularization=True)
    _loss, out = t.view_step_direct(cam, gts[1], 1500)
    assert "depth_l1" in out and "render" in out
    g = out["pose_grad"].double().cpu()
    trans, _ = _identity_sides(p, cam, cam.camera_center)
    assert float(torch.linalg.norm(trans)) > 0
    assert _rel(g[:3], trans) <= 1e-5, (g[:3], trans)
    # the view's contribution is what landed in the camera's row (table starts at zero; pads untouched)
    row = p.camera_pose_grad[p.camera_pose_index(cam.image_name)].cpu()
    assert torch.equal(row[:6], out["pose_grad"].cpu()) and not row[6:].any()


@pytest.mark.parametrize("sh", ["degree0", "degree3_dc_only"])
def test_rotation_identity(cuda_device, sh):
    """Turning the camera about its centre by phi = turning every Gaussian's mean and orientation about the centre by
    R^T phi, except for the SH view direction (absent at degree 0 and with the higher bands zero)."""
    dev = cuda_device
    p, cams, gts, tr = _setup(dev, sh_degree=0 if sh == "degree0" else 3, zero_high_bands=sh != "degree0")
    cam = cams[2]
    t = tr.ViewShardedTrainer(p, torch.zeros(3, device=dev), start_iteration=1500, train_poses=True)
    _loss, out = t.view_step_direct(cam, gts[2], 1500)
    g = out["pose_grad"].double().cpu()
    trans, rot = _identity_sides(p, cam, cam.camera_center)
    assert _rel(g[:3], trans) <= 1e-5, (g[:3], trans)
    assert _rel(g[3:], rot) <= 1e-4, (g[3:], rot)


def _xi(dev):
    return torch.tensor([0.02, -0.015, 0.03, 0.004, -0.003, 0.002], dtype=torch.float32, device=dev)


def test_apply_off_zero_matches_float64(cuda_device):
    from hidegs_b200 import camera_pose as cp
    dev = cuda_device
    p, cams, _gts, _tr = _setup(dev, n=1000)
    with torch.no_grad():
        p._camera_pose[1, :6] = _xi(dev)
        p._camera_pose[2, :6] = 0.5 * _xi(dev)
    for k, cam in enumerate(cams):
        buf = p._corrected_matrices(k, cam.world_view_transform, cam.full_proj_transform, cam.camera_center).double().cpu()
        V = cam.world_view_transform.double().cpu()
        C = torch.from_numpy(cp.pose_matrix(p._camera_pose[k, :6].detach().double().cpu().numpy()))
        V2 = V @ C.T
        P2 = V2 @ cam.projection_matrix.double().cpu()
        c2 = torch.linalg.inv(V2)[3, :3]
        assert torch.allclose(buf[:16].view(4, 4), V2, rtol=1e-6, atol=1e-6)
        assert torch.allclose(buf[16:32].view(4, 4), P2, rtol=1e-6, atol=1e-6)
        assert torch.allclose(buf[32:35], c2, rtol=0, atol=1e-6)
        assert buf[35] == 0
        if k == 0:  # a zero row gives the input camera bit for bit
            assert torch.equal(buf[:16].float(), cam.world_view_transform.cpu().reshape(-1))
            assert torch.equal(buf[16:32].float(), cam.full_proj_transform.cpu().reshape(-1))
            assert torch.equal(buf[32:35].float(), cam.camera_center.cpu().reshape(-1))
    corrected = p.corrected_camera(cams[1])
    assert torch.equal(corrected.world_view_transform.reshape(-1),
                       p._corrected_matrices(1, cams[1].world_view_transform, cams[1].full_proj_transform,
                                             cams[1].camera_center)[:16])


def test_gradient_off_zero_matches_float64_autograd(cuda_device):
    """At xi != 0 the trained gradient is float64 autograd of xi -> W2C(xi), contracted with the left-perturbation
    gradient (g, tau) of the corrected camera (which the two identities give at SH degree 0)."""
    from hidegs_b200 import camera_pose as cp
    dev = cuda_device
    p, cams, gts, tr = _setup(dev, sh_degree=0)
    k = 1
    with torch.no_grad():
        p._camera_pose[k, :6] = _xi(dev)
    cam = cams[k]
    t = tr.ViewShardedTrainer(p, torch.zeros(3, device=dev), start_iteration=1500, train_poses=True)
    _loss, out = t.view_step_direct(cam, gts[k], 1500)
    got = out["pose_grad"].double().cpu()
    cc = p.corrected_camera(cam)
    g_t, tau = _identity_sides(p, cc, cc.camera_center)
    W2C0 = cam.world_view_transform.double().cpu().T
    xi0 = p._camera_pose[k, :6].detach().double().cpu()
    M0 = torch.from_numpy(cp.pose_matrix(xi0.numpy())) @ W2C0

    def W2C(xi):
        phi, rho = xi[3:], xi[:3]
        th = torch.linalg.norm(phi)
        K = torch.zeros(3, 3, dtype=torch.float64)
        K = K.index_put((torch.tensor([0, 0, 1, 1, 2, 2]), torch.tensor([1, 2, 0, 2, 0, 1])),
                        torch.stack([-phi[2], phi[1], phi[2], -phi[0], -phi[1], phi[0]]))
        E = torch.eye(3, dtype=torch.float64) + torch.sin(th) / th * K + (1 - torch.cos(th)) / th ** 2 * K @ K
        C = torch.eye(4, dtype=torch.float64)
        C = torch.cat([torch.cat([E, rho.view(3, 1)], 1), C[3:]], 0)
        return C @ W2C0

    xi = xi0.clone().requires_grad_(True)
    D = W2C(xi) @ torch.linalg.inv(M0)  # the left increment (I + [d]x, dt) to first order
    vee = 0.5 * torch.stack([D[2, 1] - D[1, 2], D[0, 2] - D[2, 0], D[1, 0] - D[0, 1]])
    (g_t @ D[:3, 3] + tau @ vee).backward()
    want = xi.grad
    assert _rel(got[:3], want[:3]) <= 1e-5, (got, want)
    assert _rel(got[3:], want[3:]) <= 1e-4, (got, want)


def test_pose_gradient_is_deterministic_and_chunk_invariant(cuda_device):
    """The reduction adds no run-to-run variation of its own.  The per-Gaussian rows it sums come from the blend
    backward's float atomics, so two training views agree to atomic order only; with an upstream gradient on pixels
    spaced wider than any footprint every row receives at most one contribution, and then two runs, with the
    per-Gaussian part in 1 or in 4 slot ranges, and the finish give the same bits."""
    dev = cuda_device
    runs = []
    for _ in range(2):
        p, cams, gts, tr = _setup(dev)
        t = tr.ViewShardedTrainer(p, torch.zeros(3, device=dev), start_iteration=1500, train_poses=True)
        runs.append(t.view_step_direct(cams[0], gts[0], 1500)[1]["pose_grad"].double().cpu())
    assert _rel(runs[0], runs[1]) <= 1e-5
    import raster_utils as ru
    from hidegs_b200 import synthetic as syn
    from hidegs_b200._geometry_lib import lib
    W, H = 768, 480
    case = ru.build_case(20_000, W, H, seed=5)
    case["scales"] = case["scales"].clamp(max=0.025)  # footprints of at most ~17 px: many sparse pixels fit
    case["all_map"] = syn.geometry_all_map(case["means3D"], case["scales"], case["rotations"], case["cam"])
    fa = ru.op_args(case, dev)
    fwd = ru.OUR_C.rasterize_gaussians(*fa)
    # alpha >= 1/255 reaches at most sqrt(2 ln 255) = 3.33 sigma, the radius is ceil(3 sigma): 3 radii apart is enough
    step = 3 * int(fwd[2].max()) + 3
    keep = torch.zeros(H, W)
    keep[step // 2::step, step // 2::step] = 1.0
    assert keep.sum() >= 32, step
    grads = {k: v * keep for k, v in syn.upstream_grads(W, H).items()}
    N = case["P"]
    nbytes = int(lib().hg_camera_pose_workspace_bytes(N))
    ws = []
    for n_chunks in (1, 1, 4, 4):
        w = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
        ranges = []
        ru.OUR_C.rasterize_gaussians_backward(*ru.bwd_args(fa, fwd, grads, dev), pose_workspace=w,
                                              chunk_hook=(n_chunks, lambda c, a, b: ranges.append((a, b))))
        assert len(ranges) == n_chunks
        ws.append(w)
    torch.cuda.synchronize()
    part = (N + 127) // 128 * 64
    for w in ws[1:]:
        assert torch.equal(w[:part], ws[0][:part])
    sums = ws[0][:part].view(torch.float64)
    assert bool(torch.isfinite(sums).all()) and float(sums.abs().sum()) > 0
    table = torch.zeros(1, 8, device=dev)
    out = [torch.zeros(1, 8, device=dev) for _ in range(2)]
    for o in out:
        assert lib().hg_camera_pose_grad_finish(table.data_ptr(), 1, 0, N, ws[0].data_ptr(), o.data_ptr(), None,
                                                torch.cuda.current_stream().cuda_stream) == 0
    assert torch.equal(out[0], out[1]) and bool(out[0][0, :6].abs().gt(0).all())


def test_finite_differences(cuda_device):
    """Central differences of the forward loss against the analytic gradient.  Loose (cosine >= 0.99) because the
    backward the rasterizer is built on is not the derivative of its forward: the 2-D dilation is 0.3 px^2 in the
    backward against 0.1 in the forward (the reference's quirk), and the frustum clamp and the near cull are piecewise."""
    dev = cuda_device
    p, cams, gts, tr = _setup(dev, n=20_000)
    k = 1
    t = tr.ViewShardedTrainer(p, torch.zeros(3, device=dev), train_poses=True)
    base = p._camera_pose.detach().clone()

    def loss_at(xi6):
        with torch.no_grad():
            p._camera_pose.copy_(base)
            p._camera_pose[k, :6] += xi6
        p._grad_dirty = False
        return float(t.view_step_direct(cams[k], gts[k], 10)[0])
    _l, out = t.view_step_direct(cams[k], gts[k], 10)
    analytic = out["pose_grad"].double().cpu()
    steps = [2e-3] * 3 + [4e-4] * 3
    fd = torch.zeros(6, dtype=torch.float64)
    for i in range(6):
        e = torch.zeros(6, device=dev)
        e[i] = steps[i]
        fd[i] = (loss_at(e) - loss_at(-e)) / (2 * steps[i])
    cos = float(analytic @ fd / (torch.linalg.norm(analytic) * torch.linalg.norm(fd)))
    assert cos >= 0.99, (analytic, fd, cos)


def _opt(**kw):
    from hidegs_b200 import trainer as tr
    return type("Opt", (tr.OptimizationParams,), kw)


def test_zero_lr_step_equals_plain_step(cuda_device):
    dev = cuda_device
    res = {}
    for on in (False, True):
        p, cams, gts, tr = _setup(dev)
        t = tr.ViewShardedTrainer(p, torch.zeros(3, device=dev), opt=_opt(pose_lr_translation=0.0, pose_lr_rotation=0.0),
                                  start_iteration=1500, train_poses=on)
        views = list(zip(cams, gts))
        loss = t.step(views)
        res[on] = (float(loss), t.visible.clone(), p.param_arena.clone(), p)
    (l0, v0, a0, _), (l1, v1, a1, p1) = res[False], res[True]
    assert abs(l1 - l0) <= 1e-6 * abs(l0)
    assert torch.equal(v0, v1)
    diff = (a1 - a0).abs()
    assert float((diff > 1e-3).float().mean()) <= 1e-3 and float(diff.median()) <= 1e-6
    assert not p1._camera_pose.detach().any()  # zero rates: the table does not move
    assert bool(p1.camera_pose_grad[:, :6].abs().sum(1).gt(0).all())  # though every camera got a gradient


def test_recovery_of_perturbed_cameras(cuda_device):
    """Ground truths rendered from the true cameras; 2 of 3 cameras start 0.5 % of the scene depth and 0.3 degrees
    off.  With the Gaussians frozen the pose errors fall at least 5x in a fixed budget; with the pose rates at 0 they
    stay where they were."""
    from hidegs_b200 import gaussian_renderer as gr
    dev = cuda_device
    W, H = 256, 160
    depth = 5.0
    g = torch.Generator().manual_seed(9)
    err = torch.zeros(3, 6)
    for k in (1, 2):
        d = torch.randn(3, generator=g)
        a = torch.randn(3, generator=g)
        err[k, :3] = 0.005 * depth * d / d.norm()
        err[k, 3:] = math.radians(0.3) * a / a.norm()
    # photometric terms only: the Gaussians are frozen and the ground truths are their own renders
    frozen = dict(position_lr_init=0.0, feature_lr=0.0, opacity_lr=0.0, scaling_lr=0.0, rotation_lr=0.0,
                  single_view_weight=0.0)
    final = {}
    for lr_on in (True, False):
        p, cams, _gts, tr = _setup(dev, n=20_000, W=W, H=H)
        with torch.no_grad():
            gts = [gr.render(c, p, tr.PipelineParams, torch.zeros(3, device=dev))["render"].clamp(0, 1).detach()
                   for c in cams]
            p._camera_pose[:, :6] = err.to(dev)
        p.begin_view()
        rates = dict(pose_lr_translation=2e-3, pose_lr_rotation=4e-4) if lr_on else dict(pose_lr_translation=0.0,
                                                                                         pose_lr_rotation=0.0)
        t = tr.ViewShardedTrainer(p, torch.zeros(3, device=dev), opt=_opt(**frozen, **rates), train_poses=True)
        views = list(zip(cams, gts))
        for _ in range(200):
            t.step(views)
        final[lr_on] = p._camera_pose.detach()[:, :6].cpu().double()
    e0 = err.double()
    for k in (1, 2):
        t0, r0 = float(e0[k, :3].norm()), float(e0[k, 3:].norm())
        t1, r1 = float(final[True][k, :3].norm()), float(final[True][k, 3:].norm())
        assert t1 <= t0 / 5 and r1 <= r0 / 5, (k, t0, t1, r0, r1)
    assert torch.equal(final[False], e0.float().double())
    assert not final[True][0].abs().gt(5e-3).any()  # the true camera stays close to true


def test_camera_pose_multi_gpu_ranks_stay_identical(cuda_device):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    world = torch.cuda.device_count()
    env = dict(os.environ, PYTHONPATH=ROOT)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr",
           "127.0.0.1", "--master-port", "29547", os.path.join(ROOT, "tools", "pose_probe.py"), "--check"]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    out = json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])
    assert out["world"] == world
    assert out["ranks_identical"] and out["equals_single_process"], out
    assert out["table_moved"] > 0, out


def test_camera_pose_interfaces(cuda_device, tmp_path):
    from hidegs_b200 import ply_io
    from hidegs_b200 import synthetic as syn
    dev = cuda_device
    p, cams, gts, tr = _setup(dev, n=5000)
    t = tr.ViewShardedTrainer(p, torch.zeros(3, device=dev), train_poses=True)
    stranger = syn.default_camera(320, 208).to(dev)
    stranger.image_name = "nobody"
    before = (p.param_arena.clone(), p._camera_pose.detach().clone(), t.iteration)
    with pytest.raises(ValueError, match="nobody"):
        t.step([(cams[0], gts[0]), (stranger, gts[0])])
    assert torch.equal(p.param_arena, before[0]) and torch.equal(p._camera_pose.detach(), before[1])
    assert t.iteration == before[2]
    with pytest.raises(ValueError):
        tr.ViewShardedTrainer(tr.GaussianParams.from_scene(syn.make_scene(100, seed=1), dev), torch.zeros(3, device=dev),
                              train_poses=True)
    # a step moves the rendered cameras' rows only; densify-style resize leaves the table alone
    p.setup_camera_poses(list(NAMES) + ["unused"])
    t = tr.ViewShardedTrainer(p, torch.zeros(3, device=dev), train_poses=True,
                              opt=_opt(pose_lr_translation=1e-3, pose_lr_rotation=1e-3))
    t.step(list(zip(cams, gts)))
    moved = p._camera_pose.detach().abs().sum(1)
    assert bool((moved[:3] > 0).all()) and float(moved[3]) == 0.0 and not p._camera_pose.detach()[:, 6:].any()
    table = p._camera_pose.detach().clone()
    p.resize(p.param_arena.clone(), p.N)
    assert torch.equal(p._camera_pose.detach(), table)
    # save / load round trip, corrected camera matches the saved W2C
    path = str(tmp_path / "camera_poses.json")
    p.save_camera_poses(path, cams)
    q = tr.GaussianParams.from_scene(syn.make_scene(100, seed=1), dev)
    q.setup_camera_poses(list(NAMES) + ["unused"], poses=ply_io.load_camera_poses(path))
    assert torch.equal(q._camera_pose.detach(), table)
    saved = json.load(open(path))
    for cam in cams:
        cc = p.corrected_camera(cam)
        w2c = np.array(saved[cam.image_name]["w2c"])
        assert np.allclose(cc.world_view_transform.double().cpu().numpy().T, w2c, atol=1e-6)
        assert cc.image_width == cam.image_width and torch.equal(cc.projection_matrix, cam.projection_matrix)
