"""3DGS-MCMC densification over the training arenas (hg_mcmc_regularizer / hg_mcmc_inject_noise / hg_mcmc_relocate /
hg_mcmc_grow, trainer.mcmc_*, ViewShardedTrainer(mcmc=True)) against the PyTorch restatement (oracle/mcmc_oracle.py)
with the draws and normals injected; the Philox paths on their own; the trainer end to end; two or more ranks."""
import json
import math
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _model(N, dev, seed, dead_frac=0.3):
    """Random raw parameters (a `dead_frac` share of the rows with opacity logit -8, o = 3.4e-4) and random moments."""
    from hidegs_b200 import trainer as tr
    g = torch.Generator().manual_seed(seed)
    op = torch.randn(N, 1, generator=g) * 1.5
    op = op.clamp_min(-2.9)  # live rows well above min_opacity (o >= 0.052)
    op[torch.rand(N, generator=g) < dead_frac] = -8.0
    t = dict(xyz=torch.randn(N, 3, generator=g) * 2.0, features=torch.randn(N, 16, 3, generator=g), opacity=op,
             scaling=torch.empty(N, 3).uniform_(math.log(0.005), math.log(0.5), generator=g),
             rotation=torch.randn(N, 4, generator=g))
    params = tr.GaussianParams(*[t[k].to(dev) for k in ("xyz", "features", "opacity", "scaling", "rotation")])
    adam = tr.ArenaAdam(params)
    n = params.param_arena.numel()
    adam.exp_avg.copy_(torch.randn(n, generator=g).to(dev))
    adam.exp_avg_sq.copy_(torch.rand(n, generator=g).to(dev))
    for a in (adam.exp_avg, adam.exp_avg_sq):  # pad floats stay zero, as in the trainer's arenas
        _zero_pads(a, N)
    return params, adam


def _zero_pads(a, N):
    from hidegs_b200 import trainer as tr
    starts, total = tr.arena_layout(N)
    for name, w in tr.GROUPS:
        end = starts[name] + N * w
        a[end:(end + 3) // 4 * 4] = 0.0


def _split(a, N):
    """{group: [N, w]} views of an arena of N rows."""
    from hidegs_b200 import trainer as tr
    starts, _ = tr.arena_layout(N)
    return {name: a[starts[name]:starts[name] + N * w].view(N, w) for name, w in tr.GROUPS}


def _dicts(params, adam):
    N = params.N
    sh = lambda d: {k: (x.view(N, 16, 3) if k == "features" else x) for k, x in d.items()}  # noqa: E731
    return (sh(_split(params.param_arena, N)), sh(_split(adam.exp_avg, N)), sh(_split(adam.exp_avg_sq, N)))


def _ulp_diff(a, b):
    return (a.contiguous().view(torch.int32).long() - b.contiguous().view(torch.int32).long()).abs()


def _compare(arenas, N, want, touched):
    """Kernel arenas (param, exp_avg, exp_avg_sq of N rows) against the oracle's dicts: opacity / scaling within 1 ulp,
    everything else bit-identical; moments exactly zero on the `touched` rows; pads zero."""
    from hidegs_b200 import trainer as tr
    for a, w, kind in zip(arenas, want, "pmv"):
        got = _split(a, N)
        for name, wd in tr.GROUPS:
            ref = w[name].reshape(N, wd)
            if kind == "p" and name in ("opacity", "scaling"):
                d = _ulp_diff(got[name], ref)
                assert int(d.max()) <= 1, (name, int(d.max()))
            else:
                assert torch.equal(got[name], ref), (kind, name)
            if kind != "p":
                assert not got[name][touched].any(), (kind, name)
        starts, _ = tr.arena_layout(N)
        for name, wd in tr.GROUPS:
            end = starts[name] + N * wd
            assert not a[end:(end + 3) // 4 * 4].any(), ("pad", kind, name)


@pytest.mark.parametrize("N", [1024, 30001])
def test_regularizer_matches_float64(cuda_device, N):
    from hidegs_b200 import trainer as tr
    from oracle import mcmc_oracle as mo
    dev = cuda_device
    params, _ = _model(N, dev, seed=N)
    ws = tr.mcmc_workspace(N, dev)
    grad = torch.zeros_like(params.param_arena)
    loss = torch.full((), 2.0, device=dev)
    val = tr.mcmc_regularizer(params.param_arena, grad, N, 0.01, 0.02, grad_mult=3.0, loss_mult=2.0, loss=loss,
                              workspace=ws)
    ref, gx, gy = mo.regularizer(params.leaves["opacity"], params.leaves["scaling"], 0.01, 0.02)
    assert abs(float(val) - float(ref)) <= 1e-6 * float(ref)
    assert abs(float(loss) - (2.0 + 2.0 * float(ref))) <= 1e-6 * (2.0 + 2.0 * float(ref))
    g = _split(grad, N)
    for got, want in ((g["opacity"], 3.0 * gx), (g["scaling"], 3.0 * gy)):
        err = (got.double() - want).abs() / want.abs()
        assert float(err.max()) <= 1e-6, float(err.max())
    others = torch.ones_like(grad, dtype=torch.bool)
    sl = params.slices
    others[sl["opacity"]] = False
    others[sl["scaling"]] = False
    assert not grad[others].any()
    # bit-identical on a second run (the same workspace: its counter was left at zero), and accumulated onto a gradient
    grad2 = torch.zeros_like(grad)
    val2 = tr.mcmc_regularizer(params.param_arena, grad2, N, 0.01, 0.02, grad_mult=3.0, workspace=ws)
    assert torch.equal(grad2, grad) and torch.equal(val2, val)
    base = torch.randn(grad.shape, generator=torch.Generator().manual_seed(1)).to(dev)
    acc = base.clone()
    tr.mcmc_regularizer(params.param_arena, acc, N, 0.01, 0.02, grad_mult=3.0, workspace=ws)
    assert torch.equal(acc[others], base[others])
    assert torch.equal(acc[~others], base[~others] + grad[~others])
    # both weights 0: no launch, nothing changes
    assert tr.mcmc_regularizer(params.param_arena, acc, N, 0.0, 0.0, workspace=ws) is None


def test_noise_matches_oracle_with_injected_normals(cuda_device):
    from hidegs_b200 import trainer as tr
    from oracle import mcmc_oracle as mo
    dev = cuda_device
    N = 30001
    params, _ = _model(N, dev, seed=3, dead_frac=0.5)
    lv = params.leaves
    with torch.no_grad():  # opacities that open the gate (o < 0.02) on half the rows
        lv["opacity"][::2] = torch.empty((N + 1) // 2, 1).uniform_(-9.0, -4.0, generator=torch.Generator().manual_seed(6))
    z = torch.randn(N, 3, generator=torch.Generator().manual_seed(5)).to(dev)
    x0 = lv["xyz"].detach().clone()
    scale = tr.OptimizationParams.position_lr_init * tr.OptimizationParams.mcmc_noise_lr
    ref = mo.noise_delta(lv["opacity"], lv["scaling"], lv["rotation"], z, scale)
    tr.mcmc_inject_noise(params.param_arena, N, scale, normals=z)
    got = lv["xyz"].detach().double() - x0.double()  # (exact in double)
    # 1e-6 of the row's magnitude, plus the rounding of xyz + delta to float
    o = torch.sigmoid(lv["opacity"].double()).view(-1)
    gate = torch.sigmoid(100.0 * ((1.0 - o) - 0.995))
    mag = torch.exp(2 * lv["scaling"].double()).amax(1) * z.double().abs().sum(1) * gate * scale
    tol = 1e-6 * mag[:, None] + lv["xyz"].detach().double().abs() * 2.0 ** -24
    assert bool(((got - ref).abs() <= tol).all()), float(((got - ref).abs() / tol).max())
    assert int((ref.abs() > 1e-3).any(1).sum()) > 1000  # the noise moved many rows visibly
    # every other float is left alone
    rest = torch.ones_like(params.param_arena, dtype=torch.bool)
    rest[params.slices["xyz"]] = False
    before = params.param_arena.clone()
    tr.mcmc_inject_noise(params.param_arena, N, scale, normals=z)
    assert torch.equal(params.param_arena[rest], before[rest])


def test_noise_philox_draws(cuda_device):
    """Philox normals: the same seed gives the same bits, another seed others; over 2M draws (identity rotation, unit
    scale, closed-to-transparent opacity) the normals have mean 0 and variance 1 within 5e-3."""
    from hidegs_b200 import trainer as tr
    dev = cuda_device
    N = 666_667
    args = (torch.zeros(N, 3, device=dev), torch.zeros(N, 16, 3, device=dev), torch.full((N, 1), -30.0, device=dev),
            torch.zeros(N, 3, device=dev), torch.tensor([[1.0, 0.0, 0.0, 0.0]], device=dev).repeat(N, 1))
    runs = []
    for seed in (7, 7, 8):
        p = tr.GaussianParams(*args)
        tr.mcmc_inject_noise(p.param_arena, N, 1.0, seed=seed)
        runs.append(p.leaves["xyz"].detach().clone())
    assert torch.equal(runs[0], runs[1]) and not torch.equal(runs[0], runs[2])
    o = torch.sigmoid(torch.tensor(-30.0, dtype=torch.float64))
    gate = float(torch.sigmoid(100.0 * ((1.0 - o) - 0.995)))
    z = runs[0].double().view(-1) / gate
    assert z.numel() >= 2_000_000
    assert abs(float(z.mean())) <= 5e-3 and abs(float(z.var()) - 1.0) <= 5e-3, (float(z.mean()), float(z.var()))


def test_relocation_sampler(cuda_device):
    """1M dead rows drawn from 1000 live ones weighted by opacity: chi-square p > 1e-3 with a fixed seed; no dead row
    is ever a source; two runs are bit-identical."""
    from scipy.stats import chisquare
    from hidegs_b200 import trainer as tr
    dev = cuda_device
    n_live, n_dead = 1000, 1_000_000
    N = n_live + n_dead
    g = torch.Generator().manual_seed(11)
    live = torch.randperm(N, generator=g)[:n_live].sort().values
    op = torch.full((N, 1), -8.0)
    op[live] = torch.empty(n_live, 1).uniform_(-4.0, 4.0, generator=g)
    feats = torch.zeros(N, 16, 3)
    feats[:, 0, 0] = torch.arange(N, dtype=torch.float32)  # row tags (exact below 2^24)
    params = tr.GaussianParams(torch.randn(N, 3, generator=g).to(dev), feats.to(dev), op.to(dev),
                               torch.full((N, 3), -3.0).to(dev), torch.randn(N, 4, generator=g).to(dev))
    adam = tr.ArenaAdam(params)
    m0, v0 = adam.exp_avg.clone(), adam.exp_avg_sq.clone()
    p0 = params.param_arena.clone()
    counts = tr.mcmc_relocate_arenas(params.param_arena, adam.exp_avg, adam.exp_avg_sq, N, 0.005, seed=123)[3]
    assert int(counts["dead"]) == n_dead and int(counts["alive"]) == n_live
    tags = params.leaves["features"].detach()[:, 0, 0].long().cpu()
    dead = torch.ones(N, dtype=torch.bool)
    dead[live] = False
    src = tags[dead]
    is_live = torch.zeros(N, dtype=torch.bool)
    is_live[live] = True
    assert bool(is_live[src].all())  # never a dead row
    hist = torch.bincount(src, minlength=N)[live].double()
    w = torch.sigmoid(op[live].view(-1).float()).double()
    expected = w / w.sum() * n_dead
    p = chisquare(hist.numpy(), expected.numpy()).pvalue
    assert p > 1e-3, p
    # the same seed on the same inputs: the same bits
    p2 = p0.clone()
    m2, v2 = m0.clone(), v0.clone()
    tr.mcmc_relocate_arenas(p2, m2, v2, N, 0.005, seed=123)
    assert torch.equal(p2, params.param_arena) and torch.equal(m2, adam.exp_avg) and torch.equal(v2, adam.exp_avg_sq)
    # every dead row is a copy of its source
    assert torch.equal(params.leaves["rotation"].detach()[dead.to(dev)].cpu(),
                       params.leaves["rotation"].detach().cpu()[src])


@pytest.mark.parametrize("N", [1, 30001])
def test_relocate_matches_oracle(cuda_device, N):
    from hidegs_b200 import trainer as tr
    from oracle import mcmc_oracle as mo
    dev = cuda_device
    params, adam = _model(N, dev, seed=17 + N, dead_frac=0.3 if N > 1 else 0.0)
    t, m, v = _dicts(params, adam)
    o = torch.sigmoid(params.leaves["opacity"].detach().view(-1))
    dead = (~(o > 0.005)).nonzero().view(-1)
    live = (o > 0.005).nonzero().view(-1)
    g = torch.Generator().manual_seed(2)
    sources = live.cpu()[torch.randint(0, live.numel(), (dead.numel(),), generator=g)]
    sources[: min(10, sources.numel())] = live[0].cpu()  # one row drawn many times
    want = mo.relocate(t, m, v, sources.to(dev), 0.005)
    out = tr.mcmc_relocate_arenas(params.param_arena, adam.exp_avg, adam.exp_avg_sq, N, 0.005, sources=sources)
    assert int(out[3]["dead"]) == dead.numel() and int(out[3]["alive"]) == live.numel()
    touched = torch.zeros(N, dtype=torch.bool, device=dev)
    touched[dead] = True
    touched[sources.to(dev)] = True
    _compare(out[:3], N, want, touched)
    if N > 1:
        assert dead.numel() > 1000
        o2 = torch.sigmoid(params.leaves["opacity"].detach().view(-1))
        assert bool((o2 > 0.005).all())  # no row is dead right after a relocation


def test_relocate_nothing_to_do(cuda_device):
    """No dead row, or no live row: the arenas are left bit-identical."""
    from hidegs_b200 import trainer as tr
    dev = cuda_device
    for logit in (2.0, -8.0):
        params, adam = _model(5000, dev, seed=4, dead_frac=0.0)
        with torch.no_grad():
            params.leaves["opacity"].fill_(logit)
        before = [a.clone() for a in (params.param_arena, adam.exp_avg, adam.exp_avg_sq)]
        counts = tr.mcmc_relocate_arenas(params.param_arena, adam.exp_avg, adam.exp_avg_sq, 5000, 0.005, seed=1)[3]
        assert int(counts["dead"]) == (0 if logit > 0 else 5000)
        assert all(torch.equal(a, b) for a, b in zip((params.param_arena, adam.exp_avg, adam.exp_avg_sq), before))


@pytest.mark.parametrize("N", [1, 30001])
def test_grow_matches_oracle(cuda_device, N):
    from hidegs_b200 import trainer as tr
    from oracle import mcmc_oracle as mo
    dev = cuda_device
    params, adam = _model(N, dev, seed=5 + N)
    t, m, v = _dicts(params, adam)
    n2 = tr.mcmc_grow_target(N, 10 * N, 1.05) if N > 1 else 2
    g = torch.Generator().manual_seed(3)
    sources = torch.randint(0, N, (n2 - N,), generator=g)
    sources[: min(8, sources.numel())] = 0
    want = mo.grow(t, m, v, sources.to(dev), 0.005)
    before = [a.clone() for a in (params.param_arena, adam.exp_avg, adam.exp_avg_sq)]
    out = tr.mcmc_grow_arenas(params.param_arena, adam.exp_avg, adam.exp_avg_sq, N, n2, 0.005, sources=sources)
    assert out[3] == dict(added=n2 - N, n=n2)
    assert n2 == (int(1.05 * N) if N > 1 else 2)
    touched = torch.zeros(n2, dtype=torch.bool, device=dev)
    touched[N:] = True
    touched[sources.to(dev)] = True
    _compare(out[:3], n2, want, touched)
    # the old arenas are not touched
    assert all(torch.equal(a, b) for a, b in zip((params.param_arena, adam.exp_avg, adam.exp_avg_sq), before))
    # Philox draws: bit-identical across runs
    a = tr.mcmc_grow_arenas(params.param_arena, adam.exp_avg, adam.exp_avg_sq, N, n2, 0.005, seed=9)
    b = tr.mcmc_grow_arenas(params.param_arena, adam.exp_avg, adam.exp_avg_sq, N, n2, 0.005, seed=9)
    assert all(torch.equal(x, y) for x, y in zip(a[:3], b[:3]))


def _scene(dev, dead_frac=0.3):
    from test_trainer_gpu import _setup
    sc, cams, gts, tr = _setup(dev)
    g = torch.Generator().manual_seed(21)
    op = sc["opacity"].clamp_min(0.05)
    op[torch.rand(op.shape[0], generator=g) < dead_frac] = 3e-4
    sc = dict(sc, opacity=op)
    return sc, list(zip(cams, gts)), tr


def test_trainer_mcmc_end_to_end(cuda_device):
    dev = cuda_device
    sc, views, tr = _scene(dev)
    opt = type("Sched", (tr.OptimizationParams,), dict(mcmc_refine_from_iter=0, mcmc_refine_until_iter=1_000,
                                                        mcmc_refine_interval=3))
    params = tr.GaussianParams.from_scene(sc, dev)
    N0 = params.N
    cap = int(1.2 * N0)
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), opt=opt, mcmc=True, mcmc_cap_max=cap)
    # an explicit relocation first: no row is dead right after it
    o = torch.sigmoid(params.leaves["opacity"].detach())
    assert float((o <= 0.005).float().mean()) > 0.25
    counts = trainer.relocate_dead(seed=5)
    assert int(counts["dead"]) > 0.25 * N0
    assert bool((torch.sigmoid(params.leaves["opacity"].detach()) > 0.005).all())
    sizes, losses, n = [], [], N0
    for _ in range(15):
        losses.append(float(trainer.step(views).item()))
        if trainer.iteration % 3 == 0:
            n = tr.mcmc_grow_target(n, cap, 1.05)
        sizes.append(params.N)
        assert params.N == n <= cap
    assert sizes[-1] == cap and len(set(sizes)) > 3, sizes
    assert all(math.isfinite(x) for x in losses), losses
    assert trainer.adam.step_count == 15 and trainer.adam.exp_avg.numel() == params.param_arena.numel()
    for name, leaf in params.leaves.items():
        assert leaf.data_ptr() == params.param_arena[params.slices[name]].data_ptr(), name
        assert leaf.grad.data_ptr() == params.grad_arena[params.slices[name]].data_ptr(), name
    assert trainer.visible.numel() == params.N


def _image_loss_after(dev, refine, steps=30):
    sc, views, tr = _scene(dev)
    opt = type("Sched", (tr.OptimizationParams,), dict(mcmc_refine_from_iter=0,
                                                        mcmc_refine_until_iter=1_000 if refine else 0,
                                                        mcmc_refine_interval=5))
    params = tr.GaussianParams.from_scene(sc, dev)
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), opt=opt, mcmc=True,
                                    mcmc_cap_max=int(1.2 * params.N))
    for _ in range(steps):
        trainer.step(views)
    from hidegs_b200 import loss_utils as lu
    total = 0.0
    with torch.no_grad():
        for cam, gt in views:
            params.begin_view()
            img = trainer.view_loss(cam, gt, trainer.iteration)[1]["render"]
            total += float(lu.l1_loss(img.clamp(0, 1), gt))
    return total / len(views)


def test_trainer_mcmc_refinement_lowers_the_image_loss(cuda_device):
    """Same scene (30 % dead rows), same seeds, 30 steps: the mean L1 image loss is lower with refinement every 5
    steps than with mcmc_refine_until_iter = 0 (regulariser and noise in both).  Measured on a B200: 0.051715 with
    refinement, 0.052433 without."""
    dev = cuda_device
    with_refine = _image_loss_after(dev, True)
    without = _image_loss_after(dev, False)
    print("image L1 after 30 steps: refine %.6f, no refine %.6f" % (with_refine, without))
    assert with_refine < without, (with_refine, without)


def test_refinement_makes_no_host_synchronisation(cuda_device):
    dev = cuda_device
    sc, views, tr = _scene(dev)
    params = tr.GaussianParams.from_scene(sc, dev)
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), mcmc=True, mcmc_cap_max=2 * params.N)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        trainer.relocate_dead()
        counts = trainer.grow()
        trainer._mcmc_schedule()
        tr.mcmc_regularizer(params.param_arena, params.grad_arena, params.N, 0.01, 0.01, workspace=trainer._mcmc_ws)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert counts["n"] == params.N == int(1.05 * len(sc["opacity"]))


def test_mcmc_off_keeps_the_constant_position_rate(cuda_device):
    """mcmc=False (the default): no MCMC state, the xyz rate stays position_lr_init x spatial_lr_scale, N unchanged."""
    dev = cuda_device
    sc, views, tr = _scene(dev, dead_frac=0.0)
    params = tr.GaussianParams.from_scene(sc, dev)
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev))
    for _ in range(2):
        trainer.step(views)
    assert not trainer.mcmc and not hasattr(trainer, "_mcmc_ws")
    assert trainer.adam.lr["xyz"] == tr.OptimizationParams.position_lr_init and params.N == len(sc["opacity"])


def test_mcmc_multi_gpu_ranks_stay_identical(cuda_device):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    world = torch.cuda.device_count()
    env = dict(os.environ, PYTHONPATH=ROOT)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr",
           "127.0.0.1", "--master-port", "29547", os.path.join(ROOT, "tools", "mcmc_probe.py"), "--check"]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    out = json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])
    assert out["world"] == world
    assert out["ranks_identical"] and out["n_after"] > out["n_before"], out
    assert out["losses_finite"], out
