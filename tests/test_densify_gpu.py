"""Adaptive density control over the training arenas (hg_densify_plan / hg_densify_apply / hg_reset_opacity,
trainer.densify_arenas, ViewShardedTrainer.densify_and_prune / reset_opacity) against graphdeco 3DGS restated in
PyTorch (oracle/density_oracle.py), with the split draws injected; the RNG path on its own; the trainer end to end;
two or more ranks; and the C-ABI's argument checks (CPU)."""
import ctypes
import json
import math
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


def _random_model(N, dev, seed, split_all=False):
    """Raw parameters, moments and statistics with non-empty clone, split and prune sets (extent 5: percent_dense
    threshold 0.05, world-space size threshold 0.5)."""
    from hidegs_b200 import trainer as tr
    g = torch.Generator().manual_seed(seed)
    t = dict(xyz=torch.randn(N, 3, generator=g) * 2.0, features=torch.randn(N, 16, 3, generator=g),
             opacity=torch.randn(N, 1, generator=g) * 3.0,
             scaling=torch.empty(N, 3).uniform_(math.log(0.005), math.log(1.0), generator=g),
             rotation=torch.randn(N, 4, generator=g))
    accum = torch.rand(N, generator=g)
    if split_all:
        t["opacity"] = torch.full((N, 1), 4.0)
        t["scaling"] = torch.empty(N, 3).uniform_(math.log(0.06), math.log(0.4), generator=g)
        accum = torch.ones(N)
    accum[torch.rand(N, generator=g) < 0.05] = float("nan")
    params = tr.GaussianParams(*[t[k].to(dev) for k in ("xyz", "features", "opacity", "scaling", "rotation")])
    adam = tr.ArenaAdam(params)
    m, v = {}, {}
    for name, w in tr.GROUPS:
        sl = params.slices[name]
        adam.exp_avg[sl] = torch.randn(N * w, generator=g).to(dev)
        adam.exp_avg_sq[sl] = torch.rand(N * w, generator=g).to(dev)
        shape = (N, 16, 3) if name == "features" else (N, w)
        m[name], v[name] = adam.exp_avg[sl].view(shape).clone(), adam.exp_avg_sq[sl].view(shape).clone()
    denom = torch.randint(0, 5, (N,), generator=g).float().to(dev)
    radii = torch.rand(N, generator=g).to(dev) * 100.0
    return params, adam, accum.to(dev), denom, radii, m, v


def _split_samples(params, accum, max_grad, extent, seed, percent_dense=0.01):
    """The tensor torch.normal(mean=0, std=stds.repeat(2, 1)) of densify_and_split, drawn on the host."""
    g = accum.nan_to_num(0.0)
    sc = torch.exp(params.leaves["scaling"].detach())
    S = (g >= max_grad) & (sc.max(dim=1).values > percent_dense * extent)
    stds = sc[S].repeat(2, 1)
    z = torch.randn(stds.shape, generator=torch.Generator().manual_seed(seed)).to(stds.device)
    return stds * z


def _oracle(params, adam_step, accum, denom, radii, m, v):
    from oracle import density_oracle as do
    t = {k: params.leaves[k].detach().clone() for k in do.NAMES}
    return do.GaussianModel(t, m, v, adam_step, accum, denom, radii)


def _ulp_diff(a, b):
    return (a.contiguous().view(torch.int32).long() - b.contiguous().view(torch.int32).long()).abs()


def _compare(ours, counts, om, samples):
    """`ours` = (param arena, exp_avg, exp_avg_sq) of N' rows against the oracle model after its densify."""
    from oracle import density_oracle as do
    from hidegs_b200 import trainer as tr
    n = counts["n"]
    assert n == om._xyz.shape[0], (counts, om._xyz.shape)
    starts, total = tr.arena_layout(n)
    assert ours[0].numel() == total
    c0 = om.first_child_row
    widths = dict(tr.GROUPS)
    for name in do.NAMES:
        w = widths[name]
        st = om.state(name)
        want = dict(p=getattr(om, "_" + name).detach().reshape(n, w), m=st["exp_avg"].reshape(n, w),
                    v=st["exp_avg_sq"].reshape(n, w))
        got = {k: a[starts[name]:starts[name] + n * w].view(n, w) for k, a in zip("pmv", ours)}
        for k in "mv":  # kept rows keep their moments, clones and children start at zero: bit-equal everywhere
            assert torch.equal(got[k], want[k]), (name, k)
        if name in ("features", "opacity", "rotation"):  # copied raw
            assert torch.equal(got["p"], want["p"]), name
            continue
        assert torch.equal(got["p"][:c0], want["p"][:c0]), name  # kept rows and clones: bit-equal
        a, b = got["p"][c0:], want["p"][c0:]
        if a.numel() == 0:
            pass
        elif name == "scaling":
            assert int(_ulp_diff(a, b).max()) <= 1, name
        else:  # xyz: R s + xyz, the oracle's bmm sums in an unknown order: 1e-6 of the largest operand of the row
            s = samples[om.kept_children]
            mag = torch.maximum(b.abs().amax(dim=1, keepdim=True), s.abs().amax(dim=1, keepdim=True))
            assert bool(((a - b).abs() <= 1e-6 * mag).all()), float(((a - b).abs() / mag).max())
        # pad floats stay zero
        pad = ours[0][starts[name] + n * w:(starts[name] + n * w + 3) // 4 * 4]
        assert not pad.any()


@gpu
@pytest.mark.parametrize("N", [1, 1000, 30001])
@pytest.mark.parametrize("max_screen_size", [None, 20])
def test_densify_matches_oracle(cuda_device, N, max_screen_size):
    from hidegs_b200 import trainer as tr
    dev = cuda_device
    params, adam, accum, denom, radii, m, v = _random_model(N, dev, seed=N)
    max_grad, min_opacity, extent = 0.5, 0.05, 5.0
    samples = _split_samples(params, accum, max_grad, extent, seed=7)
    om = _oracle(params, 17, accum, denom, radii, m, v)
    ours = tr.densify_arenas(params.param_arena, adam.exp_avg, adam.exp_avg_sq, N, accum, max_grad, min_opacity, extent,
                             max_screen_size, samples=samples)
    om.densify_and_prune(max_grad, min_opacity, extent, max_screen_size, samples=samples)
    counts = ours[3]
    if N >= 1000:
        assert counts["cloned"] > 0 and counts["split"] > 0 and counts["pruned"] > 0, counts
    _compare(ours[:3], counts, om, samples)
    assert int(om.state("xyz")["step"]) == 17
    for s in (om.xyz_gradient_accum, om.denom, om.max_radii2D):
        assert s.shape[0] == counts["n"] and not s.any()


@gpu
def test_densify_boundaries(cuda_device):
    """g == max_grad clones or splits; smax == percent_dense * extent clones; sigmoid(opacity) == min_opacity is
    kept; NaN statistic and never-visited rows are not densified; nothing selected leaves the arenas bit-identical;
    the screen-size test sees the zeroed statistics (graphdeco quirk): a huge max_radii2D does not prune."""
    from hidegs_b200 import trainer as tr
    dev = cuda_device
    s_small, s_big = math.log(0.01), math.log(0.2)
    thr = float(torch.exp(torch.tensor(s_small, device=dev)))  # fp32 exp, as the kernel and torch see it
    o_edge = 0.3
    min_op = float(torch.sigmoid(torch.tensor(o_edge, device=dev)))
    rows = [  # (accum, scaling (log), opacity logit)
        (0.5, s_small, 2.0),          # 0: g == max_grad, smax == threshold: clone
        (0.5, s_big, 2.0),            # 1: g == max_grad, large: split
        (float("nan"), s_big, 2.0),   # 2: NaN: nothing
        (0.0, s_big, 2.0),            # 3: never visited: nothing
        (0.9, s_small, o_edge),       # 4: opacity exactly at min_opacity: kept, and cloned
        (0.1, s_small, o_edge - 1.0),  # 5: transparent: pruned
    ]
    N = len(rows)
    xyz = torch.randn(N, 3, device=dev)
    feats = torch.randn(N, 16, 3, device=dev)
    params = tr.GaussianParams(xyz, feats, torch.tensor([[r[2]] for r in rows], device=dev),
                               torch.tensor([[r[1]] * 3 for r in rows], device=dev), torch.randn(N, 4, device=dev))
    adam = tr.ArenaAdam(params)
    adam.exp_avg.normal_()
    adam.exp_avg_sq.uniform_()
    accum = torch.tensor([r[0] for r in rows], device=dev)
    new_p, new_m, new_v, counts = tr.densify_arenas(params.param_arena, adam.exp_avg, adam.exp_avg_sq, N, accum, 0.5,
                                                    min_op, thr, None, seed=3, percent_dense=1.0)
    assert counts == dict(kept=4, cloned=2, split=1, pruned=1, n=N + 2 + 1 - 1), counts
    starts, _ = tr.arena_layout(counts["n"])
    op = new_p[starts["opacity"]:starts["opacity"] + counts["n"]]
    # [rows 0, 2, 3, 4] ++ [clones of 0, 4] ++ [child 1 of 1] ++ [child 2 of 1]
    src = torch.tensor([0, 2, 3, 4, 0, 4, 1, 1], device=dev)
    assert torch.equal(op, params.leaves["opacity"].detach()[src, 0])
    # the size test against a huge max_radii2D never prunes: only the world-space test does (scales far below 0.1 extent)
    g = torch.Generator().manual_seed(1)
    n2 = 257
    p2 = tr.GaussianParams(torch.randn(n2, 3, device=dev), torch.randn(n2, 16, 3, device=dev),
                           torch.full((n2, 1), 3.0, device=dev), torch.full((n2, 3), math.log(0.01), device=dev),
                           torch.randn(n2, 4, device=dev))
    a2 = tr.ArenaAdam(p2)
    for name, w in tr.GROUPS:
        a2.exp_avg[p2.slices[name]] = torch.randn(n2 * w, generator=g).to(dev)
    radii = torch.full((n2,), 1e9, device=dev)
    acc = torch.zeros(n2, device=dev)
    from oracle import density_oracle as do
    om = do.GaussianModel({k: p2.leaves[k].detach() for k in do.NAMES},
                          {k: a2.exp_avg[p2.slices[k]].view(p2.leaves[k].shape) for k in do.NAMES},
                          {k: a2.exp_avg_sq[p2.slices[k]].view(p2.leaves[k].shape) for k in do.NAMES}, 5, acc,
                          torch.ones(n2, device=dev), radii)
    om.densify_and_prune(0.5, 0.005, 5.0, 20)
    out = tr.densify_arenas(p2.param_arena, a2.exp_avg, a2.exp_avg_sq, n2, acc, 0.5, 0.005, 5.0, 20)
    assert out[3] == dict(kept=n2, cloned=0, split=0, pruned=0, n=n2) and om._xyz.shape[0] == n2
    # nothing selected, nothing pruned: the three arenas come back bit-identical
    for a, b in zip(out[:3], (p2.param_arena, a2.exp_avg, a2.exp_avg_sq)):
        assert torch.equal(a, b)


@gpu
def test_densify_everything_pruned(cuda_device):
    from hidegs_b200 import trainer as tr
    from hidegs_b200._geometry_lib import lib as G
    dev = cuda_device
    N = 1000
    params = tr.GaussianParams(torch.randn(N, 3, device=dev), torch.randn(N, 16, 3, device=dev),
                               torch.full((N, 1), -8.0, device=dev), torch.full((N, 3), -3.0, device=dev),
                               torch.randn(N, 4, device=dev))
    accum = torch.ones(N, device=dev)
    ws = torch.empty(int(G().hg_densify_workspace_bytes(N)), dtype=torch.uint8, device=dev)
    starts, _ = tr.arena_layout(N)
    off = (ctypes.c_int64 * 5)(*[starts[n] for n, _ in tr.GROUPS])
    out = [ctypes.c_int64(-1) for _ in range(4)]
    rc = G().hg_densify_plan(params.param_arena.data_ptr(), off, N, accum.data_ptr(), 0, 0.5, 0.005, 5.0, 0.0, 0.01,
                             ws.data_ptr(), *[ctypes.byref(o) for o in out], torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    assert [o.value for o in out] == [0, N, 0, 0]  # every row cloned (small) and every row and clone pruned
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), densification_stats=True)
    trainer.xyz_gradient_accum.fill_(1.0)
    before = params.param_arena
    with pytest.raises(ValueError, match="no Gaussians"):
        trainer.densify_and_prune(0.5, 0.005, 5.0)
    assert params.N == N and params.param_arena is before


@gpu
def test_densify_rng(cuda_device):
    """Philox children: the same seed gives the same bits, another seed other children; R^T (xyz' - xyz) / s is
    standard normal per axis; the two children of a row differ."""
    from hidegs_b200 import trainer as tr
    from oracle import density_oracle as do
    dev = cuda_device
    N = 60_001
    params, adam, accum, *_ = _random_model(N, dev, seed=5, split_all=True)
    accum = torch.ones(N, device=dev)
    args = (params.param_arena, adam.exp_avg, adam.exp_avg_sq, N, accum, 0.5, 0.005, 5.0)
    a = tr.densify_arenas(*args, seed=123)
    b = tr.densify_arenas(*args, seed=123)
    c = tr.densify_arenas(*args, seed=124)
    assert a[3] == dict(kept=0, cloned=0, split=N, pruned=0, n=2 * N)
    assert all(torch.equal(x, y) for x, y in zip(a[:3], b[:3]))
    starts, _ = tr.arena_layout(2 * N)
    xa = a[0][starts["xyz"]:starts["xyz"] + 6 * N].view(2 * N, 3)
    xc = c[0][starts["xyz"]:starts["xyz"] + 6 * N].view(2 * N, 3)
    assert not torch.equal(xa, xc)
    x0 = params.leaves["xyz"].detach()
    R = do.build_rotation(params.leaves["rotation"].detach())
    s = torch.exp(params.leaves["scaling"].detach())
    z1 = torch.bmm(R.transpose(1, 2), (xa[:N] - x0).unsqueeze(-1)).squeeze(-1) / s
    z2 = torch.bmm(R.transpose(1, 2), (xa[N:] - x0).unsqueeze(-1)).squeeze(-1) / s
    z = torch.cat([z1, z2]).double()
    n = z.shape[0]
    assert n >= 100_000
    mean, std = z.mean(0), z.std(0)
    assert bool((mean.abs() <= 5.0 / math.sqrt(n)).all()), mean
    assert bool(((std - 1.0).abs() <= 0.02).all()), std
    assert bool((xa[:N] != xa[N:]).any(dim=1).all())  # the two children of every row differ


@gpu
def test_reset_opacity_matches_oracle(cuda_device):
    from hidegs_b200 import trainer as tr
    dev = cuda_device
    N = 30001
    params, adam, accum, denom, radii, m, v = _random_model(N, dev, seed=9)
    om = _oracle(params, 4, accum, denom, radii, m, v)
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev))
    trainer.adam = adam
    before = [t.clone() for t in (params.param_arena, adam.exp_avg, adam.exp_avg_sq)]
    trainer.reset_opacity()
    om.reset_opacity()
    sl = params.slices["opacity"]
    assert int(_ulp_diff(params.param_arena[sl], om._opacity.detach().reshape(-1)).max()) <= 1
    assert not adam.exp_avg[sl].any() and not adam.exp_avg_sq[sl].any()
    keep = torch.ones_like(before[0], dtype=torch.bool)
    keep[sl] = False
    for a, b in zip((params.param_arena, adam.exp_avg, adam.exp_avg_sq), before):
        assert torch.equal(a[keep], b[keep])


@gpu
def test_trainer_densify_end_to_end(cuda_device):
    """On the 30k synthetic scene: a densify changes N, the leaves and their .grad alias the new arenas, the direct
    executor still matches the autograd path, and a short schedule keeps the step count and lowers the loss."""
    from test_trainer_gpu import _setup
    dev = cuda_device
    sc, cams, gts, tr = _setup(dev)
    views = list(zip(cams, gts))
    params = tr.GaussianParams.from_scene(sc, dev, spatial_order=True)
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), densification_stats=True, start_iteration=1500)
    trainer.step(views)
    acc = trainer.xyz_gradient_accum.view(-1)
    thr = float(acc[acc > 0].quantile(0.8))
    assert abs(tr.cameras_extent(cams) - 1.1 * 0.15) <= 1e-6  # two centres 0.3 apart
    extent = 1.0
    N0 = params.N
    counts = trainer.densify_and_prune(thr, 0.005, extent, seed=11)
    assert params.N == counts["n"] != N0 and counts["cloned"] + counts["split"] > 0
    assert params.order is None and trainer.adam.step_count == 1
    assert trainer.adam.exp_avg.numel() == params.param_arena.numel() == params.grad_arena.numel()
    for name, leaf in params.leaves.items():
        assert leaf.data_ptr() == params.param_arena[params.slices[name]].data_ptr(), name
        assert leaf.grad.data_ptr() == params.grad_arena[params.slices[name]].data_ptr(), name
        assert leaf.shape[0] == params.N
    # the direct executor against the autograd path after the resize (test_direct_view_executor_matches_autograd)
    arenas, losses = {}, {}
    for direct in (True, False):
        params.zero_grad()
        ls = []
        for cam, gt in views:
            if direct:
                loss, _ = trainer.view_step_direct(cam, gt, 2000)
            else:
                loss, _ = trainer.view_loss(cam, gt, 2000)
                loss.backward()
            ls.append(float(loss.detach()))
        arenas[direct], losses[direct] = params.grad_arena.clone(), ls
    assert all(abs(x - y) <= 1e-6 * abs(y) + 1e-9 for x, y in zip(losses[True], losses[False]))
    err = (arenas[True] - arenas[False]).abs().max().item()
    assert err <= 1e-5 * arenas[False].abs().max().item() + 1e-12, err
    # the opt-in schedule: one densify after step 4 (0.9 quantile of the statistic; it perturbs the render, so the loss
    # jumps once), then 16 more steps
    opt = type("Sched", (tr.OptimizationParams,), dict(densify_from_iter=1500, densify_until_iter=1505,
                                                        densification_interval=4, opacity_reset_interval=100_000,
                                                        densify_grad_threshold=float(acc[acc > 0].quantile(0.9))))
    p2 = tr.GaussianParams.from_scene(sc, dev)
    t2 = tr.ViewShardedTrainer(p2, torch.zeros(3, device=dev), opt=opt, start_iteration=1500, densify=True,
                               scene_extent=extent)
    sizes, losses = [], []
    for _ in range(20):
        losses.append(float(t2.step(views).item()))
        sizes.append(p2.N)
    assert len(set(sizes)) > 1, sizes
    assert t2.adam.step_count == 20
    assert all(math.isfinite(x) for x in losses) and losses[-1] < losses[0], losses


@gpu
def test_densify_multi_gpu_ranks_stay_identical(cuda_device):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    world = torch.cuda.device_count()
    env = dict(os.environ, PYTHONPATH=ROOT)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr",
           "127.0.0.1", "--master-port", "29541", os.path.join(ROOT, "tools", "densify_probe.py"), "--check"]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    out = json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])
    assert out["world"] == world
    assert out["ranks_identical"] and out["equals_single_process"], out
    assert out["n_after"] != out["n_before"]
    assert out["step_loss_finite"] and out["ranks_identical_after_step"], out


def test_densify_abi_rejects_bad_arguments():
    """Argument checks before any CUDA work: no device needed (pointers are never dereferenced)."""
    from hidegs_b200 import _lib
    from hidegs_b200._geometry_lib import lib as G
    L = G()
    off = (ctypes.c_int64 * 5)(0, 4, 52, 56, 60)
    out = [ctypes.c_int64(0) for _ in range(4)]
    refs = [ctypes.byref(o) for o in out]
    fake = 4096
    assert L.hg_densify_plan(fake, off, -1, fake, 0, 0.5, 0.005, 1.0, 0.0, 0.01, fake, *refs, None) == 1
    assert b"bad argument" in L.hg_last_error()
    assert L.hg_densify_plan(None, off, 1, fake, 0, 0.5, 0.005, 1.0, 0.0, 0.01, fake, *refs, None) == 1
    assert L.hg_densify_plan(fake, off, 1, None, 0, 0.5, 0.005, 1.0, 0.0, 0.01, fake, *refs, None) == 1
    assert L.hg_densify_plan(fake, off, 1, fake, 0, 0.5, 0.005, 1.0, 0.0, 0.01, None, *refs, None) == 1
    assert L.hg_densify_plan(fake, off, 1, fake, 3, 0.5, 0.005, 1.0, 0.0, 0.01, fake, *refs, None) == 1
    assert b"skybox" in L.hg_last_error()
    bad_off = (ctypes.c_int64 * 5)(0, 2, 52, 56, 60)  # a group not on 16 bytes
    assert L.hg_densify_plan(fake, bad_off, 1, fake, 0, 0.5, 0.005, 1.0, 0.0, 0.01, fake, *refs, None) == 1
    assert L.hg_densify_apply(fake, fake, fake, off, -1, fake, fake, fake, off, 1, None, 0, fake, None) == 1
    assert L.hg_densify_apply(fake, None, fake, off, 1, fake, fake, fake, off, 1, None, 0, fake, None) == 1
    assert L.hg_densify_apply(fake, fake, fake, off, 1, None, fake, fake, off, 1, None, 0, fake, None) == 1
    assert L.hg_densify_apply(fake, fake, fake, off, 1, fake, fake, fake, off, 3, None, 0, fake, None) == 1  # N' > 2N
    assert b"hg_densify_apply" in L.hg_last_error()
    assert L.hg_reset_opacity(fake, fake, fake, -1, None) == 1
    assert L.hg_reset_opacity(None, fake, fake, 1, None) == 1
    assert b"hg_reset_opacity" in L.hg_last_error()
    assert L.hg_densify_workspace_bytes(1000) >= 1000
    assert _lib.lib() is L
