"""3DGS-MCMC densification, the parts that need no GPU: the oracle's relocation formula against a float64 / math.comb
restatement, the refinement schedule and growth arithmetic, the position learning-rate schedule, the C-ABI's argument
checks (pointers are never dereferenced) and the trainer's refusals."""
import ctypes
import math

import pytest
import torch

from oracle import mcmc_oracle as mo


def _denominator(op, n):
    return sum(math.comb(i - 1, k) * (-1.0) ** k / math.sqrt(k + 1) * op ** (k + 1)
               for i in range(1, n + 1) for k in range(i))


def test_relocation_formula_identity_and_restatement():
    """n = 1 returns (o, s); 1 - (1 - o')^n == o over a grid of o and n = 1..51; s' against a plain-Python
    restatement of the double sum."""
    grid = [0.005, 0.01, 0.05, 0.1, 0.3, 0.5, 0.7, 0.9, 0.99, 0.999]
    o = torch.tensor(grid, dtype=torch.float64)
    s = torch.rand(len(grid), 3, generator=torch.Generator().manual_seed(0), dtype=torch.float64) + 0.01
    op, s2 = mo.relocation(o, s, torch.ones(len(grid), dtype=torch.int64))
    assert torch.allclose(op, o, rtol=0, atol=1e-15) and torch.allclose(s2, s, rtol=1e-15, atol=0)
    for n in range(1, 52):
        op, s2 = mo.relocation(o, s, torch.full((len(grid),), n))
        assert float((1.0 - (1.0 - op) ** n - o).abs().max()) <= 1e-12, n
        for i, oi in enumerate(grid):
            o_p = 1.0 - (1.0 - oi) ** (1.0 / n)
            want = s[i] * oi / _denominator(o_p, n)
            assert torch.allclose(s2[i], want, rtol=1e-12, atol=0), (n, oi)
    # n is clamped to [1, 51]; the opacity clamp
    a = mo.relocation(o, s, torch.full((len(grid),), 80))
    b = mo.relocation(o, s, torch.full((len(grid),), 51))
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    op, _ = mo.relocation(torch.tensor([0.006, 1.0 - 1e-12]), s[:2], torch.tensor([51, 2]), min_opacity=0.005)
    assert float(op[0]) == 0.005 and float(op[1]) == 1.0 - 2.0 ** -23


def test_refinement_schedule_and_growth_arithmetic():
    from hidegs_b200 import trainer as tr
    o = tr.OptimizationParams
    assert (o.mcmc_refine_from_iter, o.mcmc_refine_until_iter, o.mcmc_refine_interval) == (500, 25_000, 100)
    assert (o.mcmc_min_opacity, o.mcmc_grow_factor, o.mcmc_noise_lr) == (0.005, 1.05, 5e5)
    assert (o.mcmc_opacity_reg, o.mcmc_scale_reg) == (0.01, 0.01)
    refining = [it for it in range(0, 30_001) if tr.mcmc_refines(it, o)]
    assert refining[0] == 600 and refining[-1] == 24_900 and len(refining) == 244  # 500 and 25000 themselves excluded
    assert all(it % 100 == 0 for it in refining)
    sched = type("S", (o,), dict(mcmc_refine_from_iter=0, mcmc_refine_until_iter=10, mcmc_refine_interval=3))
    assert [it for it in range(20) if tr.mcmc_refines(it, sched)] == [3, 6, 9]
    assert tr.mcmc_grow_target(1000, 10_000, 1.05) == 1050
    assert tr.mcmc_grow_target(2_000_000, 10_000_000, 1.05) == int(1.05 * 2_000_000)
    assert tr.mcmc_grow_target(999, 10_000, 1.05) == int(1.05 * 999) == 1048
    assert tr.mcmc_grow_target(1000, 1020, 1.05) == 1020  # capped
    assert tr.mcmc_grow_target(1020, 1020, 1.05) == 1020  # at the cap: unchanged
    assert tr.mcmc_grow_target(10, 1000, 1.05) == 10      # int(10.5) = 10: nothing to add
    # the growth rule from N0 under a cap: N never exceeds it and stops there
    n, seen = 30_000, []
    for _ in range(10):
        n = tr.mcmc_grow_target(n, 36_000, 1.05)
        seen.append(n)
    assert seen[:4] == [31_500, 33_075, 34_728, 36_000] and set(seen[3:]) == {36_000}


def test_position_lr_schedule():
    from hidegs_b200 import trainer as tr
    from hidegs_b200.optim import get_expon_lr_func
    o = tr.OptimizationParams
    assert (o.position_lr_final, o.position_lr_delay_mult, o.position_lr_max_steps) == (1.6e-6, 0.01, 30_000)
    p = tr.GaussianParams(torch.zeros(4, 3), torch.zeros(4, 16, 3), torch.zeros(4, 1), torch.zeros(4, 3),
                          torch.tensor([[1.0, 0, 0, 0]] * 4))
    p.fused = True  # (pretend: the schedule is host arithmetic; no kernel runs in the constructor below)
    ref = get_expon_lr_func(o.position_lr_init, o.position_lr_final, lr_delay_mult=o.position_lr_delay_mult,
                            max_steps=o.position_lr_max_steps)
    import hidegs_b200.trainer as trm
    orig = trm.mcmc_workspace
    trm.mcmc_workspace = lambda N, dev: torch.zeros(1, dtype=torch.uint8)
    try:
        t = tr.ViewShardedTrainer(p, torch.zeros(3), mcmc=True, mcmc_cap_max=8)
    finally:
        trm.mcmc_workspace = orig
    for it in (0, 1, 500, 7000, 15_000, 29_999, 30_000, 40_000):
        assert t.xyz_lr(it) == ref(it)
    assert t.xyz_lr(0) == o.position_lr_init and abs(t.xyz_lr(30_000) - o.position_lr_final) <= 1e-18
    # log-linear in between: the geometric mean at half way
    assert math.isclose(t.xyz_lr(15_000), math.sqrt(o.position_lr_init * o.position_lr_final), rel_tol=1e-12)


def test_mcmc_abi_rejects_bad_arguments():
    from hidegs_b200 import _lib
    from hidegs_b200._geometry_lib import lib as G
    L = G()
    off = (ctypes.c_int64 * 5)(0, 4, 52, 56, 60)
    bad_off = (ctypes.c_int64 * 5)(0, 2, 52, 56, 60)  # a group not on 16 bytes
    fake = 1 << 20  # never dereferenced: every call below fails its argument check first
    out = fake
    # regulariser
    assert L.hg_mcmc_regularizer(fake, fake, off, -1, 0, 0.01, 0.01, 1.0, 1.0, None, None, fake, None) == 1
    assert b"hg_mcmc_regularizer" in L.hg_last_error()
    assert L.hg_mcmc_regularizer(None, fake, off, 1, 0, 0.01, 0.01, 1.0, 1.0, None, None, fake, None) == 1
    assert L.hg_mcmc_regularizer(fake, None, off, 1, 0, 0.01, 0.01, 1.0, 1.0, None, None, fake, None) == 1
    assert L.hg_mcmc_regularizer(fake, fake, off, 1, 0, 0.01, 0.01, 1.0, 1.0, None, None, None, None) == 1
    assert L.hg_mcmc_regularizer(fake, fake, bad_off, 1, 0, 0.01, 0.01, 1.0, 1.0, None, None, fake, None) == 1
    assert L.hg_mcmc_regularizer(fake, fake, off, 1, 0, -0.01, 0.01, 1.0, 1.0, None, None, fake, None) == 1
    assert L.hg_mcmc_regularizer(fake, fake, off, 1, 2, 0.01, 0.01, 1.0, 1.0, None, None, fake, None) == 1
    assert b"skybox" in L.hg_last_error()
    assert L.hg_mcmc_regularizer(None, None, None, 0, 0, 0.01, 0.01, 1.0, 1.0, None, None, None, None) == 0  # N = 0
    # noise
    assert L.hg_mcmc_inject_noise(fake, off, -1, 0, 1.0, None, 0, None) == 1
    assert L.hg_mcmc_inject_noise(None, off, 1, 0, 1.0, None, 0, None) == 1
    assert L.hg_mcmc_inject_noise(fake + 4, off, 1, 0, 1.0, None, 0, None) == 1  # arena not on 16 bytes
    assert L.hg_mcmc_inject_noise(fake, bad_off, 1, 0, 1.0, None, 0, None) == 1
    assert L.hg_mcmc_inject_noise(fake, off, 1, 1, 1.0, None, 0, None) == 1
    assert b"skybox" in L.hg_last_error()
    # relocate
    args = lambda **k: [k.get("p", fake), k.get("m", fake), k.get("v", fake), k.get("off", off), k.get("N", 1),  # noqa: E731
                        k.get("sky", 0), k.get("mo", 0.005), None, k.get("ns", 0), 0, out, k.get("ws", fake), None]
    assert L.hg_mcmc_relocate(*args(N=-1)) == 1
    assert b"hg_mcmc_relocate" in L.hg_last_error()
    assert L.hg_mcmc_relocate(*args(N=(1 << 30) + 1)) == 1
    assert L.hg_mcmc_relocate(*args(p=None)) == 1
    assert L.hg_mcmc_relocate(*args(m=None)) == 1
    assert L.hg_mcmc_relocate(*args(v=fake + 8)) == 1
    assert L.hg_mcmc_relocate(*args(ws=None)) == 1
    assert L.hg_mcmc_relocate(*args(off=bad_off)) == 1
    assert L.hg_mcmc_relocate(*args(off=None)) == 1
    assert L.hg_mcmc_relocate(*args(mo=1.0)) == 1
    assert L.hg_mcmc_relocate(*args(ns=-1)) == 1
    assert L.hg_mcmc_relocate(*args(sky=5)) == 1
    assert b"skybox" in L.hg_last_error()
    # grow: N < N' <= 2 N ("cap < N" reaches the library as N' <= N)
    noff = (ctypes.c_int64 * 5)(0, 8, 104, 108, 116)  # the layout of 2 rows
    gargs = lambda **k: [fake, fake, fake, k.get("off", off), k.get("N", 1), k.get("np", fake), fake, fake,  # noqa: E731
                         k.get("noff", noff), k.get("nn", 2), k.get("sky", 0), 0.005, None, 0, k.get("ws", fake), None]
    assert L.hg_mcmc_grow(*gargs(N=-1)) == 1
    assert b"hg_mcmc_grow" in L.hg_last_error()
    assert L.hg_mcmc_grow(*gargs(N=0, nn=0)) == 1
    assert L.hg_mcmc_grow(*gargs(nn=1)) == 1      # N' = N
    assert L.hg_mcmc_grow(*gargs(N=2, nn=1)) == 1  # N' < N
    assert L.hg_mcmc_grow(*gargs(nn=3)) == 1      # N' > 2 N
    assert L.hg_mcmc_grow(*gargs(np=None)) == 1
    assert L.hg_mcmc_grow(*gargs(np=fake + 4)) == 1
    assert L.hg_mcmc_grow(*gargs(ws=None)) == 1
    assert L.hg_mcmc_grow(*gargs(noff=bad_off)) == 1
    assert L.hg_mcmc_grow(*gargs(sky=1)) == 1
    assert b"skybox" in L.hg_last_error()
    # the workspace: counter | regulariser partials | sampling buffers, each part 256-byte aligned, + 256 of slack
    up = lambda b: (b + 255) // 256 * 256  # noqa: E731
    N = 1000
    want = 256 + 256 + up(2 * 1 * 8) + up(8 * N) + 3 * up(4 * N) + 2 * up(8 * 4) + 2 * up(4 * 4) + up(16)
    assert L.hg_mcmc_workspace_bytes(N) == want
    assert L.hg_mcmc_workspace_bytes(-3) == L.hg_mcmc_workspace_bytes(0)
    assert _lib.lib() is L


def _cpu_params(n=10):
    from hidegs_b200 import trainer as tr
    g = torch.Generator().manual_seed(0)
    return tr.GaussianParams(torch.randn(n, 3, generator=g), torch.randn(n, 16, 3, generator=g),
                             torch.randn(n, 1, generator=g), torch.randn(n, 3, generator=g) - 3,
                             torch.randn(n, 4, generator=g))


def test_mcmc_trainer_refusals():
    from hidegs_b200 import trainer as tr
    bg = torch.zeros(3)
    p = _cpu_params()
    with pytest.raises(ValueError, match="densify"):
        tr.ViewShardedTrainer(p, bg, mcmc=True, mcmc_cap_max=100, densify=True, scene_extent=1.0)
    with pytest.raises(ValueError, match="mcmc_cap_max"):
        tr.ViewShardedTrainer(p, bg, mcmc=True, mcmc_cap_max=9)
    with pytest.raises(ValueError, match="mcmc_cap_max"):
        tr.ViewShardedTrainer(p, bg, mcmc=True)
    with pytest.raises(ValueError, match="CUDA"):
        tr.ViewShardedTrainer(p, bg, mcmc=True, mcmc_cap_max=100)
    sky = _cpu_params()
    sky.skybox_points = 4
    with pytest.raises(ValueError, match="skybox"):
        tr.ViewShardedTrainer(sky, bg, mcmc=True, mcmc_cap_max=100)
    bad = type("O", (tr.OptimizationParams,), dict(mcmc_grow_factor=2.5))
    with pytest.raises(ValueError, match="grow_factor"):
        tr.ViewShardedTrainer(p, bg, opt=bad, mcmc=True, mcmc_cap_max=100)
    # nothing changed, and the default is off
    assert p.N == 10 and p.order is None
    t = tr.ViewShardedTrainer(p, bg)
    assert not t.mcmc
    with pytest.raises(RuntimeError, match="mcmc=True"):
        t.relocate_dead()
    with pytest.raises(RuntimeError, match="mcmc=True"):
        t.grow()
    with pytest.raises(ValueError, match="2 N"):
        tr.mcmc_grow_arenas(p.param_arena, p.param_arena, p.param_arena, 10, 21)
