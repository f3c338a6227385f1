"""3DGS-MCMC densification over the training arenas (ViewShardedTrainer(mcmc=True), DESIGN.md §3 / §4).

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/mcmc_probe.py --check
        a 30k-Gaussian scene with 30 % dead rows, the views split over the ranks, six steps with a refinement every
        second one (cap 1.2 N): the parameter and moment arenas of all ranks are bit-identical after every step.  One
        JSON line (rank 0).
    python tools/mcmc_probe.py --time [--sizes 2000000 6000000 --steps 10 --rounds 3 --views 4]
        one GPU: CUDA-event times of the regulariser (48 B/row) and noise (56 B/row) kernels against the 6544 GB/s of
        BASELINE.md §2; one refinement (relocate with 10 % dead rows, then grow 2M -> 2.1M); the configs[3] training
        step with mcmc on (outside the refinement window) and off, alternated in one run; the card's name and power
        limit.  The step comparison rebuilds both trainers from the same scene every round.  One JSON line.
"""
import argparse
import json
import math
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from hidegs_b200 import trainer as tr  # noqa: E402
from exposure_probe import card  # noqa: E402


def check():
    rank, local, world = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    from hidegs_b200 import synthetic as syn
    W, H = 320, 208
    sc = syn.make_scene(30_000, seed=2, log_scale_mean=math.log(0.01 * 1920.0 / W))
    g = torch.Generator().manual_seed(21)
    op = sc["opacity"].clamp_min(0.05)
    op[torch.rand(op.shape[0], generator=g) < 0.3] = 3e-4
    sc = dict(sc, opacity=op)
    cams = [syn.default_camera(W, H, eye=(dx, 0.0, -5.0)).to(dev) for dx in (0.0, 0.3, -0.3, 0.15)]
    gts = [torch.nn.functional.avg_pool2d(torch.rand(1, 3, H, W, generator=g), 5, stride=1, padding=2)[0].clamp(0, 1)
           .to(dev) for _ in cams]
    opt = type("Sched", (tr.OptimizationParams,), dict(mcmc_refine_from_iter=0, mcmc_refine_until_iter=1_000,
                                                        mcmc_refine_interval=2))
    params = tr.GaussianParams.from_scene(sc, dev)
    n0 = params.N
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), opt=opt, mcmc=True, mcmc_cap_max=int(1.2 * n0))

    def identical(ts):
        ok = True
        for t in ts:
            t0 = t.clone()
            dist.broadcast(t0, 0)
            flag = torch.tensor([int(torch.equal(t0, t))], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            ok = ok and bool(flag.item())
        return ok
    views = list(zip(cams, gts))
    same, finite, sizes = True, True, []
    for _ in range(6):
        loss = trainer.step(views[rank::world], total_views=len(views))
        finite = finite and bool(torch.isfinite(loss).item())
        same = same and identical([params.param_arena, trainer.adam.exp_avg, trainer.adam.exp_avg_sq])
        sizes.append(params.N)
    out = {"world": world, "nvls": params.exchange is not None, "n_before": n0, "n_after": params.N, "sizes": sizes,
           "ranks_identical": same, "losses_finite": finite}
    if rank == 0:
        print(json.dumps(out))
    dist.destroy_process_group()


def _events(fn, reps):
    """Median CUDA-event time of fn() in ms over `reps` calls (one warm-up call first)."""
    fn()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return sorted(ms)[len(ms) // 2]


def _model(N, dev, dead_frac, seed=0):
    g = torch.Generator().manual_seed(seed)
    op = (torch.randn(N, 1, generator=g) * 1.5).clamp_min(-2.9)
    op[torch.rand(N, generator=g) < dead_frac] = -8.0
    p = tr.GaussianParams(torch.randn(N, 3, generator=g).to(dev), torch.randn(N, 16, 3, generator=g).to(dev), op.to(dev),
                          torch.empty(N, 3).uniform_(math.log(0.005), math.log(0.5), generator=g).to(dev),
                          torch.randn(N, 4, generator=g).to(dev))
    return p


def kernel_times(dev, sizes, reps=50):
    out = {}
    for N in sizes:
        p = _model(N, dev, 0.1)
        grad = torch.zeros_like(p.param_arena)
        ws = tr.mcmc_workspace(N, dev)
        reg_ms = _events(lambda: tr.mcmc_regularizer(p.param_arena, grad, N, 0.01, 0.01, workspace=ws), reps)
        noise_ms = _events(lambda: tr.mcmc_inject_noise(p.param_arena, N, 80.0, seed=1), reps)
        out[str(N)] = {"regularizer_ms": round(reg_ms, 4), "regularizer_GBps": round(48 * N / (reg_ms * 1e-3) / 1e9, 1),
                       "regularizer_share_of_6544": round(48 * N / (reg_ms * 1e-3) / 1e9 / 6544, 3),
                       "noise_ms": round(noise_ms, 4), "noise_GBps": round(56 * N / (noise_ms * 1e-3) / 1e9, 1),
                       "noise_share_of_6544": round(56 * N / (noise_ms * 1e-3) / 1e9 / 6544, 3)}
        del p, grad, ws
        torch.cuda.empty_cache()
    return out


def refinement_time(dev, N=2_000_000, reps=10):
    """relocate (10 % dead rows) then grow N -> int(1.05 N), on fresh copies of the same arenas every rep."""
    p = _model(N, dev, 0.1, seed=1)
    m = torch.zeros_like(p.param_arena)
    v = torch.zeros_like(p.param_arena)
    ws = tr.mcmc_workspace(N, dev)
    n2 = tr.mcmc_grow_target(N, 10 * N, 1.05)
    ms, reloc_ms = [], []
    for r in range(reps + 1):
        a = [p.param_arena.clone(), m.clone(), v.clone()]
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        counts = tr.mcmc_relocate_arenas(a[0], a[1], a[2], N, 0.005, seed=r, workspace=ws)[3]
        e[1].record()
        out = tr.mcmc_grow_arenas(a[0], a[1], a[2], N, n2, 0.005, seed=r, workspace=ws)
        e[2].record()
        e[2].synchronize()
        if r:  # (the first pass loads the modules)
            ms.append(e[0].elapsed_time(e[2]))
            reloc_ms.append(e[0].elapsed_time(e[1]))
        del out, a
    return {"N": N, "n_after_grow": n2, "dead": int(counts["dead"]), "relocate_ms": round(sorted(reloc_ms)[reps // 2], 4),
            "relocate_then_grow_ms": round(sorted(ms)[reps // 2], 4)}


def step_times(dev, steps, rounds, nviews):
    import bench
    from hidegs_b200 import synthetic as syn
    W, H = bench.WIDTH, bench.HEIGHT
    scene = syn.make_scene(2_000_000, seed=0)
    cams = [bench.camera_for(0, s).to(dev) for s in range(nviews)]
    g = torch.Generator(device=dev).manual_seed(11)
    gts = [torch.nn.functional.avg_pool2d(torch.rand(1, 3, H, W, generator=g, device=dev), 5, stride=1, padding=2)[0]
           .clamp(0, 1) for _ in cams]
    # outside the refinement window: what every step pays (regulariser, position schedule, noise)
    opt = type("NoRefine", (tr.OptimizationParams,), dict(mcmc_refine_from_iter=10 ** 9))
    views = list(zip(cams, gts))

    def make(on):
        params = tr.GaussianParams.from_scene(scene, dev, spatial_order=True)
        return tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), opt=opt, cache_ground_truth=True,
                                     start_iteration=tr.OptimizationParams.freq_warmup_iterations, mcmc=on,
                                     mcmc_cap_max=params.N if on else None)
    # every round starts both trainers from the same scene: the regulariser and the noise change the model, and with it
    # the rendering work of later steps, which is not the per-step cost of the MCMC passes
    ms = {False: [], True: []}
    for _ in range(rounds):
        for on in (False, True):
            trainer = make(on)
            for _ in range(3):  # warm-up: modules, ground-truth caches, allocator
                trainer.step(views)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                loss = trainer.step(views)
            e1.record()
            torch.cuda.synchronize()
            assert torch.isfinite(loss).item()
            ms[on].append(e0.elapsed_time(e1) / steps)
            del trainer
    off_ms, on_ms = sorted(ms[False])[len(ms[False]) // 2], sorted(ms[True])[len(ms[True]) // 2]
    torch.cuda.empty_cache()
    return {"workload": "configs[3] recipe on one GPU: 2M Gaussians, %dx%d, %d views per step, ground-truth cache on, "
                        "mcmc outside its refinement window; both trainers rebuilt from the scene every round" % (W, H, nviews),
            "steps_per_round": steps,
            "rounds": rounds, "ms_per_step_off": [round(x, 3) for x in ms[False]],
            "ms_per_step_on": [round(x, 3) for x in ms[True]], "median_off": round(off_ms, 3),
            "median_on": round(on_ms, 3), "on_over_off": round(on_ms / off_ms, 4)}


def timing(sizes, steps, rounds, nviews):
    dev = torch.device("cuda", 0)
    name, power = card()
    res = {"card": name, "power_limit": power, "peak_GBps": 6544, "kernels": kernel_times(dev, sizes),
           "refinement": refinement_time(dev), "step": step_times(dev, steps, rounds, nviews)}
    print(json.dumps(res))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--time", action="store_true")
    ap.add_argument("--sizes", type=int, nargs="*", default=[2_000_000, 6_000_000])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--views", type=int, default=4)
    a = ap.parse_args()
    if a.check:
        check()
    else:
        timing(a.sizes, a.steps, a.rounds, a.views)
