"""Densify and prune over the training arenas (trainer.densify_arenas, DESIGN.md §3 / §4).

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/densify_probe.py --check
        every rank holds different densification statistics; after ViewShardedTrainer.densify_and_prune the arenas of
        all ranks are bit-identical and equal a single-process densify on the MAX / SUM-combined statistics; a training
        step then runs on the re-created gradient exchange.  One JSON line (rank 0).
    python tools/densify_probe.py --time [--sizes 2000000 6000000]
        one GPU: kernel time (CUDA events around plan and apply), end-to-end time of densify_arenas and of the PyTorch
        formulation (oracle/density_oracle.py) on the same inputs, bytes moved over kernel time against the 6544 GB/s
        of BASELINE.md §2, and the card's name and power limit.  One JSON line.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from hidegs_b200 import trainer as tr  # noqa: E402

ROW_BYTES = 4 * sum(w for _, w in tr.GROUPS)  # 236: one row of one arena


def _model(N, dev, seed):
    g = torch.Generator().manual_seed(seed)
    p = tr.GaussianParams(torch.randn(N, 3, generator=g).to(dev) * 2.0, torch.randn(N, 16, 3, generator=g).to(dev),
                          (torch.randn(N, 1, generator=g) * 3.0).to(dev),
                          torch.empty(N, 3).uniform_(math.log(0.005), math.log(1.0), generator=g).to(dev),
                          torch.randn(N, 4, generator=g).to(dev))
    return p, g


def check():
    rank, local, world = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    from hidegs_b200 import synthetic as syn
    W, H = 320, 208
    sc = syn.make_scene(30_000, seed=2, log_scale_mean=math.log(0.01 * 1920.0 / W))
    cams = [syn.default_camera(W, H, eye=(dx, 0.0, -5.0)).to(dev) for dx in (0.0, 0.3)]
    g = torch.Generator().manual_seed(4)
    gts = [torch.nn.functional.avg_pool2d(torch.rand(1, 3, H, W, generator=g), 5, stride=1, padding=2)[0].clamp(0, 1)
           .to(dev) for _ in cams]
    params = tr.GaussianParams.from_scene(sc, dev)
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), densification_stats=True, start_iteration=1500)
    N = params.N
    # different statistics on every rank
    gr = torch.Generator().manual_seed(1000 + rank)
    trainer.xyz_gradient_accum.copy_(torch.rand(N, 1, generator=gr).to(dev))
    trainer.denom.copy_(torch.randint(0, 4, (N, 1), generator=gr).float().to(dev))
    trainer.max_radii2D.copy_(torch.rand(N, generator=gr).to(dev) * 50)
    trainer.adam.exp_avg[params.slices["xyz"]] = 0.5  # moments that the kept rows must carry over
    stats = [trainer.xyz_gradient_accum.clone(), trainer.denom.clone(), trainer.max_radii2D.clone()]
    old = [params.param_arena.clone(), trainer.adam.exp_avg.clone(), trainer.adam.exp_avg_sq.clone()]
    counts = trainer.densify_and_prune(0.9, 0.005, 1.0, 20, seed=77)
    after = [params.param_arena, trainer.adam.exp_avg, trainer.adam.exp_avg_sq]
    # the single-process densify on the combined statistics
    dist.all_reduce(stats[0], op=dist.ReduceOp.MAX)
    ref = tr.densify_arenas(old[0], old[1], old[2], N, stats[0].view(-1), 0.9, 0.005, 1.0, 20, seed=77)
    same_single = all(torch.equal(a, b) for a, b in zip(after, ref[:3]))

    def identical(ts):
        ok = True
        for t in ts:
            t0 = t.clone()
            dist.broadcast(t0, 0)
            flag = torch.tensor([int(torch.equal(t0, t))], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            ok = ok and bool(flag.item())
        return ok
    out = {"world": world, "nvls": params.exchange is not None, "n_before": N, "n_after": params.N, "counts": counts,
           "ranks_identical": identical(after), "equals_single_process": same_single}
    loss = trainer.step(list(zip(cams, gts))[rank::world], total_views=len(cams))
    torch.cuda.synchronize()
    out["step_loss_finite"] = bool(torch.isfinite(loss).item())
    out["ranks_identical_after_step"] = identical([params.param_arena])
    flag = torch.tensor([int(out["ranks_identical"] and same_single)], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    out["equals_single_process"] = out["equals_single_process"] and bool(flag.item())
    if rank == 0:
        print(json.dumps(out))
    dist.destroy_process_group()


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        power = q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def timing(sizes, reps):
    from oracle import density_oracle as do
    dev = torch.device("cuda", 0)
    name, power = card()
    res = {"card": name, "power_limit": power, "peak_GBps": 6544, "sizes": {}}
    for N in sizes:
        p, g = _model(N, dev, seed=N)
        m = torch.randn(p.param_arena.numel(), generator=g).to(dev)
        v = torch.rand(p.param_arena.numel(), generator=g).to(dev)
        accum = torch.rand(N, generator=g).to(dev)
        args = (p.param_arena, m, v, N, accum, 0.9, 0.005, 5.0, 20)
        out = tr.densify_arenas(*args, seed=1)  # warm-up (module load)
        counts = out[3]
        del out
        # kernel time: events around the plan (incl. its one read-back) and the apply, from the library directly
        ev = []
        orig_apply = tr._G().hg_densify_apply
        orig_plan = tr._G().hg_densify_plan

        def wrap(fn, slot):
            def f(*a):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                rc = fn(*a)
                e1.record()
                ev.append((slot, e0, e1))
                return rc
            return f
        L = tr._G()
        L.hg_densify_plan, L.hg_densify_apply = wrap(orig_plan, "plan"), wrap(orig_apply, "apply")
        try:
            e2e = []
            for r in range(reps):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = tr.densify_arenas(*args, seed=r)
                torch.cuda.synchronize()
                e2e.append(time.perf_counter() - t0)
                del out
        finally:
            L.hg_densify_plan, L.hg_densify_apply = orig_plan, orig_apply
        plan_ms = sorted(e0.elapsed_time(e1) for s, e0, e1 in ev if s == "plan")
        apply_ms = sorted(e0.elapsed_time(e1) for s, e0, e1 in ev if s == "apply")
        kern_ms = plan_ms[len(plan_ms) // 2] + apply_ms[len(apply_ms) // 2]
        n2 = counts["n"]
        # parameters of every source row, the moments of the kept ones, accum, the flag byte (written, read), every
        # float of the three new arenas
        nbytes = N * (ROW_BYTES + 4 + 2) + counts["kept"] * 2 * ROW_BYTES + 3 * n2 * ROW_BYTES
        # the PyTorch formulation on the same inputs
        starts, _ = tr.arena_layout(N)
        shape = {k: ((N, 16, 3) if k == "features" else (N, w)) for k, w in tr.GROUPS}

        def part(a, k):
            return a[starts[k]:starts[k] + N * dict(tr.GROUPS)[k]].view(shape[k])
        oracle_s = []
        for r in range(max(1, reps // 2)):
            om = do.GaussianModel({k: part(p.param_arena, k) for k in do.NAMES}, {k: part(m, k) for k in do.NAMES},
                                  {k: part(v, k) for k in do.NAMES}, 1, accum, torch.ones(N, device=dev),
                                  torch.zeros(N, device=dev))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            om.densify_and_prune(0.9, 0.005, 5.0, 20)
            torch.cuda.synchronize()
            oracle_s.append(time.perf_counter() - t0)
            del om
        res["sizes"][str(N)] = {
            "counts": counts, "plan_ms": plan_ms[len(plan_ms) // 2], "apply_ms": apply_ms[len(apply_ms) // 2],
            "kernel_ms": kern_ms, "e2e_ms": 1e3 * sorted(e2e)[len(e2e) // 2],
            "oracle_e2e_ms": 1e3 * sorted(oracle_s)[len(oracle_s) // 2], "bytes": nbytes,
            "GBps_kernel": nbytes / (kern_ms * 1e-3) / 1e9, "share_of_6544": nbytes / (kern_ms * 1e-3) / 1e9 / 6544}
        del p, m, v, accum
        torch.cuda.empty_cache()
    print(json.dumps(res))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--time", action="store_true")
    ap.add_argument("--sizes", type=int, nargs="*", default=[2_000_000, 6_000_000])
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    if a.check:
        check()
    else:
        timing(a.sizes, a.reps)
