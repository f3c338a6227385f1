"""Per-image exposure in the training step (ViewShardedTrainer(train_exposure=True), DESIGN.md §3 / §4).

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/exposure_probe.py --check
        cameras of four named images spread over the ranks; after a few steps the exposure tables of all ranks are
        bit-identical and equal, within 1e-6 relative, the table of a single process (run on every rank before the
        process group exists) that renders all views of every step.  One JSON line (rank 0).
    python tools/exposure_probe.py --time [--steps 10 --rounds 3]
        one GPU, configs[4] recipe (2M-Gaussian UAV slab, 1920x1080, 8 views per step, ground-truth cache): the step time
        with train_exposure on and off, alternated in one run; CUDA-event kernel times at 1920x1080 of
        hg_exposure_apply + hg_training_image_grad_exposure against clamp + hg_training_image_grad (inputs rotated over
        four buffer sets, 0.5 GB, so that they come from HBM, not L2), algorithmic bytes over kernel time against the
        6544 GB/s of BASELINE.md §2; the card's name and power limit.  One JSON line.
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from hidegs_b200 import trainer as tr  # noqa: E402


def _check_setup(dev):
    from hidegs_b200 import synthetic as syn
    W, H = 320, 208
    sc = syn.make_scene(30_000, seed=2, log_scale_mean=math.log(0.01 * 1920.0 / W))
    cams = []
    for k, (dx, dy) in enumerate(((0.0, 0.0), (0.3, 0.0), (0.0, 0.25), (-0.3, 0.1))):
        c = syn.default_camera(W, H, eye=(dx, dy, -5.0)).to(dev)
        c.image_name = "img_%d" % k
        cams.append(c)
    g = torch.Generator().manual_seed(4)
    gts = [torch.nn.functional.avg_pool2d(torch.rand(1, 3, H, W, generator=g), 5, stride=1, padding=2)[0].clamp(0, 1)
           .to(dev) for _ in cams]
    return sc, cams, gts


# the views of every step: camera indices (a repeated camera, and a camera that sits out a step)
CHECK_STEPS = ([0, 1, 2, 3, 0], [1, 2, 0], [3, 3, 1, 0])


def _run(sc, cams, gts, dev, rank, world):
    params = tr.GaussianParams.from_scene(sc, dev)
    params.setup_exposures([c.image_name for c in cams])
    # past the exposure lr's delay ramp, so that the table moves
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), train_exposure=True, start_iteration=6000)
    for ids in CHECK_STEPS:
        views = [(cams[i], gts[i]) for i in ids]
        trainer.step(views[rank::world], total_views=len(views))
    torch.cuda.synchronize()
    return params._exposure.detach().clone()


def check():
    rank, local, world = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sc, cams, gts = _check_setup(dev)
    single = _run(sc, cams, gts, dev, 0, 1)  # before the process group exists: plain arenas, world 1
    dist.init_process_group("nccl", device_id=dev)
    table = _run(sc, cams, gts, dev, rank, world)
    t0 = table.clone()
    dist.broadcast(t0, 0)
    same = torch.tensor([int(torch.equal(t0, table))], device=dev)
    err = (table - single).abs().max() / single.abs().max()
    moved = (single - torch.eye(3, 4, device=dev)).abs().max()
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    dist.all_reduce(err, op=dist.ReduceOp.MAX)
    out = {"world": world, "ranks_identical": bool(same.item()), "max_rel_err_vs_single_process": float(err),
           "equals_single_process": bool(float(err) <= 1e-6), "table_moved": float(moved)}
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


def kernel_times(dev, H=1080, W=1920, reps=200, sets=4):
    """CUDA-event time per call (mean over `reps` calls, inputs rotated over `sets` buffer sets)."""
    from hidegs_b200 import loss_utils as lu
    L = lu._L()
    st = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device=dev).manual_seed(0)
    hw = H * W
    bufs = []
    for _ in range(sets):
        color = torch.rand(3, H, W, generator=g, device=dev) * 1.2 - 0.1
        gt = torch.rand(3, H, W, generator=g, device=dev)
        gs = torch.randn(3, H, W, generator=g, device=dev) / (3 * hw)
        gf = torch.randn(3, H, W, generator=g, device=dev) / (3 * hw)
        out = torch.empty_like(color)
        img = torch.empty_like(color)
        bufs.append((color, gt, gs, gf, out, img))
    E = (torch.eye(3, 4, device=dev) + 0.05 * torch.randn(3, 4, generator=g, device=dev)).contiguous()
    eg = torch.zeros(12, device=dev)
    wf = torch.ones((), device=dev)
    ws = torch.zeros(int(L.hg_exposure_grad_workspace_bytes(H, W)), dtype=torch.uint8, device=dev)

    def clamp(b):
        torch.clamp(b[0], 0, 1, out=b[5])

    def grad(b):
        rc = L.hg_training_image_grad(b[0].data_ptr(), b[1].data_ptr(), b[2].data_ptr(), b[3].data_ptr(), 3 * hw, 0.8,
                                      -0.2, wf.data_ptr(), b[4].data_ptr(), st)
        assert rc == 0

    def apply(b):
        rc = L.hg_exposure_apply(b[0].data_ptr(), E.data_ptr(), H, W, b[5].data_ptr(), st)
        assert rc == 0

    def grad_exp(b):
        rc = L.hg_training_image_grad_exposure(b[0].data_ptr(), E.data_ptr(), b[1].data_ptr(), b[2].data_ptr(),
                                               b[3].data_ptr(), H, W, 0.8, -0.2, wf.data_ptr(), b[4].data_ptr(),
                                               eg.data_ptr(), ws.data_ptr(), st)
        assert rc == 0
    res = {}
    nbytes = {"clamp": 24 * hw, "hg_training_image_grad": 60 * hw, "hg_exposure_apply": 24 * hw,
              "hg_training_image_grad_exposure": 60 * hw}
    fns = {"clamp": clamp, "hg_training_image_grad": grad, "hg_exposure_apply": apply,
           "hg_training_image_grad_exposure": grad_exp}
    for _ in range(2):  # second pass: the reported one (the first loads modules and warms clocks)
        for name, fn in fns.items():
            for i in range(sets):
                fn(bufs[i])
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(reps):
                fn(bufs[i % sets])
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / reps
            res[name] = {"us": round(us, 2), "bytes": nbytes[name], "GBps": round(nbytes[name] / (us * 1e-6) / 1e9, 1),
                         "share_of_6544": round(nbytes[name] / (us * 1e-6) / 1e9 / 6544, 3)}
    base = res["clamp"]["us"] + res["hg_training_image_grad"]["us"]
    new = res["hg_exposure_apply"]["us"] + res["hg_training_image_grad_exposure"]["us"]
    res["pair_us_off"], res["pair_us_on"] = round(base, 2), round(new, 2)
    res["grad_ratio_exposure_over_plain"] = round(res["hg_training_image_grad_exposure"]["us"]
                                                  / res["hg_training_image_grad"]["us"], 3)
    return res


def timing(steps, rounds):
    from hidegs_b200 import synthetic as syn
    dev = torch.device("cuda", 0)
    name, power = card()
    W, H = 1920, 1080
    scene = syn.make_uav_scene(2_000_000, seed=0)
    cams = []
    for j in range(8):  # bench.py's views of one GPU: the first 8 of its Latin-square order
        c = syn.uav_camera(0, j, width=W, height=H).to(dev)
        c.image_name = "uav_0_%d" % j
        cams.append(c)
    g = torch.Generator(device=dev).manual_seed(11)
    gts = [torch.nn.functional.avg_pool2d(torch.rand(1, 3, H, W, generator=g, device=dev), 5, stride=1, padding=2)[0]
           .clamp(0, 1) for _ in cams]
    trainers = {}
    for on in (False, True):
        params = tr.GaussianParams.from_scene(scene, dev, spatial_order=True)
        if on:
            params.setup_exposures([c.image_name for c in cams])
        trainers[on] = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), cache_ground_truth=True,
                                             start_iteration=tr.OptimizationParams.freq_warmup_iterations,
                                             train_exposure=on)
    views = list(zip(cams, gts))
    for on in (False, True):  # warm-up: modules, ground-truth caches, allocator
        for _ in range(3):
            trainers[on].step(views)
    torch.cuda.synchronize()
    ms = {False: [], True: []}
    for _ in range(rounds):
        for on in (False, True):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                loss = trainers[on].step(views)
            e1.record()
            torch.cuda.synchronize()
            assert torch.isfinite(loss).item()
            ms[on].append(e0.elapsed_time(e1) / steps)
    off_ms, on_ms = sorted(ms[False])[len(ms[False]) // 2], sorted(ms[True])[len(ms[True]) // 2]
    del trainers
    torch.cuda.empty_cache()
    res = {"card": name, "power_limit": power, "peak_GBps": 6544,
           "step": {"workload": "configs[4] recipe on one GPU: 2M-Gaussian UAV slab, %dx%d, 8 views per step, ground-truth "
                                "cache on" % (W, H), "steps_per_round": steps, "rounds": rounds,
                    "ms_per_step_off": [round(x, 3) for x in ms[False]], "ms_per_step_on": [round(x, 3) for x in ms[True]],
                    "median_off": round(off_ms, 3), "median_on": round(on_ms, 3),
                    "on_over_off": round(on_ms / off_ms, 4)},
           "kernels_1080p": kernel_times(dev)}
    print(json.dumps(res))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--time", action="store_true")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if a.check:
        check()
    else:
        timing(a.steps, a.rounds)
