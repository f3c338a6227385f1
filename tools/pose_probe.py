"""Camera pose refinement in the training step (ViewShardedTrainer(train_poses=True), DESIGN.md §3 / §4).

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/pose_probe.py --check
        cameras of four named images, three of them off their true pose, spread over the ranks; after a few steps the
        pose tables of all ranks are bit-identical and equal, within float tolerance, the table of a single process
        (run on every rank before the process group exists) that renders all views of every step.  One JSON line.
    python tools/pose_probe.py --time [--steps 10 --rounds 3]
        one GPU: the configs[4] step (2M-Gaussian UAV slab, 1920x1080, 8 views per step, ground-truth cache) with
        train_poses on and off, alternated in one run; CUDA-event times (the library's per-stage events) of the
        per-Gaussian backward, default against pose variant, and of hg_prologue_backward against
        hg_prologue_backward_pose, at config 2's size (6M-Gaussian UAV slab, 3840x2160; every Gaussian one slot, as the
        pose variant needs); the card's name and power limit.  One JSON line.
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

CHECK_STEPS = ([0, 1, 2, 3, 0], [1, 2, 0], [3, 3, 1, 0])


def _check_setup(dev):
    from hidegs_b200 import gaussian_renderer as gr
    from hidegs_b200 import synthetic as syn
    W, H = 320, 208
    sc = syn.make_scene(30_000, seed=2, log_scale_mean=math.log(0.01 * 1920.0 / W))
    cams = []
    for k, (dx, dy) in enumerate(((0.0, 0.0), (0.3, 0.0), (0.0, 0.25), (-0.3, 0.1))):
        c = syn.default_camera(W, H, eye=(dx, dy, -5.0)).to(dev)
        c.image_name = "img_%d" % k
        cams.append(c)
    params = tr.GaussianParams.from_scene(sc, dev)
    with torch.no_grad():
        gts = [gr.render(c, params, tr.PipelineParams, torch.zeros(3, device=dev))["render"].clamp(0, 1).detach()
               for c in cams]
    g = torch.Generator().manual_seed(5)
    start = {c.image_name: (0.01 * torch.randn(6, generator=g) * (k > 0)).tolist() for k, c in enumerate(cams)}
    return sc, cams, gts, start


class _Opt(tr.OptimizationParams):
    pose_lr_translation = 1e-3
    pose_lr_rotation = 1e-3


def _run(sc, cams, gts, start, dev, rank, world):
    params = tr.GaussianParams.from_scene(sc, dev)
    params.setup_camera_poses([c.image_name for c in cams], poses=start)
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), opt=_Opt, train_poses=True)
    for ids in CHECK_STEPS:
        views = [(cams[i], gts[i]) for i in ids]
        trainer.step(views[rank::world], total_views=len(views))
    torch.cuda.synchronize()
    return params._camera_pose.detach().clone()


def check():
    rank, local, world = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sc, cams, gts, start = _check_setup(dev)
    single = _run(sc, cams, gts, start, dev, 0, 1)  # before the process group exists: plain arenas, world 1
    dist.init_process_group("nccl", device_id=dev)
    table = _run(sc, cams, gts, start, dev, rank, world)
    t0 = table.clone()
    dist.broadcast(t0, 0)
    same = torch.tensor([int(torch.equal(t0, table))], device=dev)
    err = (table - single).abs().max() / single.abs().max()
    first = torch.tensor([start[c.image_name] for c in cams], device=dev)
    moved = (single[:, :6] - first).abs().max()
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    dist.all_reduce(err, op=dist.ReduceOp.MAX)
    # the ranks sum their views' gradients in another order than one process does: float tolerance, not bits
    out = {"world": world, "ranks_identical": bool(same.item()), "max_rel_err_vs_single_process": float(err),
           "equals_single_process": bool(float(err) <= 1e-5), "table_moved": float(moved)}
    if rank == 0:
        print(json.dumps(out))
    dist.destroy_process_group()


def kernel_times(dev, reps=20):
    """Per-stage CUDA-event times (hg_profile_*) of the rasterizer's per-Gaussian backward, default and pose variant,
    and CUDA-event times of the prologue backward, at config 2's size."""
    from hidegs_b200 import _lib, synthetic as syn
    from hidegs_b200._geometry_lib import lib as G
    from hidegs_b200.diff_gaussian_rasterization import _C
    W, H = 3840, 2160
    scene = syn.make_uav_scene(6_000_000, seed=0)
    cam = syn.uav_camera(3, 4, width=W, height=H).to(dev)
    rs = syn.raster_settings(cam, dev)
    N = scene["means3D"].size(0)
    x = {k: v.to(dev).contiguous() for k, v in scene.items()}
    e = torch.empty(0, device=dev)
    all_map = torch.zeros(N, 5, device=dev)
    fwd = _C.rasterize_gaussians(rs.bg, rs.render_indices, rs.parent_indices, rs.interpolation_weights, rs.num_node_kids,
                                 x["means3D"], e, all_map, x["opacity"], x["scales"], x["rotations"], 1.0, e,
                                 rs.viewmatrix, rs.projmatrix, rs.tanfovx, rs.tanfovy, H, W, x["shs"], 3, rs.campos,
                                 False, True, False, True)
    g = syn.upstream_grads(W, H)
    g = {k: v.to(dev) for k, v in g.items()}
    args = (rs.bg, fwd[4], rs.render_indices, rs.parent_indices, rs.interpolation_weights, rs.num_node_kids,
            x["means3D"], fwd[2], e, all_map, x["opacity"], x["scales"], x["rotations"], 1.0, e, rs.viewmatrix,
            rs.projmatrix, rs.tanfovx, rs.tanfovy, g["color"], g["all_map"], g["plane_depth"], g["invdepth"], x["shs"], 3,
            rs.campos, fwd[6], fwd[0], fwd[7], fwd[8], True, False)
    ws = torch.empty(int(G().hg_camera_pose_workspace_bytes(N)), dtype=torch.uint8, device=dev)
    sink = torch.zeros_like(x["shs"])
    res = {"gaussians": N, "image": [W, H], "num_rendered": int(fwd[0])}
    for _ in range(2):  # second pass reported
        for name, kw in (("preprocess_bwd", {}), ("preprocess_bwd_pose", {"pose_workspace": ws})):
            _C.rasterize_gaussians_backward(*args, sh_sink=(sink, 0.0), skip_culled_rows=True, **kw)
            torch.cuda.synchronize()
            _lib.profile_collect()
            _lib.profile_enable(True)
            for _ in range(reps):
                _C.rasterize_gaussians_backward(*args, sh_sink=(sink, 0.0), skip_culled_rows=True, **kw)
            torch.cuda.synchronize()
            st = _lib.profile_collect()
            _lib.profile_enable(False)
            res[name + "_us"] = round(st["preprocess_bwd"][0] * 1e3 / st["preprocess_bwd"][1], 2)
    # prologue backward over the same rows (the rasterizer's outputs as its gradients)
    gb = _C.rasterize_gaussians_backward(*args, sh_sink=(sink, 0.0), skip_culled_rows=True)
    raw_s, raw_o = torch.log(x["scales"]), torch.zeros(N, 1, device=dev)
    d = [torch.empty(N, w, device=dev) for w in (3, 1, 3, 4)]
    radii = fwd[2]
    stream = torch.cuda.current_stream().cuda_stream

    def pro(pose):
        a = (raw_s.data_ptr(), x["rotations"].data_ptr(), raw_o.data_ptr(), x["means3D"].data_ptr(), N, 48,
             radii.data_ptr(), rs.viewmatrix.data_ptr(), rs.campos.data_ptr(), gb[3].data_ptr(), None, gb[2].data_ptr(),
             gb[6].data_ptr(), gb[7].data_ptr(), gb[8].data_ptr(), None, None, 0.0, d[0].data_ptr(), None,
             d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr())
        rc = G().hg_prologue_backward_pose(*a, ws.data_ptr(), stream) if pose else G().hg_prologue_backward(*a, stream)
        assert rc == 0
    for _ in range(2):
        for name, pose in (("prologue_bwd", False), ("prologue_bwd_pose", True)):
            pro(pose)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                pro(pose)
            e1.record()
            torch.cuda.synchronize()
            res[name + "_us"] = round(e0.elapsed_time(e1) * 1e3 / reps, 2)
    res["preprocess_bwd_pose_over_default"] = round(res["preprocess_bwd_pose_us"] / res["preprocess_bwd_us"], 4)
    res["prologue_bwd_pose_over_default"] = round(res["prologue_bwd_pose_us"] / res["prologue_bwd_us"], 4)
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
            params.setup_camera_poses([c.image_name for c in cams])
        trainers[on] = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), cache_ground_truth=True,
                                             start_iteration=tr.OptimizationParams.freq_warmup_iterations,
                                             train_poses=on)
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
    res = {"card": name, "power_limit": power,
           "step": {"workload": "configs[4] recipe on one GPU: 2M-Gaussian UAV slab, %dx%d, 8 views per step, ground-truth "
                                "cache on" % (W, H), "steps_per_round": steps, "rounds": rounds,
                    "ms_per_step_off": [round(x, 3) for x in ms[False]], "ms_per_step_on": [round(x, 3) for x in ms[True]],
                    "median_off": round(off_ms, 3), "median_on": round(on_ms, 3),
                    "per_view_ms_off": round(off_ms / 8, 3), "per_view_ms_on": round(on_ms / 8, 3),
                    "on_over_off": round(on_ms / off_ms, 4)},
           "kernels_config2": kernel_times(dev)}
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
