#!/usr/bin/env python
"""bench.py — headline benchmark of the rasterizer hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1], SURVEY.md §8(d) config 2): synthetic 1M-Gaussian
scene, SH degree 3, one 1920x1080 view per step, rasterizer forward + backward with
all outputs on (colour, 5-channel geometry map, plane depth, inverse depth).
One "step" = one view forward+backward per GPU; with N > 1 every rank renders its own
camera of the replicated scene and the ranks all-reduce the 59-float/Gaussian gradient
arena over NCCL (view-sharded data parallelism, weak scaling).

Rank 0 prints ONE JSON line:
  value     fwd+bwd Mpix/s with every input resident in HBM (CUDA events, max over ranks)
  e2e       same metric through the public API (GaussianRasterizer + autograd) with the
            step's host inputs (camera matrices + ground-truth image, pinned) copied H2D
            and the loss read back D2H inside the timed region
  roofline  dominant kernel: algorithmic bytes / live CUDA-event time vs measured HBM peak
  cpu_baseline  the CPU restatement (oracle/) timed on the host cores on the same workload

`--impl reference` runs the UNMODIFIED reference CUDA rasterizer rebuilt for sm_100
(oracle/_ref/ref_rasterizer_C.so) on the same inputs / metric; the reference has no CPU
implementation of this path, so its own implementation is timed on the same GPU.  If that
build is absent the CPU restatement is timed instead (kind "port").

`--dump-outputs DIR` writes what the last timed step of the device-resident leg returned (rank 0) as DIR/<name>.npy
in float32 (integer outputs as float64): the forward's images and per-Gaussian radii / observe counts, num_rendered,
and the nine gradient arrays of the backward.  Larger outputs are stored as a fixed sample that depends only on their
shape (seeded pixel and Gaussian indices, at most DUMP_PIXELS / DUMP_GAUSSIANS of them, about 52 MB in all at the
default workload), so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark may run from a read-only tree: it leaves no __pycache__ behind

import numpy as np  # noqa: E402
import torch  # noqa: E402

N_GAUSS = int(os.environ.get("HG_BENCH_N", 1_000_000))
WIDTH = int(os.environ.get("HG_BENCH_W", 1920))
HEIGHT = int(os.environ.get("HG_BENCH_H", 1080))
METRIC = "fwd+bwd Mpix/s @1M Gaussians 1080p"
UNIT = "Mpix/s"
DUMP_PIXELS = 1 << 18     # sampled pixels of every image output (10 floats each over colour, all_map and depths)
DUMP_GAUSSIANS = 1 << 17  # sampled Gaussian rows of every per-Gaussian output (78 floats each)
GRAD_NAMES = ("dL_dmeans2D", "dL_dcolors", "dL_dopacity", "dL_dmeans3D", "dL_dcov3D", "dL_dsh", "dL_dscales",
              "dL_drotations", "dL_dall_map")  # the order rasterize_gaussians_backward returns them in


# ----------------------------------------------------------------------------- helpers
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    # no measurement on this machine: the HBM copy bandwidth the project measured on a B200 (BASELINE.md §2)
    return 6544.0, "BASELINE.md §2 (measured on a B200; power limit not recorded)"


def camera_for(rank, step):
    """Rank/step specific camera around the config-2 pose (rank 0, step 0 == the BASELINE pose)."""
    from hidegs_b200 import synthetic as syn
    dx = 0.25 * ((rank * 7 + step * 3) % 5 - 2) if (rank or step) else 0.0
    dy = 0.15 * ((rank * 5 + step) % 3 - 1) if (rank or step) else 0.0
    return syn.default_camera(WIDTH, HEIGHT, eye=(dx, dy, -5.0))


def _sample(n, k, seed):
    """Sorted indices of a fixed seeded sample of k of n elements (all of them when n <= k)."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False))


def dump_outputs(out_dir, fwd, grads):
    """Write the outputs of one rasterizer forward + backward call (see --dump-outputs) to out_dir/<name>.npy."""
    R, color, radii, observe, all_map, plane_depth, geom, binning, img, invdepth = fwd
    os.makedirs(out_dir, exist_ok=True)
    pix = torch.from_numpy(_sample(color.shape[1] * color.shape[2], DUMP_PIXELS, seed=1)).to(color.device)
    rows = torch.from_numpy(_sample(radii.shape[0], DUMP_GAUSSIANS, seed=2)).to(radii.device)
    out = {"num_rendered": np.array([R], np.float64)}
    for name, t in (("color", color), ("all_map", all_map), ("plane_depth", plane_depth), ("invdepth", invdepth)):
        out[name] = t.reshape(t.shape[0], -1).index_select(1, pix).float().cpu().numpy()
    for name, t in (("radii", radii), ("out_observe", observe)):
        out[name] = t.index_select(0, rows).cpu().numpy().astype(np.float64)
    for name, t in zip(GRAD_NAMES, grads):
        if t is not None:  # dL_dsh is None where the backward writes SH factors for a multi-GPU exchange instead
            out[name] = t.index_select(0, rows).float().cpu().numpy()
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def stage_bytes(N, Nv, R, HW, T):
    """Algorithmic bytes per launch of each stage (DESIGN.md §4, from SURVEY.md §8(d))."""
    return {
        "preprocess_fwd": 56 * N + 335 * Nv,   # always: xyz+scale+rot+opacity 44, radii/tiles/observe 12; visible: SH 192, all_map 20, record 64, cov3D 24, depth/rect/clamp 13, ...
        "scan": 8 * N + 16 * N,   # tile-count scan + depth sort of the slots (>= one read + one write of 8-byte pairs)
        "binning": 12 * N + 16 * Nv + (8 + 16 + 4) * R + 8 * T,   # depth-order scan, emit 8R, tile sort >= 16R, ranges 4R
        "blend_fwd": 68 * R + 48 * HW + 8 * T,  # id 4 + record 64 per instance; 12 floats out per pixel
        "accum_zero": 64 * N,
        "blend_bwd": 68 * R + 72 * HW + 128 * Nv + 8 * T,  # gathers; 18 floats in per pixel; accumulator RMW
        "preprocess_bwd": 4 * N + (64 + 44 + 24 + 192 + 1 + 32) * Nv + 324 * N,  # rows read + all gradient rows written
    }


# ----------------------------------------------------------------------------- arms
def load_scene(dev):
    from hidegs_b200 import synthetic as syn
    sc = syn.make_scene(N_GAUSS, seed=0)
    return {k: v.to(dev) for k, v in sc.items()}, sc


def op_tuple(C, scene, cam, all_map, dev, bg):
    e_i = torch.empty(0, dtype=torch.int32, device=dev)
    e_f = torch.empty(0, dtype=torch.float32, device=dev)
    return (bg, e_i, e_i, e_f, e_i, scene["means3D"], e_f, all_map, scene["opacity"], scene["scales"],
            scene["rotations"], 1.0, e_f, cam.world_view_transform, cam.full_proj_transform, cam.tanfovx, cam.tanfovy,
            HEIGHT, WIDTH, scene["shs"], 3, cam.camera_center, False, True, False, True)


def bwd_tuple(fa, fwd, g):
    (bg, indices, parents, ts, kids, means3D, colors, all_map, opacity, scales, rotations, sm, cov3D, view, proj, tfx,
     tfy, H, W, sh, degree, campos, prefiltered, render_geo, debug, do_depth) = fa
    R, color, radii, observe, out_all_map, plane_depth, geom, binning, img, invdepth = fwd
    return (bg, out_all_map, indices, parents, ts, kids, means3D, radii, colors, all_map, opacity, scales, rotations, sm,
            cov3D, view, proj, tfx, tfy, g["color"], g["all_map"], g["plane_depth"], g["invdepth"], sh, degree, campos,
            geom, R, binning, img, render_geo, debug)


class RefAutograd(torch.autograd.Function):
    """Autograd glue around the reference's `_C` operators, as its own
    diff_gaussian_rasterization/__init__.py:42-155 wires them (that Python file is not
    shipped to the GPU box; only the compiled operators are)."""

    @staticmethod
    def forward(ctx, C, fa, means3D, sh, opacity, scales, rotations, all_map):
        out = C.rasterize_gaussians(*fa)
        ctx.C, ctx.fa, ctx.out = C, fa, out
        ctx.mark_non_differentiable(out[2], out[3])
        return out[1], out[2], out[3], out[4], out[5], out[9]

    @staticmethod
    def backward(ctx, g_color, _r, _o, g_all_map, g_plane, g_inv):
        g = dict(color=g_color.contiguous(), all_map=g_all_map.contiguous(), plane_depth=g_plane.contiguous(),
                 invdepth=g_inv.contiguous())
        (d2, dcol, dop, dm3, dcov, dsh, dsc, drot, dam) = ctx.C.rasterize_gaussians_backward(*bwd_tuple(ctx.fa, ctx.out, g))
        return None, None, dm3, dsh, dop, dsc, drot, dam


def run_gpu_arm(args, impl):
    import torch.distributed as dist
    from hidegs_b200 import _lib, synthetic as syn
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if impl == "reference" and rank != 0:
        return  # the reference is single-GPU: rank 0 alone runs it
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    ddp = world > 1 and impl == "ours"
    host_placement = None
    if ddp:
        # one process per GPU: keep each on the cores of its GPU's NUMA node (before NCCL and torch start their threads)
        if os.environ.get("HG_BENCH_PIN", "1") != "0":
            from hidegs_b200.parallel import pin_host_to_gpu_node
            host_placement = pin_host_to_gpu_node(dev)
        dist.init_process_group("nccl", device_id=dev)

    if impl == "ours":
        from hidegs_b200.diff_gaussian_rasterization import _C as C
    else:
        sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
        import ref_rasterizer_C as C

    scene, scene_cpu = load_scene(dev)
    bg = torch.zeros(3, device=dev)
    K, Wm = args.steps, args.warmup
    cams = [camera_for(rank, s) for s in range(K + Wm)]
    all_maps = [syn.geometry_all_map(scene["means3D"], scene["scales"], scene["rotations"], c.to(dev)) for c in cams[:1]]
    g = {k: v.to(dev) for k, v in syn.upstream_grads(WIDTH, HEIGHT, seed=1).items()}
    HW = WIDTH * HEIGHT
    from hidegs_b200 import parallel

    # With an NVSwitch multicast mapping the backward writes its gradients straight into symmetric memory and the
    # exchange is ONE in-fabric kernel (hg_nvls_allreduce_f32); otherwise NCCL sums the arena in place.
    # Default (HG_EXCHANGE_FACTORED=0 restores the whole-arena sum): the SH block does not travel.  dL/dSH of a view is
    # the outer product of the SH basis at the view direction with three clamp-masked colour gradients, so the backward
    # writes those three factors, the ranks all-gather them (12 B per Gaussian and rank) and all-reduce only the 11
    # non-SH floats, and every rank rebuilds the summed SH rows locally (parallel.FactoredExchange): (44 + 12 world) B
    # per Gaussian through the fabric instead of 236 B.
    exchange = factored = None
    if ddp and os.environ.get("HG_EXCHANGE_FACTORED", "1") == "1":
        factored = parallel.FactoredExchange(N_GAUSS, dev, 16, arena_numel=N_GAUSS * 80)
    elif ddp and parallel.prefer_nvls(dev):
        exchange = parallel.SymmetricArena(N_GAUSS * 80, dev)   # 80 floats / Gaussian: the whole backward arena

    # Opt-in (HG_EXCHANGE_OVERLAP=1): overlapped with the per-Gaussian backward — preprocess_bwd is issued in 2 slot
    # ranges and the first range's five parameter blocks travel (one in-fabric kernel on a side stream) while the second
    # range is computed.  Measured on 8 B200: 2.797 vs 2.844 ms per step in tools/overlap_probe.py (one camera per
    # rank), but 2.906 vs 2.844 ms in this bench's loop (a different camera every step: the ranks' skew makes the
    # extra cross-rank barriers cost more than the 0.08 ms they can hide), so the single call stays the default.
    overlap = None
    if exchange is not None and os.environ.get("HG_EXCHANGE_OVERLAP", "0") == "1":
        overlap = parallel.OverlappedBackwardExchange(exchange, N_GAUSS, 16,
                                                      n_chunks=int(os.environ.get("HG_EXCHANGE_CHUNKS", 2)))

    def pack_and_allreduce(grads):
        # (dL_dmeans2D, dL_dcolors, dL_dopacity, dL_dmeans3D, dL_dcov3D, dL_dsh, dL_dscales, dL_drotations, dL_dall_map)
        # xyz 3 | sh 48 | opacity 1 | scale 3 | rot 4 = 59 floats per Gaussian, contiguous in the backward's arena
        if exchange is not None and grads[3].data_ptr() == exchange.tensor.data_ptr():
            exchange.all_reduce_(59 * N_GAUSS)
        else:
            parallel.allreduce_gradients((grads[3], grads[5], grads[2], grads[6], grads[7]))

    def exchange_check():
        """Driver-visible correctness of the gradient exchange the timed steps use: every rank fills the 59-float arena
        with its own seeded pattern, the chosen exchange sums it in place, and the result is compared with
        torch.distributed.all_reduce (NCCL) of a copy; the replicas must be bit-identical across ranks."""
        n = 59 * N_GAUSS
        gen = torch.Generator(device=dev).manual_seed(4321 + rank)
        pattern = torch.randn(n, generator=gen, device=dev)
        want = pattern.clone()
        dist.all_reduce(want, op=dist.ReduceOp.SUM)
        if exchange is not None:
            got = exchange.tensor[:n]
            got.copy_(pattern)
            exchange.all_reduce_(n)
        else:
            got = pattern.clone()
            parallel.allreduce_gradients((got,))
        torch.cuda.synchronize()
        err = (got - want).abs().max().reshape(1)
        scale = want.abs().max().reshape(1)
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
        first = got.clone()
        dist.broadcast(first, src=0)
        same = torch.tensor([1.0 if torch.equal(first, got) else 0.0], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        return {"max_abs_err": float(err), "max_abs_value": float(scale), "replicas_identical": bool(same.item() == 1.0),
                "vs": "torch.distributed.all_reduce (NCCL) of the same seeded per-rank pattern, %d floats" % n,
                "kernel": "hg_nvls_allreduce_f32" if exchange is not None else "ncclAllReduce"}

    def factored_check():
        """The same check for the factored exchange, end to end on this rank's first view: plain backward + NCCL
        all_reduce of the 59-float arena against factor backward + FactoredExchange.finish."""
        n = 59 * N_GAUSS
        cams[0].to(dev)
        fa = op_tuple(C, scene, cams[0], all_maps[0], dev, bg)
        fwd = C.rasterize_gaussians(*fa)
        p = C.rasterize_gaussians_backward(*bwd_tuple(fa, fwd, g))
        want = torch.cat([p[3].reshape(-1), p[5].reshape(-1), p[2].reshape(-1), p[6].reshape(-1), p[7].reshape(-1)])
        dist.all_reduce(want, op=dist.ReduceOp.SUM)
        C.rasterize_gaussians_backward(*bwd_tuple(fa, fwd, g), **factored.backward_kwargs())
        got = factored.finish(scene["means3D"], 3)[:n]
        torch.cuda.synchronize()
        err = (got - want).abs().max().reshape(1)
        scale = want.abs().max().reshape(1)
        rel_l2 = ((got - want).double().norm() / want.double().norm()).float().reshape(1)
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
        dist.all_reduce(rel_l2, op=dist.ReduceOp.MAX)
        first = got.clone()
        dist.broadcast(first, src=0)
        same = torch.tensor([1.0 if torch.equal(first, got) else 0.0], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        # two runs of the backward differ by the order of their atomic adds (~1e-7 relative per element, more on the few
        # largest ones), so the gate is the relative L2 error of the whole arena plus a loose bound on the worst element
        return {"max_abs_err": float(err), "max_abs_value": float(scale), "rel_l2_err": float(rel_l2),
                "replicas_identical": bool(same.item() == 1.0), "tolerance": {"rel_l2_err": 1e-5, "max_abs_err_over_max": 1e-4},
                "vs": "plain backward + torch.distributed.all_reduce (NCCL) of the 59-float arena, %d floats, each rank "
                      "its own view" % n,
                "kernel": ("hg_nvls_exchange_f32" if factored.symmetric is not None else
                           "ncclAllReduce x2 + ncclAllGather") + " + hg_sh_gradient_from_factors"}

    xcheck = (factored_check() if factored is not None else exchange_check()) if ddp else None
    if xcheck is not None:
        ok = xcheck["replicas_identical"]
        if "rel_l2_err" in xcheck:
            ok = ok and xcheck["rel_l2_err"] <= 1e-5 and xcheck["max_abs_err"] <= 1e-4 * xcheck["max_abs_value"]
        else:
            ok = ok and xcheck["max_abs_err"] <= 1e-5 * xcheck["max_abs_value"]
        if not ok:
            raise SystemExit("gradient exchange check failed: %s" % json.dumps(xcheck))

    # ------------------------------------------------ device-resident leg ("value")
    def step_resident(s):
        cam = cams[s]
        fa = op_tuple(C, scene, cam, all_maps[0], dev, bg)
        fwd = C.rasterize_gaussians(*fa)
        if factored is not None:
            grads = C.rasterize_gaussians_backward(*bwd_tuple(fa, fwd, g), **factored.backward_kwargs())
            factored.finish(scene["means3D"], 3)
        elif overlap is not None:
            grads = C.rasterize_gaussians_backward(*bwd_tuple(fa, fwd, g), **overlap.backward_kwargs())
            overlap.finish()
        else:
            kw = dict(grad_arena=exchange.tensor) if exchange is not None else {}
            grads = C.rasterize_gaussians_backward(*bwd_tuple(fa, fwd, g), **kw)
            if ddp:
                pack_and_allreduce(grads)
        # only the last timed step's gradients outlive the call (for --dump-outputs)
        return fwd, (grads if s == Wm + K - 1 else None)

    for c in cams:
        c.to(dev)
    for s in range(Wm):
        fwd, grads = step_resident(s)
    torch.cuda.synchronize()
    if ddp:
        dist.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    if impl == "ours":
        _lib.lib().hg_reset_launch_count()
        _lib.profile_enable(True)
        _lib.profile_collect()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    torch.cuda.synchronize()
    e0.record()
    for s in range(Wm, Wm + K):
        fwd, grads = step_resident(s)
    e1.record()
    torch.cuda.synchronize()
    if ddp:
        dist.barrier()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop()
    launches, stages = None, None
    if impl == "ours":
        _lib.profile_enable(False)
        stages = _lib.profile_collect()
        launches = int(_lib.lib().hg_launch_count())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, fwd, grads)
    del grads
    R = int(fwd[0])
    Nv = int((fwd[2] > 0).sum())
    t_ms = torch.tensor([ms_total], device=dev)
    if ddp:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_step = float(t_ms) / K
    value = world * HW / (ms_step * 1e-3) / 1e6 if impl == "ours" else HW / (ms_step * 1e-3) / 1e6

    # ------------------------------------------------ end-to-end leg ("e2e"): public API + host inputs
    if impl == "ours":
        from hidegs_b200.diff_gaussian_rasterization import GaussianRasterizer
    params = {k: scene[k].clone().requires_grad_(True) for k in ("means3D", "shs", "opacity", "scales", "rotations")}
    if factored is not None:  # the autograd backward writes into the exchange's arena, the SH block as factors
        params["means3D"]._hg_grad_arena = factored.tensor
        params["shs"]._hg_grad_factor = factored.my_factors
    elif exchange is not None:  # the autograd backward of every e2e step writes its gradients into the symmetric arena
        params["means3D"]._hg_grad_arena = exchange.tensor
    gen = torch.Generator().manual_seed(7)
    gt_host = torch.rand(3, HEIGHT, WIDTH, generator=gen).pin_memory()
    cam_host = [torch.cat([c.world_view_transform.flatten().cpu(), c.full_proj_transform.flatten().cpu(),
                           c.camera_center.cpu()]).pin_memory() for c in cams]
    # the other outputs receive FIXED upstream gradients (d/dx of mean(x * 1e-3 g)) through torch.autograd.backward's
    # grad_tensors: every output of the rasterizer carries a gradient, without probe kernels in the timed region
    w_geo = (g["all_map"] * (1e-3 / g["all_map"].numel())).contiguous()
    w_pd = (g["plane_depth"] * (1e-3 / g["plane_depth"].numel())).contiguous()
    w_inv = (g["invdepth"] * (1e-3 / g["invdepth"].numel())).contiguous()
    if impl == "ours":
        from hidegs_b200.loss_utils import l1_loss as l1
    else:
        def l1(network_output, gt):  # utils/loss_utils.py:18-19 of the reference, verbatim
            return torch.abs((network_output - gt)).mean()
    h2d_bytes = gt_host.numel() * 4 + cam_host[0].numel() * 4
    am_param = all_maps[0].clone().requires_grad_(True)
    # The ground-truth image (24.9 MB) is uploaded on a copy stream while the forward renders; the loss waits for it.
    copy_stream = torch.cuda.Stream(device=dev)
    gt_dev = [torch.empty_like(gt_host, device=dev) for _ in range(2)]
    gt_free = [torch.cuda.Event() for _ in range(2)]
    for ev in gt_free:
        ev.record()

    # Loss read-back: non-blocking pinned copy for both arms (measured on both: faster than a blocking .item() per step,
    # 2.75 vs 2.86 ms ours, 16.5 vs 24.8 ms reference).  HG_BENCH_E2E_SYNC=1 forces the blocking read.
    blocking_readback = os.environ.get("HG_BENCH_E2E_SYNC") == "1"
    loss_host = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_read = [torch.cuda.Event() for _ in range(2)]
    for ev in loss_read:
        ev.record()

    def step_e2e(s):
        cam = cams[s]
        main = torch.cuda.current_stream()
        gt = gt_dev[s & 1]
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(gt_free[s & 1])  # the step that last read this buffer has finished
            gt.copy_(gt_host, non_blocking=True)
            gt_ready = torch.cuda.Event()
            gt_ready.record(copy_stream)
        cd = cam_host[s].to(dev, non_blocking=True)
        view, proj, campos = cd[:16].view(4, 4), cd[16:32].view(4, 4), cd[32:35]
        for p in params.values():
            p.grad = None
        if impl == "ours":
            rs = syn.raster_settings(cam, dev)._replace(viewmatrix=view, projmatrix=proj, campos=campos, bg=bg)
            means2D = torch.zeros_like(params["means3D"], requires_grad=True)
            color, radii, obs, amap, pdepth, inv = GaussianRasterizer(rs)(
                means3D=params["means3D"], means2D=means2D, opacities=params["opacity"], shs=params["shs"],
                scales=params["scales"], rotations=params["rotations"], all_map=am_param)
        else:
            e_i = torch.empty(0, dtype=torch.int32, device=dev)
            e_f = torch.empty(0, dtype=torch.float32, device=dev)
            fa = (bg, e_i, e_i, e_f, e_i, params["means3D"], e_f, am_param, params["opacity"], params["scales"],
                  params["rotations"], 1.0, e_f, view, proj, cam.tanfovx, cam.tanfovy, HEIGHT, WIDTH, params["shs"], 3,
                  campos, False, True, False, True)
            color, radii, obs, amap, pdepth, inv = RefAutograd.apply(C, fa, params["means3D"], params["shs"],
                                                                     params["opacity"], params["scales"],
                                                                     params["rotations"], am_param)
        main.wait_event(gt_ready)
        # L1 through each side's own loss function (the reference's utils/loss_utils.l1_loss is torch.abs(a - b).mean();
        # ours is the fused drop-in of the same name); the geometry / depth outputs get their fixed upstream gradients
        loss = l1(color, gt)
        torch.autograd.backward([loss, amap, pdepth, inv], [None, w_geo.view_as(amap), w_pd.view_as(pdepth),
                                                            w_inv.view_as(inv)])
        gt_free[s & 1].record(main)
        if factored is not None:
            factored.finish(params["means3D"].detach(), 3)
        elif ddp:
            pack_and_allreduce((None, None, params["opacity"].grad, params["means3D"].grad, None, params["shs"].grad,
                                params["scales"].grad, params["rotations"].grad))
        # D2H read of the step's result: copied into pinned memory every step; the host consumes it one step later
        # (as a training loop's logging does), so the copy never drains the launch queue.  Both arms share this harness.
        if blocking_readback:
            return float(loss.item())
        slot = s & 1
        prev = float(loss_host[1 - slot].item()) if loss_read[1 - slot].query() else None
        loss_host[slot].copy_(loss.detach(), non_blocking=True)
        loss_read[slot].record(main)
        return prev

    # Untimed warm-up: at least W steps, and enough of them for torch's caching allocator to have
    # seen the step's peak working set (its first steps call cudaMalloc, 10-30 ms each).
    # Every camera of the run is visited once here: the binning part of the workspace is sized from the largest
    # num_rendered seen so far, so a first-time view can still trigger one cudaMalloc.
    for s in range(max(Wm + K, 8)):
        step_e2e(s % (Wm + K))
    torch.cuda.synchronize()
    if ddp:
        dist.barrier()
    # Five timed passes of K steps; the MEDIAN pass is reported and min / max are printed beside it (the reference's
    # per-call tensor resizes make single passes of ITS arm vary with allocator state; ours varies by < 1 %).
    passes = []
    for _pass in range(5):
        e0.record()
        for s in range(Wm, Wm + K):
            step_e2e(s)
        e1.record()
        torch.cuda.synchronize()  # every step's loss has reached the host
        if not blocking_readback:
            last_loss = float(loss_host[(Wm + K - 1) & 1].item())
            assert last_loss == last_loss, "e2e loss is NaN"
        if ddp:
            dist.barrier()
        passes.append(e0.elapsed_time(e1))
    best = float(np.median(passes))
    t2 = torch.tensor([best], device=dev)
    if ddp:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    ms_e2e = float(t2) / K
    e2e_value = (world if impl == "ours" else 1) * HW / (ms_e2e * 1e-3) / 1e6

    train = train_c3 = losses = None
    if impl == "ours" and not os.environ.get("HG_BENCH_SKIP_TRAIN"):
        # free the rasterizer legs' buffers before the 2M-Gaussian training legs
        del params, am_param, scene, all_maps
        torch.cuda.empty_cache()
        n_train = int(os.environ.get("HG_BENCH_TRAIN_N", 2_000_000))
        train = train_leg(dev, rank, world, ddp, steps=K, warmup=3, views_per_rank=8, n_gauss=n_train,
                          recipe="uav")
        torch.cuda.empty_cache()
        # the same step with every ground-truth-only quantity recomputed at every visit (SURVEY.md §8(d): both)
        unc_uav = train_leg(dev, rank, world, ddp, steps=K, warmup=3, views_per_rank=8, n_gauss=n_train,
                            recipe="uav", cache_gt=False)
        train["views_per_s_uncached_ground_truth"] = unc_uav["views_per_s"]
        train["ms_per_step_uncached_ground_truth"] = unc_uav["ms_per_step"]
        if world == 1:
            torch.cuda.empty_cache()
            train_c3 = train_leg(dev, rank, world, False, steps=K, warmup=3, views_per_rank=1,
                                 n_gauss=n_train, recipe="c2")
            torch.cuda.empty_cache()
            # the same step with every ground-truth-only quantity recomputed at every visit (no per-camera cache)
            unc = train_leg(dev, rank, world, False, steps=K, warmup=3, views_per_rank=1,
                            n_gauss=n_train, recipe="c2", cache_gt=False)
            train_c3["views_per_s_uncached_ground_truth"] = unc["views_per_s"]
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import loss_bench
            losses = loss_bench.measure(dev, iters=K, warmup=3, cpu=not os.environ.get("HG_BENCH_SKIP_CPU"))

    if rank != 0:
        if ddp:
            dist.destroy_process_group()
        return

    line = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world if impl == "ours" else 1,
        "steps": K, "warmup": Wm, "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: 1M Gaussians, SH degree 3, one 1920x1080 view fwd+bwd per GPU per step"
                               if (N_GAUSS, WIDTH, HEIGHT) == (1_000_000, 1920, 1080) else
                               "REDUCED %d Gaussians %dx%d" % (N_GAUSS, WIDTH, HEIGHT),
                   "gaussians": N_GAUSS, "width": WIDTH, "height": HEIGHT, "visible": Nv, "num_rendered": R,
                   "outputs": "color+all_map+plane_depth+invdepth", "parallelism": "view-sharded dp%d" % world,
                   "host_placement_rank0": host_placement,
                   "exchange": (None if not ddp else
                                ("factored: %s; %d B per Gaussian through the fabric instead of 236"
                                 % ("ONE in-fabric kernel (hg_nvls_exchange_f32: 11 non-SH floats summed with "
                                    "multimem.ld_reduce, 3 colour-gradient factors per rank gathered with multimem.st)"
                                    if factored.symmetric is not None else
                                    "nccl all_reduce of the 11 non-SH floats + all_gather of 3 colour-gradient factors "
                                    "per rank", 44 + 12 * world)
                                 + ", SH rows rebuilt locally (hg_sh_gradient_from_factors)") if factored is not None else
                                ("nvls multimem kernel, 236 MB arena, overlapped with preprocess_bwd in %d slot ranges"
                                 % overlap.n_chunks) if overlap is not None else
                                "nvls multimem kernel (hg_nvls_allreduce_f32), 236 MB arena" if exchange is not None
                                else "nccl all_reduce, 236 MB arena"),
                   "l2": "inputs_exceed_l2 (SH 192 MB + records 64 MB + sort buffers > 126 MB)"},
        "clocks": clocks,
        "e2e": {"value": round(e2e_value, 2), "unit": UNIT, "ms_per_step": round(ms_e2e, 4),
                "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                "d2h": ("loss read with a blocking .item() every step" if blocking_readback else
                        "loss copied to pinned host memory every step (non-blocking), consumed one step later"),
                "api": "GaussianRasterizer(settings)(...) + l1_loss (each side's own utils.loss_utils.l1_loss) + torch.autograd.backward (fixed upstream gradients for all_map / plane_depth / invdepth); ground-truth upload on a copy "
                       "stream, overlapped with the forward",
                "timed_passes": "5 x K steps, median pass reported",
                "ms_per_step_min_median_max": [round(min(passes) / K, 4), round(float(np.median(passes)) / K, 4),
                                               round(max(passes) / K, 4)]},
    }
    if impl == "ours":
        bytes_per = stage_bytes(N_GAUSS, Nv, R, HW, ((WIDTH + 15) // 16) * ((HEIGHT + 15) // 16))
        peak, how = measured_peaks()
        per_stage = {k: round(v[0] / max(v[1], 1), 4) for k, v in stages.items()}
        dom = max(stages, key=lambda k: stages[k][0])
        dom_ms = stages[dom][0] / max(stages[dom][1], 1)
        achieved = bytes_per[dom] / (dom_ms * 1e-3) / 1e9
        traffic = issue_pct = None
        tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp))
            traffic = tj.get(dom)
            issue_pct = tj.get("_issue_active_pct", {}).get(dom)
        hbm = {"achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
               "algorithmic_bytes": bytes_per[dom], "peak_source": how}
        sm_ghz = (clocks.get("sm_mhz") or 1965.0) / 1e3
        issue_peak = 148 * 4 * sm_ghz  # G warp-instructions / s: 148 SMs x 4 schedulers x 1 issue / clock
        warp_inst = packed = None
        if os.path.exists(tp):
            warp_inst = json.load(open(tp)).get("_warp_instructions", {}).get(dom)
            packed = json.load(open(tp)).get("_packed_fp32_instructions", {}).get(dom)
        if dom.startswith("blend") and warp_inst:
            # the blend kernels gather L2-resident records and are bound by instruction issue (DESIGN.md §4): the
            # fraction is quoted against THAT roof, the HBM figure is kept beside it
            ach = warp_inst / (dom_ms * 1e-3) / 1e9
            line["roofline"] = {"kernel": dom, "bound": "issue", "achieved": round(ach, 1), "peak": round(issue_peak, 1),
                                "unit": "Gwarp-inst/s", "frac": round(ach / issue_peak, 4), "traffic": traffic,
                                "warp_instructions_per_launch_ncu": warp_inst,
                                "peak_source": "148 SM x 4 schedulers x median SM clock under load (%.0f MHz)" % (sm_ghz * 1e3),
                                "issue_active_pct_ncu": issue_pct, "frac_hbm": hbm["frac"], "hbm": hbm}
            if packed:
                # FADD2 / FMUL2 / FFMA2 retire two FP32 operations per issue slot at the same 128 FMA / clk / SM: `frac`
                # counts them once (= how busy the issue port is), this figure counts them twice (= the scalar-
                # equivalent instruction rate, the unit SURVEY.md 8(d) quotes the blend loops in)
                line["roofline"]["packed_fp32_instructions_per_launch_ncu"] = packed
                line["roofline"]["frac_scalar_equivalent"] = round((warp_inst + packed) / (dom_ms * 1e-3) / 1e9 / issue_peak, 4)
        else:
            line["roofline"] = dict(kernel=dom, bound="hbm", traffic=traffic, **hbm)
        line["roofline"].update({"kernel_ms": round(dom_ms, 4), "stage_ms": per_stage,
                                 "share_of_step": round(stages[dom][0] / max(sum(v[0] for v in stages.values()), 1e-9), 3)})
        # every HBM-bound stage against the measured copy bandwidth
        line["roofline"]["stages_hbm_frac"] = {
            k: round(bytes_per[k] / (max(per_stage[k], 1e-9) * 1e-3) / 1e9 / peak, 4)
            for k in ("preprocess_fwd", "scan", "binning", "preprocess_bwd") if k in per_stage}
        line["gpu_launches"] = launches
        if train is not None:
            line["train"] = train
        if train_c3 is not None:
            line["train_config3"] = train_c3
        if losses is not None:
            line["losses_config0"] = losses
            line["roofline_losses"] = {"bound": "hbm", "achieved": losses["achieved_gbs"], "peak": peak, "unit": "GB/s",
                                       "frac": round(losses["achieved_gbs"] / peak, 4),
                                       "algorithmic_bytes": losses["algorithmic_bytes"], "ms": losses["gpu_ms"],
                                       "launches": losses.get("gpu_launches"),
                                       "note": "SURVEY.md §8(d): 115 B per level-0 pixel for L1 + SSIM + frequency "
                                               "regulariser fwd+bwd (3 levels), ground truth recomputed every call"}
        if xcheck is not None:
            line["exchange_check"] = xcheck
        if not os.environ.get("HG_BENCH_SKIP_CPU"):
            line["cpu_baseline"] = cpu_baseline(scene_cpu)
    else:
        line["impl"] = "reference"
        line["cpu_baseline"] = {"value": line["value"], "unit": UNIT, "cores": 0, "kind": "reference",
                                "sample": "unmodified reference CUDA rasterizer rebuilt for sm_100 (oracle/_ref), full "
                                          "workload on the same B200; the reference has no CPU implementation of this path"}
    print(json.dumps(line), flush=True)
    if ddp:
        dist.destroy_process_group()


def make_gt_images(n, dev, seed=11):
    """Synthetic ground-truth images (config-1 recipe: blurred uniform noise), generated on the device, kept on the
    HOST in pinned memory: the training loop copies one per view, like a data loader would."""
    import torch.nn.functional as F
    g = torch.Generator(device=dev).manual_seed(seed)
    out = []
    for _ in range(n):
        x = torch.rand(1, 3, HEIGHT, WIDTH, generator=g, device=dev)
        out.append(F.avg_pool2d(x, 5, stride=1, padding=2)[0].clamp(0, 1).cpu().pin_memory())
    return out


def train_leg(dev, rank, world, ddp, steps, warmup, views_per_rank, n_gauss, recipe, cache_gt=True):
    """Training views/s (BASELINE.json metric 2): full HiDeGS step = render (prologue + rasterizer + epilogue) + L1 +
    SSIM + frequency regularisation + scale regularisation + single-view normal term, backward, gradient all-reduce
    over the ranks, fused Adam.  `recipe`: "uav" = configs[4] (8x8 survey cameras over the 400 m x 224 m slab, views
    sharded views[rank::world]) or "c2" = configs[3] (config-2 scene / camera)."""
    import torch.distributed as dist
    from hidegs_b200 import synthetic as syn, trainer as tr, _lib
    if recipe == "uav":
        scene = syn.make_uav_scene(n_gauss, seed=0)
        # Latin-square order: views[rank::world] hands every rank one camera of every row AND every column of the
        # survey grid, so the ranks' loads match (edge cameras see less of the slab than central ones)
        cams_all = [syn.uav_camera(i, (j + i) % 8, width=WIDTH, height=HEIGHT).to(dev) for i in range(8) for j in range(8)]
    else:
        scene = syn.make_scene(n_gauss, seed=0)
        cams_all = [camera_for(r, s).to(dev) for r in range(8) for s in range(8)]
    total_views = views_per_rank * world
    my_views = list(range(total_views))[rank::world]
    cams = [cams_all[i] for i in my_views]
    gts = make_gt_images(views_per_rank, dev, seed=11 + rank)
    # the model stores its Gaussians along a Morton curve (a one-off permutation at load time; results are invariant)
    spatial = os.environ.get("HG_BENCH_SPATIAL_ORDER", "1") != "0"
    params = tr.GaussianParams.from_scene(scene, dev, spatial_order=spatial)
    # the run resumes at the end of the regulariser's warm-up (frequency_regularization.py:1594: the frequency / scale
    # terms are zero before iteration 1000), so that every timed step carries the full loss
    trainer = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), cache_ground_truth=cache_gt,
                                    start_iteration=tr.OptimizationParams.freq_warmup_iterations)

    # Ground-truth images travel host -> device on a copy stream, one event per view (the losses of a view wait for
    # its image only), double buffered across steps: the uploads of step k+1 are issued at the start of step k.
    copy_stream = torch.cuda.Stream(device=dev)
    gt_dev = [[torch.empty_like(g, device=dev) for g in gts] for _ in range(2)]
    step_done = [torch.cuda.Event() for _ in range(2)]
    for ev in step_done:
        ev.record()
    counter = [0]

    uploaded = [None, None]  # per buffer: the "image has arrived" events of the step whose images it holds

    def upload(par):
        """This rank's ground-truth images of ONE step -> buffer `par`, on the copy stream."""
        evs = []
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(step_done[par])  # the step that last read this buffer has finished
            for g, d in zip(gts, gt_dev[par]):
                d.copy_(g, non_blocking=True)
                ready = torch.cuda.Event()
                ready.record(copy_stream)
                evs.append(ready)
        uploaded[par] = evs

    def step():
        par = counter[0] & 1
        counter[0] += 1
        if uploaded[par] is None:  # first call only
            upload(par)
        views = list(zip(cams, gt_dev[par], uploaded[par]))
        uploaded[par] = None
        # The loader runs ONE STEP AHEAD: the images of the next step travel while this one computes (one upload set per
        # step, inside the timed region, as before).  Issued at the start of their own step they arrive just in time at
        # 25 GB/s, and late on ranks whose host link delivers less: on an 8-GPU box four ranks sat at 8 x 24.9 MB /
        # 13.2 ms = 15 GB/s, whatever views they were dealt.
        upload(par ^ 1)
        loss = trainer.step(views, total_views=total_views)
        step_done[par].record(torch.cuda.current_stream())
        return loss

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    balance = None
    if ddp and os.environ.get("HG_BENCH_BALANCE", "1") != "0":
        # Re-shard the step's views by measured device time: the ranks meet at the gradient exchange, so the step runs at
        # the pace of the slowest rank.  A view's time is (cost of the view) x (pace of the GPU it ran on) — the GPUs of
        # one box do not run at exactly the same pace (measured: +-6 % between the halves of an 8-GPU box) — so every
        # view is timed on TWO ranks (its own shard, then the next rank's shard) and the two factors are separated by
        # alternating least squares before the assignment.  (num_rendered alone left 13.2 - 14.4 ms across 8 ranks.)
        def timed_shard(view_ids):
            cams[:] = [cams_all[i] for i in view_ids]
            trainer._gt_cache.clear()
            step()                     # (builds the per-camera ground-truth caches)
            trainer.time_views = True
            step()
            trainer.time_views = False
            return [(i, rank, t_) for i, t_ in zip(view_ids, trainer.last_view_ms())]
        every = list(range(total_views))
        mine = timed_shard(my_views) + timed_shard(every[(rank + 1) % world::world])
        table = [None] * world
        dist.all_gather_object(table, mine)
        meas = [m for part in table for m in part]
        cost, speeds = [1.0] * total_views, [1.0] * world
        for _ in range(20):            # t = cost[i] * pace[r]
            for i in range(total_views):
                v = [t_ / speeds[r_] for j, r_, t_ in meas if j == i]
                cost[i] = sum(v) / len(v)
            for r_ in range(world):
                v = [t_ / cost[j] for j, q, t_ in meas if q == r_]
                speeds[r_] = sum(v) / len(v)
            norm = sum(speeds) / world
            speeds = [x / norm for x in speeds]
        before = [speeds[r] * sum(cost[i] for i in every[r::world]) for r in range(world)]
        shards = tr.balance_views(cost, world, speeds)
        after = [speeds[r] * sum(cost[i] for i in sh) for r, sh in enumerate(shards)]
        balance = {"view_ms_per_rank_before": [round(x, 3) for x in before],
                   "view_ms_per_rank_after_predicted": [round(x, 3) for x in after],
                   "rank_pace": [round(x, 3) for x in speeds]}
        my_views = shards[rank]
        cams[:] = [cams_all[i] for i in my_views]
        trainer._gt_cache.clear()
        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        # Feedback on what the ranks then actually take for their views (the whole phase, CUDA events of two steps): the
        # sum of separately timed views misses what a rank's host side adds between them, so every rank's pace is
        # corrected by measured / predicted and the views are dealt again, at most three times.
        rounds = []
        for _ in range(int(os.environ.get("HG_BENCH_BALANCE_FEEDBACK", "3"))):
            trainer.timing = []
            step()
            step()
            torch.cuda.synchronize()
            mine_ms = sum(e[0].elapsed_time(e[1]) for e in trainer.timing) / len(trainer.timing)
            trainer.timing = None
            got = [None] * world
            dist.all_gather_object(got, mine_ms)
            rounds.append([round(x, 3) for x in got])
            pred = [speeds[r] * sum(cost[i] for i in sh) for r, sh in enumerate(shards)]
            speeds = [speeds[r] * got[r] / pred[r] for r in range(world)]
            norm = sum(speeds) / world
            speeds = [x / norm for x in speeds]
            new_shards = tr.balance_views(cost, world, speeds)
            if new_shards == shards:
                break
            shards = new_shards
            my_views = shards[rank]
            cams[:] = [cams_all[i] for i in my_views]
            trainer._gt_cache.clear()
            step()  # (rebuilds the per-camera ground-truth caches)
            torch.cuda.synchronize()
        balance["views_ms_per_rank_measured_per_feedback_round"] = rounds
        balance["rank_pace_final"] = [round(x, 3) for x in speeds]
    if ddp:
        dist.barrier()
    _lib.lib().hg_reset_launch_count()
    trainer.timing = []
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    if ddp:
        dist.barrier()
    last = float(loss.item())
    # where the step goes on this rank: its views (render + losses + backward), then exchange + union + Adam
    t_views = sum(e[0].elapsed_time(e[1]) for e in trainer.timing) / steps
    t_tail = sum(e[1].elapsed_time(e[2]) for e in trainer.timing) / steps
    trainer.timing = None
    t = torch.tensor([e0.elapsed_time(e1), t_views, -t_views, t_tail, -t_tail], device=dev)
    if ddp:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t[0]) / steps
    phases = {"views_ms_max_over_ranks": round(float(t[1]), 3), "views_ms_min_over_ranks": round(-float(t[2]), 3),
              "exchange_union_adam_ms_max": round(float(t[3]), 3), "exchange_union_adam_ms_min": round(-float(t[4]), 3),
              "note": "per rank, CUDA events: start -> last view's backward queued work done -> Adam done; the tail of a "
                      "rank that finishes its views early includes its wait for the slowest rank at the exchange"}
    if balance is not None:
        phases["balance"] = balance
    return {"views_per_s": round(total_views / (ms_step * 1e-3), 2), "ms_per_step": round(ms_step, 3),
            "ms_per_view": round(ms_step / views_per_rank, 3), "views_per_rank_per_step": views_per_rank,
            "views_per_step": total_views, "gaussians": n_gauss, "steps": steps, "warmup": warmup,
            "loss_last_step_rank0": round(last, 6), "gpu_launches": int(_lib.lib().hg_launch_count()),
            "ground_truth_cache": bool(cache_gt), "gaussian_layout": "morton order" if spatial else "as generated",
            "allreduce_bytes_per_step": params.grad_arena.numel() * 4 if world > 1 else 0, "phases": phases,
            "h2d_bytes_per_step": views_per_rank * 3 * HEIGHT * WIDTH * 4,
            "workload": ("configs[4]: view-sharded training, %d UAV survey cameras per step over the 2M-Gaussian slab, %dx%d, "
                         "views sharded over the ranks (views[rank::world], then re-sharded by the measured device time per view), one fp32 gradient "
                         "all-reduce + fused Adam per step" % (total_views, WIDTH, HEIGHT))
            if recipe == "uav" else
            ("configs[3]: full HiDeGS training step (L1 + SSIM + frequency + scale reg + single-view normal term) on the "
             "config-2 scene with %d Gaussians, %d view(s) per step" % (n_gauss, total_views))}


def cpu_baseline(scene_cpu, iters=3, tile_step=1):
    """CPU restatement (oracle port) on the host cores, same workload."""
    from hidegs_b200 import synthetic as syn
    from oracle.raster_oracle import OracleRasterizer
    cores = os.cpu_count() or 1
    cam = syn.default_camera(WIDTH, HEIGHT)
    am = syn.geometry_all_map(scene_cpu["means3D"], scene_cpu["scales"], scene_cpu["rotations"], cam)
    o = OracleRasterizer(bg=np.zeros(3, np.float32), viewmatrix=cam.world_view_transform.numpy(),
                         projmatrix=cam.full_proj_transform.numpy(), campos=cam.camera_center.numpy(),
                         means3D=scene_cpu["means3D"].numpy(), opacities=scene_cpu["opacity"].numpy(),
                         image_height=HEIGHT, image_width=WIDTH, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy,
                         shs=scene_cpu["shs"].numpy(), all_map=am.numpy(), scales=scene_cpu["scales"].numpy(),
                         rotations=scene_cpu["rotations"].numpy(), sh_degree=3, nthreads=cores)
    g = syn.upstream_grads(WIDTH, HEIGHT, seed=1)
    gn = {k: v.numpy() for k, v in g.items()}
    ts = []
    for _ in range(iters):
        t0 = time.perf_counter()
        o.forward(tile_step=tile_step)
        o.backward(gn["color"], gn["all_map"], gn["plane_depth"], gn["invdepth"], tile_step=tile_step)
        ts.append(time.perf_counter() - t0)
    t = float(np.median(ts))
    frac = 1.0 / tile_step
    return {"value": round(WIDTH * HEIGHT * frac / t / 1e6, 4), "unit": UNIT, "cores": cores, "kind": "port",
            "seconds": round(t, 2),
            "sample": "oracle/raster_oracle.c (C restatement of the reference algorithm), %d pthreads, full scene, "
                      "%s fwd+bwd, median of %d iteration(s)" % (cores, "every %d-th tile of the view" % tile_step if tile_step > 1 else "whole 1080p view", iters)}


def run_cpu_reference(args):
    """--impl reference without the reference CUDA build: time the CPU restatement."""
    from hidegs_b200 import synthetic as syn
    sc = syn.make_scene(N_GAUSS, seed=0)
    cb = cpu_baseline(sc, iters=max(1, min(args.steps, 3)))
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(cb["seconds"] * 1e3, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[1]: 1M Gaussians, SH degree 3, one 1920x1080 view fwd+bwd"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", 0))
    if args.impl == "reference":
        have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "ref_rasterizer_C.so"))
        if rank != 0:
            return
        if have_ref and torch.cuda.is_available():
            run_gpu_arm(args, "reference")
        elif args.dump_outputs:
            raise SystemExit("--dump-outputs needs the GPU arm: the CPU restatement is timed here, not the device path")
        else:
            run_cpu_reference(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the rasterizer has no CPU fallback")
    run_gpu_arm(args, "ours")


if __name__ == "__main__":
    main()
