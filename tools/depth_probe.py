"""Monocular inverse-depth supervision in the training step (ViewShardedTrainer(depth_regularization=True), DESIGN.md
§3 / §4).

    python tools/depth_probe.py --time [--steps 10 --rounds 3 --views 4]
        one GPU, in one run, with the card's name and power limit:
        1. CUDA-event time per call of hg_invdepth_l1 at 1920x1080 and 3840x2160, with and without a mask, over many
           launches with the inputs rotated over enough buffer sets (>= 512 MB) that they come from HBM, not the
           126 MB L2; algorithmic bytes (16 HW with a mask, 12 HW without) over kernel time against the 6544 GB/s of
           BASELINE.md §2 (measured HBM bandwidth of a B200) and the 7700 GB/s of the data sheet;
        2. the training step at the configs[3] recipe (config-2 scene: 2M Gaussians, 1920x1080, `--views` views per
           step, ground-truth cache) with the term on and off, alternated; per view.  With the term on, every view has
           a reliable prior with a fractional mask, so every view runs the kernel and the DEPTH variant of the blend
           backward.
        One JSON line.
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from hidegs_b200 import trainer as tr  # noqa: E402

HBM_MEASURED_GBPS = 6544   # BASELINE.md §2
HBM_DATASHEET_GBPS = 7700  # NVIDIA HGX B200 data sheet, per GPU


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        power = q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def kernel_times(dev, H, W, masked, reps=400):
    """CUDA-event time per call of hg_invdepth_l1 (mean over `reps` calls after a warm pass)."""
    from hidegs_b200 import loss_utils as lu
    L = lu._L()
    st = torch.cuda.current_stream().cuda_stream
    hw = H * W
    nbytes = (16 if masked else 12) * hw
    sets = max(2, math.ceil(512e6 / nbytes))
    g = torch.Generator(device=dev).manual_seed(0)
    bufs = []
    for _ in range(sets):
        inv = torch.rand(1, H, W, generator=g, device=dev)
        mono = inv + 0.05 * torch.randn(1, H, W, generator=g, device=dev)
        mask = torch.rand(1, H, W, generator=g, device=dev) if masked else None
        bufs.append((inv, mono, mask, torch.empty_like(inv)))
    value = torch.empty((), device=dev)
    loss = torch.zeros((), device=dev)
    ws = torch.zeros(int(L.hg_invdepth_l1_workspace_bytes(H, W)), dtype=torch.uint8, device=dev)

    def call(b):
        rc = L.hg_invdepth_l1(b[0].data_ptr(), b[1].data_ptr(), b[2].data_ptr() if b[2] is not None else None, H, W,
                              0.5, b[3].data_ptr(), value.data_ptr(), loss.data_ptr(), ws.data_ptr(), st)
        assert rc == 0
    for b in bufs:
        call(b)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        call(bufs[i % sets])
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / reps
    gbps = nbytes / (us * 1e-6) / 1e9
    return {"us": round(us, 2), "bytes": nbytes, "GBps": round(gbps, 1), "buffer_sets": sets,
            "share_of_measured_6544": round(gbps / HBM_MEASURED_GBPS, 3),
            "share_of_datasheet_7700": round(gbps / HBM_DATASHEET_GBPS, 3)}


def step_times(dev, steps, rounds, nviews):
    import bench
    from hidegs_b200 import gaussian_renderer as gr, synthetic as syn
    from hidegs_b200.ply_io import attach_depth_prior
    W, H = bench.WIDTH, bench.HEIGHT
    scene = syn.make_scene(2_000_000, seed=0)
    cams = [bench.camera_for(0, s).to(dev) for s in range(nviews)]
    g = torch.Generator(device=dev).manual_seed(11)
    gts = [torch.nn.functional.avg_pool2d(torch.rand(1, 3, H, W, generator=g, device=dev), 5, stride=1, padding=2)[0]
           .clamp(0, 1) for _ in cams]
    # priors: the scene's own inverse depth, off by a few per cent (residual of mixed sign), fractional masks
    probe = tr.GaussianParams.from_scene(scene, dev, spatial_order=True)
    with torch.no_grad():
        for c in cams:
            inv = gr.render(c, probe, tr.PipelineParams, torch.zeros(3, device=dev))["depth"].detach()
            noise = 1.0 + 0.05 * torch.randn(inv.shape, generator=g, device=dev)
            attach_depth_prior(c, inv * noise, mask=torch.rand(inv.shape, generator=g, device=dev))
    del probe
    trainers = {}
    for on in (False, True):
        params = tr.GaussianParams.from_scene(scene, dev, spatial_order=True)
        trainers[on] = tr.ViewShardedTrainer(params, torch.zeros(3, device=dev), cache_ground_truth=True,
                                             start_iteration=tr.OptimizationParams.freq_warmup_iterations,
                                             depth_regularization=on)
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
            ms[on].append(e0.elapsed_time(e1) / steps / nviews)
    off_ms, on_ms = sorted(ms[False])[len(ms[False]) // 2], sorted(ms[True])[len(ms[True]) // 2]
    return {"workload": "configs[3] recipe: config-2 scene, 2M Gaussians, %dx%d, %d views per step, ground-truth cache on"
                        % (W, H, nviews), "steps_per_round": steps, "rounds": rounds,
            "ms_per_view_off": [round(x, 3) for x in ms[False]], "ms_per_view_on": [round(x, 3) for x in ms[True]],
            "median_off": round(off_ms, 3), "median_on": round(on_ms, 3), "delta_ms_per_view": round(on_ms - off_ms, 3),
            "on_over_off": round(on_ms / off_ms, 4)}


def timing(steps, rounds, nviews):
    if not torch.cuda.is_available():
        raise SystemExit("depth_probe.py --time needs a CUDA device")
    dev = torch.device("cuda", 0)
    name, power = card()
    kernels = {}
    for H, W in ((1080, 1920), (2160, 3840)):
        for masked in (True, False):
            kernels["%dx%d_%s" % (W, H, "mask" if masked else "no_mask")] = kernel_times(dev, H, W, masked)
    torch.cuda.empty_cache()
    res = {"card": name, "power_limit": power, "kernel_hg_invdepth_l1": kernels,
           "step": step_times(dev, steps, rounds, nviews)}
    print(json.dumps(res))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--time", action="store_true")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--views", type=int, default=4)
    a = ap.parse_args()
    if not a.time:
        ap.error("nothing to do: pass --time")
    timing(a.steps, a.rounds, a.views)
