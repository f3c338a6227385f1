#!/usr/bin/env python
"""Diagnostic: per-term, per-parameter-group agreement of ViewShardedTrainer.view_step_direct with the oracle
composition of tests/test_trainer_gpu.py (reference rasterizer + oracle losses).  GPU box only."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402
import test_step_oracle_gpu as S  # noqa: E402
from hidegs_b200 import trainer as tr  # noqa: E402


def main():
    dev = torch.device("cuda", 0)
    sc = S._scene()
    [(cam, gt)] = S._views(dev, S.TWO_EYES[:1])
    bg = torch.zeros(3, device=dev)
    variants = {"l1+ssim": dict(lambda_freq=0.0, lambda_scale=0.0, single_view_weight=0.0),
                "+freq": dict(lambda_scale=0.0, single_view_weight=0.0),
                "+scale": dict(single_view_weight=0.0),
                "normal only": dict(lambda_freq=0.0, lambda_scale=0.0, lambda_dssim=0.0),
                "all": {}}
    for (backend, raster), (name, kw) in ((b, v) for b in S._backends() for v in variants.items()):
        opt = type("Opt", (tr.OptimizationParams,), kw)
        params = tr.GaussianParams.from_scene(sc, dev)
        raw = {k: v.detach().clone() for k, v in params.leaves.items()}
        trainer = tr.ViewShardedTrainer(params, bg, opt=opt)
        params.zero_grad()
        loss, pkg = trainer.view_step_direct(cam, gt, 2000)

        def compose():
            leaves = {k: v.clone().requires_grad_(True) for k, v in raw.items()}
            return S._oracle_view(leaves, cam, gt, bg, dev, 2000, opt, raster)[0], leaves
        want, leaves = compose()
        line = ["%-10s %-12s loss %.6g vs %.6g" % (backend, name, float(loss), want)]
        for n, _w in tr.GROUPS:
            a = params.grad_arena[params.slices[n]].view(leaves[n].shape).double().cpu()
            b = leaves[n].grad.double().cpu()
            l2 = float((a - b).norm()) / max(float(b.norm()), 1e-30)
            line.append("%s %.2e (|b| %.2e)" % (n, l2, float(b.norm())))
        print("  ".join(line), flush=True)
        # two evaluations of the composition against each other: the noise floor of the comparison
        if name == "all":
            want2, leaves2 = compose()
            print("  %s vs itself: " % backend + "  ".join(
                "%s %.2e" % (n, float((leaves[n].grad - leaves2[n].grad).double().norm()) / float(leaves2[n].grad.double().norm()))
                for n, _w in tr.GROUPS), flush=True)


if __name__ == "__main__":
    main()
