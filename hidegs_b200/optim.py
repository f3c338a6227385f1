"""Fused Adam for the Gaussian parameter groups: the update of the reference's scene/OurAdam.py (`Adam.step(relevant)`,
:106-337 — torch.optim.Adam arithmetic, optionally restricted to the rows `relevant` selects) as ONE kernel per
parameter tensor through hg_adam_step (include/hidegs_geometry.h), without the gather / scatter copies and the
`.item()` host sync of `_single_tensor_adam`.

    opt = Adam([{"params": [xyz], "lr": 1.6e-4, "name": "xyz"}, ...], lr=0.0, eps=1e-15)
    opt.step(relevant)      # relevant: empty tensor (all rows), int64 index tensor, or bool mask over the rows
"""
import numpy as np
import torch

from . import _lib
from ._geometry_lib import lib as _G


class Adam(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0, amsgrad=False):
        if weight_decay != 0 or amsgrad:
            raise NotImplementedError("hidegs_b200.optim.Adam: weight_decay / amsgrad are not used by the reference")
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=0, amsgrad=False))

    @torch.no_grad()
    def step(self, relevant=None, closure=None, grad_scale=1.0):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        mask = idx = None
        if relevant is not None and relevant.numel() != 0:
            if relevant.dtype == torch.bool:
                mask = relevant.contiguous().view(torch.uint8)
            else:
                idx = relevant.to(torch.int64).contiguous()
        for group in self.param_groups:
            beta1, beta2 = group["betas"]
            for p in group["params"]:
                if p.grad is None:
                    continue
                if not p.is_cuda or p.dtype != torch.float32 or not p.is_contiguous():
                    raise RuntimeError("hidegs_b200.optim.Adam needs contiguous float32 CUDA parameters")
                state = self.state[p]
                if len(state) == 0:
                    state["step"] = 0
                    state["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    state["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                state["step"] += 1
                if p.numel() == 0:
                    continue
                g = p.grad.contiguous()
                rows = p.size(0) if p.dim() > 0 else 1
                width = p.numel() // max(rows, 1)
                with torch.cuda.device(p.device):
                    rc = _G().hg_adam_step(
                        p.data_ptr(), g.data_ptr(), state["exp_avg"].data_ptr(), state["exp_avg_sq"].data_ptr(), rows,
                        width, mask.data_ptr() if mask is not None else None, idx.data_ptr() if idx is not None else None,
                        idx.numel() if idx is not None else 0, float(group["lr"]), float(beta1), float(beta2),
                        float(group["eps"]), int(state["step"]), float(grad_scale), 0, 0.0, torch.cuda.current_stream().cuda_stream)
                _lib.check(rc, "adam_step")
        return loss


def get_expon_lr_func(lr_init, lr_final, lr_delay_steps=0, lr_delay_mult=1.0, max_steps=1000000):
    """graphdeco 3DGS's learning-rate schedule (utils/general_utils.py get_expon_lr_func): log-linear from lr_init at
    step 0 to lr_final at max_steps (held there after), times a delay factor that rises from lr_delay_mult to 1 along a
    quarter sine over the first lr_delay_steps steps.  A negative step, or lr_init = lr_final = 0, gives 0."""
    def helper(step):
        if step < 0 or (lr_init == 0.0 and lr_final == 0.0):
            return 0.0
        if lr_delay_steps > 0:
            delay_rate = lr_delay_mult + (1 - lr_delay_mult) * np.sin(0.5 * np.pi * np.clip(step / lr_delay_steps, 0, 1))
        else:
            delay_rate = 1.0
        t = np.clip(step / max_steps, 0, 1)
        log_lerp = np.exp(np.log(lr_init) * (1 - t) + np.log(lr_final) * t)
        return float(delay_rate * log_lerp)
    return helper
