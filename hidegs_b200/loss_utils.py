"""Drop-in for the reference's utils/loss_utils.py (same function names and signatures), backed by
fused sm_100a kernels through the C-ABI of include/hidegs_losses.h.

  l1_loss(network_output, gt)                      utils/loss_utils.py:18-19
  l2_loss(network_output, gt)                      utils/loss_utils.py:21-22
  ssim(img1, img2, window_size=11, size_average=True)   :34-64
  get_img_grad_weight(img, beta=2.0)               :66-78
  lncc(ref, nea)                                   :80-115

CUDA tensors only (no CPU fallback).  Each loss computes its value and the gradient w.r.t. the
rendered image in one pass; autograd's backward only scales that gradient.
"""
import torch

from . import _lib
from ._losses_lib import lib as _L


def _check_cuda(*ts):
    for t in ts:
        if not t.is_cuda:
            raise RuntimeError("hidegs_b200 losses need CUDA tensors (there is no CPU path)")
        if t.dtype != torch.float32:
            raise RuntimeError("hidegs_b200 losses expect float32 tensors, got %s" % t.dtype)


def _ws(nbytes, device):
    return torch.empty(int(nbytes), dtype=torch.uint8, device=device)


def _stream():
    return torch.cuda.current_stream().cuda_stream


class _PixelLoss(torch.autograd.Function):
    """forward: value only (both images read once); backward: one kernel, the upstream scalar read on the device."""

    @staticmethod
    def forward(ctx, a, b, l2):
        _check_cuda(a, b)
        if a.shape != b.shape:
            raise RuntimeError("l1/l2 loss: shapes differ %s vs %s" % (tuple(a.shape), tuple(b.shape)))
        a_c, b_c = a.contiguous(), b.contiguous()
        out = torch.empty(1, dtype=torch.float32, device=a.device)
        with torch.cuda.device(a.device):
            ws = _ws(_L().hg_reduce_workspace_bytes(a_c.numel()), a.device)
            fn = _L().hg_l2_loss if l2 else _L().hg_l1_loss
            rc = fn(a_c.data_ptr(), b_c.data_ptr(), a_c.numel(), out.data_ptr(), None, ws.data_ptr(), _stream())
        _lib.check(rc, "l2_loss" if l2 else "l1_loss")
        ctx.save_for_backward(a_c, b_c)
        ctx.l2 = bool(l2)
        return out.reshape(())

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        need_a, need_b = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if not (need_a or need_b):
            return None, None, None
        ga = torch.empty_like(a) if need_a else None
        gb = torch.empty_like(b) if need_b else None
        gs = g.detach().reshape(1).to(dtype=torch.float32).contiguous()
        with torch.cuda.device(a.device):
            rc = _L().hg_pixel_loss_backward(a.data_ptr(), b.data_ptr(), a.numel(), int(ctx.l2), gs.data_ptr(),
                                             ga.data_ptr() if need_a else None, gb.data_ptr() if need_b else None, _stream())
        _lib.check(rc, "pixel_loss_backward")
        return ga, gb, None


def l1_loss(network_output, gt):
    return _PixelLoss.apply(network_output, gt, False)


def l2_loss(network_output, gt):
    return _PixelLoss.apply(network_output, gt, True)


class _SSIM(torch.autograd.Function):
    """ssim (loss_utils.py:24-64).  window 11 (every call site of the reference): the tiled shared-memory kernels;
    any other odd window: the two-pass kernels of hg_ssim_window."""

    @staticmethod
    def _fwd(x, y, B, C, H, W, window, out, maps):
        if window == 11:
            ws = _ws(_L().hg_ssim_workspace_bytes(B, C, H, W), x.device)
            rc = _L().hg_ssim(x.data_ptr(), y.data_ptr(), B, C, H, W, out.data_ptr(), maps.data_ptr() if maps is not None else None,
                              ws.data_ptr(), _stream())
        else:
            ws = _ws(_L().hg_ssim_window_workspace_bytes(B, C, H, W), x.device)
            rc = _L().hg_ssim_window(x.data_ptr(), y.data_ptr(), B, C, H, W, window, out.data_ptr(),
                                     maps.data_ptr() if maps is not None else None, ws.data_ptr(), _stream())
        _lib.check(rc, "ssim")

    @staticmethod
    def _bwd(x, y, maps, gs, B, C, H, W, window, grad):
        if window == 11:
            rc = _L().hg_ssim_backward(x.data_ptr(), y.data_ptr(), maps.data_ptr(), gs.data_ptr(), B, C, H, W, grad.data_ptr(),
                                       _stream())
        else:
            ws = _ws(_L().hg_ssim_window_workspace_bytes(B, C, H, W), x.device)
            rc = _L().hg_ssim_window_backward(x.data_ptr(), y.data_ptr(), maps.data_ptr(), gs.data_ptr(), B, C, H, W, window,
                                              grad.data_ptr(), ws.data_ptr(), _stream())
        _lib.check(rc, "ssim_backward")

    @staticmethod
    def forward(ctx, img1, img2, size_average, window=11):
        _check_cuda(img1, img2)
        if img1.shape != img2.shape or img1.dim() not in (3, 4):
            raise RuntimeError("ssim: expected two (C,H,W) or (B,C,H,W) tensors of the same shape")
        x, y = img1.contiguous(), img2.contiguous()
        B = x.size(0) if x.dim() == 4 else 1
        C, H, W = x.shape[-3:]
        need1, need2 = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        out = torch.empty(B, dtype=torch.float32, device=x.device)
        maps = torch.empty((3,) + tuple(x.shape), dtype=torch.float32, device=x.device) if need1 else None
        with torch.cuda.device(x.device):
            _SSIM._fwd(x, y, B, C, H, W, window, out, maps)
        ctx.save_for_backward(x, y)
        ctx.maps, ctx.dims, ctx.size_average, ctx.need2, ctx.window = maps, (B, C, H, W), size_average, need2, window
        if size_average:
            return out.mean() if B > 1 else out.reshape(())
        if x.dim() != 4:
            raise RuntimeError("ssim(size_average=False) needs a batched (B,C,H,W) input, as in the reference")
        return out

    @staticmethod
    def backward(ctx, g):
        x, y = ctx.saved_tensors
        B, C, H, W = ctx.dims
        if ctx.size_average:  # mean over the batch: every item receives g / B (no kernel for the usual B == 1)
            gs = g.detach().reshape(1) if B == 1 else (g.detach().reshape(1) / B).expand(B)
        else:
            gs = g.detach()
        gs = gs.contiguous().float()
        g1 = g2 = None
        with torch.cuda.device(x.device):
            if ctx.needs_input_grad[0]:
                g1 = torch.empty_like(x)
                _SSIM._bwd(x, y, ctx.maps, gs, B, C, H, W, ctx.window, g1)
            if ctx.need2:  # SSIM is symmetric in its arguments: swap roles for d/d img2
                out = torch.empty(B, dtype=torch.float32, device=x.device)
                maps = torch.empty((3,) + tuple(x.shape), dtype=torch.float32, device=x.device)
                _SSIM._fwd(y, x, B, C, H, W, ctx.window, out, maps)
                g2 = torch.empty_like(x)
                _SSIM._bwd(y, x, maps, gs, B, C, H, W, ctx.window, g2)
        return g1, g2, None, None


def ssim(img1, img2, window_size=11, size_average=True):
    window_size = int(window_size)
    if window_size < 1 or window_size > 63 or window_size % 2 == 0:
        # an even window makes the reference's conv2d(padding=window_size // 2) return maps one pixel larger than the
        # images; no call site uses one
        raise ValueError("hidegs_b200.ssim: window_size must be odd and in 1..63 (got %d)" % window_size)
    return _SSIM.apply(img1, img2, size_average, window_size)


def _invdepth_l1_launch(invdepth, mono, mask, weight, grad, value, loss_inout, ws):
    """hg_invdepth_l1 on contiguous [.., H, W] fp32 CUDA tensors (mask may be None, loss_inout may be None)."""
    H, W = invdepth.shape[-2:]
    with torch.cuda.device(invdepth.device):
        rc = _L().hg_invdepth_l1(invdepth.data_ptr(), mono.data_ptr(), mask.data_ptr() if mask is not None else None,
                                 H, W, float(weight), grad.data_ptr(), value.data_ptr(),
                                 loss_inout.data_ptr() if loss_inout is not None else None, ws.data_ptr(), _stream())
    _lib.check(rc, "invdepth_l1")


class _InvDepthL1(torch.autograd.Function):
    """mean |(invdepth - mono) * mask|: value and unit-weight gradient in one pass (hg_invdepth_l1); the backward scales
    that gradient by the upstream scalar.  The prior and the mask receive no gradient."""

    @staticmethod
    def forward(ctx, invdepth, mono, mask):
        ts = (invdepth, mono) + ((mask,) if mask is not None else ())
        _check_cuda(*ts)
        if any(t.shape != invdepth.shape for t in ts) or invdepth.dim() < 2 or invdepth.numel() != \
                invdepth.size(-1) * invdepth.size(-2):
            raise RuntimeError("inverse_depth_l1: expected [1, H, W] / [H, W] tensors of one shape, got %s"
                               % [tuple(t.shape) for t in ts])
        x, m = invdepth.contiguous(), mono.contiguous()
        k = mask.contiguous() if mask is not None else None
        H, W = x.shape[-2:]
        grad = torch.empty_like(x)
        value = torch.empty((), dtype=torch.float32, device=x.device)
        ws = torch.zeros(int(_L().hg_invdepth_l1_workspace_bytes(H, W)), dtype=torch.uint8, device=x.device)
        _invdepth_l1_launch(x, m, k, 1.0, grad, value, None, ws)
        ctx.save_for_backward(grad)
        return value

    @staticmethod
    def backward(ctx, g):
        (grad,) = ctx.saved_tensors
        return grad * g.detach().reshape(()), None, None


def inverse_depth_l1(invdepth, mono, mask=None):
    """mean_{H,W} |(invdepth - mono) * mask| (graphdeco's Ll1depth without its weight; DESIGN.md §3 "Depth
    regularisation"): `invdepth` the rendered inverse depth [1, H, W], `mono` the camera's prior, `mask` a float map or
    None for all ones.  Differentiable w.r.t. `invdepth` only."""
    return _InvDepthL1.apply(invdepth, mono, mask)


def get_img_grad_weight(img, beta=2.0):
    """Edge-aware weight map of an image (used on ground-truth images; returned without autograd history)."""
    _check_cuda(img)
    if img.dim() != 3:
        raise RuntimeError("get_img_grad_weight expects a (C,H,W) image")
    x = img.detach().contiguous()
    C, H, W = x.shape
    out = torch.empty((H, W), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        ws = _ws(_L().hg_img_grad_weight_workspace_bytes(H, W), x.device)
        rc = _L().hg_img_grad_weight(x.data_ptr(), C, H, W, out.data_ptr(), ws.data_ptr(), _stream())
    _lib.check(rc, "get_img_grad_weight")
    return out


class _LNCC(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ref, nea):
        _check_cuda(ref, nea)
        if ref.shape != nea.shape or ref.dim() != 2:
            raise RuntimeError("lncc expects two (batch, patch*patch) tensors of the same shape")
        r, n = ref.contiguous(), nea.contiguous()
        bs, tps = n.shape
        ncc = torch.empty((bs, 1), dtype=torch.float32, device=r.device)
        mask = torch.empty((bs, 1), dtype=torch.bool, device=r.device)
        with torch.cuda.device(r.device):
            rc = _L().hg_lncc(r.data_ptr(), n.data_ptr(), bs, tps, ncc.data_ptr(), mask.data_ptr(), _stream())
        _lib.check(rc, "lncc")
        ctx.save_for_backward(r, n)
        ctx.mark_non_differentiable(mask)
        return ncc, mask

    @staticmethod
    def backward(ctx, g_ncc, _g_mask):
        r, n = ctx.saved_tensors
        bs, tps = n.shape
        gr, gn = torch.empty_like(r), torch.empty_like(n)
        g = g_ncc.contiguous().float()
        with torch.cuda.device(r.device):
            rc = _L().hg_lncc_backward(r.data_ptr(), n.data_ptr(), g.data_ptr(), bs, tps, gr.data_ptr(), gn.data_ptr(), _stream())
        _lib.check(rc, "lncc_backward")
        return gr, gn


def lncc(ref, nea):
    return _LNCC.apply(ref, nea)
