"""ctypes prototypes of include/hidegs_losses.h (same shared library as the rasterizer)."""
import ctypes

from . import _lib

EXPORTED_SYMBOLS = (
    "hg_reduce_workspace_bytes", "hg_l1_loss", "hg_l2_loss", "hg_pixel_loss_backward", "hg_freq_total", "hg_training_image_grad", "hg_exposure_apply", "hg_exposure_grad_workspace_bytes",
    "hg_training_image_grad_exposure", "hg_invdepth_l1_workspace_bytes", "hg_invdepth_l1", "hg_training_loss_value", "hg_ssim_workspace_bytes", "hg_ssim", "hg_ssim_backward",
    "hg_ssim_window_workspace_bytes", "hg_ssim_window", "hg_ssim_window_backward",
    "hg_img_grad_weight_workspace_bytes", "hg_img_grad_weight", "hg_lncc", "hg_lncc_backward",
    "hg_scale_reg_workspace_bytes", "hg_scale_reg", "hg_fft2_workspace_bytes", "hg_fft2_r2c", "hg_fft2_c2r",
    "hg_freq_loss_workspace_bytes", "hg_freq_loss", "hg_freq_forward", "hg_freq_backward", "hg_freq_gt_state_bytes", "hg_freq_gt_prepare", "hg_freq_loss_cached", "hg_hf_mask_workspace_bytes", "hg_hf_mask",
)
FREQ_STATS = 24
_ready = False


def lib():
    global _ready
    L = _lib.lib()
    if _ready:
        return L
    vp, i32, i64, sz, f32 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t, ctypes.c_float
    proto = {
        "hg_reduce_workspace_bytes": (sz, [i64]),
        "hg_l1_loss": (ctypes.c_int, [vp, vp, i64, vp, vp, vp, vp]),
        "hg_l2_loss": (ctypes.c_int, [vp, vp, i64, vp, vp, vp, vp]),
        "hg_pixel_loss_backward": (ctypes.c_int, [vp, vp, i64, i32, vp, vp, vp, vp]),
        "hg_freq_total": (ctypes.c_int, [vp, vp, vp, f32, f32, vp, vp]),
        "hg_training_image_grad": (ctypes.c_int, [vp, vp, vp, vp, i64, f32, f32, vp, vp, vp]),
        "hg_exposure_apply": (ctypes.c_int, [vp, vp, i32, i32, vp, vp]),
        "hg_exposure_grad_workspace_bytes": (sz, [i32, i32]),
        "hg_training_image_grad_exposure": (ctypes.c_int, [vp, vp, vp, vp, vp, i32, i32, f32, f32, vp, vp, vp, vp, vp]),
        "hg_invdepth_l1_workspace_bytes": (sz, [i32, i32]),
        "hg_invdepth_l1": (ctypes.c_int, [vp, vp, vp, i32, i32, f32, vp, vp, vp, vp, vp]),
        "hg_training_loss_value": (ctypes.c_int, [vp, vp, vp, vp, f32, vp, vp]),
        "hg_ssim_workspace_bytes": (sz, [i32, i32, i32, i32]),
        "hg_ssim": (ctypes.c_int, [vp, vp, i32, i32, i32, i32, vp, vp, vp, vp]),
        "hg_ssim_backward": (ctypes.c_int, [vp, vp, vp, vp, i32, i32, i32, i32, vp, vp]),
        "hg_ssim_window_workspace_bytes": (sz, [i32, i32, i32, i32]),
        "hg_ssim_window": (ctypes.c_int, [vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, vp]),
        "hg_ssim_window_backward": (ctypes.c_int, [vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, vp, vp]),
        "hg_img_grad_weight_workspace_bytes": (sz, [i32, i32]),
        "hg_img_grad_weight": (ctypes.c_int, [vp, i32, i32, i32, vp, vp, vp]),
        "hg_lncc": (ctypes.c_int, [vp, vp, i32, i32, vp, vp, vp]),
        "hg_lncc_backward": (ctypes.c_int, [vp, vp, vp, i32, i32, vp, vp, vp]),
        "hg_scale_reg_workspace_bytes": (sz, [i64]),
        "hg_scale_reg": (ctypes.c_int, [vp, i64, vp, vp, i64, vp, vp, vp, vp]),
        "hg_fft2_workspace_bytes": (sz, [i32, i32]),
        "hg_fft2_r2c": (ctypes.c_int, [vp, i32, i32, vp, vp, vp]),
        "hg_fft2_c2r": (ctypes.c_int, [vp, i32, i32, vp, ctypes.c_int, vp, vp]),
        "hg_freq_loss_workspace_bytes": (sz, [i32, i32, i32]),
        "hg_freq_loss": (ctypes.c_int, [vp, vp, i32, i32, i32, vp, vp, vp, vp]),
        "hg_freq_forward": (ctypes.c_int, [vp, vp, vp, i32, i32, i32, f32, vp, vp, vp, vp, vp]),
        "hg_freq_backward": (ctypes.c_int, [vp, i32, i32, i32, i32, vp, vp, vp, vp]),
        "hg_freq_gt_state_bytes": (sz, [i32, i32, i32]),
        "hg_freq_gt_prepare": (ctypes.c_int, [vp, i32, i32, i32, vp, vp]),
        "hg_freq_loss_cached": (ctypes.c_int, [vp, vp, i32, i32, i32, vp, vp, vp, vp]),
        "hg_hf_mask_workspace_bytes": (sz, [i32, i32]),
        "hg_hf_mask": (ctypes.c_int, [vp, i32, i32, f32, vp, vp, vp, vp]),
    }
    for name, (res, args) in proto.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _ready = True
    return L
