/*
 * hidegs_losses.h — C-ABI of the B200-native HiDeGS training losses.
 *
 * Every entry point takes device pointers (fp32, contiguous, CHW images), sizes, scalars, a
 * caller-provided workspace and a cudaStream_t (as void*); results stay on the device (no host
 * synchronisation inside); status codes as in hidegs_raster.h.
 *
 * Reference functions replaced (paths relative to the reference tree):
 *   hg_l1_loss, hg_l2_loss      utils/loss_utils.py:18-22  l1_loss / l2_loss
 *   hg_ssim, hg_ssim_backward   utils/loss_utils.py:24-64  ssim / _ssim / create_window / gaussian
 *   hg_img_grad_weight          utils/loss_utils.py:66-78  get_img_grad_weight
 *   hg_lncc, hg_lncc_backward   utils/loss_utils.py:80-115 lncc
 *   hg_scale_reg                scripts/frequency_regularization.py:1403-1444 compute_scale_regularization
 *   hg_fft2_r2c, hg_fft2_c2r    torch.fft.fft2 / ifft2 as used at scripts/frequency_regularization.py:1110,1221,1227
 *   hg_freq_loss                scripts/frequency_regularization.py:1073-1082 build_pyramid, :1327-1360
 *                               _compute_spatial_frequency_loss, :1084-1164 compute_fft_features, :1362-1401
 *                               _compute_fft_frequency_loss, :1293-1325 compute_true_frequency_loss
 *   hg_hf_mask                  scripts/frequency_regularization.py:1166-1271 detect_true_high_frequency_regions
 *
 * Value-and-gradient convention: the losses that feed a training step return their value AND the
 * gradient w.r.t. the rendered image for a unit upstream gradient in the same call (the autograd
 * wrapper scales it by the incoming scalar), so the image is read once.
 */
#ifndef HIDEGS_LOSSES_H
#define HIDEGS_LOSSES_H

#include <stddef.h>
#include <stdint.h>
#include "hidegs_raster.h"

#ifdef __cplusplus
extern "C" {
#endif

/* mean |a-b| (l1) or mean (a-b)^2 (l2) over n elements -> out[0]; grad_a (nullable): d out / d a. */
HG_API size_t hg_reduce_workspace_bytes(int64_t n);
HG_API int hg_l1_loss(const float *a, const float *b, int64_t n, float *out, float *grad_a,
                      void *workspace, void *stream);
HG_API int hg_l2_loss(const float *a, const float *b, int64_t n, float *out, float *grad_a,
                      void *workspace, void *stream);

/* Backward of hg_l1_loss (squared = 0) / hg_l2_loss (squared = 1): grad_a = gscale[0] * d loss / d a, grad_b = -grad_a
 * (either may be NULL); gscale: DEVICE scalar (NULL = 1). */
HG_API int hg_pixel_loss_backward(const float *a, const float *b, int64_t n, int32_t squared, const float *gscale,
                                  float *grad_a, float *grad_b, void *stream);

/* Scalar tail of frequency_regularization_pyramid_scale (scripts/frequency_regularization.py:1636-1660) in one launch:
 *   out3[0] = clamp(lambda_freq * freq_loss[0] + lambda_scale * scale_loss[0] * [hf_count[0] > 0], 0, 1)
 *   out3[1] = d out3[0] / d freq_loss, out3[2] = d out3[0] / d scale_loss   (zero where the clamp saturates)
 * freq_loss / scale_loss: device scalars, either may be NULL (term absent); hf_count: pixel count of the mask. */
HG_API int hg_freq_total(const float *freq_loss, const float *scale_loss, const float *hf_count, float lambda_freq,
                         float lambda_scale, float *out3, void *stream);

/* Image gradient of the composed training loss in one pass (used by the autograd-free executor of the training step,
 * hidegs_b200/trainer.py; the reference composes the same terms with autograd: (1 - lambda) l1_loss + lambda (1 - ssim)
 * + frequency term, on render().clamp(0, 1) — utils/loss_utils.py:18-64, gaussian_renderer/__init__.py:170):
 *   out = [0 <= color <= 1] * ( w_l1 * sign(clamp(color, 0, 1) - gt) / n  +  w_ssim * g_ssim  +  w_freq[0] * g_freq )
 * color, gt, out: n floats (out may alias g_ssim or g_freq); g_ssim / g_freq: dSSIM/dimage and dfreq/dimage for a unit
 * upstream gradient, nullable; w_freq: DEVICE scalar (the clamp gate times lambda_freq), nullable = 0. */
HG_API int hg_training_image_grad(const float *color, const float *gt, const float *g_ssim, const float *g_freq,
                                  int64_t n, float w_l1, float w_ssim, const float *w_freq, float *out, void *stream);

/* Learned per-image exposure (the reference's render(..., use_trained_exp=True), gaussian_renderer/__init__.py:181-184;
 * definition in DESIGN.md §3).  exposure12: DEVICE pointer to E [3, 4] row major (12 contiguous floats; the host never
 * reads it).  Per pixel of color [3, H, W]:
 *   e[ch] = sum_c color[c] * E[c][ch] + E[ch][3]        (torch.matmul(img.permute(1, 2, 0), E[:3, :3]) + E[:3, 3])
 * hg_exposure_apply:  out = clamp(e, 0, 1)  (out may alias color).
 * hg_training_image_grad_exposure:  hg_training_image_grad on the exposed image, taken through the exposure:
 *   ge  = [0 <= e <= 1] * ( w_l1 * sign(clamp(e, 0, 1) - gt) / (3 H W)  +  w_ssim * g_ssim  +  w_freq[0] * g_freq )
 *   out[c] = sum_ch E[c][ch] * ge[ch]                   (out may alias g_ssim or g_freq)
 *   exposure_grad12[c][ch] += sum_pixels color[c] * ge[ch],   exposure_grad12[ch][3] += sum_pixels ge[ch]
 * The sums are deterministic (grid fixed by H * W, per-CTA partials, fixed-order final sum in double by the last CTA)
 * and ADDED to exposure_grad12.  workspace: hg_exposure_grad_workspace_bytes(H, W) bytes, zero-filled before its first
 * use; every call leaves its ticket counter at zero again, so one workspace serves any later call of the same or a
 * smaller size on the same stream.  With E = eye(3, 4), out equals hg_training_image_grad's bit for bit. */
HG_API int hg_exposure_apply(const float *color, const float *exposure12, int32_t H, int32_t W, float *out,
                             void *stream);
HG_API size_t hg_exposure_grad_workspace_bytes(int32_t H, int32_t W);
HG_API int hg_training_image_grad_exposure(const float *color, const float *exposure12, const float *gt,
                                           const float *g_ssim, const float *g_freq, int32_t H, int32_t W, float w_l1,
                                           float w_ssim, const float *w_freq, float *out, float *exposure_grad12,
                                           void *workspace, void *stream);

/* Monocular inverse-depth supervision (graphdeco 3DGS / hierarchical-3DGS's `Ll1depth`; definition in DESIGN.md §3
 * "Depth regularisation").  invdepth: the rasterizer's inverse depth [H, W]; mono: the camera's prior [H, W]; mask:
 * [H, W] fp32 or NULL (all ones).  One streaming pass:
 *   d = (invdepth - mono) * mask
 *   grad[p] = (weight / (H W)) * sgn(d[p]) * mask[p]          (sgn(0) = 0; weight * (1 / (H W)) rounded in fp32)
 *   value[0] = mean |d|  (unweighted)                         loss_inout[0] += weight * value[0]  (when not NULL)
 * The sum is deterministic (grid fixed by H * W, per-CTA partials, fixed-order final sum in double by the last CTA) and
 * does not depend on the alignment of the pointers.  weight is a host float: no host read, no synchronisation.
 * workspace: hg_invdepth_l1_workspace_bytes(H, W) bytes, zero-filled before its first use; every call leaves its
 * ticket counter at zero again, so one workspace serves any later call of the same or a smaller size on the same
 * stream. */
HG_API size_t hg_invdepth_l1_workspace_bytes(int32_t H, int32_t W);
HG_API int hg_invdepth_l1(const float *invdepth, const float *mono, const float *mask, int32_t H, int32_t W,
                          float weight, float *grad, float *value, float *loss_inout, void *workspace, void *stream);

/* Value of the composed training loss of one view (the sum a training loop forms from the reference's pieces:
 * `(1.0 - lambda_dssim) * l1_loss(...) + lambda_dssim * (1.0 - ssim(...))` plus up to two more device scalars, e.g. the
 * total of frequency_regularization_pyramid_scale and the normal term), the Python expression's operations in its
 * order, one launch.  All pointers are DEVICE scalars; extra0 / extra1 nullable. */
HG_API int hg_training_loss_value(const float *l1, const float *ssim, const float *extra0, const float *extra1,
                                  float lambda_dssim, float *out, void *stream);

/* SSIM with the reference's 11x11 sigma=1.5 window, zero padding 5, C1=1e-4, C2=9e-4.
 * img1/img2: [B,C,H,W].  out[b] = mean over (C,H,W) of the SSIM map of batch item b (the Python
 * wrapper averages over b for size_average=True).  If `maps` != NULL (3*B*C*H*W floats) the three
 * partial-derivative maps needed by hg_ssim_backward are stored. */
HG_API size_t hg_ssim_workspace_bytes(int32_t B, int32_t C, int32_t H, int32_t W);
HG_API int hg_ssim(const float *img1, const float *img2, int32_t B, int32_t C, int32_t H, int32_t W,
                   float *out, float *maps, void *workspace, void *stream);
/* grad_img1 = d (sum_b gscale[b] * out[b]) / d img1, gscale: device [B]. */
HG_API int hg_ssim_backward(const float *img1, const float *img2, const float *maps, const float *gscale,
                            int32_t B, int32_t C, int32_t H, int32_t W, float *grad_img1, void *stream);

/* ssim(img1, img2, window_size) for any odd window_size in 1..63 (loss_utils.py:24-64 with a non-default window;
 * hg_ssim / hg_ssim_backward are the tiled kernels of the default 11).  Same outputs and derivative maps; `workspace` of
 * hg_ssim_window_workspace_bytes() bytes is needed by both calls (its contents need not survive between them). */
HG_API size_t hg_ssim_window_workspace_bytes(int32_t B, int32_t C, int32_t H, int32_t W);
HG_API int hg_ssim_window(const float *img1, const float *img2, int32_t B, int32_t C, int32_t H, int32_t W,
                          int32_t window_size, float *out, float *maps, void *workspace, void *stream);
HG_API int hg_ssim_window_backward(const float *img1, const float *img2, const float *maps, const float *gscale,
                                   int32_t B, int32_t C, int32_t H, int32_t W, int32_t window_size, float *grad_img1,
                                   void *workspace, void *stream);

/* get_img_grad_weight: img [C,H,W] -> out [H,W] (border = 1.0). */
HG_API size_t hg_img_grad_weight_workspace_bytes(int32_t H, int32_t W);
HG_API int hg_img_grad_weight(const float *img, int32_t C, int32_t H, int32_t W, float *out,
                              void *workspace, void *stream);

/* lncc: ref/nea [bs,tps] -> ncc [bs], mask [bs] (u8: ncc < 0.9). */
HG_API int hg_lncc(const float *ref, const float *nea, int32_t bs, int32_t tps, float *ncc,
                   uint8_t *mask, void *stream);
HG_API int hg_lncc_backward(const float *ref, const float *nea, const float *grad_ncc, int32_t bs,
                            int32_t tps, float *grad_ref, float *grad_nea, void *stream);

/* compute_scale_regularization on index list `vis` (int64 [n_vis]; out-of-range entries ignored, as
 * in the reference) or a bool mask (u8 [N], n_vis < 0).  out[0] = loss; grad_scaling [N,3] (nullable)
 * is fully written (zeros where no gradient flows). */
HG_API size_t hg_scale_reg_workspace_bytes(int64_t n);
HG_API int hg_scale_reg(const float *scaling, int64_t N, const int64_t *vis_idx, const uint8_t *vis_mask,
                        int64_t n_vis, float *out, float *grad_scaling, void *workspace, void *stream);

/* 2-D FFT of a real H x W image -> half spectrum [H, W/2+1] interleaved complex (unnormalised, as
 * torch.fft.fft2), and the inverse (normalised by 1/(H*W), as torch.fft.ifft2 of a Hermitian
 * spectrum; real output).  1 < W, H <= 4096; sizes 2^a 3^b 5^c use radix-4/2/3/5 butterflies, other
 * prime factors a generic O(R^2) butterfly. */
HG_API size_t hg_fft2_workspace_bytes(int32_t H, int32_t W);
HG_API int hg_fft2_r2c(const float *img, int32_t H, int32_t W, float *spec, void *workspace, void *stream);
HG_API int hg_fft2_c2r(const float *spec, int32_t H, int32_t W, float *img, int scale_by_inverse_size,
                       void *workspace, void *stream);

/* Frequency regulariser core: rendered/gt [3,H,W].  Writes
 *   stats[0]  freq_loss (clamp(sum_l w_l level_l, 0, 0.1))
 *   stats[1 + 6*l + {0..5}]  level l: spatial, fft, level (clamped), mag, phase, band   (l < levels <= 3)
 *   stats[19..22]  band energies of the level-0 ground-truth spectrum
 * and, if grad_rendered != NULL, d freq_loss / d rendered [3,H,W]. */
#define HG_FREQ_STATS 24
HG_API size_t hg_freq_loss_workspace_bytes(int32_t H, int32_t W, int32_t levels);
HG_API int hg_freq_loss(const float *rendered, const float *gt, int32_t H, int32_t W, int32_t levels,
                        float *stats, float *grad_rendered, void *workspace, void *stream);

/* The same regulariser as two calls, for callers that keep the forward state until a backward arrives (autograd):
 *   hg_freq_forward   value + stats (as hg_freq_loss); the ground truth comes either as the image `gt` or as a state
 *                     prepared by hg_freq_gt_prepare (`gt_state`, then `gt` may be NULL).  If hf_mask != NULL the
 *                     high-frequency mask of the same ground truth (hg_hf_mask: mask [H,W], hf_count[0] = sum) is produced
 *                     by the same launches (its row / column transforms ride the regulariser's kernels).
 *   hg_freq_backward  grad_rendered [3,H,W] = gscale[0] * d freq_loss / d rendered (gscale: DEVICE scalar, NULL = 1) from
 *                     the state hg_freq_forward left in `workspace` (same H, W, levels, gt_state; forward_had_hf_mask
 *                     tells whether that forward call produced the mask, which fixes the workspace layout).
 * Six launches in total (nine with the mask); the scalar epilogue runs in the last CTA of the column kernel. */
HG_API int hg_freq_forward(const float *rendered, const float *gt, void *gt_state, int32_t H, int32_t W, int32_t levels,
                           float hf_thresh, float *hf_mask, float *hf_count, float *stats, void *workspace,
                           void *stream);
HG_API int hg_freq_backward(void *gt_state, int32_t H, int32_t W, int32_t levels, int32_t forward_had_hf_mask,
                            const float *gscale, float *grad_rendered, void *workspace, void *stream);

/* The ground-truth side of hg_freq_loss (gray pyramid of gt, its spectra, the level-0 band sums) depends on the camera's
 * image only.  A training loop that revisits a camera prepares it once (hg_freq_gt_prepare into a caller-owned state of
 * hg_freq_gt_state_bytes bytes) and calls hg_freq_loss_cached, which is hg_freq_loss minus that work (3 of the 6
 * forward FFTs); results are bit-identical to the uncached call. */
HG_API size_t hg_freq_gt_state_bytes(int32_t H, int32_t W, int32_t levels);
HG_API int hg_freq_gt_prepare(const float *gt, int32_t H, int32_t W, int32_t levels, void *gt_state, void *stream);
HG_API int hg_freq_loss_cached(const float *rendered, void *gt_state, int32_t H, int32_t W, int32_t levels,
                               float *stats, float *grad_rendered, void *workspace, void *stream);

/* detect_true_high_frequency_regions on gt [3,H,W] -> mask [H,W] float (0/1); count[0] = sum(mask). */
HG_API size_t hg_hf_mask_workspace_bytes(int32_t H, int32_t W);
HG_API int hg_hf_mask(const float *gt, int32_t H, int32_t W, float thresh, float *mask, float *count,
                      void *workspace, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* HIDEGS_LOSSES_H */
