// exposure.cu — learned per-image exposure of the training step (the reference's `render(..., use_trained_exp=True)`,
// gaussian_renderer/__init__.py:181-184) as sm_100a kernels: the exposed, clamped image, and the composed image gradient
// of the training loss through the exposure with the 12 exposure sums, in one pass.  Definition: DESIGN.md §3
// "Per-image exposure".
//
// An exposure is 12 contiguous fp32 on the device (E [3, 4], row major); the host never reads it.  Per pixel
//   e[ch] = c[0] E[0][ch] + c[1] E[1][ch] + c[2] E[2][ch] + E[ch][3]      image = clamp(e, 0, 1)
// (torch.matmul(img.permute(1, 2, 0), E[:3, :3]) + E[:3, 3]: the pixel row vector times E[:3, :3]).
#include "common.cuh"
#include "reduce.cuh"
#include "../../include/hidegs_losses.h"

namespace hg {

namespace {

constexpr int kExpThreads = 256;
constexpr int kExpPix = 4;                              // pixels per thread of the gradient kernel
constexpr int kExpPixPerCta = kExpThreads * kExpPix;    // the grid depends on H * W only
constexpr size_t kExpCounterBytes = 256;                // [0]: ticket counter of the last-CTA reduction

// The exposed value of channel ch: ONE fma chain, shared by both kernels, so the clamp gate and the L1 sign of the
// backward see exactly the image the losses saw.  With E = eye(3, 4) every product is by an exact 0 or 1 and the
// result equals c[ch] bit for bit (up to the sign of a zero).
__device__ __forceinline__ float exposed(const float (&E)[12], int ch, float c0, float c1, float c2) {
  return __fmaf_rn(c0, E[ch], __fmaf_rn(c1, E[4 + ch], __fmaf_rn(c2, E[8 + ch], E[4 * ch + 3])));
}

__device__ __forceinline__ void load_exposure(const float* __restrict__ e12, float (&E)[12]) {
#pragma unroll
  for (int k = 0; k < 12; ++k) E[k] = __ldg(e12 + k);
}

// Sum of v[0..11] over the CTA in a fixed order (warp butterflies in double, then the 8 warps in index order); the
// result lands in out12[0..11] (shared), valid after the call (it ends with a barrier).
__device__ __forceinline__ void cta_sum12(double (&v)[12], double (*sm)[12], double* out12) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 12; ++k) v[k] = warp_sum_double(v[k]);
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 12; ++k) sm[warp][k] = v[k];
  }
  __syncthreads();
  if (threadIdx.x < 12) {
    double s = 0.0;
    for (int w = 0; w < kExpThreads / 32; ++w) s += sm[w][threadIdx.x];
    out12[threadIdx.x] = s;
  }
  __syncthreads();
}

// image = clamp(e, 0, 1), thread per pixel over the three CHW planes (out may be color itself)
__global__ void __launch_bounds__(kExpThreads)
exposure_apply_kernel(const float* color, const float* __restrict__ e12, int64_t hw, float* out) {
  const int64_t i = (int64_t)blockIdx.x * kExpThreads + threadIdx.x;
  if (i >= hw) return;
  float E[12];
  load_exposure(e12, E);
  const float c0 = color[i], c1 = color[hw + i], c2 = color[2 * hw + i];
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) out[ch * hw + i] = fminf(fmaxf(exposed(E, ch, c0, c1, c2), 0.f), 1.f);
}

// ge = [0 <= e <= 1] (w_l1 sign(clamp(e) - gt) / n + w_ssim g_ssim + w_freq g_freq)   (training_image_grad_kernel's
// arithmetic on e);  out[c] = sum_ch E[c][ch] ge[ch];  and the exposure sums
//   dE[c][ch] = sum c[c] ge[ch],  dE[ch][3] = sum ge[ch]
// per thread in fp32 over its kExpPix pixels, per CTA in double (fixed order) -> partial[cta][12]; the last CTA to
// finish adds the sum over the CTAs (index order, double) onto eg12 and re-arms the counter.
__global__ void __launch_bounds__(kExpThreads)
exposure_image_grad_kernel(const float* __restrict__ color, const float* __restrict__ e12, const float* __restrict__ gt,
                           const float* g_ssim, const float* g_freq, int64_t hw, float w_l1_over_n, float w_ssim,
                           const float* __restrict__ w_freq, float* out, double* __restrict__ partial,
                           unsigned* __restrict__ counter, float* __restrict__ eg12) {
  __shared__ double sm[kExpThreads / 32][12];
  __shared__ double s12[12];
  __shared__ int s_last;
  float E[12];
  load_exposure(e12, E);
  const float wf = w_freq ? __ldg(w_freq) : 0.f;
  float acc[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) acc[k] = 0.f;
  const int64_t base = (int64_t)blockIdx.x * kExpPixPerCta + threadIdx.x;
  // every input of the thread's pixels first (out may alias g_ssim / g_freq: a thread writes only its own pixels,
  // after it has read them)
  float c[kExpPix][3], t[kExpPix][3], s[kExpPix][3], f[kExpPix][3];
#pragma unroll
  for (int k = 0; k < kExpPix; ++k) {
    const int64_t i = base + k * kExpThreads;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      const bool in = i < hw;
      const int64_t j = ch * hw + i;
      c[k][ch] = in ? color[j] : 0.f;
      t[k][ch] = in ? gt[j] : 0.f;
      s[k][ch] = (in && g_ssim) ? g_ssim[j] : 0.f;
      f[k][ch] = (in && g_freq) ? g_freq[j] : 0.f;
    }
  }
#pragma unroll
  for (int k = 0; k < kExpPix; ++k) {
    const int64_t i = base + k * kExpThreads;
    if (i >= hw) break;
    float ge[3];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      const float e = exposed(E, ch, c[k][0], c[k][1], c[k][2]);
      const float d = fminf(fmaxf(e, 0.f), 1.f) - t[k][ch];
      float g = (d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f)) * w_l1_over_n;
      if (g_ssim) g = fmaf(w_ssim, s[k][ch], g);
      if (g_freq) g = fmaf(wf, f[k][ch], g);
      ge[ch] = (e >= 0.f && e <= 1.f) ? g : 0.f;  // d clamp(e, 0, 1) / de
    }
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) {
      // (identity: 1 * ge[cc] plus exact zeros = ge[cc], hg_training_image_grad's value)
      out[cc * hw + i] = __fmaf_rn(E[4 * cc], ge[0], __fmaf_rn(E[4 * cc + 1], ge[1], __fmul_rn(E[4 * cc + 2], ge[2])));
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) acc[4 * cc + ch] = __fmaf_rn(c[k][cc], ge[ch], acc[4 * cc + ch]);
      acc[4 * cc + 3] = __fadd_rn(acc[4 * cc + 3], ge[cc]);
    }
  }
  double v[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) v[k] = (double)acc[k];
  cta_sum12(v, sm, s12);
  if (threadIdx.x < 12) {
    partial[(size_t)blockIdx.x * 12 + threadIdx.x] = s12[threadIdx.x];
    __threadfence();
  }
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(counter, 1u) == gridDim.x - 1 ? 1 : 0;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
#pragma unroll
  for (int k = 0; k < 12; ++k) v[k] = 0.0;
  for (int b = threadIdx.x; b < (int)gridDim.x; b += kExpThreads) {
#pragma unroll
    for (int k = 0; k < 12; ++k) v[k] += __ldcg(partial + (size_t)b * 12 + k);
  }
  cta_sum12(v, sm, s12);
  if (threadIdx.x < 12) eg12[threadIdx.x] = __fadd_rn(eg12[threadIdx.x], (float)s12[threadIdx.x]);
  if (threadIdx.x == 0) *counter = 0u;  // ready for the next call on this workspace
}

int64_t grad_ctas(int64_t hw) { return (hw + kExpPixPerCta - 1) / kExpPixPerCta; }

}  // namespace

}  // namespace hg

using namespace hg;

extern "C" {

int hg_exposure_apply(const float* color, const float* exposure12, int32_t H, int32_t W, float* out, void* st_) {
  if (!color || !exposure12 || !out || H <= 0 || W <= 0) {
    set_error("hg_exposure_apply: bad argument (NULL pointer or H, W <= 0)");
    return HG_ERR_INVALID_ARG;
  }
  cudaStream_t st = (cudaStream_t)st_;
  const int64_t hw = (int64_t)H * W;
  exposure_apply_kernel<<<(unsigned)((hw + kExpThreads - 1) / kExpThreads), kExpThreads, 0, st>>>(color, exposure12,
                                                                                                  hw, out);
  HG_POST_LAUNCH(false, st, "exposure_apply");
  return HG_OK;
}

size_t hg_exposure_grad_workspace_bytes(int32_t H, int32_t W) {
  if (H <= 0 || W <= 0) return 0;
  return kExpCounterBytes + sizeof(double) * 12 * (size_t)grad_ctas((int64_t)H * W);
}

int hg_training_image_grad_exposure(const float* color, const float* exposure12, const float* gt, const float* g_ssim,
                                    const float* g_freq, int32_t H, int32_t W, float w_l1, float w_ssim,
                                    const float* w_freq, float* out, float* exposure_grad12, void* workspace,
                                    void* st_) {
  if (!color || !exposure12 || !gt || !out || !exposure_grad12 || !workspace || H <= 0 || W <= 0) {
    set_error("hg_training_image_grad_exposure: bad argument (NULL pointer or H, W <= 0)");
    return HG_ERR_INVALID_ARG;
  }
  cudaStream_t st = (cudaStream_t)st_;
  const int64_t hw = (int64_t)H * W;
  const int64_t n = 3 * hw;
  unsigned* counter = (unsigned*)workspace;
  double* partial = (double*)((char*)workspace + kExpCounterBytes);
  exposure_image_grad_kernel<<<(unsigned)grad_ctas(hw), kExpThreads, 0, st>>>(
      color, exposure12, gt, g_ssim, g_freq, hw, w_l1 / (float)n, w_ssim, w_freq, out, partial, counter,
      exposure_grad12);
  HG_POST_LAUNCH(false, st, "training_image_grad_exposure");
  return HG_OK;
}

}  // extern "C"
