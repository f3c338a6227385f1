// depth_loss.cu — monocular inverse-depth supervision of the training step (graphdeco 3DGS / hierarchical-3DGS's
// `Ll1depth`) as one sm_100a streaming pass: the value of the masked depth L1 and its gradient w.r.t. the rendered
// inverse depth.  Definition: DESIGN.md §3 "Depth regularisation".
//
//   d = (invdepth - mono) * mask                    value = mean_{H,W} |d|
//   grad = (weight / (H W)) * sgn(d) * mask         (sgn(0) = 0, as torch's abs backward)
//
// Every quad of 4 consecutive pixels is read with one float4 load per input where all base pointers are 16-byte
// aligned, with 4 scalar loads otherwise and for the tail quad of H W % 4 != 0.  Both paths hand the pixels to the
// same per-thread sum in the same order, so the value does not depend on the alignment of the views.
#include "common.cuh"
#include "reduce.cuh"
#include "../../include/hidegs_losses.h"

namespace hg {

namespace {

constexpr int kDepThreads = 256;
constexpr int kDepQuads = 4;                                   // quads (4 pixels) per thread
constexpr int64_t kDepPixPerCta = 4LL * kDepQuads * kDepThreads; // the grid depends on H * W only
constexpr size_t kDepCounterBytes = 256;                       // [0]: ticket counter of the last-CTA reduction

// One pixel: its gradient (c = weight / (H W), rounded as torch's mean backward: weight * (1 / (H W))) and |d|.
template <bool kMask>
__device__ __forceinline__ float pixel(float inv, float mono, float m, float c, double& acc) {
  const float r = __fsub_rn(inv, mono);
  const float d = kMask ? __fmul_rn(r, m) : r;
  const float s = d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f);
  acc += (double)fabsf(d);
  const float g = __fmul_rn(c, s);
  return kMask ? __fmul_rn(g, m) : g;
}

// Thread t of CTA b takes quads b * (kDepQuads * T) + k * T + t, k = 0..kDepQuads-1 (coalesced float4 per k); the
// per-thread double sum runs over the quads in k order and the 4 pixels of a quad in order; the CTA sum is a fixed
// warp butterfly + warp-index order -> partial[b].  The last CTA to finish sums the partials in a fixed order
// (cta_sum_strided), writes value, adds weight * value onto loss_inout and re-arms the counter.
template <bool kVec, bool kMask>
__global__ void __launch_bounds__(kDepThreads)
invdepth_l1_kernel(const float* __restrict__ inv, const float* __restrict__ mono, const float* __restrict__ mask,
                   int64_t n, float weight, float c, float* __restrict__ grad, float* __restrict__ value,
                   float* __restrict__ loss_inout, double* __restrict__ partial, unsigned* __restrict__ counter) {
  __shared__ double sm[32];
  __shared__ int s_last;
  double acc = 0.0;
  const int64_t q0 = (int64_t)blockIdx.x * (kDepQuads * kDepThreads) + threadIdx.x;
#pragma unroll
  for (int k = 0; k < kDepQuads; ++k) {
    const int64_t q = q0 + (int64_t)k * kDepThreads;
    const int64_t e = 4 * q;
    if (e >= n) break;
    if (kVec && e + 4 <= n) {
      const float4 a = __ldcs(reinterpret_cast<const float4*>(inv) + q);
      const float4 b = __ldcs(reinterpret_cast<const float4*>(mono) + q);
      const float4 m = kMask ? __ldcs(reinterpret_cast<const float4*>(mask) + q) : make_float4(1.f, 1.f, 1.f, 1.f);
      float4 g;
      g.x = pixel<kMask>(a.x, b.x, m.x, c, acc);
      g.y = pixel<kMask>(a.y, b.y, m.y, c, acc);
      g.z = pixel<kMask>(a.z, b.z, m.z, c, acc);
      g.w = pixel<kMask>(a.w, b.w, m.w, c, acc);
      __stcs(reinterpret_cast<float4*>(grad) + q, g);
    } else {
      for (int j = 0; j < 4 && e + j < n; ++j) {
        const int64_t i = e + j;
        grad[i] = pixel<kMask>(__ldcs(inv + i), __ldcs(mono + i), kMask ? __ldcs(mask + i) : 1.f, c, acc);
      }
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  acc = warp_sum_double(acc);
  if (lane == 0) sm[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < kDepThreads / 32; ++w) s += sm[w];
    partial[blockIdx.x] = s;
    __threadfence();
    s_last = atomicAdd(counter, 1u) == gridDim.x - 1 ? 1 : 0;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  // (__ldcg: the other CTAs' partials are read from L2, past this SM's L1)
  double a0 = 0.0;
  for (int b = threadIdx.x; b < (int)gridDim.x; b += kDepThreads) a0 += __ldcg(partial + b);
  a0 = warp_sum_double(a0);
  __syncthreads();
  if (lane == 0) sm[warp] = a0;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < kDepThreads / 32; ++w) s += sm[w];
    const float v = (float)(s / (double)n);
    *value = v;
    if (loss_inout) *loss_inout = __fadd_rn(*loss_inout, __fmul_rn(weight, v));  // (torch: loss + w * value)
    *counter = 0u;  // ready for the next call on this workspace
  }
}

int64_t depth_ctas(int64_t n) { return (n + kDepPixPerCta - 1) / kDepPixPerCta; }

template <bool kVec, bool kMask>
void launch(const float* inv, const float* mono, const float* mask, int64_t n, float weight, float c, float* grad,
            float* value, float* loss_inout, double* partial, unsigned* counter, cudaStream_t st) {
  invdepth_l1_kernel<kVec, kMask><<<(unsigned)depth_ctas(n), kDepThreads, 0, st>>>(
      inv, mono, mask, n, weight, c, grad, value, loss_inout, partial, counter);
}

}  // namespace

}  // namespace hg

using namespace hg;

extern "C" {

size_t hg_invdepth_l1_workspace_bytes(int32_t H, int32_t W) {
  if (H <= 0 || W <= 0) return 0;
  return kDepCounterBytes + sizeof(double) * (size_t)depth_ctas((int64_t)H * W);
}

int hg_invdepth_l1(const float* invdepth, const float* mono, const float* mask, int32_t H, int32_t W, float weight,
                   float* grad, float* value, float* loss_inout, void* workspace, void* st_) {
  if (!invdepth || !mono || !grad || !value || !workspace || H <= 0 || W <= 0) {
    set_error("hg_invdepth_l1: bad argument (NULL pointer or H, W <= 0)");
    return HG_ERR_INVALID_ARG;
  }
  cudaStream_t st = (cudaStream_t)st_;
  const int64_t n = (int64_t)H * W;
  const float c = weight * (1.0f / (float)n);  // torch's mean backward: grad * (1 / numel) in fp32
  unsigned* counter = (unsigned*)workspace;
  double* partial = (double*)((char*)workspace + kDepCounterBytes);
  auto a16 = [](const void* p) { return ((uintptr_t)p & 15u) == 0; };
  const bool vec = a16(invdepth) && a16(mono) && a16(grad) && (!mask || a16(mask));
  if (vec) {
    if (mask) launch<true, true>(invdepth, mono, mask, n, weight, c, grad, value, loss_inout, partial, counter, st);
    else launch<true, false>(invdepth, mono, mask, n, weight, c, grad, value, loss_inout, partial, counter, st);
  } else {
    if (mask) launch<false, true>(invdepth, mono, mask, n, weight, c, grad, value, loss_inout, partial, counter, st);
    else launch<false, false>(invdepth, mono, mask, n, weight, c, grad, value, loss_inout, partial, counter, st);
  }
  HG_POST_LAUNCH(false, st, "invdepth_l1");
  return HG_OK;
}

}  // extern "C"
