// geometry.cu — per-Gaussian prologue and per-pixel epilogue of the reference's render(), the single-view
// normal-consistency loss, and the fused Adam step (see include/hidegs_geometry.h).
//
// Replaces the PyTorch op chains of
//   gaussian_renderer/__init__.py:161-169  (input_all_map)  + scene/gaussian_model.py:150-166 (get_normal)
//   gaussian_renderer/__init__.py:21-33,200-201 (render_normal * alpha) + utils/graphics_utils.py:17-23,108-166
//   scene/OurAdam.py:249-337 (_single_tensor_adam / _single_tensor_adam2)
// All kernels are HBM-bound streaming passes (one read of every input, one write of every output).
#include "common.cuh"
#include "reduce.cuh"
#include "../../include/hidegs_geometry.h"

#include <climits>
#include <cmath>

namespace hg {

namespace {

// ------------------------------------------------------------------------------------------------
// Per-Gaussian prologue.
struct View {
  float v[16];   // world_view_transform, row-vector convention: p_view_j = sum_i p_i v[4 i + j] + v[12 + j]
  float cam[3];
};

// Column m of pytorch3d's quaternion_to_matrix(q), q = (r, i, j, k), two_s = 2 / |q|^2.
__device__ __forceinline__ void rot_column(const float4 q, int m, float s, float col[3]) {
  const float r = q.x, i = q.y, j = q.z, k = q.w;
  if (m == 0) {
    col[0] = 1.f - s * (j * j + k * k); col[1] = s * (i * j + k * r); col[2] = s * (i * k - j * r);
  } else if (m == 1) {
    col[0] = s * (i * j - k * r); col[1] = 1.f - s * (i * i + k * k); col[2] = s * (j * k + i * r);
  } else {
    col[0] = s * (i * k + j * r); col[1] = s * (j * k - i * r); col[2] = 1.f - s * (i * i + j * j);
  }
}

__device__ __forceinline__ int argmin3(float a, float b, float c) {
  // first minimum wins, as torch.min(dim) does on ties
  int m = 0;
  float v = a;
  if (b < v) { v = b; m = 1; }
  if (c < v) { m = 2; }
  return m;
}

// One row of input_all_map and (BACKWARD) of its gradient: `m` = index of the smallest scaling axis, `q` the rotation as
// the renderer sees it (activated).  out5 / g5 point at the row's five floats.  POSE: the camera side of the row's
// gradient is added to pose[0..5]: dL/drho = g4 n_cam, and the torque n_cam x dL/dn_cam + p_cam x dL/dp_cam, in which
// the two terms of d = n_cam . p_cam cancel (d does not change when the camera turns), leaving n_cam x g5[0..2].
template <bool BACKWARD, bool POSE = false>
__device__ __forceinline__ void all_map_row(const View& V, const float px, const float py, const float pz, const int m,
                                            const float4 q, float* __restrict__ out5, const float* __restrict__ g5,
                                            float (&dxyz)[3], float4& drot, float* pose = nullptr) {
  const float qq = q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w;
  const float s = 2.0f / qq;
  float col[3];
  rot_column(q, m, s, col);
  const float facing = col[0] * (V.cam[0] - px) + col[1] * (V.cam[1] - py) + col[2] * (V.cam[2] - pz);
  const float flip = facing < 0.0f ? -1.0f : 1.0f;
  const float nx = flip * col[0], ny = flip * col[1], nz = flip * col[2];
  float ln[3], pc[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    ln[j] = nx * V.v[j] + ny * V.v[4 + j] + nz * V.v[8 + j];
    pc[j] = px * V.v[j] + py * V.v[4 + j] + pz * V.v[8 + j] + V.v[12 + j];
  }
  const float d = ln[0] * pc[0] + ln[1] * pc[1] + ln[2] * pc[2];
  if (!BACKWARD) {
    out5[0] = ln[0]; out5[1] = ln[1]; out5[2] = ln[2]; out5[3] = 1.0f; out5[4] = fabsf(d);
    return;
  }
  const float sg = d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f);  // d|d|/dd, 0 at 0 as torch.abs
  const float g4 = g5[4] * sg;
  float dln[3], dpc[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    dln[j] = g5[j] + g4 * pc[j];
    dpc[j] = g4 * ln[j];
  }
  if constexpr (POSE) {
    pose[0] += dpc[0]; pose[1] += dpc[1]; pose[2] += dpc[2];
    pose[3] += ln[1] * g5[2] - ln[2] * g5[1];
    pose[4] += ln[2] * g5[0] - ln[0] * g5[2];
    pose[5] += ln[0] * g5[1] - ln[1] * g5[0];
  }
  float dn[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    dn[i] = dln[0] * V.v[4 * i] + dln[1] * V.v[4 * i + 1] + dln[2] * V.v[4 * i + 2];
    dxyz[i] = dpc[0] * V.v[4 * i] + dpc[1] * V.v[4 * i + 1] + dpc[2] * V.v[4 * i + 2];
  }
  // column = e_m + s * A_m(q):  dL/dq = s * J_A^T G + (G . A_m) ds/dq,  ds/dq = -s^2 q
  const float G0 = flip * dn[0], G1 = flip * dn[1], G2 = flip * dn[2];
  const float r = q.x, i = q.y, j = q.z, k = q.w;
  float dr, di, dj, dk, GA;
  if (m == 0) {
    // A = [-(j^2+k^2), ij+kr, ik-jr]
    GA = G0 * (-(j * j + k * k)) + G1 * (i * j + k * r) + G2 * (i * k - j * r);
    dr = G1 * k - G2 * j;
    di = G1 * j + G2 * k;
    dj = -2.f * j * G0 + G1 * i - G2 * r;
    dk = -2.f * k * G0 + G1 * r + G2 * i;
  } else if (m == 1) {
    // A = [ij-kr, -(i^2+k^2), jk+ir]
    GA = G0 * (i * j - k * r) + G1 * (-(i * i + k * k)) + G2 * (j * k + i * r);
    dr = -G0 * k + G2 * i;
    di = G0 * j - 2.f * i * G1 + G2 * r;
    dj = G0 * i + G2 * k;
    dk = -G0 * r - 2.f * k * G1 + G2 * j;
  } else {
    // A = [ik+jr, jk-ir, -(i^2+j^2)]
    GA = G0 * (i * k + j * r) + G1 * (j * k - i * r) + G2 * (-(i * i + j * j));
    dr = G0 * j - G1 * i;
    di = G0 * k - G1 * r - 2.f * i * G2;
    dj = G0 * r + G1 * k - 2.f * j * G2;
    dk = G0 * i + G1 * j;
  }
  const float c = -s * s * GA;
  drot = make_float4(s * dr + c * r, s * di + c * i, s * dj + c * j, s * dk + c * k);
}

template <bool BACKWARD>
__global__ void __launch_bounds__(256)
all_map_kernel(const float* __restrict__ xyz, const float* __restrict__ scaling, const float* __restrict__ rotation,
               const float* __restrict__ viewmatrix, const float* __restrict__ campos, const int64_t N,
               float* __restrict__ out, const float* __restrict__ dL_dall_map, float* __restrict__ dL_dxyz,
               float* __restrict__ dL_drot) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  // the 19 camera floats are read through the pointers (uniform, L1-resident): no host round trip
  View V;
#pragma unroll
  for (int i = 0; i < 16; ++i) V.v[i] = __ldg(viewmatrix + i);
#pragma unroll
  for (int i = 0; i < 3; ++i) V.cam[i] = __ldg(campos + i);
  const float px = xyz[3 * n], py = xyz[3 * n + 1], pz = xyz[3 * n + 2];
  const int m = argmin3(scaling[3 * n], scaling[3 * n + 1], scaling[3 * n + 2]);
  const float4 q = __ldg(reinterpret_cast<const float4*>(rotation) + n);
  float dxyz[3];
  float4 drot;
  all_map_row<BACKWARD>(V, px, py, pz, m, q, BACKWARD ? nullptr : out + 5 * n, BACKWARD ? dL_dall_map + 5 * n : nullptr,
                        dxyz, drot);
  if (BACKWARD) {
    dL_dxyz[3 * n] = dxyz[0]; dL_dxyz[3 * n + 1] = dxyz[1]; dL_dxyz[3 * n + 2] = dxyz[2];
    reinterpret_cast<float4*>(dL_drot)[n] = drot;
  }
}

// ------------------------------------------------------------------------------------------------
// Parameter activations.
__global__ void __launch_bounds__(256)
activate_kernel(const float* __restrict__ rs, const float* __restrict__ rr, const float* __restrict__ ro, const int64_t N,
                float* __restrict__ s, float* __restrict__ r, float* __restrict__ o) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
#pragma unroll
  for (int i = 0; i < 3; ++i) s[3 * n + i] = expf(rs[3 * n + i]);
  o[n] = 1.0f / (1.0f + expf(-ro[n]));
  const float4 q = __ldg(reinterpret_cast<const float4*>(rr) + n);
  const float inv = 1.0f / fmaxf(sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w), 1e-12f);
  reinterpret_cast<float4*>(r)[n] = make_float4(q.x * inv, q.y * inv, q.z * inv, q.w * inv);
}

// per-Gaussian part: xyz (pass-through), opacity, scaling, rotation
__global__ void __launch_bounds__(256)
activate_bwd_kernel(const float* __restrict__ rs, const float* __restrict__ rr, const float* __restrict__ ro,
                    const int64_t N, const float* __restrict__ g_xyz, const float* __restrict__ g_o,
                    const float* __restrict__ g_s, const float* __restrict__ g_r, const float beta,
                    float* __restrict__ d_xyz, float* __restrict__ d_o, float* __restrict__ d_s,
                    float* __restrict__ d_r) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const bool acc = beta != 0.0f;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const float gx = g_xyz ? g_xyz[3 * n + i] : 0.f;
    d_xyz[3 * n + i] = acc ? d_xyz[3 * n + i] + gx : gx;
    const float gs = g_s ? g_s[3 * n + i] * expf(rs[3 * n + i]) : 0.f;
    d_s[3 * n + i] = acc ? d_s[3 * n + i] + gs : gs;
  }
  {
    const float sg = 1.0f / (1.0f + expf(-ro[n]));
    const float go = g_o ? g_o[n] * sg * (1.0f - sg) : 0.f;
    d_o[n] = acc ? d_o[n] + go : go;
  }
  {
    const float4 q = __ldg(reinterpret_cast<const float4*>(rr) + n);
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    if (g_r) g = __ldg(reinterpret_cast<const float4*>(g_r) + n);
    const float len = sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w);
    float4 d;
    if (len > 1e-12f) {
      const float inv = 1.0f / len;
      const float4 y = make_float4(q.x * inv, q.y * inv, q.z * inv, q.w * inv);
      const float t = y.x * g.x + y.y * g.y + y.z * g.z + y.w * g.w;
      d = make_float4((g.x - y.x * t) * inv, (g.y - y.y * t) * inv, (g.z - y.z * t) * inv, (g.w - y.w * t) * inv);
    } else {  // clamp_min saturated: the denominator is the constant eps
      d = make_float4(g.x * 1e12f, g.y * 1e12f, g.z * 1e12f, g.w * 1e12f);
    }
    float4* dst = reinterpret_cast<float4*>(d_r) + n;
    if (acc) {
      const float4 p = *dst;
      d = make_float4(p.x + d.x, p.y + d.y, p.z + d.z, p.w + d.w);
    }
    *dst = d;
  }
}

// Everything between the rasterizer's backward and the raw-parameter gradient arena of a training view, in ONE pass over
// the rows the view rendered: all_map backward (its xyz / rotation gradients join the rasterizer's), the scale
// regulariser's gradient (g_s_extra * *extra_scale), the activation chain rule (exp / sigmoid / normalize) and the
// accumulation dst = beta * dst + grad.  Rows with radii <= 0 carry no gradient in any of these terms: they are
// skipped (beta = 1) or zero-filled (beta = 0) without reading their gradient rows — which the rasterizer's backward
// therefore need not write (HG_BWD_SKIP_CULLED_ROWS).  Replaces all_map_kernel<true>, two adds, one addcmul and
// activate_bwd_kernel (five passes over N rows) of the executor.
template <bool POSE>
__device__ __forceinline__ void
prologue_bwd_row(const int64_t n, const float* __restrict__ rs, const float* __restrict__ rr, const float* __restrict__ ro,
                 const float* __restrict__ xyz, const int* __restrict__ radii,
                 const float* __restrict__ viewmatrix, const float* __restrict__ campos,
                 const float* __restrict__ g_xyz, const float* __restrict__ g_o, const float* __restrict__ g_s,
                 const float* __restrict__ g_r, const float* __restrict__ g_all_map,
                 const float* __restrict__ g_s_extra, const float* __restrict__ extra_scale, const float beta,
                 float* __restrict__ d_xyz, float* __restrict__ d_o, float* __restrict__ d_s,
                 float* __restrict__ d_r, float* pose) {
  const bool acc = beta != 0.0f;
  float4* const dst_r = reinterpret_cast<float4*>(d_r) + n;
  if (radii && radii[n] <= 0) {
    if (!acc) {
      d_xyz[3 * n] = d_xyz[3 * n + 1] = d_xyz[3 * n + 2] = 0.f;
      d_s[3 * n] = d_s[3 * n + 1] = d_s[3 * n + 2] = 0.f;
      d_o[n] = 0.f;
      *dst_r = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    return;
  }
  const float4 q = __ldg(reinterpret_cast<const float4*>(rr) + n);
  const float len = sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w);
  const float inv = 1.0f / fmaxf(len, 1e-12f);
  const float4 y = make_float4(q.x * inv, q.y * inv, q.z * inv, q.w * inv);  // the activated rotation
  const float r0 = rs[3 * n], r1 = rs[3 * n + 1], r2 = rs[3 * n + 2];
  const float e[3] = {expf(r0), expf(r1), expf(r2)};                         // the activated scaling
  float gx[3] = {0.f, 0.f, 0.f};
  float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
  if (g_xyz) { gx[0] = g_xyz[3 * n]; gx[1] = g_xyz[3 * n + 1]; gx[2] = g_xyz[3 * n + 2]; }
  if (g_r) g = __ldg(reinterpret_cast<const float4*>(g_r) + n);
  if (g_all_map) {
    View V;
#pragma unroll
    for (int i = 0; i < 16; ++i) V.v[i] = __ldg(viewmatrix + i);
#pragma unroll
    for (int i = 0; i < 3; ++i) V.cam[i] = __ldg(campos + i);
    float dxyz[3];
    float4 drot;
    all_map_row<true, POSE>(V, xyz[3 * n], xyz[3 * n + 1], xyz[3 * n + 2], argmin3(e[0], e[1], e[2]), y, nullptr,
                            g_all_map + 5 * n, dxyz, drot, pose);
    gx[0] += dxyz[0]; gx[1] += dxyz[1]; gx[2] += dxyz[2];
    g = make_float4(g.x + drot.x, g.y + drot.y, g.z + drot.z, g.w + drot.w);
  }
  const float xs = (g_s_extra && extra_scale) ? __ldg(extra_scale) : 1.0f;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    d_xyz[3 * n + i] = acc ? d_xyz[3 * n + i] + gx[i] : gx[i];
    float gs = g_s ? g_s[3 * n + i] : 0.f;
    if (g_s_extra) gs = fmaf(g_s_extra[3 * n + i], xs, gs);  // torch.addcmul(g_s, extra, scale)
    gs *= e[i];
    d_s[3 * n + i] = acc ? d_s[3 * n + i] + gs : gs;
  }
  {
    const float sg = 1.0f / (1.0f + expf(-ro[n]));
    const float go = g_o ? g_o[n] * sg * (1.0f - sg) : 0.f;
    d_o[n] = acc ? d_o[n] + go : go;
  }
  {
    float4 d;
    if (len > 1e-12f) {
      const float t = y.x * g.x + y.y * g.y + y.z * g.z + y.w * g.w;
      d = make_float4((g.x - y.x * t) * inv, (g.y - y.y * t) * inv, (g.z - y.z * t) * inv, (g.w - y.w * t) * inv);
    } else {  // clamp_min saturated: the denominator is the constant eps
      d = make_float4(g.x * 1e12f, g.y * 1e12f, g.z * 1e12f, g.w * 1e12f);
    }
    if (acc) {
      const float4 p = *dst_r;
      d = make_float4(p.x + d.x, p.y + d.y, p.z + d.z, p.w + d.w);
    }
    *dst_r = d;
  }
}

// POSE: the rows' camera-side all_map gradients (all_map_row) summed over the CTA in double in a fixed order (warp
// butterflies, then the 8 warps in index order) -> pose_partial[blockIdx.x][0..5]; the grid depends on N only.
template <bool POSE>
__global__ void __launch_bounds__(kPosePrologueRows)
prologue_bwd_kernel(const float* __restrict__ rs, const float* __restrict__ rr, const float* __restrict__ ro,
                    const float* __restrict__ xyz, const int64_t N, const int* __restrict__ radii,
                    const float* __restrict__ viewmatrix, const float* __restrict__ campos,
                    const float* __restrict__ g_xyz, const float* __restrict__ g_o, const float* __restrict__ g_s,
                    const float* __restrict__ g_r, const float* __restrict__ g_all_map,
                    const float* __restrict__ g_s_extra, const float* __restrict__ extra_scale, const float beta,
                    float* __restrict__ d_xyz, float* __restrict__ d_o, float* __restrict__ d_s,
                    float* __restrict__ d_r, double* __restrict__ pose_partial) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float pose[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (n < N)
    prologue_bwd_row<POSE>(n, rs, rr, ro, xyz, radii, viewmatrix, campos, g_xyz, g_o, g_s, g_r, g_all_map, g_s_extra,
                           extra_scale, beta, d_xyz, d_o, d_s, d_r, pose);
  if constexpr (POSE) {
    __shared__ double s_pose[kPosePrologueRows / 32][6];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const double w = warp_sum_double((double)pose[k]);
      if (lane == 0) s_pose[warp][k] = w;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
      double a = 0.0;
#pragma unroll
      for (int w = 0; w < kPosePrologueRows / 32; ++w) a += s_pose[w][threadIdx.x];
      pose_partial[(size_t)blockIdx.x * kPosePartialStride + threadIdx.x] = a;
    }
  }
}

// features: dst = beta * dst + g, float4 grid-stride
__global__ void __launch_bounds__(256)
axpby4_kernel(const float4* __restrict__ g, const int64_t n4, const float beta, float4* __restrict__ dst) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 v = g ? __ldg(g + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (beta != 0.0f) {
      const float4 p = dst[i];
      v = make_float4(p.x + v.x, p.y + v.y, p.z + v.z, p.w + v.w);
    }
    dst[i] = v;
  }
}

// ------------------------------------------------------------------------------------------------
// Depth -> normal.
struct Unproj {
  float i00, i20, i11, i21;  // entries of K^-1: X = (u z) i00 + z i20, Y = (v z) i11 + z i21
  float wm1, hm1;            // W - 1, H - 1 (the reference builds pixel coords as arange/(W-1)*(W-1))
};

__device__ __forceinline__ float3 unproject(const Unproj& U, int x, int y, float z) {
  const float u = ((float)x / U.wm1) * U.wm1, v = ((float)y / U.hm1) * U.hm1;
  return make_float3((u * z) * U.i00 + z * U.i20, (v * z) * U.i11 + z * U.i21, z);
}
__device__ __forceinline__ float3 sub3(float3 a, float3 b) { return make_float3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ float3 cross3(float3 a, float3 b) {
  return make_float3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__device__ __forceinline__ float dot3(float3 a, float3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }

constexpr float kNormEps = 1e-12f;  // torch.nn.functional.normalize eps

// Unit normal of the centre (y, x) from the four neighbouring depths; also returns a, b, |n|.
__device__ __forceinline__ float3 centre_normal(const Unproj& U, int x, int y, float zl, float zr, float zt, float zb,
                                                float3& a, float3& b, float& len) {
  a = sub3(unproject(U, x + 1, y, zr), unproject(U, x - 1, y, zl));  // left -> right
  b = sub3(unproject(U, x, y - 1, zt), unproject(U, x, y + 1, zb));  // bottom -> top
  const float3 n = cross3(a, b);
  len = sqrtf(dot3(n, n));
  const float inv = 1.0f / fmaxf(len, kNormEps);
  return make_float3(n.x * inv, n.y * inv, n.z * inv);
}

__global__ void __launch_bounds__(256)
depth_normal_kernel(const float* __restrict__ depth, const float* __restrict__ alpha, const int H, const int W,
                    const Unproj U, float* __restrict__ out) {
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (x >= W || y >= H) return;
  const size_t HW = (size_t)H * W, p = (size_t)y * W + x;
  float3 n = make_float3(0.f, 0.f, 0.f);
  if (x >= 1 && x <= W - 2 && y >= 1 && y <= H - 2) {
    float3 a, b;
    float len;
    n = centre_normal(U, x, y, __ldg(depth + p - 1), __ldg(depth + p + 1), __ldg(depth + p - W), __ldg(depth + p + W),
                      a, b, len);
  }
  const float al = alpha ? __ldg(alpha + p) : 1.0f;
  out[p] = n.x * al;
  out[HW + p] = n.y * al;
  out[2 * HW + p] = n.z * al;
}

// Forward value of the fused loss: per-pixel  iw * sum_c |dn_c * alpha - rn_c|, block partial sums.
__global__ void __launch_bounds__(256)
normal_loss_fwd_kernel(const float* __restrict__ depth, const float* __restrict__ all_map,
                       const float* __restrict__ iw, const int H, const int W, const Unproj U,
                       double* __restrict__ partial) {
  __shared__ float red[8];
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  float term = 0.f;
  if (x < W && y < H) {
    const size_t HW = (size_t)H * W, p = (size_t)y * W + x;
    float3 n = make_float3(0.f, 0.f, 0.f);
    if (x >= 1 && x <= W - 2 && y >= 1 && y <= H - 2) {
      float3 a, b;
      float len;
      n = centre_normal(U, x, y, __ldg(depth + p - 1), __ldg(depth + p + 1), __ldg(depth + p - W),
                        __ldg(depth + p + W), a, b, len);
    }
    const float al = __ldg(all_map + 3 * HW + p);
    const float e = fabsf(n.x * al - __ldg(all_map + p)) + fabsf(n.y * al - __ldg(all_map + HW + p)) +
                    fabsf(n.z * al - __ldg(all_map + 2 * HW + p));
    term = (iw ? __ldg(iw + p) : 1.0f) * e;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) term += __shfl_xor_sync(0xffffffffu, term, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = term;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += red[i];
    partial[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = (double)s;
  }
}

__global__ void __launch_bounds__(1024)
normal_loss_finalize_kernel(const double* __restrict__ partial, int n, double scale, float* __restrict__ out) {
  __shared__ double sm[32];
  const double s = cta_sum_strided(partial, n, 1, 0, sm);
  if (threadIdx.x == 0) out[0] = (float)(s * scale);
}

// Backward w.r.t. the depth: gather form over a 32x8 tile.  Stage 1 evaluates, for every centre of the tile
// plus a 1-pixel halo, the gradients G1 = dL/d(P_right - P_left) and G2 = dL/d(P_top - P_bottom); stage 2 lets
// every pixel collect the four centres it is a neighbour of.
//   FUSED = false: upstream gradient dL/ddepth_normal [3,H,W] is read from memory;
//   FUSED = true : it is derived from the loss (coef * iw * sign(dn*alpha - rn) * alpha) and dL/dall_map is written.
constexpr int kTX = 32, kTY = 8;
template <bool FUSED>
__global__ void __launch_bounds__(kTX * kTY)
depth_normal_bwd_kernel(const float* __restrict__ depth, const float* __restrict__ alpha,
                        const float* __restrict__ dL_dnormal, const float* __restrict__ all_map,
                        const float* __restrict__ iw, const float coef, const int H, const int W, const Unproj U,
                        float* __restrict__ dL_ddepth, float* __restrict__ dL_dall_map) {
  __shared__ float sz[kTY + 4][kTX + 4];
  __shared__ float sg[6][kTY + 2][kTX + 2 + 1];
  const int x0 = blockIdx.x * kTX, y0 = blockIdx.y * kTY;
  const int tid = threadIdx.x;
  const size_t HW = (size_t)H * W;
  for (int i = tid; i < (kTY + 4) * (kTX + 4); i += kTX * kTY) {
    const int r = i / (kTX + 4), c = i - r * (kTX + 4);
    const int y = y0 + r - 2, x = x0 + c - 2;
    sz[r][c] = (y >= 0 && y < H && x >= 0 && x < W) ? __ldg(depth + (size_t)y * W + x) : 0.f;
  }
  __syncthreads();
  for (int i = tid; i < (kTY + 2) * (kTX + 2); i += kTX * kTY) {
    const int r = i / (kTX + 2), c = i - r * (kTX + 2);
    const int y = y0 + r - 1, x = x0 + c - 1;
    float3 G1 = make_float3(0.f, 0.f, 0.f), G2 = G1;
    const bool in_img = y >= 0 && y < H && x >= 0 && x < W;
    const bool centre = x >= 1 && x <= W - 2 && y >= 1 && y <= H - 2;
    const size_t p = in_img ? (size_t)y * W + x : 0;
    float3 g = make_float3(0.f, 0.f, 0.f);
    float3 nh = g, a = g, b = g;
    float len = 0.f;
    if (centre) nh = centre_normal(U, x, y, sz[r + 1][c], sz[r + 1][c + 2], sz[r][c + 1], sz[r + 2][c + 1], a, b, len);
    if (in_img) {
      if (FUSED) {
        const float al = __ldg(all_map + 3 * HW + p);
        const float w = coef * (iw ? __ldg(iw + p) : 1.0f);
        const float e0 = nh.x * al - __ldg(all_map + p), e1 = nh.y * al - __ldg(all_map + HW + p),
                    e2 = nh.z * al - __ldg(all_map + 2 * HW + p);
        const float s0 = e0 > 0.f ? w : (e0 < 0.f ? -w : 0.f), s1 = e1 > 0.f ? w : (e1 < 0.f ? -w : 0.f),
                    s2 = e2 > 0.f ? w : (e2 < 0.f ? -w : 0.f);
        g = make_float3(s0 * al, s1 * al, s2 * al);
        // the pixel belongs to this CTA's interior exactly once: write dL/drendered_normal there
        if (r >= 1 && r <= kTY && c >= 1 && c <= kTX && dL_dall_map) {
          dL_dall_map[p] = -s0;
          dL_dall_map[HW + p] = -s1;
          dL_dall_map[2 * HW + p] = -s2;
          dL_dall_map[3 * HW + p] = 0.f;
          dL_dall_map[4 * HW + p] = 0.f;
        }
      } else {
        const float al = alpha ? __ldg(alpha + p) : 1.0f;
        g = make_float3(__ldg(dL_dnormal + p) * al, __ldg(dL_dnormal + HW + p) * al, __ldg(dL_dnormal + 2 * HW + p) * al);
      }
    }
    if (centre) {
      float3 dn;
      if (len > kNormEps) {
        const float t = dot3(nh, g), inv = 1.0f / len;
        dn = make_float3((g.x - nh.x * t) * inv, (g.y - nh.y * t) * inv, (g.z - nh.z * t) * inv);
      } else {
        dn = make_float3(g.x / kNormEps, g.y / kNormEps, g.z / kNormEps);
      }
      G1 = cross3(b, dn);  // n = a x b  ->  dL/da = b x dn
      G2 = cross3(dn, a);  //                dL/db = dn x a
    }
    sg[0][r][c] = G1.x; sg[1][r][c] = G1.y; sg[2][r][c] = G1.z;
    sg[3][r][c] = G2.x; sg[4][r][c] = G2.y; sg[5][r][c] = G2.z;
  }
  __syncthreads();
  const int lx = tid & 31, ly = tid >> 5;
  const int x = x0 + lx, y = y0 + ly;
  if (x >= W || y >= H) return;
  const int r = ly + 1, c = lx + 1;
  // p is the right neighbour of centre (y, x-1), the left one of (y, x+1), the top one of (y+1, x), the bottom
  // one of (y-1, x)
  const float dPx = sg[0][r][c - 1] - sg[0][r][c + 1] + sg[3][r + 1][c] - sg[3][r - 1][c];
  const float dPy = sg[1][r][c - 1] - sg[1][r][c + 1] + sg[4][r + 1][c] - sg[4][r - 1][c];
  const float dPz = sg[2][r][c - 1] - sg[2][r][c + 1] + sg[5][r + 1][c] - sg[5][r - 1][c];
  const float u = ((float)x / U.wm1) * U.wm1, v = ((float)y / U.hm1) * U.hm1;
  dL_ddepth[(size_t)y * W + x] = dPx * (u * U.i00 + U.i20) + dPy * (v * U.i11 + U.i21) + dPz;
}

int make_unproj(hg_intrinsics K, int H, int W, Unproj* U) {
  if (H < 3 || W < 3 || !(K.fx != 0.f) || !(K.fy != 0.f)) {
    set_error("depth normal: needs H, W >= 3 and non-zero focal lengths");
    return HG_ERR_INVALID_ARG;
  }
  U->i00 = (float)(1.0 / (double)K.fx);
  U->i20 = (float)(-(double)K.cx / (double)K.fx);
  U->i11 = (float)(1.0 / (double)K.fy);
  U->i21 = (float)(-(double)K.cy / (double)K.fy);
  U->wm1 = (float)(W - 1);
  U->hm1 = (float)(H - 1);
  return HG_OK;
}

// ------------------------------------------------------------------------------------------------
// Adam.
struct AdamArgs {
  float beta1, beta2, one_m_b1, one_m_b2, step_size, inv_bc2_sqrt, eps, grad_scale;
  float step_size_head;  // step size of the first `head_cols` columns of every row (the SH DC term)
  int head_cols;
};

__device__ __forceinline__ void adam_update(float& p, float g, float& m, float& v, const AdamArgs& a, float step_size) {
  g *= a.grad_scale;
  m = m * a.beta1 + a.one_m_b1 * g;             // exp_avg.mul_(beta1).add_(grad, alpha=1-beta1)
  v = v * a.beta2 + a.one_m_b2 * (g * g);       // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1-beta2)
  const float denom = sqrtf(v) * a.inv_bc2_sqrt + a.eps;
  p = p - step_size * (m / denom);              // param.addcdiv_(exp_avg, denom, value=-step_size)
}
__device__ __forceinline__ float adam_step_of(const AdamArgs& a, int col) {
  return col < a.head_cols ? a.step_size_head : a.step_size;
}

__global__ void __launch_bounds__(256)
adam_dense_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                  const int64_t n, const int row_width, const uint8_t* __restrict__ visible, const AdamArgs a) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int64_t row = i / row_width;
    if (visible && !visible[row]) continue;
    float pp = p[i], mm = m[i], vv = v[i];
    adam_update(pp, __ldg(g + i), mm, vv, a, adam_step_of(a, (int)(i - row * row_width)));
    p[i] = pp; m[i] = mm; v[i] = vv;
  }
}

__global__ void __launch_bounds__(256)
adam_dense4_kernel(float4* __restrict__ p, const float4* __restrict__ g, float4* __restrict__ m,
                   float4* __restrict__ v, const int64_t n4, const AdamArgs a) {  // head_cols == 0 only
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 pp = p[i], mm = m[i], vv = v[i];
    const float4 gg = __ldg(g + i);
    adam_update(pp.x, gg.x, mm.x, vv.x, a, a.step_size);
    adam_update(pp.y, gg.y, mm.y, vv.y, a, a.step_size);
    adam_update(pp.z, gg.z, mm.z, vv.z, a, a.step_size);
    adam_update(pp.w, gg.w, mm.w, vv.w, a, a.step_size);
    p[i] = pp; m[i] = mm; v[i] = vv;
  }
}

// row_width % 4 == 0: whole float4s belong to one row, masked rows cost no memory traffic
__global__ void __launch_bounds__(256)
adam_masked4_kernel(float4* __restrict__ p, const float4* __restrict__ g, float4* __restrict__ m,
                    float4* __restrict__ v, const int64_t n4, const int row_width4,
                    const uint8_t* __restrict__ visible, const AdamArgs a) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const int64_t row = i / row_width4;
    if (visible && !visible[row]) continue;
    const int c0 = 4 * (int)(i - row * row_width4);
    float4 pp = p[i], mm = m[i], vv = v[i];
    const float4 gg = __ldg(g + i);
    adam_update(pp.x, gg.x, mm.x, vv.x, a, adam_step_of(a, c0));
    adam_update(pp.y, gg.y, mm.y, vv.y, a, adam_step_of(a, c0 + 1));
    adam_update(pp.z, gg.z, mm.z, vv.z, a, adam_step_of(a, c0 + 2));
    adam_update(pp.w, gg.w, mm.w, vv.w, a, adam_step_of(a, c0 + 3));
    p[i] = pp; m[i] = mm; v[i] = vv;
  }
}

// add_densification_stats (scene/gaussian_model.py:763-765) + the max_radii2D update of the training loop
__global__ void __launch_bounds__(256)
densification_stats_kernel(const float* __restrict__ grad_means2D, const int* __restrict__ radii, const int64_t N,
                           float* __restrict__ accum, float* __restrict__ denom, float* __restrict__ max_radii2D) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const int r = radii[n];
  if (r <= 0) return;
  const float gx = grad_means2D[3 * n], gy = grad_means2D[3 * n + 1];
  accum[n] = fmaxf(sqrtf(gx * gx + gy * gy), accum[n]);
  denom[n] += 1.0f;
  if (max_radii2D) max_radii2D[n] = fmaxf(max_radii2D[n], (float)r);
}

__global__ void __launch_bounds__(256)
adam_indexed_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                    const int64_t n_rows, const int row_width, const int64_t* __restrict__ idx, const int64_t n_idx,
                    const AdamArgs a) {
  const int64_t total = n_idx * row_width;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
    const int64_t e = t / row_width;
    int64_t row = idx[e];
    if (row < 0) row += n_rows;  // negative indices wrap, as torch indexing does
    if (row < 0 || row >= n_rows) continue;
    const int col = (int)(t - e * row_width);
    const int64_t i = row * row_width + col;
    float pp = p[i], mm = m[i], vv = v[i];
    adam_update(pp, __ldg(g + i), mm, vv, a, adam_step_of(a, col));
    p[i] = pp; m[i] = mm; v[i] = vv;
  }
}

}  // namespace
}  // namespace hg

using namespace hg;

extern "C" {

int hg_geometry_all_map(const float* xyz, const float* scaling, const float* rotation, const float* viewmatrix,
                        const float* campos, int64_t N, float* out_all_map, void* st_) {
  if (N < 0 || (N > 0 && (!xyz || !scaling || !rotation || !viewmatrix || !campos || !out_all_map))) {
    set_error("hg_geometry_all_map: bad argument");
    return HG_ERR_INVALID_ARG;
  }
  if (N == 0) return HG_OK;
  if (((uintptr_t)rotation & 15) != 0) {
    set_error("hg_geometry_all_map: rotation must be 16-byte aligned");
    return HG_ERR_INVALID_ARG;
  }
  cudaStream_t st = (cudaStream_t)st_;
  all_map_kernel<false><<<(unsigned)((N + 255) / 256), 256, 0, st>>>(xyz, scaling, rotation, viewmatrix, campos, N,
                                                                      out_all_map, nullptr, nullptr, nullptr);
  HG_POST_LAUNCH(false, st, "geometry_all_map");
  return HG_OK;
}

int hg_geometry_all_map_backward(const float* xyz, const float* scaling, const float* rotation,
                                 const float* viewmatrix, const float* campos, int64_t N, const float* dL_dall_map,
                                 float* dL_dxyz, float* dL_drotation, void* st_) {
  if (N < 0 || (N > 0 && (!xyz || !scaling || !rotation || !viewmatrix || !campos || !dL_dall_map || !dL_dxyz ||
                          !dL_drotation))) {
    set_error("hg_geometry_all_map_backward: bad argument");
    return HG_ERR_INVALID_ARG;
  }
  if (N == 0) return HG_OK;
  if ((((uintptr_t)rotation | (uintptr_t)dL_drotation) & 15) != 0) {
    set_error("hg_geometry_all_map_backward: rotation pointers must be 16-byte aligned");
    return HG_ERR_INVALID_ARG;
  }
  cudaStream_t st = (cudaStream_t)st_;
  all_map_kernel<true><<<(unsigned)((N + 255) / 256), 256, 0, st>>>(xyz, scaling, rotation, viewmatrix, campos, N,
                                                                     nullptr, dL_dall_map, dL_dxyz, dL_drotation);
  HG_POST_LAUNCH(false, st, "geometry_all_map_bwd");
  return HG_OK;
}

int hg_activate_params(const float* raw_scaling, const float* raw_rotation, const float* raw_opacity, int64_t N,
                       float* scaling, float* rotation, float* opacity, void* st_) {
  if (N < 0 || (N > 0 && (!raw_scaling || !raw_rotation || !raw_opacity || !scaling || !rotation || !opacity)) ||
      (((uintptr_t)raw_rotation | (uintptr_t)rotation) & 15) != 0) {
    set_error("hg_activate_params: bad argument (rotation arrays must be 16-byte aligned)");
    return HG_ERR_INVALID_ARG;
  }
  if (N == 0) return HG_OK;
  cudaStream_t st = (cudaStream_t)st_;
  activate_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(raw_scaling, raw_rotation, raw_opacity, N, scaling, rotation,
                                                                 opacity);
  HG_POST_LAUNCH(false, st, "activate_params");
  return HG_OK;
}

int hg_activate_params_backward(const float* raw_scaling, const float* raw_rotation, const float* raw_opacity, int64_t N,
                                int32_t F, const float* g_xyz, const float* g_features, const float* g_opacity,
                                const float* g_scaling, const float* g_rotation, float beta, float* d_xyz,
                                float* d_features, float* d_opacity, float* d_scaling, float* d_rotation, void* st_) {
  if (N < 0 || F < 0 || !(beta == 0.0f || beta == 1.0f) ||
      (N > 0 && (!raw_scaling || !raw_rotation || !raw_opacity || !d_xyz || !d_opacity || !d_scaling || !d_rotation ||
                 (F > 0 && !d_features))) ||
      (((uintptr_t)raw_rotation | (uintptr_t)g_rotation | (uintptr_t)d_rotation | (uintptr_t)g_features |
        (uintptr_t)d_features) & 15) != 0 || ((N * (int64_t)F) & 3) != 0) {
    set_error("hg_activate_params_backward: bad argument (rotation / feature arrays must be 16-byte aligned, N*F % 4 == 0)");
    return HG_ERR_INVALID_ARG;
  }
  if (N == 0) return HG_OK;
  cudaStream_t st = (cudaStream_t)st_;
  activate_bwd_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(raw_scaling, raw_rotation, raw_opacity, N, g_xyz,
                                                                     g_opacity, g_scaling, g_rotation, beta, d_xyz,
                                                                     d_opacity, d_scaling, d_rotation);
  HG_POST_LAUNCH(false, st, "activate_params_bwd");
  if (F > 0 && g_features) {  // NULL: the feature gradient already sits in d_features (rasterizer SH sink)
    axpby4_kernel<<<148 * 8, 256, 0, st>>>((const float4*)g_features, N * (int64_t)F / 4, beta, (float4*)d_features);
    HG_POST_LAUNCH(false, st, "features_grad_accumulate");
  }
  return HG_OK;
}

}  // extern "C"

// hg_prologue_backward and hg_prologue_backward_pose: pose_workspace == NULL is the plain prologue backward.
static int prologue_backward_impl(const float* raw_scaling, const float* raw_rotation, const float* raw_opacity,
                                  const float* xyz, int64_t N, int32_t F, const int32_t* radii, const float* viewmatrix,
                                  const float* campos, const float* g_xyz, const float* g_features,
                                  const float* g_opacity, const float* g_scaling, const float* g_rotation,
                                  const float* g_all_map, const float* g_scaling_extra, const float* extra_scale,
                                  float beta, float* d_xyz, float* d_features, float* d_opacity, float* d_scaling,
                                  float* d_rotation, void* pose_workspace, void* st_) {
  if (pose_workspace && (N > INT32_MAX || (reinterpret_cast<uintptr_t>(pose_workspace) & 15))) {
    set_error("hg_prologue_backward_pose: bad argument (N must fit int32, the workspace must be 16-byte aligned)");
    return HG_ERR_INVALID_ARG;
  }
  if (N < 0 || F < 0 || !(beta == 0.0f || beta == 1.0f) ||
      (N > 0 && (!raw_scaling || !raw_rotation || !raw_opacity || !d_xyz || !d_opacity || !d_scaling || !d_rotation ||
                 (g_all_map && (!xyz || !viewmatrix || !campos)) || (F > 0 && g_features && !d_features))) ||
      (((uintptr_t)raw_rotation | (uintptr_t)g_rotation | (uintptr_t)d_rotation | (uintptr_t)g_features |
        (uintptr_t)d_features) & 15) != 0 || (g_features && ((N * (int64_t)F) & 3) != 0)) {
    set_error("hg_prologue_backward: bad argument (rotation / feature arrays must be 16-byte aligned, N*F % 4 == 0)");
    return HG_ERR_INVALID_ARG;
  }
  if (N == 0) return HG_OK;
  cudaStream_t st = (cudaStream_t)st_;
  double* const pose_partial = static_cast<double*>(pose_workspace);
  auto kernel = pose_partial ? prologue_bwd_kernel<true> : prologue_bwd_kernel<false>;
  kernel<<<(unsigned)((N + kPosePrologueRows - 1) / kPosePrologueRows), kPosePrologueRows, 0, st>>>(
      raw_scaling, raw_rotation, raw_opacity, xyz, N, radii, viewmatrix, campos, g_xyz, g_opacity, g_scaling, g_rotation,
      g_all_map, g_scaling_extra, extra_scale, beta, d_xyz, d_opacity, d_scaling, d_rotation, pose_partial);
  HG_POST_LAUNCH(false, st, pose_partial ? "prologue_bwd_pose" : "prologue_bwd");
  if (F > 0 && g_features) {  // NULL: the feature gradient already sits in d_features (rasterizer SH sink)
    axpby4_kernel<<<148 * 8, 256, 0, st>>>((const float4*)g_features, N * (int64_t)F / 4, beta, (float4*)d_features);
    HG_POST_LAUNCH(false, st, "features_grad_accumulate");
  }
  return HG_OK;
}

extern "C" {

int hg_prologue_backward(const float* raw_scaling, const float* raw_rotation, const float* raw_opacity, const float* xyz,
                         int64_t N, int32_t F, const int32_t* radii, const float* viewmatrix, const float* campos,
                         const float* g_xyz, const float* g_features, const float* g_opacity, const float* g_scaling,
                         const float* g_rotation, const float* g_all_map, const float* g_scaling_extra,
                         const float* extra_scale, float beta, float* d_xyz, float* d_features, float* d_opacity,
                         float* d_scaling, float* d_rotation, void* st_) {
  return prologue_backward_impl(raw_scaling, raw_rotation, raw_opacity, xyz, N, F, radii, viewmatrix, campos, g_xyz,
                                g_features, g_opacity, g_scaling, g_rotation, g_all_map, g_scaling_extra, extra_scale,
                                beta, d_xyz, d_features, d_opacity, d_scaling, d_rotation, nullptr, st_);
}

int hg_prologue_backward_pose(const float* raw_scaling, const float* raw_rotation, const float* raw_opacity,
                              const float* xyz, int64_t N, int32_t F, const int32_t* radii, const float* viewmatrix,
                              const float* campos, const float* g_xyz, const float* g_features, const float* g_opacity,
                              const float* g_scaling, const float* g_rotation, const float* g_all_map,
                              const float* g_scaling_extra, const float* extra_scale, float beta, float* d_xyz,
                              float* d_features, float* d_opacity, float* d_scaling, float* d_rotation,
                              void* pose_workspace, void* st_) {
  if (!pose_workspace) {
    set_error("hg_prologue_backward_pose: pose_workspace is NULL");
    return HG_ERR_INVALID_ARG;
  }
  return prologue_backward_impl(raw_scaling, raw_rotation, raw_opacity, xyz, N, F, radii, viewmatrix, campos, g_xyz,
                                g_features, g_opacity, g_scaling, g_rotation, g_all_map, g_scaling_extra, extra_scale,
                                beta, d_xyz, d_features, d_opacity, d_scaling, d_rotation,
                                static_cast<char*>(pose_workspace) + camera_pose_prologue_offset(N), st_);
}

int hg_depth_normal(const float* plane_depth, const float* alpha, int32_t H, int32_t W, hg_intrinsics K,
                    float* out_normal, void* st_) {
  if (!plane_depth || !out_normal) {
    set_error("hg_depth_normal: NULL pointer");
    return HG_ERR_INVALID_ARG;
  }
  Unproj U;
  int rc = make_unproj(K, H, W, &U);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)st_;
  const dim3 grid((W + 31) / 32, (H + 7) / 8);
  depth_normal_kernel<<<grid, 256, 0, st>>>(plane_depth, alpha, H, W, U, out_normal);
  HG_POST_LAUNCH(false, st, "depth_normal");
  return HG_OK;
}

int hg_depth_normal_backward(const float* plane_depth, const float* alpha, const float* dL_dnormal, int32_t H,
                             int32_t W, hg_intrinsics K, float* dL_dplane_depth, void* st_) {
  if (!plane_depth || !dL_dnormal || !dL_dplane_depth) {
    set_error("hg_depth_normal_backward: NULL pointer");
    return HG_ERR_INVALID_ARG;
  }
  Unproj U;
  int rc = make_unproj(K, H, W, &U);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)st_;
  const dim3 grid((W + kTX - 1) / kTX, (H + kTY - 1) / kTY);
  depth_normal_bwd_kernel<false><<<grid, kTX * kTY, 0, st>>>(plane_depth, alpha, dL_dnormal, nullptr, nullptr, 0.f, H,
                                                             W, U, dL_dplane_depth, nullptr);
  HG_POST_LAUNCH(false, st, "depth_normal_bwd");
  return HG_OK;
}

size_t hg_normal_consistency_workspace_bytes(int32_t H, int32_t W) {
  const size_t blocks = (size_t)((W + 31) / 32) * ((H + 7) / 8);
  return blocks * sizeof(double) + 256;
}

int hg_normal_consistency_loss(const float* plane_depth, const float* all_map, const float* image_weight, int32_t H,
                               int32_t W, hg_intrinsics K, float weight, float* out_loss, float* dL_dplane_depth,
                               float* dL_dall_map, void* ws, void* st_) {
  if (!plane_depth || !all_map || !out_loss || !ws || ((dL_dplane_depth == nullptr) != (dL_dall_map == nullptr))) {
    set_error("hg_normal_consistency_loss: bad argument");
    return HG_ERR_INVALID_ARG;
  }
  Unproj U;
  int rc = make_unproj(K, H, W, &U);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)st_;
  double* partial = (double*)(((uintptr_t)ws + 255) / 256 * 256);
  const dim3 grid((W + 31) / 32, (H + 7) / 8);
  const double scale = (double)weight / ((double)H * (double)W);
  normal_loss_fwd_kernel<<<grid, 256, 0, st>>>(plane_depth, all_map, image_weight, H, W, U, partial);
  HG_POST_LAUNCH(false, st, "normal_loss_fwd");
  normal_loss_finalize_kernel<<<1, 1024, 0, st>>>(partial, (int)(grid.x * grid.y), scale, out_loss);
  HG_POST_LAUNCH(false, st, "normal_loss_finalize");
  if (dL_dplane_depth) {
    depth_normal_bwd_kernel<true><<<grid, kTX * kTY, 0, st>>>(plane_depth, nullptr, nullptr, all_map, image_weight,
                                                              (float)scale, H, W, U, dL_dplane_depth, dL_dall_map);
    HG_POST_LAUNCH(false, st, "normal_loss_bwd");
  }
  return HG_OK;
}

int hg_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n_rows,
                 int32_t row_width, const uint8_t* visible_mask, const int64_t* visible_idx, int64_t n_idx, double lr,
                 double beta1, double beta2, double eps, int32_t step, float grad_scale, int32_t head_cols,
                 double head_lr, void* st_) {
  if (n_rows < 0 || row_width <= 0 || step < 1 || (visible_mask && visible_idx) || n_idx < 0 || head_cols < 0 ||
      head_cols > row_width ||
      (n_rows > 0 && (!param || !grad || !exp_avg || !exp_avg_sq))) {
    set_error("hg_adam_step: bad argument");
    return HG_ERR_INVALID_ARG;
  }
  const int64_t n = n_rows * row_width;
  if (n == 0) return HG_OK;
  cudaStream_t st = (cudaStream_t)st_;
  // bias corrections in double, as Python evaluates `1 - beta ** step` and `lr / bias_correction1`
  const double bc1 = 1.0 - std::pow(beta1, (double)step);
  const double bc2 = 1.0 - std::pow(beta2, (double)step);
  AdamArgs a;
  a.beta1 = (float)beta1; a.beta2 = (float)beta2;
  a.one_m_b1 = (float)(1.0 - beta1);
  a.one_m_b2 = (float)(1.0 - beta2);
  a.step_size = (float)(lr / bc1);
  a.inv_bc2_sqrt = (float)(1.0 / std::sqrt(bc2));
  a.eps = (float)eps;
  a.grad_scale = grad_scale;
  a.head_cols = head_cols;
  a.step_size_head = (float)(head_lr / bc1);
  const int blocks = 148 * 8;
  if (visible_idx) {
    if (n_idx == 0) return HG_OK;
    adam_indexed_kernel<<<blocks, 256, 0, st>>>(param, grad, exp_avg, exp_avg_sq, n_rows, row_width, visible_idx, n_idx, a);
  } else if (!visible_mask && head_cols == 0 && n % 4 == 0 &&
             (((uintptr_t)param | (uintptr_t)grad | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) & 15) == 0) {
    adam_dense4_kernel<<<blocks, 256, 0, st>>>((float4*)param, (const float4*)grad, (float4*)exp_avg, (float4*)exp_avg_sq,
                                               n / 4, a);
  } else if (row_width % 4 == 0 &&
             (((uintptr_t)param | (uintptr_t)grad | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) & 15) == 0) {
    adam_masked4_kernel<<<blocks, 256, 0, st>>>((float4*)param, (const float4*)grad, (float4*)exp_avg,
                                                (float4*)exp_avg_sq, n / 4, row_width / 4, visible_mask, a);
  } else {
    adam_dense_kernel<<<blocks, 256, 0, st>>>(param, grad, exp_avg, exp_avg_sq, n, row_width, visible_mask, a);
  }
  HG_POST_LAUNCH(false, st, "adam_step");
  return HG_OK;
}

int hg_densification_stats(const float* grad_means2D, const int32_t* radii, int64_t N, float* xyz_gradient_accum,
                           float* denom, float* max_radii2D, void* st_) {
  if (N < 0 || (N > 0 && (!grad_means2D || !radii || !xyz_gradient_accum || !denom))) {
    set_error("hg_densification_stats: bad argument");
    return HG_ERR_INVALID_ARG;
  }
  if (N == 0) return HG_OK;
  cudaStream_t st = (cudaStream_t)st_;
  densification_stats_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(grad_means2D, radii, N, xyz_gradient_accum, denom,
                                                                            max_radii2D);
  HG_POST_LAUNCH(false, st, "densification_stats");
  return HG_OK;
}

}  // extern "C"
