// camera_pose.cu — per-image camera pose refinement of the training step (DESIGN.md §3 "Camera pose refinement"):
// the corrected camera of a view, and the fixed-order finish of the view's pose gradient.
//
// Image k owns xi_k = (rho, phi) (row k of an [n, 8] fp32 table: rho 3 | phi 3 | 2 zero pads), applied in the camera
// frame: p_cam' = Exp(phi) p_cam + rho, i.e. W2C' = [Exp(phi) | rho] W2C, in the row-vector convention of the
// rasterizer: viewmatrix' = viewmatrix C^T.  The host never reads the table.
//
// The pose variants of the per-Gaussian backward (preprocess_bwd.cu) and of the prologue backward (geometry.cu) leave
// one row of partial sums per CTA: [0..2] dL/drho and [3..5] the torque tau of the left perturbation
// p_cam' -> Exp(d) p_cam' (which also turns rho).  hg_camera_pose_grad_finish sums them in double in a fixed order and
// adds onto the camera's gradient row
//   dL/drho = g,   dL/dphi = J_l(phi)^T (tau - rho x g)
// (changing phi alone turns p_cam' - rho, not rho: hence the rho x g term; J_l is the SO(3) left Jacobian).
#include "common.cuh"
#include "reduce.cuh"
#include "../../include/hidegs_geometry.h"

#include <climits>

namespace hg {

namespace {

constexpr int kFinishThreads = 512;

// Exp(phi) - I = a K + b K^2 and J_l(phi) = I + c K + d K^2 (K = [phi]x), with the series near 0: at phi = 0 both
// corrections are EXACT zeros, so the corrected camera of a zero row is the input camera bit for bit.
__device__ void so3_coeffs(const double p[3], double& a, double& b, double& c, double& d) {
  const double t2 = p[0] * p[0] + p[1] * p[1] + p[2] * p[2];
  if (t2 < 1e-8) {
    a = 1.0 - t2 / 6.0 + t2 * t2 / 120.0;
    b = 0.5 - t2 / 24.0 + t2 * t2 / 720.0;
    c = b;
    d = 1.0 / 6.0 - t2 / 120.0 + t2 * t2 / 5040.0;
  } else {
    const double t = sqrt(t2), s = sin(t), co = cos(t);
    a = s / t;
    b = (1.0 - co) / t2;
    c = b;
    d = (t - s) / (t2 * t);
  }
}

__device__ void skew_terms(const double p[3], double K[3][3], double K2[3][3]) {
  K[0][0] = 0.0;   K[0][1] = -p[2]; K[0][2] = p[1];
  K[1][0] = p[2];  K[1][1] = 0.0;   K[1][2] = -p[0];
  K[2][0] = -p[1]; K[2][1] = p[0];  K[2][2] = 0.0;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) K2[i][j] = K[i][0] * K[0][j] + K[i][1] * K[1][j] + K[i][2] * K[2][j];
}

// out[0..15] viewmatrix', out[16..31] projmatrix', out[32..34] campos' (row-vector convention, as the rasterizer reads
// them).  Every correction is formed as a difference and added last, in double:
//   viewmatrix' = V + V D,                      D = C^T - I = [[Em^T, 0], [rho^T, 0]],  Em = Exp(phi) - I
//   projmatrix' = P + V D (V^-1 P)              (= viewmatrix' times the intrinsic projection V^-1 P)
//   campos'     = c - R^T Exp(phi)^T rho        (the centre moves with rho only)
__global__ void camera_pose_apply_kernel(const float* __restrict__ view, const float* __restrict__ proj,
                                         const float* __restrict__ campos, const float* __restrict__ row,
                                         float* __restrict__ out) {
  if (threadIdx.x != 0) return;
  double V[4][4], P[4][4];
  for (int i = 0; i < 16; ++i) {
    V[i / 4][i % 4] = (double)view[i];
    P[i / 4][i % 4] = (double)proj[i];
  }
  const double rho[3] = {(double)row[0], (double)row[1], (double)row[2]};
  const double phi[3] = {(double)row[3], (double)row[4], (double)row[5]};
  double a, b, c, d, K[3][3], K2[3][3];
  so3_coeffs(phi, a, b, c, d);
  skew_terms(phi, K, K2);
  double Em[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) Em[i][j] = a * K[i][j] + b * K2[i][j];
  double D[4][4] = {};
  for (int k = 0; k < 3; ++k)
    for (int j = 0; j < 3; ++j) D[k][j] = Em[j][k];
  for (int j = 0; j < 3; ++j) D[3][j] = rho[j];
  double VD[4][4];
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) VD[i][j] = V[i][0] * D[0][j] + V[i][1] * D[1][j] + V[i][2] * D[2][j] + V[i][3] * D[3][j];
  // V^-1 of the rigid viewmatrix [[A, 0], [t^T, 1]]: [[A^T, 0], [-t^T A^T, 1]]
  double Vi[4][4] = {};
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) Vi[i][j] = V[j][i];
  for (int j = 0; j < 3; ++j) Vi[3][j] = -(V[3][0] * V[j][0] + V[3][1] * V[j][1] + V[3][2] * V[j][2]);
  Vi[3][3] = 1.0;
  double P0[4][4];
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) P0[i][j] = Vi[i][0] * P[0][j] + Vi[i][1] * P[1][j] + Vi[i][2] * P[2][j] + Vi[i][3] * P[3][j];
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) {
      out[4 * i + j] = (float)(V[i][j] + VD[i][j]);
      const double dp = VD[i][0] * P0[0][j] + VD[i][1] * P0[1][j] + VD[i][2] * P0[2][j] + VD[i][3] * P0[3][j];
      out[16 + 4 * i + j] = (float)(P[i][j] + dp);
    }
  double er[3];  // Exp(phi)^T rho
  for (int j = 0; j < 3; ++j) er[j] = rho[j] + Em[0][j] * rho[0] + Em[1][j] * rho[1] + Em[2][j] * rho[2];
  for (int i = 0; i < 3; ++i)
    out[32 + i] = (float)((double)campos[i] - (V[i][0] * er[0] + V[i][1] * er[1] + V[i][2] * er[2]));
  out[35] = 0.f;
}

// Sum of the 6 leading doubles of n_a rows of `pa` and then of n_b rows of `pb` (stride kPosePartialStride) over one
// CTA: per thread in row order, then warp butterflies, then the warps in index order.  The bits depend on (n_a, n_b)
// only.  Thread 0 applies the result to the camera's gradient row.
__global__ void __launch_bounds__(kFinishThreads)
camera_pose_finish_kernel(const double* __restrict__ pa, int n_a, const double* __restrict__ pb, int n_b,
                          const float* __restrict__ row, float* __restrict__ grad_row, float* __restrict__ view6) {
  __shared__ double sm[kFinishThreads / 32][6];
  double s[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  for (int i = threadIdx.x; i < n_a; i += kFinishThreads) {
    const double2* r = reinterpret_cast<const double2*>(pa + (size_t)i * kPosePartialStride);
    const double2 x = r[0], y = r[1], z = r[2];
    s[0] += x.x; s[1] += x.y; s[2] += y.x; s[3] += y.y; s[4] += z.x; s[5] += z.y;
  }
  for (int i = threadIdx.x; i < n_b; i += kFinishThreads) {
    const double2* r = reinterpret_cast<const double2*>(pb + (size_t)i * kPosePartialStride);
    const double2 x = r[0], y = r[1], z = r[2];
    s[0] += x.x; s[1] += x.y; s[2] += y.x; s[3] += y.y; s[4] += z.x; s[5] += z.y;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    const double w = warp_sum_double(s[k]);
    if (lane == 0) sm[warp][k] = w;
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  double t[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  for (int w = 0; w < kFinishThreads / 32; ++w)
    for (int k = 0; k < 6; ++k) t[k] += sm[w][k];
  const double rho[3] = {(double)row[0], (double)row[1], (double)row[2]};
  const double phi[3] = {(double)row[3], (double)row[4], (double)row[5]};
  const double* g = t;
  const double q[3] = {t[3] - (rho[1] * g[2] - rho[2] * g[1]), t[4] - (rho[2] * g[0] - rho[0] * g[2]),
                       t[5] - (rho[0] * g[1] - rho[1] * g[0])};
  double a, b, c, d, K[3][3], K2[3][3];
  so3_coeffs(phi, a, b, c, d);
  skew_terms(phi, K, K2);
  float out[6];
  for (int j = 0; j < 3; ++j) {
    out[j] = (float)g[j];
    // (J_l^T q)_j = q_j + sum_i (c K[i][j] + d K2[i][j]) q_i
    double v = q[j];
    for (int i = 0; i < 3; ++i) v += (c * K[i][j] + d * K2[i][j]) * q[i];
    out[3 + j] = (float)v;
  }
  for (int k = 0; k < 6; ++k) {
    grad_row[k] = __fadd_rn(grad_row[k], out[k]);
    if (view6) view6[k] = out[k];
  }
}

}  // namespace

}  // namespace hg

using namespace hg;

extern "C" {

int hg_camera_pose_apply(const float* viewmatrix, const float* projmatrix, const float* campos, const float* pose_table,
                         int32_t n_poses, int32_t index, float* out, void* st_) {
  if (!viewmatrix || !projmatrix || !campos || !pose_table || !out || n_poses <= 0 || index < 0 || index >= n_poses) {
    set_error("hg_camera_pose_apply: bad argument (NULL pointer, or index %d outside the table of %d poses)", index,
              n_poses);
    return HG_ERR_INVALID_ARG;
  }
  cudaStream_t st = (cudaStream_t)st_;
  camera_pose_apply_kernel<<<1, 32, 0, st>>>(viewmatrix, projmatrix, campos, pose_table + (size_t)index * 8, out);
  HG_POST_LAUNCH(false, st, "camera_pose_apply");
  return HG_OK;
}

size_t hg_camera_pose_workspace_bytes(int64_t N) {
  if (N <= 0 || N > INT32_MAX) return 0;
  return camera_pose_workspace_bytes(N);
}

int hg_camera_pose_grad_finish(const float* pose_table, int32_t n_poses, int32_t index, int64_t N, const void* workspace,
                               float* pose_grad_table, float* view_grad6, void* st_) {
  if (!pose_table || !workspace || !pose_grad_table || n_poses <= 0 || index < 0 || index >= n_poses || N <= 0 ||
      N > INT32_MAX || (reinterpret_cast<uintptr_t>(workspace) & 15)) {
    set_error("hg_camera_pose_grad_finish: bad argument (NULL pointer, index %d outside the table of %d poses, N %lld, "
              "or a workspace that is not 16-byte aligned)", index, n_poses, (long long)N);
    return HG_ERR_INVALID_ARG;
  }
  cudaStream_t st = (cudaStream_t)st_;
  const char* ws = static_cast<const char*>(workspace);
  const int n_a = (int)((N + kPoseRasterSlots - 1) / kPoseRasterSlots);
  const int n_b = (int)((N + kPosePrologueRows - 1) / kPosePrologueRows);
  camera_pose_finish_kernel<<<1, kFinishThreads, 0, st>>>(
      reinterpret_cast<const double*>(ws), n_a, reinterpret_cast<const double*>(ws + camera_pose_prologue_offset(N)),
      n_b, pose_table + (size_t)index * 8, pose_grad_table + (size_t)index * 8, view_grad6);
  HG_POST_LAUNCH(false, st, "camera_pose_grad_finish");
  return HG_OK;
}

}  // extern "C"
