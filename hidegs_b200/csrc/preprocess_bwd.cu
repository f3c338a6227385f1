// preprocess_bwd.cu — per-Gaussian backward: accumulator row -> parameter grads.
//
// Fuses the reference's two backward kernels computeCov2DCUDA
// (cuda_rasterizer/backward.cu:147-326) and preprocessCUDA<3>
// (backward.cu:398-496, with computeColorFromSH :23-142 and computeCov3D
// :330-393) into ONE pass that reads the 64-byte accumulator row produced by
// the backward blend and writes every user-visible gradient row exactly once
// (rows of culled Gaussians are written as zeros, so callers need no memset:
// the reference zero-fills 324 B per Gaussian with eleven torch::zeros,
// rasterize_points.cu:195-206).
//
// Reference quirks reproduced on purpose: the dilation constant is 0.3 here
// although the forward used 0.1 (backward.cu:211 vs forward.cu:356); the mean
// used for the projection Jacobians is the raw source mean even when a parent
// interpolation was active; with a parent, own opacity/scale/rotation/SH/mean
// gradients are zeroed and (1-t) x mean gradient is pushed to the parent
// (backward.cu:459-495).
#include "common.cuh"
#include "reduce.cuh"
#include "sh_stage.cuh"

namespace hg {

namespace {

constexpr int kThreads = kPoseRasterSlots;
constexpr int kWarps = kThreads / 32;
constexpr int kShStrideMax = 48 + 1;  // M <= 16 coefficients x 3 channels, odd stride

__device__ __forceinline__ void store_or_add3(float* dst, float a, float b, float c, bool atomic) {
  if (atomic) {
    atomicAdd(dst, a);
    atomicAdd(dst + 1, b);
    atomicAdd(dst + 2, c);
  } else {
    dst[0] = a;
    dst[1] = b;
    dst[2] = c;
  }
}

// POSE (camera pose refinement, DESIGN.md §3): every rendered slot also forms the camera side of its gradient — the
// gradient g_p w.r.t. its camera-frame mean over every path, and the torque p_cam x g_p(non-SH) + vee(G - G^T) with
// G = dL/dW W^T of the covariance path (the SH view direction moves with the camera centre, i.e. with rho only) — and
// the CTA writes the sum of these six numbers (double, fixed order) to pose_partial[global block][0..5].
template <bool POSE>
__global__ void __launch_bounds__(kThreads)
preprocess_bwd_kernel(const int P, const int block0, const int D, const int M, const int* __restrict__ indices,
                      const int* __restrict__ parent_indices, const float* __restrict__ ts,
                      const float* __restrict__ means3D, const int* __restrict__ radii,
                      const float* __restrict__ shs, const uint8_t* __restrict__ clamped,
                      const float* __restrict__ opacities, const float* __restrict__ scales,
                      const float* __restrict__ rotations, const float scale_modifier,
                      const float* __restrict__ cov3Ds, const bool cov_precomp,
                      const float* __restrict__ viewmatrix, const float* __restrict__ projmatrix,
                      const float* __restrict__ campos, const float h_x, const float h_y,
                      const float tan_fovx, const float tan_fovy,
                      const float* __restrict__ accum, const bool has_invdepth,
                      const bool prezeroed, float* __restrict__ dL_dmeans2D,
                      float* __restrict__ dL_dconic, float* __restrict__ dL_dopacity,
                      float* __restrict__ dL_dcolors, float* __restrict__ dL_dinvdepths,
                      float* __restrict__ dL_dmeans3D, float* __restrict__ dL_dcov3D,
                      float* __restrict__ dL_dsh, float* __restrict__ dL_dscales,
                      float* __restrict__ dL_drotations, float* __restrict__ dL_dall_map,
                      float* __restrict__ sh_sink, const float sh_beta, float* __restrict__ sh_factor,
                      double* __restrict__ pose_partial) {
  // SH rows (read AND written, 2 x 192 B per Gaussian at degree 3: 60 % of this kernel's traffic) move through a
  // per-warp shared-memory tile with coalesced 128-bit accesses when the warp's rows are contiguous (no index
  // remap); each thread then works on its own row of the tile.
  __shared__ float s_sh[kWarps][32 * kShStrideMax];
  const int t_idx = (blockIdx.x + block0) * kThreads + threadIdx.x;  // block0: first block of this chunk
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool in_range = t_idx < P;
  const int row = 3 * M;
  const bool alive = in_range && radii[t_idx] > 0;
  const uint32_t alive_mask = __ballot_sync(0xffffffffu, alive);
  const bool staged = shs != nullptr && indices == nullptr && (row & 3) == 0 &&
                      ((reinterpret_cast<uintptr_t>(shs) | reinterpret_cast<uintptr_t>(dL_dsh)) & 15) == 0;
  float* const tile = s_sh[warp];
  const size_t warp_base = (size_t)((blockIdx.x + block0) * kThreads + warp * 32) * row;
  const size_t sh_total = (size_t)P * row;
  // The thread's own rows are requested BEFORE the cooperative SH staging so that both are in flight together.
  float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, a2 = a0, a3 = a0;
  float mx = 0.f, my = 0.f, mz = 0.f;
  float pre_c3[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, pre_opacity = 0.f, pre_scale[3] = {0.f, 0.f, 0.f};
  float4 pre_rot = make_float4(0.f, 0.f, 0.f, 0.f);
  uint8_t pre_clamped = 0;
  if (alive) {
    const float4* ar = reinterpret_cast<const float4*>(accum) + 4 * (size_t)t_idx;
    a0 = __ldg(ar); a1 = __ldg(ar + 1); a2 = __ldg(ar + 2); a3 = __ldg(ar + 3);
    const size_t gpre = indices ? (size_t)__ldg(indices + t_idx) : (size_t)t_idx;
    mx = __ldg(means3D + 3 * gpre); my = __ldg(means3D + 3 * gpre + 1); mz = __ldg(means3D + 3 * gpre + 2);
    const float* c3p = cov_precomp ? (cov3Ds + 6 * gpre) : (cov3Ds + 6 * (size_t)t_idx);
#pragma unroll
    for (int i = 0; i < 6; ++i) pre_c3[i] = __ldg(c3p + i);
    pre_opacity = __ldg(opacities + gpre);
    if (scales) {
      pre_scale[0] = __ldg(scales + 3 * gpre); pre_scale[1] = __ldg(scales + 3 * gpre + 1); pre_scale[2] = __ldg(scales + 3 * gpre + 2);
      pre_rot = __ldg((const float4*)rotations + gpre);
    }
    if (shs) pre_clamped = clamped[t_idx];
  }
  if (staged && alive_mask) {
    if (row == 48) stage_sh_rows<48>(shs, warp_base, sh_total, row, lane, tile, alive_mask);
    else stage_sh_rows<0>(shs, warp_base, sh_total, row, lane, tile, alive_mask);
    __syncwarp();
  }
  // camera side of this slot's gradient (POSE): [0..2] dL/drho, [3..5] torque; zero for culled slots
  float pose[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  do {  // single-trip block: `break` = this thread is done (it still joins the cooperative store below)
  if (!in_range) break;
  const int idx = indices ? __ldg(indices + t_idx) : t_idx;
  const size_t g = (size_t)idx;

  if (!alive) {
    if (sh_factor) sh_factor[3 * g] = sh_factor[3 * g + 1] = sh_factor[3 * g + 2] = 0.f;
    if (prezeroed) break;
    // Culled slot: its gradient rows are all zero.
    dL_dmeans2D[3 * g] = dL_dmeans2D[3 * g + 1] = dL_dmeans2D[3 * g + 2] = 0.f;
    if (dL_dconic) dL_dconic[4 * g] = dL_dconic[4 * g + 1] = dL_dconic[4 * g + 2] = dL_dconic[4 * g + 3] = 0.f;
    dL_dopacity[g] = 0.f;
    dL_dcolors[3 * g] = dL_dcolors[3 * g + 1] = dL_dcolors[3 * g + 2] = 0.f;
    if (dL_dinvdepths) dL_dinvdepths[g] = 0.f;
    dL_dmeans3D[3 * g] = dL_dmeans3D[3 * g + 1] = dL_dmeans3D[3 * g + 2] = 0.f;
#pragma unroll
    for (int i = 0; i < 6; ++i) dL_dcov3D[6 * g + i] = 0.f;
    if (!sh_factor && !staged)
      for (int i = 0; i < row; ++i) dL_dsh[g * row + i] = 0.f;
    dL_dscales[3 * g] = dL_dscales[3 * g + 1] = dL_dscales[3 * g + 2] = 0.f;
    dL_drotations[4 * g] = dL_drotations[4 * g + 1] = dL_drotations[4 * g + 2] = dL_drotations[4 * g + 3] = 0.f;
#pragma unroll
    for (int i = 0; i < 5; ++i) dL_dall_map[5 * g + i] = 0.f;
    break;
  }

  // ---- accumulator row --------------------------------------------------------
  const float dcol[3] = {a0.x, a0.y, a0.z};
  const float dinvd = a0.w;
  const float dam[5] = {a1.x, a1.y, a1.z, a1.w, a2.x};
  const float dm2x = a2.y, dm2y = a2.z;
  const float dcon_x = a2.w, dcon_y = a3.x, dcon_z = a3.y;
  const float dopac_raw = a3.z;

  dL_dmeans2D[3 * g] = dm2x;
  dL_dmeans2D[3 * g + 1] = dm2y;
  dL_dmeans2D[3 * g + 2] = 0.f;
  if (dL_dconic) {
    dL_dconic[4 * g] = dcon_x;
    dL_dconic[4 * g + 1] = dcon_y;
    dL_dconic[4 * g + 2] = 0.f;
    dL_dconic[4 * g + 3] = dcon_z;
  }
  dL_dcolors[3 * g] = dcol[0];
  dL_dcolors[3 * g + 1] = dcol[1];
  dL_dcolors[3 * g + 2] = dcol[2];
  if (dL_dinvdepths) dL_dinvdepths[g] = dinvd;
#pragma unroll
  for (int i = 0; i < 5; ++i) dL_dall_map[5 * g + i] = dam[i];

  float v[16], pm[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    v[i] = __ldg(viewmatrix + i);
    pm[i] = __ldg(projmatrix + i);
  }

  // ---- conic -> 2-D covariance -> 3-D covariance / mean (backward.cu:147-326) --
  const float V00 = pre_c3[0], V01 = pre_c3[1], V02 = pre_c3[2], V11 = pre_c3[3], V12 = pre_c3[4], V22 = pre_c3[5];

  float tx = v[0] * mx + v[4] * my + v[8] * mz + v[12];
  float ty = v[1] * mx + v[5] * my + v[9] * mz + v[13];
  const float pcx = tx, pcy = ty;  // (POSE) the camera-frame mean before the frustum clamp
  const float tz = v[2] * mx + v[6] * my + v[10] * mz + v[14];
  const float limx = 1.3f * tan_fovx, limy = 1.3f * tan_fovy;
  const float txtz = tx / tz, tytz = ty / tz;
  tx = fminf(limx, fmaxf(-limx, txtz)) * tz;
  ty = fminf(limy, fmaxf(-limy, tytz)) * tz;
  const float x_grad_mul = (txtz < -limx || txtz > limx) ? 0.f : 1.f;
  const float y_grad_mul = (tytz < -limy || tytz > limy) ? 0.f : 1.f;

  const float J00 = h_x / tz, J02 = -(h_x * tx) / (tz * tz);
  const float J11 = h_y / tz, J12 = -(h_y * ty) / (tz * tz);
  // T[c][r] = W[0|1][r] * Jcc + W[2][r] * Jc2
  const float T00 = v[0] * J00 + v[2] * J02, T01 = v[4] * J00 + v[6] * J02,
              T02 = v[8] * J00 + v[10] * J02;
  const float T10 = v[1] * J11 + v[2] * J12, T11 = v[5] * J11 + v[6] * J12,
              T12 = v[9] * J11 + v[10] * J12;
  // V * T0 and V * T1
  const float VT0x = V00 * T00 + V01 * T01 + V02 * T02;
  const float VT0y = V01 * T00 + V11 * T01 + V12 * T02;
  const float VT0z = V02 * T00 + V12 * T01 + V22 * T02;
  const float VT1x = V00 * T10 + V01 * T11 + V02 * T12;
  const float VT1y = V01 * T10 + V11 * T11 + V12 * T12;
  const float VT1z = V02 * T10 + V12 * T11 + V22 * T12;
  float c_xx = T00 * VT0x + T01 * VT0y + T02 * VT0z;
  const float c_xy = T00 * VT1x + T01 * VT1y + T02 * VT1z;
  float c_yy = T10 * VT1x + T11 * VT1y + T12 * VT1z;

  constexpr float h_var = 0.3f;  // sic: backward.cu:211
  const float det_cov = c_xx * c_yy - c_xy * c_xy;
  c_xx += h_var;
  c_yy += h_var;
  const float det_cov_plus_h = c_xx * c_yy - c_xy * c_xy;
  const float ratio = det_cov / det_cov_plus_h;
  const float h_scale = sqrtf(fmaxf(0.000025f, ratio));
  const float d_h_scale = dopac_raw * pre_opacity;
  float dopac = dopac_raw * h_scale;
  const float d_inside_root = (ratio <= 0.000025f) ? 0.f : d_h_scale / (2.f * h_scale);

  float dL_dc_xx, dL_dc_xy, dL_dc_yy;
  {
    const float x = c_xx, y = c_yy, z = c_xy, w = h_var;
    const float den = w * w + w * (x + y) + x * y - z * z;
    const float denom_f = d_inside_root / (den * den);
    dL_dc_xx = w * (w * y + y * y + z * z) * denom_f;
    dL_dc_yy = w * (w * x + x * x + z * z) * denom_f;
    dL_dc_xy = -2.f * w * z * (w + x + y) * denom_f;
  }

  const float denom = c_xx * c_yy - c_xy * c_xy;
  const float denom2inv = 1.0f / ((denom * denom) + 0.0000001f);
  float dV[6];
  if (denom2inv != 0.f) {
    dL_dc_xx += denom2inv * (-c_yy * c_yy * dcon_x + 2.f * c_xy * c_yy * dcon_y +
                             (denom - c_xx * c_yy) * dcon_z);
    dL_dc_yy += denom2inv * (-c_xx * c_xx * dcon_z + 2.f * c_xx * c_xy * dcon_y +
                             (denom - c_xx * c_yy) * dcon_x);
    dL_dc_xy += denom2inv * 2.f *
                (c_xy * c_yy * dcon_x - (denom + 2.f * c_xy * c_xy) * dcon_y + c_xx * c_xy * dcon_z);
    dV[0] = T00 * T00 * dL_dc_xx + T00 * T10 * dL_dc_xy + T10 * T10 * dL_dc_yy;
    dV[3] = T01 * T01 * dL_dc_xx + T01 * T11 * dL_dc_xy + T11 * T11 * dL_dc_yy;
    dV[5] = T02 * T02 * dL_dc_xx + T02 * T12 * dL_dc_xy + T12 * T12 * dL_dc_yy;
    dV[1] = 2.f * T00 * T01 * dL_dc_xx + (T00 * T11 + T01 * T10) * dL_dc_xy + 2.f * T10 * T11 * dL_dc_yy;
    dV[2] = 2.f * T00 * T02 * dL_dc_xx + (T00 * T12 + T02 * T10) * dL_dc_xy + 2.f * T10 * T12 * dL_dc_yy;
    dV[4] = 2.f * T02 * T01 * dL_dc_xx + (T01 * T12 + T02 * T11) * dL_dc_xy + 2.f * T11 * T12 * dL_dc_yy;
  } else {
#pragma unroll
    for (int i = 0; i < 6; ++i) dV[i] = 0.f;
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) dL_dcov3D[6 * g + i] = dV[i];

  // dL/dT (upper 2x3), dL/dJ, dL/dt
  const float dT00 = 2.f * VT0x * dL_dc_xx + VT1x * dL_dc_xy;
  const float dT01 = 2.f * VT0y * dL_dc_xx + VT1y * dL_dc_xy;
  const float dT02 = 2.f * VT0z * dL_dc_xx + VT1z * dL_dc_xy;
  const float dT10 = 2.f * VT1x * dL_dc_yy + VT0x * dL_dc_xy;
  const float dT11 = 2.f * VT1y * dL_dc_yy + VT0y * dL_dc_xy;
  const float dT12 = 2.f * VT1z * dL_dc_yy + VT0z * dL_dc_xy;
  const float dJ00 = v[0] * dT00 + v[4] * dT01 + v[8] * dT02;
  const float dJ02 = v[2] * dT00 + v[6] * dT01 + v[10] * dT02;
  const float dJ11 = v[1] * dT10 + v[5] * dT11 + v[9] * dT12;
  const float dJ12 = v[2] * dT10 + v[6] * dT11 + v[10] * dT12;
  const float itz = 1.f / tz, itz2 = itz * itz, itz3 = itz2 * itz;
  const float dtx = x_grad_mul * -h_x * itz2 * dJ02;
  const float dty = y_grad_mul * -h_y * itz2 * dJ12;
  float dtz = -h_x * itz2 * dJ00 - h_y * itz2 * dJ11 + (2.f * h_x * tx) * itz3 * dJ02 +
              (2.f * h_y * ty) * itz3 * dJ12;
  if (has_invdepth) dtz -= dinvd / (tz * tz);
  if constexpr (POSE) {
    // torque of the covariance path: G = J^T A, A = dL/dT W^T (2 x 3; A00, A02, A11, A12 are the dJ above)
    const float A01 = v[1] * dT00 + v[5] * dT01 + v[9] * dT02;
    const float A10 = v[0] * dT10 + v[4] * dT11 + v[8] * dT12;
    pose[3] = (J02 * A01 + J12 * dJ11) - J11 * dJ12;  // G21 - G12
    pose[4] = J00 * dJ02 - (J02 * dJ00 + J12 * A10);  // G02 - G20
    pose[5] = J11 * A10 - J00 * A01;                  // G10 - G01
  }
  float dmean_x = v[0] * dtx + v[1] * dty + v[2] * dtz;
  float dmean_y = v[4] * dtx + v[5] * dty + v[6] * dtz;
  float dmean_z = v[8] * dtx + v[9] * dty + v[10] * dtz;

  // ---- 2-D mean -> 3-D mean (backward.cu:433-449) ------------------------------
  {
    const float hw = pm[3] * mx + pm[7] * my + pm[11] * mz + pm[15];
    const float m_w = 1.0f / (hw + 0.0000001f);
    const float mul1 = (pm[0] * mx + pm[4] * my + pm[8] * mz + pm[12]) * m_w * m_w;
    const float mul2 = (pm[1] * mx + pm[5] * my + pm[9] * mz + pm[13]) * m_w * m_w;
    dmean_x += (pm[0] * m_w - pm[3] * mul1) * dm2x + (pm[1] * m_w - pm[3] * mul2) * dm2y;
    dmean_y += (pm[4] * m_w - pm[7] * mul1) * dm2x + (pm[5] * m_w - pm[7] * mul2) * dm2y;
    dmean_z += (pm[8] * m_w - pm[11] * mul1) * dm2x + (pm[9] * m_w - pm[11] * mul2) * dm2y;
  }

  if constexpr (POSE) {  // + p_cam x g_p over every path but the SH view direction (g_p = W dL/dmean)
    const float gx = v[0] * dmean_x + v[4] * dmean_y + v[8] * dmean_z;
    const float gy = v[1] * dmean_x + v[5] * dmean_y + v[9] * dmean_z;
    const float gz = v[2] * dmean_x + v[6] * dmean_y + v[10] * dmean_z;
    pose[3] += pcy * gz - tz * gy;
    pose[4] += tz * gx - pcx * gz;
    pose[5] += pcx * gy - pcy * gx;
  }

  // Parent handling decides what survives (backward.cu:459-495).
  int parent_id = -1;
  if (parent_indices) parent_id = __ldg(parent_indices + t_idx);
  const bool has_parent = parent_id != -1;

  // ---- SH backward (backward.cu:23-142) -----------------------------------------
  if (shs) {
    float* out = staged ? tile + lane * (row | 1) : dL_dsh + g * row;
    const float ox = mx - __ldg(campos), oy = my - __ldg(campos + 1), oz = mz - __ldg(campos + 2);
    const float len = sqrtf(ox * ox + oy * oy + oz * oz);
    const float x = ox / len, y = oy / len, z = oz / len;
    const uint8_t cb = pre_clamped;
    const float dr = (cb & 1) ? 0.f : dcol[0], dg = (cb & 2) ? 0.f : dcol[1],
                db = (cb & 4) ? 0.f : dcol[2];
    const float* sh = staged ? tile + lane * (row | 1) : shs + g * row;
    float basis[16];
    float ddx = 0.f, ddy = 0.f, ddz = 0.f;
    // s(k) = <sh[k], dL/dRGB>   (every s(k) is taken before the row is overwritten with the gradient below)
    auto s = [&](int k) { return sh[3 * k] * dr + sh[3 * k + 1] * dg + sh[3 * k + 2] * db; };
    basis[0] = SH_C0;
    int nb = 1;
    if (D > 0) {
      basis[1] = -SH_C1 * y;
      basis[2] = SH_C1 * z;
      basis[3] = -SH_C1 * x;
      nb = 4;
      ddx = -SH_C1 * s(3);
      ddy = -SH_C1 * s(1);
      ddz = SH_C1 * s(2);
      if (D > 1) {
        const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
        basis[4] = SH_C2_0 * xy;
        basis[5] = SH_C2_1 * yz;
        basis[6] = SH_C2_2 * (2.f * zz - xx - yy);
        basis[7] = SH_C2_3 * xz;
        basis[8] = SH_C2_4 * (xx - yy);
        nb = 9;
        const float s4 = s(4), s5 = s(5), s6 = s(6), s7 = s(7), s8 = s(8);
        ddx += SH_C2_0 * y * s4 + SH_C2_2 * 2.f * -x * s6 + SH_C2_3 * z * s7 + SH_C2_4 * 2.f * x * s8;
        ddy += SH_C2_0 * x * s4 + SH_C2_1 * z * s5 + SH_C2_2 * 2.f * -y * s6 + SH_C2_4 * 2.f * -y * s8;
        ddz += SH_C2_1 * y * s5 + SH_C2_2 * 4.f * z * s6 + SH_C2_3 * x * s7;
        if (D > 2) {
          basis[9] = SH_C3_0 * y * (3.f * xx - yy);
          basis[10] = SH_C3_1 * xy * z;
          basis[11] = SH_C3_2 * y * (4.f * zz - xx - yy);
          basis[12] = SH_C3_3 * z * (2.f * zz - 3.f * xx - 3.f * yy);
          basis[13] = SH_C3_4 * x * (4.f * zz - xx - yy);
          basis[14] = SH_C3_5 * z * (xx - yy);
          basis[15] = SH_C3_6 * x * (xx - 3.f * yy);
          nb = 16;
          const float s9 = s(9), s10 = s(10), s11 = s(11), s12 = s(12), s13 = s(13), s14 = s(14),
                      s15 = s(15);
          ddx += SH_C3_0 * s9 * 6.f * xy + SH_C3_1 * s10 * yz + SH_C3_2 * s11 * -2.f * xy +
                 SH_C3_3 * s12 * -6.f * xz + SH_C3_4 * s13 * (-3.f * xx + 4.f * zz - yy) +
                 SH_C3_5 * s14 * 2.f * xz + SH_C3_6 * s15 * 3.f * (xx - yy);
          ddy += SH_C3_0 * s9 * 3.f * (xx - yy) + SH_C3_1 * s10 * xz +
                 SH_C3_2 * s11 * (-3.f * yy + 4.f * zz - xx) + SH_C3_3 * s12 * -6.f * yz +
                 SH_C3_4 * s13 * -2.f * xy + SH_C3_5 * s14 * -2.f * yz + SH_C3_6 * s15 * -6.f * xy;
          ddz += SH_C3_1 * s10 * xy + SH_C3_2 * s11 * 8.f * yz +
                 SH_C3_3 * s12 * 3.f * (2.f * zz - xx - yy) + SH_C3_4 * s13 * 8.f * xz +
                 SH_C3_5 * s14 * (xx - yy);
        }
      }
    }
    if (nb > M) nb = M;
    // With a parent the reference zeroes the (48-float) SH gradient row again.
    const float keep = has_parent ? 0.f : 1.f;
    if (sh_factor) {
      // factored exchange (include/hidegs_exchange.h): dL/dSH is the outer product basis(view direction) x dL/dRGB, so
      // only the three clamp-masked colour gradients leave this kernel; hg_sh_gradient_from_factors rebuilds the rows
      sh_factor[3 * g] = keep * dr;
      sh_factor[3 * g + 1] = keep * dg;
      sh_factor[3 * g + 2] = keep * db;
    } else {
      for (int k = 0; k < M; ++k) {
        const float bk = (k < nb) ? basis[k] * keep : 0.f;
        if (k < nb || !prezeroed || staged) {
          out[3 * k] = bk * dr;
          out[3 * k + 1] = bk * dg;
          out[3 * k + 2] = bk * db;
        }
      }
    }
    // d(normalised dir)/d(mean)  (auxiliary.h:132-142)
    const float sum2 = ox * ox + oy * oy + oz * oz;
    const float invsum32 = 1.0f / sqrtf(sum2 * sum2 * sum2);
    dmean_x += ((sum2 - ox * ox) * ddx - oy * ox * ddy - oz * ox * ddz) * invsum32;
    dmean_y += (-ox * oy * ddx + (sum2 - oy * oy) * ddy - oz * oy * ddz) * invsum32;
    dmean_z += (-ox * oz * ddx - oy * oz * ddy + (sum2 - oz * oz) * ddz) * invsum32;
  }

  // ---- 3-D covariance -> scale / rotation (backward.cu:330-393) -------------------
  float dsx = 0.f, dsy = 0.f, dsz = 0.f, dqr = 0.f, dqx = 0.f, dqy = 0.f, dqz = 0.f;
  if (scales) {
    const float4 q4 = pre_rot;
    const float r = q4.x, x = q4.y, y = q4.z, z = q4.w;
    const float s0 = scale_modifier * pre_scale[0], s1 = scale_modifier * pre_scale[1],
                s2 = scale_modifier * pre_scale[2];
    // R[c][r] as constructed in the forward (glm column-major argument order).
    const float R[3][3] = {{1.f - 2.f * (y * y + z * z), 2.f * (x * y - r * z), 2.f * (x * z + r * y)},
                           {2.f * (x * y + r * z), 1.f - 2.f * (x * x + z * z), 2.f * (y * z - r * x)},
                           {2.f * (x * z - r * y), 2.f * (y * z + r * x), 1.f - 2.f * (x * x + y * y)}};
    const float sc[3] = {s0, s1, s2};
    // Symmetric dL/dSigma with halved off-diagonals.
    const float S[3][3] = {{dV[0], 0.5f * dV[1], 0.5f * dV[2]},
                           {0.5f * dV[1], dV[3], 0.5f * dV[4]},
                           {0.5f * dV[2], 0.5f * dV[4], dV[5]}};
    // dM[c][k] = 2 * sum_j M[j][k] * S[c][j],  M[j][k] = sc[k] * R[j][k]
    float Dr[3][3];  // dL/dR[c][k]
    float ds[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float dM = 2.f * (sc[k] * R[0][k] * S[c][0] + sc[k] * R[1][k] * S[c][1] +
                                sc[k] * R[2][k] * S[c][2]);
        ds[k] += R[c][k] * dM;
        Dr[c][k] = sc[k] * dM;
      }
    }
    // The reference stores dL/dscale without the scale_modifier chain factor.
    dsx = ds[0];
    dsy = ds[1];
    dsz = ds[2];
    dqr = 2.f * (-z * Dr[0][1] + y * Dr[0][2] + z * Dr[1][0] - x * Dr[1][2] - y * Dr[2][0] + x * Dr[2][1]);
    dqx = 2.f * (y * Dr[0][1] + z * Dr[0][2] + y * Dr[1][0] - 2.f * x * Dr[1][1] - r * Dr[1][2] +
                 z * Dr[2][0] + r * Dr[2][1] - 2.f * x * Dr[2][2]);
    dqy = 2.f * (-2.f * y * Dr[0][0] + x * Dr[0][1] + r * Dr[0][2] + x * Dr[1][0] + z * Dr[1][2] -
                 r * Dr[2][0] + z * Dr[2][1] - 2.f * y * Dr[2][2]);
    dqz = 2.f * (-2.f * z * Dr[0][0] - r * Dr[0][1] + x * Dr[0][2] + r * Dr[1][0] - 2.f * z * Dr[1][1] +
                 y * Dr[1][2] + x * Dr[2][0] + y * Dr[2][1]);
  }

  if constexpr (POSE) {  // dL/drho = W dL/dmean over every path (the camera centre moves by -R^T rho)
    pose[0] = v[0] * dmean_x + v[4] * dmean_y + v[8] * dmean_z;
    pose[1] = v[1] * dmean_x + v[5] * dmean_y + v[9] * dmean_z;
    pose[2] = v[2] * dmean_x + v[6] * dmean_y + v[10] * dmean_z;
  }

  if (has_parent) {
    const float t = __ldg(ts + t_idx);
    dopac = 0.f;
    dsx = dsy = dsz = 0.f;
    dqr = dqx = dqy = dqz = 0.f;
    float* pdst = dL_dmeans3D + 3 * (size_t)parent_id;
    atomicAdd(pdst, (1.0f - t) * dmean_x);
    atomicAdd(pdst + 1, (1.0f - t) * dmean_y);
    atomicAdd(pdst + 2, (1.0f - t) * dmean_z);
    dmean_x = dmean_y = dmean_z = 0.f;
  }

  dL_dopacity[g] = dopac;
  store_or_add3(dL_dmeans3D + 3 * g, dmean_x, dmean_y, dmean_z, parent_indices != nullptr);
  if (scales || !prezeroed) {
    dL_dscales[3 * g] = dsx;
    dL_dscales[3 * g + 1] = dsy;
    dL_dscales[3 * g + 2] = dsz;
    dL_drotations[4 * g] = dqr;
    dL_drotations[4 * g + 1] = dqx;
    dL_drotations[4 * g + 2] = dqy;
    dL_drotations[4 * g + 3] = dqz;
  }
  } while (0);
  if (sh_factor) {  // the view's camera centre rides behind the factors: [3 P .. 3 P + 2]
    if (blockIdx.x == 0 && block0 == 0 && threadIdx.x < 3) sh_factor[3 * (size_t)P + threadIdx.x] = __ldg(campos + threadIdx.x);
  } else if (staged && sh_sink) {  // accumulate straight into the caller's gradient arena (launcher guarantees `staged`)
    if (alive_mask || sh_beta == 0.f) {
      __syncwarp();
      unstage_sh_rows_accum(sh_sink, warp_base, sh_total, row, lane, tile, alive_mask, sh_beta);
    }
  } else if (staged && (alive_mask || !prezeroed)) {
    __syncwarp();
    unstage_sh_rows(dL_dsh, warp_base, sh_total, row, lane, tile, alive_mask, !prezeroed);
  }
  if constexpr (POSE) {  // warp butterflies in double, then the 4 warps in index order: bits fixed by the slot count
    __shared__ double s_pose[kWarps][6];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const double w = warp_sum_double((double)pose[k]);
      if (lane == 0) s_pose[warp][k] = w;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
      double acc = 0.0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) acc += s_pose[w][threadIdx.x];
      pose_partial[(size_t)(blockIdx.x + block0) * kPosePartialStride + threadIdx.x] = acc;
    }
  }
}

// dL/dSH rows rebuilt from the factors of `n_views` views (factored gradient exchange, include/hidegs_exchange.h):
//   dL_dsh[g][k][c] = beta * dL_dsh[g][k][c] + sum_v basis_k(normalize(mean_g - campos_v)) * factor_v[g][c]
// with the basis expressions of the SH backward above, summed in view order (every rank forms the same bits).  Thread
// per Gaussian, 3 M accumulators in registers, rows leave through the per-warp tile as coalesced 128-bit stores.
__global__ void __launch_bounds__(kThreads)
sh_from_factors_kernel(const int N, const int D, const int M, const int n_views, const float* __restrict__ means3D,
                       const float* __restrict__ factors, const size_t view_stride, float* __restrict__ dL_dsh,
                       const float beta, const bool vector_rows) {
  __shared__ float s_sh[kWarps][32 * kShStrideMax];
  const int g = blockIdx.x * kThreads + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row = 3 * M;
  float acc[48];
#pragma unroll
  for (int i = 0; i < 48; ++i) acc[i] = 0.f;
  if (g < N) {
    const float mx = __ldg(means3D + 3 * (size_t)g), my = __ldg(means3D + 3 * (size_t)g + 1),
                mz = __ldg(means3D + 3 * (size_t)g + 2);
    for (int v = 0; v < n_views; ++v) {
      const float* fv = factors + (size_t)v * view_stride;
      const float dr = __ldg(fv + 3 * (size_t)g), dg = __ldg(fv + 3 * (size_t)g + 1), db = __ldg(fv + 3 * (size_t)g + 2);
      if (dr == 0.f && dg == 0.f && db == 0.f) continue;  // culled (or fully clamped) in that view
      const float ox = mx - __ldg(fv + 3 * (size_t)N), oy = my - __ldg(fv + 3 * (size_t)N + 1),
                  oz = mz - __ldg(fv + 3 * (size_t)N + 2);
      const float len = sqrtf(ox * ox + oy * oy + oz * oz);
      const float x = ox / len, y = oy / len, z = oz / len;
      float basis[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) basis[k] = 0.f;
      basis[0] = SH_C0;
      if (D > 0) {
        basis[1] = -SH_C1 * y;
        basis[2] = SH_C1 * z;
        basis[3] = -SH_C1 * x;
        if (D > 1) {
          const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
          basis[4] = SH_C2_0 * xy;
          basis[5] = SH_C2_1 * yz;
          basis[6] = SH_C2_2 * (2.f * zz - xx - yy);
          basis[7] = SH_C2_3 * xz;
          basis[8] = SH_C2_4 * (xx - yy);
          if (D > 2) {
            basis[9] = SH_C3_0 * y * (3.f * xx - yy);
            basis[10] = SH_C3_1 * xy * z;
            basis[11] = SH_C3_2 * y * (4.f * zz - xx - yy);
            basis[12] = SH_C3_3 * z * (2.f * zz - 3.f * xx - 3.f * yy);
            basis[13] = SH_C3_4 * x * (4.f * zz - xx - yy);
            basis[14] = SH_C3_5 * z * (xx - yy);
            basis[15] = SH_C3_6 * x * (xx - 3.f * yy);
          }
        }
      }
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        acc[3 * k] += basis[k] * dr;
        acc[3 * k + 1] += basis[k] * dg;
        acc[3 * k + 2] += basis[k] * db;
      }
    }
  }
  if (vector_rows) {
    float* const tile = s_sh[warp];
    float* const mine = tile + lane * (row | 1);
#pragma unroll
    for (int i = 0; i < 48; ++i)
      if (i < row) mine[i] = acc[i];
    __syncwarp();
    const size_t warp_base = (size_t)(blockIdx.x * kThreads + warp * 32) * row;
    if (warp_base < (size_t)N * row)
      unstage_sh_rows_accum(dL_dsh, warp_base, (size_t)N * row, row, lane, tile, 0xffffffffu, beta);
  } else if (g < N) {
#pragma unroll
    for (int i = 0; i < 48; ++i)
      if (i < row) {
        float* d = dL_dsh + (size_t)g * row + i;
        *d = beta != 0.f ? fmaf(beta, *d, acc[i]) : acc[i];
      }
  }
}

}  // namespace

int launch_sh_from_factors(int N, int D, int M, int n_views, const float* means3D, const float* factors,
                           size_t view_stride, float* dL_dsh, float beta, cudaStream_t stream) {
  const bool vector_rows = ((3 * M) & 3) == 0 && (reinterpret_cast<uintptr_t>(dL_dsh) & 15) == 0;
  sh_from_factors_kernel<<<(N + kThreads - 1) / kThreads, kThreads, 0, stream>>>(N, D, M, n_views, means3D, factors,
                                                                                view_stride, dL_dsh, beta, vector_rows);
  HG_POST_LAUNCH(false, stream, "sh_from_factors");
  return HG_OK;
}

int launch_preprocess_bwd(const hg_raster_inputs& in, const GeomState& g, const int* radii,
                          float focal_x, float focal_y, const float* accum, bool has_invdepth,
                          float* dL_dmeans2D, float* dL_dconic, float* dL_dopacity,
                          float* dL_dcolors, float* dL_dinvdepths, float* dL_dmeans3D,
                          float* dL_dcov3D, float* dL_dsh, float* dL_dscales,
                          float* dL_drotations, float* dL_dall_map, cudaStream_t stream, int slot_begin,
                          int slot_end, float* sh_sink, float sh_beta, float* sh_factor, bool skip_culled_rows,
                          double* pose_partial) {
  // "prezeroed": the kernel leaves the rows of culled slots alone — because the caller zero-filled the arrays (index
  // remap / parents: rows are scattered and accumulated), or because it never reads them (HG_BWD_SKIP_CULLED_ROWS)
  const bool prezeroed = in.indices != nullptr || in.parent_indices != nullptr || skip_culled_rows;
  const float* cov = in.cov3D_precomp ? in.cov3D_precomp : g.cov3D;
  // [slot_begin, slot_end): the slots this launch covers (slot_begin a multiple of the block size; -1 = to the end)
  if (slot_end < 0 || slot_end > in.P) slot_end = in.P;
  if (sh_sink) {  // the sink is written by the staged (coalesced, contiguous-rows) path only
    const int row = 3 * in.M;
    if (!in.shs || in.indices || in.parent_indices || (row & 3) ||
        ((reinterpret_cast<uintptr_t>(in.shs) | reinterpret_cast<uintptr_t>(dL_dsh) | reinterpret_cast<uintptr_t>(sh_sink)) & 15)) {
      set_error("preprocess_bwd: an SH gradient sink needs SH input, no index remap, 3*M %% 4 == 0 and 16-byte aligned arrays");
      return HG_ERR_INVALID_ARG;
    }
  }
  if (sh_factor && (!in.shs || in.indices || in.parent_indices || sh_sink)) {
    set_error("preprocess_bwd: SH gradient factors need SH input, no index remap and no SH sink");
    return HG_ERR_INVALID_ARG;
  }
  if (pose_partial && (in.indices || in.parent_indices)) {
    set_error("preprocess_bwd: the camera pose gradient needs contiguous slots (no render or parent indices)");
    return HG_ERR_INVALID_ARG;
  }
  if (slot_begin % kThreads != 0 || slot_begin >= slot_end) {
    set_error("preprocess_bwd: bad slot range [%d, %d)", slot_begin, slot_end);
    return HG_ERR_INVALID_ARG;
  }
  auto kernel = pose_partial ? preprocess_bwd_kernel<true> : preprocess_bwd_kernel<false>;
  kernel<<<(slot_end - slot_begin + kThreads - 1) / kThreads, kThreads, 0, stream>>>(
      slot_end, slot_begin / kThreads, in.D, in.M, in.indices, in.parent_indices, in.ts, in.means3D, radii, in.shs, g.clamped,
      in.opacities, in.scales, in.rotations, in.scale_modifier, cov, in.cov3D_precomp != nullptr,
      in.viewmatrix, in.projmatrix, in.campos, focal_x, focal_y, in.tan_fovx, in.tan_fovy, accum,
      has_invdepth, prezeroed, dL_dmeans2D, dL_dconic, dL_dopacity, dL_dcolors, dL_dinvdepths,
      dL_dmeans3D, dL_dcov3D, dL_dsh, dL_dscales, dL_drotations, dL_dall_map, sh_sink, sh_beta, sh_factor, pose_partial);
  HG_POST_LAUNCH(in.debug, stream, pose_partial ? "preprocess_bwd_pose" : "preprocess_bwd");
  return HG_OK;
}

int preprocess_bwd_block_slots() { return kThreads; }

}  // namespace hg
