// preprocess.cu — per-Gaussian projection / covariance / SH colour / tile bounds.
//
// Replaces preprocessCUDA<3> of the reference (cuda_rasterizer/forward.cu:218-435)
// together with computeCov3D (:181-215), computeCov2D (:141-176),
// computeColorFromSH[Interp] (:25-138) and getRect/ndc2Pix/transformPoint*
// (auxiliary.h:53-102), plus the frustum test checkFrustum
// (rasterizer_impl.cu:54-66).
//
// Design (B200): one thread per rendered slot, 128-thread CTAs.  Every value
// that decides a sort key (depth bits, tile rectangle) or an alpha (conic,
// opacity) is computed with explicit __f*_rn intrinsics in exactly the
// operation order that nvcc 12.9 / ptxas emit for the reference source
// (verified against the reference's PTX and SASS), so that keys, radii and
// conics are bit-identical without depending on contraction heuristics.
// SH rows (192 B each) are fetched warp-cooperatively with coalesced LDG.128
// into shared memory and read back transposed; results go out as one 64-byte
// splat record per slot plus the SoA arrays the binning stage reads.
#include "common.cuh"
#include "tile_instances.cuh"
#include "sh_stage.cuh"

namespace hg {

namespace {

constexpr int kThreads = 128;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxShFloats = 48;              // M <= 16 coefficients x 3 channels
constexpr int kShStrideMax = kMaxShFloats + 1;  // odd stride => conflict-free transposed reads

struct ShSmem {
  const float* s;
  __device__ __forceinline__ float operator()(int k, int c) const { return s[k * 3 + c]; }
};
struct ShGlobal {
  const float* g;
  __device__ __forceinline__ float operator()(int k, int c) const { return __ldg(g + k * 3 + c); }
};
struct ShInterp {  // computeColorFromSHInterp / interp(), forward.cu:78-84
  const float* a;
  const float* b;
  float t;
  __device__ __forceinline__ float operator()(int k, int c) const {
    return t * __ldg(a + k * 3 + c) + (1.0f - t) * __ldg(b + k * 3 + c);
  }
};

// SH -> RGB (forward.cu:25-76).  Returns the unclamped-at-zero colour + 0.5.
template <typename F>
__device__ __forceinline__ void eval_sh(int deg, const F& sh, float dx, float dy, float dz,
                                        float* out) {
  const float len = sqrtf(dx * dx + dy * dy + dz * dz);
  const float x = dx / len, y = dy / len, z = dz / len;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float r = SH_C0 * sh(0, c);
    if (deg > 0) {
      r = r - SH_C1 * y * sh(1, c) + SH_C1 * z * sh(2, c) - SH_C1 * x * sh(3, c);
      if (deg > 1) {
        const float xx = x * x, yy = y * y, zz = z * z;
        const float xy = x * y, yz = y * z, xz = x * z;
        r = r + SH_C2_0 * xy * sh(4, c) + SH_C2_1 * yz * sh(5, c) +
            SH_C2_2 * (2.0f * zz - xx - yy) * sh(6, c) + SH_C2_3 * xz * sh(7, c) +
            SH_C2_4 * (xx - yy) * sh(8, c);
        if (deg > 2) {
          r = r + SH_C3_0 * y * (3.0f * xx - yy) * sh(9, c) + SH_C3_1 * xy * z * sh(10, c) +
              SH_C3_2 * y * (4.0f * zz - xx - yy) * sh(11, c) +
              SH_C3_3 * z * (2.0f * zz - 3.0f * xx - 3.0f * yy) * sh(12, c) +
              SH_C3_4 * x * (4.0f * zz - xx - yy) * sh(13, c) +
              SH_C3_5 * z * (xx - yy) * sh(14, c) + SH_C3_6 * x * (xx - 3.0f * yy) * sh(15, c);
        }
      }
    }
    out[c] = r + 0.5f;
  }
}


// Sigma = (S R)^T (S R) in the reference's exact operation order
// (forward.cu:181-215; PTX fma chains + the ptxas fusions of the quaternion
// products).  q = (r, x, y, z) is NOT normalised.
__device__ __forceinline__ void cov3d_ref(float sx, float sy, float sz, float mod, float r,
                                          float x, float y, float z, float* c) {
  const float s0 = __fmul_rn(mod, sx), s1 = __fmul_rn(mod, sy), s2 = __fmul_rn(mod, sz);
  const float yy = __fmul_rn(y, y), zz = __fmul_rn(z, z);
  const float rx = __fmul_rn(r, x), xz = __fmul_rn(z, x), rz = __fmul_rn(z, r);
  const float a_yz = __fadd_rn(yy, zz);          // y^2 + z^2
  const float a_xz = __fmaf_rn(x, x, zz);        // x^2 + z^2
  const float a_xy = __fmaf_rn(x, x, yy);        // x^2 + y^2
  const float yz_m_rx = __fmaf_rn(z, y, -rx);
  const float yz_p_rx = __fmaf_rn(z, y, rx);
  const float xz_p_ry = __fmaf_rn(y, r, xz);
  const float xz_m_ry = __fmaf_rn(y, -r, xz);
  const float xy_m_rz = __fmaf_rn(y, x, -rz);
  const float xy_p_rz = __fmaf_rn(y, x, rz);
  // Rotation matrix columns (glm column-major constructor order).
  const float R00 = __fsub_rn(1.0f, __fadd_rn(a_yz, a_yz));
  const float R01 = __fadd_rn(xy_m_rz, xy_m_rz);
  const float R02 = __fadd_rn(xz_p_ry, xz_p_ry);
  const float R10 = __fadd_rn(xy_p_rz, xy_p_rz);
  const float R11 = __fsub_rn(1.0f, __fadd_rn(a_xz, a_xz));
  const float R12 = __fadd_rn(yz_m_rx, yz_m_rx);
  const float R20 = __fadd_rn(xz_m_ry, xz_m_ry);
  const float R21 = __fadd_rn(yz_p_rx, yz_p_rx);
  const float R22 = __fsub_rn(1.0f, __fadd_rn(a_xy, a_xy));
  // M = S * R  (the zero terms of the diagonal S add exact zeros).
  const float M00 = __fmul_rn(s0, R00), M01 = __fmul_rn(s1, R01), M02 = __fmul_rn(s2, R02);
  const float M10 = __fmul_rn(s0, R10), M11 = __fmul_rn(s1, R11), M12 = __fmul_rn(s2, R12);
  const float M20 = __fmul_rn(s0, R20), M21 = __fmul_rn(s1, R21), M22 = __fmul_rn(s2, R22);
  // Sigma = M^T M, upper triangle.
  c[0] = __fmaf_rn(M02, M02, __fmaf_rn(M00, M00, __fmul_rn(M01, M01)));
  c[1] = __fmaf_rn(M12, M02, __fmaf_rn(M10, M00, __fmul_rn(M11, M01)));
  c[2] = __fmaf_rn(M22, M02, __fmaf_rn(M20, M00, __fmul_rn(M21, M01)));
  c[3] = __fmaf_rn(M12, M12, __fmaf_rn(M10, M10, __fmul_rn(M11, M11)));
  c[4] = __fmaf_rn(M22, M12, __fmaf_rn(M20, M10, __fmul_rn(M21, M11)));
  c[5] = __fmaf_rn(M22, M22, __fmaf_rn(M20, M20, __fmul_rn(M21, M21)));
}

// EWA projection of the 3-D covariance (forward.cu:141-176) in the reference's
// operation order.  v = view matrix (16 floats), t = view-space mean.
__device__ __forceinline__ void cov2d_ref(float tx, float ty, float tz, float focal_x,
                                          float focal_y, float tan_fovx, float tan_fovy,
                                          const float* c, const float* v, float& cxx, float& cxy,
                                          float& cyy) {
  const float limx = __fmul_rn(tan_fovx, 1.3f), limy = __fmul_rn(tan_fovy, 1.3f);
  const float txtz = __fdiv_rn(tx, tz), tytz = __fdiv_rn(ty, tz);
  const float ux = fminf(limx, fmaxf(-limx, txtz));
  const float uy = fminf(limy, fmaxf(-limy, tytz));
  const float tz2 = __fmul_rn(tz, tz);
  const float J00 = __fdiv_rn(focal_x, tz);
  const float J02 = __fdiv_rn(__fmul_rn(focal_x, __fmul_rn(ux, -tz)), tz2);
  const float J11 = __fdiv_rn(focal_y, tz);
  const float J12 = __fdiv_rn(__fmul_rn(focal_y, __fmul_rn(uy, -tz)), tz2);
  // T = W * J (third column of J is zero).
  const float T00 = __fmaf_rn(v[2], J02, __fmul_rn(v[0], J00));
  const float T01 = __fmaf_rn(v[6], J02, __fmul_rn(v[4], J00));
  const float T02 = __fmaf_rn(v[10], J02, __fmul_rn(v[8], J00));
  const float T10 = __fmaf_rn(v[2], J12, __fmul_rn(v[1], J11));
  const float T11 = __fmaf_rn(v[6], J12, __fmul_rn(v[5], J11));
  const float T12 = __fmaf_rn(v[10], J12, __fmul_rn(v[9], J11));
  // A = T^T * Vrk^T
  const float A00 = __fmaf_rn(T02, c[2], __fmaf_rn(T00, c[0], __fmul_rn(T01, c[1])));
  const float A01 = __fmaf_rn(T12, c[2], __fmaf_rn(T10, c[0], __fmul_rn(T11, c[1])));
  const float A10 = __fmaf_rn(T02, c[4], __fmaf_rn(T00, c[1], __fmul_rn(T01, c[3])));
  const float A11 = __fmaf_rn(T12, c[4], __fmaf_rn(T10, c[1], __fmul_rn(T11, c[3])));
  const float A20 = __fmaf_rn(T02, c[5], __fmaf_rn(T00, c[2], __fmul_rn(T01, c[4])));
  const float A21 = __fmaf_rn(T12, c[5], __fmaf_rn(T10, c[2], __fmul_rn(T11, c[4])));
  // cov = A * T
  cxx = __fmaf_rn(T02, A20, __fmaf_rn(T00, A00, __fmul_rn(T01, A10)));
  cxy = __fmaf_rn(T02, A21, __fmaf_rn(T00, A01, __fmul_rn(T01, A11)));
  cyy = __fmaf_rn(T12, A21, __fmaf_rn(T10, A01, __fmul_rn(T11, A11)));
}

__global__ void __launch_bounds__(kThreads)
preprocess_fwd_kernel(const int P, const int N, const int D, const int M,
                      const int* __restrict__ indices, const int* __restrict__ parent_indices,
                      const float* __restrict__ ts, const float* __restrict__ means3D,
                      const float* __restrict__ scales, const float scale_modifier,
                      const float* __restrict__ rotations, const float* __restrict__ opacities,
                      const float* __restrict__ shs, const float* __restrict__ cov3D_precomp,
                      const float* __restrict__ colors_precomp,
                      const float* __restrict__ all_map, const float* __restrict__ viewmatrix,
                      const float* __restrict__ projmatrix, const float* __restrict__ campos,
                      const int W, const int H, const float tan_fovx, const float tan_fovy,
                      const float focal_x, const float focal_y, const uint32_t grid_x,
                      const uint32_t grid_y, int* __restrict__ radii,
                      int* __restrict__ out_observe, float* __restrict__ depths,
                      uint32_t* __restrict__ tiles_touched, uint2* __restrict__ rects,
                      float* __restrict__ cov3Ds, uint8_t* __restrict__ clamped,
                      float4* __restrict__ records, uint32_t* __restrict__ tile_ctr,
                      const int ctr_stride) {
  __shared__ float s_sh[kWarps][32 * kShStrideMax];

  const int t_idx = blockIdx.x * kThreads + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const bool in_range = t_idx < P;

  bool alive = in_range;
  float pre_s[3] = {0.f, 0.f, 0.f}, pre_o = 0.f, pre_am[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  float4 pre_q = make_float4(0.f, 0.f, 0.f, 0.f);
  int r_idx = 0, p_idx = -1;
  float t = 0.0f;
  bool has_parent = false;
  float px = 0, py = 0, pz = 0;     // (possibly parent-interpolated) world mean
  float depth = 0, pix_x = 0, pix_y = 0;
  float conic_a = 0, conic_b = 0, conic_c = 0, opac = 0;
  uint32_t minx = 0, miny = 0, maxx = 0, maxy = 0;
  int my_radius = 0;

  if (in_range) {
    r_idx = indices ? __ldg(indices + t_idx) : t_idx;
    radii[t_idx] = 0;
    tiles_touched[t_idx] = 0;
    out_observe[t_idx] = 0;

    px = __ldg(means3D + 3 * (size_t)r_idx);
    py = __ldg(means3D + 3 * (size_t)r_idx + 1);
    pz = __ldg(means3D + 3 * (size_t)r_idx + 2);
    // Everything else this slot will need is requested now, next to the mean (one round trip instead of a chain of
    // dependent ones; culled slots pay ~32 bytes of traffic that share their neighbours' sectors anyway).
    if (cov3D_precomp == nullptr) {
      pre_s[0] = __ldg(scales + 3 * (size_t)r_idx);
      pre_s[1] = __ldg(scales + 3 * (size_t)r_idx + 1);
      pre_s[2] = __ldg(scales + 3 * (size_t)r_idx + 2);
      pre_q = __ldg((const float4*)rotations + r_idx);
    }
    pre_o = __ldg(opacities + r_idx);
    if (all_map) {
#pragma unroll
      for (int c = 0; c < 5; ++c) pre_am[c] = __ldg(all_map + 5 * (size_t)t_idx + c);
    }
    if (parent_indices) {
      p_idx = __ldg(parent_indices + t_idx);
      if (p_idx != -1) {
        has_parent = true;
        t = __ldg(ts + t_idx);
        const float omt = __fsub_rn(1.0f, t);
        px = __fmaf_rn(px, t, __fmul_rn(omt, __ldg(means3D + 3 * (size_t)p_idx)));
        py = __fmaf_rn(py, t, __fmul_rn(omt, __ldg(means3D + 3 * (size_t)p_idx + 1)));
        pz = __fmaf_rn(pz, t, __fmul_rn(omt, __ldg(means3D + 3 * (size_t)p_idx + 2)));
      }
    }

    float v[16], pm[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      v[i] = __ldg(viewmatrix + i);
      pm[i] = __ldg(projmatrix + i);
    }

    // Screen-space position and view depth (forward.cu:311-317).
    const float hx = __fadd_rn(pm[12], dot3_ref(pm[0], pm[4], pm[8], px, py, pz));
    const float hy = __fadd_rn(pm[13], dot3_ref(pm[1], pm[5], pm[9], px, py, pz));
    const float hw = __fadd_rn(pm[15], dot3_ref(pm[3], pm[7], pm[11], px, py, pz));
    const float p_w = __frcp_rn(__fadd_rn(hw, 0.0000001f));
    const float proj_x = __fmul_rn(hx, p_w), proj_y = __fmul_rn(hy, p_w);
    depth = __fadd_rn(v[14], dot3_ref(v[2], v[6], v[10], px, py, pz));
    alive = !(depth <= 0.2f);  // NaN passes, as in the reference's `<=` test

    if (alive) {
      float c3[6];
      if (cov3D_precomp == nullptr) {
        float sx = pre_s[0], sy = pre_s[1], sz = pre_s[2];
        const float4 q4 = pre_q;
        float qr = q4.x, qx = q4.y, qy = q4.z, qz = q4.w;
        if (has_parent) {  // forward.cu:332-343
          const float omt = __fsub_rn(1.0f, t);
          sx = __fmaf_rn(t, sx, __fmul_rn(omt, __ldg(scales + 3 * (size_t)p_idx)));
          sy = __fmaf_rn(t, sy, __fmul_rn(omt, __ldg(scales + 3 * (size_t)p_idx + 1)));
          sz = __fmaf_rn(t, sz, __fmul_rn(omt, __ldg(scales + 3 * (size_t)p_idx + 2)));
          float4 o4 = __ldg((const float4*)rotations + p_idx);
          const float dotp = __fadd_rn(__fmaf_rn(qr, o4.x, __fmul_rn(qx, o4.y)),
                                       __fmaf_rn(qy, o4.z, __fmul_rn(qz, o4.w)));
          if (dotp < 0.0f) { o4.x = -o4.x; o4.y = -o4.y; o4.z = -o4.z; o4.w = -o4.w; }
          qr = __fmaf_rn(t, qr, __fmul_rn(omt, o4.x));
          qx = __fmaf_rn(t, qx, __fmul_rn(omt, o4.y));
          qy = __fmaf_rn(t, qy, __fmul_rn(omt, o4.z));
          qz = __fmaf_rn(t, qz, __fmul_rn(omt, o4.w));
        }
        cov3d_ref(sx, sy, sz, scale_modifier, qr, qx, qy, qz, c3);
#pragma unroll
        for (int i = 0; i < 6; ++i) cov3Ds[6 * (size_t)t_idx + i] = c3[i];
      } else {
        // The reference leaves its cov3D pointer unset on this path
        // (forward.cu:326-350); we use the precomputed matrix of the source row
        // as the original 3DGS rasterizer does.
#pragma unroll
        for (int i = 0; i < 6; ++i) c3[i] = __ldg(cov3D_precomp + 6 * (size_t)r_idx + i);
      }

      const float tx = __fadd_rn(v[12], dot3_ref(v[0], v[4], v[8], px, py, pz));
      const float ty = __fadd_rn(v[13], dot3_ref(v[1], v[5], v[9], px, py, pz));
      float cxx, cxy, cyy;
      cov2d_ref(tx, ty, depth, focal_x, focal_y, tan_fovx, tan_fovy, c3, v, cxx, cxy, cyy);

      // Dilation 0.1 and anti-aliasing scale (forward.cu:355-364).
      const float cxy2 = __fmul_rn(cxy, cxy);
      const float det_cov = __fmaf_rn(cxx, cyy, -cxy2);
      const float dxx = __fadd_rn(cxx, 0.1f), dyy = __fadd_rn(cyy, 0.1f);
      const float det = __fmaf_rn(dxx, dyy, -cxy2);
      const float h_scale = __fsqrt_rn(fmaxf(0.000025f, __fdiv_rn(det_cov, det)));
      alive = det != 0.0f;
      if (alive) {
        const float det_inv = __frcp_rn(det);
        conic_a = __fmul_rn(dyy, det_inv);
        conic_b = __fmul_rn(-cxy, det_inv);
        conic_c = __fmul_rn(dxx, det_inv);
        const float mid = __fmul_rn(0.5f, __fadd_rn(dxx, dyy));
        const float disc = __fsqrt_rn(fmaxf(0.1f, __fmaf_rn(mid, mid, -det)));
        const float lam = fmaxf(__fadd_rn(mid, disc), __fsub_rn(mid, disc));
        my_radius = __float2int_rz(ceilf(__fmul_rn(3.0f, __fsqrt_rn(lam))));
        pix_x = ndc2pix_ref(proj_x, W);
        pix_y = ndc2pix_ref(proj_y, H);
        // rects path of the reference (forward.cu:390-395), always active.
        const int ex = __float2int_rz(ceilf(__fmul_rn(3.0f, __fsqrt_rn(dxx))));
        const int ey = __float2int_rz(ceilf(__fmul_rn(3.0f, __fsqrt_rn(dyy))));
        get_rect_ref(pix_x, pix_y, ex, ey, grid_x, grid_y, minx, miny, maxx, maxy);
        alive = ((maxx - minx) * (maxy - miny)) != 0;
        float o = pre_o;
        if (has_parent) o = __fmaf_rn(t, o, __fmul_rn(__fsub_rn(1.0f, t), __ldg(opacities + p_idx)));
        opac = __fmul_rn(o, h_scale);
      }
    }
  }

  // ---- colour ---------------------------------------------------------------
  float rgb[3] = {0.f, 0.f, 0.f};
  uint8_t clamp_bits = 0;
  const bool need_sh = (colors_precomp == nullptr);
  if (need_sh) {
    const int row = M * 3;
    // Fast path: rows of this warp are contiguous -> coalesced staging.  The float4 staging skips the float4s of
    // culled rows, which is only exact when no float4 straddles two rows (row % 4 == 0), and needs 16-byte aligned
    // shs; other widths and misaligned views are staged float by float.  Either way the colour comes from the one
    // eval_sh below, so a view of the same rows at another alignment gives the same bits.
    const bool staged = (indices == nullptr) && (parent_indices == nullptr);
    if (staged) {
      const unsigned any = __ballot_sync(0xffffffffu, alive);
      if (any) {
        const int stride = row | 1;
        const int warp_first = blockIdx.x * kThreads + warp * 32;
        const size_t base = (size_t)warp_first * row;         // float index of the warp's first row
        const size_t total = (size_t)N * row;
        float* dst = s_sh[warp];
        // rows of culled slots are skipped
        if ((row & 3) == 0 && (reinterpret_cast<uintptr_t>(shs) & 15) == 0) {
          if (row == 48) stage_sh_rows<48>(shs, base, total, row, lane, dst, any);
          else stage_sh_rows<0>(shs, base, total, row, lane, dst, any);
        } else {
          stage_sh_rows_scalar(shs, base, total, row, lane, dst, any);
        }
        __syncwarp();
        if (alive) {
          const float cx = __ldg(campos), cy = __ldg(campos + 1), cz = __ldg(campos + 2);
          eval_sh(D, ShSmem{dst + lane * stride}, px - cx, py - cy, pz - cz, rgb);
        }
      }
    } else if (alive) {
      const float cx = __ldg(campos), cy = __ldg(campos + 1), cz = __ldg(campos + 2);
      // Direction uses the un-interpolated source mean (forward.cu:30,91).
      const float ox = __ldg(means3D + 3 * (size_t)r_idx), oy = __ldg(means3D + 3 * (size_t)r_idx + 1),
                  oz = __ldg(means3D + 3 * (size_t)r_idx + 2);
      if (has_parent)
        eval_sh(D, ShInterp{shs + (size_t)r_idx * row, shs + (size_t)p_idx * row, t}, ox - cx,
                oy - cy, oz - cz, rgb);
      else
        eval_sh(D, ShGlobal{shs + (size_t)r_idx * row}, ox - cx, oy - cy, oz - cz, rgb);
    }
    if (alive) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        if (rgb[c] < 0.0f) clamp_bits |= (1u << c);
        rgb[c] = fmaxf(rgb[c], 0.0f);
      }
    }
  } else if (alive) {
#pragma unroll
    for (int c = 0; c < 3; ++c) rgb[c] = __ldg(colors_precomp + 3 * (size_t)t_idx + c);
  }

  // Instances per tile (the bucket sizes of binning.cu): one RED per (splat, tile), the warp's instances spread evenly
  // over its lanes whatever the rectangle sizes.
  {
    const uint32_t width = maxx - minx;
    const WarpInstances wi(alive ? width * (maxy - miny) : 0u, minx | (miny << 16), width, lane);
    for (uint32_t j0 = 0; j0 < wi.total; j0 += 32) {
      int owner;
      uint32_t tile;
      if (wi.at(j0, grid_x, owner, tile)) atomicAdd(tile_ctr + (size_t)tile * ctr_stride, 1u);
    }
  }
  if (!alive) return;

  const float* am = pre_am;
  depths[t_idx] = depth;
  radii[t_idx] = my_radius;
  rects[t_idx] = make_uint2(minx | (miny << 16), maxx | (maxy << 16));
  // With a parent the reference records the clamp flags in `p_clamped` (forward.cu:411) but its
  // backward reads `clamped` (backward.cu:453), which that path never wrote: the flags are
  // effectively "not clamped".  We store exactly that instead of uninitialised memory.
  clamped[t_idx] = has_parent ? (uint8_t)0 : clamp_bits;
  tiles_touched[t_idx] = (maxy - miny) * (maxx - minx);
  float4* rec = records + 4 * (size_t)t_idx;
  rec[0] = make_float4(pix_x, pix_y, conic_a, conic_b);
  rec[1] = make_float4(conic_c, opac, rgb[0], rgb[1]);
  rec[2] = make_float4(rgb[2], __frcp_rn(depth), am[0], am[1]);
  rec[3] = make_float4(am[2], am[3], am[4], __int_as_float(t_idx));  // the record carries its own slot id
}

__global__ void mark_visible_kernel(int P, const float* __restrict__ means3D,
                                    const float* __restrict__ viewmatrix,
                                    uint8_t* __restrict__ present) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= P) return;
  const float x = means3D[3 * (size_t)idx], y = means3D[3 * (size_t)idx + 1],
              z = means3D[3 * (size_t)idx + 2];
  const float d = __fadd_rn(__ldg(viewmatrix + 14),
                            dot3_ref(__ldg(viewmatrix + 2), __ldg(viewmatrix + 6),
                                     __ldg(viewmatrix + 10), x, y, z));
  present[idx] = (d <= 0.2f) ? 0 : 1;
}

}  // namespace

int launch_preprocess_fwd(const hg_raster_inputs& in, const GeomState& g, int* radii,
                          int* out_observe, dim3 grid, float focal_x, float focal_y,
                          cudaStream_t stream) {
  const int blocks = (in.P + kThreads - 1) / kThreads;
  preprocess_fwd_kernel<<<blocks, kThreads, 0, stream>>>(
      in.P, in.N, in.D, in.M, in.indices, in.parent_indices, in.ts, in.means3D, in.scales,
      in.scale_modifier, in.rotations, in.opacities, in.shs, in.cov3D_precomp, in.colors_precomp,
      in.all_map, in.viewmatrix, in.projmatrix, in.campos, in.W, in.H, in.tan_fovx, in.tan_fovy,
      focal_x, focal_y, grid.x, grid.y, radii, out_observe, g.depths, g.tiles_touched, g.rects,
      g.cov3D, g.clamped, g.records, g.tile_ctr, g.ctr_stride);
  HG_POST_LAUNCH(in.debug, stream, "preprocess_fwd");
  return HG_OK;
}

int launch_mark_visible(int P, const float* means3D, const float* viewmatrix,
                        const float* projmatrix, uint8_t* present, cudaStream_t stream) {
  (void)projmatrix;
  if (P <= 0) return HG_OK;
  mark_visible_kernel<<<(P + 255) / 256, 256, 0, stream>>>(P, means3D, viewmatrix, present);
  HG_POST_LAUNCH(false, stream, "mark_visible");
  return HG_OK;
}

}  // namespace hg
