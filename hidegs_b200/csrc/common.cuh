// common.cuh — shared definitions of the B200-native HiDeGS rasterizer.
//
// State layout (our own; opaque to callers, see hg_raster_layout):
//   geometry buffer : depths f32[P] | tiles_touched u32[P] | point_offsets u32[P] (diagnostics only)
//                     | rects u32[P,2] (packed tile bounds) | cov3D f32[P,6]
//                     | clamped u8[P] | records f32[P,16]
//                     | tile_ctr u32[T, stride] (count, cursor) | list_a u32[T] | list_b u32[T] | xl_off u32[T]
//                     | binning header u32[16]
//   image buffer    : final_T f32[HW] | n_contrib u32[HW] | ranges u32[T,2]
//   binning buffer  : vals u32[R] (= point_list) | pairs u32[R,2] (depth bits, slot; bucketed by tile)
//                     | scratch for lists beyond shared memory (binning.cu)
//
// Splat record (64 B, one per rendered slot, written by preprocess, gathered by
// both blend kernels with four LDG.128):
//   [0] x  [1] y  [2] conic.a  [3] conic.b | [4] conic.c  [5] opacity*AA  [6] r  [7] g
//   [8] b  [9] 1/depth  [10] am0  [11] am1 | [12] am2  [13] am3  [14] am4  [15] slot id (bits)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include "../../include/hidegs_raster.h"

#define HG_BLOCK_SIZE (HG_BLOCK_X * HG_BLOCK_Y)
#define HG_REC_FLOATS 16

namespace hg {

// ---- error plumbing ---------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define HG_CUDA_TRY(expr)                                                        \
  do {                                                                           \
    cudaError_t _e = (expr);                                                     \
    if (_e != cudaSuccess) {                                                     \
      hg::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__,         \
                    cudaGetErrorString(_e));                                     \
      return HG_ERR_CUDA;                                                        \
    }                                                                            \
  } while (0)

// After a kernel launch: always catch launch-config errors; in debug mode also
// synchronise (mirrors CHECK_CUDA of the reference, auxiliary.h:23-30).
#define HG_POST_LAUNCH(debug, stream, what)                                      \
  do {                                                                           \
    hg::count_launch();                                                          \
    cudaError_t _e = cudaGetLastError();                                         \
    if (_e == cudaSuccess && (debug)) _e = cudaStreamSynchronize(stream);        \
    if (_e != cudaSuccess) {                                                     \
      hg::set_error("kernel %s failed: %s", what, cudaGetErrorString(_e));       \
      return HG_ERR_CUDA;                                                        \
    }                                                                            \
  } while (0)

// ---- layout -----------------------------------------------------------------
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct GeomState {
  float* depths;
  uint32_t* tiles_touched;
  uint32_t* point_offsets;
  uint2* rects;
  float* cov3D;
  uint8_t* clamped;
  float4* records;
  uint32_t* tile_ctr;     // per tile, `ctr_stride` words apart: [0] instances (REDs of preprocess_fwd), [1] list offset,
                          // after the scatter the END of its list
  int ctr_stride;
  uint32_t* list_a;       // short lists from the front, medium lists from the back
  uint32_t* list_b;       // long lists from the front, lists beyond shared memory from the back
  uint32_t* xl_off;       // scratch offset (in pairs) of the k-th list beyond shared memory
  uint32_t* bin_header;   // see tile_scan_kernel
};
struct ImageState {
  float* final_T;
  uint32_t* n_contrib;
  uint2* ranges;
};
struct BinState {
  uint32_t* vals;     // point_list
  uint2* pairs;       // (depth bits, slot) of every instance, bucketed by tile
  uint32_t* scratch;  // only for lists beyond shared memory
};

size_t binning_scratch_bytes(uint32_t beyond_pairs);

static inline GeomState geom_from(char* base, const hg_raster_layout& L) {
  GeomState g;
  g.depths = (float*)(base + L.depths);
  g.tiles_touched = (uint32_t*)(base + L.tiles_touched);
  g.point_offsets = (uint32_t*)(base + L.point_offsets);
  g.rects = (uint2*)(base + L.rects);
  g.cov3D = (float*)(base + L.cov3D);
  g.clamped = (uint8_t*)(base + L.clamped);
  g.records = (float4*)(base + L.records);
  g.tile_ctr = (uint32_t*)(base + L.tile_ctr);
  g.ctr_stride = (int)L.ctr_stride;
  g.list_a = (uint32_t*)(base + L.tile_lists);
  g.list_b = g.list_a + L.tiles;
  g.xl_off = g.list_b + L.tiles;
  g.bin_header = (uint32_t*)(base + L.bin_header);
  return g;
}
static inline ImageState image_from(char* base, const hg_raster_layout& L) {
  ImageState s;
  s.final_T = (float*)(base + L.final_T);
  s.n_contrib = (uint32_t*)(base + L.n_contrib);
  s.ranges = (uint2*)(base + L.ranges);
  return s;
}
static inline BinState bin_from(char* base, const hg_raster_layout& L) {
  BinState b;
  b.vals = (uint32_t*)(base + L.vals);
  b.pairs = (uint2*)(base + L.pairs);
  b.scratch = (uint32_t*)(base + L.binning_bytes);
  return b;
}

// Buffers handed out by torch are 512-B aligned; we align every sub-array to
// 256 B relative to the base, and the base itself is re-aligned by the caller.
static inline char* align_ptr(char* p, size_t a) {
  return (char*)(((uintptr_t)p + a - 1) / a * a);
}

// ---- per-Gaussian accumulator row written by the backward blend -------------
//   [0..2] dL/drgb  [3] dL/dinvdepth  [4..8] dL/dall_map  [9] dL/dmean2D.x
//   [10] dL/dmean2D.y  [11] dL/dconic.xx  [12] dL/dconic.xy  [13] dL/dconic.yy
//   [14] dL/dopacity (w.r.t. opacity*AA)  [15] unused
#define HG_ACC_FLOATS 16

// ---- kernels launchers (one per translation unit) ---------------------------
int launch_preprocess_fwd(const hg_raster_inputs& in, const GeomState& g, int* radii,
                          int* out_observe, dim3 grid, float focal_x, float focal_y,
                          cudaStream_t stream);
int launch_tile_scan(const GeomState& g, const ImageState& img, int T, uint32_t* host_header, cudaStream_t stream,
                     bool debug);
int launch_debug_keys(int P, int T, const GeomState& g, const BinState& b, const int* radii, int R,
                      dim3 grid, uint64_t* keys_unsorted, uint32_t* vals_unsorted, uint64_t* keys_sorted,
                      cudaStream_t stream);
int launch_binning(const hg_raster_inputs& in, const GeomState& g, const BinState& b, int T, dim3 grid,
                   const uint32_t* header_host, cudaStream_t stream);
int launch_blend_fwd(const hg_raster_inputs& in, const GeomState& g, const BinState& b,
                     const ImageState& img, dim3 grid, float focal_x, float focal_y,
                     float* out_color, float* out_invdepth, int* out_observe, float* out_all_map,
                     float* out_plane_depth, bool empty_scene, cudaStream_t stream);
int launch_blend_bwd(const hg_raster_inputs& in, const GeomState& g, const BinState& b,
                     const ImageState& img, dim3 grid, float focal_x, float focal_y,
                     const float* all_map_pixels, const float* dL_dpix,
                     const float* dL_dout_all_map, const float* dL_dout_plane_depth,
                     const float* dL_dout_invdepth, float* accum, cudaStream_t stream);
int launch_preprocess_bwd(const hg_raster_inputs& in, const GeomState& g, const int* radii,
                          float focal_x, float focal_y, const float* accum, bool has_invdepth,
                          float* dL_dmeans2D, float* dL_dconic, float* dL_dopacity,
                          float* dL_dcolors, float* dL_dinvdepths, float* dL_dmeans3D,
                          float* dL_dcov3D, float* dL_dsh, float* dL_dscales,
                          float* dL_drotations, float* dL_dall_map, cudaStream_t stream, int slot_begin = 0,
                          int slot_end = -1, float* sh_sink = nullptr, float sh_beta = 0.f,
                          float* sh_factor = nullptr, bool skip_culled_rows = false,
                          double* pose_partial = nullptr);
// Camera pose gradient partials (camera_pose.cu): one row of kPosePartialStride doubles ([0..2] dL/drho, [3..5] the
// torque) per CTA of the pose variants of the per-Gaussian backward (128-slot CTAs) and of the prologue backward
// (256-row CTAs).  The CTA counts depend on the Gaussian count only.
constexpr int kPosePartialStride = 8;
constexpr int kPoseRasterSlots = 128;
constexpr int kPosePrologueRows = 256;
// pose workspace of N Gaussians: [rasterizer partials | prologue partials], each part 256-byte aligned
static inline size_t camera_pose_prologue_offset(int64_t N) {
  return align_up((size_t)((N + kPoseRasterSlots - 1) / kPoseRasterSlots) * kPosePartialStride * sizeof(double), 256);
}
static inline size_t camera_pose_workspace_bytes(int64_t N) {
  return camera_pose_prologue_offset(N) +
         align_up((size_t)((N + kPosePrologueRows - 1) / kPosePrologueRows) * kPosePartialStride * sizeof(double), 256);
}
int launch_sh_from_factors(int N, int D, int M, int n_views, const float* means3D, const float* factors,
                           size_t view_stride, float* dL_dsh, float beta, cudaStream_t stream);
int preprocess_bwd_block_slots();
int launch_mark_visible(int P, const float* means3D, const float* viewmatrix,
                        const float* projmatrix, uint8_t* present, cudaStream_t stream);

// ---- device helpers -----------------------------------------------------------
#ifdef __CUDACC__

// Spherical-harmonics constants (auxiliary.h:34-51).
__device__ constexpr float SH_C0 = 0.28209479177387814f;
__device__ constexpr float SH_C1 = 0.4886025119029199f;
__device__ constexpr float SH_C2_0 = 1.0925484305920792f;
__device__ constexpr float SH_C2_1 = -1.0925484305920792f;
__device__ constexpr float SH_C2_2 = 0.31539156525252005f;
__device__ constexpr float SH_C2_3 = -1.0925484305920792f;
__device__ constexpr float SH_C2_4 = 0.5462742152960396f;
__device__ constexpr float SH_C3_0 = -0.5900435899266435f;
__device__ constexpr float SH_C3_1 = 2.890611442640554f;
__device__ constexpr float SH_C3_2 = -0.4570457994644658f;
__device__ constexpr float SH_C3_3 = 0.3731763325901154f;
__device__ constexpr float SH_C3_4 = -0.4570457994644658f;
__device__ constexpr float SH_C3_5 = 1.445305721320277f;
__device__ constexpr float SH_C3_6 = -0.5900435899266435f;

// m[a]*x + m[b]*y + m[c]*z as the reference's compiled code evaluates it
// (auxiliary.h:83-102 after nvcc contraction): fma(z, mc, fma(x, ma, y*mb)).
__device__ __forceinline__ float dot3_ref(float ma, float mb, float mc, float x, float y, float z) {
  return __fmaf_rn(z, mc, __fmaf_rn(x, ma, __fmul_rn(y, mb)));
}

// ndc2Pix (auxiliary.h:53-56): evaluated in double, fma-contracted.
__device__ __forceinline__ float ndc2pix_ref(float v, int S) {
  return (float)__dmul_rn(__fma_rn(__dadd_rn((double)v, 1.0), (double)S, -1.0), 0.5);
}

// Tile bounds from a pixel centre and an integer extent (auxiliary.h:70-80).
__device__ __forceinline__ void get_rect_ref(float px, float py, int ex, int ey, uint32_t gx,
                                             uint32_t gy, uint32_t& minx, uint32_t& miny,
                                             uint32_t& maxx, uint32_t& maxy) {
  const float fx = (float)ex, fy = (float)ey;
  minx = min(gx, (uint32_t)max(0, __float2int_rz(__fmul_rn(__fsub_rn(px, fx), 0.0625f))));
  miny = min(gy, (uint32_t)max(0, __float2int_rz(__fmul_rn(__fsub_rn(py, fy), 0.0625f))));
  maxx = min(gx, (uint32_t)max(0, __float2int_rz(__fmul_rn(
                     __fadd_rn(__fadd_rn(__fadd_rn(px, fx), 16.0f), -1.0f), 0.0625f))));
  maxy = min(gy, (uint32_t)max(0, __float2int_rz(__fmul_rn(
                     __fadd_rn(__fadd_rn(__fadd_rn(py, fy), 16.0f), -1.0f), 0.0625f))));
}

#endif  // __CUDACC__

}  // namespace hg
