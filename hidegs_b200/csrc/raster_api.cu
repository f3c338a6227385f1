// raster_api.cu — extern "C" entry points (see include/hidegs_raster.h).
//
// Host-side orchestration that replaces CudaRasterizer::Rasterizer::forward /
// backward (cuda_rasterizer/rasterizer_impl.cu:203-405, 409-535).
#include "common.cuh"
#include "../../include/hidegs_exchange.h"

#include <cstdlib>

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <atomic>
#include <mutex>
#include <vector>

namespace hg {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

static constexpr size_t kAlign = 256;

// ---- optional per-stage device timing (CUDA events on the launch stream) ------
// Events are only recorded while profiling is enabled and are resolved lazily in
// hg_profile_collect(), so the timed region gains no host synchronisation.
static std::atomic<int> g_prof_on{0};
static std::mutex g_prof_mu;
struct ProfRec { int stage; cudaEvent_t a, b; };
static std::vector<ProfRec> g_prof;

struct StageTimer {
  int stage; cudaStream_t st; cudaEvent_t a = nullptr, b = nullptr; bool on;
  StageTimer(int stage_, cudaStream_t st_) : stage(stage_), st(st_), on(g_prof_on.load() != 0) {
    if (on) {
      if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) { on = false; return; }
      cudaEventRecord(a, st);
    }
  }
  ~StageTimer() {
    if (on) {
      cudaEventRecord(b, st);
      std::lock_guard<std::mutex> lk(g_prof_mu);
      g_prof.push_back({stage, a, b});
    }
  }
};

// Pinned landing slot for the binning header (num_rendered + list counts) and the event that signals its arrival (one per host thread and device).
struct HostSlot { uint32_t* value = nullptr; uint32_t* device_value = nullptr; cudaEvent_t ready = nullptr; int device = -1; };
static HostSlot* host_slot() {
  static thread_local HostSlot slots[16];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) { set_error("cudaGetDevice failed"); return nullptr; }
  HostSlot& s = slots[dev];
  if (s.device != dev) {
    if (cudaHostAlloc((void**)&s.value, 64, cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer((void**)&s.device_value, s.value, 0) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.ready, cudaEventDisableTiming) != cudaSuccess) {
      set_error("allocating the pinned num_rendered slot failed: %s", cudaGetErrorString(cudaGetLastError()));
      return nullptr;
    }
    s.device = dev;
  }
  return &s;
}

static void fill_layout(int32_t P, int32_t W, int32_t H, int64_t R, hg_raster_layout* L) {
  memset(L, 0, sizeof(*L));
  const size_t p = (size_t)(P > 0 ? P : 0);
  const size_t hw = (size_t)W * H;
  const size_t tiles = (size_t)((W + HG_BLOCK_X - 1) / HG_BLOCK_X) * ((H + HG_BLOCK_Y - 1) / HG_BLOCK_Y);
  const size_t r = (size_t)(R > 0 ? R : 0);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t at = off;
    off = align_up(off + bytes, kAlign);
    return at;
  };
  // geometry
  L->depths = take(p * 4);
  L->tiles_touched = take(p * 4);
  L->point_offsets = take(p * 4);
  L->rects = take(p * 8);
  L->cov3D = take(p * 24);
  L->clamped = take(p);
  L->records = take(p * HG_REC_FLOATS * 4);
  L->tiles = tiles;
  // (count, cursor) interleaved.  Measured and dropped: one 128-byte line per tile — the REDs / atomics do not run
  // faster, and zero-filling and scanning 1 MB instead of 64 KB cost 15 us.
  L->ctr_stride = 2;
  L->tile_ctr = take(tiles * L->ctr_stride * 4);
  L->tile_lists = take(tiles * 12);
  L->bin_header = take(64);
  L->geom_bytes = off + kAlign;
  // image
  off = 0;
  L->final_T = take(hw * 4);
  L->n_contrib = take(hw * 4);
  L->ranges = take(tiles * 8);
  L->image_bytes = off + kAlign;
  // binning
  off = 0;
  L->vals = take(r * 4);  // first: the backward only needs the sorted list
  L->pairs = take(r * 8);
  L->binning_bytes = off + kAlign;
}

static int validate(const hg_raster_inputs* in) {
  if (!in) { set_error("inputs is NULL"); return HG_ERR_INVALID_ARG; }
  if (in->P < 0 || in->N < 0 || in->W <= 0 || in->H <= 0) {
    set_error("bad sizes P=%d N=%d W=%d H=%d", in->P, in->N, in->W, in->H);
    return HG_ERR_INVALID_ARG;
  }
  if (in->W > 65535 * HG_BLOCK_X || in->H > 65535 * HG_BLOCK_Y) {
    set_error("image too large for the 16-bit tile rectangle encoding");
    return HG_ERR_INVALID_ARG;
  }
  if (in->P == 0) return HG_OK;
  if (!in->means3D || !in->opacities || !in->background || !in->viewmatrix || !in->projmatrix ||
      !in->campos) {
    set_error("a mandatory pointer (means3D/opacities/bg/view/proj/campos) is NULL");
    return HG_ERR_INVALID_ARG;
  }
  if ((in->shs == nullptr) == (in->colors_precomp == nullptr)) {
    set_error("Please provide excatly one of either SHs or precomputed colors!");
    return HG_ERR_INVALID_ARG;
  }
  const bool has_sr = in->scales != nullptr && in->rotations != nullptr;
  if (has_sr == (in->cov3D_precomp != nullptr) || ((in->scales != nullptr) != (in->rotations != nullptr))) {
    set_error("Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!");
    return HG_ERR_INVALID_ARG;
  }
  if (reinterpret_cast<uintptr_t>(in->rotations) & 15) {  // read as one float4 per Gaussian
    set_error("rotations must be 16-byte aligned (got %p)", (const void*)in->rotations);
    return HG_ERR_INVALID_ARG;
  }
  if (in->shs && (in->M <= 0 || in->M > 16 || in->D < 0 || (in->D + 1) * (in->D + 1) > in->M)) {
    set_error("SH degree %d does not fit %d coefficients (max 16)", in->D, in->M);
    return HG_ERR_INVALID_ARG;
  }
  if (in->parent_indices && !in->ts) {
    set_error("parent_indices given without interpolation weights");
    return HG_ERR_INVALID_ARG;
  }
  return HG_OK;
}

}  // namespace hg

using namespace hg;

extern "C" {

const char* hg_last_error(void) { return g_err; }
const char* hg_version(void) { return "hidegs_b200 0.1.0 sm_100a"; }
int64_t hg_launch_count(void) { return (int64_t)g_launches.load(); }
void hg_reset_launch_count(void) { g_launches.store(0); }

int hg_raster_layout_query(int32_t P, int32_t W, int32_t H, int64_t R, hg_raster_layout* out) {
  if (!out || P < 0 || W <= 0 || H <= 0 || R < 0) {
    set_error("hg_raster_layout_query: bad argument");
    return HG_ERR_INVALID_ARG;
  }
  fill_layout(P, W, H, R, out);
  return HG_OK;
}

size_t hg_raster_backward_accum_bytes(int32_t P) {
  return (size_t)(P > 0 ? P : 0) * HG_ACC_FLOATS * sizeof(float) + kAlign;
}

int hg_raster_forward(const hg_raster_inputs* in, hg_alloc_fn geom_alloc, void* geom_ctx,
                      hg_alloc_fn binning_alloc, void* binning_ctx, hg_alloc_fn image_alloc,
                      void* image_ctx, float* out_color, float* out_invdepth,
                      int32_t* out_observe, float* out_all_map, float* out_plane_depth,
                      int32_t* radii, int32_t* num_rendered, void* stream_) {
  g_err[0] = 0;
  int rc = validate(in);
  if (rc) return rc;
  if (!geom_alloc || !binning_alloc || !image_alloc || !out_color || !out_all_map ||
      !out_plane_depth || (in->P > 0 && (!out_observe || !radii))) {
    set_error("hg_raster_forward: a mandatory output/allocator is NULL");
    return HG_ERR_INVALID_ARG;
  }
  cudaStream_t stream = (cudaStream_t)stream_;
  int backup = 0;
  if (!num_rendered) num_rendered = &backup;
  *num_rendered = 0;
  const size_t HW = (size_t)in->W * in->H;

  if (in->P == 0) {  // rasterize_points.cu:100: nothing is launched, outputs stay zero
    HG_CUDA_TRY(cudaMemsetAsync(out_color, 0, 3 * HW * sizeof(float), stream));
    if (out_invdepth) HG_CUDA_TRY(cudaMemsetAsync(out_invdepth, 0, HW * sizeof(float), stream));
    HG_CUDA_TRY(cudaMemsetAsync(out_all_map, 0, 5 * HW * sizeof(float), stream));
    HG_CUDA_TRY(cudaMemsetAsync(out_plane_depth, 0, HW * sizeof(float), stream));
    return HG_OK;
  }

  hg_raster_layout L;
  fill_layout(in->P, in->W, in->H, 0, &L);
  char* geom_raw = geom_alloc(geom_ctx, L.geom_bytes);
  char* img_raw = image_alloc(image_ctx, L.image_bytes);
  if (!geom_raw || !img_raw) {
    set_error("scratch allocator returned NULL");
    return HG_ERR_ALLOC;
  }
  GeomState g = geom_from(align_ptr(geom_raw, kAlign), L);
  ImageState img = image_from(align_ptr(img_raw, kAlign), L);

  const float focal_y = in->H / (2.0f * in->tan_fovy);
  const float focal_x = in->W / (2.0f * in->tan_fovx);
  const dim3 grid((in->W + HG_BLOCK_X - 1) / HG_BLOCK_X, (in->H + HG_BLOCK_Y - 1) / HG_BLOCK_Y, 1);

  const int T = (int)(grid.x * grid.y);
  {
    StageTimer t(HG_STAGE_PREPROCESS_FWD, stream);
    HG_CUDA_TRY(cudaMemsetAsync(g.tile_ctr, 0, (size_t)T * g.ctr_stride * sizeof(uint32_t), stream));
    rc = launch_preprocess_fwd(*in, g, radii, out_observe, grid, focal_x, focal_y, stream);
  }
  if (rc) return rc;
  // R is part of the API contract (returned to Python as an int,
  // diff_gaussian_rasterization/__init__.py:89-93), so one sync is unavoidable.  The scan kernel stores R and the
  // counts of the sort's work lists straight into mapped pinned host memory (one slot + event per host thread and
  // device): no copy operation behind the kernel, the host wakes on the kernel's own completion event.
  HostSlot* slot = host_slot();
  if (!slot) return HG_ERR_CUDA;
  {
    StageTimer t(HG_STAGE_SCAN, stream);
    rc = launch_tile_scan(g, img, T, slot->device_value, stream, in->debug != 0);
    if (rc) return rc;
    HG_CUDA_TRY(cudaEventRecord(slot->ready, stream));
  }
  HG_CUDA_TRY(cudaEventSynchronize(slot->ready));
  uint32_t header[8];
  memcpy(header, slot->value, sizeof(header));
  const uint32_t R = header[0];
  if (R > 0x7fffffffu) {
    set_error("%u tile instances exceed the 31-bit num_rendered of the API", R);
    return HG_ERR_INVALID_ARG;
  }
  *num_rendered = (int)R;

  BinState b{};
  if (R > 0) {
    hg_raster_layout LB;
    fill_layout(in->P, in->W, in->H, (int64_t)R, &LB);
    char* bin_raw = binning_alloc(binning_ctx, LB.binning_bytes + binning_scratch_bytes(header[5]));
    if (!bin_raw) {
      set_error("binning allocator returned NULL");
      return HG_ERR_ALLOC;
    }
    b = bin_from(align_ptr(bin_raw, kAlign), LB);
    {
      StageTimer t(HG_STAGE_BINNING, stream);
      rc = launch_binning(*in, g, b, T, grid, header, stream);
    }
    if (rc) return rc;
  }
  StageTimer t(HG_STAGE_BLEND_FWD, stream);
  return launch_blend_fwd(*in, g, b, img, grid, focal_x, focal_y, out_color, out_invdepth,
                          out_observe, out_all_map, out_plane_depth, R == 0, stream);
}

int hg_raster_backward(const hg_raster_inputs* in, int32_t R, const int32_t* radii,
                       const char* geom_buffer, const char* binning_buffer,
                       const char* image_buffer, const float* all_map_pixels,
                       const float* dL_dpix, const float* dL_dout_all_map,
                       const float* dL_dout_plane_depth, const float* dL_dout_invdepth,
                       char* accum, float* dL_dmeans2D, float* dL_dconic, float* dL_dopacity,
                       float* dL_dcolors, float* dL_dinvdepths, float* dL_dmeans3D,
                       float* dL_dcov3D, float* dL_dsh, float* dL_dscales, float* dL_drotations,
                       float* dL_dall_map, void* stream_) {
  return hg_raster_backward_chunked(in, R, radii, geom_buffer, binning_buffer, image_buffer, all_map_pixels, dL_dpix,
                                    dL_dout_all_map, dL_dout_plane_depth, dL_dout_invdepth, accum, dL_dmeans2D, dL_dconic,
                                    dL_dopacity, dL_dcolors, dL_dinvdepths, dL_dmeans3D, dL_dcov3D, dL_dsh, dL_dscales,
                                    dL_drotations, dL_dall_map, 1, nullptr, nullptr, nullptr, 0.f, nullptr, 0, stream_);
}

}  // extern "C"

// hg_raster_backward_chunked and hg_raster_backward_pose: pose_workspace == NULL is the plain backward.
static int raster_backward_impl(const hg_raster_inputs* in, int32_t R, const int32_t* radii, const char* geom_buffer,
                                const char* binning_buffer, const char* image_buffer, const float* all_map_pixels,
                                const float* dL_dpix, const float* dL_dout_all_map, const float* dL_dout_plane_depth,
                                const float* dL_dout_invdepth, char* accum, float* dL_dmeans2D, float* dL_dconic,
                                float* dL_dopacity, float* dL_dcolors, float* dL_dinvdepths, float* dL_dmeans3D,
                                float* dL_dcov3D, float* dL_dsh, float* dL_dscales, float* dL_drotations,
                                float* dL_dall_map, int32_t n_chunks, hg_chunk_fn on_chunk, void* chunk_ctx,
                                float* sh_sink, float sh_beta, float* sh_factor, int32_t flags, void* pose_workspace,
                                void* stream_) {
  g_err[0] = 0;
  int rc = validate(in);
  if (rc) return rc;
  if (pose_workspace && (in->indices || in->parent_indices || in->N != in->P ||
                         (reinterpret_cast<uintptr_t>(pose_workspace) & 15))) {
    set_error("hg_raster_backward_pose: the camera pose gradient needs every Gaussian as one slot (no render or parent "
              "indices, P == N) and a 16-byte aligned workspace");
    return HG_ERR_INVALID_ARG;
  }
  if (in->P == 0) return HG_OK;
  if (!radii || !geom_buffer || !image_buffer || !dL_dpix || !accum || !dL_dmeans2D ||
      !dL_dopacity || !dL_dcolors || !dL_dmeans3D || !dL_dcov3D || (in->shs && !dL_dsh) || !dL_dscales ||
      !dL_drotations || !dL_dall_map || (R > 0 && !binning_buffer) ||
      (in->render_geo && (!all_map_pixels || !dL_dout_all_map || !dL_dout_plane_depth)) ||
      ((dL_dout_invdepth != nullptr) != (dL_dinvdepths != nullptr))) {
    set_error("hg_raster_backward: a mandatory pointer is NULL");
    return HG_ERR_INVALID_ARG;
  }
  cudaStream_t stream = (cudaStream_t)stream_;
  hg_raster_layout L;
  fill_layout(in->P, in->W, in->H, R, &L);
  GeomState g = geom_from(align_ptr(const_cast<char*>(geom_buffer), kAlign), L);
  ImageState img = image_from(align_ptr(const_cast<char*>(image_buffer), kAlign), L);
  BinState b{};
  if (R > 0) b = bin_from(align_ptr(const_cast<char*>(binning_buffer), kAlign), L);

  const float focal_y = in->H / (2.0f * in->tan_fovy);
  const float focal_x = in->W / (2.0f * in->tan_fovx);
  const dim3 grid((in->W + HG_BLOCK_X - 1) / HG_BLOCK_X, (in->H + HG_BLOCK_Y - 1) / HG_BLOCK_Y, 1);

  float* acc = (float*)align_ptr(accum, kAlign);
  {
    StageTimer t(HG_STAGE_ACCUM_ZERO, stream);
    HG_CUDA_TRY(cudaMemsetAsync(acc, 0, (size_t)in->P * HG_ACC_FLOATS * sizeof(float), stream));
  }
  if (R > 0) {
    StageTimer t(HG_STAGE_BLEND_BWD, stream);
    rc = launch_blend_bwd(*in, g, b, img, grid, focal_x, focal_y, all_map_pixels, dL_dpix,
                          dL_dout_all_map, dL_dout_plane_depth, dL_dout_invdepth, acc, stream);
    if (rc) return rc;
  }
  StageTimer t(HG_STAGE_PREPROCESS_BWD, stream);
  // The per-Gaussian backward in slot ranges: once the kernel of a range completes, the rows of those Gaussians are
  // final in EVERY gradient array, and the caller's hook may start shipping them (gradient exchange of view-sharded
  // training, include/hidegs_exchange.h) while the next range is still being computed.  An index remap scatters the
  // rows, so it keeps one range.
  if (n_chunks < 1 || in->indices || in->parent_indices) n_chunks = 1;
  // (Measured and dropped: laying the zero rows of culled slots down with memsets when R < 2 P — the UAV views cull
  // 80 % of the slots — was 1 % SLOWER than letting the culled threads store them; what helps sparse views is a
  // spatially coherent Gaussian order, GaussianParams.from_scene(spatial_order=True): -9 % per training step.)
  const int unit = preprocess_bwd_block_slots();
  const int per = (int)align_up((size_t)(in->P + n_chunks - 1) / n_chunks, (size_t)unit);
  int chunk = 0;
  for (int p0 = 0; p0 < in->P; p0 += per, ++chunk) {
    const int p1 = p0 + per < in->P ? p0 + per : in->P;
    rc = launch_preprocess_bwd(*in, g, radii, focal_x, focal_y, acc, dL_dout_invdepth != nullptr,
                               dL_dmeans2D, dL_dconic, dL_dopacity, dL_dcolors, dL_dinvdepths,
                               dL_dmeans3D, dL_dcov3D, dL_dsh, dL_dscales, dL_drotations,
                               dL_dall_map, stream, p0, p1, sh_sink, sh_beta, sh_factor,
                               (flags & HG_BWD_SKIP_CULLED_ROWS) != 0, static_cast<double*>(pose_workspace));
    if (rc) return rc;
    if (on_chunk) on_chunk(chunk_ctx, chunk, p0, p1, stream_);
  }
  return HG_OK;
}

extern "C" {

int hg_raster_backward_chunked(const hg_raster_inputs* in, int32_t R, const int32_t* radii,
                               const char* geom_buffer, const char* binning_buffer,
                               const char* image_buffer, const float* all_map_pixels,
                               const float* dL_dpix, const float* dL_dout_all_map,
                               const float* dL_dout_plane_depth, const float* dL_dout_invdepth,
                               char* accum, float* dL_dmeans2D, float* dL_dconic, float* dL_dopacity,
                               float* dL_dcolors, float* dL_dinvdepths, float* dL_dmeans3D,
                               float* dL_dcov3D, float* dL_dsh, float* dL_dscales, float* dL_drotations,
                               float* dL_dall_map, int32_t n_chunks, hg_chunk_fn on_chunk, void* chunk_ctx,
                               float* sh_sink, float sh_beta, float* sh_factor, int32_t flags, void* stream_) {
  return raster_backward_impl(in, R, radii, geom_buffer, binning_buffer, image_buffer, all_map_pixels, dL_dpix,
                              dL_dout_all_map, dL_dout_plane_depth, dL_dout_invdepth, accum, dL_dmeans2D, dL_dconic,
                              dL_dopacity, dL_dcolors, dL_dinvdepths, dL_dmeans3D, dL_dcov3D, dL_dsh, dL_dscales,
                              dL_drotations, dL_dall_map, n_chunks, on_chunk, chunk_ctx, sh_sink, sh_beta, sh_factor,
                              flags, nullptr, stream_);
}

int hg_raster_backward_pose(const hg_raster_inputs* in, int32_t R, const int32_t* radii,
                            const char* geom_buffer, const char* binning_buffer,
                            const char* image_buffer, const float* all_map_pixels,
                            const float* dL_dpix, const float* dL_dout_all_map,
                            const float* dL_dout_plane_depth, const float* dL_dout_invdepth,
                            char* accum, float* dL_dmeans2D, float* dL_dconic, float* dL_dopacity,
                            float* dL_dcolors, float* dL_dinvdepths, float* dL_dmeans3D,
                            float* dL_dcov3D, float* dL_dsh, float* dL_dscales, float* dL_drotations,
                            float* dL_dall_map, int32_t n_chunks, hg_chunk_fn on_chunk, void* chunk_ctx,
                            float* sh_sink, float sh_beta, float* sh_factor, int32_t flags, void* pose_workspace,
                            void* stream_) {
  if (!pose_workspace) {
    g_err[0] = 0;
    set_error("hg_raster_backward_pose: pose_workspace is NULL");
    return HG_ERR_INVALID_ARG;
  }
  return raster_backward_impl(in, R, radii, geom_buffer, binning_buffer, image_buffer, all_map_pixels, dL_dpix,
                              dL_dout_all_map, dL_dout_plane_depth, dL_dout_invdepth, accum, dL_dmeans2D, dL_dconic,
                              dL_dopacity, dL_dcolors, dL_dinvdepths, dL_dmeans3D, dL_dcov3D, dL_dsh, dL_dscales,
                              dL_drotations, dL_dall_map, n_chunks, on_chunk, chunk_ctx, sh_sink, sh_beta, sh_factor,
                              flags, pose_workspace, stream_);
}

int hg_raster_debug_keys(int32_t P, int32_t W, int32_t H, int32_t R, const int32_t* radii, const char* geom_buffer,
                         const char* binning_buffer, uint64_t* keys_unsorted, uint32_t* vals_unsorted,
                         uint64_t* keys_sorted, void* stream_) {
  g_err[0] = 0;
  if (P < 0 || W <= 0 || H <= 0 || R < 0) {
    set_error("hg_raster_debug_keys: bad sizes");
    return HG_ERR_INVALID_ARG;
  }
  if (P == 0 || R == 0) return HG_OK;
  if (!radii || !geom_buffer || !binning_buffer) {
    set_error("hg_raster_debug_keys: a mandatory pointer is NULL");
    return HG_ERR_INVALID_ARG;
  }
  hg_raster_layout L;
  fill_layout(P, W, H, R, &L);
  GeomState g = geom_from(align_ptr(const_cast<char*>(geom_buffer), kAlign), L);
  BinState b = bin_from(align_ptr(const_cast<char*>(binning_buffer), kAlign), L);
  const dim3 grid((W + HG_BLOCK_X - 1) / HG_BLOCK_X, (H + HG_BLOCK_Y - 1) / HG_BLOCK_Y, 1);
  return launch_debug_keys(P, (int)(grid.x * grid.y), g, b, radii, R, grid, keys_unsorted, vals_unsorted, keys_sorted,
                           (cudaStream_t)stream_);
}

int hg_sh_gradient_from_factors(int32_t N, int32_t D, int32_t M, int32_t n_views, const float* means3D,
                                const float* factors, int64_t view_stride, float* dL_dsh, float beta, void* stream_) {
  g_err[0] = 0;
  if (N < 0 || n_views < 0 || M <= 0 || M > 16 || D < 0 || (D + 1) * (D + 1) > M || view_stride < 3 * (int64_t)N + 3 ||
      (N > 0 && (!means3D || !dL_dsh || (n_views > 0 && !factors)))) {
    set_error("hg_sh_gradient_from_factors: bad argument (N %d, D %d, M %d, views %d, stride %lld)", N, D, M, n_views,
              (long long)view_stride);
    return HG_ERR_INVALID_ARG;
  }
  if (N == 0) return HG_OK;
  return launch_sh_from_factors(N, D, M, n_views, means3D, factors, (size_t)view_stride, dL_dsh, beta,
                                (cudaStream_t)stream_);
}

void hg_profile_enable(int on) { g_prof_on.store(on ? 1 : 0); }

int hg_profile_collect(double* ms_per_stage, int64_t* count_per_stage, int n_stages) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (int i = 0; i < n_stages; ++i) {
    if (ms_per_stage) ms_per_stage[i] = 0.0;
    if (count_per_stage) count_per_stage[i] = 0;
  }
  int rc = HG_OK;
  for (auto& r : g_prof) {
    float ms = 0.f;
    cudaError_t e = cudaEventSynchronize(r.b);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, r.a, r.b);
    if (e != cudaSuccess) {
      set_error("hg_profile_collect: %s", cudaGetErrorString(e));
      rc = HG_ERR_CUDA;
    } else if (r.stage >= 0 && r.stage < n_stages) {
      if (ms_per_stage) ms_per_stage[r.stage] += ms;
      if (count_per_stage) count_per_stage[r.stage] += 1;
    }
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  g_prof.clear();
  return rc;
}

int hg_mark_visible(int32_t P, const float* means3D, const float* viewmatrix,
                    const float* projmatrix, uint8_t* present, void* stream) {
  g_err[0] = 0;
  if (P < 0 || (P > 0 && (!means3D || !viewmatrix || !present))) {
    set_error("hg_mark_visible: bad argument");
    return HG_ERR_INVALID_ARG;
  }
  return launch_mark_visible(P, means3D, viewmatrix, projmatrix, present, (cudaStream_t)stream);
}

}  // extern "C"
