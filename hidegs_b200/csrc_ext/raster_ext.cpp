// raster_ext.cpp — the thin PyTorch C++ extension of the drop-in rasterizer (`diff_gaussian_rasterization._C`).
//
// Same operator names, argument order and return tuples as the reference's pybind module
// (submodules/hierarchy-rasterizer/ext.cpp:15-18, rasterize_points.h:18-80, rasterize_points.cu:35-279); the compute is
// the C-ABI of include/hidegs_raster.h (libhidegs_b200.so).  This file only does what rasterize_points.cu does around
// CudaRasterizer::Rasterizer::forward / backward: shape checks, output / scratch tensors, pointer unwrapping, the
// current CUDA stream, status -> exception.  Differences from the reference glue, all host-side:
//   * ONE scratch allocation per forward (geometry | image | backward accumulator | binning) instead of three growable
//     byte tensors (rasterize_points.cu:27-33, 91-97); the binning part is sized from the largest num_rendered this
//     (device, P, W, H) has produced so far — an allocation-size memo, results never depend on it;
//   * outputs are torch::empty (the library writes every element), the reference zero-fills 7 tensors per call;
//   * ONE flat gradient arena per backward whose first 59 floats / Gaussian are xyz | sh | opacity | scale | rotation.
// Per-call extensions (keyword arguments of rasterize_gaussians_backward; no module state):
//   sh_sink / sh_beta   accumulate dL/dSH into a caller tensor (hg_raster_backward_chunked)
//   skip_culled_rows    leave the gradient rows of culled slots unwritten (HG_BWD_SKIP_CULLED_ROWS)
//   sh_factor           write the three colour-gradient factors per Gaussian instead of the SH rows (factored exchange)
//   grad_arena          caller-owned flat fp32 tensor the gradients are written into (e.g. multicast symmetric memory)
//   n_chunks/chunk_hook issue the per-Gaussian backward in slot ranges and call hook(chunk, slot_begin, slot_end)
#include <torch/extension.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>

#include <mutex>
#include <tuple>
#include <unordered_map>

#include "../../include/hidegs_raster.h"

namespace {

constexpr int64_t kRound = 32ll << 20;  // scratch size granularity (bytes)

inline int64_t up(int64_t n, int64_t a) { return (n + a - 1) / a * a; }

void check(int rc, const char* what) {
  TORCH_CHECK(rc == HG_OK, what, " failed (status ", rc, "): ", hg_last_error());
}

// data pointer of a tensor, NULL for an empty / undefined one (reference: empty == absent)
template <typename T>
const T* ptr(const torch::Tensor& t) {
  return (t.defined() && t.numel() != 0) ? t.data_ptr<T>() : nullptr;
}
template <typename T>
T* mptr(torch::Tensor& t) {
  return (t.defined() && t.numel() != 0) ? t.data_ptr<T>() : nullptr;
}

torch::Tensor f32(const torch::Tensor& t, const char* name) {
  if (!t.defined()) return t;
  if (t.numel() != 0)
    TORCH_CHECK(t.scalar_type() == torch::kFloat32 && t.is_cuda(), name, ": expected a float32 CUDA tensor, got ",
                t.scalar_type(), " on ", t.device());
  return t.contiguous();
}
// The library reads rotations as one float4 per row; a contiguous view that starts off a 16-byte boundary (e.g.
// params[1:]) is copied into fresh storage so that the drop-in API keeps accepting it.
torch::Tensor f32_aligned16(const torch::Tensor& t, const char* name) {
  torch::Tensor c = f32(t, name);
  if (c.defined() && c.numel() != 0 && reinterpret_cast<uintptr_t>(c.data_ptr()) % 16 != 0) return c.clone();
  return c;
}
torch::Tensor i32(const torch::Tensor& t, const char* name) {
  if (!t.defined()) return t;
  if (t.numel() != 0)
    TORCH_CHECK(t.scalar_type() == torch::kInt32 && t.is_cuda(), name, ": expected an int32 CUDA tensor, got ",
                t.scalar_type(), " on ", t.device());
  return t.contiguous();
}

// Allocation-size memo: largest num_rendered seen per (device, P, W, H).  Sizes the binning part of the forward's
// single scratch block so that the steady state needs no second allocation; never changes a result.
struct CapacityMemo {
  std::mutex mu;
  std::unordered_map<uint64_t, int64_t> seen;
  static uint64_t key(int dev, int P, int W, int H) {
    uint64_t k = (uint64_t)(uint32_t)P;
    k = k * 1000003ull + (uint32_t)W;
    k = k * 1000003ull + (uint32_t)H;
    return k * 131ull + (uint32_t)dev;
  }
  int64_t get(uint64_t k) {
    std::lock_guard<std::mutex> lk(mu);
    auto it = seen.find(k);
    return it == seen.end() ? 0 : it->second;
  }
  void raise(uint64_t k, int64_t r) {
    std::lock_guard<std::mutex> lk(mu);
    auto& v = seen[k];
    if (r > v) v = r;
  }
};
CapacityMemo& memo() {
  static CapacityMemo m;
  return m;
}

// The forward's scratch block and the three allocator callbacks the library asks for memory through
// (std::function<char*(size_t)> of rasterizer.h:34-36 as plain C callbacks with a context pointer).
struct Workspace {
  torch::Tensor block, binning;
  int64_t geom_bytes = 0, image_bytes = 0, accum_bytes = 0, off_image = 0, off_accum = 0, off_binning = 0, binning_cap = 0;
  bool failed = false;
  static char* alloc_geom(void* c, size_t n) {
    auto* w = static_cast<Workspace*>(c);
    return (int64_t)n <= w->geom_bytes ? reinterpret_cast<char*>(w->block.data_ptr()) : nullptr;
  }
  static char* alloc_image(void* c, size_t n) {
    auto* w = static_cast<Workspace*>(c);
    return (int64_t)n <= w->image_bytes ? reinterpret_cast<char*>(w->block.data_ptr()) + w->off_image : nullptr;
  }
  static char* alloc_binning(void* c, size_t n) {
    auto* w = static_cast<Workspace*>(c);
    try {
      if ((int64_t)n <= w->binning_cap) {
        w->binning = w->block.narrow(0, w->off_binning, (int64_t)n);
      } else {  // a view with more instances than any before: its own block, the memo is raised afterwards
        w->binning = torch::empty({up((int64_t)n, kRound)}, w->block.options());
      }
      return reinterpret_cast<char*>(w->binning.data_ptr());
    } catch (...) {  // surfaces as HG_ERR_ALLOC
      w->failed = true;
      return nullptr;
    }
  }
};

void layout_offsets(int P, int W, int H, int64_t* off_image, int64_t* off_accum, int64_t* geom_bytes, int64_t* image_bytes,
                    int64_t* accum_bytes) {
  hg_raster_layout L0;
  check(hg_raster_layout_query(P, W, H, 0, &L0), "hg_raster_layout_query");
  *geom_bytes = (int64_t)L0.geom_bytes;
  *image_bytes = (int64_t)L0.image_bytes;
  *accum_bytes = (int64_t)hg_raster_backward_accum_bytes(P);
  *off_image = up(*geom_bytes, 256);
  *off_accum = *off_image + up(*image_bytes, 256);
}

hg_raster_inputs make_inputs(int P, int N, int degree, int M, int W, int H, float tan_fovx, float tan_fovy,
                             float scale_modifier, bool prefiltered, bool render_geo, bool debug, const torch::Tensor& bg,
                             const torch::Tensor& viewmatrix, const torch::Tensor& projmatrix, const torch::Tensor& campos,
                             const torch::Tensor& indices, const torch::Tensor& parent_indices, const torch::Tensor& ts,
                             const torch::Tensor& kids, const torch::Tensor& means3D, const torch::Tensor& sh,
                             const torch::Tensor& colors, const torch::Tensor& all_map, const torch::Tensor& opacity,
                             const torch::Tensor& scales, const torch::Tensor& rotations, const torch::Tensor& cov3D) {
  hg_raster_inputs s{};
  s.P = P; s.N = N; s.D = degree; s.M = M; s.W = W; s.H = H;
  s.tan_fovx = tan_fovx; s.tan_fovy = tan_fovy; s.scale_modifier = scale_modifier;
  s.prefiltered = prefiltered; s.render_geo = render_geo; s.debug = debug;
  s.background = ptr<float>(bg); s.viewmatrix = ptr<float>(viewmatrix); s.projmatrix = ptr<float>(projmatrix);
  s.campos = ptr<float>(campos);
  s.indices = ptr<int32_t>(indices); s.parent_indices = ptr<int32_t>(parent_indices);
  s.ts = ptr<float>(ts); s.kids = ptr<int32_t>(kids);
  s.means3D = ptr<float>(means3D); s.shs = ptr<float>(sh); s.colors_precomp = ptr<float>(colors);
  s.all_map = ptr<float>(all_map); s.opacities = ptr<float>(opacity); s.scales = ptr<float>(scales);
  s.rotations = ptr<float>(rotations); s.cov3D_precomp = ptr<float>(cov3D);
  return s;
}

// RasterizeGaussiansCUDA (rasterize_points.cu:35-147)
std::tuple<int, torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor,
           torch::Tensor, torch::Tensor>
rasterize_gaussians(torch::Tensor background, torch::Tensor indices, torch::Tensor parent_indices, torch::Tensor ts,
                    torch::Tensor kids, torch::Tensor means3D, torch::Tensor colors, torch::Tensor all_map,
                    torch::Tensor opacity, torch::Tensor scales, torch::Tensor rotations, double scale_modifier,
                    torch::Tensor cov3D_precomp, torch::Tensor viewmatrix, torch::Tensor projmatrix, double tan_fovx,
                    double tan_fovy, int64_t image_height, int64_t image_width, torch::Tensor sh, int64_t degree,
                    torch::Tensor campos, bool prefiltered, bool render_geo, bool debug, bool do_depth) {
  TORCH_CHECK(means3D.dim() == 2 && means3D.size(1) == 3, "means3D must have dimensions (num_points, 3)");
  TORCH_CHECK(means3D.is_cuda(), "hidegs_b200 rasterizer needs CUDA tensors (there is no CPU path)");
  const auto dev = means3D.device();
  background = f32(background, "bg"); viewmatrix = f32(viewmatrix, "viewmatrix"); projmatrix = f32(projmatrix, "projmatrix");
  campos = f32(campos, "campos"); means3D = f32(means3D, "means3D"); colors = f32(colors, "colors_precomp");
  all_map = f32(all_map, "all_map"); opacity = f32(opacity, "opacities"); scales = f32(scales, "scales");
  rotations = f32_aligned16(rotations, "rotations"); cov3D_precomp = f32(cov3D_precomp, "cov3D_precomp"); sh = f32(sh, "shs");
  ts = f32(ts, "interpolation_weights");
  indices = i32(indices, "render_indices"); parent_indices = i32(parent_indices, "parent_indices");
  kids = i32(kids, "num_node_kids");

  const int N = (int)means3D.size(0);
  const int P = indices.numel() == 0 ? N : (int)indices.size(0);
  const int H = (int)image_height, W = (int)image_width;
  const int M = sh.numel() != 0 ? (int)sh.size(1) : 0;
  TORCH_CHECK(!(P != 0 && all_map.numel() != 0 && all_map.size(0) < P), "all_map must have one row per rendered slot");

  c10::cuda::CUDAGuard guard(dev);
  cudaStream_t stream = at::cuda::getCurrentCUDAStream();
  const auto bytes = torch::TensorOptions().dtype(torch::kUInt8).device(dev);
  const auto fopt = torch::TensorOptions().dtype(torch::kFloat32).device(dev);
  const auto iopt = torch::TensorOptions().dtype(torch::kInt32).device(dev);

  Workspace ws;  // largest block first: keeps the caching allocator from splitting it
  layout_offsets(P, W, H, &ws.off_image, &ws.off_accum, &ws.geom_bytes, &ws.image_bytes, &ws.accum_bytes);
  ws.off_binning = ws.off_accum + up(ws.accum_bytes, 256);
  const uint64_t key = CapacityMemo::key(dev.index(), P, W, H);
  const int64_t hint = memo().get(key);
  if (hint > 0) {
    hg_raster_layout LB;
    check(hg_raster_layout_query(P, W, H, up(hint + hint / 8 + 4096, 1 << 18), &LB), "hg_raster_layout_query");
    ws.binning_cap = up((int64_t)LB.binning_bytes, kRound);
  }
  ws.block = torch::empty({ws.off_binning + ws.binning_cap}, bytes);
  ws.binning = ws.block.narrow(0, 0, 0);

  // The library writes every element of these outputs (no zero fill).  All float images come from one allocation and
  // both int vectors from another: two blocks of constant size per view instead of six.
  const int64_t HW = (int64_t)H * W;
  const int nd = do_depth ? 1 : 0;
  torch::Tensor out_f = torch::empty({(9 + nd) * HW}, fopt);
  torch::Tensor out_color = out_f.narrow(0, 0, 3 * HW).view({3, H, W});
  torch::Tensor out_all_map = out_f.narrow(0, 3 * HW, 5 * HW).view({5, H, W});
  torch::Tensor out_plane_depth = out_f.narrow(0, 8 * HW, HW).view({1, H, W});
  torch::Tensor out_invdepth = out_f.narrow(0, 9 * HW, nd * HW).view({nd, H, W});
  torch::Tensor out_i = torch::empty({2 * (int64_t)P}, iopt);
  torch::Tensor radii = out_i.narrow(0, 0, P), out_observe = out_i.narrow(0, P, P);

  hg_raster_inputs in = make_inputs(P, N, (int)degree, M, W, H, (float)tan_fovx, (float)tan_fovy, (float)scale_modifier,
                                    prefiltered, render_geo, debug, background, viewmatrix, projmatrix, campos, indices,
                                    parent_indices, ts, kids, means3D, sh, colors, all_map, opacity, scales, rotations,
                                    cov3D_precomp);
  int32_t rendered = 0;
  const int rc = hg_raster_forward(&in, Workspace::alloc_geom, &ws, Workspace::alloc_binning, &ws, Workspace::alloc_image,
                                   &ws, mptr<float>(out_color), mptr<float>(out_invdepth), mptr<int32_t>(out_observe),
                                   mptr<float>(out_all_map), mptr<float>(out_plane_depth), mptr<int32_t>(radii), &rendered,
                                   stream);
  check(rc, "rasterize_gaussians");
  memo().raise(key, rendered);
  torch::Tensor imgBuffer = ws.block.narrow(0, ws.off_image, ws.image_bytes);
  return std::make_tuple((int)rendered, out_color, radii, out_observe, out_all_map, out_plane_depth, ws.block, ws.binning,
                         imgBuffer, out_invdepth);
}

struct ChunkCtx {
  py::object hook;
  std::exception_ptr error;
};
void on_chunk(void* c, int32_t chunk, int32_t p0, int32_t p1, void* /*stream*/) {
  auto* ctx = static_cast<ChunkCtx*>(c);
  if (ctx->error) return;
  try {
    ctx->hook(chunk, p0, p1);
  } catch (...) {  // must not unwind through the C frame
    ctx->error = std::current_exception();
  }
}

// RasterizeGaussiansBackwardCUDA (rasterize_points.cu:149-279)
py::tuple rasterize_gaussians_backward(torch::Tensor background, torch::Tensor all_map_pixels, torch::Tensor indices,
                                       torch::Tensor parent_indices, torch::Tensor ts, torch::Tensor kids,
                                       torch::Tensor means3D, torch::Tensor radii, torch::Tensor colors,
                                       torch::Tensor all_maps, torch::Tensor opacities, torch::Tensor scales,
                                       torch::Tensor rotations, double scale_modifier, torch::Tensor cov3D_precomp,
                                       torch::Tensor viewmatrix, torch::Tensor projmatrix, double tan_fovx, double tan_fovy,
                                       torch::Tensor dL_dout_color, torch::Tensor dL_dout_all_map,
                                       torch::Tensor dL_dout_plane_depth, torch::Tensor dL_dout_invdepth, torch::Tensor sh,
                                       int64_t degree, torch::Tensor campos, torch::Tensor geomBuffer, int64_t R,
                                       torch::Tensor binningBuffer, torch::Tensor imageBuffer, bool render_geo, bool debug,
                                       c10::optional<torch::Tensor> sh_sink, double sh_beta,
                                       c10::optional<torch::Tensor> grad_arena, int64_t n_chunks, py::object chunk_hook,
                                       c10::optional<torch::Tensor> sh_factor, bool skip_culled_rows) {
  const auto dev = means3D.device();
  background = f32(background, "bg"); viewmatrix = f32(viewmatrix, "viewmatrix"); projmatrix = f32(projmatrix, "projmatrix");
  campos = f32(campos, "campos"); means3D = f32(means3D, "means3D"); colors = f32(colors, "colors_precomp");
  all_maps = f32(all_maps, "all_map"); opacities = f32(opacities, "opacities"); scales = f32(scales, "scales");
  rotations = f32_aligned16(rotations, "rotations"); cov3D_precomp = f32(cov3D_precomp, "cov3D_precomp"); sh = f32(sh, "shs");
  ts = f32(ts, "interpolation_weights"); all_map_pixels = f32(all_map_pixels, "all_map_pixels");
  indices = i32(indices, "render_indices"); parent_indices = i32(parent_indices, "parent_indices");
  kids = i32(kids, "num_node_kids"); radii = i32(radii, "radii");
  dL_dout_color = f32(dL_dout_color, "dL_dout_color"); dL_dout_all_map = f32(dL_dout_all_map, "dL_dout_all_map");
  dL_dout_plane_depth = f32(dL_dout_plane_depth, "dL_dout_plane_depth");
  dL_dout_invdepth = f32(dL_dout_invdepth, "dL_dout_invdepth");

  const int64_t fullP = means3D.size(0);
  const int P = indices.numel() == 0 ? (int)fullP : (int)indices.size(0);
  const int H = (int)dL_dout_color.size(1), W = (int)dL_dout_color.size(2);
  const int M = sh.numel() != 0 ? (int)sh.size(1) : 0;
  // With an index remap or parents the library accumulates into pre-zeroed rows.
  const bool prezero = indices.numel() != 0 || parent_indices.numel() != 0 || P == 0;
  const bool has_depth_grad = dL_dout_invdepth.defined() && dL_dout_invdepth.numel() != 0;

  c10::cuda::CUDAGuard guard(dev);
  cudaStream_t stream = at::cuda::getCurrentCUDAStream();
  const auto fopt = torch::TensorOptions().dtype(torch::kFloat32).device(dev);

  // One flat fp32 arena per backward.  The trainable parameters come first (xyz 3 | sh 3M | opacity 1 | scale 3 |
  // rotation 4 = 59 floats per Gaussian at M = 16), so the view-sharded trainer can all-reduce arena[:59 N] in place
  // without a pack kernel.  Every block starts on a multiple of 4 floats (float4 paths of the backward).
  const int64_t widths[10] = {3, 3 * M, 1, 3, 4, 3, 3, 6, 5, has_depth_grad ? 1 : 0};
  int64_t offs[10], total = 0;
  for (int i = 0; i < 10; ++i) { offs[i] = total; total += up(fullP * widths[i], 4); }
  torch::Tensor arena;
  if (grad_arena.has_value() && grad_arena->defined()) {  // caller-owned arena (e.g. multicast symmetric memory)
    arena = *grad_arena;
    TORCH_CHECK(arena.numel() >= total && arena.scalar_type() == torch::kFloat32 && arena.device() == dev &&
                    arena.is_contiguous(),
                "grad_arena: need a contiguous float32 tensor of at least ", total, " elements on ", dev);
    arena = arena.flatten().narrow(0, 0, total);
    if (prezero) arena.zero_();
  } else {
    arena = prezero ? torch::zeros({total}, fopt) : torch::empty({total}, fopt);
  }
  auto block = [&](int i, std::vector<int64_t> shape) { return arena.narrow(0, offs[i], fullP * widths[i]).view(shape); };
  torch::Tensor dL_dmeans3D = block(0, {fullP, 3}), dL_dsh = block(1, {fullP, M, 3}), dL_dopacity = block(2, {fullP, 1});
  torch::Tensor dL_dscales = block(3, {fullP, 3}), dL_drotations = block(4, {fullP, 4}), dL_dmeans2D = block(5, {fullP, 3});
  torch::Tensor dL_dcolors = block(6, {fullP, 3}), dL_dcov3D = block(7, {fullP, 6}), dL_dall_map = block(8, {fullP, 5});
  torch::Tensor dL_dinvdepths = has_depth_grad ? block(9, {fullP, 1}) : torch::zeros({0, 1}, fopt);

  bool sink_used = false;
  if (P != 0) {
    // the accumulator lives inside the forward's scratch block; a foreign geometry buffer gets a separate one
    int64_t off_image, off_accum, geom_bytes, image_bytes, accum_bytes;
    layout_offsets(P, W, H, &off_image, &off_accum, &geom_bytes, &image_bytes, &accum_bytes);
    torch::Tensor own_accum;
    char* accum;
    if (geomBuffer.numel() >= off_accum + accum_bytes) {
      accum = reinterpret_cast<char*>(geomBuffer.data_ptr()) + off_accum;
    } else {
      own_accum = torch::empty({accum_bytes}, torch::TensorOptions().dtype(torch::kUInt8).device(dev));
      accum = reinterpret_cast<char*>(own_accum.data_ptr());
    }
    hg_raster_inputs in = make_inputs(P, (int)fullP, (int)degree, M, W, H, (float)tan_fovx, (float)tan_fovy,
                                      (float)scale_modifier, false, render_geo, debug, background, viewmatrix, projmatrix,
                                      campos, indices, parent_indices, ts, kids, means3D, sh, colors, all_maps, opacities,
                                      scales, rotations, cov3D_precomp);
    float* sink_ptr = nullptr;
    if (sh_sink.has_value() && sh_sink->defined()) {
      TORCH_CHECK(sh_sink->scalar_type() == torch::kFloat32 && sh_sink->is_contiguous() &&
                      sh_sink->numel() == fullP * 3 * M && sh_sink->device() == dev,
                  "sh_sink must be a contiguous fp32 tensor of the SH gradient's shape");
      // (checked here as well as in the library: sh_sink_supported() is the caller's test)
      TORCH_CHECK(sh.numel() != 0 && indices.numel() == 0 && parent_indices.numel() == 0 && (3 * M) % 4 == 0,
                  "an SH gradient sink needs SH input, no index remap and 3*M a multiple of 4");
      sink_ptr = sh_sink->data_ptr<float>();
      sink_used = true;
    }
    float* factor_ptr = nullptr;
    if (sh_factor.has_value() && sh_factor->defined()) {
      TORCH_CHECK(sh_factor->scalar_type() == torch::kFloat32 && sh_factor->is_contiguous() &&
                      sh_factor->numel() >= 3 * fullP + 3 && sh_factor->device() == dev,
                  "sh_factor must be a contiguous fp32 tensor of at least 3 N + 3 elements");
      TORCH_CHECK(sh.numel() != 0 && indices.numel() == 0 && parent_indices.numel() == 0 && !sink_used,
                  "SH gradient factors need SH input, no index remap and no SH sink");
      factor_ptr = sh_factor->data_ptr<float>();
      sink_used = true;  // the SH rows are not written: no dL_dsh is returned
    }
    const bool hooked = !chunk_hook.is_none() && n_chunks > 0 && !prezero;
    ChunkCtx cctx{hooked ? chunk_hook : py::none(), nullptr};
    int rc;
    if (sink_ptr || factor_ptr || hooked || skip_culled_rows) {
      rc = hg_raster_backward_chunked(
          &in, (int32_t)R, ptr<int32_t>(radii), reinterpret_cast<const char*>(geomBuffer.data_ptr()),
          reinterpret_cast<const char*>(binningBuffer.data_ptr()), reinterpret_cast<const char*>(imageBuffer.data_ptr()),
          ptr<float>(all_map_pixels), ptr<float>(dL_dout_color), ptr<float>(dL_dout_all_map),
          ptr<float>(dL_dout_plane_depth), has_depth_grad ? ptr<float>(dL_dout_invdepth) : nullptr, accum,
          mptr<float>(dL_dmeans2D), nullptr, mptr<float>(dL_dopacity), mptr<float>(dL_dcolors),
          has_depth_grad ? mptr<float>(dL_dinvdepths) : nullptr, mptr<float>(dL_dmeans3D), mptr<float>(dL_dcov3D),
          mptr<float>(dL_dsh), mptr<float>(dL_dscales), mptr<float>(dL_drotations), mptr<float>(dL_dall_map),
          hooked ? (int32_t)n_chunks : 1, hooked ? on_chunk : nullptr, &cctx, sink_ptr, (float)sh_beta, factor_ptr,
          skip_culled_rows ? HG_BWD_SKIP_CULLED_ROWS : 0, stream);
      if (cctx.error) std::rethrow_exception(cctx.error);
    } else {
      rc = hg_raster_backward(
          &in, (int32_t)R, ptr<int32_t>(radii), reinterpret_cast<const char*>(geomBuffer.data_ptr()),
          reinterpret_cast<const char*>(binningBuffer.data_ptr()), reinterpret_cast<const char*>(imageBuffer.data_ptr()),
          ptr<float>(all_map_pixels), ptr<float>(dL_dout_color), ptr<float>(dL_dout_all_map),
          ptr<float>(dL_dout_plane_depth), has_depth_grad ? ptr<float>(dL_dout_invdepth) : nullptr, accum,
          mptr<float>(dL_dmeans2D), nullptr, mptr<float>(dL_dopacity), mptr<float>(dL_dcolors),
          has_depth_grad ? mptr<float>(dL_dinvdepths) : nullptr, mptr<float>(dL_dmeans3D), mptr<float>(dL_dcov3D),
          mptr<float>(dL_dsh), mptr<float>(dL_dscales), mptr<float>(dL_drotations), mptr<float>(dL_dall_map), stream);
    }
    check(rc, "rasterize_gaussians_backward");
  }
  py::object sh_out = sink_used ? py::object(py::none()) : py::cast(dL_dsh);
  return py::make_tuple(dL_dmeans2D, dL_dcolors, dL_dopacity, dL_dmeans3D, dL_dcov3D, sh_out, dL_dscales, dL_drotations,
                        dL_dall_map);
}

// Whether a backward over these inputs can accumulate its SH gradient into a sink (contiguous rows, 16-byte rows).
bool sh_sink_supported(c10::optional<torch::Tensor> sh, c10::optional<torch::Tensor> indices,
                       c10::optional<torch::Tensor> parent_indices) {
  if (!sh.has_value() || !sh->defined() || sh->numel() == 0) return false;
  if (indices.has_value() && indices->defined() && indices->numel() != 0) return false;
  if (parent_indices.has_value() && parent_indices->defined() && parent_indices->numel() != 0) return false;
  return (3 * sh->size(1)) % 4 == 0 && reinterpret_cast<uintptr_t>(sh->data_ptr()) % 16 == 0;
}

// markVisible (rasterizer_impl.cu:145-157).  The reference's Python calls `_C.mark_visible`
// (diff_gaussian_rasterization/__init__.py:187) but never binds it (ext.cpp:15-18); it is bound here.
torch::Tensor mark_visible(torch::Tensor positions, torch::Tensor viewmatrix, torch::Tensor projmatrix) {
  positions = f32(positions, "positions"); viewmatrix = f32(viewmatrix, "viewmatrix"); projmatrix = f32(projmatrix, "projmatrix");
  TORCH_CHECK(positions.is_cuda(), "hidegs_b200 rasterizer needs CUDA tensors (there is no CPU path)");
  const int64_t P = positions.size(0);
  torch::Tensor present = torch::empty({P}, torch::TensorOptions().dtype(torch::kBool).device(positions.device()));
  if (P) {
    c10::cuda::CUDAGuard guard(positions.device());
    check(hg_mark_visible((int32_t)P, ptr<float>(positions), ptr<float>(viewmatrix), ptr<float>(projmatrix),
                          reinterpret_cast<uint8_t*>(present.data_ptr()), at::cuda::getCurrentCUDAStream()),
          "mark_visible");
  }
  return present;
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "hidegs_b200 rasterizer operators (thin torch extension over the C-ABI of include/hidegs_raster.h)";
  m.def("rasterize_gaussians", &rasterize_gaussians);
  m.def("rasterize_gaussians_backward", &rasterize_gaussians_backward, py::arg("background"), py::arg("all_map_pixels"),
        py::arg("indices"), py::arg("parent_indices"), py::arg("ts"), py::arg("kids"), py::arg("means3D"), py::arg("radii"),
        py::arg("colors"), py::arg("all_maps"), py::arg("opacities"), py::arg("scales"), py::arg("rotations"),
        py::arg("scale_modifier"), py::arg("cov3D_precomp"), py::arg("viewmatrix"), py::arg("projmatrix"),
        py::arg("tan_fovx"), py::arg("tan_fovy"), py::arg("dL_dout_color"), py::arg("dL_dout_all_map"),
        py::arg("dL_dout_plane_depth"), py::arg("dL_dout_invdepth"), py::arg("sh"), py::arg("degree"), py::arg("campos"),
        py::arg("geomBuffer"), py::arg("R"), py::arg("binningBuffer"), py::arg("imageBuffer"), py::arg("render_geo"),
        py::arg("debug"), py::arg("sh_sink") = py::none(), py::arg("sh_beta") = 0.0, py::arg("grad_arena") = py::none(),
        py::arg("n_chunks") = 0, py::arg("chunk_hook") = py::none(), py::arg("sh_factor") = py::none(), py::arg("skip_culled_rows") = false);
  m.def("mark_visible", &mark_visible);
  m.def("sh_sink_supported", &sh_sink_supported, py::arg("sh"), py::arg("indices") = py::none(),
        py::arg("parent_indices") = py::none());
}
