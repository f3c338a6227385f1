/*
 * hidegs_raster.h — C-ABI of the B200-native HiDeGS rasterizer hot path.
 *
 * This header is the drop-in boundary.  Every entry point takes only POD
 * (device pointers, sizes, scalars, a cudaStream_t passed as void*) and
 * returns an int status (0 = ok, otherwise see hg_status).  No C++ exceptions
 * cross the ABI and no torch types appear in any signature.
 *
 * Reference interfaces each entry point replaces (paths relative to the
 * reference tree, submodules/hierarchy-rasterizer/):
 *
 *   hg_raster_forward   <- CudaRasterizer::Rasterizer::forward
 *                          (cuda_rasterizer/rasterizer.h:33-72,
 *                           cuda_rasterizer/rasterizer_impl.cu:203-405), as
 *                          driven by RasterizeGaussiansCUDA
 *                          (rasterize_points.cu:35-147)
 *   hg_raster_backward  <- CudaRasterizer::Rasterizer::backward
 *                          (cuda_rasterizer/rasterizer.h:74-117,
 *                           cuda_rasterizer/rasterizer_impl.cu:409-535), as
 *                          driven by RasterizeGaussiansBackwardCUDA
 *                          (rasterize_points.cu:149-279)
 *   hg_mark_visible     <- CudaRasterizer::Rasterizer::markVisible
 *                          (cuda_rasterizer/rasterizer_impl.cu:145-157)
 *   hg_alloc_fn         <- std::function<char*(size_t)> geometryBuffer /
 *                          binningBuffer / imageBuffer
 *                          (cuda_rasterizer/rasterizer.h:34-36)
 *   hg_raster_layout    <- GeometryState/ImageState/BinningState::fromChunk
 *                          (cuda_rasterizer/rasterizer_impl.cu:159-199); the
 *                          layout itself is this library's own (SoA + one
 *                          64-byte splat record per slot) and is only exposed
 *                          so that parity tests can read keys / ranges.
 *
 * Conventions kept from the reference: a NULL pointer means "tensor absent"
 * (rasterizer_impl.cu:376,471,506; forward.cu:276,290,328,402,503); matrices
 * are the 16 floats of a row-vector-convention 4x4 (cameras.py:127-129) read
 * as in auxiliary.h:83-102; quaternions are NOT normalised here
 * (forward.cu:190).
 */
#ifndef HIDEGS_RASTER_H
#define HIDEGS_RASTER_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define HG_API __attribute__((visibility("default")))
#else
#define HG_API
#endif

#define HG_NUM_CHANNELS 3 /* config.h:15 */
#define HG_NUM_ALL_MAP 5  /* config.h:16 */
#define HG_BLOCK_X 16     /* config.h:17 */
#define HG_BLOCK_Y 16     /* config.h:18 */

enum hg_status {
  HG_OK = 0,
  HG_ERR_INVALID_ARG = 1, /* bad shape / missing mandatory pointer        */
  HG_ERR_CUDA = 2,        /* a CUDA runtime call or kernel launch failed  */
  HG_ERR_ALLOC = 3        /* a scratch allocator callback returned NULL   */
};

/* Scratch allocator: must return a device pointer to >= bytes bytes that
 * stays valid until the matching backward call has completed. */
typedef char *(*hg_alloc_fn)(void *ctx, size_t bytes);

/* Per-call inputs shared by forward and backward (all pointers are device
 * pointers, nullable where the reference accepts an empty tensor). */
typedef struct hg_raster_inputs {
  int32_t P;      /* rendered slots: indices ? len(indices) : N           */
  int32_t N;      /* rows of means3D ("fullP", rasterize_points.cu:184)   */
  int32_t D;      /* active SH degree                                     */
  int32_t M;      /* SH coefficients per channel (0 if shs absent)        */
  int32_t W, H;   /* image size                                           */
  float tan_fovx, tan_fovy;
  float scale_modifier;
  int32_t prefiltered;
  int32_t render_geo;
  int32_t debug;  /* synchronise + check after every launch               */
  const float *background;     /* [3]                                     */
  const float *viewmatrix;     /* [16]                                    */
  const float *projmatrix;     /* [16]                                    */
  const float *campos;         /* [3]                                     */
  const int32_t *indices;        /* [P] or NULL                           */
  const int32_t *parent_indices; /* [P] or NULL                           */
  const float *ts;               /* interpolation weights or NULL         */
  const int32_t *kids;           /* num_node_kids or NULL                 */
  const float *means3D;        /* [N,3]                                   */
  const float *shs;            /* [N,M,3] or NULL                         */
  const float *colors_precomp; /* [N,3] or NULL                           */
  const float *all_map;        /* [P,5] or NULL                           */
  const float *opacities;      /* [N,1]                                   */
  const float *scales;         /* [N,3] or NULL                           */
  const float *rotations;      /* [N,4] or NULL; 16-byte aligned (read as one float4 per row;
                                  forward and backward return HG_ERR_INVALID_ARG otherwise) */
  const float *cov3D_precomp;  /* [N,6] or NULL                           */
} hg_raster_inputs;

/* Byte offsets of the arrays inside the three opaque scratch buffers
 * (test/diagnostic accessor). */
typedef struct hg_raster_layout {
  /* geometry buffer (depends on P and on the tile grid of W x H) */
  size_t geom_bytes;
  size_t depths;        /* f32[P] view depth of visible slots (culled slots: undefined) */
  size_t tiles_touched; /* u32[P]; 0 for culled slots                     */
  size_t point_offsets; /* u32[P] inclusive prefix sum; only filled by hg_raster_debug_keys */
  size_t rects;         /* u32[P,2] tile bounds: minx|miny<<16, maxx|maxy<<16 */
  size_t cov3D;         /* f32[P,6]                                       */
  size_t clamped;       /* u8[P] bit0..2 = r,g,b clamped                  */
  size_t records;       /* f32[P,16] splat record, see DESIGN.md          */
  size_t tiles;         /* T = number of 16x16 tiles (a count, not an offset) */
  size_t ctr_stride;    /* words between the counters of consecutive tiles (a count, not an offset) */
  size_t tile_ctr;      /* u32[T, ctr_stride]: [t][0] instances of tile t, [t][1] end of its list in pairs / vals */
  size_t tile_lists;    /* u32[3,T] work lists of the per-tile sort, by list length */
  size_t bin_header;    /* u32[16]: R, list counts, work counters         */
  /* image buffer */
  size_t image_bytes;
  size_t final_T;   /* f32[H*W]                                           */
  size_t n_contrib; /* u32[H*W]                                           */
  size_t ranges;    /* u32[T,2]                                           */
  /* binning buffer (sized for R instances; lists too long for shared memory add sort scratch behind it) */
  size_t binning_bytes;
  size_t vals;      /* u32[R] == reference point_list                     */
  size_t pairs;     /* u32[R,2] (depth bits, slot) of every instance, bucketed by tile, arrival order */
} hg_raster_layout;

HG_API int hg_raster_layout_query(int32_t P, int32_t W, int32_t H, int64_t R,
                           hg_raster_layout *out);

/* Forward.  Outputs are fully written by the call (no pre-zeroing needed):
 *   out_color [3,H,W], out_invdepth [1,H,W] or NULL (do_depth=false),
 *   out_observe [P] i32, out_all_map [5,H,W], out_plane_depth [1,H,W],
 *   radii [P] i32.  *num_rendered receives R (host int, one stream sync as in
 *   rasterizer_impl.cu:329-330). */
HG_API int hg_raster_forward(const hg_raster_inputs *in,
                      hg_alloc_fn geom_alloc, void *geom_ctx,
                      hg_alloc_fn binning_alloc, void *binning_ctx,
                      hg_alloc_fn image_alloc, void *image_ctx,
                      float *out_color, float *out_invdepth,
                      int32_t *out_observe, float *out_all_map,
                      float *out_plane_depth, int32_t *radii,
                      int32_t *num_rendered, void *stream);

/* Backward.  `accum` is caller-provided scratch of
 * hg_raster_backward_accum_bytes(P) bytes (contents ignored).  All gradient
 * outputs are fully written (rows of culled Gaussians receive zeros), except
 * when in->indices != NULL, in which case the caller must pre-zero them
 * (rows that no slot maps to are not touched; the same holds when
 * in->parent_indices != NULL, because parents receive atomic pushes).  dL_dconic and dL_dinvdepths
 * may be NULL. */
HG_API size_t hg_raster_backward_accum_bytes(int32_t P);

HG_API int hg_raster_backward(const hg_raster_inputs *in, int32_t R,
                       const int32_t *radii,
                       const char *geom_buffer, const char *binning_buffer,
                       const char *image_buffer,
                       const float *all_map_pixels,     /* [5,H,W]        */
                       const float *dL_dpix,            /* [3,H,W]        */
                       const float *dL_dout_all_map,    /* [5,H,W]        */
                       const float *dL_dout_plane_depth,/* [1,H,W]        */
                       const float *dL_dout_invdepth,   /* [1,H,W] or NULL*/
                       char *accum,
                       float *dL_dmeans2D,   /* [N,3] */
                       float *dL_dconic,     /* [N,2,2] or NULL */
                       float *dL_dopacity,   /* [N,1] */
                       float *dL_dcolors,    /* [N,3] */
                       float *dL_dinvdepths, /* [N,1] or NULL */
                       float *dL_dmeans3D,   /* [N,3] */
                       float *dL_dcov3D,     /* [N,6] */
                       float *dL_dsh,        /* [N,M,3] (may be NULL when shs is) */
                       float *dL_dscales,    /* [N,3] */
                       float *dL_drotations, /* [N,4] */
                       float *dL_dall_map,   /* [N,5] */
                       void *stream);

/* hg_raster_backward with the per-Gaussian part (backward.cu:147-326, 398-496) issued in `n_chunks` slot ranges.
 * Right after the kernel of slots [slot_begin, slot_end) has been QUEUED on `stream`, `on_chunk(chunk_ctx, chunk,
 * slot_begin, slot_end, stream)` is called on the host: once that kernel completes, rows slot_begin..slot_end-1 of
 * every gradient array are final, so the hook can record an event and start the gradient exchange of those rows on
 * another stream (include/hidegs_exchange.h) while the remaining ranges are computed.  Range boundaries are multiples
 * of 128 slots.  With render indices / parent indices (scattered rows) a single range is used.
 * `sh_sink` (optional, [N, M, 3], 16-byte aligned): the SH gradient is ACCUMULATED there, sink = sh_beta * sink + grad
 * (sh_beta 0 or 1), instead of being written to dL_dsh — the gradient arena of a multi-view training step, replacing
 * autograd's AccumulateGrad pass over the largest parameter block; rows of culled Gaussians are zero-filled when
 * sh_beta == 0 and not touched otherwise.  Needs SH input, no index remap and 3 M a multiple of 4.
 * `sh_factor` (optional, [3 N + 4] floats; excludes sh_sink): the SH gradient rows are NOT written at all; instead the
 * three clamp-masked colour gradients of every Gaussian go to sh_factor[3 g .. 3 g + 2] (zeros for culled slots) and
 * the view's camera centre to sh_factor[3 N .. 3 N + 2].  dL/dSH is the outer product of the SH basis at the view
 * direction with exactly these three numbers, so a data-parallel step ships 12 bytes per Gaussian and view instead of
 * 192 and rebuilds the summed rows with hg_sh_gradient_from_factors (include/hidegs_exchange.h).
 * `flags`: HG_BWD_SKIP_CULLED_ROWS = the gradient rows of culled slots (radii <= 0) are NOT written (they are zeros by
 * definition; the reference zero-fills 324 B per Gaussian for them): for a consumer that looks at `radii` first, such
 * as hg_prologue_backward (include/hidegs_geometry.h) — a sparse view then costs no gradient traffic for the
 * Gaussians it does not see.  The SH sink keeps its own rule (sh_beta). */
#define HG_BWD_SKIP_CULLED_ROWS 1
typedef void (*hg_chunk_fn)(void *chunk_ctx, int32_t chunk, int32_t slot_begin, int32_t slot_end, void *stream);
HG_API int hg_raster_backward_chunked(const hg_raster_inputs *in, int32_t R,
                       const int32_t *radii,
                       const char *geom_buffer, const char *binning_buffer,
                       const char *image_buffer,
                       const float *all_map_pixels,     /* [5,H,W]        */
                       const float *dL_dpix,            /* [3,H,W]        */
                       const float *dL_dout_all_map,    /* [5,H,W]        */
                       const float *dL_dout_plane_depth,/* [1,H,W]        */
                       const float *dL_dout_invdepth,   /* [1,H,W] or NULL*/
                       char *accum,
                       float *dL_dmeans2D,   /* [N,3] */
                       float *dL_dconic,     /* [N,2,2] or NULL */
                       float *dL_dopacity,   /* [N,1] */
                       float *dL_dcolors,    /* [N,3] */
                       float *dL_dinvdepths, /* [N,1] or NULL */
                       float *dL_dmeans3D,   /* [N,3] */
                       float *dL_dcov3D,     /* [N,6] */
                       float *dL_dsh,        /* [N,M,3] (may be NULL when shs is) */
                       float *dL_dscales,    /* [N,3] */
                       float *dL_drotations, /* [N,4] */
                       float *dL_dall_map,   /* [N,5] */
                       int32_t n_chunks, hg_chunk_fn on_chunk,
                                       void *chunk_ctx, float *sh_sink, float sh_beta, float *sh_factor,
                                       int32_t flags, void *stream);

/* hg_raster_backward_chunked that also forms the camera side of the gradient, for per-image camera pose refinement
 * (DESIGN.md §3 "Camera pose refinement"; viewmatrix / projmatrix / campos are the view's CORRECTED camera, e.g. the
 * output of hg_camera_pose_apply, include/hidegs_geometry.h).  Every rendered slot sums dL/dp_cam over every path and
 * its torque; each 128-slot CTA of the per-Gaussian part writes the sum of its slots (double, fixed order) to its row
 * of `pose_workspace` (hg_camera_pose_workspace_bytes(N) bytes, 16-byte aligned; rows are indexed by the global CTA,
 * so n_chunks does not change a bit).  hg_prologue_backward_pose adds the all_map part and hg_camera_pose_grad_finish
 * turns both into the camera's gradient row.  Needs every Gaussian as one slot: render / parent indices and P != N are
 * rejected.  Every other argument as in hg_raster_backward_chunked. */
HG_API int hg_raster_backward_pose(const hg_raster_inputs *in, int32_t R,
                       const int32_t *radii,
                       const char *geom_buffer, const char *binning_buffer,
                       const char *image_buffer,
                       const float *all_map_pixels, const float *dL_dpix, const float *dL_dout_all_map,
                       const float *dL_dout_plane_depth, const float *dL_dout_invdepth,
                       char *accum, float *dL_dmeans2D, float *dL_dconic, float *dL_dopacity,
                       float *dL_dcolors, float *dL_dinvdepths, float *dL_dmeans3D, float *dL_dcov3D,
                       float *dL_dsh, float *dL_dscales, float *dL_drotations, float *dL_dall_map,
                       int32_t n_chunks, hg_chunk_fn on_chunk, void *chunk_ctx, float *sh_sink, float sh_beta,
                       float *sh_factor, int32_t flags, void *pose_workspace, void *stream);

/* Test / diagnostic accessor.  The library never materialises the reference's 64-bit tile|depth keys: it buckets the
 * tile instances by tile (counts from the preprocess pass, one scan, one scatter) and sorts every tile's list by
 * (depth, slot) in shared memory -- same final order as the reference's global 45..47-bit sort, one pass over the
 * instances in HBM instead of six.  This call reconstructs, from the buffers of a finished forward, what the reference holds:
 *   keys_unsorted [R] u64, vals_unsorted [R] u32   duplicateWithKeys output (ascending slot, y-major / x-minor)
 *   keys_sorted   [R] u64                          binningState.point_list_keys after the sort
 * (any of the three may be NULL).  `radii` as returned by the forward. */
HG_API int hg_raster_debug_keys(int32_t P, int32_t W, int32_t H, int32_t R, const int32_t *radii,
                                const char *geom_buffer, const char *binning_buffer,
                                uint64_t *keys_unsorted, uint32_t *vals_unsorted, uint64_t *keys_sorted,
                                void *stream);

/* Frustum test of rasterizer_impl.cu:54-66 (present[i] = p_view.z > 0.2). */
HG_API int hg_mark_visible(int32_t P, const float *means3D, const float *viewmatrix,
                    const float *projmatrix, uint8_t *present, void *stream);

/* Launch counter: number of kernels this library has launched since the last
 * hg_reset_launch_count() (used for bench.py's gpu_launches). */
HG_API int64_t hg_launch_count(void);
HG_API void hg_reset_launch_count(void);

/* Optional per-stage device timing.  While enabled, every stage launched by
 * hg_raster_forward / hg_raster_backward is bracketed by CUDA events on the
 * launch stream (no host synchronisation is added); hg_profile_collect()
 * synchronises, sums the elapsed milliseconds and launch counts per stage into
 * the caller's arrays (n_stages entries, indexed by hg_stage) and clears the
 * record.  Used by bench.py for the live roofline numbers. */
enum hg_stage {
  HG_STAGE_PREPROCESS_FWD = 0,
  HG_STAGE_SCAN = 1,    /* tile counts -> list offsets, tile ranges, R, work lists (one CTA) */
  HG_STAGE_BINNING = 2, /* instance scatter + per-tile sorts */
  HG_STAGE_BLEND_FWD = 3,
  HG_STAGE_ACCUM_ZERO = 4,
  HG_STAGE_BLEND_BWD = 5,
  HG_STAGE_PREPROCESS_BWD = 6,
  HG_STAGE_COUNT = 7
};
HG_API void hg_profile_enable(int on);
HG_API int hg_profile_collect(double *ms_per_stage, int64_t *count_per_stage, int n_stages);

/* Text of the last error on this host thread ("" if none). */
HG_API const char *hg_last_error(void);

/* Library identification: "hidegs_b200 <version> sm_100a". */
HG_API const char *hg_version(void);

#ifdef __cplusplus
}
#endif
#endif /* HIDEGS_RASTER_H */
