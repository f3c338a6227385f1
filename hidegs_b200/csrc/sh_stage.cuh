// sh_stage.cuh — warp-cooperative, coalesced movement of 32 consecutive SH rows (<= 192 B each) between global
// memory and a per-warp shared-memory tile with an odd row stride (conflict-free per-thread row access).
#pragma once
#include <cuda_runtime.h>

namespace hg {

// Warp-cooperative, coalesced load of 32 consecutive SH rows into shared memory
// (row-major, odd stride).  ROW > 0 fixes the row length at compile time.  The row length must be a multiple of 4
// and `shs + base` 16-byte aligned (checked by the caller): the loads are float4s, and the float4s of rows whose bit
// in `row_mask` is clear are skipped, which leaves no live float unloaded only when no float4 straddles two rows.
template <int ROW>
__device__ __forceinline__ void stage_sh_rows(const float* __restrict__ shs, size_t base,
                                              size_t total, int row_rt, int lane, float* dst,
                                              uint32_t row_mask = 0xffffffffu) {
  const int row = ROW > 0 ? ROW : row_rt;
  const int stride = row | 1;
  const int nfloat = 32 * row;  // multiple of 4
  // Loads are issued in groups of kGroup independent LDG.128 before any of them is consumed, so a warp keeps
  // several 512-byte requests in flight (the staging is latency bound otherwise).
  constexpr int kGroup = 4;
  for (int i0 = lane * 4; i0 < nfloat; i0 += 128 * kGroup) {
    float4 val[kGroup];
#pragma unroll
    for (int u = 0; u < kGroup; ++u) {
      const int i = i0 + 128 * u;
      const size_t gi = base + i;
      val[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      // skip rows nobody will read (row % 4 == 0: a float4 never straddles rows)
      if (i < nfloat && ((row_mask >> (i / row)) & 1u)) {
        if (gi + 3 < total) {
          val[u] = __ldg((const float4*)(shs + gi));
        } else {
          val[u].x = gi < total ? __ldg(shs + gi) : 0.f;
          val[u].y = gi + 1 < total ? __ldg(shs + gi + 1) : 0.f;
          val[u].z = gi + 2 < total ? __ldg(shs + gi + 2) : 0.f;
        }
      }
    }
#pragma unroll
    for (int u = 0; u < kGroup; ++u) {
      const int i = i0 + 128 * u;
      if (i < nfloat && ((row_mask >> (i / row)) & 1u)) {
        const float e[4] = {val[u].x, val[u].y, val[u].z, val[u].w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int f = i + k;
          dst[(f / row) * stride + (f % row)] = e[k];
        }
      }
    }
  }
}

// The same for any row length and alignment: one float per lane and step (still coalesced), each loaded only when
// its own row's bit in `row_mask` is set; kGroup independent loads are in flight before any is stored.
__device__ __forceinline__ void stage_sh_rows_scalar(const float* __restrict__ shs, size_t base, size_t total, int row,
                                                     int lane, float* dst, uint32_t row_mask) {
  const int stride = row | 1;
  const int nfloat = 32 * row;
  constexpr int kGroup = 4;
#pragma unroll 1
  for (int i0 = lane; i0 < nfloat; i0 += 32 * kGroup) {
    float val[kGroup];
#pragma unroll
    for (int u = 0; u < kGroup; ++u) {
      const int i = i0 + 32 * u;
      val[u] = (i < nfloat && ((row_mask >> (i / row)) & 1u) && base + i < total) ? __ldg(shs + base + i) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < kGroup; ++u) {
      const int i = i0 + 32 * u;
      if (i < nfloat) dst[(i / row) * stride + i % row] = val[u];
    }
  }
}

// The inverse: rows of the tile -> global, coalesced float4 stores.  Rows whose bit in `row_mask` is clear are
// written as zeros if `zero_others`, else left untouched.  `row` must be a multiple of 4 and `dst + base` 16-byte
// aligned (checked by the caller).
__device__ __forceinline__ void unstage_sh_rows(float* __restrict__ dst, size_t base, size_t total, int row, int lane,
                                                const float* src, uint32_t row_mask, bool zero_others) {
  const int stride = row | 1;
  const int nfloat = 32 * row;
  for (int i = lane * 4; i < nfloat; i += 128) {
    const size_t gi = base + i;
    if (gi >= total) break;
    const int r = i / row, c = i - r * row;
    float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
    if ((row_mask >> r) & 1u) {
      const float* s = src + r * stride + c;
      val = make_float4(s[0], s[1], s[2], s[3]);
    } else if (!zero_others) {
      continue;
    }
    *reinterpret_cast<float4*>(dst + gi) = val;
  }
}

// Accumulating variant for a caller-owned gradient sink: live rows do dst = beta * dst + row (beta = 0: plain store,
// dst is not read); rows whose bit is clear are zero-filled when beta == 0 and NOT TOUCHED otherwise — a culled
// Gaussian costs no traffic in any view but the first of a step.
__device__ __forceinline__ void unstage_sh_rows_accum(float* __restrict__ dst, size_t base, size_t total, int row, int lane,
                                                      const float* src, uint32_t row_mask, float beta) {
  const int stride = row | 1;
  const int nfloat = 32 * row;
  for (int i = lane * 4; i < nfloat; i += 128) {
    const size_t gi = base + i;
    if (gi >= total) break;
    const int r = i / row, c = i - r * row;
    float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
    if ((row_mask >> r) & 1u) {
      const float* s = src + r * stride + c;
      val = make_float4(s[0], s[1], s[2], s[3]);
      if (beta != 0.f) {
        const float4 old = *reinterpret_cast<const float4*>(dst + gi);
        val.x = fmaf(beta, old.x, val.x);
        val.y = fmaf(beta, old.y, val.y);
        val.z = fmaf(beta, old.z, val.z);
        val.w = fmaf(beta, old.w, val.w);
      }
    } else if (beta != 0.f) {
      continue;
    }
    *reinterpret_cast<float4*>(dst + gi) = val;
  }
}

}  // namespace hg
