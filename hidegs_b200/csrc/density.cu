// density.cu — adaptive density control over the training arenas (include/hidegs_geometry.h, DESIGN.md §3
// "Densify and prune"): graphdeco 3DGS densify_and_clone / densify_and_split / densification_postfix / prune_points
// and reset_opacity, as passes over the flat SoA arenas instead of ~60 small torch ops per call.
//
//   1. densify_plan_kernel   one thread per source row: clone / split / prune decisions -> one flag byte per row,
//                            per-CTA counts of the output sections
//   2. densify_scan_kernel   ONE CTA: per-CTA section bases, section sizes and N' (read back with one synchronisation)
//   3. densify_apply_kernel  one streaming pass: every output row of every group into the new parameter arena and both
//                            new Adam moment arenas (kept rows keep their moments, new rows start at zero)
//
// Output order (each section in source order):
//   [rows not split, kept] ++ [clones, kept] ++ [first child of every split row, kept] ++ [second child, kept]
// The two children of a row share one prune decision, so both child sections have the same size.
#include "common.cuh"
#include "../../include/hidegs_geometry.h"

#include <curand_philox4x32_x.h>

namespace hg {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr uint32_t kAll = 0xffffffffu;
constexpr int kGroupWidth[5] = {3, 48, 1, 3, 4};  // xyz | features | opacity | scaling | rotation (trainer.GROUPS)

// flag bits of a source row
constexpr uint32_t kKeep = 1u;       // the row itself is in the output (not split, not pruned)
constexpr uint32_t kClone = 2u;      // its clone is in the output
constexpr uint32_t kChildren = 4u;   // its two children are in the output
constexpr uint32_t kSplit = 8u;      // the row is split (pruned children included): index into the injected samples
constexpr uint32_t kCloneSel = 16u;  // the row is cloned (pruned clones included): reported count only

struct Offsets {
  int64_t g[5];  // start of every group, in floats
};

struct Thresholds {
  float max_grad, min_opacity, pd_thr, big_thr;
  int big;  // max_screen_size given: world-space size test
};

// torch.max(dim) propagates NaN
__device__ __forceinline__ float nanmax(float a, float b) { return (a > b || a != a) ? a : b; }

__device__ __forceinline__ float smax_of(float e0, float e1, float e2) { return nanmax(nanmax(e0, e1), e2); }

// the same expressions as activate_kernel (geometry.cu), so that every decision matches torch's exp / sigmoid bits
__device__ __forceinline__ float sigmoid_of(float x) { return 1.0f / (1.0f + expf(-x)); }

// x / 1.6 as torch evaluates a float32 tensor divided by a Python scalar: times the fp32 reciprocal
__device__ __forceinline__ float div16(float x) { return __fmul_rn(x, 1.0f / 1.6f); }

// ---- 1. decisions ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
densify_plan_kernel(const float* __restrict__ param, const Offsets o, const int64_t N, const float* __restrict__ accum,
                    const Thresholds t, uint8_t* __restrict__ flags, uint4* __restrict__ cta_counts,
                    uint32_t* __restrict__ cta_clone_sel) {
  __shared__ uint32_t s_cnt[5][kWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  uint32_t f = 0;
  if (n < N) {
    float g = accum[n];
    if (g != g) g = 0.0f;  // grads[grads.isnan()] = 0
    const float* s = param + o.g[3] + 3 * n;
    const float e0 = expf(s[0]), e1 = expf(s[1]), e2 = expf(s[2]);
    const float smax = smax_of(e0, e1, e2);
    const bool low = sigmoid_of(param[o.g[2] + n]) < t.min_opacity;
    // clone: norm(grads, dim=-1) >= threshold; split: padded_grad >= threshold (clones carry zero and are never split)
    const bool clone = fabsf(g) >= t.max_grad && smax <= t.pd_thr;
    const bool split = g >= t.max_grad && smax > t.pd_thr;
    // a clone is a copy of its row: one prune decision for both
    const bool pruned = low || (t.big && smax > t.big_thr);
    if (!split && !pruned) f |= kKeep;
    if (clone) f |= kCloneSel | (pruned ? 0u : kClone);
    if (split) {
      // children: scaling' = log(exp(scaling) / 1.6); the size test sees exp(scaling')
      const float c = smax_of(expf(logf(div16(e0))), expf(logf(div16(e1))), expf(logf(div16(e2))));
      f |= kSplit | ((low || (t.big && c > t.big_thr)) ? 0u : kChildren);
    }
    flags[n] = (uint8_t)f;
  }
  const uint32_t b0 = __ballot_sync(kAll, f & kKeep), b1 = __ballot_sync(kAll, f & kClone);
  const uint32_t b2 = __ballot_sync(kAll, f & kChildren), b3 = __ballot_sync(kAll, f & kSplit);
  const uint32_t b4 = __ballot_sync(kAll, f & kCloneSel);
  if (lane == 0) {
    s_cnt[0][warp] = __popc(b0); s_cnt[1][warp] = __popc(b1); s_cnt[2][warp] = __popc(b2);
    s_cnt[3][warp] = __popc(b3); s_cnt[4][warp] = __popc(b4);
  }
  __syncthreads();
  if (threadIdx.x < 5) {
    uint32_t v = 0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) v += s_cnt[threadIdx.x][w];
    if (threadIdx.x < 4) reinterpret_cast<uint32_t*>(cta_counts + blockIdx.x)[threadIdx.x] = v;
    else cta_clone_sel[blockIdx.x] = v;
  }
}

// ---- 2. section bases -----------------------------------------------------------------------------------------------
// One CTA, rounds of 1024 consecutive CTA counts (one per thread), as tile_scan_kernel (binning.cu).
// header: [0] kept rows [1] kept clones [2] kept children per child section [3] split rows [4] cloned rows [5] N'
__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t u = __shfl_up_sync(kAll, v, o);
    if (lane >= o) v += u;
  }
  return v;
}

__global__ void __launch_bounds__(1024)
densify_scan_kernel(const uint4* __restrict__ cta_counts, const uint32_t* __restrict__ cta_clone_sel, const int nb,
                    uint4* __restrict__ cta_base, long long* __restrict__ header) {
  __shared__ uint32_t s_warp[2][4][32];
  __shared__ uint32_t s_sel[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t carry[4] = {0u, 0u, 0u, 0u};
  uint32_t sel = 0;
  int round = 0;
  for (int base = 0; base < nb; base += 1024, round ^= 1) {
    const int t = base + tid;
    uint4 c4 = make_uint4(0u, 0u, 0u, 0u);
    if (t < nb) {
      c4 = cta_counts[t];
      sel += cta_clone_sel[t];
    }
    const uint32_t c[4] = {c4.x, c4.y, c4.z, c4.w};
    uint32_t incl[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      incl[k] = warp_incl_scan(c[k], lane);
      if (lane == 31) s_warp[round][k][warp] = incl[k];  // double-buffered: one barrier per round
    }
    __syncthreads();
    uint32_t start[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t wsum = s_warp[round][k][lane];
      const uint32_t wincl = warp_incl_scan(wsum, lane);
      start[k] = carry[k] + __shfl_sync(kAll, wincl - wsum, warp) + incl[k] - c[k];
      carry[k] += __shfl_sync(kAll, wincl, 31);
    }
    if (t < nb) cta_base[t] = make_uint4(start[0], start[1], start[2], start[3]);
  }
  sel = __reduce_add_sync(kAll, sel);
  if (lane == 0) s_sel[warp] = sel;
  __syncthreads();
  if (tid == 0) {
    long long cs = 0;
    for (int w = 0; w < 32; ++w) cs += s_sel[w];
    header[0] = carry[0]; header[1] = carry[1]; header[2] = carry[2]; header[3] = carry[3]; header[4] = cs;
    header[5] = (long long)carry[0] + carry[1] + 2ll * carry[2];
  }
}

// ---- 3. the new arenas ----------------------------------------------------------------------------------------------
struct Arenas {
  const float* p;
  const float* m;
  const float* v;
};
struct NewArenas {
  float* p;
  float* m;
  float* v;
};

// rotation -> R of graphdeco's build_rotation (utils/general_utils.py): r / |r|, no epsilon.  Every operation is
// the separate round-to-nearest step torch takes (no contraction), so R has the oracle's bits.
__device__ __forceinline__ void build_rotation(float4 r, float R[3][3]) {
  const float n2 = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(r.x, r.x), __fmul_rn(r.y, r.y)), __fmul_rn(r.z, r.z)),
                             __fmul_rn(r.w, r.w));
  const float nrm = sqrtf(n2);
  const float w = __fdiv_rn(r.x, nrm), x = __fdiv_rn(r.y, nrm), y = __fdiv_rn(r.z, nrm), z = __fdiv_rn(r.w, nrm);
  auto diag = [](float a, float b) { return __fsub_rn(1.f, __fmul_rn(2.f, __fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b)))); };
  auto minus = [](float a, float b, float c, float d) { return __fmul_rn(2.f, __fsub_rn(__fmul_rn(a, b), __fmul_rn(c, d))); };
  auto plus = [](float a, float b, float c, float d) { return __fmul_rn(2.f, __fadd_rn(__fmul_rn(a, b), __fmul_rn(c, d))); };
  R[0][0] = diag(y, z); R[0][1] = minus(x, y, w, z); R[0][2] = plus(x, z, w, y);
  R[1][0] = plus(x, y, w, z); R[1][1] = diag(x, z); R[1][2] = minus(y, z, w, x);
  R[2][0] = minus(x, z, w, y); R[2][1] = plus(y, z, w, x); R[2][2] = diag(x, y);
}

// three standard normal draws for (row, child): Philox4x32-10, key = seed, counter = (row, child); Box-Muller
__device__ __forceinline__ void normal3(uint2 key, int64_t row, uint32_t child, float z[3]) {
  const uint4 r = curand_Philox4x32_10(make_uint4((uint32_t)row, (uint32_t)((uint64_t)row >> 32), child, 0u), key);
  // uniforms in (0, 1]: 24-bit mantissa grid, never 0 (log)
  const float u0 = ((r.x >> 8) + 1u) * (1.0f / 16777216.0f), u1 = (r.y >> 8) * (1.0f / 16777216.0f);
  const float u2 = ((r.z >> 8) + 1u) * (1.0f / 16777216.0f), u3 = (r.w >> 8) * (1.0f / 16777216.0f);
  const float ra = sqrtf(-2.0f * logf(u0)), rb = sqrtf(-2.0f * logf(u2));
  float sa, ca;
  sincospif(2.0f * u1, &sa, &ca);
  z[0] = ra * ca; z[1] = ra * sa; z[2] = rb * cospif(2.0f * u3);
}

// one row of a narrow group (W floats) to its output positions: the kept row with its moments, new rows with zeros
template <int W>
__device__ __forceinline__ void put_rows(const Arenas& a, const NewArenas& d, int64_t src, int64_t dst_off,
                                         const float (&x)[W], uint32_t f, int64_t pk, int64_t pc) {
  if (f & kKeep) {
#pragma unroll
    for (int i = 0; i < W; ++i) {
      d.p[dst_off + W * pk + i] = x[i];
      d.m[dst_off + W * pk + i] = a.m[src + i];
      d.v[dst_off + W * pk + i] = a.v[src + i];
    }
  }
  if (f & kClone) {
#pragma unroll
    for (int i = 0; i < W; ++i) {
      d.p[dst_off + W * pc + i] = x[i];
      d.m[dst_off + W * pc + i] = 0.0f;
      d.v[dst_off + W * pc + i] = 0.0f;
    }
  }
}

template <int W>
__device__ __forceinline__ void put_new_row(const NewArenas& d, int64_t dst, const float (&x)[W]) {
#pragma unroll
  for (int i = 0; i < W; ++i) {
    d.p[dst + i] = x[i];
    d.m[dst + i] = 0.0f;
    d.v[dst + i] = 0.0f;
  }
}

__global__ void __launch_bounds__(kThreads)
densify_apply_kernel(const Arenas a, const Offsets oo, const int64_t N, const NewArenas d, const Offsets no,
                     const int64_t Nn, const uint8_t* __restrict__ flags, const uint4* __restrict__ cta_base,
                     const long long* __restrict__ header, const float* __restrict__ samples, const uint2 key) {
  __shared__ uint32_t s_cnt[4][kWarps];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t n = (int64_t)blockIdx.x * kThreads + tid;
  if (blockIdx.x == 0 && tid < 20) {  // pad floats of every group (up to the next 16 bytes) are zero
    const int g = tid >> 2;
    const int64_t end = no.g[g] + Nn * (g == 1 ? 48 : g == 2 ? 1 : g == 4 ? 4 : 3), i = end + (tid & 3);
    if (i < (end + 3) / 4 * 4) d.p[i] = d.m[i] = d.v[i] = 0.0f;
  }
  const uint32_t f = n < N ? flags[n] : 0u;
  // in-CTA ranks of the four sections: the same warp-ballot scan every launch shape gives the same positions
  const uint32_t b[4] = {__ballot_sync(kAll, f & kKeep), __ballot_sync(kAll, f & kClone),
                         __ballot_sync(kAll, f & kChildren), __ballot_sync(kAll, f & kSplit)};
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 4; ++k) s_cnt[k][warp] = __popc(b[k]);
  }
  __syncthreads();
  if ((b[0] | b[1] | b[2]) == 0) return;  // nothing of this warp reaches the output
  const uint32_t lt = (1u << lane) - 1u;
  uint32_t r[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    uint32_t pre = 0;
    for (int w = 0; w < warp; ++w) pre += s_cnt[k][w];
    r[k] = pre + __popc(b[k] & lt);
  }
  const uint4 cb = cta_base[blockIdx.x];
  const long long kept = header[0], clones = header[1], children = header[2], n_split = header[3];
  const int64_t pk = (int64_t)cb.x + r[0];                      // kept row
  const int64_t pc = kept + (int64_t)cb.y + r[1];               // clone
  const int64_t p1 = kept + clones + (int64_t)cb.z + r[2];      // first child
  const int64_t p2 = p1 + children;                             // second child
  const int64_t si = (int64_t)cb.w + r[3];                      // row of the injected samples (first child)
  // a position beyond the caller's N' (a plan of other inputs) writes nothing
  const bool ok = !((f & kKeep) && pk >= Nn) && !((f & kClone) && pc >= Nn) && !((f & kChildren) && p2 >= Nn);
  const uint32_t fw = ok ? f : 0u;

  if (fw & (kKeep | kClone | kChildren)) {
    float op[1] = {a.p[oo.g[2] + n]};
    float xyz[3], sc[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      xyz[i] = a.p[oo.g[0] + 3 * n + i];
      sc[i] = a.p[oo.g[3] + 3 * n + i];
    }
    const float4 q4 = reinterpret_cast<const float4*>(a.p + oo.g[4])[n];
    float rot[4] = {q4.x, q4.y, q4.z, q4.w};
    put_rows<3>(a, d, oo.g[0] + 3 * n, no.g[0], xyz, fw, pk, pc);
    put_rows<1>(a, d, oo.g[2] + n, no.g[2], op, fw, pk, pc);
    put_rows<3>(a, d, oo.g[3] + 3 * n, no.g[3], sc, fw, pk, pc);
    if (fw & kKeep) {
      const int64_t s4 = oo.g[4] / 4 + n, d4 = no.g[4] / 4 + pk;
      reinterpret_cast<float4*>(d.p)[d4] = q4;
      reinterpret_cast<float4*>(d.m)[d4] = reinterpret_cast<const float4*>(a.m)[s4];
      reinterpret_cast<float4*>(d.v)[d4] = reinterpret_cast<const float4*>(a.v)[s4];
    }
    if (fw & kClone) put_new_row<4>(d, no.g[4] + 4 * pc, rot);
    if (fw & kChildren) {
      float R[3][3];
      build_rotation(q4, R);
      const float e[3] = {expf(sc[0]), expf(sc[1]), expf(sc[2])};
      float csc[3];
#pragma unroll
      for (int i = 0; i < 3; ++i) csc[i] = logf(div16(e[i]));
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        float s[3];
        if (samples) {  // torch.normal(mean=0, std=stds.repeat(2, 1)): rows [first children | second children]
          const float* sp = samples + 3 * (si + (c ? n_split : 0));
          s[0] = sp[0]; s[1] = sp[1]; s[2] = sp[2];
        } else {
          float z[3];
          normal3(key, n, (uint32_t)c, z);
          s[0] = e[0] * z[0]; s[1] = e[1] * z[1]; s[2] = e[2] * z[2];
        }
        float cx[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) cx[i] = (R[i][0] * s[0] + R[i][1] * s[1] + R[i][2] * s[2]) + xyz[i];
        const int64_t p = c ? p2 : p1;
        put_new_row<3>(d, no.g[0] + 3 * p, cx);
        put_new_row<1>(d, no.g[2] + p, op);
        put_new_row<3>(d, no.g[3] + 3 * p, csc);
        put_new_row<4>(d, no.g[4] + 4 * p, rot);
      }
    }
  }

  // features: 48 floats = 12 float4 per row; the warp moves its 32 rows together (coalesced 16-byte accesses)
  const int64_t row0 = n - lane;
  const float4* fs = reinterpret_cast<const float4*>(a.p + oo.g[1]) + row0 * 12;
  const float4* fm = reinterpret_cast<const float4*>(a.m + oo.g[1]) + row0 * 12;
  const float4* fv = reinterpret_cast<const float4*>(a.v + oo.g[1]) + row0 * 12;
  float4* dp = reinterpret_cast<float4*>(d.p + no.g[1]);
  float4* dm = reinterpret_cast<float4*>(d.m + no.g[1]);
  float4* dv = reinterpret_cast<float4*>(d.v + no.g[1]);
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
  for (int k = 0; k < 12; ++k) {
    const int j = lane + 32 * k, rr = j / 12, c = j - 12 * rr;
    const uint32_t g = __shfl_sync(kAll, fw, rr);
    const int64_t qk = __shfl_sync(kAll, pk, rr), qc = __shfl_sync(kAll, pc, rr);
    const int64_t q1 = __shfl_sync(kAll, p1, rr), q2 = __shfl_sync(kAll, p2, rr);
    if (!(g & (kKeep | kClone | kChildren))) continue;
    const float4 x = fs[j];
    if (g & kKeep) {
      dp[qk * 12 + c] = x;
      dm[qk * 12 + c] = fm[j];
      dv[qk * 12 + c] = fv[j];
    }
    if (g & kClone) {
      dp[qc * 12 + c] = x; dm[qc * 12 + c] = zero; dv[qc * 12 + c] = zero;
    }
    if (g & kChildren) {
      dp[q1 * 12 + c] = x; dm[q1 * 12 + c] = zero; dv[q1 * 12 + c] = zero;
      dp[q2 * 12 + c] = x; dm[q2 * 12 + c] = zero; dv[q2 * 12 + c] = zero;
    }
  }
}

// ---- reset_opacity --------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
reset_opacity_kernel(float* __restrict__ op, float* __restrict__ m, float* __restrict__ v, const int64_t N) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    const float s = sigmoid_of(op[i]);
    const float x = (s < 0.01f || s != s) ? s : 0.01f;  // torch.min propagates NaN
    op[i] = logf(x / (1.0f - x));                      // inverse_sigmoid
    m[i] = 0.0f;
    v[i] = 0.0f;
  }
}

struct Workspace {
  uint8_t* flags;
  uint4* counts;
  uint32_t* clone_sel;
  uint4* base;
  long long* header;
};

static Workspace workspace_of(void* ws, int64_t N) {
  const size_t nb = (size_t)((N + kThreads - 1) / kThreads);
  char* p = (char*)(((uintptr_t)ws + 255) / 256 * 256);
  Workspace w;
  w.flags = (uint8_t*)p;
  p += align_up((size_t)N, 256);
  w.counts = (uint4*)p;
  p += align_up(nb * sizeof(uint4), 256);
  w.clone_sel = (uint32_t*)p;
  p += align_up(nb * sizeof(uint32_t), 256);
  w.base = (uint4*)p;
  p += align_up(nb * sizeof(uint4), 256);
  w.header = (long long*)p;
  return w;
}

// the layout the trainer builds (GaussianParams): every group starts on 16 bytes and holds N rows
static bool offsets_ok(const int64_t* off, int64_t N) {
  if (!off) return false;
  for (int g = 0; g < 5; ++g) {
    if (off[g] < 0 || (off[g] & 3) != 0) return false;
    if (g < 4 && off[g] + N * kGroupWidth[g] > off[g + 1]) return false;
  }
  return true;
}

constexpr int64_t kMaxRows = (int64_t)1 << 30;  // N' <= 2 N stays below 2^31 (32-bit per-CTA bases)

}  // namespace
}  // namespace hg

using namespace hg;

extern "C" {

size_t hg_densify_workspace_bytes(int64_t N) {
  if (N < 0) N = 0;
  const size_t nb = (size_t)((N + kThreads - 1) / kThreads);
  return 256 + align_up((size_t)N, 256) + 2 * align_up(nb * sizeof(uint4), 256) + align_up(nb * sizeof(uint32_t), 256) +
         64;
}

int hg_densify_plan(const float* param, const int64_t* group_offsets, int64_t N, const float* accum,
                    int32_t skybox_points, double max_grad, double min_opacity, double extent, double max_screen_size,
                    double percent_dense, void* workspace, int64_t* out_kept, int64_t* out_cloned, int64_t* out_split,
                    int64_t* out_new_n, void* st_) {
  if (skybox_points != 0) {
    set_error("hg_densify_plan: models with skybox points are not supported (skybox_points = %d)", (int)skybox_points);
    return HG_ERR_INVALID_ARG;
  }
  if (N < 0 || N > kMaxRows || !out_kept || !out_cloned || !out_split || !out_new_n || max_screen_size < 0.0 ||
      (N > 0 && (!param || !accum || !workspace || !offsets_ok(group_offsets, N) || ((uintptr_t)param & 15) != 0))) {
    set_error("hg_densify_plan: bad argument (N in [0, 2^30], non-NULL pointers, 16-byte aligned arena with the "
              "GaussianParams group layout, max_screen_size >= 0)");
    return HG_ERR_INVALID_ARG;
  }
  *out_kept = *out_cloned = *out_split = *out_new_n = 0;
  if (N == 0) return HG_OK;
  cudaStream_t st = (cudaStream_t)st_;
  Offsets o;
  for (int g = 0; g < 5; ++g) o.g[g] = group_offsets[g];
  // Python floats: the products are formed in double and narrowed, as torch compares a float32 tensor with a scalar
  Thresholds t;
  t.max_grad = (float)max_grad;
  t.min_opacity = (float)min_opacity;
  t.pd_thr = (float)(percent_dense * extent);
  t.big_thr = (float)(0.1 * extent);
  t.big = max_screen_size > 0.0;
  Workspace w = workspace_of(workspace, N);
  const int nb = (int)((N + kThreads - 1) / kThreads);
  densify_plan_kernel<<<nb, kThreads, 0, st>>>(param, o, N, accum, t, w.flags, w.counts, w.clone_sel);
  HG_POST_LAUNCH(false, st, "densify_plan");
  densify_scan_kernel<<<1, 1024, 0, st>>>(w.counts, w.clone_sel, nb, w.base, w.header);
  HG_POST_LAUNCH(false, st, "densify_scan");
  // N' sizes the new arenas: the one synchronisation of a densify
  long long h[6];
  HG_CUDA_TRY(cudaMemcpyAsync(h, w.header, sizeof(h), cudaMemcpyDeviceToHost, st));
  HG_CUDA_TRY(cudaStreamSynchronize(st));
  *out_kept = h[0];
  *out_cloned = h[4];
  *out_split = h[3];
  *out_new_n = h[5];
  return HG_OK;
}

int hg_densify_apply(const float* old_param, const float* old_exp_avg, const float* old_exp_avg_sq,
                     const int64_t* old_offsets, int64_t N, float* new_param, float* new_exp_avg, float* new_exp_avg_sq,
                     const int64_t* new_offsets, int64_t new_n, const float* samples, uint64_t seed,
                     const void* workspace, void* st_) {
  if (N < 0 || N > kMaxRows || new_n < 0 || new_n > 2 * N ||
      (N > 0 && (!old_param || !old_exp_avg || !old_exp_avg_sq || !workspace || !offsets_ok(old_offsets, N))) ||
      (new_n > 0 && (!new_param || !new_exp_avg || !new_exp_avg_sq || !offsets_ok(new_offsets, new_n))) ||
      (((uintptr_t)old_param | (uintptr_t)old_exp_avg | (uintptr_t)old_exp_avg_sq | (uintptr_t)new_param |
        (uintptr_t)new_exp_avg | (uintptr_t)new_exp_avg_sq) & 15) != 0) {
    set_error("hg_densify_apply: bad argument (non-NULL 16-byte aligned arenas with the GaussianParams group layout, "
              "0 <= N' <= 2 N)");
    return HG_ERR_INVALID_ARG;
  }
  if (N == 0 || new_n == 0) return HG_OK;
  cudaStream_t st = (cudaStream_t)st_;
  Offsets oo, no;
  for (int g = 0; g < 5; ++g) {
    oo.g[g] = old_offsets[g];
    no.g[g] = new_offsets[g];
  }
  Workspace w = workspace_of(const_cast<void*>(workspace), N);
  const Arenas a{old_param, old_exp_avg, old_exp_avg_sq};
  const NewArenas d{new_param, new_exp_avg, new_exp_avg_sq};
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  const int nb = (int)((N + kThreads - 1) / kThreads);
  densify_apply_kernel<<<nb, kThreads, 0, st>>>(a, oo, N, d, no, new_n, w.flags, w.base, w.header, samples, key);
  HG_POST_LAUNCH(false, st, "densify_apply");
  return HG_OK;
}

int hg_reset_opacity(float* opacity, float* exp_avg, float* exp_avg_sq, int64_t N, void* st_) {
  if (N < 0 || (N > 0 && (!opacity || !exp_avg || !exp_avg_sq))) {
    set_error("hg_reset_opacity: bad argument");
    return HG_ERR_INVALID_ARG;
  }
  if (N == 0) return HG_OK;
  cudaStream_t st = (cudaStream_t)st_;
  const int64_t blocks = (N + kThreads - 1) / kThreads;
  reset_opacity_kernel<<<(unsigned)(blocks < 148 * 8 ? blocks : 148 * 8), kThreads, 0, st>>>(opacity, exp_avg, exp_avg_sq,
                                                                                            N);
  HG_POST_LAUNCH(false, st, "reset_opacity");
  return HG_OK;
}

}  // extern "C"
