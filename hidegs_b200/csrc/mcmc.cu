// mcmc.cu — 3DGS-MCMC densification over the training arenas (include/hidegs_geometry.h, DESIGN.md §3
// "MCMC densification"): the opacity / scale regulariser, opacity-gated position noise, relocation of dead Gaussians
// onto live ones, and capped growth, as passes over the flat SoA arenas.  Nothing here reads back to the host.
//
//   regulariser   mcmc_reg_kernel: gradient RMW + per-CTA double partials, the last CTA sums them in a fixed order
//   noise         mcmc_noise_kernel: one thread per row, xyz += c sigma(100 ((1 - o) - 0.995)) R diag(s^2) R^T z
//   sampling      mcmc_weights_kernel  per-CTA inclusive double scan of the weights, dead counts, zeroed draw counts
//                 mcmc_scan_kernel     ONE CTA: exclusive bases of the CTA sums and dead counts (fixed order)
//                 mcmc_finalize_kernel cdf = base + local; dead rows compacted in row order (relocation)
//                 mcmc_draw_kernel     draw j: Philox uniform -> smallest i with cdf[i] > u cdf[N-1]; integer counts
//   relocate      mcmc_relocate_sources_kernel (o', s') of every drawn row, moments zeroed;
//                 mcmc_relocate_copy_kernel dead row d_j <- its source, moments zeroed
//   grow          mcmc_grow_copy_kernel old arenas -> new arenas (sources with (o', s') and zero moments);
//                 mcmc_grow_append_kernel rows N + j <- source j of the new arena, zero moments
#include <cfloat>

#include "common.cuh"
#include "sampling.cuh"
#include "../../include/hidegs_geometry.h"

namespace hg {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr uint32_t kAll = 0xffffffffu;
constexpr int kGroupWidth[5] = {3, 48, 1, 3, 4};  // xyz | features | opacity | scaling | rotation (trainer.GROUPS)
constexpr int kRegRows = 4;                       // rows per thread of the regulariser
constexpr int64_t kRegRowsPerCta = (int64_t)kRegRows * kThreads;
constexpr int kNMax = 51;                         // relocation ratio cap (gsplat's binoms table)
constexpr uint32_t kPurposeRelocate = 0u, kPurposeGrow = 1u, kPurposeNoise = 2u;  // Philox counter word 2
constexpr int64_t kMaxRows = (int64_t)1 << 30;    // int32 row indices in the draw buffers; N' <= 2 N < 2^31

struct Offsets {
  int64_t g[5];  // start of every group, in floats
};

// ---- workspace ------------------------------------------------------------------------------------------------------
// [counter (regulariser ticket, zero between calls) | regulariser partials | sampling buffers].  The sampling passes
// never touch the first two parts, so one workspace serves the regulariser of every step and the refinements.
struct Workspace {
  unsigned* counter;
  double* reg_partial;  // 2 per regulariser CTA
  double* cdf;          // N
  int* counts;          // N: draws per row
  int* dead_idx;        // N: dead rows in row order (relocation)
  int* src;             // N: source of draw slot j
  double* block_sum;    // per weights CTA
  double* block_base;
  uint32_t* block_dead;
  uint32_t* dead_base;
  long long* header;    // [0] dead rows [1] alive rows
};

static size_t workspace_layout(void* ws, int64_t N, Workspace* w) {
  if (N < 0) N = 0;
  const size_t nb = (size_t)((N + kThreads - 1) / kThreads), nr = (size_t)((N + kRegRowsPerCta - 1) / kRegRowsPerCta);
  const size_t parts[11] = {256, 2 * nr * sizeof(double), (size_t)N * sizeof(double), (size_t)N * sizeof(int),
                            (size_t)N * sizeof(int), (size_t)N * sizeof(int), nb * sizeof(double), nb * sizeof(double),
                            nb * sizeof(uint32_t), nb * sizeof(uint32_t), 2 * sizeof(long long)};
  char* p = (char*)(((uintptr_t)ws + 255) / 256 * 256);
  size_t off[11], total = 0;
  for (int i = 0; i < 11; ++i) {
    off[i] = total;
    total += align_up(parts[i], 256);
  }
  if (w) {
    w->counter = (unsigned*)(p + off[0]);
    w->reg_partial = (double*)(p + off[1]);
    w->cdf = (double*)(p + off[2]);
    w->counts = (int*)(p + off[3]);
    w->dead_idx = (int*)(p + off[4]);
    w->src = (int*)(p + off[5]);
    w->block_sum = (double*)(p + off[6]);
    w->block_base = (double*)(p + off[7]);
    w->block_dead = (uint32_t*)(p + off[8]);
    w->dead_base = (uint32_t*)(p + off[9]);
    w->header = (long long*)(p + off[10]);
  }
  return 256 + total;  // (room to re-align the base)
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

static bool a16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

// ---- regulariser ----------------------------------------------------------------------------------------------------
// Thread t of CTA b takes rows b * kRegRowsPerCta + k * kThreads + t, k = 0..kRegRows-1.  d sigmoid / dx = t / (1 + t)^2
// with t = exp(-|x|): o (1 - o) without the cancellation of 1 - o near o = 1.
__global__ void __launch_bounds__(kThreads)
mcmc_reg_kernel(const float* __restrict__ param, float* __restrict__ grad, const Offsets o, const int64_t N,
                const float c_op, const float c_sc, const double w_op, const double w_sc, const double loss_mult,
                float* __restrict__ value, float* __restrict__ loss_inout, double* __restrict__ partial,
                unsigned* __restrict__ counter) {
  __shared__ double sm[2][kWarps];
  __shared__ int s_last;
  double acc_o = 0.0, acc_s = 0.0;
  const int64_t r0 = (int64_t)blockIdx.x * kRegRowsPerCta + threadIdx.x;
#pragma unroll
  for (int k = 0; k < kRegRows; ++k) {
    const int64_t n = r0 + (int64_t)k * kThreads;
    if (n >= N) break;
    const float x = param[o.g[2] + n];
    const float t = expf(-fabsf(x));
    const float u = 1.0f + t;
    acc_o += (double)sigmoid_of(x);
    grad[o.g[2] + n] = __fadd_rn(grad[o.g[2] + n], __fmul_rn(c_op, t / (u * u)));  // (no contraction)
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const float s = expf(param[o.g[3] + 3 * n + a]);
      acc_s += (double)s;
      grad[o.g[3] + 3 * n + a] = __fadd_rn(grad[o.g[3] + 3 * n + a], __fmul_rn(c_sc, s));
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int of = 16; of > 0; of >>= 1) {
    acc_o += __shfl_xor_sync(kAll, acc_o, of);
    acc_s += __shfl_xor_sync(kAll, acc_s, of);
  }
  if (lane == 0) {
    sm[0][warp] = acc_o;
    sm[1][warp] = acc_s;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double so = 0.0, ss = 0.0;
    for (int w = 0; w < kWarps; ++w) {
      so += sm[0][w];
      ss += sm[1][w];
    }
    partial[2 * blockIdx.x] = so;
    partial[2 * blockIdx.x + 1] = ss;
    __threadfence();
    s_last = atomicAdd(counter, 1u) == gridDim.x - 1 ? 1 : 0;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  // (__ldcg: the other CTAs' partials are read from L2, past this SM's L1)
  double a0 = 0.0, a1 = 0.0;
  for (int b = threadIdx.x; b < (int)gridDim.x; b += kThreads) {
    a0 += __ldcg(partial + 2 * b);
    a1 += __ldcg(partial + 2 * b + 1);
  }
#pragma unroll
  for (int of = 16; of > 0; of >>= 1) {
    a0 += __shfl_xor_sync(kAll, a0, of);
    a1 += __shfl_xor_sync(kAll, a1, of);
  }
  __syncthreads();
  if (lane == 0) {
    sm[0][warp] = a0;
    sm[1][warp] = a1;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double so = 0.0, ss = 0.0;
    for (int w = 0; w < kWarps; ++w) {
      so += sm[0][w];
      ss += sm[1][w];
    }
    const double reg = w_op * so + w_sc * ss;
    if (value) *value = (float)reg;
    if (loss_inout) *loss_inout = __fadd_rn(*loss_inout, (float)(loss_mult * reg));
    *counter = 0u;  // ready for the next call on this workspace
  }
}

// ---- position noise -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
mcmc_noise_kernel(float* __restrict__ param, const Offsets o, const int64_t N, const float scale,
                  const float* __restrict__ normals, const uint2 key) {
  const int64_t n = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (n >= N) return;
  const float op = sigmoid_of(param[o.g[2] + n]);
  const float gate = 1.0f / (1.0f + expf(-100.0f * ((1.0f - op) - 0.995f)));
  const float4 q4 = reinterpret_cast<const float4*>(param + o.g[4])[n];
  float R[3][3];
  build_rotation(q4, R);
  float z[3];
  if (normals) {
    z[0] = normals[3 * n]; z[1] = normals[3 * n + 1]; z[2] = normals[3 * n + 2];
  } else {
    normal3(key, n, kPurposeNoise, z);
  }
  float s2[3], v[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const float s = expf(param[o.g[3] + 3 * n + a]);
    s2[a] = s * s;
    v[a] = (z[a] * gate) * scale;
  }
  // (R diag(s^2) R^T) v = R (s^2 * (R^T v))
  float w[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) w[a] = s2[a] * (R[0][a] * v[0] + R[1][a] * v[1] + R[2][a] * v[2]);
  float* xyz = param + o.g[0] + 3 * n;
#pragma unroll
  for (int i = 0; i < 3; ++i) xyz[i] += R[i][0] * w[0] + R[i][1] * w[1] + R[i][2] * w[2];
}

// ---- sampling -------------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T warp_incl_scan(T v, int lane) {
#pragma unroll
  for (int of = 1; of < 32; of <<= 1) {
    const T u = __shfl_up_sync(kAll, v, of);
    if (lane >= of) v += u;
  }
  return v;
}

// dead = !(o > min_opacity): o <= min_opacity, and NaN
__device__ __forceinline__ bool is_dead(const float* __restrict__ opacity, int64_t n, float min_opacity) {
  return !(sigmoid_of(opacity[n]) > min_opacity);
}

// weights w = o over the candidates (alive rows for relocation, every row for growth; NaN weighs 0); cdf = the
// CTA-local inclusive scan (warp Hillis-Steele, then the sum of the earlier warps in warp order)
__global__ void __launch_bounds__(kThreads)
mcmc_weights_kernel(const float* __restrict__ opacity, const int64_t N, const float min_opacity, const int relocate,
                    double* __restrict__ cdf, double* __restrict__ block_sum, uint32_t* __restrict__ block_dead,
                    int* __restrict__ counts) {
  __shared__ double s_w[kWarps];
  __shared__ uint32_t s_d[kWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  double w = 0.0;
  bool dead = false;
  if (n < N) {
    const float o = sigmoid_of(opacity[n]);
    dead = !(o > min_opacity);
    if (relocate ? !dead : o > 0.0f) w = (double)o;
    counts[n] = 0;
  }
  const double v = warp_incl_scan(w, lane);
  const uint32_t b = __ballot_sync(kAll, dead);
  if (lane == 31) s_w[warp] = v;
  if (lane == 0) s_d[warp] = __popc(b);
  __syncthreads();
  double base = 0.0;
  for (int k = 0; k < warp; ++k) base += s_w[k];
  if (n < N) cdf[n] = base + v;
  if (threadIdx.x == 0) {
    double t = 0.0;
    uint32_t d = 0;
    for (int k = 0; k < kWarps; ++k) {
      t += s_w[k];
      d += s_d[k];
    }
    block_sum[blockIdx.x] = t;
    block_dead[blockIdx.x] = d;
  }
}

// One CTA, rounds of 1024 consecutive CTA sums (one per thread), as densify_scan_kernel: exclusive bases
__global__ void __launch_bounds__(1024)
mcmc_scan_kernel(const double* __restrict__ block_sum, const uint32_t* __restrict__ block_dead, const int nb,
                 const int64_t N, double* __restrict__ block_base, uint32_t* __restrict__ dead_base,
                 long long* __restrict__ header, long long* __restrict__ out_counts) {
  __shared__ double s_w[2][32];
  __shared__ uint32_t s_d[2][32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double carry = 0.0;
  uint32_t dcarry = 0;
  int round = 0;
  for (int base = 0; base < nb; base += 1024, round ^= 1) {
    const int t = base + tid;
    const double w = t < nb ? block_sum[t] : 0.0;
    const uint32_t d = t < nb ? block_dead[t] : 0u;
    const double iw = warp_incl_scan(w, lane);
    const uint32_t id = warp_incl_scan(d, lane);
    if (lane == 31) {  // double-buffered: one barrier per round
      s_w[round][warp] = iw;
      s_d[round][warp] = id;
    }
    __syncthreads();
    const double ew = __shfl_up_sync(kAll, iw, 1);
    const double wi = warp_incl_scan(s_w[round][lane], lane);
    const double we = __shfl_up_sync(kAll, wi, 1);
    const double wpre = __shfl_sync(kAll, lane == 0 ? 0.0 : we, warp);
    const uint32_t di = warp_incl_scan(s_d[round][lane], lane);
    const uint32_t dpre = __shfl_sync(kAll, di - s_d[round][lane], warp);
    if (t < nb) {
      block_base[t] = carry + (wpre + (lane == 0 ? 0.0 : ew));
      dead_base[t] = dcarry + dpre + id - d;
    }
    carry += __shfl_sync(kAll, wi, 31);
    dcarry += __shfl_sync(kAll, di, 31);
  }
  if (tid == 0) {
    header[0] = dcarry;
    header[1] = N - (long long)dcarry;
    if (out_counts) {
      out_counts[0] = dcarry;
      out_counts[1] = N - (long long)dcarry;
    }
  }
}

__global__ void __launch_bounds__(kThreads)
mcmc_finalize_kernel(const float* __restrict__ opacity, const int64_t N, const float min_opacity, const int relocate,
                     double* __restrict__ cdf, const double* __restrict__ block_base,
                     const uint32_t* __restrict__ dead_base, int* __restrict__ dead_idx) {
  __shared__ uint32_t s_d[kWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (n < N) cdf[n] = block_base[blockIdx.x] + cdf[n];
  if (!relocate) return;
  const bool dead = n < N && is_dead(opacity, n, min_opacity);
  const uint32_t b = __ballot_sync(kAll, dead);
  if (lane == 0) s_d[warp] = __popc(b);
  __syncthreads();
  if (!dead) return;
  uint32_t r = dead_base[blockIdx.x] + __popc(b & ((1u << lane) - 1u));
  for (int k = 0; k < warp; ++k) r += s_d[k];
  dead_idx[r] = (int)n;
}

// draw j < n_draws (relocation: the dead count on the device; growth: the host's n_new): its source row, or -1
__global__ void __launch_bounds__(kThreads)
mcmc_draw_kernel(const double* __restrict__ cdf, const int64_t N, const long long* __restrict__ header,
                 const int64_t n_draws_host, const int relocate, const int64_t* __restrict__ sources,
                 const int64_t n_sources, const uint2 key, int* __restrict__ src, int* __restrict__ counts) {
  const int64_t j = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  const int64_t n_draws = relocate ? (int64_t)header[0] : n_draws_host;
  if (j >= n_draws) return;
  int s = -1;
  if (sources) {
    if (j < n_sources && sources[j] >= 0 && sources[j] < N) s = (int)sources[j];
  } else {
    const double total = cdf[N - 1];
    const uint4 r = curand_Philox4x32_10(
        make_uint4((uint32_t)j, (uint32_t)((uint64_t)j >> 32), relocate ? kPurposeRelocate : kPurposeGrow, 0u), key);
    const double u = (double)(((uint64_t)(r.x >> 5) << 26) | (uint64_t)(r.y >> 6)) * (1.0 / 9007199254740992.0);
    if (!relocate && !(total > 0.0)) {
      s = (int)min((int64_t)(u * (double)N), N - 1);  // growth with no positive weight: uniform over the rows
    } else if (total > 0.0) {
      double t = u * total;
      if (!(t < total)) t = nextafter(total, 0.0);  // u total rounded up to total: the last row that reaches it
      int64_t lo = 0, hi = N - 1;
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(cdf + mid) > t) hi = mid;
        else lo = mid + 1;
      }
      s = (int)lo;
    }
  }
  src[j] = s;
  if (s >= 0) atomicAdd(counts + s, 1);
}

// (o', s') of a row drawn c >= 1 times, evaluated in double and rounded once (DESIGN.md §3 "MCMC densification")
__device__ __forceinline__ void relocated(float logit, const float (&logs)[3], int c, double min_opacity, float& new_logit,
                          float (&new_logs)[3]) {
  const double o = (double)sigmoid_of(logit);
  const int n = min(max(c + 1, 1), kNMax);
  const double op = 1.0 - pow(1.0 - o, 1.0 / (double)n);
  double denom = 0.0;
  for (int i = 1; i <= n; ++i) {
    double binom = 1.0, pw = op, inner = 0.0;  // C(i-1, k), o'^(k+1)
    for (int k = 0; k < i; ++k) {
      const double term = binom / sqrt((double)(k + 1)) * pw;
      inner += (k & 1) ? -term : term;
      binom = binom * (double)(i - 1 - k) / (double)(k + 1);
      pw *= op;
    }
    denom += inner;
  }
  const double oc = fmin(fmax(op, min_opacity), 1.0 - (double)FLT_EPSILON);
  new_logit = (float)log(oc / (1.0 - oc));
#pragma unroll
  for (int a = 0; a < 3; ++a) new_logs[a] = (float)log((double)expf(logs[a]) * o / denom);
}

template <int W>
__device__ __forceinline__ void zero_row(float* __restrict__ m, float* __restrict__ v, int64_t at) {
#pragma unroll
  for (int i = 0; i < W; ++i) m[at + i] = v[at + i] = 0.0f;
}

// every row drawn at least once: (o', s') in place, all 59 moments zeroed
__global__ void __launch_bounds__(kThreads)
mcmc_relocate_sources_kernel(float* __restrict__ p, float* __restrict__ m, float* __restrict__ v, const Offsets o,
                             const int64_t N, const int* __restrict__ counts, const double min_opacity) {
  const int64_t n = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (n >= N) return;
  const int c = counts[n];
  if (c == 0) return;
  const float logs[3] = {p[o.g[3] + 3 * n], p[o.g[3] + 3 * n + 1], p[o.g[3] + 3 * n + 2]};
  float nl, ns[3];
  relocated(p[o.g[2] + n], logs, c, min_opacity, nl, ns);
  p[o.g[2] + n] = nl;
#pragma unroll
  for (int a = 0; a < 3; ++a) p[o.g[3] + 3 * n + a] = ns[a];
  zero_row<3>(m, v, o.g[0] + 3 * n);
  zero_row<48>(m, v, o.g[1] + 48 * n);
  zero_row<1>(m, v, o.g[2] + n);
  zero_row<3>(m, v, o.g[3] + 3 * n);
  zero_row<4>(m, v, o.g[4] + 4 * n);
}

template <int W>
__device__ __forceinline__ void copy_row(const float* __restrict__ from, float* __restrict__ to, int64_t s, int64_t d) {
#pragma unroll
  for (int i = 0; i < W; ++i) to[d + i] = from[s + i];
}

// slot j < dead count: dead row d_j <- its (already updated) source, its moments zeroed
__global__ void __launch_bounds__(kThreads)
mcmc_relocate_copy_kernel(float* __restrict__ p, float* __restrict__ m, float* __restrict__ v, const Offsets o,
                          const long long* __restrict__ header, const int* __restrict__ dead_idx,
                          const int* __restrict__ src) {
  const int64_t j = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (j >= header[0]) return;
  const int64_t s = src[j];
  if (s < 0) return;
  const int64_t d = dead_idx[j];
  copy_row<3>(p, p, o.g[0] + 3 * s, o.g[0] + 3 * d);
  copy_row<1>(p, p, o.g[2] + s, o.g[2] + d);
  copy_row<3>(p, p, o.g[3] + 3 * s, o.g[3] + 3 * d);
  reinterpret_cast<float4*>(p + o.g[4])[d] = reinterpret_cast<const float4*>(p + o.g[4])[s];
  const float4* fs = reinterpret_cast<const float4*>(p + o.g[1]) + 12 * s;
  float4* fd = reinterpret_cast<float4*>(p + o.g[1]) + 12 * d;
#pragma unroll
  for (int k = 0; k < 12; ++k) fd[k] = fs[k];
  zero_row<3>(m, v, o.g[0] + 3 * d);
  zero_row<48>(m, v, o.g[1] + 48 * d);
  zero_row<1>(m, v, o.g[2] + d);
  zero_row<3>(m, v, o.g[3] + 3 * d);
  zero_row<4>(m, v, o.g[4] + 4 * d);
}

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

template <int W>
__device__ __forceinline__ void move_row(const Arenas& a, const NewArenas& d, int64_t s, int64_t t, const float (&x)[W],
                                         bool src) {
#pragma unroll
  for (int i = 0; i < W; ++i) {
    d.p[t + i] = x[i];
    d.m[t + i] = src ? 0.0f : a.m[s + i];
    d.v[t + i] = src ? 0.0f : a.v[s + i];
  }
}

// rows 0..N-1 of the new arenas: the old rows, drawn rows with (o', s') and zero moments; pads zeroed
__global__ void __launch_bounds__(kThreads)
mcmc_grow_copy_kernel(const Arenas a, const Offsets oo, const int64_t N, const NewArenas d, const Offsets no,
                      const int64_t Nn, const int* __restrict__ counts, const double min_opacity) {
  const int tid = threadIdx.x, lane = tid & 31;
  const int64_t n = (int64_t)blockIdx.x * kThreads + tid;
  if (blockIdx.x == 0 && tid < 20) {  // pad floats of every group (up to the next 16 bytes) are zero
    const int g = tid >> 2;  // (selects, not an indexed load: a dynamic index would put `no` in local memory)
    const int64_t start = g == 0 ? no.g[0] : g == 1 ? no.g[1] : g == 2 ? no.g[2] : g == 3 ? no.g[3] : no.g[4];
    const int64_t end = start + Nn * (g == 1 ? 48 : g == 2 ? 1 : g == 4 ? 4 : 3), i = end + (tid & 3);
    if (i < (end + 3) / 4 * 4) d.p[i] = d.m[i] = d.v[i] = 0.0f;
  }
  const bool live = n < N;
  const int c = live ? counts[n] : 0;
  if (live) {
    float xyz[3], op[1], sc[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      xyz[i] = a.p[oo.g[0] + 3 * n + i];
      sc[i] = a.p[oo.g[3] + 3 * n + i];
    }
    op[0] = a.p[oo.g[2] + n];
    if (c) {
      float nl, ns[3];
      relocated(op[0], sc, c, min_opacity, nl, ns);
      op[0] = nl;
      sc[0] = ns[0]; sc[1] = ns[1]; sc[2] = ns[2];
    }
    move_row<3>(a, d, oo.g[0] + 3 * n, no.g[0] + 3 * n, xyz, c);
    move_row<1>(a, d, oo.g[2] + n, no.g[2] + n, op, c);
    move_row<3>(a, d, oo.g[3] + 3 * n, no.g[3] + 3 * n, sc, c);
    const int64_t s4 = oo.g[4] / 4 + n, d4 = no.g[4] / 4 + n;
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    reinterpret_cast<float4*>(d.p)[d4] = reinterpret_cast<const float4*>(a.p)[s4];
    reinterpret_cast<float4*>(d.m)[d4] = c ? zero : reinterpret_cast<const float4*>(a.m)[s4];
    reinterpret_cast<float4*>(d.v)[d4] = c ? zero : reinterpret_cast<const float4*>(a.v)[s4];
  }
  // features: 48 floats = 12 float4 per row; the warp moves its 32 rows together (coalesced 16-byte accesses)
  const int64_t row0 = n - lane;
  const float4* fs = reinterpret_cast<const float4*>(a.p + oo.g[1]) + row0 * 12;
  const float4* fm = reinterpret_cast<const float4*>(a.m + oo.g[1]) + row0 * 12;
  const float4* fv = reinterpret_cast<const float4*>(a.v + oo.g[1]) + row0 * 12;
  float4* dp = reinterpret_cast<float4*>(d.p + no.g[1]) + row0 * 12;
  float4* dm = reinterpret_cast<float4*>(d.m + no.g[1]) + row0 * 12;
  float4* dv = reinterpret_cast<float4*>(d.v + no.g[1]) + row0 * 12;
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  const uint32_t lv = __ballot_sync(kAll, live), sr = __ballot_sync(kAll, c != 0);
#pragma unroll 4
  for (int k = 0; k < 12; ++k) {
    const int j = lane + 32 * k, rr = j / 12;
    if (!((lv >> rr) & 1u)) continue;
    const bool s = (sr >> rr) & 1u;
    dp[j] = fs[j];
    dm[j] = s ? zero : fm[j];
    dv[j] = s ? zero : fv[j];
  }
}

// rows N + j of the new arenas: copies of source j as the copy kernel left it, zero moments
__global__ void __launch_bounds__(kThreads)
mcmc_grow_append_kernel(const NewArenas d, const Offsets no, const int64_t N, const int64_t n_new,
                        const int* __restrict__ src) {
  const int64_t j = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (j >= n_new) return;
  const int64_t s = src[j], t = N + j;
  if (s < 0) return;
  copy_row<3>(d.p, d.p, no.g[0] + 3 * s, no.g[0] + 3 * t);
  copy_row<1>(d.p, d.p, no.g[2] + s, no.g[2] + t);
  copy_row<3>(d.p, d.p, no.g[3] + 3 * s, no.g[3] + 3 * t);
  reinterpret_cast<float4*>(d.p + no.g[4])[t] = reinterpret_cast<const float4*>(d.p + no.g[4])[s];
  const float4* fs = reinterpret_cast<const float4*>(d.p + no.g[1]) + 12 * s;
  float4* fd = reinterpret_cast<float4*>(d.p + no.g[1]) + 12 * t;
#pragma unroll
  for (int k = 0; k < 12; ++k) fd[k] = fs[k];
  zero_row<3>(d.m, d.v, no.g[0] + 3 * t);
  zero_row<48>(d.m, d.v, no.g[1] + 48 * t);
  zero_row<1>(d.m, d.v, no.g[2] + t);
  zero_row<3>(d.m, d.v, no.g[3] + 3 * t);
  zero_row<4>(d.m, d.v, no.g[4] + 4 * t);
}

// weights, bases, cdf and (relocation) the dead list: four launches, no host read
static int build_cdf(const float* opacity, int64_t N, float min_opacity, int relocate, const Workspace& w,
                     long long* out_counts, cudaStream_t st) {
  const int nb = (int)((N + kThreads - 1) / kThreads);
  mcmc_weights_kernel<<<nb, kThreads, 0, st>>>(opacity, N, min_opacity, relocate, w.cdf, w.block_sum, w.block_dead,
                                               w.counts);
  HG_POST_LAUNCH(false, st, "mcmc_weights");
  mcmc_scan_kernel<<<1, 1024, 0, st>>>(w.block_sum, w.block_dead, nb, N, w.block_base, w.dead_base, w.header,
                                       out_counts);
  HG_POST_LAUNCH(false, st, "mcmc_scan");
  mcmc_finalize_kernel<<<nb, kThreads, 0, st>>>(opacity, N, min_opacity, relocate, w.cdf, w.block_base, w.dead_base,
                                                w.dead_idx);
  HG_POST_LAUNCH(false, st, "mcmc_finalize");
  return HG_OK;
}

static uint2 key_of(uint64_t seed) { return make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)); }

}  // namespace
}  // namespace hg

using namespace hg;

extern "C" {

size_t hg_mcmc_workspace_bytes(int64_t N) { return workspace_layout(nullptr, N, nullptr); }

int hg_mcmc_regularizer(const float* param, float* grad, const int64_t* group_offsets, int64_t N,
                        int32_t skybox_points, double opacity_reg, double scale_reg, double grad_mult,
                        double loss_mult, float* value, float* loss_inout, void* workspace, void* st_) {
  if (skybox_points != 0) {
    set_error("hg_mcmc_regularizer: models with skybox points are not supported (skybox_points = %d)",
              (int)skybox_points);
    return HG_ERR_INVALID_ARG;
  }
  if (N < 0 || N > kMaxRows || !(opacity_reg >= 0.0) || !(scale_reg >= 0.0) ||
      (N > 0 && (!param || !grad || !workspace || !offsets_ok(group_offsets, N)))) {
    set_error("hg_mcmc_regularizer: bad argument (N in [0, 2^30], non-NULL arenas and workspace with the "
              "GaussianParams group layout, weights >= 0)");
    return HG_ERR_INVALID_ARG;
  }
  if (N == 0 || (opacity_reg == 0.0 && scale_reg == 0.0)) return HG_OK;
  cudaStream_t st = (cudaStream_t)st_;
  Offsets o;
  for (int g = 0; g < 5; ++g) o.g[g] = group_offsets[g];
  Workspace w;
  workspace_layout(workspace, N, &w);
  // d/dx of opacity_reg mean o = opacity_reg / N o (1 - o); of scale_reg mean s = scale_reg / (3 N) s; times grad_mult
  const double w_op = opacity_reg / (double)N, w_sc = scale_reg / (3.0 * (double)N);
  const unsigned nr = (unsigned)((N + kRegRowsPerCta - 1) / kRegRowsPerCta);
  mcmc_reg_kernel<<<nr, kThreads, 0, st>>>(param, grad, o, N, (float)(grad_mult * w_op), (float)(grad_mult * w_sc),
                                           w_op, w_sc, loss_mult, value, loss_inout, w.reg_partial, w.counter);
  HG_POST_LAUNCH(false, st, "mcmc_regularizer");
  return HG_OK;
}

int hg_mcmc_inject_noise(float* param, const int64_t* group_offsets, int64_t N, int32_t skybox_points, double scale,
                         const float* normals, uint64_t seed, void* st_) {
  if (skybox_points != 0) {
    set_error("hg_mcmc_inject_noise: models with skybox points are not supported (skybox_points = %d)",
              (int)skybox_points);
    return HG_ERR_INVALID_ARG;
  }
  if (N < 0 || N > kMaxRows || (N > 0 && (!param || !a16(param) || !offsets_ok(group_offsets, N)))) {
    set_error("hg_mcmc_inject_noise: bad argument (N in [0, 2^30], non-NULL 16-byte aligned arena with the "
              "GaussianParams group layout)");
    return HG_ERR_INVALID_ARG;
  }
  if (N == 0) return HG_OK;
  cudaStream_t st = (cudaStream_t)st_;
  Offsets o;
  for (int g = 0; g < 5; ++g) o.g[g] = group_offsets[g];
  const unsigned nb = (unsigned)((N + kThreads - 1) / kThreads);
  mcmc_noise_kernel<<<nb, kThreads, 0, st>>>(param, o, N, (float)scale, normals, key_of(seed));
  HG_POST_LAUNCH(false, st, "mcmc_inject_noise");
  return HG_OK;
}

int hg_mcmc_relocate(float* param, float* exp_avg, float* exp_avg_sq, const int64_t* group_offsets, int64_t N,
                     int32_t skybox_points, double min_opacity, const int64_t* sources, int64_t n_sources,
                     uint64_t seed, int64_t* out_counts, void* workspace, void* st_) {
  if (skybox_points != 0) {
    set_error("hg_mcmc_relocate: models with skybox points are not supported (skybox_points = %d)", (int)skybox_points);
    return HG_ERR_INVALID_ARG;
  }
  if (N < 0 || N > kMaxRows || n_sources < 0 || !(min_opacity >= 0.0 && min_opacity < 1.0) ||
      (N > 0 && (!param || !exp_avg || !exp_avg_sq || !workspace || !offsets_ok(group_offsets, N) ||
                 !a16(param) || !a16(exp_avg) || !a16(exp_avg_sq)))) {
    set_error("hg_mcmc_relocate: bad argument (N in [0, 2^30], non-NULL 16-byte aligned arenas with the "
              "GaussianParams group layout, a workspace, 0 <= min_opacity < 1, n_sources >= 0)");
    return HG_ERR_INVALID_ARG;
  }
  cudaStream_t st = (cudaStream_t)st_;
  if (N == 0) {
    if (out_counts) HG_CUDA_TRY(cudaMemsetAsync(out_counts, 0, 2 * sizeof(int64_t), st));
    return HG_OK;
  }
  Offsets o;
  for (int g = 0; g < 5; ++g) o.g[g] = group_offsets[g];
  Workspace w;
  workspace_layout(workspace, N, &w);
  const float mo = (float)min_opacity;  // (a float32 tensor compared with a Python float)
  int rc = build_cdf(param + o.g[2], N, mo, 1, w, (long long*)out_counts, st);
  if (rc != HG_OK) return rc;
  const unsigned nb = (unsigned)((N + kThreads - 1) / kThreads);
  mcmc_draw_kernel<<<nb, kThreads, 0, st>>>(w.cdf, N, w.header, 0, 1, sources, sources ? n_sources : 0, key_of(seed),
                                            w.src, w.counts);
  HG_POST_LAUNCH(false, st, "mcmc_draw");
  mcmc_relocate_sources_kernel<<<nb, kThreads, 0, st>>>(param, exp_avg, exp_avg_sq, o, N, w.counts, min_opacity);
  HG_POST_LAUNCH(false, st, "mcmc_relocate_sources");
  mcmc_relocate_copy_kernel<<<nb, kThreads, 0, st>>>(param, exp_avg, exp_avg_sq, o, w.header, w.dead_idx, w.src);
  HG_POST_LAUNCH(false, st, "mcmc_relocate_copy");
  return HG_OK;
}

int hg_mcmc_grow(const float* old_param, const float* old_exp_avg, const float* old_exp_avg_sq,
                 const int64_t* old_offsets, int64_t N, float* new_param, float* new_exp_avg, float* new_exp_avg_sq,
                 const int64_t* new_offsets, int64_t new_n, int32_t skybox_points, double min_opacity,
                 const int64_t* sources, uint64_t seed, void* workspace, void* st_) {
  if (skybox_points != 0) {
    set_error("hg_mcmc_grow: models with skybox points are not supported (skybox_points = %d)", (int)skybox_points);
    return HG_ERR_INVALID_ARG;
  }
  if (N <= 0 || N > kMaxRows || new_n <= N || new_n > 2 * N || !(min_opacity >= 0.0 && min_opacity < 1.0) ||
      !old_param || !old_exp_avg || !old_exp_avg_sq || !new_param || !new_exp_avg || !new_exp_avg_sq || !workspace ||
      !offsets_ok(old_offsets, N) || !offsets_ok(new_offsets, new_n) || !a16(old_param) || !a16(old_exp_avg) ||
      !a16(old_exp_avg_sq) || !a16(new_param) || !a16(new_exp_avg) || !a16(new_exp_avg_sq)) {
    set_error("hg_mcmc_grow: bad argument (N in [1, 2^30], N < N' <= 2 N, non-NULL 16-byte aligned arenas with the "
              "GaussianParams group layout, a workspace, 0 <= min_opacity < 1)");
    return HG_ERR_INVALID_ARG;
  }
  cudaStream_t st = (cudaStream_t)st_;
  Offsets oo, no;
  for (int g = 0; g < 5; ++g) {
    oo.g[g] = old_offsets[g];
    no.g[g] = new_offsets[g];
  }
  Workspace w;
  workspace_layout(workspace, N, &w);
  const int64_t n_new = new_n - N;
  int rc = build_cdf(old_param + oo.g[2], N, (float)min_opacity, 0, w, nullptr, st);
  if (rc != HG_OK) return rc;
  const unsigned nb = (unsigned)((N + kThreads - 1) / kThreads), nd = (unsigned)((n_new + kThreads - 1) / kThreads);
  mcmc_draw_kernel<<<nd, kThreads, 0, st>>>(w.cdf, N, w.header, n_new, 0, sources, sources ? n_new : 0, key_of(seed),
                                            w.src, w.counts);
  HG_POST_LAUNCH(false, st, "mcmc_draw");
  const Arenas a{old_param, old_exp_avg, old_exp_avg_sq};
  const NewArenas d{new_param, new_exp_avg, new_exp_avg_sq};
  mcmc_grow_copy_kernel<<<nb, kThreads, 0, st>>>(a, oo, N, d, no, new_n, w.counts, min_opacity);
  HG_POST_LAUNCH(false, st, "mcmc_grow_copy");
  mcmc_grow_append_kernel<<<nd, kThreads, 0, st>>>(d, no, N, n_new, w.src);
  HG_POST_LAUNCH(false, st, "mcmc_grow_append");
  return HG_OK;
}

}  // extern "C"
