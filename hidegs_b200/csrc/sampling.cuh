// sampling.cuh — per-row helpers shared by the passes over the training arenas (density.cu, mcmc.cu): the activations
// with torch's bits, graphdeco's build_rotation, and the Philox4x32-10 / Box-Muller normals.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <curand_philox4x32_x.h>

namespace hg {

// the same expressions as activate_kernel (geometry.cu), so that every decision matches torch's exp / sigmoid bits
__device__ __forceinline__ float sigmoid_of(float x) { return 1.0f / (1.0f + expf(-x)); }

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

}  // namespace hg
