// rsc_morton.cuh -- bounding box and Morton quantisation shared by the octree (rsc_octree.cu) and the k-nearest-neighbour
// search of the normal estimator (rsc_normals.cu).
#pragma once
#include <string.h>

#include "rsc_common.cuh"

namespace rsc {

// order-preserving float <-> uint encoding for atomicMin/atomicMax
__device__ __forceinline__ uint32_t f2ord(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ inline float ord2f(uint32_t o) {
  const uint32_t u = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

// per-axis min / max (f2ord-encoded) of soa[a * n_pad + i], i < n, folded into mm[0..2] / mm[3..5].
// finite_only: points with a non-finite coordinate are left out.
__global__ void __launch_bounds__(256) bbox_kernel(const float* __restrict__ soa, int64_t n, int64_t n_pad, uint32_t* __restrict__ mm,
                                                   bool finite_only);

struct Quant {
  double lo[3], w[3], scale;
  int D;
  uint32_t qmax;
};

// cell coordinate of x on axis a: floor((x - lo) / w * 2^D) in float64, clamped to [0, qmax] -- exactly as the oracle
// computes it
__device__ __forceinline__ uint32_t quantise(float x, const Quant& q, int a) {
  const double t = __dmul_rn(__ddiv_rn(__dsub_rn((double)x, q.lo[a]), q.w[a]), q.scale);
  long long v = (long long)floor(t);
  v = v < 0 ? 0 : (v > (long long)q.qmax ? (long long)q.qmax : v);
  return (uint32_t)v;
}

}  // namespace rsc
