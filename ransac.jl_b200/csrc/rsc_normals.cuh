// rsc_normals.cuh -- the exact k-nearest-neighbour search of rsc_normals.cu as an internal step, shared by
// rsc_estimate_normals and rsc_orient_normals (rsc_orient.cu), so that orientation reuses the search instead of a copy.
#pragma once
#include "rsc_common.cuh"
#include "rsc_morton.cuh"

namespace rsc {

// device allocations of one call, released on every return path
struct Allocs {
  void* p[24] = {};
  int np = 0;
  cudaError_t get(void** out, size_t bytes) {
    if (np == 24) return cudaErrorMemoryAllocation;
    cudaError_t e = cudaMalloc(out, bytes ? bytes : 16);
    if (e == cudaSuccess) p[np++] = *out;
    return e;
  }
  ~Allocs() {
    for (int i = 0; i < np; ++i) cudaFree(p[i]);
  }
};

// what knn_prepare leaves on the device (owned by `al`): about 48 B per point
struct KnnSearch {
  Allocs al;
  int64_t n = 0, nf = 0;    // points, finite points
  Quant q;
  float* aos = nullptr;     // [3 n] the input, AoS by point index
  float* soa = nullptr;     // [3 n] the finite points first, SoA in Morton order
  const uint64_t* keys = nullptr;  // [n] sorted Morton keys
  const uint32_t* perm = nullptr;  // [n] sorted position -> point index
  unsigned long long* cnt = nullptr;  // [0] finite points, [1] distances evaluated
};

// uploads xyz[3 n], sorts the finite points by Morton key and builds the sorted SoA; synchronises.
int32_t knn_prepare(rsc_ctx* ctx, const float* xyz, int64_t n, KnnSearch& S);

// one warp per query over the prepared search.  d_nrm: [3 n] PCA normals (sign rule or towards viewpoint), or null
// for the lists alone; d_nbr: [n k] int64 lists or null; d_lists: [n k] int32 lists or null (not with d_nbr).
// Enqueues only.
int32_t knn_run(rsc_ctx* ctx, const KnnSearch& S, int32_t k, const double* viewpoint, float* d_nrm, int64_t* d_nbr,
                int32_t* d_lists);

}  // namespace rsc
