// rsc_normals.cuh -- the exact k-nearest-neighbour search of rsc_normals.cu as an internal step, shared by
// rsc_estimate_normals and rsc_orient_normals (rsc_orient.cu), so that orientation reuses the search instead of a copy,
// and the collective steps of their sharded forms (rsc_*_normals_shard, DESIGN.md section 8).
#pragma once
#include <functional>

#include "rsc_common.cuh"
#include "rsc_morton.cuh"

namespace rsc {

// device allocations of one call, released on every return path
struct Allocs {
  static constexpr int kMax = 32;
  void* p[kMax] = {};
  int np = 0;
  cudaError_t get(void** out, size_t bytes) {
    if (np == kMax) return cudaErrorMemoryAllocation;
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
  // the sort's scratch (knn_reserve)
  uint64_t* keys_buf[2] = {nullptr, nullptr};
  uint32_t* idx_buf[2] = {nullptr, nullptr};
  uint32_t* mm = nullptr;
  void* tmp = nullptr;
  size_t tmp_bytes = 0;
};

// knn_reserve, uploads xyz[3 n] into S.aos, then knn_sort; synchronises.
int32_t knn_prepare(rsc_ctx* ctx, const float* xyz, int64_t n, KnnSearch& S);

// every device buffer of the search of n points: S.aos and the sort's scratch.  Allocates only.
int32_t knn_reserve(rsc_ctx* ctx, int64_t n, KnnSearch& S);

// from S.aos[3 S.n], already on the device (knn_reserve): sorts the finite points by Morton key and builds the sorted
// SoA; synchronises.
int32_t knn_sort(rsc_ctx* ctx, KnnSearch& S);

// one warp per query over the prepared search, for the queries at sorted positions [p_begin, p_end) ([0, n): every
// point).  d_nrm: [3 n] PCA normals (sign rule or towards viewpoint), or null for the lists alone; d_nbr: [n k] int64
// lists or null; d_lists: [n k] int32 lists or null (not with d_nbr).  Rows of points outside the range are not
// written.  Enqueues only.
int32_t knn_run(rsc_ctx* ctx, const KnnSearch& S, int32_t k, const double* viewpoint, float* d_nrm, int64_t* d_nbr,
                int32_t* d_lists, int64_t p_begin, int64_t p_end);

// ---- the sharded forms: every rank holds the rows [off, off + n) of a cloud of n_global points ----

// this rank's own argument problem for shard_check, or null (n = 0 allows null pointers)
const char* shard_own_problem(int64_t n, int64_t off, int64_t n_global, int32_t k, const void* xyz, const void* out);

// collective argument check (two all-reduces).  `own`: this rank's own problem (null: none); `opt`: this rank passes
// the optional row array (nbr, nrm_in), which must be all or none over the non-empty ranks; *opt_on: some rank does.
// Between the two all-reduces, when the arguments agree, reserve(*opt_on) allocates every buffer of the collective
// steps; its failure (false) counts as this rank's problem, so all ranks return together.
int32_t shard_check(rsc_ctx* ctx, Allocs& al, const char* fn, const char* own, int64_t n, int64_t n_global, int32_t k,
                    const double* viewpoint, bool opt, const std::function<bool(bool)>& reserve, bool* opt_on);

// the device buffers of the collective steps, owned by a KnnSearch's Allocs
struct ShardBufs {
  int W = 4;                         // int32 words per gathered record: xyz, (normal,) coverage
  int64_t words = 0;                 // int32 words of the row buffer
  int32_t* rec = nullptr;            // [n_global W] gathered records
  unsigned long long* cnt = nullptr; // [3] coverage counters
  int32_t* rows = nullptr;           // [words] rows returned to their owners
  float* nrm = nullptr;              // [3 n_global] gathered normals (with_nrm), else null
  // knn_reserve(n_global) and the buffers above; false on an allocation failure
  bool reserve(rsc_ctx* ctx, int64_t n_global, bool with_nrm, int64_t row_words, KnnSearch& S);
};

// this rank's share of the search: the sorted positions [p_begin, p_end)
struct ShardSlice {
  int64_t p_begin = 0, p_end = 0;
};

// RSC_NORMALS_TRACE=1: the sharded calls synchronise between their phases and print their times to stderr
struct PhaseClock {
  bool on = false;
  double t = 0.0, ms[5] = {0.0, 0.0, 0.0, 0.0, 0.0};  // gather, prepare, search, exchange, forest
  PhaseClock();
  void mark(rsc_ctx* ctx, int phase);
  void print(const char* fn, rsc_ctx* ctx) const;
};

// gathers every rank's xyz (and nrm, when B.nrm is not null) into S (and B.nrm) on every rank with
// one all-reduce, checks that the ranges tile [0, n_global), runs knn_sort and picks this rank's slice: the
// non-empty ranks split the finite points into equal contiguous runs in range order, the last one also takes the
// non-finite tail.  Synchronises.
int32_t shard_gather(rsc_ctx* ctx, const char* fn, const float* xyz, const float* nrm, int64_t off, int64_t n,
                     int64_t n_global, KnnSearch& S, const ShardBufs& B, ShardSlice& sl, PhaseClock& clk);

// the per-point scratch of orient_forest on n points (the union-find, the per-component minima, F's edges, ...)
struct OrientScratch {
  double* u = nullptr;
  uint32_t *word = nullptr, *link = nullptr, *cnt = nullptr;
  unsigned long long *offs = nullptr, *best_w = nullptr, *best_e = nullptr, *tree = nullptr, *scal = nullptr;
};
// allocates it (and zeroes the counters on the context stream)
int32_t orient_reserve(rsc_ctx* ctx, Allocs& al, int64_t n, OrientScratch& O);

// everything of rsc_orient_normals after the search, on n points: d_xyz [3 n] AoS, d_nrm [3 n] (oriented in place),
// d_lists [n k] int32; edges / stats (host, nullable) as in rsc.h.  The graph's edge lists are allocated from `al`.
// Synchronises.
int32_t orient_forest(rsc_ctx* ctx, Allocs& al, const OrientScratch& O, const float* d_xyz, float* d_nrm,
                      const int32_t* d_lists, int64_t n, int32_t k, int64_t* edges, int64_t* stats);

}  // namespace rsc
