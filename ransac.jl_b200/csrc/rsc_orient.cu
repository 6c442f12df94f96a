// rsc_orient.cu -- consistent normal signs without a viewpoint: the minimum spanning forest of the k-NN graph, signs
// propagated along it (rsc_orient_normals, DESIGN.md section 8).
//
// Vertices are the points with finite coordinates and a finite non-zero normal; u = n / |n| in float64.  The graph
// joins i and j (both vertices, i != j) when j is in N(i), the exact k-NN list of rsc_estimate_normals; the weight is
// w = 1 - |d|, d = u_i . u_j, and edges are ordered by (w, lo, hi), a strict total order, so the forest F is unique.
// It is built by Borůvka rounds over a parity union-find: every vertex holds its representative and the parity of its
// sign relative to it, packed into one word (rep << 1 | parity), so a word read alone is always consistent.
//   - each component with a crossing edge selects the minimum one by (w, lo, hi), for both endpoint components;
//   - it hooks to the component across that edge (when two choose the same edge the lower representative stays the
//     root) with parity par[lo] ^ par[hi] ^ (d < 0), and the edge joins F;
//   - pointer jumping flattens the hooks, XOR-ing the parities, and every vertex is relabelled;
//   - the edge list is compacted to the edges that still cross components; the rounds stop when none is left.
// The parity of v relative to its tree's root r is then the XOR of the flip bits (d < 0) along the unique tree path
// from r to v, which is the propagation rule s(c) = s(p) * sign(d(p, c)); it does not depend on the schedule.  Each
// tree is rooted at its vertex of largest float32 z (lowest index on ties, one 64-bit atomicMax) and its sign makes
// u_r.z positive (the largest-magnitude rule when u_r.z == 0).  The output is the input normal with its sign bit
// flipped or not.  Built with -fmad=false: u and d round like the oracle's (oracle/orient_oracle.py orient_mst).
#include <cub/device/device_radix_sort.cuh>

#include <cmath>

#include "rsc_normals.cuh"

namespace rsc {
namespace {

constexpr uint32_t kNotVertex = 0xffffffffu;  // union-find word of a point that is not a vertex
constexpr uint64_t kNone = ~(uint64_t)0;
constexpr int kTileEdges = 4096;               // edges per block of the compaction (256 threads x 16)
constexpr int kMaxRounds = 40;                 // > log2(2^31): a round that does not halve the components is a bug

struct Edge {
  uint64_t w;    // order-preserving bits of w = 1 - |d|
  uint64_t key;  // lo << 32 | hi
};

__device__ __forceinline__ uint64_t d2ord(double w) {
  const uint64_t b = (uint64_t)__double_as_longlong(w);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

__device__ __forceinline__ double dot_u(const double* __restrict__ u, int64_t a, int64_t b) {
  return (u[3 * a] * u[3 * b] + u[3 * a + 1] * u[3 * b + 1]) + u[3 * a + 2] * u[3 * b + 2];
}

// vertex test, unit vectors, singleton components
__global__ void __launch_bounds__(256) setup_kernel(const float* __restrict__ xyz, const float* __restrict__ nrm, int64_t n,
                                                    double* __restrict__ u, uint32_t* __restrict__ word,
                                                    unsigned long long* __restrict__ nvert) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool vert = false;
  if (i < n) {
    const float x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2];
    const double a = nrm[3 * i], b = nrm[3 * i + 1], c = nrm[3 * i + 2];
    const double len2 = (a * a + b * b) + c * c;
    vert = isfinite(x) && isfinite(y) && isfinite(z) && isfinite(a) && isfinite(b) && isfinite(c) && len2 > 0.0;
    if (vert) {
      const double len = sqrt(len2);
      u[3 * i] = a / len, u[3 * i + 1] = b / len, u[3 * i + 2] = c / len;
    }
    word[i] = vert ? (uint32_t)i << 1 : kNotVertex;
  }
  const int cnt = __syncthreads_count(vert);
  if (threadIdx.x == 0 && cnt) atomicAdd(nvert, (unsigned long long)cnt);
}

// the edge {i, j} of row i is kept once: from row i when i < j, or when i is not in N(j)
template <bool kWrite>
__global__ void __launch_bounds__(256) edges_kernel(const int32_t* __restrict__ lists, int k, int64_t n,
                                                    const uint32_t* __restrict__ word, const double* __restrict__ u,
                                                    uint32_t* __restrict__ cnt, const unsigned long long* __restrict__ offs,
                                                    Edge* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t c = 0;
  Edge* dst = kWrite ? out + offs[i] : nullptr;
  if (word[i] != kNotVertex) {
    for (int t = 0; t < k; ++t) {
      const int32_t j = lists[i * k + t];
      if (j < 0 || j == i || word[j] == kNotVertex) continue;
      bool keep = i < j;
      if (!keep) {
        keep = true;
        for (int s = 0; s < k; ++s) keep = keep && lists[(int64_t)j * k + s] != (int32_t)i;
      }
      if (!keep) continue;
      if (kWrite) {
        const uint64_t lo = (uint64_t)min((int64_t)j, i), hi = (uint64_t)max((int64_t)j, i);
        dst[c] = Edge{d2ord(1.0 - fabs(dot_u(u, (int64_t)lo, (int64_t)hi))), lo << 32 | hi};
      }
      ++c;
    }
  }
  if (!kWrite) cnt[i] = c;
}

__global__ void __launch_bounds__(256) reset_kernel(int64_t n, unsigned long long* __restrict__ a, unsigned long long* __restrict__ b) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] = kNone, b[i] = kNone;
}

// minimum w of the edges at each component, both endpoints (every edge of the list crosses components)
__global__ void __launch_bounds__(256) min_w_kernel(const Edge* __restrict__ e, int64_t m, const uint32_t* __restrict__ word,
                                                    unsigned long long* __restrict__ best_w) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < m; t += (int64_t)gridDim.x * blockDim.x) {
    const Edge x = e[t];
    const uint32_t cu = word[x.key >> 32] >> 1, cv = word[x.key & 0xffffffffu] >> 1;
    if (x.w < *(volatile unsigned long long*)(best_w + cu)) atomicMin(best_w + cu, (unsigned long long)x.w);
    if (x.w < *(volatile unsigned long long*)(best_w + cv)) atomicMin(best_w + cv, (unsigned long long)x.w);
  }
}

// then the minimum (lo, hi) among the edges of that weight
__global__ void __launch_bounds__(256) min_key_kernel(const Edge* __restrict__ e, int64_t m, const uint32_t* __restrict__ word,
                                                      const unsigned long long* __restrict__ best_w,
                                                      unsigned long long* __restrict__ best_e) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < m; t += (int64_t)gridDim.x * blockDim.x) {
    const Edge x = e[t];
    const uint32_t cu = word[x.key >> 32] >> 1, cv = word[x.key & 0xffffffffu] >> 1;
    if (x.w == best_w[cu]) atomicMin(best_e + cu, (unsigned long long)x.key);
    if (x.w == best_w[cv]) atomicMin(best_e + cv, (unsigned long long)x.key);
  }
}

// every representative with a selected edge hooks to the component across it, except the lower representative of two
// that selected the same edge; link[r] = (new parent << 1 | parity of r relative to it), the edge joins F
__global__ void __launch_bounds__(256) hook_kernel(int64_t n, const uint32_t* __restrict__ word,
                                                   const unsigned long long* __restrict__ best_e, const double* __restrict__ u,
                                                   uint32_t* __restrict__ link, unsigned long long* __restrict__ tree,
                                                   unsigned long long* __restrict__ ntree) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const uint32_t wr = word[r];
  if (wr != (uint32_t)r << 1) return;  // not a representative (or not a vertex)
  const uint64_t e = best_e[r];
  uint32_t l = (uint32_t)r << 1;
  if (e != kNone) {
    const int64_t lo = (int64_t)(e >> 32), hi = (int64_t)(e & 0xffffffffu);
    const uint32_t wl = word[lo], wh = word[hi];
    const uint32_t other = ((wl >> 1) == (uint32_t)r ? wh : wl) >> 1;
    if (!(best_e[other] == e && (uint32_t)r < other)) {
      const uint32_t flip = dot_u(u, lo, hi) < 0.0 ? 1u : 0u;
      l = other << 1 | ((wl ^ wh ^ flip) & 1u);
      tree[atomicAdd(ntree, 1ull)] = e;
    }
  }
  link[r] = l;
}

// one pointer-jumping step over the representatives; *changed is set while some link is not a root
__global__ void __launch_bounds__(256) jump_kernel(int64_t n, const uint32_t* __restrict__ word, uint32_t* link, int* changed) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n || word[r] != (uint32_t)r << 1) return;
  const uint32_t x = *(volatile uint32_t*)(link + r);
  const uint32_t y = *(volatile uint32_t*)(link + (x >> 1));
  if ((y >> 1) != (x >> 1)) {
    *(volatile uint32_t*)(link + r) = (y & ~1u) | ((x ^ y) & 1u);
    *changed = 1;
  }
}

__global__ void __launch_bounds__(256) relabel_kernel(int64_t n, uint32_t* __restrict__ word, const uint32_t* __restrict__ link) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  const uint32_t w = word[v];
  if (w == kNotVertex) return;
  const uint32_t l = link[w >> 1];
  word[v] = (l & ~1u) | ((w ^ l) & 1u);
}

__device__ __forceinline__ bool crossing(const Edge& x, const uint32_t* __restrict__ word) {
  return (word[x.key >> 32] >> 1) != (word[x.key & 0xffffffffu] >> 1);
}

// stable compaction of the edges that still cross components: counts per tile, scan_u32, scatter
__global__ void __launch_bounds__(256) cross_count_kernel(const Edge* __restrict__ e, int64_t m, const uint32_t* __restrict__ word,
                                                          uint32_t* __restrict__ cnt) {
  const int64_t base = (int64_t)blockIdx.x * kTileEdges;
  int c = 0;
  for (int it = 0; it < kTileEdges / 256; ++it) {
    const int64_t t = base + it * 256 + threadIdx.x;
    c += __syncthreads_count(t < m && crossing(e[t], word));
  }
  if (threadIdx.x == 0) cnt[blockIdx.x] = (uint32_t)c;
}

__global__ void __launch_bounds__(256) cross_scatter_kernel(const Edge* __restrict__ e, int64_t m, const uint32_t* __restrict__ word,
                                                            const unsigned long long* __restrict__ offs, Edge* __restrict__ out) {
  __shared__ int wc[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t base = (int64_t)blockIdx.x * kTileEdges;
  unsigned long long run = offs[blockIdx.x];
  for (int it = 0; it < kTileEdges / 256; ++it) {
    const int64_t t = base + it * 256 + threadIdx.x;
    Edge x;
    const bool keep = t < m && crossing(x = e[t], word);
    const unsigned b = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) wc[warp] = __popc(b);
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      before += w < warp ? wc[w] : 0;
      total += wc[w];
    }
    if (keep) out[run + before + __popc(b & ((1u << lane) - 1u))] = x;
    run += total;
    __syncthreads();
  }
}

// each tree's root: largest float32 z, lowest index on ties (-0 counts as +0)
__global__ void __launch_bounds__(256) root_kernel(int64_t n, const float* __restrict__ xyz, const uint32_t* __restrict__ word,
                                                   unsigned long long* __restrict__ root) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  const uint32_t w = word[v];
  if (w == kNotVertex) return;
  const float z = xyz[3 * v + 2];
  const uint64_t key = (uint64_t)f2ord(z == 0.f ? 0.f : z) << 32 | (uint64_t)(0xffffffffu - (uint32_t)v);
  atomicMax(root + (w >> 1), (unsigned long long)key);
}

__global__ void __launch_bounds__(256) sign_kernel(int64_t n, const uint32_t* __restrict__ word,
                                                   const unsigned long long* __restrict__ root, const double* __restrict__ u,
                                                   const float* in, float* out) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  const uint32_t w = word[v];
  uint32_t flip = 0;
  if (w != kNotVertex) {
    const int64_t r = 0xffffffffu - (uint32_t)(root[w >> 1] & 0xffffffffu);
    const double x = u[3 * r], y = u[3 * r + 1], z = u[3 * r + 2];
    bool neg = z < 0.0;
    if (z == 0.0) {  // the sign rule of rsc_estimate_normals: the largest-magnitude component positive, first on ties
      double big = x;
      if (fabs(y) > fabs(big)) big = y;
      neg = big < 0.0;
    }
    flip = (neg ? 1u : 0u) ^ ((w ^ word[r]) & 1u);
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) out[3 * v + a] = __uint_as_float(__float_as_uint(in[3 * v + a]) ^ (flip << 31));
}

__global__ void __launch_bounds__(256) pairs_kernel(const unsigned long long* __restrict__ keys, int64_t m, int64_t* __restrict__ out) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m) return;
  out[2 * t] = (int64_t)(keys[t] >> 32);
  out[2 * t + 1] = (int64_t)(keys[t] & 0xffffffffu);
}

inline unsigned blocks_of(int64_t n) { return (unsigned)((n + 255) / 256); }

}  // namespace
}  // namespace rsc

using namespace rsc;

#define ORI_CUDA(expr) RSC_CUDA(ctx, (expr))

int32_t rsc::orient_reserve(rsc_ctx* ctx, Allocs& al, int64_t n, OrientScratch& O) {
  ORI_CUDA(al.get((void**)&O.u, (size_t)n * 24));
  ORI_CUDA(al.get((void**)&O.word, (size_t)n * 4));
  ORI_CUDA(al.get((void**)&O.link, (size_t)n * 4));
  ORI_CUDA(al.get((void**)&O.cnt, (size_t)n * 4));
  ORI_CUDA(al.get((void**)&O.offs, (size_t)n * 8));
  ORI_CUDA(al.get((void**)&O.best_w, (size_t)n * 8));
  ORI_CUDA(al.get((void**)&O.best_e, (size_t)n * 8));
  ORI_CUDA(al.get((void**)&O.tree, (size_t)n * 8));
  ORI_CUDA(al.get((void**)&O.scal, 4 * 8));  // [0] vertices, [1] tree edges, [2] edges, [3] changed
  ORI_CUDA(cudaMemsetAsync(O.scal, 0, 4 * 8, ctx->stream));
  return RSC_OK;
}

int32_t rsc::orient_forest(rsc_ctx* ctx, Allocs& al, const OrientScratch& O, const float* d_xyz, float* d_nrm,
                           const int32_t* d_lists, int64_t n, int32_t k, int64_t* edges, int64_t* stats) {
  cudaStream_t st = ctx->stream;
  double* d_u = O.u;
  uint32_t *d_word = O.word, *d_link = O.link, *d_cnt = O.cnt;
  unsigned long long *d_best_w = O.best_w, *d_best_e = O.best_e, *d_tree = O.tree, *d_offs = O.offs, *d_scal = O.scal;

  const unsigned nb = blocks_of(n);
  setup_kernel<<<nb, 256, 0, st>>>(d_xyz, d_nrm, n, d_u, d_word, d_scal);
  ORI_CUDA(cudaGetLastError());
  edges_kernel<false><<<nb, 256, 0, st>>>(d_lists, k, n, d_word, d_u, d_cnt, nullptr, nullptr);
  ORI_CUDA(cudaGetLastError());
  if (int32_t rc = scan_u32(ctx, d_cnt, (int)n, d_offs, d_scal + 2, st)) return rc;
  unsigned long long got[3];
  ORI_CUDA(cudaMemcpyAsync(got, d_scal, 3 * 8, cudaMemcpyDeviceToHost, st));
  ORI_CUDA(cudaStreamSynchronize(st));
  const int64_t nvert = (int64_t)got[0];
  int64_t m = (int64_t)got[2];
  Edge* d_e[2] = {nullptr, nullptr};
  for (int b = 0; b < 2; ++b) ORI_CUDA(al.get((void**)&d_e[b], (size_t)m * sizeof(Edge)));
  uint32_t* d_tcnt = nullptr;
  unsigned long long* d_toff = nullptr;
  const int64_t max_tiles = (m + kTileEdges - 1) / kTileEdges;
  ORI_CUDA(al.get((void**)&d_tcnt, (size_t)max_tiles * 4));
  ORI_CUDA(al.get((void**)&d_toff, (size_t)max_tiles * 8));
  edges_kernel<true><<<nb, 256, 0, st>>>(d_lists, k, n, d_word, d_u, nullptr, d_offs, d_e[0]);
  ORI_CUDA(cudaGetLastError());

  const unsigned grid = (unsigned)ctx->sm_count * 16;
  int64_t rounds = 0;
  int cur = 0;
  while (m > 0) {
    if (++rounds > kMaxRounds) return fail(ctx, RSC_E_STATE, "orient_normals: Boruvka rounds did not converge");
    reset_kernel<<<nb, 256, 0, st>>>(n, d_best_w, d_best_e);
    ORI_CUDA(cudaGetLastError());
    min_w_kernel<<<grid, 256, 0, st>>>(d_e[cur], m, d_word, d_best_w);
    ORI_CUDA(cudaGetLastError());
    min_key_kernel<<<grid, 256, 0, st>>>(d_e[cur], m, d_word, d_best_w, d_best_e);
    ORI_CUDA(cudaGetLastError());
    hook_kernel<<<nb, 256, 0, st>>>(n, d_word, d_best_e, d_u, d_link, d_tree, d_scal + 1);
    ORI_CUDA(cudaGetLastError());
    for (int changed = 1; changed;) {
      ORI_CUDA(cudaMemsetAsync(d_scal + 3, 0, 4, st));
      jump_kernel<<<nb, 256, 0, st>>>(n, d_word, d_link, (int*)(d_scal + 3));
      ORI_CUDA(cudaGetLastError());
      ORI_CUDA(cudaMemcpyAsync(&changed, d_scal + 3, 4, cudaMemcpyDeviceToHost, st));
      ORI_CUDA(cudaStreamSynchronize(st));
    }
    relabel_kernel<<<nb, 256, 0, st>>>(n, d_word, d_link);
    ORI_CUDA(cudaGetLastError());
    const int tiles = (int)((m + kTileEdges - 1) / kTileEdges);
    cross_count_kernel<<<tiles, 256, 0, st>>>(d_e[cur], m, d_word, d_tcnt);
    ORI_CUDA(cudaGetLastError());
    if (int32_t rc = scan_u32(ctx, d_tcnt, tiles, d_toff, d_scal + 2, st)) return rc;
    cross_scatter_kernel<<<tiles, 256, 0, st>>>(d_e[cur], m, d_word, d_toff, d_e[cur ^ 1]);
    ORI_CUDA(cudaGetLastError());
    unsigned long long left = 0;
    ORI_CUDA(cudaMemcpyAsync(&left, d_scal + 2, 8, cudaMemcpyDeviceToHost, st));
    ORI_CUDA(cudaStreamSynchronize(st));
    m = (int64_t)left;
    cur ^= 1;
  }

  // roots and signs (d_best_w holds the root keys)
  ORI_CUDA(cudaMemsetAsync(d_best_w, 0, (size_t)n * 8, st));
  root_kernel<<<nb, 256, 0, st>>>(n, d_xyz, d_word, d_best_w);
  ORI_CUDA(cudaGetLastError());
  sign_kernel<<<nb, 256, 0, st>>>(n, d_word, d_best_w, d_u, d_nrm, d_nrm);
  ORI_CUDA(cudaGetLastError());
  unsigned long long ntree = 0;
  ORI_CUDA(cudaMemcpyAsync(&ntree, d_scal + 1, 8, cudaMemcpyDeviceToHost, st));
  ORI_CUDA(cudaStreamSynchronize(st));
  if (edges && ntree) {  // F's edges in ascending (lo, hi) order
    cub::DoubleBuffer<unsigned long long> kb(d_tree, d_best_e);
    size_t tmp_bytes = 0;
    void* d_tmp = nullptr;
    ORI_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, kb, (int)ntree, 0, 64, st));
    ORI_CUDA(al.get(&d_tmp, tmp_bytes));
    ORI_CUDA(cub::DeviceRadixSort::SortKeys(d_tmp, tmp_bytes, kb, (int)ntree, 0, 64, st));
    int64_t* d_pairs = reinterpret_cast<int64_t*>(d_e[0]);  // the edge lists are free now; 16 B per edge either way
    pairs_kernel<<<blocks_of((int64_t)ntree), 256, 0, st>>>(kb.Current(), (int64_t)ntree, d_pairs);
    ORI_CUDA(cudaGetLastError());
    if (int32_t rc = staged_d2h(ctx, edges, d_pairs, (size_t)ntree * 16, st)) return rc;
  }
  if (stats) {
    stats[0] = nvert;
    stats[1] = (int64_t)ntree;
    stats[2] = nvert - (int64_t)ntree;
    stats[3] = rounds;
  }
  return RSC_OK;
}

extern "C" int32_t rsc_orient_normals(rsc_ctx* ctx, const float* xyz, int64_t n, int32_t k, const float* nrm_in, float* nrm_out,
                                      int64_t* edges, int64_t* stats) {
  if (!ctx) return RSC_E_ARG;
  if (!xyz || !nrm_out) return fail(ctx, RSC_E_ARG, "orient_normals: xyz and nrm_out must not be NULL");
  if (k < 3 || k > 32) return fail(ctx, RSC_E_ARG, "orient_normals: k must be in [3, 32]");
  if (n < 1 || n >= ((int64_t)1 << 31)) return fail(ctx, RSC_E_ARG, "orient_normals: n must be in [1, 2^31)");
  KnnSearch S;
  OrientScratch O;
  if (int32_t rc = knn_prepare(ctx, xyz, n, S)) return rc;
  cudaStream_t st = ctx->stream;
  float* d_nrm = nullptr;
  int32_t* d_lists = nullptr;
  ORI_CUDA(S.al.get((void**)&d_nrm, (size_t)n * 12));
  ORI_CUDA(S.al.get((void**)&d_lists, (size_t)n * k * 4));
  if (int32_t rc = orient_reserve(ctx, S.al, n, O)) return rc;
  if (nrm_in) ORI_CUDA(cudaMemcpyAsync(d_nrm, nrm_in, (size_t)n * 12, cudaMemcpyHostToDevice, st));
  // one search: the lists, and the normals too when none are given
  if (int32_t rc = knn_run(ctx, S, k, nullptr, nrm_in ? nullptr : d_nrm, nullptr, d_lists, 0, n)) return rc;
  if (int32_t rc = orient_forest(ctx, S.al, O, S.aos, d_nrm, d_lists, n, k, edges, stats)) return rc;
  if (int32_t rc = staged_d2h(ctx, nrm_out, d_nrm, (size_t)n * 12, st)) return rc;
  return RSC_OK;
}

extern "C" int32_t rsc_orient_normals_shard(rsc_ctx* ctx, const float* xyz, int64_t n, int64_t global_offset, int64_t n_global,
                                            int32_t k, const float* nrm_in, float* nrm_out, int64_t* edges, int64_t* stats) {
  constexpr const char* fn = "orient_normals_shard";
  if (!ctx) return RSC_E_ARG;
  KnnSearch S;
  ShardBufs B;
  OrientScratch O;
  PhaseClock clk;
  bool given = false;
  // given normals travel with the coordinates; estimated ones come back with the lists: [n_global k] int32 lists,
  // then [3 n_global] normals, zero-filled and completed by one all-reduce
  auto reserve = [&](bool with_nrm) {
    return B.reserve(ctx, n_global, with_nrm, n_global * ((int64_t)k + (with_nrm ? 0 : 3)), S) &&
           orient_reserve(ctx, S.al, n_global, O) == RSC_OK;
  };
  if (int32_t rc = shard_check(ctx, S.al, fn, shard_own_problem(n, global_offset, n_global, k, xyz, nrm_out), n, n_global, k,
                               nullptr, nrm_in != nullptr, reserve, &given))
    return rc;
  ShardSlice sl;
  if (int32_t rc = shard_gather(ctx, fn, xyz, nrm_in, global_offset, n, n_global, S, B, sl, clk)) return rc;
  clk.mark(ctx, 1);
  const int64_t words = B.words;
  int32_t* d_rows = B.rows;
  float* d_nrm = given ? B.nrm : reinterpret_cast<float*>(d_rows + (int64_t)k * n_global);
  cudaStream_t st = ctx->stream;
  ORI_CUDA(cudaMemsetAsync(d_rows, 0, (size_t)words * 4, st));
  if (int32_t rc = knn_run(ctx, S, k, nullptr, given ? nullptr : d_nrm, nullptr, d_rows, sl.p_begin, sl.p_end)) return rc;
  clk.mark(ctx, 2);
  if (int32_t rc = rsc_ctx_allreduce(ctx, d_rows, words, st)) return rc;
  clk.mark(ctx, 3);
  // the forest, replicated on identical inputs: identical on every rank
  if (int32_t rc = orient_forest(ctx, S.al, O, S.aos, d_nrm, d_rows, n_global, k, edges, stats)) return rc;
  if (n > 0)
    if (int32_t rc = staged_d2h(ctx, nrm_out, d_nrm + 3 * global_offset, (size_t)n * 12, st)) return rc;
  ORI_CUDA(cudaStreamSynchronize(st));
  clk.mark(ctx, 4);
  clk.print(fn, ctx);
  return RSC_OK;
}
#undef ORI_CUDA
