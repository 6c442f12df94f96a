// rsc_octree.cu -- flattened octree of the cloud for the level-weighted cell sampler (SURVEY 8(f)-1).
//
// Replaces the RegionTrees octree of the reference (octree.jl:158-244: cells split while they hold
// more than 8 points, children halve every axis of the parent box) by a Morton-ordered grid
// hierarchy: points are quantised to D = nlevels-1 bits per axis inside the cloud's bounding box,
// sorted by their interleaved code, and a level-l cell is the contiguous range of sorted positions
// sharing the top 3(l-1) code bits -- no tree is stored.  Per point: its Morton rank (inv), and
// leafdepth = the first level at which its cell holds <= 8 points (what findleaf + cell depth give in
// the reference, fitting.jl:397-401).  The sampler (rsc_fit.cu) additionally keeps pc.isenabled in
// Morton order with a rank/select index, so that "the j-th enabled point of a cell" is O(log n).
//
// The semantics (quantisation, bit order, tie order, leafdepth) are restated in
// oracle/ransac_oracle.py::MortonOctree; tests compare the two bit for bit.
#include <cub/device/device_radix_sort.cuh>

#include "rsc_common.cuh"
#include "rsc_morton.cuh"

namespace rsc {

__global__ void __launch_bounds__(256) bbox_kernel(const float* __restrict__ soa, int64_t n, int64_t n_pad, uint32_t* __restrict__ mm,
                                                   bool finite_only) {
  uint32_t lo[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, hi[3] = {0u, 0u, 0u};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float x = soa[i], y = soa[n_pad + i], z = soa[2 * n_pad + i];
    if (finite_only && !(isfinite(x) && isfinite(y) && isfinite(z))) continue;
    const float v[3] = {x, y, z};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const uint32_t o = f2ord(v[a]);
      lo[a] = min(lo[a], o);
      hi[a] = max(hi[a], o);
    }
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    lo[a] = __reduce_min_sync(0xffffffffu, lo[a]);
    hi[a] = __reduce_max_sync(0xffffffffu, hi[a]);
  }
  if ((threadIdx.x & 31) == 0)
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      atomicMin(mm + a, lo[a]);
      atomicMax(mm + 3 + a, hi[a]);
    }
}

__global__ void __launch_bounds__(256) morton_kernel(const float* __restrict__ soa, int64_t n, int64_t n_pad, Quant q,
                                                     uint32_t* __restrict__ codes, uint32_t* __restrict__ idx) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t c[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) c[a] = quantise(soa[a * n_pad + i], q, a);
  uint32_t code = 0;
  for (int b = q.D - 1; b >= 0; --b) code = (code << 3) | (((c[0] >> b) & 1u) << 2) | (((c[1] >> b) & 1u) << 1) | ((c[2] >> b) & 1u);
  codes[i] = code;
  idx[i] = (uint32_t)i;
}

__global__ void __launch_bounds__(256) invert_kernel(const uint32_t* __restrict__ perm, int64_t n, uint32_t* __restrict__ inv) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) inv[perm[i]] = (uint32_t)i;
}

// first position in codes[lo, hi) whose code is >= key
__device__ __forceinline__ int64_t lower_bound_u32(const uint32_t* __restrict__ codes, int64_t lo, int64_t hi, uint64_t key) {
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if ((uint64_t)__ldg(codes + mid) < key)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(256) leafdepth_kernel(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ perm,
                                                        int64_t n, int nlevels, uint8_t* __restrict__ leafdepth) {
  const int64_t pos = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pos >= n) return;
  const int D = nlevels - 1;
  const uint32_t code = codes[pos];
  int64_t a = 0, b = n;  // range of the level-1 cell (root)
  int ld = nlevels;
  for (int l = 1; l <= nlevels; ++l) {
    if (l > 1) {  // children nest: search inside the parent's range only
      const int shift = 3 * (D - (l - 1));
      const uint64_t lo_key = (uint64_t)(code >> shift) << shift;
      const int64_t na = lower_bound_u32(codes, a, b, lo_key);
      const int64_t nb = lower_bound_u32(codes, na, b, lo_key + ((uint64_t)1 << shift));
      a = na, b = nb;
    }
    if (b - a <= 8) {
      ld = l;
      break;
    }
  }
  leafdepth[perm[pos]] = (uint8_t)ld;
}

// pc.isenabled in Morton order: bit p of en_sorted = enabled[perm[p]]
__global__ void __launch_bounds__(256) gather_sorted_enabled_kernel(const uint32_t* __restrict__ enabled,
                                                                     const uint32_t* __restrict__ perm, int64_t n,
                                                                     int64_t words, uint32_t* __restrict__ en_sorted) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // one sorted position per thread
  const int64_t w = p >> 5;
  if (w >= words) return;
  bool on = false;
  if (p < n) {
    const uint32_t i = __ldg(perm + p);
    on = (__ldg(enabled + (i >> 5)) >> (i & 31)) & 1u;
  }
  const uint32_t v = __ballot_sync(0xffffffffu, on);
  if ((threadIdx.x & 31) == 0) en_sorted[w] = v;
}

int32_t cells_refresh_enabled(rsc_cloud* cloud, cudaStream_t st) {
  rsc_ctx* ctx = cloud->ctx;
  rsc_cells& c = cloud->cells;
  if (c.nlevels == 0 || c.en_valid) return RSC_OK;
  const int64_t words = cloud->n_pad / 32;
  gather_sorted_enabled_kernel<<<(unsigned)((cloud->n_pad + 255) / 256), 256, 0, st>>>(cloud->enabled, c.perm, cloud->n, words,
                                                                                       c.en_sorted);
  RSC_CUDA(ctx, cudaGetLastError());
  c.en_valid = true;
  c.sel_valid = false;
  return RSC_OK;
}

void cells_release(rsc_cloud* cloud) {
  rsc_cells& c = cloud->cells;
  if (c.codes) cudaFree(c.codes);
  if (c.perm) cudaFree(c.perm);
  if (c.perm64) cudaFree(c.perm64);
  if (c.inv) cudaFree(c.inv);
  if (c.leafdepth) cudaFree(c.leafdepth);
  if (c.en_sorted) cudaFree(c.en_sorted);
  if (c.msoa) cudaFree(c.msoa);
  if (c.tiles) cudaFree(c.tiles);
  c.selbuf.release();
  c = rsc_cells();
}

// ---- Morton view of a subset copy for the culled scorer (rsc_cull.cu) ------------------------------------
__global__ void __launch_bounds__(256) cull_view_gather_kernel(const float* __restrict__ soa, int64_t m_pad, const int64_t* __restrict__ idx,
                                                               const uint32_t* __restrict__ perm, int64_t m, float* __restrict__ csoa,
                                                               int64_t* __restrict__ cidx) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= m_pad) return;
  const bool real = p < m;
  const int64_t j = real ? (int64_t)perm[p] : 0;
#pragma unroll
  for (int f = 0; f < 6; ++f) csoa[f * m_pad + p] = real ? soa[f * m_pad + j] : 0.f;
  if (real) cidx[p] = idx[j];
}

// The subset's points sorted by a 30-bit Morton code (10 bits per axis inside the subset's bounding box; only the
// ORDER matters, for how small the tiles' bounding spheres are -- counts do not depend on it), the cloud indices
// and pc.isenabled in that order, and the spheres.  Kept with the subset until its coordinates change.
int32_t subset_cull_view(rsc_cloud* cloud, rsc_subset& s, cudaStream_t st) {
  rsc_ctx* ctx = cloud->ctx;
  if (s.csoa) return RSC_OK;
  if (s.m >= ((int64_t)1 << 31)) return fail(ctx, RSC_E_ARG, "culled scorer: subset too large");
  const int64_t m = s.m, words = s.m_pad / 32;
  const int64_t nsph = (int64_t)cull_sphere_count(s.m_pad);
  auto bail = [&](cudaError_t e, const char* what) {
    s.release_cull_view();
    return fail_cuda(ctx, e, what);
  };
  cudaError_t e;
#define CV(expr) \
  if ((e = (expr)) != cudaSuccess) return bail(e, #expr)
  CV(cudaMalloc(&s.csoa, (size_t)6 * s.m_pad * sizeof(float)));
  CV(cudaMalloc(&s.cen, (size_t)words * 4));
  CV(cudaMalloc(&s.cidx, (size_t)(m > 0 ? m : 1) * sizeof(int64_t)));
  CV(cudaMalloc(&s.ctiles, (size_t)nsph * sizeof(float4)));
  // temporaries live in a scratch buffer of the context (no cudaMalloc / cudaFree per view: a cudaFree in the middle
  // of a run synchronises the device and was seen to take tens of milliseconds): codes in/out, positions in/out,
  // bounding box, CUB's workspace
  const size_t mm1 = (size_t)(m > 0 ? m : 1);
  const size_t o_cout = (mm1 * 4 + 255) / 256 * 256, o_iin = 2 * o_cout, o_perm = 3 * o_cout, o_mm = 4 * o_cout, o_tmp = o_mm + 256;
  size_t tmp_bytes = 0;
  CV(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const uint32_t*)nullptr,
                                     (uint32_t*)nullptr, (int)mm1, 0, 30, st));
  CV(ctx->viewtmp.ensure(o_tmp + tmp_bytes + 16));
  char* b = ctx->viewtmp.as<char>();
  uint32_t* codes_in = reinterpret_cast<uint32_t*>(b);
  uint32_t* codes_out = reinterpret_cast<uint32_t*>(b + o_cout);
  uint32_t* idx_in = reinterpret_cast<uint32_t*>(b + o_iin);
  uint32_t* perm = reinterpret_cast<uint32_t*>(b + o_perm);
  uint32_t* mm = reinterpret_cast<uint32_t*>(b + o_mm);
  if (m > 0) {
    const uint32_t init[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
    CV(cudaMemcpyAsync(mm, init, sizeof(init), cudaMemcpyHostToDevice, st));
    bbox_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(s.soa, m, s.m_pad, mm, false);
    CV(cudaGetLastError());
    uint32_t got[6];
    CV(cudaMemcpyAsync(got, mm, sizeof(got), cudaMemcpyDeviceToHost, st));
    CV(cudaStreamSynchronize(st));
    Quant q;
    q.D = 10;
    q.scale = 1024.0;
    q.qmax = 1023u;
    for (int a = 0; a < 3; ++a) {
      const double lo = (double)ord2f(got[a]), hi = (double)ord2f(got[3 + a]);
      q.lo[a] = lo;
      q.w[a] = hi - lo;
      if (!(q.w[a] > 0.0)) q.w[a] = 1.0;
    }
    morton_kernel<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(s.soa, m, s.m_pad, q, codes_in, idx_in);
    CV(cudaGetLastError());
    CV(cub::DeviceRadixSort::SortPairs(b + o_tmp, tmp_bytes, codes_in, codes_out, idx_in, perm, (int)m, 0, 30, st));
  }
  cull_view_gather_kernel<<<(unsigned)((s.m_pad + 255) / 256), 256, 0, st>>>(s.soa, s.m_pad, s.idx, perm, m, s.csoa, s.cidx);
  CV(cudaGetLastError());
  {
    PointSet ps;
    ps.x = s.csoa, ps.y = s.csoa + s.m_pad, ps.z = s.csoa + 2 * s.m_pad;
    ps.n = m, ps.n_pad = s.m_pad;
    if (int32_t rc = cull_tile_spheres(ctx, ps, reinterpret_cast<float4*>(s.ctiles), st)) {
      s.release_cull_view();
      return rc;
    }
  }
#undef CV
  // pc.isenabled in the new order (stream order keeps the scratch buffer safe: everything above was enqueued on st)
  if (int32_t rc = refresh_subsets_enabled(cloud, st)) return rc;
  return RSC_OK;
}

}  // namespace rsc

using namespace rsc;

extern "C" {

int32_t rsc_cloud_build_cells(rsc_cloud* cloud, int32_t nlevels) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (nlevels < 1 || nlevels > 11) return fail(ctx, RSC_E_ARG, "build_cells: nlevels must be 1..11 (30-bit Morton codes)");
  if (cloud->n <= 0 || cloud->n >= ((int64_t)1 << 31)) return fail(ctx, RSC_E_ARG, "build_cells: cloud size must be below 2^31 points per shard");
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if (int32_t rcr = cloud_ready(cloud)) return rcr;
  cudaStream_t st = ctx->stream;
  cells_release(cloud);
  rsc_cells& c = cloud->cells;
  const int64_t n = cloud->n;
  uint32_t *codes_in = nullptr, *idx_in = nullptr, *mm = nullptr;
  void* tmp = nullptr;
  auto bail = [&](cudaError_t e, const char* what) {
    if (codes_in) cudaFree(codes_in);
    if (idx_in) cudaFree(idx_in);
    if (mm) cudaFree(mm);
    if (tmp) cudaFree(tmp);
    cells_release(cloud);
    return fail_cuda(ctx, e, what);
  };
  cudaError_t e;
#define OCT(expr)                         \
  if ((e = (expr)) != cudaSuccess) return bail(e, #expr)
  OCT(cudaMalloc(&c.codes, (size_t)n * 4));
  OCT(cudaMalloc(&c.perm, (size_t)n * 4));
  OCT(cudaMalloc(&c.inv, (size_t)n * 4));
  OCT(cudaMalloc(&c.leafdepth, (size_t)n));
  OCT(cudaMalloc(&c.en_sorted, (size_t)(cloud->n_pad / 32) * 4));
  OCT(cudaMalloc(&codes_in, (size_t)n * 4));
  OCT(cudaMalloc(&idx_in, (size_t)n * 4));
  OCT(cudaMalloc(&mm, 6 * 4));
  const uint32_t init[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
  OCT(cudaMemcpyAsync(mm, init, sizeof(init), cudaMemcpyHostToDevice, st));
  bbox_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(cloud->soa, n, cloud->n_pad, mm, false);
  OCT(cudaGetLastError());
  uint32_t got[6];
  OCT(cudaMemcpyAsync(got, mm, sizeof(got), cudaMemcpyDeviceToHost, st));
  OCT(cudaStreamSynchronize(st));
  Quant q;
  q.D = nlevels - 1;
  q.scale = (double)((uint64_t)1 << q.D);
  q.qmax = (1u << q.D) - 1u;
  for (int a = 0; a < 3; ++a) {
    const double lo = (double)ord2f(got[a]), hi = (double)ord2f(got[3 + a]);
    q.lo[a] = lo;
    q.w[a] = hi - lo;
    if (!(q.w[a] > 0.0)) q.w[a] = 1.0;  // degenerate axis (also NaN): everything lands in cell 0
    c.lo[a] = q.lo[a], c.w[a] = q.w[a];
  }
  morton_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(cloud->soa, n, cloud->n_pad, q, codes_in, idx_in);
  OCT(cudaGetLastError());
  size_t tmp_bytes = 0;
  const int end_bit = q.D > 0 ? 3 * q.D : 1;
  OCT(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, codes_in, c.codes, idx_in, c.perm, (int)n, 0, end_bit, st));
  OCT(cudaMalloc(&tmp, tmp_bytes ? tmp_bytes : 16));
  OCT(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, codes_in, c.codes, idx_in, c.perm, (int)n, 0, end_bit, st));  // stable
  invert_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(c.perm, n, c.inv);
  OCT(cudaGetLastError());
  leafdepth_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(c.codes, c.perm, n, nlevels, c.leafdepth);
  OCT(cudaGetLastError());
  OCT(cudaStreamSynchronize(st));
#undef OCT
  cudaFree(codes_in), cudaFree(idx_in), cudaFree(mm), cudaFree(tmp);
  c.nlevels = nlevels;
  c.en_valid = false;
  c.sel_valid = false;
  return RSC_OK;
}

int32_t rsc_cloud_cells_levels(const rsc_cloud* cloud) { return cloud ? cloud->cells.nlevels : 0; }

int32_t rsc_cloud_get_cells(rsc_cloud* cloud, uint32_t* codes_sorted, uint32_t* perm, uint8_t* leafdepth) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  const rsc_cells& c = cloud->cells;
  if (c.nlevels == 0) return fail(ctx, RSC_E_STATE, "get_cells: rsc_cloud_build_cells has not been called");
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  RSC_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (codes_sorted) RSC_CUDA(ctx, cudaMemcpy(codes_sorted, c.codes, (size_t)cloud->n * 4, cudaMemcpyDeviceToHost));
  if (perm) RSC_CUDA(ctx, cudaMemcpy(perm, c.perm, (size_t)cloud->n * 4, cudaMemcpyDeviceToHost));
  if (leafdepth) RSC_CUDA(ctx, cudaMemcpy(leafdepth, c.leafdepth, (size_t)cloud->n, cudaMemcpyDeviceToHost));
  return RSC_OK;
}

}  // extern "C"
