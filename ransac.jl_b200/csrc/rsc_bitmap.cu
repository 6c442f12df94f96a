// rsc_bitmap.cu -- parameter-space bitmap + largest connected component (extension, SURVEY 8(f)-4).
//
// The paper's third compatibility criterion -- "the point must be part of the largest connected
// component in the parameter space bitmap of the shape" -- which the reference documents and leaves
// out (docs/src/ransac.md:106-112; src/parameterspacebitmap.jl is dead code: bitmapparameters :12-46,
// largestconncomp :60-109, restated and pinned in oracle/ransac_oracle.py).  Here it is a filter on an
// inlier list, defined in oracle/ransac_oracle.py::bitmap_filter and implemented on the device:
//   1. bm_param_kernel   2-D parameters of every listed point on the shape, FP64, explicit roundings
//                        (plane: the reference's project2plane frame, plane.jl:82-103 / utilities.jl:84-92;
//                        sphere: Lambert's equal-area cylinder; cylinder: unrolled; cone: azimuth x slant
//                        distance) + per-CTA min / max
//   2. host              cell sizes from the bounding box and beta (the oracle's arithmetic, float64)
//   3. bm_bin_kernel     cell of every point, bitmap
//   4. union-find on the grid (4- or 8-connected, x wraps where the azimuth does): bm_init / bm_merge
//                        (atomicMin hooking) / bm_flatten; component sizes in CELLS; arg-max with ties to the
//                        smallest root = the component met first in column-major order, like
//                        argmax(component_lengths(label_components(...))) in the reference
//   5. bm_keep_kernel + scan + compaction: the points of that component, in input order
// Compiled with -fmad=false (the parameters must round like the oracle's).
#include <math.h>

#include "rsc_exact.cuh"

namespace rsc {

struct BmFrame {
  int type;
  double o[3];   // origin: plane point / sphere centre / cylinder centre / cone apex
  double ox[3], oy[3], oz[3];
  double R;      // sphere / cylinder radius
};

constexpr int kBmThreads = 256;

__global__ void __launch_bounds__(kBmThreads) bm_param_kernel(const float* __restrict__ soa, int64_t n_pad, const int64_t* __restrict__ idx,
                                                              int64_t n, BmFrame f, double2* __restrict__ uv,
                                                              double* __restrict__ partial /*[grid][4]: umin umax vmin vmax*/) {
  __shared__ double red[4][kBmThreads / 32];
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  double u = 0, v = 0;
  const bool live = i < n;
  if (live) {
    const int64_t p = idx[i];
    const ex::V3 P = {(double)soa[p], (double)soa[n_pad + p], (double)soa[2 * n_pad + p]};
    const ex::V3 V = ex::sub(P, ex::V3{f.o[0], f.o[1], f.o[2]});
    const ex::V3 ox = {f.ox[0], f.ox[1], f.ox[2]}, oy = {f.oy[0], f.oy[1], f.oy[2]}, oz = {f.oz[0], f.oz[1], f.oz[2]};
    if (f.type == RSC_PLANE) {
      u = ex::dot(V, ox);
      v = ex::dot(V, oy);
    } else if (f.type == RSC_SPHERE) {
      const double r = __dsqrt_rn(ex::dot(V, V));
      u = ex::mul(f.R, atan2(V.y, V.x));
      v = ex::mul(f.R, __ddiv_rn(V.z, r));
    } else if (f.type == RSC_CYLINDER) {
      u = ex::mul(f.R, atan2(ex::dot(V, oy), ex::dot(V, ox)));
      v = ex::dot(V, oz);
    } else {  // cone: raw azimuth and slant distance; the azimuth is scaled on the host side of step 2
      u = atan2(ex::dot(V, oy), ex::dot(V, ox));
      v = __dsqrt_rn(ex::dot(V, V));
    }
    uv[i] = make_double2(u, v);
  }
  const double inf = __longlong_as_double(0x7ff0000000000000ll);
  double a[4] = {live ? u : inf, live ? u : -inf, live ? v : inf, live ? v : -inf};
#pragma unroll
  for (int d = 16; d; d >>= 1) {
    a[0] = fmin(a[0], __shfl_xor_sync(0xffffffffu, a[0], d));
    a[1] = fmax(a[1], __shfl_xor_sync(0xffffffffu, a[1], d));
    a[2] = fmin(a[2], __shfl_xor_sync(0xffffffffu, a[2], d));
    a[3] = fmax(a[3], __shfl_xor_sync(0xffffffffu, a[3], d));
  }
  if ((threadIdx.x & 31) == 0)
    for (int k = 0; k < 4; ++k) red[k][threadIdx.x >> 5] = a[k];
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kBmThreads / 32; ++w) {
      a[0] = fmin(a[0], red[0][w]), a[1] = fmax(a[1], red[1][w]);
      a[2] = fmin(a[2], red[2][w]), a[3] = fmax(a[3], red[3][w]);
    }
    for (int k = 0; k < 4; ++k) partial[(size_t)blockIdx.x * 4 + k] = a[k];
  }
}

struct BmGrid {
  double su, umin, bu, vmin, bv;  // u = su * raw u
  int nu, nv, wrap, eight;
};

__global__ void bm_bin_kernel(const double2* __restrict__ uv, int64_t n, BmGrid g, int32_t* __restrict__ cell, uint8_t* __restrict__ bitmap) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double u = ex::mul(g.su, uv[i].x), v = uv[i].y;
  long long ix = (long long)floor(__ddiv_rn(ex::sub(u, g.umin), g.bu));
  long long iy = (long long)floor(__ddiv_rn(ex::sub(v, g.vmin), g.bv));
  ix = ix < 0 ? 0 : (ix > g.nu - 1 ? g.nu - 1 : ix);
  iy = iy < 0 ? 0 : (iy > g.nv - 1 ? g.nv - 1 : iy);
  const int c = (int)(ix + (long long)g.nu * iy);
  cell[i] = c;
  bitmap[c] = 1;
}

__global__ void bm_init_kernel(const uint8_t* __restrict__ bitmap, int ncells, int32_t* __restrict__ parent, int32_t* __restrict__ size) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ncells) return;
  parent[c] = bitmap[c] ? c : -1;
  size[c] = 0;
}

__device__ __forceinline__ int bm_find(const int32_t* parent, int c) {
  const volatile int32_t* vp = parent;  // other threads hook roots while we walk
  int p = vp[c];
  while (p != c) {
    c = p;
    p = vp[c];
  }
  return c;
}

__device__ inline void bm_union(int32_t* parent, int a, int b) {
  while (true) {
    a = bm_find(parent, a);
    b = bm_find(parent, b);
    if (a == b) return;
    if (a > b) {
      const int t = a;
      a = b;
      b = t;
    }
    const int old = atomicMin(&parent[b], a);  // hook the larger root under the smaller
    if (old == b) return;
    b = old;
  }
}

__global__ void bm_merge_kernel(BmGrid g, int32_t* __restrict__ parent) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= g.nu * g.nv || parent[c] < 0) return;
  const int x = c % g.nu, y = c / g.nu;
  auto link = [&](int ux, int uy) {
    if (g.wrap) ux = (ux + g.nu) % g.nu;
    if (ux < 0 || ux >= g.nu || uy < 0 || uy >= g.nv) return;
    const int d = ux + g.nu * uy;
    if (d != c && parent[d] >= 0) bm_union(parent, c, d);
  };
  link(x + 1, y);
  link(x, y + 1);
  if (g.eight) {
    link(x + 1, y + 1);
    link(x - 1, y + 1);
  }
}

__global__ void bm_flatten_kernel(int ncells, int32_t* __restrict__ parent, int32_t* __restrict__ size) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ncells || parent[c] < 0) return;
  const int r = bm_find(parent, c);
  parent[c] = r;
  atomicAdd(&size[r], 1);
}

// [0] = max over roots of (cells << 32 | 0xffffffff - root), [1] = number of components
__global__ void bm_best_kernel(int ncells, const int32_t* __restrict__ parent, const int32_t* __restrict__ size,
                               unsigned long long* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ncells || size[c] <= 0) return;  // size is only non-zero at roots
  atomicMax(out, ((unsigned long long)(uint32_t)size[c] << 32) | (unsigned long long)(0xffffffffu - (uint32_t)c));
  atomicAdd(out + 1, 1ull);
}

__global__ void bm_keep_kernel(const int32_t* __restrict__ cell, int64_t n, const int32_t* __restrict__ parent,
                               const unsigned long long* __restrict__ best, uint32_t* __restrict__ keep) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int root = (int)(0xffffffffu - (uint32_t)(best[0] & 0xffffffffull));
  keep[i] = parent[cell[i]] == root ? 1u : 0u;
}

__global__ void bm_compact_kernel(const int64_t* __restrict__ idx, int64_t n, const uint32_t* __restrict__ keep,
                                  const unsigned long long* __restrict__ offs, int64_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && keep[i]) out[offs[i]] = idx[i];
}

// host: the frame of the shape, in the oracle's operation order (oracle/ransac_oracle.py::shape_parameters2d)
static void h_normalize(const double* a, double* o) {
  const double inv = 1.0 / sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
  o[0] = inv * a[0], o[1] = inv * a[1], o[2] = inv * a[2];
}
static void h_cross(const double* a, const double* b, double* o) {
  o[0] = a[1] * b[2] - a[2] * b[1], o[1] = a[2] * b[0] - a[0] * b[2], o[2] = a[0] * b[1] - a[1] * b[0];
}
// utilities.jl:84-92 with the smallest component taken by magnitude (oracle: stable_orthogonal; the reference's
// version returns the zero vector for e.g. (0, 0, -1))
static void h_arbitrary_orthogonal(const double* vec, double* o) {
  double v[3];
  h_normalize(vec, v);
  const double a[3] = {fabs(v[0]), fabs(v[1]), fabs(v[2])};
  const bool b0 = (a[0] < a[1]) && (a[0] < a[2]);
  const bool b1 = (a[1] <= a[0]) && (a[1] < a[2]);
  const bool b2 = (a[2] <= a[0]) && (a[2] <= a[1]);
  const double rv[3] = {b0 ? 1.0 : 0.0, b1 ? 1.0 : 0.0, b2 ? 1.0 : 0.0};
  h_cross(v, rv, o);
}

// d_idx: n local point indices (device); d_out: capacity n (device).  Synchronises `st`.
int32_t bitmap_filter_dev(rsc_cloud* cloud, const rsc_cand& cand, double beta, bool eight, const int64_t* d_idx, int64_t n,
                          int64_t* d_out, int64_t* out_n, int32_t* info, cudaStream_t st) {
  rsc_ctx* ctx = cloud->ctx;
  if (info) info[0] = info[1] = info[2] = info[3] = 0;
  *out_n = 0;
  if (n <= 0) return RSC_OK;
  if (!(beta > 0.0)) return fail(ctx, RSC_E_ARG, "bitmap_filter: beta must be positive");
  if (n >= 2147483647LL) return fail(ctx, RSC_E_ARG, "bitmap_filter: too many points");
  BmFrame f;
  f.type = cand.type;
  f.R = 1.0;
  const double* p = cand.p;
  double axis[3];
  switch (cand.type) {
    case RSC_PLANE:
      f.o[0] = p[0], f.o[1] = p[1], f.o[2] = p[2];
      h_normalize(p + 3, f.oz);
      break;
    case RSC_SPHERE:
      f.o[0] = p[0], f.o[1] = p[1], f.o[2] = p[2];
      f.R = p[3];
      f.oz[0] = 0, f.oz[1] = 0, f.oz[2] = 1;
      break;
    case RSC_CYLINDER:
      f.o[0] = p[3], f.o[1] = p[4], f.o[2] = p[5];
      f.R = p[6];
      h_normalize(p, f.oz);
      break;
    case RSC_CONE:
      f.o[0] = p[0], f.o[1] = p[1], f.o[2] = p[2];
      h_normalize(p + 3, f.oz);
      break;
    default:
      return fail(ctx, RSC_E_ARG, "bitmap_filter: unknown shape type");
  }
  if (cand.type == RSC_SPHERE) {
    f.ox[0] = 1, f.ox[1] = 0, f.ox[2] = 0, f.oy[0] = 0, f.oy[1] = 1, f.oy[2] = 0;
  } else {
    double t[3];
    h_arbitrary_orthogonal(f.oz, t);
    h_normalize(t, f.ox);
    h_cross(f.oz, f.ox, axis);
    h_normalize(axis, f.oy);
  }
  const int grid = (int)((n + kBmThreads - 1) / kBmThreads);
  // scratch: uv [n] double2 | partial [grid][4] | cell [n] | keep [n] | offs [n+1]
  auto al = [](size_t b) { return (b + 255) / 256 * 256; };
  const size_t o_part = al((size_t)n * 16), o_cell = o_part + al((size_t)grid * 32), o_keep = o_cell + al((size_t)n * 4);
  const size_t o_offs = o_keep + al((size_t)n * 4), o_best = o_offs + al((size_t)(n + 1) * 8), total = o_best + 256;
  RSC_CUDA(ctx, ctx->lsqbuf.ensure(total));
  char* b = ctx->lsqbuf.as<char>();
  double2* uv = (double2*)b;
  double* partial = (double*)(b + o_part);
  int32_t* cell = (int32_t*)(b + o_cell);
  uint32_t* keep = (uint32_t*)(b + o_keep);
  unsigned long long* offs = (unsigned long long*)(b + o_offs);
  unsigned long long* best = (unsigned long long*)(b + o_best);
  bm_param_kernel<<<grid, kBmThreads, 0, st>>>(cloud->soa, cloud->n_pad, d_idx, n, f, uv, partial);
  RSC_CUDA(ctx, cudaGetLastError());
  std::vector<double> hp((size_t)grid * 4);
  RSC_CUDA(ctx, cudaMemcpyAsync(hp.data(), partial, hp.size() * 8, cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaStreamSynchronize(st));
  double umin = hp[0], umax = hp[1], vmin = hp[2], vmax = hp[3];
  for (int k = 1; k < grid; ++k) {
    umin = fmin(umin, hp[4 * k]), umax = fmax(umax, hp[4 * k + 1]);
    vmin = fmin(vmin, hp[4 * k + 2]), vmax = fmax(vmax, hp[4 * k + 3]);
  }
  if (!(umin == umin) || !(vmin == vmin) || !isfinite(umin) || !isfinite(umax) || !isfinite(vmin) || !isfinite(vmax))
    return fail(ctx, RSC_E_ARG, "bitmap_filter: a point has no finite parameters on this shape (on the axis / at the centre?)");
  // cell sizes: oracle/ransac_oracle.py::bitmap_filter, float64, round half to even
  BmGrid g;
  g.eight = eight ? 1 : 0;
  g.su = 1.0;
  g.wrap = cand.type != RSC_PLANE;
  double period = 0.0;
  if (cand.type == RSC_CONE) {
    double rref = fabs(sin(p[6] / 2)) * (0.5 * (vmin + vmax));
    if (!(rref > 1e-300)) rref = 1e-300;
    g.su = rref;
    period = 2 * M_PI * rref;
  } else if (cand.type == RSC_SPHERE) {
    period = 2 * M_PI * p[3];
  } else if (cand.type == RSC_CYLINDER) {
    period = 2 * M_PI * p[6];
  }
  const double nvd = fmax(1.0, nearbyint((vmax - vmin) / beta));
  g.vmin = vmin;
  g.bv = vmax > vmin ? (vmax - vmin) / nvd : 1.0;
  double nud;
  if (!g.wrap) {
    nud = fmax(1.0, nearbyint((umax - umin) / beta));
    g.umin = umin;
    g.bu = umax > umin ? (umax - umin) / nud : 1.0;
  } else {
    if (!(period > 0.0) || !isfinite(period)) return fail(ctx, RSC_E_ARG, "bitmap_filter: the shape has no positive radius");
    nud = fmax(3.0, nearbyint(period / beta));
    g.umin = -period / 2;
    g.bu = period / nud;
  }
  if (nud * nvd > (double)(1 << 26)) return fail(ctx, RSC_E_ARG, "bitmap_filter: more than 2^26 cells: beta is too small for this shape's extent");
  g.nu = (int)nud;
  g.nv = (int)nvd;
  const int ncells = g.nu * g.nv;
  const size_t o_par = al((size_t)ncells), o_size = o_par + al((size_t)ncells * 4);
  RSC_CUDA(ctx, ctx->cullbuf.ensure(o_size + al((size_t)ncells * 4)));
  uint8_t* bitmap = ctx->cullbuf.as<uint8_t>();
  int32_t* parent = (int32_t*)(ctx->cullbuf.as<char>() + o_par);
  int32_t* size = (int32_t*)(ctx->cullbuf.as<char>() + o_size);
  RSC_CUDA(ctx, cudaMemsetAsync(bitmap, 0, (size_t)ncells, st));
  RSC_CUDA(ctx, cudaMemsetAsync(best, 0, 16, st));
  bm_bin_kernel<<<grid, kBmThreads, 0, st>>>(uv, n, g, cell, bitmap);
  RSC_CUDA(ctx, cudaGetLastError());
  const int cgrid = (ncells + 255) / 256;
  bm_init_kernel<<<cgrid, 256, 0, st>>>(bitmap, ncells, parent, size);
  bm_merge_kernel<<<cgrid, 256, 0, st>>>(g, parent);
  bm_flatten_kernel<<<cgrid, 256, 0, st>>>(ncells, parent, size);
  bm_best_kernel<<<cgrid, 256, 0, st>>>(ncells, parent, size, best);
  RSC_CUDA(ctx, cudaGetLastError());
  bm_keep_kernel<<<grid, kBmThreads, 0, st>>>(cell, n, parent, best, keep);
  RSC_CUDA(ctx, cudaGetLastError());
  if (int32_t rc = scan_u32(ctx, keep, (int)n, offs, offs + n, st)) return rc;
  bm_compact_kernel<<<grid, kBmThreads, 0, st>>>(d_idx, n, keep, offs, d_out);
  RSC_CUDA(ctx, cudaGetLastError());
  unsigned long long hb[2] = {0, 0}, kept = 0;
  RSC_CUDA(ctx, cudaMemcpyAsync(hb, best, 16, cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaMemcpyAsync(&kept, offs + n, 8, cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaStreamSynchronize(st));
  *out_n = (int64_t)kept;
  if (info) info[0] = g.nu, info[1] = g.nv, info[2] = (int32_t)hb[1], info[3] = (int32_t)(hb[0] >> 32);
  return RSC_OK;
}

}  // namespace rsc

using namespace rsc;

extern "C" int32_t rsc_ctx_set_bitmap(rsc_ctx* ctx, double beta, int32_t eight) {
  if (!ctx) return RSC_E_ARG;
  if (!(beta > 0.0)) return fail(ctx, RSC_E_ARG, "set_bitmap: beta must be positive");
  ctx->bitmap_beta = beta;
  ctx->bitmap_eight = eight != 0;
  return RSC_OK;
}

extern "C" int32_t rsc_bitmap_filter(rsc_cloud* cloud, const rsc_cand* cand, double beta, int32_t eight, const int64_t* idx, int64_t n,
                                     int64_t* out_idx, int64_t* out_n, int32_t* info) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (!cand || !out_n || n < 0 || (n > 0 && (!idx || !out_idx))) return fail(ctx, RSC_E_ARG, "bitmap_filter: null arguments");
  if (cloud->exact()) return fail(ctx, RSC_E_STATE, "bitmap_filter: the bitmap filter does not support exact clouds yet");
  *out_n = 0;
  if (n == 0) {
    if (info) info[0] = info[1] = info[2] = info[3] = 0;
    return RSC_OK;
  }
  for (int64_t i = 0; i < n; ++i)
    if (idx[i] < 0 || idx[i] >= cloud->n) return fail(ctx, RSC_E_ARG, "bitmap_filter: index out of range");
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if (int32_t rc = cloud_ready(cloud)) return rc;
  cudaStream_t st = ctx->stream;
  RSC_CUDA(ctx, ctx->misc.ensure((size_t)n * 8));
  RSC_CUDA(ctx, ctx->misc2.ensure((size_t)n * 8));
  RSC_CUDA(ctx, cudaMemcpyAsync(ctx->misc.p, idx, (size_t)n * 8, cudaMemcpyHostToDevice, st));
  int32_t rc = bitmap_filter_dev(cloud, *cand, beta, eight != 0, ctx->misc.as<int64_t>(), n, ctx->misc2.as<int64_t>(), out_n, info, st);
  if (rc) return rc;
  if (*out_n > 0) RSC_CUDA(ctx, cudaMemcpy(out_idx, ctx->misc2.p, (size_t)*out_n * 8, cudaMemcpyDeviceToHost));
  return RSC_OK;
}
