// rsc_normals.cu -- oriented PCA normals of the k nearest neighbours (rsc_estimate_normals, DESIGN.md section 8).
//
// N(i) is the k_eff = min(k, finite points) finite points j smallest in (d2(i, j), j) order, with
// d2 = ((xj-xi)^2 + (yj-yi)^2) + (zj-zi)^2 in float64 (no FMA: this file is compiled with -fmad=false), so the lists
// are the oracle's (oracle/normals_oracle.py) bit for bit.  The search is exact by construction:
//   - finite points are quantised to 21 bits per axis inside their bounding box (the octree's float64 formula,
//     rsc_morton.cuh), interleaved into 63-bit Morton keys and sorted; a level-l cell (2^(l-1) cells per axis) is
//     a contiguous range of sorted keys;
//   - one warp per query, queries in Morton order.  The search starts at the deepest level whose cell around the
//     query holds >= k_eff points, scans the 27 cells around it and keeps the best k in lanes, sorted across the warp;
//   - it accepts when the k-th d2 < r_safe^2, r_safe = the distance from the query to the boundary of the 3x3x3 block
//     minus a bound on the quantisation's float64 rounding: every point outside the block is then strictly farther
//     than the k-th.  Otherwise it rescans one level up; level 2 and level 1 cover the whole box.
// Then, in the same warp: the float64 covariance of N(i) in list order, cyclic Jacobi, the sign rule, and the stores
// by original index.  rsc_orient_normals (rsc_orient.cu) runs the same search through knn_prepare / knn_run
// (rsc_normals.cuh) and keeps the lists on the device as int32.  The sharded forms (rsc_*_normals_shard) gather the
// cloud on every rank, sort it identically there and give each rank a contiguous run of the sorted queries.
#include <cub/device/device_radix_sort.cuh>

#include <chrono>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>

#include "rsc_normals.cuh"

namespace rsc {
namespace {

constexpr int kKeyBits = 21;                        // bits per axis of the Morton keys: levels 1 .. kKeyBits + 1
constexpr uint64_t kNonFinite = ~(uint64_t)0;       // key of a point with a non-finite coordinate: sorts last
constexpr double kTau = 0x1p-40;                    // degenerate neighbourhood: middle eigenvalue <= kTau * largest
constexpr int kJacobiSweeps = 16;
constexpr int kWarpsPerBlock = 8;

__global__ void __launch_bounds__(256) aos_to_soa_kernel(const float* __restrict__ aos, int64_t n, float* __restrict__ soa) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
#pragma unroll
  for (int a = 0; a < 3; ++a) soa[a * n + i] = aos[3 * i + a];
}

__device__ __forceinline__ uint64_t interleave(uint32_t cx, uint32_t cy, uint32_t cz, int bits) {
  uint64_t key = 0;
  for (int b = bits - 1; b >= 0; --b)
    key = (key << 3) | ((uint64_t)((cx >> b) & 1u) << 2) | ((uint64_t)((cy >> b) & 1u) << 1) | (uint64_t)((cz >> b) & 1u);
  return key;
}

__global__ void __launch_bounds__(256) keys_kernel(const float* __restrict__ soa, int64_t n, Quant q, uint64_t* __restrict__ keys,
                                                   uint32_t* __restrict__ idx, unsigned long long* __restrict__ n_finite) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool fin = false;
  if (i < n) {
    const float x = soa[i], y = soa[n + i], z = soa[2 * n + i];
    fin = isfinite(x) && isfinite(y) && isfinite(z);
    keys[i] = fin ? interleave(quantise(x, q, 0), quantise(y, q, 1), quantise(z, q, 2), kKeyBits) : kNonFinite;
    idx[i] = (uint32_t)i;
  }
  const int c = __syncthreads_count(fin);
  if (threadIdx.x == 0 && c) atomicAdd(n_finite, (unsigned long long)c);
}

__global__ void __launch_bounds__(256) gather_sorted_kernel(const float* __restrict__ aos, const uint32_t* __restrict__ perm, int64_t n,
                                                            float* __restrict__ soa) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const int64_t j = perm[p];
#pragma unroll
  for (int a = 0; a < 3; ++a) soa[a * n + p] = aos[3 * j + a];
}

// first position in keys[lo, hi) whose key is >= key
__device__ __forceinline__ int32_t lower_bound_u64(const uint64_t* __restrict__ keys, int32_t lo, int32_t hi, uint64_t key) {
  while (lo < hi) {
    const int32_t mid = (int32_t)(((uint32_t)lo + (uint32_t)hi) >> 1);
    if (__ldg(keys + mid) < key)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

// (d, j) < (e, k) in lexicographic order
__device__ __forceinline__ bool lex_less(double d, int32_t j, double e, int32_t k) { return d < e || (d == e && j < k); }

__device__ __forceinline__ double dist2(double xi, double yi, double zi, double xj, double yj, double zj) {
  const double dx = __dsub_rn(xj, xi), dy = __dsub_rn(yj, yi), dz = __dsub_rn(zj, zi);
  return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// one Jacobi rotation zeroing a[p][q] of the symmetric 3x3 matrix a; v accumulates the rotations (columns = eigenvectors)
template <int P, int Q>
__device__ __forceinline__ void jacobi_rotate(double (&a)[3][3], double (&v)[3][3]) {
  const double apq = a[P][Q];
  if (apq == 0.0) return;
  const double g = 100.0 * fabs(apq);
  if (fabs(a[P][P]) + g == fabs(a[P][P]) && fabs(a[Q][Q]) + g == fabs(a[Q][Q])) {  // negligible: drop it
    a[P][Q] = a[Q][P] = 0.0;
    return;
  }
  const double theta = (a[Q][Q] - a[P][P]) / (2.0 * apq);
  double t = 1.0 / (fabs(theta) + sqrt(theta * theta + 1.0));
  if (fabs(theta) > 1e150) t = 0.5 / fabs(theta);  // theta^2 would overflow
  if (theta < 0.0) t = -t;
  const double c = 1.0 / sqrt(t * t + 1.0), s = t * c, tau = s / (1.0 + c);
  a[P][P] -= t * apq;
  a[Q][Q] += t * apq;
  a[P][Q] = a[Q][P] = 0.0;
  constexpr int R = 3 - P - Q;
  const double arp = a[R][P], arq = a[R][Q];
  a[R][P] = a[P][R] = arp - s * (arq + arp * tau);
  a[R][Q] = a[Q][R] = arq + s * (arp - arq * tau);
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const double vp = v[r][P], vq = v[r][Q];
    v[r][P] = vp - s * (vq + vp * tau);
    v[r][Q] = vq + s * (vp - vq * tau);
  }
}

struct Eig {
  double val, x, y, z;
};
__device__ __forceinline__ void sort2(Eig& a, Eig& b) {
  if (b.val < a.val) {
    const Eig t = a;
    a = b;
    b = t;
  }
}

struct NormalsArgs {
  const uint64_t* keys;  // [n] sorted Morton keys (finite points first)
  const uint32_t* perm;  // [n] sorted position -> point index
  const float* sx;       // [3 n] sorted SoA coordinates
  int32_t n, nf, k, keff;
  int32_t p0, p1;        // the queries: sorted positions [p0, p1)
  Quant q;
  double vp[3];
  int has_vp;
  float* nrm;     // [3 n] AoS, by point index
  int64_t* nbr;   // [n k] or null
  int32_t* lists; // [n k]: the int32 lists of the kLists32 instantiations
  unsigned long long* pairs;
};

// kPca = false: the lists alone, no covariance and no normal.  kLists32: the lists go to A.lists as int32 (always
// written) instead of A.nbr.  <true, false> is rsc_estimate_normals' kernel.
template <bool kPca, bool kLists32>
__global__ void __launch_bounds__(256, 2) knn_normals_kernel(const NormalsArgs A) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
  const float* sy = A.sx + A.n;
  const float* sz = A.sx + 2 * (int64_t)A.n;
  const int k = A.k, keff = A.keff;
  long long pairs = 0;
  // positions and candidate counters are 64-bit: p + nwarps and base + 32 may pass 2^31 - 1 for n close to it
  for (int64_t p = A.p0 + (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5); p < A.p1; p += nwarps) {
    const uint32_t i = __ldg(A.perm + p);
    if (p >= A.nf) {  // non-finite point: zero normal, empty row
      if (kPca && lane < 3) A.nrm[3 * (int64_t)i + lane] = 0.f;
      if (kLists32) {
        if (lane < k) A.lists[(int64_t)i * k + lane] = -1;
      } else if (A.nbr && lane < k) {
        A.nbr[(int64_t)i * k + lane] = -1;
      }
      continue;
    }
    const uint64_t key = __ldg(A.keys + p);
    const double xi = A.sx[p], yi = sy[p], zi = sz[p];
    // start level: the deepest one whose cell around the query holds >= k_eff points (lane l-1 looks at level l)
    int level;
    {
      bool enough = false;
      if (lane <= kKeyBits) {
        const int shift = 3 * (kKeyBits - lane);
        const uint64_t lo_key = (key >> shift) << shift;
        const int32_t a = lower_bound_u64(A.keys, 0, (int32_t)p, lo_key);
        const int32_t b = lower_bound_u64(A.keys, (int32_t)p + 1, A.nf, lo_key + ((uint64_t)1 << shift));
        enough = b - a >= keff;
      }
      level = 32 - __clz(__ballot_sync(0xffffffffu, enough));  // lane 0 (the whole box) always holds enough
    }
    uint32_t qc[3] = {0u, 0u, 0u};  // the query's finest cell
    for (int b = kKeyBits - 1; b >= 0; --b) {
      qc[0] |= (uint32_t)((key >> (3 * b + 2)) & 1u) << b;
      qc[1] |= (uint32_t)((key >> (3 * b + 1)) & 1u) << b;
      qc[2] |= (uint32_t)((key >> (3 * b)) & 1u) << b;
    }
    // lane t < k holds the t-th best (d2, j) so far and the sorted position of j; empty: (inf, INT_MAX)
    double ld = INFINITY;
    int32_t lj = INT_MAX, lp = 0;
    double bound_d = INFINITY;  // (d2, j) of the k-th of the level below: every member of N(i) is <= it
    int32_t bound_j = INT_MAX;
    for (;;) {
      const int bits = level - 1;
      const int down = kKeyBits - bits;
      const uint32_t ncell = 1u << bits;
      // lane c < 27: the c-th cell of the 3x3x3 block (lane 0 the query's own) as a range of sorted positions
      int32_t cb = 0, ce = 0;
      if (lane < 27) {
        const int o = lane == 0 ? 13 : (lane <= 13 ? lane - 1 : lane);
        const int d[3] = {o / 9 - 1, (o / 3) % 3 - 1, o % 3 - 1};
        uint32_t c[3];
        bool in = true;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          const int64_t v = (int64_t)(qc[a] >> down) + d[a];
          in = in && v >= 0 && v < (int64_t)ncell;
          c[a] = (uint32_t)v;
        }
        if (in) {
          const int shift = 3 * down;
          const uint64_t lo_key = interleave(c[0], c[1], c[2], bits) << shift;
          cb = lower_bound_u64(A.keys, 0, A.nf, lo_key);
          ce = lower_bound_u64(A.keys, cb, A.nf, lo_key + ((uint64_t)1 << shift));
        }
      }
      const int32_t sz_c = ce - cb;
      int32_t incl = sz_c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      const int32_t excl = incl - sz_c;
      const int32_t total = __shfl_sync(0xffffffffu, incl, 31);
      ld = INFINITY, lj = INT_MAX, lp = 0;
      for (int64_t base = 0; base < total; base += 32) {
        const int64_t v = base + lane;
        int lo = 0, hi = 26;  // the cell of candidate v: the first c with incl[c] > v
#pragma unroll
        for (int s = 0; s < 5; ++s) {
          const int mid = (lo + hi) >> 1;
          const int32_t im = __shfl_sync(0xffffffffu, incl, mid);
          if (lo < hi) {
            if (im <= v)
              lo = mid + 1;
            else
              hi = mid;
          }
        }
        const int32_t pc = __shfl_sync(0xffffffffu, cb, lo) + (int32_t)(v - __shfl_sync(0xffffffffu, excl, lo));
        const double kd = __shfl_sync(0xffffffffu, ld, k - 1);
        const int32_t kj = __shfl_sync(0xffffffffu, lj, k - 1);
        double cd = INFINITY;
        int32_t cj = INT_MAX;
        bool keep = false;
        if (v < total) {
          cj = (int32_t)__ldg(A.perm + pc);
          cd = dist2(xi, yi, zi, A.sx[pc], sy[pc], sz[pc]);
          keep = lex_less(cd, cj, kd, kj) && !lex_less(bound_d, bound_j, cd, cj);
        }
        pairs += min((int64_t)32, total - base);
        unsigned m = __ballot_sync(0xffffffffu, keep);
        while (m) {  // insert the survivors one by one into the sorted list
          const int src = __ffs(m) - 1;
          m &= m - 1;
          const double nd = __shfl_sync(0xffffffffu, cd, src);
          const int32_t nj = __shfl_sync(0xffffffffu, cj, src);
          const int32_t np = __shfl_sync(0xffffffffu, pc, src);
          const int pos = __popc(__ballot_sync(0xffffffffu, lex_less(ld, lj, nd, nj)));
          const double ud = __shfl_up_sync(0xffffffffu, ld, 1);
          const int32_t uj = __shfl_up_sync(0xffffffffu, lj, 1);
          const int32_t up = __shfl_up_sync(0xffffffffu, lp, 1);
          if (pos < k) {
            if (lane > pos && lane < k) ld = ud, lj = uj, lp = up;
            if (lane == pos) ld = nd, lj = nj, lp = np;
          }
        }
      }
      const double kd = __shfl_sync(0xffffffffu, ld, k - 1);
      // r_safe: every finite point outside the block is farther than this from the query (DESIGN.md section 8)
      double r = INFINITY;
      const double xq[3] = {xi, yi, zi};
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        const int64_t qa = qc[a] >> down;
        const double h = A.q.w[a] / (double)ncell;  // exact: a power of two
        const double e = 0x1p-48 * (fabs(A.q.lo[a]) + A.q.w[a] + fabs(xq[a]));
        if (qa >= 2) r = fmin(r, (xq[a] - (A.q.lo[a] + (double)(qa - 1) * h)) - e);
        if (qa + 2 < (int64_t)ncell) r = fmin(r, ((A.q.lo[a] + (double)(qa + 2) * h) - xq[a]) - e);
      }
      if (r == INFINITY || (r > 0.0 && kd < (r * r) * (1.0 - 0x1p-40))) break;
      bound_d = kd;
      bound_j = __shfl_sync(0xffffffffu, lj, k - 1);
      --level;
    }
    if (kLists32) {
      if (lane < k) A.lists[(int64_t)i * k + lane] = lane < keff ? lj : -1;
      if (!kPca) continue;
    } else if (A.nbr && lane < k) {
      A.nbr[(int64_t)i * k + lane] = lane < keff ? (int64_t)lj : -1;
    }
    // covariance of N(i), summed in list order
    const double px = lane < keff ? (double)A.sx[lp] : 0.0, py = lane < keff ? (double)sy[lp] : 0.0,
                 pz = lane < keff ? (double)sz[lp] : 0.0;
    double mx = 0.0, my = 0.0, mz = 0.0;
    for (int t = 0; t < keff; ++t) {
      mx += __shfl_sync(0xffffffffu, px, t);
      my += __shfl_sync(0xffffffffu, py, t);
      mz += __shfl_sync(0xffffffffu, pz, t);
    }
    mx /= keff, my /= keff, mz /= keff;
    double a[3][3] = {{0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}};
    for (int t = 0; t < keff; ++t) {
      const double dx = __shfl_sync(0xffffffffu, px, t) - mx, dy = __shfl_sync(0xffffffffu, py, t) - my,
                   dz = __shfl_sync(0xffffffffu, pz, t) - mz;
      a[0][0] += dx * dx, a[0][1] += dx * dy, a[0][2] += dx * dz;
      a[1][1] += dy * dy, a[1][2] += dy * dz, a[2][2] += dz * dz;
    }
    a[0][0] /= keff, a[0][1] /= keff, a[0][2] /= keff, a[1][1] /= keff, a[1][2] /= keff, a[2][2] /= keff;
    a[1][0] = a[0][1], a[2][0] = a[0][2], a[2][1] = a[1][2];
    double v[3][3] = {{1.0, 0.0, 0.0}, {0.0, 1.0, 0.0}, {0.0, 0.0, 1.0}};
    for (int s = 0; s < kJacobiSweeps && (a[0][1] != 0.0 || a[0][2] != 0.0 || a[1][2] != 0.0); ++s) {
      jacobi_rotate<0, 1>(a, v);
      jacobi_rotate<0, 2>(a, v);
      jacobi_rotate<1, 2>(a, v);
    }
    // eigenpairs in ascending order (a stable sorting network: ties keep the lower column first)
    Eig e[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) e[c] = Eig{a[c][c], v[0][c], v[1][c], v[2][c]};
    sort2(e[0], e[1]);
    sort2(e[1], e[2]);
    sort2(e[0], e[1]);
    double n[3] = {0.0, 0.0, 0.0};
    if (keff >= 3 && e[1].val > kTau * e[2].val) {
      n[0] = e[0].x, n[1] = e[0].y, n[2] = e[0].z;
      const double len = sqrt((n[0] * n[0] + n[1] * n[1]) + n[2] * n[2]);
      n[0] /= len, n[1] /= len, n[2] /= len;
      bool flip;
      if (A.has_vp) {
        flip = ((n[0] * (A.vp[0] - xi) + n[1] * (A.vp[1] - yi)) + n[2] * (A.vp[2] - zi)) < 0.0;
      } else {
        double big = n[0];  // the component of largest magnitude, the first on ties
        if (fabs(n[1]) > fabs(big)) big = n[1];
        if (fabs(n[2]) > fabs(big)) big = n[2];
        flip = big < 0.0;
      }
      if (flip) n[0] = -n[0], n[1] = -n[1], n[2] = -n[2];
    }
    if (lane < 3) A.nrm[3 * (int64_t)i + lane] = (float)(lane == 0 ? n[0] : (lane == 1 ? n[1] : n[2]));
  }
  if (lane == 0 && A.pairs && pairs) atomicAdd(A.pairs, (unsigned long long)pairs);
}

// sharded forms: this rank's rows into the zero-filled all-reduce records of W int32 words by point index -- the
// coordinate bits, the normal bits when given, and a coverage word: 3 on the range's first row, 1 on the others
__global__ void __launch_bounds__(256) shard_pack_kernel(const float* __restrict__ xyz, const float* __restrict__ nrm, int64_t n,
                                                         int64_t off, int W, int32_t* __restrict__ rec) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int32_t* r = rec + (off + i) * W;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    r[a] = __float_as_int(xyz[3 * i + a]);
    if (nrm) r[3 + a] = __float_as_int(nrm[3 * i + a]);
  }
  r[W - 1] = i == 0 ? 3 : 1;
}

// the summed records back to AoS; cnt[0] rows covered by no range or by several, cnt[1] ranges starting before off,
// cnt[2] ranges (non-empty ones)
__global__ void __launch_bounds__(256) shard_unpack_kernel(const int32_t* __restrict__ rec, int64_t n, int64_t off, int W,
                                                           float* __restrict__ aos, float* __restrict__ nrm,
                                                           unsigned long long* __restrict__ cnt) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool bad = false, start = false;
  if (i < n) {
    const int32_t* r = rec + i * W;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      aos[3 * i + a] = __int_as_float(r[a]);
      if (nrm) nrm[3 * i + a] = __int_as_float(r[3 + a]);
    }
    const int32_t c = r[W - 1];
    bad = c != 1 && c != 3;
    start = c == 3;
  }
  const int nb = __syncthreads_count(bad), ns = __syncthreads_count(start), nbefore = __syncthreads_count(start && i < off);
  if (threadIdx.x == 0) {
    if (nb) atomicAdd(cnt, (unsigned long long)nb);
    if (nbefore) atomicAdd(cnt + 1, (unsigned long long)nbefore);
    if (ns) atomicAdd(cnt + 2, (unsigned long long)ns);
  }
}

}  // namespace
}  // namespace rsc

using namespace rsc;

#define NRM_CUDA(expr) RSC_CUDA(ctx, (expr))

int32_t rsc::knn_prepare(rsc_ctx* ctx, const float* xyz, int64_t n, KnnSearch& S) {
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if (int32_t rc = knn_reserve(ctx, n, S)) return rc;
  NRM_CUDA(cudaMemcpyAsync(S.aos, xyz, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
  return knn_sort(ctx, S);
}

int32_t rsc::knn_reserve(rsc_ctx* ctx, int64_t n, KnnSearch& S) {
  Allocs& al = S.al;
  S.n = n;
  NRM_CUDA(al.get((void**)&S.aos, (size_t)n * 12));
  NRM_CUDA(al.get((void**)&S.soa, (size_t)n * 12));
  for (int b = 0; b < 2; ++b) {
    NRM_CUDA(al.get((void**)&S.keys_buf[b], (size_t)n * 8));
    NRM_CUDA(al.get((void**)&S.idx_buf[b], (size_t)n * 4));
  }
  NRM_CUDA(al.get((void**)&S.mm, 6 * 4 + 2 * 8));
  S.cnt = reinterpret_cast<unsigned long long*>(S.mm + 6);
  cub::DoubleBuffer<uint64_t> kbuf(S.keys_buf[0], S.keys_buf[1]);
  cub::DoubleBuffer<uint32_t> ibuf(S.idx_buf[0], S.idx_buf[1]);
  S.tmp_bytes = 0;
  NRM_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, S.tmp_bytes, kbuf, ibuf, (int)n, 0, 64, ctx->stream));
  NRM_CUDA(al.get(&S.tmp, S.tmp_bytes));
  return RSC_OK;
}

int32_t rsc::knn_sort(rsc_ctx* ctx, KnnSearch& S) {
  cudaStream_t st = ctx->stream;
  const int64_t n = S.n;
  uint64_t* const* d_keys = S.keys_buf;
  uint32_t* const* d_idx = S.idx_buf;
  uint32_t* d_mm = S.mm;
  cub::DoubleBuffer<uint64_t> kbuf(d_keys[0], d_keys[1]);
  cub::DoubleBuffer<uint32_t> ibuf(d_idx[0], d_idx[1]);
  size_t tmp_bytes = S.tmp_bytes;
  void* d_tmp = S.tmp;

  const unsigned blocks = (unsigned)((n + 255) / 256);
  const uint32_t init[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
  NRM_CUDA(cudaMemcpyAsync(d_mm, init, sizeof(init), cudaMemcpyHostToDevice, st));
  NRM_CUDA(cudaMemsetAsync(S.cnt, 0, 2 * 8, st));
  aos_to_soa_kernel<<<blocks, 256, 0, st>>>(S.aos, n, S.soa);
  NRM_CUDA(cudaGetLastError());
  bbox_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(S.soa, n, n, d_mm, true);
  NRM_CUDA(cudaGetLastError());
  uint32_t got[6];
  NRM_CUDA(cudaMemcpyAsync(got, d_mm, sizeof(got), cudaMemcpyDeviceToHost, st));
  NRM_CUDA(cudaStreamSynchronize(st));
  Quant& q = S.q;
  q.D = kKeyBits;
  q.scale = (double)((uint64_t)1 << kKeyBits);
  q.qmax = (1u << kKeyBits) - 1u;
  for (int a = 0; a < 3; ++a) {
    const double lo = (double)ord2f(got[a]), hi = (double)ord2f(got[3 + a]);
    q.lo[a] = lo;
    q.w[a] = hi - lo;
    if (!(q.w[a] > 0.0)) q.w[a] = 1.0;  // one value on this axis, or no finite point at all
    if (!std::isfinite(q.lo[a])) q.lo[a] = 0.0;
  }
  keys_kernel<<<blocks, 256, 0, st>>>(S.soa, n, q, d_keys[0], d_idx[0], S.cnt);
  NRM_CUDA(cudaGetLastError());
  NRM_CUDA(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, kbuf, ibuf, (int)n, 0, 64, st));
  gather_sorted_kernel<<<blocks, 256, 0, st>>>(S.aos, ibuf.Current(), n, S.soa);
  NRM_CUDA(cudaGetLastError());
  unsigned long long nf = 0;
  NRM_CUDA(cudaMemcpyAsync(&nf, S.cnt, 8, cudaMemcpyDeviceToHost, st));
  NRM_CUDA(cudaStreamSynchronize(st));
  S.nf = (int64_t)nf;
  S.keys = kbuf.Current();
  S.perm = ibuf.Current();
  return RSC_OK;
}

int32_t rsc::knn_run(rsc_ctx* ctx, const KnnSearch& S, int32_t k, const double* viewpoint, float* d_nrm, int64_t* d_nbr,
                     int32_t* d_lists, int64_t p_begin, int64_t p_end) {
  if (p_end <= p_begin) return RSC_OK;
  NormalsArgs A;
  A.keys = S.keys;
  A.perm = S.perm;
  A.sx = S.soa;
  A.n = (int32_t)S.n, A.nf = (int32_t)S.nf, A.k = k, A.keff = (int32_t)std::min<int64_t>(k, S.nf);
  A.p0 = (int32_t)p_begin, A.p1 = (int32_t)p_end;
  A.q = S.q;
  A.has_vp = viewpoint != nullptr;
  for (int a = 0; a < 3; ++a) A.vp[a] = viewpoint ? viewpoint[a] : 0.0;
  A.nrm = d_nrm, A.nbr = d_nbr, A.lists = d_lists, A.pairs = S.cnt + 1;
  const int64_t want = (p_end - p_begin + kWarpsPerBlock - 1) / kWarpsPerBlock;
  const unsigned grid = (unsigned)std::min<int64_t>(want, (int64_t)ctx->sm_count * 8);
  cudaStream_t st = ctx->stream;
  if (!d_lists)
    knn_normals_kernel<true, false><<<grid, 256, 0, st>>>(A);
  else if (d_nrm)
    knn_normals_kernel<true, true><<<grid, 256, 0, st>>>(A);
  else
    knn_normals_kernel<false, true><<<grid, 256, 0, st>>>(A);
  NRM_CUDA(cudaGetLastError());
  return RSC_OK;
}

// The check's record: int32 words summed over the ranks.  Every multi-bit value travels as 16-bit pieces, so that a
// sum over up to 2^15 ranks cannot overflow; a rank compares each sum with R times its own value, R = the sum of the
// ones.
namespace {
constexpr int kRecOne = 0, kRecNonEmpty = 1, kRecN = 2, kRecNGlobal = 6, kRecK = 10, kRecHasVp = 12, kRecOpt = 13,
              kRecVp = 14, kRecWords = 26;

void put16(int32_t* rec, int at, uint64_t v, int pieces) {
  for (int p = 0; p < pieces; ++p) rec[at + p] = (int32_t)((v >> (16 * p)) & 0xffffu);
}
}  // namespace

int32_t rsc::shard_check(rsc_ctx* ctx, Allocs& al, const char* fn, const char* own, int64_t n, int64_t n_global, int32_t k,
                         const double* viewpoint, bool opt, const std::function<bool(bool)>& reserve, bool* opt_on) {
  if (!ctx->allreduce)
    return fail(ctx, RSC_E_STATE, (std::string(fn) + ": the context has no communicator (rsc_ctx_comm_init / rsc_ctx_set_allreduce)").c_str());
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  int32_t rec[kRecWords] = {}, sum[kRecWords];
  rec[kRecOne] = 1;
  rec[kRecNonEmpty] = n > 0;
  put16(rec, kRecN, (uint64_t)n, 4);
  put16(rec, kRecNGlobal, (uint64_t)n_global, 4);
  put16(rec, kRecK, (uint32_t)k, 2);
  rec[kRecHasVp] = viewpoint != nullptr;
  rec[kRecOpt] = n > 0 && opt;
  for (int a = 0; a < 3; ++a) {
    uint64_t bits = 0;
    if (viewpoint) memcpy(&bits, viewpoint + a, 8);
    put16(rec, kRecVp + 4 * a, bits, 4);
  }
  int32_t* d_rec = nullptr;
  NRM_CUDA(al.get((void**)&d_rec, sizeof(rec)));
  NRM_CUDA(cudaMemcpyAsync(d_rec, rec, sizeof(rec), cudaMemcpyHostToDevice, st));
  if (int32_t rc = rsc_ctx_allreduce(ctx, d_rec, kRecWords, st)) return rc;
  NRM_CUDA(cudaMemcpyAsync(sum, d_rec, sizeof(sum), cudaMemcpyDeviceToHost, st));
  NRM_CUDA(cudaStreamSynchronize(st));
  const int64_t R = sum[kRecOne];
  bool agree = true;
  for (int w = kRecNGlobal; w < kRecWords; ++w)
    if (w != kRecOpt) agree = agree && (int64_t)sum[w] == R * rec[w];
  uint64_t sum_n = 0;
  for (int p = 0; p < 4; ++p) sum_n += (uint64_t)(uint32_t)sum[kRecN + p] << (16 * p);
  agree = agree && sum_n == (uint64_t)n_global;
  agree = agree && (sum[kRecOpt] == 0 || sum[kRecOpt] == sum[kRecNonEmpty]);
  // every buffer the collective steps need is allocated here, so that a rank short of memory fails with its peers
  if (!own && agree && !reserve(sum[kRecOpt] > 0)) {
    cudaGetLastError();  // (an allocation failure is not sticky: clear it)
    own = "cannot allocate the device buffers of n_global points on this rank";
  }
  int32_t bad = own || !agree ? 1 : 0;
  NRM_CUDA(cudaMemcpyAsync(d_rec, &bad, 4, cudaMemcpyHostToDevice, st));
  if (int32_t rc = rsc_ctx_allreduce(ctx, d_rec, 1, st)) return rc;
  NRM_CUDA(cudaMemcpyAsync(&bad, d_rec, 4, cudaMemcpyDeviceToHost, st));
  NRM_CUDA(cudaStreamSynchronize(st));
  if (bad > 0) {
    const std::string msg = std::string(fn) + ": " +
                            (own ? own : "the ranks' arguments disagree (k, n_global, viewpoint, optional outputs, or the sum of n)");
    return fail(ctx, RSC_E_ARG, msg.c_str());
  }
  *opt_on = sum[kRecOpt] > 0;
  return RSC_OK;
}

bool rsc::ShardBufs::reserve(rsc_ctx* ctx, int64_t n_global, bool with_nrm, int64_t row_words, KnnSearch& S) {
  W = with_nrm ? 7 : 4;
  words = row_words;
  return knn_reserve(ctx, n_global, S) == RSC_OK && S.al.get((void**)&rec, (size_t)n_global * W * 4) == cudaSuccess &&
         S.al.get((void**)&cnt, 3 * 8) == cudaSuccess && S.al.get((void**)&rows, (size_t)words * 4) == cudaSuccess &&
         (!with_nrm || S.al.get((void**)&nrm, (size_t)n_global * 12) == cudaSuccess);
}

int32_t rsc::shard_gather(rsc_ctx* ctx, const char* fn, const float* xyz, const float* nrm, int64_t off, int64_t n,
                          int64_t n_global, KnnSearch& S, const ShardBufs& B, ShardSlice& sl, PhaseClock& clk) {
  cudaStream_t st = ctx->stream;
  const int W = B.W;
  int32_t* d_rec = B.rec;
  unsigned long long* d_cnt = B.cnt;
  float* d_nrm_all = B.nrm;
  NRM_CUDA(cudaMemsetAsync(d_rec, 0, (size_t)n_global * W * 4, st));
  NRM_CUDA(cudaMemsetAsync(d_cnt, 0, 3 * 8, st));
  if (n > 0) {  // this rank's rows go through S.aos and d_nrm_all, which the unpack overwrites
    NRM_CUDA(cudaMemcpyAsync(S.aos, xyz, (size_t)n * 12, cudaMemcpyHostToDevice, st));
    if (d_nrm_all) NRM_CUDA(cudaMemcpyAsync(d_nrm_all, nrm, (size_t)n * 12, cudaMemcpyHostToDevice, st));
    shard_pack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(S.aos, d_nrm_all, n, off, W, d_rec);
    NRM_CUDA(cudaGetLastError());
  }
  if (int32_t rc = rsc_ctx_allreduce(ctx, d_rec, n_global * W, st)) return rc;
  shard_unpack_kernel<<<(unsigned)((n_global + 255) / 256), 256, 0, st>>>(d_rec, n_global, off, W, S.aos, d_nrm_all, d_cnt);
  NRM_CUDA(cudaGetLastError());
  unsigned long long got[3];
  NRM_CUDA(cudaMemcpyAsync(got, d_cnt, sizeof(got), cudaMemcpyDeviceToHost, st));
  NRM_CUDA(cudaStreamSynchronize(st));
  clk.mark(ctx, 0);
  if (got[0])  // the records are identical on every rank: all of them return here
    return fail(ctx, RSC_E_ARG, (std::string(fn) + ": the ranks' ranges overlap or leave a gap in [0, n_global)").c_str());
  if (int32_t rc = knn_sort(ctx, S)) return rc;
  sl = ShardSlice{};
  if (n > 0) {
    const int64_t r = (int64_t)got[1], R = (int64_t)got[2], nf = S.nf;
    sl.p_begin = nf * r / R;
    sl.p_end = r == R - 1 ? n_global : nf * (r + 1) / R;
  }
  return RSC_OK;
}

rsc::PhaseClock::PhaseClock() {
  const char* e = getenv("RSC_NORMALS_TRACE");
  on = e && atoi(e) != 0;
  if (on) t = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

void rsc::PhaseClock::mark(rsc_ctx* ctx, int phase) {
  if (!on) return;
  cudaStreamSynchronize(ctx->stream);
  const double now = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
  ms[phase] += 1e3 * (now - t);
  t = now;
}

void rsc::PhaseClock::print(const char* fn, rsc_ctx* ctx) const {
  if (on)
    fprintf(stderr, "[%s] gather %.3f prepare %.3f search %.3f exchange %.3f forest %.3f ms | all-reduces %lld (%lld B)\n", fn,
            ms[0], ms[1], ms[2], ms[3], ms[4], (long long)ctx->allreduce_calls, (long long)ctx->allreduce_bytes);
}

extern "C" int32_t rsc_estimate_normals(rsc_ctx* ctx, const float* xyz, int64_t n, int32_t k, const double* viewpoint, float* nrm,
                                        int64_t* nbr, int64_t* pairs) {
  if (!ctx) return RSC_E_ARG;
  if (!xyz || !nrm) return fail(ctx, RSC_E_ARG, "estimate_normals: xyz and nrm must not be NULL");
  if (k < 3 || k > 32) return fail(ctx, RSC_E_ARG, "estimate_normals: k must be in [3, 32]");
  if (n < 1 || n >= ((int64_t)1 << 31)) return fail(ctx, RSC_E_ARG, "estimate_normals: n must be in [1, 2^31)");
  KnnSearch S;
  float* d_nrm = nullptr;
  int64_t* d_nbr = nullptr;
  if (int32_t rc = knn_prepare(ctx, xyz, n, S)) return rc;
  NRM_CUDA(S.al.get((void**)&d_nrm, (size_t)n * 12));
  if (nbr) NRM_CUDA(S.al.get((void**)&d_nbr, (size_t)n * k * 8));
  if (int32_t rc = knn_run(ctx, S, k, viewpoint, d_nrm, d_nbr, nullptr, 0, n)) return rc;
  cudaStream_t st = ctx->stream;
  if (int32_t rc = staged_d2h(ctx, nrm, d_nrm, (size_t)n * 12, st)) return rc;
  if (nbr)
    if (int32_t rc = staged_d2h(ctx, nbr, d_nbr, (size_t)n * k * 8, st)) return rc;
  unsigned long long np = 0;
  NRM_CUDA(cudaMemcpyAsync(&np, S.cnt + 1, 8, cudaMemcpyDeviceToHost, st));
  NRM_CUDA(cudaStreamSynchronize(st));
  if (pairs) *pairs = (int64_t)np;
  return RSC_OK;
}

const char* rsc::shard_own_problem(int64_t n, int64_t off, int64_t n_global, int32_t k, const void* xyz, const void* out) {
  if (k < 3 || k > 32) return "k must be in [3, 32]";
  if (n_global < 1 || n_global >= ((int64_t)1 << 31)) return "n_global must be in [1, 2^31)";
  if (n < 0 || off < 0 || off > n_global - n) return "[global_offset, global_offset + n) must lie in [0, n_global)";
  if (n > 0 && (!xyz || !out)) return "the coordinates and the output normals must not be NULL when n > 0";
  return nullptr;
}

extern "C" int32_t rsc_estimate_normals_shard(rsc_ctx* ctx, const float* xyz, int64_t n, int64_t global_offset, int64_t n_global,
                                              int32_t k, const double* viewpoint, float* nrm, int64_t* nbr, int64_t* pairs) {
  constexpr const char* fn = "estimate_normals_shard";
  if (!ctx) return RSC_E_ARG;
  KnnSearch S;
  ShardBufs B;
  PhaseClock clk;
  bool with_nbr = false;
  // the rows, zero-filled and completed by one all-reduce: [n_global k] int64 lists (when asked for), [3 n_global] normals
  auto reserve = [&](bool lists) { return B.reserve(ctx, n_global, false, n_global * (3 + (lists ? 2 * (int64_t)k : 0)), S); };
  if (int32_t rc = shard_check(ctx, S.al, fn, shard_own_problem(n, global_offset, n_global, k, xyz, nrm), n, n_global, k,
                               viewpoint, nbr != nullptr, reserve, &with_nbr))
    return rc;
  ShardSlice sl;
  if (int32_t rc = shard_gather(ctx, fn, xyz, nullptr, global_offset, n, n_global, S, B, sl, clk)) return rc;
  clk.mark(ctx, 1);
  const int64_t words = B.words;
  int32_t* d_rows = B.rows;
  int64_t* d_nbr = with_nbr ? reinterpret_cast<int64_t*>(d_rows) : nullptr;
  float* d_nrm = reinterpret_cast<float*>(d_rows + (with_nbr ? 2 * (int64_t)k * n_global : 0));
  cudaStream_t st = ctx->stream;
  NRM_CUDA(cudaMemsetAsync(d_rows, 0, (size_t)words * 4, st));
  if (int32_t rc = knn_run(ctx, S, k, viewpoint, d_nrm, d_nbr, nullptr, sl.p_begin, sl.p_end)) return rc;
  clk.mark(ctx, 2);
  if (int32_t rc = rsc_ctx_allreduce(ctx, d_rows, words, st)) return rc;
  if (n > 0) {
    if (int32_t rc = staged_d2h(ctx, nrm, d_nrm + 3 * global_offset, (size_t)n * 12, st)) return rc;
    if (nbr)
      if (int32_t rc = staged_d2h(ctx, nbr, d_nbr + global_offset * k, (size_t)n * k * 8, st)) return rc;
  }
  unsigned long long np = 0;
  NRM_CUDA(cudaMemcpyAsync(&np, S.cnt + 1, 8, cudaMemcpyDeviceToHost, st));
  NRM_CUDA(cudaStreamSynchronize(st));
  clk.mark(ctx, 3);
  clk.print(fn, ctx);
  if (pairs) *pairs = (int64_t)np;
  return RSC_OK;
}
#undef NRM_CUDA
