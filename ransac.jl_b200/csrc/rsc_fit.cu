// rsc_fit.cu -- K1: batched minimal-set sampling and shape fitting, one thread per minimal set.
//
// Replaces samplepointcloud4! (fitting.jl:383-430), forcefitshapes! (fitting.jl:165-173) and the four
// fit methods (plane.jl:33-57, sphere.jl:29-114, cylinder.jl:34-168, cone.jl:39-128).
//
// The fits run in FP64 (a few kFLOP per set; the tolerance on fitted parameters is 1e-5 relative and
// the cone apex solve can be ill conditioned) and this file is compiled with -fmad=false so that the
// accept/reject decisions follow the plain IEEE evaluation of the reference formulas.
// Candidates leave the kernel dense ([set][shape type] + a validity flag) and are compacted in
// (set, shape_types) order -- the reference's candidate order, which breaks score ties (Q16).
//
// Sampler: every minimal set owns a Philox4x32-10 stream (key = seed, counter = (draw/2, set id)).
// Reference semantics on the root cell (Q1): first index by rejection over all points until an
// enabled one is hit, the others uniform over the enabled points (rank -> index by select over the
// enabled bitmask), one re-draw on collision with the first, whole set dropped on any duplicate.
#include <math.h>

#include <vector>

#include "rsc_common.cuh"

namespace rsc {

struct D3 {
  double x, y, z;
};
__device__ __forceinline__ D3 operator-(D3 a, D3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ D3 operator+(D3 a, D3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
__device__ __forceinline__ D3 operator*(double s, D3 a) { return {s * a.x, s * a.y, s * a.z}; }
__device__ __forceinline__ D3 operator-(D3 a) { return {-a.x, -a.y, -a.z}; }
__device__ __forceinline__ double dot(D3 a, D3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ double norm(D3 a) { return sqrt(dot(a, a)); }
__device__ __forceinline__ D3 unit(D3 a) { return (1.0 / norm(a)) * a; }  // StaticArrays: inv(norm)*a
__device__ __forceinline__ D3 cross(D3 a, D3 b) {
  return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}

constexpr int kMaxK = 8;  // points per set the validators look at (minimal set + extra validators)

struct FitParams {
  double eps[RSC_NTYPES], cosa[RSC_NTYPES];
  double cos_par;  // cosd(parallelthrdeg)
  double sphere_par, minconeopang, collin;
  int32_t ntypes, types[RSC_MAX_ORDER];  // the fit order; user types (>= RSC_USER_TYPE0) are fitted by their own kernel
  int32_t k;
};

__device__ inline void store(rsc_cand* o, int type, int outw, D3 a, D3 b, double s) {
  o->type = type;
  o->outwards = outw;
  o->p[0] = a.x, o->p[1] = a.y, o->p[2] = a.z;
  if (type == RSC_SPHERE) {
    o->p[3] = s, o->p[4] = 0, o->p[5] = 0, o->p[6] = 0;
  } else {
    o->p[3] = b.x, o->p[4] = b.y, o->p[5] = b.z, o->p[6] = s;
  }
}

// same-side test shared by the four validators: all dots > thr -> +1, all < -thr -> -1, else 0
__device__ __forceinline__ int side(const double* d, int k, double thr) {
  bool pos = true, neg = true;
#pragma unroll
  for (int i = 0; i < k; ++i) {
    pos = pos && (d[i] > thr);
    neg = neg && (d[i] < -thr);
  }
  return pos ? 1 : (neg ? -1 : 0);
}

template <int KK>
__device__ bool fit_plane(const D3* p, const D3* n, const FitParams& f, rsc_cand* out) {
  constexpr int KA = KK ? KK : kMaxK;
  const int kk = KK ? KK : f.k;
  D3 m = unit(cross(p[1] - p[0], p[2] - p[0]));
  if (norm(m) < f.collin) return false;  // plane.jl:43 (never true: the norm is 1 or NaN, Q3)
  double d[KA];
  _Pragma("unroll") for (int i = 0; i < kk; ++i) d[i] = dot(m, unit(n[i]));
  const int sd = side(d, kk, f.cosa[RSC_PLANE]);
  if (sd == 0) return false;
  if (sd < 0) m = -1.0 * m;
  store(out, RSC_PLANE, 1, p[0], m, 0.0);
  return true;
}

template <int KK>
__device__ bool fit_sphere(const D3* v, const D3* n, const FitParams& f, rsc_cand* out) {
  constexpr int KA = KK ? KK : kMaxK;
  const int kk = KK ? KK : f.k;
  const D3 n1 = unit(n[0]), n2 = unit(n[1]);
  D3 c;
  double R;
  if (fabs(dot(n1, n2)) > f.cos_par) {  // parallel normals: midpoint sphere (sphere.jl:38-42)
    c = 0.5 * (v[0] + v[1]);
    R = norm(c - v[0]);
  } else {
    const D3 g = v[1] - v[0];
    const D3 h = cross(n2, g), kk = cross(n2, n1);
    const double nk = norm(kk), nh = norm(h);
    if (nk < f.sphere_par || nh < f.sphere_par) {  // closest approach of the two normal lines (sphere.jl:52-61)
      const D3 m2 = cross(n2, cross(n1, n2));
      const D3 m1 = cross(n1, cross(n2, n1));
      const D3 c1 = v[0] + (dot(v[1] - v[0], m2) / dot(n[0], m2)) * n[0];
      const D3 c2 = v[1] + (dot(v[0] - v[1], m1) / dot(n[1], m1)) * n[1];
      c = 0.5 * (c1 + c2);
      R = (norm(v[0] - c) + norm(v[0] - c)) / 2;  // Q5: p1 twice
    } else {
      const double t = nh / nk;
      c = dot(h, kk) > 0 ? v[0] + t * n1 : v[0] - t * n1;
      R = norm(c - v[0]);
    }
  }
  double d[KA];
  bool vert = true;
  _Pragma("unroll") for (int i = 0; i < kk; ++i) {
    vert = vert && (fabs(norm(v[i] - c) - R) < f.eps[RSC_SPHERE]);
    d[i] = dot(unit(v[i] - c), unit(n[i]));
  }
  if (!vert) return false;
  const int sd = side(d, kk, f.cosa[RSC_SPHERE]);
  if (sd == 0) return false;
  store(out, RSC_SPHERE, sd > 0, c, D3{0, 0, 0}, R);
  return true;
}

// foot of w on the plane through the origin with normal a (cylinder.jl:46-59)
__device__ __forceinline__ D3 to_plane(D3 a, D3 w) { return w + (dot(-a, w) / dot(a, a)) * a; }

// first two coordinates of p in the frame (xa, ya, za), Cramer's rule (cylinder.jl:61-85)
__device__ inline void frame2d(D3 xa, D3 ya, D3 za, D3 p, double* r) {
  const double xx = xa.x, xy = xa.y, xz = xa.z, yx = ya.x, yy = ya.y, yz = ya.z, zx = za.x, zy = za.y, zz = za.z;
  const double px = p.x, py = p.y, pz = p.z;
  const double den = xz * yy * zx - xy * yz * zx - xz * yx * zy + xx * yz * zy + xy * yx * zz - xx * yy * zz;
  const double n1 = -(pz * yy * zx) + py * yz * zx + pz * yx * zy - px * yz * zy - py * yx * zz + px * yy * zz;
  const double n2 = pz * xy * zx - py * xz * zx - pz * xx * zy + px * xz * zy + py * xx * zz - px * xy * zz;
  r[0] = -(n1 / den);
  r[1] = -(n2 / den);
}

template <int KK>
__device__ bool fit_cylinder(const D3* p, const D3* n, const FitParams& f, rsc_cand* out) {
  constexpr int KA = KK ? KK : kMaxK;
  const int kk = KK ? KK : f.k;
  if (fabs(dot(n[0], n[1])) > f.cos_par) return false;  // raw normals (Q8)
  const D3 a = unit(cross(n[0], n[1]));
  const D3 xa = unit(to_plane(a, p[0]));
  const D3 ya = unit(cross(a, xa));
  double A[2], B[2], C[2], Dd[2];
  frame2d(xa, ya, a, to_plane(a, p[0]), A);
  frame2d(xa, ya, a, to_plane(a, p[0] + n[0]), B);
  frame2d(xa, ya, a, to_plane(a, p[1]), C);
  frame2d(xa, ya, a, to_plane(a, p[1] + n[1]), Dd);
  // intersection of the two projected normal lines (cylinder.jl:87-101)
  const double ab[2] = {A[0] - B[0], A[1] - B[1]}, cd[2] = {C[0] - Dd[0], C[1] - Dd[1]};
  const double d1 = A[0] * B[1] - A[1] * B[0];
  const double d2 = C[0] * Dd[1] - C[1] * Dd[0];
  const double d3 = ab[0] * cd[1] - ab[1] * cd[0];
  const double i0 = (d1 * cd[0] - d2 * ab[0]) / d3, i1 = (d1 * cd[1] - d2 * ab[1]) / d3;
  const D3 c = i0 * xa + i1 * ya;
  double rr[2];
  for (int i = 0; i < 2; ++i) {
    const D3 q = p[i] - c;
    rr[i] = norm(q - dot(a, q) * a);
  }
  const double R = (rr[0] + rr[1]) / 2;
  double d[KA];
  bool vert = true;
  _Pragma("unroll") for (int i = 0; i < kk; ++i) {
    const D3 w = (p[i] - dot(a, p[i] - c) * a) - c;
    vert = vert && (fabs(norm(w) - R) < f.eps[RSC_CYLINDER]);
    d[i] = dot(unit(w), n[i]);
  }
  if (!vert) return false;
  const int sd = side(d, kk, f.cosa[RSC_CYLINDER]);
  if (sd == 0) return false;
  store(out, RSC_CYLINDER, sd > 0, a, c, R);
  return true;
}

// singular values of a 3 x c matrix (c = 3 or 4): one-sided Jacobi on the rows
__device__ inline void singular_values3(const double* A, int c, double* s) {
  double B[3][4];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 4; ++j) B[i][j] = j < c ? A[i * c + j] : 0.0;
  for (int sweep = 0; sweep < 60; ++sweep) {
    double off = 0.0;
    for (int i = 0; i < 2; ++i)
      for (int j = i + 1; j < 3; ++j) {
        double aii = 0, ajj = 0, aij = 0;
        for (int t = 0; t < 4; ++t) aii += B[i][t] * B[i][t], ajj += B[j][t] * B[j][t], aij += B[i][t] * B[j][t];
        if (aij == 0.0) continue;
        off = fmax(off, fabs(aij) / sqrt(aii * ajj + 1e-300));
        const double zeta = (ajj - aii) / (2.0 * aij);
        const double tt = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
        const double cs = 1.0 / sqrt(1.0 + tt * tt), sn = cs * tt;
        for (int t = 0; t < 4; ++t) {
          const double bi = B[i][t], bj = B[j][t];
          B[i][t] = cs * bi - sn * bj;
          B[j][t] = sn * bi + cs * bj;
        }
      }
    if (off <= 2.220446049250313e-16) break;  // every pair orthogonal to working precision (de Rijk's criterion)
  }
  for (int i = 0; i < 3; ++i) {
    double q = 0;
    for (int t = 0; t < 4; ++t) q += B[i][t] * B[i][t];
    s[i] = sqrt(q);
  }
}

// LinearAlgebra.rank(A) == 3 for a 3 x c matrix: all singular values > min(size)*eps*smax
__device__ inline bool full_rank3(const double* A, int c) {
  for (int i = 0; i < 3 * c; ++i)
    if (!isfinite(A[i])) return false;
  double s[3];
  singular_values3(A, c, s);
  const double tol = 3 * 2.220446049250313e-16 * fmax(s[0], fmax(s[1], s[2]));
  return s[0] > tol && s[1] > tol && s[2] > tol;
}

// x = A \ b for a 3 x 3 system: Gaussian elimination with partial pivoting (first maximum wins, one row swap per
// column -- the same pivot sequence and operation order as oracle.c::solve3), written on scalars with selects so
// that the rows stay in registers (indexing rows by a run-time pivot put the matrix in local memory)
__device__ inline bool solve3(const double* A, const double* b, double* x) {
  double r0[4] = {A[0], A[1], A[2], b[0]}, r1[4] = {A[3], A[4], A[5], b[1]}, r2[4] = {A[6], A[7], A[8], b[2]};
  auto swap_rows = [](double* u, double* v, bool doit) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const double a = u[j], c = v[j];
      u[j] = doit ? c : a;
      v[j] = doit ? a : c;
    }
  };
  {  // column 0: pivot = first row with the largest |entry|
    const bool p1 = fabs(r1[0]) > fabs(r0[0]);
    const bool p2 = fabs(r2[0]) > fabs(p1 ? r1[0] : r0[0]);
    swap_rows(r0, r1, p1 && !p2);
    swap_rows(r0, r2, p2);
    if (r0[0] == 0.0) return false;
    const double f1 = r1[0] / r0[0];
#pragma unroll
    for (int j = 0; j < 4; ++j) r1[j] -= f1 * r0[j];
    const double f2 = r2[0] / r0[0];
#pragma unroll
    for (int j = 0; j < 4; ++j) r2[j] -= f2 * r0[j];
  }
  {  // column 1
    swap_rows(r1, r2, fabs(r2[1]) > fabs(r1[1]));
    if (r1[1] == 0.0) return false;
    const double f2 = r2[1] / r1[1];
#pragma unroll
    for (int j = 1; j < 4; ++j) r2[j] -= f2 * r1[j];
  }
  if (r2[2] == 0.0) return false;
  x[2] = r2[3] / r2[2];
  x[1] = (r1[3] - r1[2] * x[2]) / r1[1];
  x[0] = ((r0[3] - r0[1] * x[1]) - r0[2] * x[2]) / r0[0];
  return true;
}

// project2cone (cone.jl:68-85) in the reference's own order: distance to the surface and the
// surface normal there, through the Rodrigues matrix of the axis perpendicular to (axis, apex->p)
__device__ inline double project2cone(D3 apex, D3 axis, double ct, double st, D3 p, D3* nrm) {
  const D3 tp = apex - p;
  const D3 tpn = unit(tp);
  const D3 rot = unit(cross(axis, tpn));
  const D3 cn = unit(cross(axis, rot));
  const D3 nv = unit(rot);
  const double v[3] = {nv.x, nv.y, nv.z};
  double R[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      const double o = v[i] * v[j];
      R[i][j] = o + ct * ((i == j ? 1.0 : 0.0) - o);
    }
  R[0][1] -= st * v[2];
  R[0][2] += st * v[1];
  R[1][0] += st * v[2];
  R[1][2] -= st * v[0];
  R[2][0] -= st * v[1];
  R[2][1] += st * v[0];
  const D3 rv = {R[0][0] * cn.x + R[0][1] * cn.y + R[0][2] * cn.z, R[1][0] * cn.x + R[1][1] * cn.y + R[1][2] * cn.z,
                 R[2][0] * cn.x + R[2][1] * cn.y + R[2][2] * cn.z};
  const D3 cur = unit(rv);
  *nrm = cur;
  return dot(-cur, -tp);
}

template <int KK>
__device__ bool fit_cone(const D3* p, const D3* n, const FitParams& f, rsc_cand* out) {
  constexpr int KA = KK ? KK : kMaxK;
  const int kk = KK ? KK : f.k;
  const double r[9] = {n[0].x, n[0].y, n[0].z, n[1].x, n[1].y, n[1].z, n[2].x, n[2].y, n[2].z};
  const double ds[3] = {dot(p[0], n[0]), dot(p[1], n[1]), dot(p[2], n[2])};
  // rank(r) == 3 && rank([r | -d]) == 3 (cone.jl:44,48).  Shortcut that cannot disagree with the SVD:
  // sigma_min(r) = |det| / (s1 s2) >= 2 |det| / |r|_F^2, the augmented matrix has sigma_min >= that of r,
  // and both tolerances are <= 3 eps |[r | -d]|_F.  Only when the bound is within a factor 1e4 of the
  // tolerance (numerically singular normals) are the singular values computed.
  const double det = r[0] * (r[4] * r[8] - r[5] * r[7]) - r[1] * (r[3] * r[8] - r[5] * r[6]) + r[2] * (r[3] * r[7] - r[4] * r[6]);
  double fr = 0.0;
  for (int i = 0; i < 9; ++i) fr += r[i] * r[i];
  const double fa = fr + ds[0] * ds[0] + ds[1] * ds[1] + ds[2] * ds[2];
  const bool clearly_full = 2.0 * fabs(det) > 1e4 * (3 * 2.220446049250313e-16) * sqrt(fa) * fr;  // false on NaN/Inf
  if (!clearly_full) {
    if (!full_rank3(r, 3)) return false;
    double rv[12];
    for (int i = 0; i < 3; ++i) {
      for (int j = 0; j < 3; ++j) rv[i * 4 + j] = r[i * 3 + j];
      rv[i * 4 + 3] = -1 * ds[i];
    }
    if (!full_rank3(rv, 4)) return false;
  }
  double ax3[3];
  if (!solve3(r, ds, ax3)) return false;
  const D3 ap = {ax3[0], ax3[1], ax3[2]};  // apex = intersection of the three tangent planes
  D3 u[3];
  for (int i = 0; i < 3; ++i) {
    const D3 d = p[i] - ap;
    const double nd = norm(d);
    u[i] = ap + D3{d.x / nd, d.y / nd, d.z / nd};
  }
  D3 ax = unit(cross(u[1] - u[0], u[2] - u[0]));
  const D3 sm = (u[0] + u[1]) + u[2];
  const D3 mid = {sm.x / 3, sm.y / 3, sm.z / 3};
  if (dot(ax, unit(mid - ap)) < 0) ax = -1.0 * ax;
  double ang[3];
  for (int i = 0; i < 3; ++i) {
    double c = dot(unit(p[i] - ap), ax);
    if (c == c) c = fmin(fmax(c, -1.0), 1.0);
    ang[i] = acos(c);
  }
  const double op = 2 * (ang[0] + ang[1] + ang[2]) / 3;  // full opening angle (Q7)
  // validatecone (cone.jl:87-115)
  const double ct = cos(-op / 2), st = sin(-op / 2);
  D3 nr[KA];
  _Pragma("unroll") for (int i = 0; i < kk; ++i)
    if (project2cone(ap, ax, ct, st, p[i], &nr[i]) > f.eps[RSC_CONE]) return false;  // signed (Q6)
  if (op < f.minconeopang) return false;
  double d[KA];
  _Pragma("unroll") for (int i = 0; i < kk; ++i) d[i] = dot(nr[i], n[i]);
  const int sd = side(d, kk, f.cosa[RSC_CONE]);
  if (sd == 0) return false;
  store(out, RSC_CONE, sd > 0, ap, ax, op);
  return true;
}

// ---- Philox4x32-10 -------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                           uint32_t* o) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
    const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
    c0 = n0, c1 = l1, c2 = n2, c3 = l0;
    k0 += 0x9E3779B9u, k1 += 0xBB67AE85u;
  }
  o[0] = c0, o[1] = c1, o[2] = c2, o[3] = c3;
}

struct SetStream {
  uint32_t k0, k1, s0, s1, ndraw, blk[4];
  __device__ SetStream(uint64_t seed, uint64_t set) : k0((uint32_t)seed), k1((uint32_t)(seed >> 32)), s0((uint32_t)set), s1((uint32_t)(set >> 32)), ndraw(0) {}
  __device__ uint64_t next() {
    const uint32_t i = ndraw++;
    if ((i & 1u) == 0) philox4x32(i >> 1, s0, s1, 0u, k0, k1, blk);
    return (i & 1u) ? ((uint64_t)blk[2] | ((uint64_t)blk[3] << 32)) : ((uint64_t)blk[0] | ((uint64_t)blk[1] << 32));
  }
  __device__ uint64_t below(uint64_t n) { return __umul64hi(next(), n); }  // rand(1:n) - 1
};

constexpr int kSelWords = 8;  // words per rank/select block (256 points): two 128-bit loads per select

__global__ void block_popc_kernel(const uint32_t* __restrict__ en, int64_t words, uint32_t* __restrict__ out, int nblk) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nblk) return;
  uint32_t s = 0;
  for (int w = 0; w < kSelWords; ++w) {
    const int64_t i = (int64_t)b * kSelWords + w;
    if (i < words) s += __popc(en[i]);
  }
  out[b] = s;
}

// index of the j-th (0-based) enabled point: binary search over the block offsets, then the
// block's 8 mask words in two 128-bit loads (n_pad is a multiple of 512, so blocks are never ragged)
__device__ inline int64_t select_enabled(const uint32_t* en, int64_t words, const unsigned long long* boff, int nblk,
                                         uint64_t j) {
  int lo = 0, hi = nblk - 1;  // last block whose offset <= j
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(boff + mid) <= j)
      lo = mid;
    else
      hi = mid - 1;
  }
  uint32_t rem = (uint32_t)(j - __ldg(boff + lo));
  const uint4* wp = reinterpret_cast<const uint4*>(en + (int64_t)lo * kSelWords);
  const uint4 A = __ldg(wp), B = __ldg(wp + 1);
  const uint32_t w[8] = {A.x, A.y, A.z, A.w, B.x, B.y, B.z, B.w};
#pragma unroll
  for (int q = 0; q < kSelWords; ++q) {
    const uint32_t c = __popc(w[q]);
    if (rem < c) return ((int64_t)lo * kSelWords + q) * 32 + __fns(w[q], 0, rem + 1);
    rem -= c;
  }
  return -1;
}

struct GatherSrc {
  const float* soa;  // cloud SoA (6 x n_pad), used when idx != nullptr or sampling
  int64_t n_pad;
  const double* P;   // explicit coordinates S x k x 3 (used when soa == nullptr)
  const double* N;
  const float* G;    // sharded storage: [S][k][6] float32 x y z nx ny nz gathered from the owning ranks
  const double* xyz64 = nullptr;  // exact clouds: the float64 coordinates the drawn points are read from instead of soa
  const double* nrm64 = nullptr;
};

// sharded storage: every rank writes the bit patterns of the drawn points it owns (zeros for the others);
// an int32 sum over the ranks then leaves every set's coordinates on every rank, bit for bit
__global__ void gather_owned_kernel(const int64_t* __restrict__ idx, int64_t nidx, const float* __restrict__ soa, int64_t n_pad,
                                    int64_t goff, int64_t n_local, float* __restrict__ out) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nidx) return;
  const int64_t g = idx[j] - goff;
  const bool mine = idx[j] >= 0 && g >= 0 && g < n_local;
#pragma unroll
  for (int f = 0; f < 6; ++f) out[j * 6 + f] = mine ? __ldg(soa + f * n_pad + g) : 0.f;
}

// samplepointcloud4! on the root cell: one thread per minimal set, writes its k indices (-1 = failed)
__global__ void __launch_bounds__(128) sample_kernel(int S, int k, uint64_t seed, uint64_t set0, int64_t n_points,
                                                     const uint32_t* __restrict__ enabled, int64_t words,
                                                     const unsigned long long* __restrict__ boff, int nblk,
                                                     const unsigned long long* __restrict__ n_enabled,
                                                     int64_t* __restrict__ idx_out) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  int64_t id[kMaxK];
  bool ok = true;
  SetStream rng(seed, set0 + (uint64_t)s);
  const uint64_t ne = *n_enabled;
  int64_t r1 = (int64_t)rng.below((uint64_t)n_points);
  if (ne == 0) {
    ok = false;
  } else {
    while (!((__ldg(enabled + (r1 >> 5)) >> (r1 & 31)) & 1u)) r1 = (int64_t)rng.below((uint64_t)n_points);
  }
  if (ok && ne < (uint64_t)k) ok = false;  // (false, 0): too few enabled points in the cell
  if (ok) {
    id[0] = r1;
    for (int q = 1; q < k; ++q) {
      int64_t c = select_enabled(enabled, words, boff, nblk, rng.below(ne));
      if (c == id[0]) c = select_enabled(enabled, words, boff, nblk, rng.below(ne));  // "try once more"
      id[q] = c;
    }
    for (int i = 1; i < k; ++i)
      for (int j = 0; j < i; ++j)
        if (id[i] == id[j]) ok = false;  // (false, 1): duplicate index
  }
  for (int q = 0; q < k; ++q) idx_out[(size_t)s * k + q] = ok ? id[q] : -1;
}

// ---- level-weighted cell sampler on the flattened octree (SURVEY 8(f)-1, rsc_octree.cu) ----------
struct CellsView {
  const uint32_t* codes;      // sorted Morton codes
  const uint32_t* perm;       // sorted position -> point index
  const uint32_t* inv;        // point index -> sorted position
  const uint8_t* leafdepth;   // by point index
  const uint32_t* en_sorted;  // isenabled in Morton order
  const unsigned long long* boff;  // rank blocks over en_sorted
  int nblk;
  int nlevels;
  double cum[11];             // cumulative level weights (host, float64, left to right)
};

// enabled points among sorted positions [0, p)
__device__ __forceinline__ uint64_t rank_sorted(const CellsView& c, int64_t p, int64_t words) {
  const int64_t blk = p / (kSelWords * 32);
  if (blk >= c.nblk) return __ldg(c.boff + c.nblk);  // p == n_pad: the total (stored behind the offsets)
  uint64_t r = __ldg(c.boff + blk);
  const int64_t w0 = blk * kSelWords, wp = p >> 5;
  for (int64_t w = w0; w < wp; ++w) r += __popc(__ldg(c.en_sorted + w));
  if (p & 31) r += __popc(__ldg(c.en_sorted + wp) & ((1u << (p & 31)) - 1u));
  return r;
}

__device__ __forceinline__ int64_t lower_bound_code(const uint32_t* __restrict__ codes, int64_t lo, int64_t hi, uint64_t key) {
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if ((uint64_t)__ldg(codes + mid) < key)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

// samplepointcloud4! (fitting.jl:383-430) with the cell of a drawn octree level: one thread per set.
// The level is DRAWN from the level distribution restricted to 1..leafdepth(r1) (docs/src/ransac.md:
// 80-82); the shipped code takes the argmax (fitting.jl:401), which never leaves level 1.
__global__ void __launch_bounds__(128) sample_cells_kernel(int S, int k, uint64_t seed, uint64_t set0, int64_t n_points,
                                                           const uint32_t* __restrict__ enabled, int64_t words, CellsView c,
                                                           int64_t* __restrict__ idx_out, int32_t* __restrict__ level_out) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  int64_t id[kMaxK];
  bool ok = true;
  int level = 0;
  SetStream rng(seed, set0 + (uint64_t)s);
  const uint64_t ne_all = __ldg(c.boff + c.nblk);
  if (ne_all == 0) {
    ok = false;
  } else {
    int64_t r1 = (int64_t)rng.below((uint64_t)n_points);
    while (!((__ldg(enabled + (r1 >> 5)) >> (r1 & 31)) & 1u)) r1 = (int64_t)rng.below((uint64_t)n_points);
    const int ld = c.leafdepth[r1];
    // level: smallest l with cum[l] > u * cum[ld]  (u = 64 random bits as a fraction)
    const double target = __dmul_rn(__dmul_rn((double)rng.next(), 5.421010862427522e-20 /* 2^-64 */), c.cum[ld - 1]);
    level = ld;
    for (int l = 1; l <= ld; ++l)
      if (c.cum[l - 1] > target) {
        level = l;
        break;
      }
    const int shift = 3 * ((c.nlevels - 1) - (level - 1));
    const uint32_t code = __ldg(c.codes + __ldg(c.inv + r1));
    const uint64_t lo_key = (uint64_t)(code >> shift) << shift;
    const int64_t a = lower_bound_code(c.codes, 0, n_points, lo_key);
    const int64_t b = lower_bound_code(c.codes, a, n_points, lo_key + ((uint64_t)1 << shift));
    const uint64_t ra = rank_sorted(c, a, words);
    const uint64_t ne = rank_sorted(c, b, words) - ra;
    if (ne < (uint64_t)k) ok = false;  // (false, 0): too few enabled points in the cell
    if (ok) {
      id[0] = r1;
      for (int q = 1; q < k; ++q) {
        int64_t p = (int64_t)__ldg(c.perm + select_enabled(c.en_sorted, words, c.boff, c.nblk, ra + rng.below(ne)));
        if (p == id[0]) p = (int64_t)__ldg(c.perm + select_enabled(c.en_sorted, words, c.boff, c.nblk, ra + rng.below(ne)));
        id[q] = p;
      }
      for (int i = 1; i < k; ++i)
        for (int j = 0; j < i; ++j)
          if (id[i] == id[j]) ok = false;  // (false, 1): duplicate index
    }
  }
  for (int q = 0; q < k; ++q) idx_out[(size_t)s * k + q] = ok ? id[q] : -1;
  level_out[s] = level;
}

// one thread per (minimal set, shape type): blockIdx.y = position in shape_types, so a warp runs
// one fit routine.  Points come from explicit coordinates (src.soa == nullptr) or from the cloud
// by index; sets whose first index is negative (failed samples) yield nothing.
// KK = 3: the minimal set of the reference's default drawN, everything in registers; KK = 0: f.k points (3..8)
template <int KK>
__global__ void __launch_bounds__(128) fit_kernel(GatherSrc src, const int64_t* __restrict__ idx, int S, FitParams f,
                                                  rsc_cand* __restrict__ dense, uint32_t* __restrict__ okmask) {
  constexpr int KA = KK ? KK : kMaxK;
  const int fk = KK ? KK : f.k;
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  const int t = blockIdx.y;
  if (f.types[t] >= RSC_NTYPES) return;  // a user position (block-uniform): its own fit kernel writes slot and ballot
  const size_t slot = (size_t)s * f.ntypes + t;
  bool ok = false;
  // (a set the sampler could not draw has idx < 0: no candidate)
  if (s < S && ((!src.G && !src.soa) || idx[(size_t)s * fk] >= 0)) {
  D3 p[KA], n[KA];
  if (src.G) {
    _Pragma("unroll") for (int q = 0; q < fk; ++q) {
      const float* g = src.G + ((size_t)s * fk + q) * 6;
      p[q] = D3{(double)g[0], (double)g[1], (double)g[2]};
      n[q] = D3{(double)g[3], (double)g[4], (double)g[5]};
    }
  } else if (src.xyz64) {
    _Pragma("unroll") for (int q = 0; q < fk; ++q) {
      const int64_t i = 3 * idx[(size_t)s * fk + q];
      p[q] = D3{__ldg(src.xyz64 + i), __ldg(src.xyz64 + i + 1), __ldg(src.xyz64 + i + 2)};
      n[q] = D3{__ldg(src.nrm64 + i), __ldg(src.nrm64 + i + 1), __ldg(src.nrm64 + i + 2)};
    }
  } else if (src.soa) {
    _Pragma("unroll") for (int q = 0; q < fk; ++q) {
      const int64_t i = idx[(size_t)s * fk + q];
      p[q] = D3{(double)__ldg(src.soa + i), (double)__ldg(src.soa + src.n_pad + i), (double)__ldg(src.soa + 2 * src.n_pad + i)};
      n[q] = D3{(double)__ldg(src.soa + 3 * src.n_pad + i), (double)__ldg(src.soa + 4 * src.n_pad + i),
                (double)__ldg(src.soa + 5 * src.n_pad + i)};
    }
  } else {
    _Pragma("unroll") for (int q = 0; q < fk; ++q) {
      const double* a = src.P + ((size_t)s * fk + q) * 3;
      const double* b = src.N + ((size_t)s * fk + q) * 3;
      p[q] = D3{a[0], a[1], a[2]};
      n[q] = D3{b[0], b[1], b[2]};
    }
  }
  rsc_cand c;
  switch (f.types[t]) {
    case RSC_PLANE:
      ok = fit_plane<KK>(p, n, f, &c);
      break;
    case RSC_SPHERE:
      ok = fit_sphere<KK>(p, n, f, &c);
      break;
    case RSC_CYLINDER:
      ok = fit_cylinder<KK>(p, n, f, &c);
      break;
    case RSC_CONE:
      ok = fit_cone<KK>(p, n, f, &c);
      break;
  }
  if (ok) dense[slot] = c;
  }
  // which of the warp's 32 sets gave a candidate of this type: one word per (group of 128 sets, type, warp)
  const uint32_t m = __ballot_sync(0xffffffffu, ok);
  if ((threadIdx.x & 31) == 0) okmask[((size_t)blockIdx.x * f.ntypes + t) * 4 + (threadIdx.x >> 5)] = m;
}

// ---- order-preserving compaction of the dense candidates (slot order = set-major, type-minor) ----------------
// The candidates are sparse (c4: ~0.1 % of the slots), so instead of a scan over all slots: the fit kernel leaves
// one ballot word per (group of 128 sets, type, warp); ONE CTA scans the groups' bit counts (a group = 4 ntypes
// words), and every candidate finds its rank inside its group from those words.
// seg (optional): the loops' segment bounds -- seg[j] = candidates of the sets before j * sets_per_iter, j = 0..nb;
// needs sets_per_iter to be a multiple of 128 (then a segment starts at a group)
__global__ void __launch_bounds__(1024) group_scan_kernel(const uint32_t* __restrict__ okmask, int G, int ntypes,
                                                          uint32_t* __restrict__ base, unsigned long long* __restrict__ out_total,
                                                          int32_t* __restrict__ seg, int sets_per_iter, int nb) {
  __shared__ uint32_t wsum[32];
  __shared__ uint32_t carry, chunk;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int g0 = 0; g0 < G; g0 += 1024) {
    const int g = g0 + tid;
    uint32_t cnt = 0;
    if (g < G)
      for (int i = 0; i < 4 * ntypes; ++i) cnt += __popc(okmask[(size_t)g * 4 * ntypes + i]);
    uint32_t inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += o;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      const uint32_t v = wsum[lane];
      uint32_t vi = v;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, vi, d);
        if (lane >= d) vi += o;
      }
      wsum[lane] = vi - v;
      if (lane == 31) chunk = vi;
    }
    __syncthreads();
    if (g < G) base[g] = carry + wsum[warp] + (inc - cnt);
    __syncthreads();
    if (tid == 0) carry += chunk;
    __syncthreads();
  }
  if (tid == 0) *out_total = carry;
  if (seg && tid <= nb) {  // (the last barrier of the loop made base[] and carry visible)
    const long long g = (long long)tid * sets_per_iter / 128;
    seg[tid] = (tid == nb || g >= G) ? (int32_t)carry : (int32_t)base[g];
  }
}

// same grid as the fit kernel: thread = (set, type)
__global__ void __launch_bounds__(128) compact_kernel(const rsc_cand* __restrict__ dense, const uint32_t* __restrict__ okmask,
                                                      const uint32_t* __restrict__ base, int ntypes, rsc_cand* __restrict__ out,
                                                      int32_t* __restrict__ out_set) {
  __shared__ uint32_t m[4 * RSC_MAX_ORDER];  // [type][warp]
  const int t = blockIdx.y, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (threadIdx.x < 4 * ntypes) m[threadIdx.x] = okmask[(size_t)blockIdx.x * 4 * ntypes + threadIdx.x];
  __syncthreads();
  if (!((m[t * 4 + w] >> lane) & 1u)) return;
  uint32_t rank = base[blockIdx.x];
  const uint32_t below = (1u << lane) - 1u;
  for (int tt = 0; tt < ntypes; ++tt) {
    for (int ww = 0; ww < w; ++ww) rank += __popc(m[tt * 4 + ww]);  // sets of earlier warps, every type
    rank += __popc(m[tt * 4 + w] & below);                            // earlier sets of this warp, every type
    if (tt < t) rank += (m[tt * 4 + w] >> lane) & 1u;                 // this set, earlier types
  }
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  out[rank] = dense[(size_t)s * ntypes + t];
  if (out_set) out_set[rank] = s;
}

__global__ void scan_u32_kernel(const uint32_t* __restrict__ counts, int n, unsigned long long* __restrict__ offsets,
                                unsigned long long* __restrict__ out_total);  // defined below

int32_t make_fit_params(rsc_ctx* ctx, const rsc_params* p, int k, FitParams* f) {
  if (!p) return fail(ctx, RSC_E_ARG, "params is null");
  if (k < 3 || k > kMaxK) return fail(ctx, RSC_E_ARG, "fit: a set needs 3..8 points (At least 3 point is needed)");
  if (p->n_shape_types < 0 || p->n_shape_types > RSC_NTYPES) return fail(ctx, RSC_E_ARG, "fit: bad n_shape_types");
  for (int t = 0; t < RSC_NTYPES; ++t) {
    f->eps[t] = p->eps[t];
    f->cosa[t] = cos(p->alpha[t]);
  }
  f->cos_par = cos(p->parallelthrdeg * (M_PI / 180.0));
  f->sphere_par = p->sphere_par;
  f->minconeopang = p->minconeopang;
  f->collin = p->collin_threshold;
  f->ntypes = p->n_shape_types;
  for (int t = 0; t < p->n_shape_types; ++t) {
    if (p->shape_types[t] < 0 || p->shape_types[t] >= RSC_NTYPES) return fail(ctx, RSC_E_ARG, "fit: unknown shape type");
    f->types[t] = p->shape_types[t];
  }
  f->k = k;
  return RSC_OK;
}

static int32_t carve(rsc_ctx* ctx, int S, int ntypes, int k, FitScratch* fs) {
  const size_t slots = (size_t)S * (ntypes > 0 ? ntypes : 1);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += (bytes + 255) / 256 * 256;
    return o;
  };
  const size_t o_dense = take(slots * sizeof(rsc_cand)), o_out = take(slots * sizeof(rsc_cand));
  const size_t groups = ((size_t)S + 127) / 128;
  const size_t o_flags = take(groups * 4 * (ntypes > 0 ? ntypes : 1) * 4), o_offs = take(groups * 4), o_total = take(8);
  const size_t o_set = take(slots * 4), o_idx = take((size_t)S * k * 8), o_level = take((size_t)S * 4);
  const size_t o_gath = take((size_t)S * k * 6 * 4);
  RSC_CUDA(ctx, ctx->fitbuf.ensure(off));
  char* b = ctx->fitbuf.as<char>();
  fs->dense = (rsc_cand*)(b + o_dense);
  fs->out = (rsc_cand*)(b + o_out);
  fs->okmask = (uint32_t*)(b + o_flags);
  fs->base = (uint32_t*)(b + o_offs);
  fs->total = (unsigned long long*)(b + o_total);
  fs->out_set = (int32_t*)(b + o_set);
  fs->idx = (int64_t*)(b + o_idx);
  fs->level = (int32_t*)(b + o_level);
  fs->gath = (float*)(b + o_gath);
  return RSC_OK;
}

// rank/select index over the enabled mask; cached on the cloud until the mask changes
int32_t build_select_index(rsc_cloud* cloud, cudaStream_t st, unsigned long long** boff, int* nblk,
                           unsigned long long** n_enabled) {
  rsc_ctx* ctx = cloud->ctx;
  // a shard samples from the replicated whole-cloud mask (same sets on every rank)
  const uint32_t* mask = cloud->is_shard() ? cloud->g_enabled : cloud->enabled;
  const int64_t words = cloud->is_shard() ? cloud->g_words : cloud->n_pad / 32;
  const int nb = (int)((words + kSelWords - 1) / kSelWords);
  RSC_CUDA(ctx, cloud->selbuf.ensure((size_t)nb * (4 + 8) + 64));
  char* b = cloud->selbuf.as<char>();
  unsigned long long* offs = (unsigned long long*)b;
  unsigned long long* total = offs + nb;
  uint32_t* cnt = (uint32_t*)(total + 1);
  if (!cloud->sel_valid) {
    block_popc_kernel<<<(nb + 255) / 256, 256, 0, st>>>(mask, words, cnt, nb);
    RSC_CUDA(ctx, cudaGetLastError());
    if (int32_t rcs = scan_u32(ctx, cnt, nb, offs, total, st)) return rcs;
    cloud->sel_valid = true;
  }
  *boff = offs;
  *nblk = nb;
  *n_enabled = total;
  return RSC_OK;
}

// exclusive scan of n counts by ONE CTA (n is small: flags of a batch, block counts of a mask);
// every thread takes 8 consecutive elements per pass, so 8192 elements cost one block-wide scan
// the same index over isenabled in Morton order (cell sampler); refreshed lazily after every change
int32_t build_cells_index(rsc_cloud* cloud, cudaStream_t st, const double* cum, CellsView* v) {
  rsc_ctx* ctx = cloud->ctx;
  rsc_cells& c = cloud->cells;
  if (c.nlevels == 0) return fail(ctx, RSC_E_STATE, "cell sampler: rsc_cloud_build_cells has not been called");
  if (int32_t rc = cells_refresh_enabled(cloud, st)) return rc;
  const int64_t words = cloud->n_pad / 32;
  const int nb = (int)((words + kSelWords - 1) / kSelWords);
  RSC_CUDA(ctx, c.selbuf.ensure((size_t)nb * (4 + 8) + 64));
  unsigned long long* offs = c.selbuf.as<unsigned long long>();
  unsigned long long* total = offs + nb;
  uint32_t* cnt = (uint32_t*)(total + 1);
  if (!c.sel_valid) {
    block_popc_kernel<<<(nb + 255) / 256, 256, 0, st>>>(c.en_sorted, words, cnt, nb);
    RSC_CUDA(ctx, cudaGetLastError());
    if (int32_t rcs = scan_u32(ctx, cnt, nb, offs, total, st)) return rcs;
    c.sel_valid = true;
  }
  v->codes = c.codes, v->perm = c.perm, v->inv = c.inv, v->leafdepth = c.leafdepth, v->en_sorted = c.en_sorted;
  v->boff = offs, v->nblk = nb, v->nlevels = c.nlevels;
  for (int l = 0; l < 11; ++l) v->cum[l] = l < c.nlevels ? cum[l] : 0.0;
  return RSC_OK;
}

__global__ void __launch_bounds__(1024) scan_u32_kernel(const uint32_t* __restrict__ counts, int n,
                                                        unsigned long long* __restrict__ offsets,
                                                        unsigned long long* __restrict__ out_total) {
  constexpr int E = 8;
  __shared__ unsigned long long wex[32];
  __shared__ unsigned long long carry, chunk_total;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < n; base += 1024 * E) {
    const int i0 = base + tid * E;
    uint32_t v[E];
#pragma unroll
    for (int e = 0; e < E; ++e) v[e] = (i0 + e < n) ? counts[i0 + e] : 0u;
    unsigned long long s = 0;
#pragma unroll
    for (int e = 0; e < E; ++e) s += v[e];
    unsigned long long inc = s;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned long long o = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += o;
    }
    if (lane == 31) wex[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      const unsigned long long t = wex[lane];
      unsigned long long ti = t;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long o = __shfl_up_sync(0xffffffffu, ti, d);
        if (lane >= d) ti += o;
      }
      wex[lane] = ti - t;
      if (lane == 31) chunk_total = ti;
    }
    __syncthreads();
    unsigned long long run = carry + wex[warp] + (inc - s);
#pragma unroll
    for (int e = 0; e < E; ++e) {
      if (i0 + e < n) offsets[i0 + e] = run;
      run += v[e];
    }
    __syncthreads();
    if (tid == 0) carry += chunk_total;
    __syncthreads();
  }
  if (tid == 0) *out_total = carry;
}

// ---- exclusive scan of n uint32 counts into 64-bit offsets (+ total), any n -------------------
// Up to 32 Ki elements one CTA does it; beyond that: per-CTA sums of 8 Ki-element tiles, a one-CTA scan
// of the tile sums, and a second pass in which every CTA scans its own tile on top of its offset.
constexpr int kScanTile = 8192;

__global__ void __launch_bounds__(1024) scan_tile_sums_kernel(const uint32_t* __restrict__ counts, int n, uint32_t* __restrict__ sums) {
  __shared__ uint32_t ws[32];
  const int base = blockIdx.x * kScanTile;
  uint32_t s = 0;
#pragma unroll
  for (int e = 0; e < kScanTile / 1024; ++e) {
    const int i = base + e * 1024 + threadIdx.x;
    if (i < n) s += counts[i];
  }
  s = __reduce_add_sync(0xffffffffu, s);
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    s = __reduce_add_sync(0xffffffffu, ws[threadIdx.x]);
    if (threadIdx.x == 0) sums[blockIdx.x] = s;
  }
}

__global__ void __launch_bounds__(1024) scan_tile_apply_kernel(const uint32_t* __restrict__ counts, int n,
                                                               const unsigned long long* __restrict__ tile_off,
                                                               unsigned long long* __restrict__ offsets) {
  constexpr int E = kScanTile / 1024;
  __shared__ unsigned long long wex[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int i0 = blockIdx.x * kScanTile + tid * E;
  uint32_t v[E];
  unsigned long long s = 0;
#pragma unroll
  for (int e = 0; e < E; ++e) {
    v[e] = (i0 + e < n) ? counts[i0 + e] : 0u;
    s += v[e];
  }
  unsigned long long inc = s;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned long long o = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += o;
  }
  if (lane == 31) wex[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const unsigned long long t = wex[lane];
    unsigned long long ti = t;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned long long o = __shfl_up_sync(0xffffffffu, ti, d);
      if (lane >= d) ti += o;
    }
    wex[lane] = ti - t;
  }
  __syncthreads();
  unsigned long long run = tile_off[blockIdx.x] + wex[warp] + (inc - s);
#pragma unroll
  for (int e = 0; e < E; ++e) {
    if (i0 + e < n) offsets[i0 + e] = run;
    run += v[e];
  }
}

int32_t scan_u32(rsc_ctx* ctx, const uint32_t* counts, int n, unsigned long long* offsets, unsigned long long* total,
                 cudaStream_t st) {
  if (n <= 4 * kScanTile) {
    scan_u32_kernel<<<1, 1024, 0, st>>>(counts, n, offsets, total);
    RSC_CUDA(ctx, cudaGetLastError());
    return RSC_OK;
  }
  const int tiles = (n + kScanTile - 1) / kScanTile;
  RSC_CUDA(ctx, ctx->scanbuf.ensure((size_t)tiles * (4 + 8) + 64));
  unsigned long long* toff = ctx->scanbuf.as<unsigned long long>();
  uint32_t* tsum = (uint32_t*)(toff + tiles + 1);
  scan_tile_sums_kernel<<<tiles, 1024, 0, st>>>(counts, n, tsum);
  RSC_CUDA(ctx, cudaGetLastError());
  scan_u32_kernel<<<1, 1024, 0, st>>>(tsum, tiles, toff, total);
  RSC_CUDA(ctx, cudaGetLastError());
  scan_tile_apply_kernel<<<tiles, 1024, 0, st>>>(counts, n, toff, offsets);
  RSC_CUDA(ctx, cudaGetLastError());
  return RSC_OK;
}

// Enqueue fit (+ sampling) for S sets; leaves compacted candidates in ctx->fitbuf (FitScratch.out),
// their count in FitScratch.total.  No synchronisation.
// size the scratch for batches of up to S sets once (the device loop grows its batches while it runs)
int32_t fit_reserve(rsc_ctx* ctx, const rsc_params* params, int S, int ntypes) {
  FitScratch fs;
  return carve(ctx, S, ntypes >= 0 ? ntypes : params->n_shape_types, params->drawN, &fs);
}

// mode 0: explicit coordinates, 1: explicit indices, 2: root-cell sampler (the reference's behaviour,
// Q1), 3: level-weighted cell sampler on the flattened octree (`cum` = cumulative level weights)
int32_t fit_enqueue(rsc_ctx* ctx, rsc_cloud* cloud, int mode, const rsc_params* params, int k, const double* dP,
                    const double* dN, const int64_t* d_idx, int S, uint64_t seed, uint64_t set0, cudaStream_t st,
                    FitScratch* fs, const double* cum, int32_t* d_seg, int sets_per_iter, int nb, const FitOrder* order) {
  if (d_seg && (sets_per_iter <= 0 || sets_per_iter % 128 || nb < 0 || nb >= 1024)) return fail(ctx, RSC_E_ARG, "fit: segment bounds need sets_per_iter % 128 == 0");
  FitParams f;
  int32_t rc;
  if (order) {  // a mixed order replaces params->shape_types
    rsc_params pb = *params;
    pb.n_shape_types = 0;
    if ((rc = make_fit_params(ctx, &pb, k, &f))) return rc;
    if (order->has_user && (mode != 2 || !cloud || cloud->is_shard())) return fail(ctx, RSC_E_STATE, "fit: user shapes fit on the root-cell sampler of a whole cloud only");
    f.ntypes = order->n;
    for (int t = 0; t < order->n; ++t) f.types[t] = order->type[t];
  } else if ((rc = make_fit_params(ctx, params, k, &f))) {
    return rc;
  }
  if ((rc = carve(ctx, S, f.ntypes, k, fs))) return rc;
  const int slots = S * f.ntypes;
  GatherSrc src{nullptr, 0, dP, dN, nullptr};
  const bool shard = cloud && cloud->is_shard();
  if (shard && mode != 2) return fail(ctx, RSC_E_STATE, "fit: a shard (sharded storage) only supports the root-cell sampler of rsc_ransac_run");
  unsigned long long *boff = nullptr, *nen = nullptr;
  int nblk = 0;
  if (mode != 0) {
    src.soa = cloud->soa;
    src.n_pad = cloud->n_pad;
    src.xyz64 = cloud->xyz64;
    src.nrm64 = cloud->nrm64;
  }
  if (mode == 3 && cloud->exact())
    return fail(ctx, RSC_E_STATE, "fit: the cell sampler (octree quantisation) does not support exact clouds yet");
  if (mode == 2 && (rc = build_select_index(cloud, st, &boff, &nblk, &nen))) return rc;
  CellsView cv;
  if (mode == 3 && (rc = build_cells_index(cloud, st, cum, &cv))) return rc;
  if (slots > 0 || (order && S > 0)) {  // (an empty order only draws)
    const int64_t* use_idx = d_idx;
    if (mode == 3) {
      sample_cells_kernel<<<(S + 127) / 128, 128, 0, st>>>(S, k, seed, set0, cloud->n, cloud->enabled, cloud->n_pad / 32, cv,
                                                           fs->idx, fs->level);
      RSC_CUDA(ctx, cudaGetLastError());
      use_idx = fs->idx;
    } else if (mode == 2 && shard) {
      // sharded storage: global indices from the replicated mask, coordinates gathered from their owners
      sample_kernel<<<(S + 127) / 128, 128, 0, st>>>(S, k, seed, set0, cloud->n_global, cloud->g_enabled, cloud->g_words, boff, nblk,
                                                     nen, fs->idx);
      RSC_CUDA(ctx, cudaGetLastError());
      const int64_t nidx = (int64_t)S * k;
      gather_owned_kernel<<<(unsigned)((nidx + 255) / 256), 256, 0, st>>>(fs->idx, nidx, cloud->soa, cloud->n_pad, cloud->global_offset,
                                                                           cloud->n, fs->gath);
      RSC_CUDA(ctx, cudaGetLastError());
      if (!ctx->allreduce || ctx->allreduce(ctx->allreduce_user, fs->gath, nidx * 6, (void*)st))
        return fail(ctx, RSC_E_NCCL, "fit: gathering the minimal sets' coordinates (all-reduce) failed");
      src.G = fs->gath;
      use_idx = fs->idx;
    } else if (mode == 2) {
      sample_kernel<<<(S + 127) / 128, 128, 0, st>>>(S, k, seed, set0, cloud->n, cloud->enabled, cloud->n_pad / 32, boff, nblk,
                                                     nen, fs->idx);
      RSC_CUDA(ctx, cudaGetLastError());
      use_idx = fs->idx;
    }
    if (slots == 0) {
      RSC_CUDA(ctx, cudaMemsetAsync(fs->total, 0, 8, st));
      ctx->stats.sets_drawn += S;
      return RSC_OK;
    }
    if (k == 3)
      fit_kernel<3><<<dim3((S + 127) / 128, f.ntypes), 128, 0, st>>>(src, use_idx, S, f, fs->dense, fs->okmask);
    else
      fit_kernel<0><<<dim3((S + 127) / 128, f.ntypes), 128, 0, st>>>(src, use_idx, S, f, fs->dense, fs->okmask);
    RSC_CUDA(ctx, cudaGetLastError());
    if (order)
      for (int t = 0; t < order->n; ++t)
        if (order->type[t] >= RSC_NTYPES && (rc = user_fit_enqueue(ctx, *order, t, cloud, use_idx, S, k, fs->dense, fs->okmask, st)))
          return rc;
    group_scan_kernel<<<1, 1024, 0, st>>>(fs->okmask, (S + 127) / 128, f.ntypes, fs->base, fs->total, d_seg, sets_per_iter, nb);
    RSC_CUDA(ctx, cudaGetLastError());
    compact_kernel<<<dim3((S + 127) / 128, f.ntypes), 128, 0, st>>>(fs->dense, fs->okmask, fs->base, f.ntypes, fs->out, fs->out_set);
    RSC_CUDA(ctx, cudaGetLastError());
  } else {
    RSC_CUDA(ctx, cudaMemsetAsync(fs->total, 0, 8, st));
    if (d_seg) RSC_CUDA(ctx, cudaMemsetAsync(d_seg, 0, (size_t)(nb + 1) * 4, st));
  }
  ctx->stats.sets_drawn += S;
  return RSC_OK;
}

static int32_t fit_finish(rsc_ctx* ctx, const FitScratch& fs, int S, int k, cudaStream_t st, rsc_cand* out,
                          int32_t* out_set, int64_t* out_idx, int32_t* out_n) {
  unsigned long long total = 0;
  RSC_CUDA(ctx, cudaMemcpyAsync(&total, fs.total, 8, cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaStreamSynchronize(st));
  *out_n = (int32_t)total;
  if (total) {
    if (out) RSC_CUDA(ctx, cudaMemcpyAsync(out, fs.out, (size_t)total * sizeof(rsc_cand), cudaMemcpyDeviceToHost, st));
    if (out_set) RSC_CUDA(ctx, cudaMemcpyAsync(out_set, fs.out_set, (size_t)total * 4, cudaMemcpyDeviceToHost, st));
  }
  if (out_idx) RSC_CUDA(ctx, cudaMemcpyAsync(out_idx, fs.idx, (size_t)S * k * 8, cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaStreamSynchronize(st));
  return RSC_OK;
}

}  // namespace rsc

using namespace rsc;

extern "C" {

void rsc_level_cumsum(const double* levelweight, int32_t nlevels, double* cum);

int32_t rsc_fit_points(rsc_ctx* ctx, const rsc_params* params, const double* p, const double* n, int32_t S, int32_t k,
                       rsc_cand* out, int32_t* out_set, int32_t* out_n) {
  if (!ctx) return RSC_E_ARG;
  if (!out_n || S < 0 || (S > 0 && (!p || !n || !out))) return fail(ctx, RSC_E_ARG, "fit_points: null arguments");
  *out_n = 0;
  if (S == 0) return RSC_OK;
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t bytes = (size_t)S * k * 3 * sizeof(double);
  RSC_CUDA(ctx, ctx->misc.ensure(bytes));
  RSC_CUDA(ctx, ctx->misc2.ensure(bytes));
  RSC_CUDA(ctx, cudaMemcpyAsync(ctx->misc.p, p, bytes, cudaMemcpyHostToDevice, st));
  RSC_CUDA(ctx, cudaMemcpyAsync(ctx->misc2.p, n, bytes, cudaMemcpyHostToDevice, st));
  FitScratch fs;
  int32_t rc = fit_enqueue(ctx, nullptr, 0, params, k, ctx->misc.as<double>(), ctx->misc2.as<double>(), nullptr, S, 0, 0, st, &fs);
  if (rc) return rc;
  return fit_finish(ctx, fs, S, k, st, out, out_set, nullptr, out_n);
}

int32_t rsc_fit_batch(rsc_cloud* cloud, const rsc_params* params, const int64_t* idx, int32_t S, rsc_cand* out,
                      int32_t* out_set, int32_t* out_n) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (!params || !out_n || S < 0 || (S > 0 && (!idx || !out))) return fail(ctx, RSC_E_ARG, "fit_batch: null arguments");
  *out_n = 0;
  if (S == 0) return RSC_OK;
  const int k = params->drawN;
  if (k < 3 || k > kMaxK) return fail(ctx, RSC_E_ARG, "fit_batch: drawN must be 3..8");
  for (int64_t i = 0; i < (int64_t)S * k; ++i)
    if (idx[i] < 0 || idx[i] >= cloud->n) return fail(ctx, RSC_E_ARG, "fit_batch: index out of range");
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if (int32_t rcr = cloud_ready(cloud)) return rcr;
  cudaStream_t st = ctx->stream;
  RSC_CUDA(ctx, ctx->misc.ensure((size_t)S * k * 8));
  RSC_CUDA(ctx, cudaMemcpyAsync(ctx->misc.p, idx, (size_t)S * k * 8, cudaMemcpyHostToDevice, st));
  FitScratch fs;
  int32_t rc = fit_enqueue(ctx, cloud, 1, params, k, nullptr, nullptr, ctx->misc.as<int64_t>(), S, 0, 0, st, &fs);
  if (rc) return rc;
  return fit_finish(ctx, fs, S, k, st, out, out_set, nullptr, out_n);
}

int32_t rsc_sample_fit(rsc_cloud* cloud, const rsc_params* params, uint64_t seed, uint64_t set0, int32_t S,
                       rsc_cand* out, int32_t* out_set, int64_t* out_idx, int32_t* out_n) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (!params || !out_n || S < 0 || (S > 0 && !out)) return fail(ctx, RSC_E_ARG, "sample_fit: null arguments");
  *out_n = 0;
  if (S == 0) return RSC_OK;
  const int k = params->drawN;
  if (k < 3 || k > kMaxK) return fail(ctx, RSC_E_ARG, "sample_fit: drawN must be 3..8");
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if (int32_t rcr = cloud_ready(cloud)) return rcr;
  cudaStream_t st = ctx->stream;
  FitScratch fs;
  int32_t rc = fit_enqueue(ctx, cloud, 2, params, k, nullptr, nullptr, nullptr, S, seed, set0, st, &fs);
  if (rc) return rc;
  return fit_finish(ctx, fs, S, k, st, out, out_set, out_idx, out_n);
}

int32_t rsc_sample_fit_user(rsc_cloud* cloud, const rsc_params* params, const void* order, int32_t norder,
                            uint64_t seed, uint64_t set0, int32_t S, rsc_cand* out, int32_t* out_set, int64_t* out_idx,
                            int32_t* out_n) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (!params || !out_n || S < 0 || (S > 0 && norder > 0 && !out) || (norder > 0 && !order))
    return fail(ctx, RSC_E_ARG, "sample_fit_user: null arguments");
  *out_n = 0;
  FitOrder fo;
  int32_t rc = make_fit_order(ctx, static_cast<const rsc_shape_slot*>(order), norder, &fo, "sample_fit_user");
  if (rc) return rc;
  if (fo.has_user && (cloud->is_shard() || cloud->range_set))
    return fail(ctx, RSC_E_STATE, "sample_fit_user: sharded or ranged clouds are not supported");
  if (S == 0) return RSC_OK;
  const int k = params->drawN;
  if (k < 3 || k > kMaxK) return fail(ctx, RSC_E_ARG, "sample_fit_user: drawN must be 3..8");
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if (int32_t rcr = cloud_ready(cloud)) return rcr;
  cudaStream_t st = ctx->stream;
  FitScratch fs;
  if ((rc = fit_enqueue(ctx, cloud, 2, params, k, nullptr, nullptr, nullptr, S, seed, set0, st, &fs, nullptr, nullptr, 0, 0, &fo)))
    return rc;
  return fit_finish(ctx, fs, S, k, st, out, out_set, out_idx, out_n);
}

int32_t rsc_sample_fit_cells(rsc_cloud* cloud, const rsc_params* params, uint64_t seed, uint64_t set0, int32_t S,
                             const double* levelweight, int32_t nlevels, rsc_cand* out, int32_t* out_set, int64_t* out_idx,
                             int32_t* out_level, int32_t* out_n) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (!params || !out_n || !levelweight || S < 0 || (S > 0 && !out)) return fail(ctx, RSC_E_ARG, "sample_fit_cells: null arguments");
  *out_n = 0;
  if (S == 0) return RSC_OK;
  if (nlevels != cloud->cells.nlevels) return fail(ctx, RSC_E_ARG, "sample_fit_cells: nlevels differs from rsc_cloud_build_cells");
  const int k = params->drawN;
  if (k < 3 || k > kMaxK) return fail(ctx, RSC_E_ARG, "sample_fit_cells: drawN must be 3..8");
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if (int32_t rcr = cloud_ready(cloud)) return rcr;
  cudaStream_t st = ctx->stream;
  double cum[11];
  rsc_level_cumsum(levelweight, nlevels, cum);
  FitScratch fs;
  int32_t rc = fit_enqueue(ctx, cloud, 3, params, k, nullptr, nullptr, nullptr, S, seed, set0, st, &fs, cum);
  if (rc) return rc;
  if (out_level) RSC_CUDA(ctx, cudaMemcpyAsync(out_level, fs.level, (size_t)S * 4, cudaMemcpyDeviceToHost, st));
  return fit_finish(ctx, fs, S, k, st, out, out_set, out_idx, out_n);
}

void rsc_level_cumsum(const double* levelweight, int32_t nlevels, double* cum) {
  double c = 0.0;
  for (int l = 0; l < nlevels && l < 11; ++l) {
    c += levelweight[l];
    cum[l] = c;
  }
}

/* octree.jl:198-205; the weights stay unchanged while no level has a score (w = 0 would give NaN).  x is the
 * Rational 9//10 there: x*sigma is Float64(9//10)*sigma, but (1-x)/length(P) stays the exact rational 1//(10 n) until
 * it meets the float term, i.e. it enters as the correctly rounded 1/(10 n) -- not as (1 - 0.9)/n, which is 1 ulp off */
void rsc_update_levelweight(double* levelweight, const double* levelscore, int32_t nlevels) {
  if (nlevels > 11) nlevels = 11;
  double w = 0.0;
  for (int i = 0; i < nlevels; ++i) w += levelscore[i] / levelweight[i];
  if (!(w > 0.0)) return;
  const double floor_w = 1.0 / (10.0 * (double)nlevels);
  double nw[11];
  for (int i = 0; i < nlevels; ++i) nw[i] = 0.9 * levelscore[i] / (w * levelweight[i]) + floor_w;
  for (int i = 0; i < nlevels; ++i) levelweight[i] = nw[i];
}

}  // extern "C"
