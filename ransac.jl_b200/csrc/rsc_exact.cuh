// rsc_exact.cuh -- FP64 re-evaluation of one (candidate, point) pair in the REFERENCE's operation
// order.  Used only for pairs whose FP32 margin falls inside the guard band, so that the inlier
// decision equals the float64 reference's (compatibles*: plane.jl:114-130, sphere.jl:144-172,
// cylinder.jl:194-221, cone.jl:132-153 with project2cone :68-85 and rodrigues utilities.jl:19-43).
//
// Every operation is an explicit round-to-nearest intrinsic: nvcc never contracts those into FMAs,
// so the rounding sequence is the one a plain IEEE evaluation of the reference source produces.
#pragma once
#include "rsc_common.cuh"

namespace rsc {
namespace ex {

struct V3 {
  double x, y, z;
};

__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ V3 sub(V3 a, V3 b) { return {sub(a.x, b.x), sub(a.y, b.y), sub(a.z, b.z)}; }
__device__ __forceinline__ V3 neg(V3 a) { return {-a.x, -a.y, -a.z}; }
__device__ __forceinline__ V3 scale(double s, V3 a) { return {mul(s, a.x), mul(s, a.y), mul(s, a.z)}; }
__device__ __forceinline__ double dot(V3 a, V3 b) {
  return add(add(mul(a.x, b.x), mul(a.y, b.y)), mul(a.z, b.z));
}
__device__ __forceinline__ double norm(V3 a) { return __dsqrt_rn(dot(a, a)); }
// StaticArrays: normalize(a) = inv(norm(a)) * a
__device__ __forceinline__ V3 normalize(V3 a) { return scale(__ddiv_rn(1.0, norm(a)), a); }
__device__ __forceinline__ V3 cross(V3 a, V3 b) {
  return {sub(mul(a.y, b.z), mul(a.z, b.y)), sub(mul(a.z, b.x), mul(a.x, b.z)),
          sub(mul(a.x, b.y), mul(a.y, b.x))};
}

// The float64 coordinates of point j of a set: on an exact cloud the caller's own, else the float32 ones widened
// (which is what the reference sees for a Float32 cloud).  Padding points (j >= n) are zero either way.
__device__ __forceinline__ void point64(const PointSet& ps, int64_t j, V3* p, V3* n) {
  if (ps.xyz64 && j < ps.n) {
    const int64_t i = 3 * (ps.map ? ps.map[j] : j);
    *p = V3{ps.xyz64[i], ps.xyz64[i + 1], ps.xyz64[i + 2]};
    *n = V3{ps.nrm64[i], ps.nrm64[i + 1], ps.nrm64[i + 2]};
  } else {
    *p = V3{(double)ps.x[j], (double)ps.y[j], (double)ps.z[j]};
    *n = V3{(double)ps.nx[j], (double)ps.ny[j], (double)ps.nz[j]};
  }
}

// cos/sin of -opang/2 for the cone's Rodrigues matrix
struct ConeTrig {
  double ct, st;
};

__device__ inline bool compat_plane(const rsc_cand& c, V3 p, V3 n, double eps, double thr) {
  V3 q = {c.p[0], c.p[1], c.p[2]};
  V3 m = {c.p[3], c.p[4], c.p[5]};
  V3 oz = normalize(m);
  double pz = dot(oz, sub(p, q));
  return (dot(m, n) > thr) && (fabs(pz) < eps);
}

__device__ inline bool compat_sphere(const rsc_cand& c, V3 p, V3 n, double eps, double thr) {
  V3 o = {c.p[0], c.p[1], c.p[2]};
  double R = c.p[3];
  V3 u = c.outwards ? normalize(sub(p, o)) : normalize(sub(o, p));
  return (dot(u, n) > thr) && (fabs(sub(norm(sub(p, o)), R)) < eps);
}

__device__ inline bool compat_cylinder(const rsc_cand& c, V3 p, V3 n, double eps, double thr) {
  V3 a = {c.p[0], c.p[1], c.p[2]};
  V3 ce = {c.p[3], c.p[4], c.p[5]};
  double R = c.p[6];
  double h = dot(a, sub(p, ce));
  V3 cn = sub(sub(p, scale(h, a)), ce);
  bool okr = fabs(sub(norm(cn), R)) < eps;
  V3 u = normalize(cn);
  if (!c.outwards) u = neg(u);
  return okr && (dot(u, n) > thr);
}

__device__ inline bool compat_cone(const rsc_cand& c, ConeTrig tr, V3 p, V3 n, double eps, double thr) {
  V3 apex = {c.p[0], c.p[1], c.p[2]};
  V3 axis = {c.p[3], c.p[4], c.p[5]};
  V3 tp = sub(apex, p);
  V3 tpn = normalize(tp);
  V3 rot = normalize(cross(axis, tpn));
  V3 cn = normalize(cross(axis, rot));
  V3 nv = normalize(rot);
  double v[3] = {nv.x, nv.y, nv.z};
  double R[3][3];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      double o = mul(v[i], v[j]);
      double e = (i == j) ? 1.0 : 0.0;
      R[i][j] = add(o, mul(tr.ct, sub(e, o)));
    }
  R[0][1] = sub(R[0][1], mul(tr.st, v[2]));
  R[0][2] = add(R[0][2], mul(tr.st, v[1]));
  R[1][0] = add(R[1][0], mul(tr.st, v[2]));
  R[1][2] = sub(R[1][2], mul(tr.st, v[0]));
  R[2][0] = sub(R[2][0], mul(tr.st, v[1]));
  R[2][1] = add(R[2][1], mul(tr.st, v[0]));
  V3 rv;
  rv.x = add(add(mul(R[0][0], cn.x), mul(R[0][1], cn.y)), mul(R[0][2], cn.z));
  rv.y = add(add(mul(R[1][0], cn.x), mul(R[1][1], cn.y)), mul(R[1][2], cn.z));
  rv.z = add(add(mul(R[2][0], cn.x), mul(R[2][1], cn.y)), mul(R[2][2], cn.z));
  V3 cur = normalize(rv);
  double dist = dot(neg(cur), neg(tp));
  V3 nr = c.outwards ? cur : neg(cur);
  return (dot(nr, n) > thr) && (fabs(dist) < eps);
}

__device__ inline bool compat(const rsc_cand& c, ConeTrig tr, const Thresh& th, V3 p, V3 n) {
  switch (c.type) {
    case RSC_PLANE:
      return compat_plane(c, p, n, th.eps_d[RSC_PLANE], th.cosa_d[RSC_PLANE]);
    case RSC_SPHERE:
      return compat_sphere(c, p, n, th.eps_d[RSC_SPHERE], th.cosa_d[RSC_SPHERE]);
    case RSC_CYLINDER:
      return compat_cylinder(c, p, n, th.eps_d[RSC_CYLINDER], th.cosa_d[RSC_CYLINDER]);
    case RSC_CONE:
      return compat_cone(c, tr, p, n, th.eps_d[RSC_CONE], th.cosa_d[RSC_CONE]);
    default:
      return false;
  }
}

}  // namespace ex
}  // namespace rsc
