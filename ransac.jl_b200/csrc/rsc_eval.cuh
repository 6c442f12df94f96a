// rsc_eval.cuh -- FP32 evaluation of one (candidate, point) pair against a compiled candidate
// record, and the record compiler (FP64 parameters -> FP32 record with folded constants).
//
// eval<T>() returns the MARGIN m = max(|dist| - eps, cos(alpha)*rho - rho*(n_shape . n_point)):
// the pair is compatible iff m < 0.  |m| <= band (a bound on the FP32 rounding error, record field
// kBandField) marks the pair ambiguous; those are re-evaluated in FP64 (rsc_exact.cuh).
//
// Closed forms used (they equal the reference's compatibles* up to rounding; SURVEY.md 8a15-a21):
//   plane    dist = o.p - o.q (o = normalize(normal));   angle: normal . n > cos(alpha)
//   sphere   v = p - c, r = |v|: | r - R | < eps;        +-(v . n) > cos(alpha) r
//   cylinder w = v - a (a.v), rho = |w|: |rho - R| < eps; +-(w . n) > cos(alpha) rho
//   cone     h = a.v, w = v - a h, rho = |w|, (c,s) = cos/sin(opang/2):
//            dist = h s - rho c;   +-(c (w.n) - s rho (a.n)) > cos(alpha) rho
// The outwards sign is folded into the record (sg = +-1 multiplies v), so a warp never branches.
//
// Operation count (FP32-pipe instructions per evaluation: plane 7, sphere 12, cylinder 18, cone 23):
//   * sphere/cylinder: d = r - R comes out of ONE fma(vv, rsqrt(vv), -R); the angle term re-uses it,
//     cos(alpha) r - s = cos(alpha) d - (s - cos(alpha) R), with -cos(alpha) R folded into the record
//     as the start value of the s chain;
//   * cone: both tests are divided by c = cos(opang/2) > 0 (sign-preserving):
//     dist/c = h tan - rho,   margin/c = rho (cos(alpha)/c + tan (a.n)) - w.n,
//     so the record carries tan, eps/c and cos(alpha)/c and the margin (and its guard band) are in
//     units of 1/c.  Cones wider than 120 degrees (c < 1/2; fits on near-planar patches produce them)
//     form their own column type kConeWide, scaled by s = sin(opang/2) instead (24 ops):
//     dist/s = h - rho cot,   margin/s = rho (cos(alpha)/s + a.n) - cot (w.n);
//     only opening angles beyond ~352.8 deg (s < 1/16) fall back to an infinite band = all-FP64.
#pragma once
#include "rsc_common.cuh"

namespace rsc {

// error-bound multipliers (units of 2^-24 * magnitude), calibrated in tests/test_guard_band.py
__host__ __device__ constexpr float kappa(int type) {
  return type == RSC_PLANE ? 8.f : type == RSC_SPHERE ? 16.f : type == RSC_CYLINDER ? 16.f : 20.f;  // both cone forms: 20
}

// Input-rounding term of an exact cloud (DESIGN.md section 4): the float32 point is the rounding of the caller's
// float64 one, |dp| <= (u/2) pmax and |dn| <= (u/2) nmax, which moves the margin the kernel evaluates by at most
// (u/2) L (plane), (3/2) u L (sphere, cylinder) or (1 + 1/sqrt 2) u L (both cone forms).  Like kappa, kappa_in
// is twice that bound in units of u L.
__host__ __device__ constexpr float kappa_in(int type) {
  return type == RSC_PLANE ? 1.f : type == RSC_SPHERE ? 3.f : type == RSC_CYLINDER ? 3.f : 4.f;
}

// column type of a candidate: its public type, except cones wider than 120 degrees (cos(opang/2) < 1/2)
__host__ __device__ inline int col_type(const rsc_cand& c) {
  if (c.type != RSC_CONE) return c.type;
  return cos(0.5 * c.p[6]) >= 0.5 ? RSC_CONE : kConeWide;  // NaN opang -> kConeWide (its record is "far")
}

__device__ __forceinline__ float fmax_nan(float a, float b) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
// one MUFU.RSQ; denormal inputs flush to zero (-> inf -> NaN margin -> FP64 path)
__device__ __forceinline__ float rsqrt_fast(float a) {
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a));
  return r;
}
__device__ __forceinline__ float fmin_nan(float a, float b) {
  float r;
  asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}

// Number of record fields each type really uses (the rest of the 12 is padding).
template <int T>
struct RecN;
template <>
struct RecN<RSC_PLANE> {
  static constexpr int n = 7;
};
template <>
struct RecN<RSC_SPHERE> {
  static constexpr int n = 6;
};
template <>
struct RecN<RSC_CYLINDER> {
  static constexpr int n = 9;
};
template <>
struct RecN<RSC_CONE> {
  static constexpr int n = 10;
};
template <>
struct RecN<kConeWide> {
  static constexpr int n = 11;
};

// r: the used fields of the record (registers).  p = (x,y,z), n = (nx,ny,nz).
template <int T>
__device__ __forceinline__ float eval(const float* r, float px, float py, float pz, float nx, float ny,
                                      float nz, float eps, float cosa) {
  if constexpr (T == RSC_PLANE) {
    // r0..2 = o, r3 = -o.q, r4..6 = -normal
    float d = fmaf(r[0], px, fmaf(r[1], py, fmaf(r[2], pz, r[3])));
    float e = fabsf(d) - eps;
    float nt = fmaf(r[4], nx, fmaf(r[5], ny, fmaf(r[6], nz, cosa)));
    return fmax_nan(e, nt);
  } else if constexpr (T == RSC_SPHERE) {
    // r0 = sg, r1..3 = -sg*center, r4 = -R, r5 = -cos(alpha)*R
    float vx = fmaf(r[0], px, r[1]), vy = fmaf(r[0], py, r[2]), vz = fmaf(r[0], pz, r[3]);
    float vv = fmaf(vx, vx, fmaf(vy, vy, vz * vz));
    float d = fmaf(vv, rsqrt_fast(vv), r[4]);
    float e = fabsf(d) - eps;
    float s = fmaf(vx, nx, fmaf(vy, ny, fmaf(vz, nz, r[5])));
    float nt = fmaf(cosa, d, -s);
    return fmax_nan(e, nt);
  } else if constexpr (T == RSC_CYLINDER) {
    // r0 = sg, r1..3 = -sg*center, r4..6 = axis, r7 = -R, r8 = -cos(alpha)*R
    float vx = fmaf(r[0], px, r[1]), vy = fmaf(r[0], py, r[2]), vz = fmaf(r[0], pz, r[3]);
    float h = fmaf(r[4], vx, fmaf(r[5], vy, r[6] * vz));
    float wx = fmaf(-r[4], h, vx), wy = fmaf(-r[5], h, vy), wz = fmaf(-r[6], h, vz);
    float ww = fmaf(wx, wx, fmaf(wy, wy, wz * wz));
    float d = fmaf(ww, rsqrt_fast(ww), r[7]);
    float e = fabsf(d) - eps;
    float wn = fmaf(wx, nx, fmaf(wy, ny, fmaf(wz, nz, r[8])));
    float nt = fmaf(cosa, d, -wn);
    return fmax_nan(e, nt);
  } else if constexpr (T == kConeWide) {
    // r0 = sg, r1..3 = -sg*apex, r4..6 = axis, r7 = sg*cot(opang/2), r8 = -eps/s, r9 = cos(alpha)/s, r10 = cot
    float vx = fmaf(r[0], px, r[1]), vy = fmaf(r[0], py, r[2]), vz = fmaf(r[0], pz, r[3]);
    float h = fmaf(r[4], vx, fmaf(r[5], vy, r[6] * vz));
    float wx = fmaf(-r[4], h, vx), wy = fmaf(-r[5], h, vy), wz = fmaf(-r[6], h, vz);
    float ww = fmaf(wx, wx, fmaf(wy, wy, wz * wz));
    float rho = ww * rsqrt_fast(ww);
    float d = fmaf(-rho, r[7], h);
    float e = fabsf(d) + r[8];
    float wn = fmaf(wx, nx, fmaf(wy, ny, wz * nz));
    float an = fmaf(r[4], nx, fmaf(r[5], ny, r[6] * nz));
    float t1 = fmaf(r[0], an, r[9]);
    float cw = r[10] * wn;
    float nt = fmaf(rho, t1, -cw);
    return fmax_nan(e, nt);
  } else {
    // r0 = sg, r1..3 = -sg*apex, r4..6 = axis, r7 = sg*tan(opang/2), r8 = -eps/c, r9 = cos(alpha)/c
    float vx = fmaf(r[0], px, r[1]), vy = fmaf(r[0], py, r[2]), vz = fmaf(r[0], pz, r[3]);
    float h = fmaf(r[4], vx, fmaf(r[5], vy, r[6] * vz));
    float wx = fmaf(-r[4], h, vx), wy = fmaf(-r[5], h, vy), wz = fmaf(-r[6], h, vz);
    float ww = fmaf(wx, wx, fmaf(wy, wy, wz * wz));
    float rho = ww * rsqrt_fast(ww);
    float d = fmaf(h, r[7], -rho);
    float e = fabsf(d) + r[8];
    float wn = fmaf(wx, nx, fmaf(wy, ny, wz * nz));
    float an = fmaf(r[4], nx, fmaf(r[5], ny, r[6] * nz));
    float t1 = fmaf(r[7], an, r[9]);
    float nt = fmaf(rho, t1, -wn);
    return fmax_nan(e, nt);
  }
}

// ---------------------------------------------------------------------------------------------
// Packed evaluation: TWO candidates per call on sm_100's 2-wide FP32 instructions (FFMA2 / FMUL2 /
// FADD2).  A scalar FFMA issues at half the FP32 lane rate on this chip (measured: tools/
// fp32_peak.cu), so the tiled kernel keeps its candidates as float2 pairs; the point's scalars are
// broadcast operands (`R.F32` in SASS) and |x| / -x are operand modifiers, i.e. free.  Each half
// performs exactly the scalar sequence of eval<T>() (same roundings, same guard band).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 bc2(float s) { return make_float2(s, s); }
__device__ __forceinline__ float2 neg2(float2 a) { return make_float2(-a.x, -a.y); }
__device__ __forceinline__ float2 abs2(float2 a) { return make_float2(fabsf(a.x), fabsf(a.y)); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 rsqrt2(float2 a) { return make_float2(rsqrt_fast(a.x), rsqrt_fast(a.y)); }
__device__ __forceinline__ float2 max2_nan(float2 a, float2 b) {
  return make_float2(fmax_nan(a.x, b.x), fmax_nan(a.y, b.y));
}

// the two terms of the margin: returns the distance term e, stores the angle term nt
template <int T>
__device__ __forceinline__ float2 eval2_terms(const float2* r, float px, float py, float pz, float nx, float ny,
                                              float nz, float eps, float cosa, float2* nt_out) {
  const float2 X = bc2(px), Y = bc2(py), Z = bc2(pz), NX = bc2(nx), NY = bc2(ny), NZ = bc2(nz);
  if constexpr (T == RSC_PLANE) {
    const float2 d = fma2(r[0], X, fma2(r[1], Y, fma2(r[2], Z, r[3])));
    const float2 e = add2(abs2(d), bc2(-eps));
    const float2 nt = fma2(r[4], NX, fma2(r[5], NY, fma2(r[6], NZ, bc2(cosa))));
    *nt_out = nt;
    return e;
  } else if constexpr (T == RSC_SPHERE) {
    const float2 vx = fma2(r[0], X, r[1]), vy = fma2(r[0], Y, r[2]), vz = fma2(r[0], Z, r[3]);
    const float2 vv = fma2(vx, vx, fma2(vy, vy, mul2(vz, vz)));
    const float2 d = fma2(vv, rsqrt2(vv), r[4]);
    const float2 e = add2(abs2(d), bc2(-eps));
    const float2 s = fma2(vx, NX, fma2(vy, NY, fma2(vz, NZ, r[5])));
    const float2 nt = fma2(bc2(cosa), d, neg2(s));
    *nt_out = nt;
    return e;
  } else if constexpr (T == RSC_CYLINDER) {
    const float2 vx = fma2(r[0], X, r[1]), vy = fma2(r[0], Y, r[2]), vz = fma2(r[0], Z, r[3]);
    const float2 h = fma2(r[4], vx, fma2(r[5], vy, mul2(r[6], vz)));
    const float2 wx = fma2(neg2(r[4]), h, vx), wy = fma2(neg2(r[5]), h, vy), wz = fma2(neg2(r[6]), h, vz);
    const float2 ww = fma2(wx, wx, fma2(wy, wy, mul2(wz, wz)));
    const float2 d = fma2(ww, rsqrt2(ww), r[7]);
    const float2 e = add2(abs2(d), bc2(-eps));
    const float2 wn = fma2(wx, NX, fma2(wy, NY, fma2(wz, NZ, r[8])));
    const float2 nt = fma2(bc2(cosa), d, neg2(wn));
    *nt_out = nt;
    return e;
  } else if constexpr (T == kConeWide) {
    const float2 vx = fma2(r[0], X, r[1]), vy = fma2(r[0], Y, r[2]), vz = fma2(r[0], Z, r[3]);
    const float2 h = fma2(r[4], vx, fma2(r[5], vy, mul2(r[6], vz)));
    const float2 wx = fma2(neg2(r[4]), h, vx), wy = fma2(neg2(r[5]), h, vy), wz = fma2(neg2(r[6]), h, vz);
    const float2 ww = fma2(wx, wx, fma2(wy, wy, mul2(wz, wz)));
    const float2 rho = mul2(ww, rsqrt2(ww));
    const float2 d = fma2(neg2(rho), r[7], h);
    const float2 e = add2(abs2(d), r[8]);
    const float2 wn = fma2(wx, NX, fma2(wy, NY, mul2(wz, NZ)));
    const float2 an = fma2(r[4], NX, fma2(r[5], NY, mul2(r[6], NZ)));
    const float2 t1 = fma2(r[0], an, r[9]);
    const float2 cw = mul2(r[10], wn);
    const float2 nt = fma2(rho, t1, neg2(cw));
    *nt_out = nt;
    return e;
  } else {
    const float2 vx = fma2(r[0], X, r[1]), vy = fma2(r[0], Y, r[2]), vz = fma2(r[0], Z, r[3]);
    const float2 h = fma2(r[4], vx, fma2(r[5], vy, mul2(r[6], vz)));
    const float2 wx = fma2(neg2(r[4]), h, vx), wy = fma2(neg2(r[5]), h, vy), wz = fma2(neg2(r[6]), h, vz);
    const float2 ww = fma2(wx, wx, fma2(wy, wy, mul2(wz, wz)));
    const float2 rho = mul2(ww, rsqrt2(ww));
    const float2 d = fma2(h, r[7], neg2(rho));
    const float2 e = add2(abs2(d), r[8]);
    const float2 wn = fma2(wx, NX, fma2(wy, NY, mul2(wz, NZ)));
    const float2 an = fma2(r[4], NX, fma2(r[5], NY, mul2(r[6], NZ)));
    const float2 t1 = fma2(r[7], an, r[9]);
    const float2 nt = fma2(rho, t1, neg2(wn));
    *nt_out = nt;
    return e;
  }
}

// margin of a candidate pair = max(distance term, angle term), NaN-propagating
template <int T>
__device__ __forceinline__ float2 eval2(const float2* r, float px, float py, float pz, float nx, float ny,
                                        float nz, float eps, float cosa) {
  float2 nt;
  const float2 e = eval2_terms<T>(r, px, py, pz, nx, ny, nz, eps, cosa, &nt);
  return max2_nan(e, nt);
}

// Lockstep evaluation of FOUR points against one candidate pair: every formula step is written for the four
// points back to back, so that consecutive packed instructions share their candidate operand (the operand-
// reuse cache then serves it and the instruction reads at most two even and two odd registers: 2 issue
// cycles instead of 3, see tools/sass_model.py).  Same operations, same roundings as eval2<T>().
template <int T>
__device__ __forceinline__ void eval2x4(const float2* r, const float* px, const float* py, const float* pz, const float* nx,
                                        const float* ny, const float* nz, float eps, float cosa, float2* m) {
#define RSC_Q for (int q = 0; q < 4; ++q)
  if constexpr (T == RSC_PLANE) {
    float2 d[4], nt[4];
#pragma unroll
    RSC_Q d[q] = fma2(r[2], bc2(pz[q]), r[3]);
#pragma unroll
    RSC_Q d[q] = fma2(r[1], bc2(py[q]), d[q]);
#pragma unroll
    RSC_Q d[q] = fma2(r[0], bc2(px[q]), d[q]);
#pragma unroll
    RSC_Q nt[q] = fma2(r[6], bc2(nz[q]), bc2(cosa));
#pragma unroll
    RSC_Q nt[q] = fma2(r[5], bc2(ny[q]), nt[q]);
#pragma unroll
    RSC_Q nt[q] = fma2(r[4], bc2(nx[q]), nt[q]);
#pragma unroll
    RSC_Q d[q] = add2(abs2(d[q]), bc2(-eps));
#pragma unroll
    RSC_Q m[q] = max2_nan(d[q], nt[q]);
  } else {
    float2 vx[4], vy[4], vz[4];
#pragma unroll
    RSC_Q vx[q] = fma2(r[0], bc2(px[q]), r[1]);
#pragma unroll
    RSC_Q vy[q] = fma2(r[0], bc2(py[q]), r[2]);
#pragma unroll
    RSC_Q vz[q] = fma2(r[0], bc2(pz[q]), r[3]);
    if constexpr (T == RSC_SPHERE) {
      float2 vv[4], s[4];
#pragma unroll
      RSC_Q vv[q] = mul2(vz[q], vz[q]);
#pragma unroll
      RSC_Q vv[q] = fma2(vy[q], vy[q], vv[q]);
#pragma unroll
      RSC_Q vv[q] = fma2(vx[q], vx[q], vv[q]);
#pragma unroll
      RSC_Q s[q] = fma2(vz[q], bc2(nz[q]), r[5]);
#pragma unroll
      RSC_Q s[q] = fma2(vy[q], bc2(ny[q]), s[q]);
#pragma unroll
      RSC_Q s[q] = fma2(vx[q], bc2(nx[q]), s[q]);
#pragma unroll
      RSC_Q vv[q] = fma2(vv[q], rsqrt2(vv[q]), r[4]);  // d
#pragma unroll
      RSC_Q s[q] = fma2(bc2(cosa), vv[q], neg2(s[q]));  // nt
#pragma unroll
      RSC_Q vv[q] = add2(abs2(vv[q]), bc2(-eps));
#pragma unroll
      RSC_Q m[q] = max2_nan(vv[q], s[q]);
    } else {
      float2 h[4], ww[4];
#pragma unroll
      RSC_Q h[q] = mul2(r[6], vz[q]);
#pragma unroll
      RSC_Q h[q] = fma2(r[5], vy[q], h[q]);
#pragma unroll
      RSC_Q h[q] = fma2(r[4], vx[q], h[q]);
#pragma unroll
      RSC_Q vx[q] = fma2(neg2(r[4]), h[q], vx[q]);  // w
#pragma unroll
      RSC_Q vy[q] = fma2(neg2(r[5]), h[q], vy[q]);
#pragma unroll
      RSC_Q vz[q] = fma2(neg2(r[6]), h[q], vz[q]);
#pragma unroll
      RSC_Q ww[q] = mul2(vz[q], vz[q]);
#pragma unroll
      RSC_Q ww[q] = fma2(vy[q], vy[q], ww[q]);
#pragma unroll
      RSC_Q ww[q] = fma2(vx[q], vx[q], ww[q]);
      if constexpr (T == RSC_CYLINDER) {
        float2 wn[4];
#pragma unroll
        RSC_Q wn[q] = fma2(vz[q], bc2(nz[q]), r[8]);
#pragma unroll
        RSC_Q wn[q] = fma2(vy[q], bc2(ny[q]), wn[q]);
#pragma unroll
        RSC_Q wn[q] = fma2(vx[q], bc2(nx[q]), wn[q]);
#pragma unroll
        RSC_Q ww[q] = fma2(ww[q], rsqrt2(ww[q]), r[7]);  // d
#pragma unroll
        RSC_Q wn[q] = fma2(bc2(cosa), ww[q], neg2(wn[q]));  // nt
#pragma unroll
        RSC_Q ww[q] = add2(abs2(ww[q]), bc2(-eps));
#pragma unroll
        RSC_Q m[q] = max2_nan(ww[q], wn[q]);
      } else {
        float2 wn[4], an[4];
#pragma unroll
        RSC_Q an[q] = mul2(r[6], bc2(nz[q]));
#pragma unroll
        RSC_Q an[q] = fma2(r[5], bc2(ny[q]), an[q]);
#pragma unroll
        RSC_Q an[q] = fma2(r[4], bc2(nx[q]), an[q]);
#pragma unroll
        RSC_Q wn[q] = mul2(vz[q], bc2(nz[q]));
#pragma unroll
        RSC_Q wn[q] = fma2(vy[q], bc2(ny[q]), wn[q]);
#pragma unroll
        RSC_Q wn[q] = fma2(vx[q], bc2(nx[q]), wn[q]);
#pragma unroll
        RSC_Q ww[q] = mul2(ww[q], rsqrt2(ww[q]));  // rho
        if constexpr (T == kConeWide) {
#pragma unroll
          RSC_Q h[q] = fma2(neg2(ww[q]), r[7], h[q]);  // d
#pragma unroll
          RSC_Q an[q] = fma2(r[0], an[q], r[9]);  // t1
#pragma unroll
          RSC_Q wn[q] = mul2(r[10], wn[q]);  // cw
        } else {
#pragma unroll
          RSC_Q h[q] = fma2(h[q], r[7], neg2(ww[q]));  // d
#pragma unroll
          RSC_Q an[q] = fma2(r[7], an[q], r[9]);  // t1
        }
#pragma unroll
        RSC_Q h[q] = add2(abs2(h[q]), r[8]);  // e
#pragma unroll
        RSC_Q an[q] = fma2(ww[q], an[q], neg2(wn[q]));  // nt
#pragma unroll
        RSC_Q m[q] = max2_nan(h[q], an[q]);
      }
    }
  }
#undef RSC_Q
}

// Packed evaluation of TWO POINTS against one candidate (the transposed mapping of rsc_cull.cu: a lane owns
// points, the candidate's record is a warp-uniform scalar operand).  Each half performs exactly the scalar
// sequence of eval<T>() (same roundings, same guard band).  r: the used fields of the record.
template <int T>
__device__ __forceinline__ float2 evalp(const float* r, float2 X, float2 Y, float2 Z, float2 NX, float2 NY, float2 NZ,
                                        float eps, float cosa) {
  if constexpr (T == RSC_PLANE) {
    const float2 d = fma2(bc2(r[0]), X, fma2(bc2(r[1]), Y, fma2(bc2(r[2]), Z, bc2(r[3]))));
    const float2 e = add2(abs2(d), bc2(-eps));
    const float2 nt = fma2(bc2(r[4]), NX, fma2(bc2(r[5]), NY, fma2(bc2(r[6]), NZ, bc2(cosa))));
    return max2_nan(e, nt);
  } else if constexpr (T == RSC_SPHERE) {
    const float2 vx = fma2(bc2(r[0]), X, bc2(r[1])), vy = fma2(bc2(r[0]), Y, bc2(r[2])), vz = fma2(bc2(r[0]), Z, bc2(r[3]));
    const float2 vv = fma2(vx, vx, fma2(vy, vy, mul2(vz, vz)));
    const float2 d = fma2(vv, rsqrt2(vv), bc2(r[4]));
    const float2 e = add2(abs2(d), bc2(-eps));
    const float2 s = fma2(vx, NX, fma2(vy, NY, fma2(vz, NZ, bc2(r[5]))));
    const float2 nt = fma2(bc2(cosa), d, neg2(s));
    return max2_nan(e, nt);
  } else {
    const float2 vx = fma2(bc2(r[0]), X, bc2(r[1])), vy = fma2(bc2(r[0]), Y, bc2(r[2])), vz = fma2(bc2(r[0]), Z, bc2(r[3]));
    const float2 h = fma2(bc2(r[4]), vx, fma2(bc2(r[5]), vy, mul2(bc2(r[6]), vz)));
    const float2 wx = fma2(bc2(-r[4]), h, vx), wy = fma2(bc2(-r[5]), h, vy), wz = fma2(bc2(-r[6]), h, vz);
    const float2 ww = fma2(wx, wx, fma2(wy, wy, mul2(wz, wz)));
    if constexpr (T == RSC_CYLINDER) {
      const float2 d = fma2(ww, rsqrt2(ww), bc2(r[7]));
      const float2 e = add2(abs2(d), bc2(-eps));
      const float2 wn = fma2(wx, NX, fma2(wy, NY, fma2(wz, NZ, bc2(r[8]))));
      const float2 nt = fma2(bc2(cosa), d, neg2(wn));
      return max2_nan(e, nt);
    } else {
      const float2 rho = mul2(ww, rsqrt2(ww));
      const float2 wn = fma2(wx, NX, fma2(wy, NY, mul2(wz, NZ)));
      const float2 an = fma2(bc2(r[4]), NX, fma2(bc2(r[5]), NY, mul2(bc2(r[6]), NZ)));
      if constexpr (T == kConeWide) {
        const float2 d = fma2(neg2(rho), bc2(r[7]), h);
        const float2 e = add2(abs2(d), bc2(r[8]));
        const float2 t1 = fma2(bc2(r[0]), an, bc2(r[9]));
        const float2 cw = mul2(bc2(r[10]), wn);
        const float2 nt = fma2(rho, t1, neg2(cw));
        return max2_nan(e, nt);
      } else {
        const float2 d = fma2(h, bc2(r[7]), neg2(rho));
        const float2 e = add2(abs2(d), bc2(r[8]));
        const float2 t1 = fma2(bc2(r[7]), an, bc2(r[9]));
        const float2 nt = fma2(rho, t1, neg2(wn));
        return max2_nan(e, nt);
      }
    }
  }
}

// runtime-type version for the (rare) slow path; `type` is a COLUMN type (col_type())
__device__ __forceinline__ float eval_any(int type, const float* r, float px, float py, float pz,
                                          float nx, float ny, float nz, float eps, float cosa) {
  switch (type) {
    case RSC_PLANE:
      return eval<RSC_PLANE>(r, px, py, pz, nx, ny, nz, eps, cosa);
    case RSC_SPHERE:
      return eval<RSC_SPHERE>(r, px, py, pz, nx, ny, nz, eps, cosa);
    case RSC_CYLINDER:
      return eval<RSC_CYLINDER>(r, px, py, pz, nx, ny, nz, eps, cosa);
    case kConeWide:
      return eval<kConeWide>(r, px, py, pz, nx, ny, nz, eps, cosa);
    default:
      return eval<RSC_CONE>(r, px, py, pz, nx, ny, nz, eps, cosa);
  }
}

// Compile one candidate (FP64 parameters) into its FP32 record.  pmax/nmax: max |p| and max |n|
// over the cloud, the scale of every intermediate and therefore of the rounding error.
// A candidate with a non-finite parameter can match nothing in the reference (NaN compares
// false); it gets a record that is far from everything so that no NaN reaches the tiled kernel.
// `col` = col_type(c) as decided by the caller (the kernel that evaluates the record must use the same form).
__device__ inline void compile_record(const rsc_cand& c, int col, const Thresh& th, float pmax, float nmax, float* r /*[12]*/) {
  const double u = 5.9604644775390625e-08;  // 2^-24
  for (int i = 0; i < kRecFields; ++i) r[i] = 0.f;
  bool finite = true;
  for (int i = 0; i < 7; ++i) finite = finite && isfinite(c.p[i]);
  double nm = nmax > 1.f ? (double)nmax : 1.0;
  double P = (double)pmax;
  double L;
  switch (c.type) {
    case RSC_PLANE: {
      double mx = c.p[3], my = c.p[4], mz = c.p[5];
      double mn = sqrt(mx * mx + my * my + mz * mz);
      double inv = 1.0 / mn;
      if (!finite || !(mn > 0.0) || !isfinite(inv)) {
        r[3] = 1e30f;  // |dist| = 1e30
        r[kBandField] = 1.f;
        return;
      }
      double ox = mx * inv, oy = my * inv, oz = mz * inv;
      double oq = ox * c.p[0] + oy * c.p[1] + oz * c.p[2];
      r[0] = (float)ox, r[1] = (float)oy, r[2] = (float)oz, r[3] = (float)(-oq);
      r[4] = (float)(-mx), r[5] = (float)(-my), r[6] = (float)(-mz);
      L = (P + fabs(oq) + 1.0) * (mn > 1.0 ? mn : 1.0) * nm;
      break;
    }
    case RSC_SPHERE: {
      double sg = c.outwards ? 1.0 : -1.0;
      if (!finite) {
        r[0] = 1.f, r[1] = 1e15f, r[4] = -1e30f, r[kBandField] = 1.f;
        return;
      }
      r[0] = (float)sg;
      r[1] = (float)(-sg * c.p[0]), r[2] = (float)(-sg * c.p[1]), r[3] = (float)(-sg * c.p[2]);
      r[4] = (float)(-c.p[3]);
      r[5] = (float)(-th.cosa_d[RSC_SPHERE] * c.p[3]);
      double cn = sqrt(c.p[0] * c.p[0] + c.p[1] * c.p[1] + c.p[2] * c.p[2]);
      L = (P + cn + fabs(c.p[3]) + 1.0) * nm;
      break;
    }
    case RSC_CYLINDER: {
      double sg = c.outwards ? 1.0 : -1.0;
      if (!finite) {
        r[0] = 1.f, r[2] = 1e15f, r[4] = 1.f, r[7] = -1e30f, r[kBandField] = 1.f;
        return;
      }
      r[0] = (float)sg;
      r[1] = (float)(-sg * c.p[3]), r[2] = (float)(-sg * c.p[4]), r[3] = (float)(-sg * c.p[5]);
      r[4] = (float)c.p[0], r[5] = (float)c.p[1], r[6] = (float)c.p[2];
      r[7] = (float)(-c.p[6]);
      r[8] = (float)(-th.cosa_d[RSC_CYLINDER] * c.p[6]);
      double cn = sqrt(c.p[3] * c.p[3] + c.p[4] * c.p[4] + c.p[5] * c.p[5]);
      double a2 = c.p[0] * c.p[0] + c.p[1] * c.p[1] + c.p[2] * c.p[2];
      L = (P + cn + fabs(c.p[6]) + 1.0) * (a2 > 1.0 ? a2 : 1.0) * nm;
      break;
    }
    default: {
      // project2cone (cone.jl:68-85) only uses the DIRECTION of the axis (every cross product with
      // it is normalised), so the closed form works on the unit axis; a zero axis matches nothing.
      double sg = c.outwards ? 1.0 : -1.0;
      const double an = sqrt(c.p[3] * c.p[3] + c.p[4] * c.p[4] + c.p[5] * c.p[5]);
      const double ia = 1.0 / an;
      const double ch = cos(0.5 * c.p[6]), sh = sin(0.5 * c.p[6]);
      const bool wide = (col == kConeWide);
      const bool needle = wide && !(sh >= 1.0 / 16.0);  // opening angle beyond ~352.8 deg (or NaN): FP64 decides
      if (!finite || !(an > 0.0) || !isfinite(ia) || needle) {
        // far from everything; a finite "needle" additionally gets an infinite band (every pair -> FP64)
        r[0] = 1.f, r[2] = 1e15f, r[4] = 1.f, r[7] = 0.f, r[8] = 0.f, r[9] = 1.f, r[10] = 0.f;
        r[kBandField] = (finite && an > 0.0 && isfinite(ia)) ? __int_as_float(0x7f800000) : 1.f;
        return;
      }
      const double sc = wide ? 1.0 / sh : 1.0 / ch;  // the margin is in units of 1/c (1/s for wide cones)
      r[0] = (float)sg;
      r[1] = (float)(-sg * c.p[0]), r[2] = (float)(-sg * c.p[1]), r[3] = (float)(-sg * c.p[2]);
      r[4] = (float)(c.p[3] * ia), r[5] = (float)(c.p[4] * ia), r[6] = (float)(c.p[5] * ia);
      r[7] = (float)(wide ? sg * ch * sc : sg * sh * sc);
      r[8] = (float)(-th.eps_d[RSC_CONE] * sc);
      r[9] = (float)(th.cosa_d[RSC_CONE] * sc);
      r[10] = (float)(wide ? ch * sc : 0.0);
      double cn = sqrt(c.p[0] * c.p[0] + c.p[1] * c.p[1] + c.p[2] * c.p[2]);
      L = (P + cn + 1.0) * nm * sc;
      break;
    }
  }
  double b = (double)(th.exact_in ? kappa(c.type) + kappa_in(c.type) : kappa(c.type)) * u * L;
  r[kBandField] = (float)(b * 1.0000002);  // round the band up, never down
}

}  // namespace rsc
