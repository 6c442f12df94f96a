// rsc_lsq.cu -- least-squares refit of a candidate before its extraction (extension, SURVEY 8(f)-4).
//
// The reference's refit keeps the candidate unchanged ("In our implementation least-square fitting is
// not used", docs/src/ransac.md:163-169; plane.jl:137-143 etc.); the paper refits it to all compatible
// points within 3 eps first.  Definition (shared with oracle/ransac_oracle.py::lsq_refine):
//   1. the point set is selected ONCE with the candidate: compatibles* with eps scaled by `band`, enabled
//      points only -- the K4 mask kernel, so the selection is the exact float64 one;
//   2. planes get the total-least-squares plane of the set (centroid + smallest-eigenvalue direction of
//      the scatter matrix); spheres, cylinders and cones a Levenberg-Marquardt minimisation of the sum
//      of squared point-to-surface distances.
// Device work per pass: one streaming kernel over the selected points that accumulates the normal
// equations J^T J (28), J^T r (7) and r^T r in float64 -- warp per 32-point mask word (zero words are
// skipped, loads are coalesced), registers -> shuffles -> one partial per CTA -> a fixed-order final sum,
// so the result does not depend on scheduling (HBM bound: N/8 B of mask words + 12 B per selected point).
// The 7x7 solve, the damping schedule and the 3x3 Jacobi run on the host in float64.
#include <math.h>
#include <string.h>

#include "rsc_common.cuh"

namespace rsc {

constexpr int kLsqPar = 7;
constexpr int kLsqAcc = kLsqPar * (kLsqPar + 1) / 2 + kLsqPar + 1;  // 36: upper triangle, gradient, cost
constexpr int kLsqThreads = 256;

struct LsqX {
  double x[kLsqPar];
  double sn, cs;  // sin/cos of the cone's half opening angle (host libm)
  int kind;
};

// residual r and Jacobian J[7] (unused entries zero) of the signed distance of point p
__device__ __forceinline__ bool lsq_point(const LsqX& q, double px, double py, double pz, double& r, double (&J)[kLsqPar]) {
#pragma unroll
  for (int i = 0; i < kLsqPar; ++i) J[i] = 0.0;
  if (q.kind == RSC_PLANE) {  // moments about the old point: A = sum v v^T, g = sum v, cost = n
    J[0] = px - q.x[0], J[1] = py - q.x[1], J[2] = pz - q.x[2];
    r = 1.0;
  } else if (q.kind == RSC_SPHERE) {
    const double vx = px - q.x[0], vy = py - q.x[1], vz = pz - q.x[2];
    const double rho = sqrt(vx * vx + vy * vy + vz * vz);
    J[0] = -vx / rho, J[1] = -vy / rho, J[2] = -vz / rho, J[3] = -1.0;
    r = rho - q.x[3];
  } else if (q.kind == RSC_CYLINDER) {
    const double ax = q.x[0], ay = q.x[1], az = q.x[2];
    const double vx = px - q.x[3], vy = py - q.x[4], vz = pz - q.x[5];
    const double h = vx * ax + vy * ay + vz * az;
    const double wx = vx - h * ax, wy = vy - h * ay, wz = vz - h * az;
    const double rho = sqrt(wx * wx + wy * wy + wz * wz);
    const double ux = wx / rho, uy = wy / rho, uz = wz / rho;
    J[0] = -h * ux, J[1] = -h * uy, J[2] = -h * uz;
    J[3] = -ux, J[4] = -uy, J[5] = -uz;
    J[6] = -1.0;
    r = rho - q.x[6];
  } else {
    const double ax = q.x[3], ay = q.x[4], az = q.x[5];
    const double vx = px - q.x[0], vy = py - q.x[1], vz = pz - q.x[2];
    const double h = vx * ax + vy * ay + vz * az;
    const double wx = vx - h * ax, wy = vy - h * ay, wz = vz - h * az;
    const double rho = sqrt(wx * wx + wy * wy + wz * wz);
    const double ux = wx / rho, uy = wy / rho, uz = wz / rho;
    const double dx = q.sn * ax - q.cs * ux, dy = q.sn * ay - q.cs * uy, dz = q.sn * az - q.cs * uz;  // d r / d v
    J[0] = -dx, J[1] = -dy, J[2] = -dz;
    J[3] = q.sn * vx + q.cs * h * ux, J[4] = q.sn * vy + q.cs * h * uy, J[5] = q.sn * vz + q.cs * h * uz;
    J[6] = h * q.cs + rho * q.sn;
    r = h * q.sn - rho * q.cs;
  }
  bool ok = isfinite(r);
#pragma unroll
  for (int i = 0; i < kLsqPar; ++i) ok = ok && isfinite(J[i]);
  return ok;  // points on the axis / at the centre are left out (like NaN comparisons in compatibles*)
}

__global__ void __launch_bounds__(kLsqThreads) lsq_accumulate_kernel(PointSet ps, const uint32_t* __restrict__ sel, LsqX q,
                                                                     double* __restrict__ partials /*[grid][36]*/) {
  __shared__ double sm[kLsqThreads / 32][kLsqAcc];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t words = ps.n_pad / 32;
  const int64_t nwarps = (int64_t)gridDim.x * (kLsqThreads / 32);
  double acc[kLsqAcc];
#pragma unroll
  for (int i = 0; i < kLsqAcc; ++i) acc[i] = 0.0;
  for (int64_t w = (int64_t)blockIdx.x * (kLsqThreads / 32) + warp; w < words; w += nwarps) {
    const uint32_t bits = sel[w];  // same address in every lane: one broadcast load
    if (bits == 0) continue;
    if (!((bits >> lane) & 1u)) continue;
    const int64_t j = w * 32 + lane;
    double r, J[kLsqPar];
    if (!lsq_point(q, (double)ps.x[j], (double)ps.y[j], (double)ps.z[j], r, J)) continue;
    int k = 0;
#pragma unroll
    for (int a = 0; a < kLsqPar; ++a)
#pragma unroll
      for (int b = a; b < kLsqPar; ++b) acc[k++] += J[a] * J[b];
#pragma unroll
    for (int a = 0; a < kLsqPar; ++a) acc[k++] += J[a] * r;
    acc[k] += r * r;
  }
#pragma unroll
  for (int i = 0; i < kLsqAcc; ++i) {
    double v = acc[i];
#pragma unroll
    for (int d = 16; d; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
    if (lane == 0) sm[warp][i] = v;
  }
  __syncthreads();
  if (threadIdx.x < kLsqAcc) {
    double v = 0.0;
    for (int wi = 0; wi < kLsqThreads / 32; ++wi) v += sm[wi][threadIdx.x];
    partials[(size_t)blockIdx.x * kLsqAcc + threadIdx.x] = v;
  }
}

__global__ void lsq_final_kernel(const double* __restrict__ partials, int nblocks, double* __restrict__ out) {
  if (threadIdx.x >= kLsqAcc) return;
  double v = 0.0;
  for (int b = 0; b < nblocks; ++b) v += partials[(size_t)b * kLsqAcc + threadIdx.x];
  out[threadIdx.x] = v;
}

// ---- host side of the minimisation (mirrors oracle/ransac_oracle.py::lsq_*) ------------------------
static int lsq_npar(int kind) { return kind == RSC_PLANE ? 3 : kind == RSC_SPHERE ? 4 : 7; }

static void lsq_pack(const rsc_cand& c, double* x) {
  for (int i = 0; i < kLsqPar; ++i) x[i] = 0.0;
  if (c.type == RSC_PLANE)
    for (int i = 0; i < 6; ++i) x[i] = c.p[i];
  else if (c.type == RSC_SPHERE)
    for (int i = 0; i < 4; ++i) x[i] = c.p[i];
  else {
    for (int i = 0; i < 7; ++i) x[i] = c.p[i];
    if (c.type == RSC_CONE) x[6] = c.p[6] / 2;  // half opening angle
  }
}

static void lsq_normalise(int kind, double* x) {
  if (kind == RSC_CYLINDER) {
    const double n = sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]);
    const double a[3] = {x[0] / n, x[1] / n, x[2] / n};
    const double d = a[0] * x[3] + a[1] * x[4] + a[2] * x[5];
    for (int i = 0; i < 3; ++i) x[i] = a[i], x[3 + i] = x[3 + i] - a[i] * d;
  } else if (kind == RSC_CONE) {
    const double n = sqrt(x[3] * x[3] + x[4] * x[4] + x[5] * x[5]);
    for (int i = 3; i < 6; ++i) x[i] = x[i] / n;
  }
}

// A x = b, A symmetric positive definite (n <= 7); false if a pivot is not positive
static bool lsq_cholesky_solve(const double (*A)[kLsqPar], const double* b, int n, double* xs) {
  double L[kLsqPar][kLsqPar] = {{0}};
  for (int j = 0; j < n; ++j) {
    double d = A[j][j];
    for (int k = 0; k < j; ++k) d -= L[j][k] * L[j][k];
    if (!(d > 0) || !isfinite(d)) return false;
    L[j][j] = sqrt(d);
    for (int i = j + 1; i < n; ++i) {
      double s = A[i][j];
      for (int k = 0; k < j; ++k) s -= L[i][k] * L[j][k];
      L[i][j] = s / L[j][j];
    }
  }
  double y[kLsqPar];
  for (int i = 0; i < n; ++i) {
    double s = b[i];
    for (int k = 0; k < i; ++k) s -= L[i][k] * y[k];
    y[i] = s / L[i][i];
  }
  for (int i = n - 1; i >= 0; --i) {
    double s = y[i];
    for (int k = i + 1; k < n; ++k) s -= L[k][i] * xs[k];
    xs[i] = s / L[i][i];
  }
  return true;
}

// eigenvector of the smallest eigenvalue of a symmetric 3x3 matrix (cyclic Jacobi, fixed sweep order)
static void lsq_smallest_eigvec3(const double M[3][3], double* out) {
  double A[3][3], V[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  memcpy(A, M, sizeof(A));
  static const int P[3] = {0, 0, 1}, Q[3] = {1, 2, 2};
  for (int sweep = 0; sweep < 30; ++sweep) {
    const double off = fabs(A[0][1]) + fabs(A[0][2]) + fabs(A[1][2]);
    if (off <= 1e-300 || off <= 1e-17 * (fabs(A[0][0]) + fabs(A[1][1]) + fabs(A[2][2]))) break;
    for (int r = 0; r < 3; ++r) {
      const int p = P[r], q = Q[r];
      if (A[p][q] == 0.0) continue;
      const double tau = (A[q][q] - A[p][p]) / (2 * A[p][q]);
      const double t = (tau >= 0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1 + tau * tau));
      const double c = 1 / sqrt(1 + t * t), s = t * c;
      double Jm[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
      Jm[p][p] = Jm[q][q] = c;
      Jm[p][q] = s, Jm[q][p] = -s;
      double T[3][3], B[3][3], W[3][3];
      for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
          T[i][j] = 0;
          for (int k = 0; k < 3; ++k) T[i][j] += Jm[k][i] * A[k][j];  // Jm^T A
        }
      for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
          B[i][j] = 0, W[i][j] = 0;
          for (int k = 0; k < 3; ++k) B[i][j] += T[i][k] * Jm[k][j], W[i][j] += V[i][k] * Jm[k][j];
        }
      memcpy(A, B, sizeof(A));
      memcpy(V, W, sizeof(V));
    }
  }
  int k = 0;
  if (A[1][1] < A[k][k]) k = 1;
  if (A[2][2] < A[k][k]) k = 2;
  for (int i = 0; i < 3; ++i) out[i] = V[i][k];
}

struct LsqSums {
  double A[kLsqPar][kLsqPar];
  double g[kLsqPar];
  double cost;
};

// one pass over the selected points (mask = first words of ctx->idxbuf, left there by refit_mask_enqueue)
static int32_t lsq_pass(rsc_cloud* cloud, int kind, const double* x, cudaStream_t st, LsqSums* out) {
  rsc_ctx* ctx = cloud->ctx;
  LsqX q;
  for (int i = 0; i < kLsqPar; ++i) q.x[i] = x[i];
  q.kind = kind;
  q.sn = kind == RSC_CONE ? sin(x[6]) : 0.0;
  q.cs = kind == RSC_CONE ? cos(x[6]) : 0.0;
  const int grid = ctx->sm_count * 4;
  RSC_CUDA(ctx, ctx->lsqbuf.ensure((size_t)(grid + 1) * kLsqAcc * sizeof(double)));
  double* partials = ctx->lsqbuf.as<double>();
  double* total = partials + (size_t)grid * kLsqAcc;
  lsq_accumulate_kernel<<<grid, kLsqThreads, 0, st>>>(view_cloud(cloud), ctx->idxbuf.as<uint32_t>(), q, partials);
  RSC_CUDA(ctx, cudaGetLastError());
  lsq_final_kernel<<<1, 64, 0, st>>>(partials, grid, total);
  RSC_CUDA(ctx, cudaGetLastError());
  double h[kLsqAcc];
  RSC_CUDA(ctx, cudaMemcpyAsync(h, total, sizeof(h), cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaStreamSynchronize(st));
  int k = 0;
  for (int a = 0; a < kLsqPar; ++a)
    for (int b = a; b < kLsqPar; ++b) out->A[a][b] = out->A[b][a] = h[k++];
  for (int a = 0; a < kLsqPar; ++a) out->g[a] = h[k++];
  out->cost = h[k];
  return RSC_OK;
}

// refine `cand` in place; *n_used = selected points, *rms = root mean square distance (NaN if unchanged)
int32_t lsq_refine(rsc_cloud* cloud, const rsc_params* params, double band, rsc_cand* cand, int64_t* n_used, double* rms,
                   cudaStream_t st) {
  rsc_ctx* ctx = cloud->ctx;
  const int kind = cand->type;
  const int npar = lsq_npar(kind);
  if (n_used) *n_used = 0;
  if (rms) *rms = NAN;
  rsc_params p3 = *params;
  p3.eps[kind] = params->eps[kind] * band;
  Thresh th = make_thresh(&p3);
  th.honour_enabled = 0xFu;
  int32_t rc = refit_mask_enqueue(cloud, th, *cand, st);
  if (rc) return rc;
  unsigned long long total = 0;
  RSC_CUDA(ctx, cudaMemcpyAsync(&total, ctx->misc2.p, 8, cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaStreamSynchronize(st));
  if (n_used) *n_used = (int64_t)total;
  if ((int64_t)total < 2 * npar) return RSC_OK;
  double x[kLsqPar];
  lsq_pack(*cand, x);
  LsqSums s;
  if (kind == RSC_PLANE) {
    if ((rc = lsq_pass(cloud, kind, x, st, &s))) return rc;
    const double cnt = s.cost;
    double mean[3], M[3][3], nv[3];
    for (int i = 0; i < 3; ++i) mean[i] = s.g[i] / cnt;
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) M[i][j] = s.A[i][j] - cnt * (mean[i] * mean[j]);
    lsq_smallest_eigvec3(M, nv);
    const double nn = sqrt(nv[0] * nv[0] + nv[1] * nv[1] + nv[2] * nv[2]);
    for (int i = 0; i < 3; ++i) nv[i] /= nn;
    if (nv[0] * x[3] + nv[1] * x[4] + nv[2] * x[5] < 0)
      for (int i = 0; i < 3; ++i) nv[i] = -nv[i];
    double out[6];
    bool fin = true;
    for (int i = 0; i < 3; ++i) out[i] = x[i] + mean[i], out[3 + i] = nv[i];
    for (int i = 0; i < 6; ++i) fin = fin && isfinite(out[i]);
    if (!fin) return RSC_OK;
    double q = 0;
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) q += nv[i] * M[i][j] * nv[j];
    for (int i = 0; i < 6; ++i) cand->p[i] = out[i];
    if (rms) *rms = sqrt((q > 0 ? q : 0.0) / cnt);
    return RSC_OK;
  }
  lsq_normalise(kind, x);
  if ((rc = lsq_pass(cloud, kind, x, st, &s))) return rc;
  double lam = 1e-3;
  for (int it = 0; it < 12; ++it) {
    double D[kLsqPar][kLsqPar], mg[kLsqPar], d[kLsqPar] = {0};
    double tr = 0;
    for (int i = 0; i < npar; ++i) tr += s.A[i][i];
    for (int i = 0; i < npar; ++i) {
      for (int j = 0; j < npar; ++j) D[i][j] = s.A[i][j];
      D[i][i] = s.A[i][i] + lam * s.A[i][i] + 1e-12 * tr / npar;
      mg[i] = -s.g[i];
    }
    bool ok = lsq_cholesky_solve(D, mg, npar, d);
    for (int i = 0; i < npar && ok; ++i) ok = isfinite(d[i]);
    if (!ok) {
      lam *= 10;
      continue;
    }
    double x1[kLsqPar] = {0};
    for (int i = 0; i < npar; ++i) x1[i] = x[i] + d[i];
    lsq_normalise(kind, x1);
    LsqSums s1;
    if ((rc = lsq_pass(cloud, kind, x1, st, &s1))) return rc;
    if (isfinite(s1.cost) && s1.cost <= s.cost) {
      const double rel = (s.cost - s1.cost) / (s.cost > 1e-300 ? s.cost : 1e-300);
      memcpy(x, x1, sizeof(x));
      s = s1;
      lam = lam / 10 > 1e-9 ? lam / 10 : 1e-9;
      if (rel < 1e-12) break;
    } else {
      lam *= 10;
    }
  }
  for (int i = 0; i < npar; ++i)
    if (!isfinite(x[i])) return RSC_OK;
  if (kind == RSC_SPHERE)
    for (int i = 0; i < 4; ++i) cand->p[i] = x[i];
  else {
    for (int i = 0; i < 7; ++i) cand->p[i] = x[i];
    if (kind == RSC_CONE) cand->p[6] = 2 * x[6];
  }
  if (rms) *rms = sqrt(s.cost / (double)total);
  return RSC_OK;
}

}  // namespace rsc

using namespace rsc;

extern "C" int32_t rsc_refit_lsq(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cand, double band, rsc_cand* out,
                                 int64_t* n_used, double* rms) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (!params || !cand || !out) return fail(ctx, RSC_E_ARG, "refit_lsq: null params/candidate/out");
  if (cand->type < 0 || cand->type >= RSC_NTYPES) return fail(ctx, RSC_E_ARG, "refit_lsq: unknown shape type");
  if (!(band > 0) || !isfinite(band)) return fail(ctx, RSC_E_ARG, "refit_lsq: band must be positive");
  if (cloud->exact()) return fail(ctx, RSC_E_STATE, "refit_lsq: the least-squares refit does not support exact clouds yet");
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if (int32_t rc = cloud_ready(cloud)) return rc;
  *out = *cand;
  return lsq_refine(cloud, params, band, out, n_used, rms, ctx->stream);
}
