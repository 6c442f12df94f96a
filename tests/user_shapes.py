"""Two user-defined shapes with device source (include/rsc.h, rsc_user_compatible) and their NumPy twins.

Each twin evaluates the same float64 operations in the same order as the CUDA source, on the cloud's float32
coordinates widened to double.  The source is compiled with --fmad=false and IEEE division / square root, so
the twin's decisions are the device's bit for bit.

  slab   p = (z0),  k = (eps, cos alpha):  |z - z0| < eps and |nz| > cos alpha
  torus  p = (center[3], r * axis[3], R),  k = (eps, cos alpha):  the tube radius r rides in the length of the
         axis (a torus has 8 parameters, rsc_cand holds 7); tube distance |sqrt((rho - R)^2 + h^2) - r| < eps with
         h = a.v, w = v - h a, rho = |w|, and the normal within alpha of the tube normal (unoriented)
"""
import math
from dataclasses import dataclass

import numpy as np

SLAB_SRC = r"""
// p = (z0); k = (eps, cos alpha)
__device__ bool rsc_user_compatible(const double p[7], int outwards, const double k[8],
                                    double x, double y, double z, double nx, double ny, double nz) {
  return fabs(z - p[0]) < k[0] && fabs(nz) > k[1];
}
"""

TORUS_SRC = r"""
// p = (center[3], r * axis[3], R); k = (eps, cos alpha)
__device__ bool rsc_user_compatible(const double p[7], int outwards, const double k[8],
                                    double x, double y, double z, double nx, double ny, double nz) {
  const double r = sqrt(p[3] * p[3] + p[4] * p[4] + p[5] * p[5]);
  const double ax = p[3] / r, ay = p[4] / r, az = p[5] / r;
  const double vx = x - p[0], vy = y - p[1], vz = z - p[2];
  const double h = ax * vx + ay * vy + az * vz;
  const double wx = vx - h * ax, wy = vy - h * ay, wz = vz - h * az;
  const double rho = sqrt(wx * wx + wy * wy + wz * wz);
  const double e = rho - p[6];
  const double dt = sqrt(e * e + h * h);
  if (!(fabs(dt - r) < k[0])) return false;
  const double s = e / rho;  // tube normal direction: w (rho - R) / rho + h a, of length dt
  const double gx = wx * s + h * ax, gy = wy * s + h * ay, gz = wz * s + h * az;
  const double dot = nx * gx + ny * gy + nz * gz;
  return fabs(dot) > k[1] * dt;
}
"""

BROKEN_SRC = r"""
__device__ bool rsc_user_compatible(const double p[7], int outwards, const double k[8],
                                    double x, double y, double z, double nx, double ny, double nz) {
  return fabs(z - p[0]) < k[0] &&& fabs(nz) > k[1];
}
"""


def constants(eps=0.3, alpha=math.radians(5)):
    return [float(eps), math.cos(alpha)]


def slab_twin(p, k, P, N):
    """bool mask of the points P, N ((M, 3) float64) compatible with the slab record p"""
    with np.errstate(invalid="ignore"):
        return (np.abs(P[:, 2] - p[0]) < k[0]) & (np.abs(N[:, 2]) > k[1])


def torus_twin(p, k, P, N):
    p = np.asarray(p, dtype=np.float64)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        r = np.sqrt(p[3] * p[3] + p[4] * p[4] + p[5] * p[5])
        ax, ay, az = p[3] / r, p[4] / r, p[5] / r
        vx, vy, vz = P[:, 0] - p[0], P[:, 1] - p[1], P[:, 2] - p[2]
        h = ax * vx + ay * vy + az * vz
        wx, wy, wz = vx - h * ax, vy - h * ay, vz - h * az
        rho = np.sqrt(wx * wx + wy * wy + wz * wz)
        e = rho - p[6]
        dt = np.sqrt(e * e + h * h)
        near = np.abs(dt - r) < k[0]
        s = e / rho
        gx, gy, gz = wx * s + h * ax, wy * s + h * ay, wz * s + h * az
        dot = N[:, 0] * gx + N[:, 1] * gy + N[:, 2] * gz
        return near & (np.abs(dot) > k[1] * dt)


def torus_record(center, axis, R, r):
    a = np.asarray(axis, dtype=np.float64)
    a = a / np.linalg.norm(a)
    return [*np.asarray(center, dtype=np.float64), *(a * r), float(R)]


def torus_points(rng, center, axis, R, r, n, noise=0.0):
    """n points on a torus and their unit tube normals (float64)"""
    a = np.asarray(axis, dtype=np.float64)
    a = a / np.linalg.norm(a)
    u = np.cross(a, [1.0, 0.0, 0.0] if abs(a[0]) < 0.9 else [0.0, 1.0, 0.0])
    u /= np.linalg.norm(u)
    v = np.cross(a, u)
    th, ph = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    radial = np.cos(th)[:, None] * u + np.sin(th)[:, None] * v
    nrm = np.cos(ph)[:, None] * radial + np.sin(ph)[:, None] * a
    pts = np.asarray(center) + R * radial + (r + rng.normal(0, noise, n))[:, None] * nrm
    return pts, nrm


def slab_classes(R):
    """the z-slab of test_plugin_gpu.py in float64 (NumpySlab: scorecandidate / refit in NumPy) and the same shape
    with device source (DeviceSlab: rsc_user_score / rsc_user_refit_extract); both keep their host fit"""

    def _m(z0, params, V, N):
        k = constants(params["slab"]["eps"], params["slab"]["alpha"])
        return slab_twin(np.array([z0]), k, V.astype(np.float64), N.astype(np.float64))

    @dataclass
    class NumpySlab(R.FittedShape):
        z0: float

        @staticmethod
        def defaultshapeparameters():
            return {"slab": {"eps": 0.3, "alpha": math.radians(5)}}

        @classmethod
        def fit(cls, p, n, pc, params):
            z = np.asarray(p, float)[:, 2]
            nz = np.abs(np.asarray(n, float)[:, 2])
            if z.max() - z.min() < 0.1 and (nz > math.cos(math.radians(5))).all():
                return cls(float(z.mean()))
            return None

        def scorecandidate(self, pc, subsetID, params):
            sub = pc.subsets[subsetID]
            m = _m(self.z0, params, pc.vertices[sub], pc.normals[sub]) & pc.isenabled[sub]
            return R.estimatescore(len(sub), pc.size, int(m.sum())), sub[m]

        def refit(self, pc, params):
            m = _m(self.z0, params, pc.vertices, pc.normals) & pc.isenabled
            return R.ExtractedShape(self, np.flatnonzero(m))

    @dataclass
    class DeviceSlab(NumpySlab):
        cuda_source = SLAB_SRC

        def device_record(self):
            return [self.z0], False

        @staticmethod
        def device_constants(params):
            return constants(params["slab"]["eps"], params["slab"]["alpha"])

        def scorecandidate(self, pc, subsetID, params):
            raise AssertionError("a device-capable shape is scored on the device")

        def refit(self, pc, params):
            raise AssertionError("a device-capable shape is refit on the device")

    return NumpySlab, DeviceSlab
