"""Two user-defined shapes that fit on the device (include/rsc.h, rsc_user_fit) and their Python / NumPy twins.

Each twin evaluates the same float64 operations in the same order as the CUDA source, on the cloud's float32
coordinates widened to double (`pc.vertices[row].astype(np.float32).astype(np.float64)`).  NVRTC compiles with
--fmad=false and IEEE division / square root, so the twins' fits and decisions are the device's bit for bit.

  slab  p = (z0),  k = (eps, cos alpha, fit tolerance):  z0 = ((z_0 + z_1) + z_2) / 3; every point of the set has
        |z_i - z0| < k[2] and |nz_i| > k[1].  Compatible: |z - z0| < eps and |nz| > cos alpha.
  zcyl  a cylinder along z, p = (cx, cy, R),  k = (eps, cos alpha):  the centre is where the xy normal lines of
        points 0 and 1 cross (Cramer's rule; rejected when the determinant is small against |n0xy| |n1xy|), R the
        distance of point 0 from it; every point of the set must pass the compatibility test.  Compatible:
        |rho - R| < eps and |(r . n)| > cos alpha * rho, r = (x - cx, y - cy), rho = |r|.
"""
import math
from dataclasses import dataclass

import numpy as np

SLAB_COMPAT = r"""
// p = (z0); k = (eps, cos alpha, fit tolerance)
__device__ bool rsc_user_compatible(const double p[7], int outwards, const double k[8],
                                    double x, double y, double z, double nx, double ny, double nz) {
  return fabs(z - p[0]) < k[0] && fabs(nz) > k[1];
}
"""

SLAB_FIT = r"""
__device__ bool rsc_user_fit(int np, const double P[8][3], const double N[8][3], const double k[8],
                             double p[7], int* outwards) {
  const double z0 = ((P[0][2] + P[1][2]) + P[2][2]) / 3.0;
  for (int i = 0; i < np; ++i)
    if (!(fabs(P[i][2] - z0) < k[2]) || !(fabs(N[i][2]) > k[1])) return false;
  p[0] = z0;
  return true;
}
"""

ZCYL_COMPAT = r"""
// p = (cx, cy, R); k = (eps, cos alpha)
__device__ bool rsc_user_compatible(const double p[7], int outwards, const double k[8],
                                    double x, double y, double z, double nx, double ny, double nz) {
  const double rx = x - p[0], ry = y - p[1];
  const double rho = sqrt(rx * rx + ry * ry);
  return fabs(rho - p[2]) < k[0] && fabs(rx * nx + ry * ny) > k[1] * rho;
}
"""

ZCYL_FIT = r"""
__device__ bool rsc_user_fit(int np, const double P[8][3], const double N[8][3], const double k[8],
                             double p[7], int* outwards) {
  const double n0x = N[0][0], n0y = N[0][1], n1x = N[1][0], n1y = N[1][1];
  const double det = n1x * n0y - n0x * n1y;
  const double l0 = sqrt(n0x * n0x + n0y * n0y), l1 = sqrt(n1x * n1x + n1y * n1y);
  if (!(fabs(det) > 0.1 * (l0 * l1))) return false;  // (nearly) parallel normals
  const double dx = P[1][0] - P[0][0], dy = P[1][1] - P[0][1];
  const double s = (n1x * dy - dx * n1y) / det;
  const double cx = P[0][0] + s * n0x, cy = P[0][1] + s * n0y;
  const double ex = P[0][0] - cx, ey = P[0][1] - cy;
  const double R = sqrt(ex * ex + ey * ey);
  for (int i = 0; i < np; ++i) {
    const double rx = P[i][0] - cx, ry = P[i][1] - cy;
    const double rho = sqrt(rx * rx + ry * ry);
    if (!(fabs(rho - R) < k[0]) || !(fabs(rx * N[i][0] + ry * N[i][1]) > k[1] * rho)) return false;
  }
  p[0] = cx, p[1] = cy, p[2] = R;
  return true;
}
"""

SLAB_SRC = SLAB_COMPAT + SLAB_FIT
ZCYL_SRC = ZCYL_COMPAT + ZCYL_FIT

BROKEN_FIT_SRC = SLAB_COMPAT + r"""
__device__ bool rsc_user_fit(int np, const double P[8][3], const double N[8][3], const double k[8],
                             double p[7], int* outwards) {
  p[0] = P[0][2] +* 2.0;
  return true;
}
"""
BROKEN_FIT_LINE = next(i + 1 for i, line in enumerate(BROKEN_FIT_SRC.split("\n")) if "+*" in line)


def slab_constants(eps=0.3, alpha=math.radians(5), tol=0.1):
    return [float(eps), math.cos(alpha), float(tol)]


def zcyl_constants(eps=0.05, alpha=math.radians(10)):
    return [float(eps), math.cos(alpha)]


def slab_fit_twin(P, N, k):
    """P, N: (np, 3) float64 -> record p or None"""
    z0 = ((P[0][2] + P[1][2]) + P[2][2]) / 3.0
    for i in range(len(P)):
        if not (abs(P[i][2] - z0) < k[2]) or not (abs(N[i][2]) > k[1]):
            return None
    return [z0]


def slab_twin(p, k, P, N):
    with np.errstate(invalid="ignore"):
        return (np.abs(P[:, 2] - p[0]) < k[0]) & (np.abs(N[:, 2]) > k[1])


def zcyl_fit_twin(P, N, k):
    n0x, n0y, n1x, n1y = float(N[0][0]), float(N[0][1]), float(N[1][0]), float(N[1][1])
    det = n1x * n0y - n0x * n1y
    l0, l1 = math.sqrt(n0x * n0x + n0y * n0y), math.sqrt(n1x * n1x + n1y * n1y)
    if not (abs(det) > 0.1 * (l0 * l1)):
        return None
    dx, dy = float(P[1][0]) - float(P[0][0]), float(P[1][1]) - float(P[0][1])
    s = (n1x * dy - dx * n1y) / det
    cx, cy = float(P[0][0]) + s * n0x, float(P[0][1]) + s * n0y
    ex, ey = float(P[0][0]) - cx, float(P[0][1]) - cy
    R = math.sqrt(ex * ex + ey * ey)
    for i in range(len(P)):
        rx, ry = float(P[i][0]) - cx, float(P[i][1]) - cy
        rho = math.sqrt(rx * rx + ry * ry)
        if not (abs(rho - R) < k[0]) or not (abs(rx * float(N[i][0]) + ry * float(N[i][1])) > k[1] * rho):
            return None
    return [cx, cy, R]


def zcyl_twin(p, k, P, N):
    with np.errstate(invalid="ignore"):
        rx, ry = P[:, 0] - p[0], P[:, 1] - p[1]
        rho = np.sqrt(rx * rx + ry * ry)
        return (np.abs(rho - p[2]) < k[0]) & (np.abs(rx * N[:, 0] + ry * N[:, 1]) > k[1] * rho)


def shape_classes(R):
    """(NumPy twins, device-scoring twins, device-fitting shapes) of the slab and the z-cylinder.

    NumPy twins fit, score and refit on the host; device-scoring twins fit on the host and score / refit with their
    compatibility source (no rsc_user_fit); device-fitting shapes carry the full source and `from_device_record`."""

    def _fit(cls, twin, p, n, params):
        P = np.asarray(p, np.float32).astype(np.float64)
        N = np.asarray(n, np.float32).astype(np.float64)
        r = twin(P, N, cls.device_constants(params))
        return None if r is None else cls.from_device_record(r, False)

    def _mask(self, params, V, N):
        return self.TWIN(np.asarray(self.device_record()[0], np.float64), self.device_constants(params), V.astype(np.float64),
                         N.astype(np.float64))

    class _Twin(R.FittedShape):
        @classmethod
        def fit(cls, p, n, pc, params):
            return _fit(cls, cls.FIT_TWIN, p, n, params)

        def scorecandidate(self, pc, subsetID, params):
            sub = pc.subsets[subsetID]
            m = _mask(self, params, pc.vertices[sub], pc.normals[sub]) & pc.isenabled[sub]
            return R.estimatescore(len(sub), pc.size, int(m.sum())), sub[m]

        def refit(self, pc, params):
            m = _mask(self, params, pc.vertices, pc.normals) & pc.isenabled
            return R.ExtractedShape(self, np.flatnonzero(m))

    @dataclass
    class NumpySlab(_Twin):
        z0: float
        FIT_TWIN = staticmethod(slab_fit_twin)
        TWIN = staticmethod(slab_twin)

        @staticmethod
        def defaultshapeparameters():
            return {"slab": {"eps": 0.3, "alpha": math.radians(5), "tol": 0.1}}

        @staticmethod
        def device_constants(params):
            s = params["slab"]
            return slab_constants(s["eps"], s["alpha"], s["tol"])

        def device_record(self):
            return [self.z0], False

        @classmethod
        def from_device_record(cls, p, outwards):
            return cls(float(p[0]))

    @dataclass
    class NumpyZCyl(_Twin):
        cx: float
        cy: float
        radius: float
        FIT_TWIN = staticmethod(zcyl_fit_twin)
        TWIN = staticmethod(zcyl_twin)

        @staticmethod
        def defaultshapeparameters():
            return {"zcyl": {"eps": 0.05, "alpha": math.radians(10)}}

        @staticmethod
        def device_constants(params):
            return zcyl_constants(params["zcyl"]["eps"], params["zcyl"]["alpha"])

        def device_record(self):
            return [self.cx, self.cy, self.radius], False

        @classmethod
        def from_device_record(cls, p, outwards):
            return cls(float(p[0]), float(p[1]), float(p[2]))

    def _scored(base, src):
        @dataclass
        class Scored(base):
            cuda_source = src

            def scorecandidate(self, pc, subsetID, params):
                raise AssertionError("a device-capable shape is scored on the device")

            def refit(self, pc, params):
                raise AssertionError("a device-capable shape is refit on the device")

        Scored.__name__ = Scored.__qualname__ = base.__name__.replace("Numpy", "Scored")
        return Scored

    def _fitted(base, src):
        @dataclass
        class Fitted(base):
            cuda_source = src

            @classmethod
            def fit(cls, p, n, pc, params):
                raise AssertionError("a device-fitting shape is fitted on the device")

        Fitted.__name__ = Fitted.__qualname__ = base.__name__.replace("Scored", "Device")
        return Fitted

    ScoredSlab, ScoredZCyl = _scored(NumpySlab, SLAB_COMPAT), _scored(NumpyZCyl, ZCYL_COMPAT)
    DeviceSlab, DeviceZCyl = _fitted(ScoredSlab, SLAB_SRC), _fitted(ScoredZCyl, ZCYL_SRC)
    return (NumpySlab, NumpyZCyl), (ScoredSlab, ScoredZCyl), (DeviceSlab, DeviceZCyl)


def zcyl_points(rng, cx, cy, R, z0, z1, n, noise=0.0):
    th = rng.uniform(0, 2 * np.pi, n)
    nrm = np.c_[np.cos(th), np.sin(th), np.zeros(n)]
    pts = np.c_[cx + (R + rng.normal(0, noise, n)) * nrm[:, 0], cy + (R + rng.normal(0, noise, n)) * nrm[:, 1], rng.uniform(z0, z1, n)]
    return pts, nrm


def slab_points(rng, z0, half, n, noise=0.02, center=(0.0, 0.0)):
    pts = np.c_[rng.uniform(-half, half, (n, 2)) + np.asarray(center), np.full(n, z0) + rng.normal(0, noise, n)]
    nrm = np.tile([0.0, 0.0, 1.0], (n, 1)) + rng.normal(0, 0.01, (n, 3))
    return pts, nrm / np.linalg.norm(nrm, axis=1, keepdims=True)


def mixed_scene(rng, n, frac_out=0.1):
    """built-in primitives (a plane wall, a sphere) + slabs + vertical cylinders + outliers, about n points, float32"""
    parts = []
    m = n // 6
    # a vertical plane x = 40
    wall = np.c_[np.full(m, 40.0) + rng.normal(0, 0.01, m), rng.uniform(-30, 30, (m, 2))]
    parts.append((wall, np.tile([1.0, 0.0, 0.0], (m, 1))))
    d = rng.normal(size=(m, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    parts.append((np.array([-30.0, 20.0, 5.0]) + 6.0 * d, d))
    parts.append(slab_points(rng, 7.0, 20.0, m))
    parts.append(slab_points(rng, -12.0, 10.0, m // 2, center=(5.0, -5.0)))
    parts.append(zcyl_points(rng, -5.0, -20.0, 4.0, -20.0, 0.0, m, noise=0.005))
    parts.append(zcyl_points(rng, 15.0, 18.0, 2.5, -25.0, -15.0, m // 2, noise=0.005))
    k = n - sum(len(p) for p, _ in parts)
    out = rng.uniform(-40, 40, (k, 3))
    on = rng.normal(size=(k, 3))
    parts.append((out, on / np.linalg.norm(on, axis=1, keepdims=True)))
    V = np.concatenate([p for p, _ in parts]).astype(np.float32)
    N = np.concatenate([q for _, q in parts])
    N = (N / np.linalg.norm(N, axis=1, keepdims=True)).astype(np.float32)
    perm = rng.permutation(len(V))
    return V[perm], N[perm]
