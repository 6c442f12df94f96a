// rsc_user_kernels.cuh -- the kernels of user-defined shapes, compiled at run time with NVRTC (rsc_user.cu).
//
// The library embeds this file as a string and compiles it together with the user's source, which defines
//
//   __device__ bool rsc_user_compatible(const double p[7], int outwards, const double k[8],
//                                       double x, double y, double z, double nx, double ny, double nz);
//
// and optionally (then the library compiles with -DRSC_USER_HAS_FIT)
//
//   __device__ bool rsc_user_fit(int np, const double P[8][3], const double N[8][3], const double k[8],
//                                double p[7], int* outwards);
//
// for sm_100a with --fmad=false and no fast-math, so that a NumPy restatement in the same operation order makes
// the same float64 decisions (DESIGN.md section 8).  The argument structs below are also compiled into the
// library itself (nvcc): one definition, one layout on both sides of the cudaLaunchKernel call.  Only plain
// types appear in them -- NVRTC sees no system header.
#pragma once

struct RscUserPoints {  // = rsc::PointSet
  const float* x;
  const float* y;
  const float* z;
  const float* nx;
  const float* ny;
  const float* nz;
  const unsigned* enabled;  // bit j%32 of word j/32 = pc.isenabled of point j
  const unsigned* valid;    // 1 for real points, 0 for padding
  long long n;
  long long n_pad;  // multiple of 512
  const double* xyz64;    // exact clouds: the caller's float64 coordinates (AoS), point j at 3 * (map ? map[j] : j)
  const double* nrm64;
  const long long* map;
};

struct RscUserCand {  // = rsc_cand (64 bytes)
  int type;
  int outwards;
  double p[7];
};

struct RscUserScoreArgs {
  RscUserPoints ps;
  const RscUserCand* cands;  // [C], one user type
  int C;
  int nk;
  double k[8];
  int* counts;       // [C], zeroed by the host
  unsigned* masks;   // nullable: candidate-major [C][words], zeroed by the host
  long long words;   // ceil(n / 32)
  const unsigned long long* d_count;  // nullable: number of candidates = min(*d_count, C) (the device loop)
  int type;                           // only records of this type are scored
  int* counts2;                       // nullable: receives the same counts as `counts`
};

struct RscUserFitArgs {
  const float* soa;      // the cloud: x | y | z | nx | ny | nz rows of n_pad floats
  long long n_pad;
  const double* xyz64;   // exact clouds: the caller's float64 coordinates (AoS [3 n]), read instead of soa
  const double* nrm64;
  const long long* idx;  // [S][np] drawn indices; a row starting with -1 is a failed sample
  int S, np;
  int npos, pos;         // positions in the fit order / this type's position
  int type;
  int nk;
  double k[8];
  RscUserCand* dense;    // [S][npos]: slot s * npos + pos, as the built-in fit kernel writes
  unsigned* okmask;      // [(S + 127) / 128][npos][4] ballot words
};

struct RscUserMaskArgs {
  RscUserPoints ps;
  RscUserCand cand;
  int nk;
  double k[8];
  unsigned* inl;  // [n_pad / 32] inlier-mask words (enabled points only)
};

#define RSC_USER_THREADS 256
#define RSC_USER_TILE 128  // candidate records staged in shared memory per pass

#ifdef __CUDACC_RTC__

__device__ bool rsc_user_compatible(const double p[7], int outwards, const double k[8], double x, double y, double z, double nx,
                                    double ny, double nz);

// The float64 coordinates of point p of a set: an exact cloud's own, else the float32 ones widened
__device__ __forceinline__ void rsc_user_point(const RscUserPoints& ps, long long p, double q[6]) {
  if (ps.xyz64 && p < ps.n) {
    const long long i = 3 * (ps.map ? ps.map[p] : p);
    q[0] = ps.xyz64[i], q[1] = ps.xyz64[i + 1], q[2] = ps.xyz64[i + 2];
    q[3] = ps.nrm64[i], q[4] = ps.nrm64[i + 1], q[5] = ps.nrm64[i + 2];
  } else {
    q[0] = __ldg(ps.x + p), q[1] = __ldg(ps.y + p), q[2] = __ldg(ps.z + p);
    q[3] = __ldg(ps.nx + p), q[4] = __ldg(ps.ny + p), q[5] = __ldg(ps.nz + p);
  }
}

// Counts (and masks) of C candidates of one user type: the transposed mapping of the small-batch scorer
// (rsc_small.cu).  A thread owns a point; the CTA stages a chunk of candidate records in shared memory and reads
// them as broadcasts; a (candidate, 32 points) group is one ballot, its POPC goes into a shared counter, and each
// CTA adds one atomic per candidate.  Candidate chunks are spread over gridDim.y.  Every pair is decided once, in
// float64, on the point's float32 coordinates widened to double (an exact cloud's float64 coordinates).
// The device loop passes a mixed batch of built-in and user records whose size may stay on the device (a.d_count):
// only records of a.type are scored, and their counts are ADDED where the built-in scorer has left zeros.
extern "C" __global__ void __launch_bounds__(RSC_USER_THREADS) rsc_user_score_kernel(const RscUserScoreArgs a) {
  __shared__ RscUserCand sc[RSC_USER_TILE];
  __shared__ int scount[RSC_USER_TILE];
  __shared__ double sk[8];
  const int lane = threadIdx.x & 31;
  if (threadIdx.x < 8) sk[threadIdx.x] = threadIdx.x < a.nk ? a.k[threadIdx.x] : 0.0;
  const int C = a.d_count && *a.d_count < (unsigned long long)a.C ? (int)*a.d_count : a.C;
  const long long ntiles = a.ps.n_pad / RSC_USER_THREADS;
  for (int c0 = blockIdx.y * RSC_USER_TILE; c0 < C; c0 += gridDim.y * RSC_USER_TILE) {
    const int ct = min(RSC_USER_TILE, C - c0);
    for (int i = threadIdx.x; i < ct; i += RSC_USER_THREADS) {
      sc[i] = a.cands[c0 + i];
      scount[i] = 0;
    }
    __syncthreads();
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
      const long long p = t * RSC_USER_THREADS + threadIdx.x;
      const unsigned live = __ldg(a.ps.enabled + (p >> 5)) & __ldg(a.ps.valid + (p >> 5));
      if (live == 0u) continue;  // warp-uniform: no enabled real point in this group
      const bool on = (live >> lane) & 1u;
      double q[6];
      rsc_user_point(a.ps, p, q);
      for (int c = 0; c < ct; ++c) {
        if (sc[c].type != a.type) continue;  // block-uniform: a record of another type in a mixed batch
        const bool ok = on && rsc_user_compatible(sc[c].p, sc[c].outwards, sk, q[0], q[1], q[2], q[3], q[4], q[5]);
        const unsigned b = __ballot_sync(0xffffffffu, ok);
        if (lane == 0 && b) {
          atomicAdd(&scount[c], __popc(b));
          if (a.masks) a.masks[(long long)(c0 + c) * a.words + (p >> 5)] = b;
        }
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < ct; i += RSC_USER_THREADS)
      if (scount[i]) {
        atomicAdd(a.counts + c0 + i, scount[i]);
        if (a.counts2) atomicAdd(a.counts2 + c0 + i, scount[i]);
      }
    __syncthreads();
  }
}

// The inlier-mask words of one candidate over the whole cloud, enabled points only: what K4's mask kernel writes
// for a built-in shape (rsc_extract.cu), so that the library's count / scan / compaction follow unchanged.
extern "C" __global__ void __launch_bounds__(RSC_USER_THREADS) rsc_user_mask_kernel(const RscUserMaskArgs a) {
  __shared__ RscUserCand sc;
  __shared__ double sk[8];
  if (threadIdx.x == 0) sc = a.cand;
  if (threadIdx.x < 8) sk[threadIdx.x] = threadIdx.x < a.nk ? a.k[threadIdx.x] : 0.0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  for (long long p = (long long)blockIdx.x * RSC_USER_THREADS + threadIdx.x; p < a.ps.n_pad;
       p += (long long)gridDim.x * RSC_USER_THREADS) {
    const unsigned live = __ldg(a.ps.enabled + (p >> 5)) & __ldg(a.ps.valid + (p >> 5));
    bool ok = false;
    if (((live >> lane) & 1u) && a.ps.xyz64) {  // (a live point is a real one: p < n)
      const long long i = 3 * (a.ps.map ? a.ps.map[p] : p);
      ok = rsc_user_compatible(sc.p, sc.outwards, sk, a.ps.xyz64[i], a.ps.xyz64[i + 1], a.ps.xyz64[i + 2], a.ps.nrm64[i],
                               a.ps.nrm64[i + 1], a.ps.nrm64[i + 2]);
    } else if ((live >> lane) & 1u) {
      ok = rsc_user_compatible(sc.p, sc.outwards, sk, __ldg(a.ps.x + p), __ldg(a.ps.y + p), __ldg(a.ps.z + p), __ldg(a.ps.nx + p),
                               __ldg(a.ps.ny + p), __ldg(a.ps.nz + p));
    }
    const unsigned b = __ballot_sync(0xffffffffu, ok);
    if (lane == 0) a.inl[p >> 5] = b;
  }
}

#ifdef RSC_USER_HAS_FIT
__device__ bool rsc_user_fit(int np, const double P[8][3], const double N[8][3], const double k[8], double p[7], int* outwards);

// K1 for one user type: one thread per minimal set, the shape of the built-in fit kernel (rsc_fit.cu).  The
// candidate goes to the same dense slot and the set's bit into the same ballot word the built-in fits use, so
// the library's group scan and compaction emit (set, position in the fit order) order unchanged.
extern "C" __global__ void __launch_bounds__(128) rsc_user_fit_kernel(const RscUserFitArgs a) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  bool ok = false;
  if (s < a.S && a.idx[(long long)s * a.np] >= 0) {
    double P[8][3], N[8][3], k[8], p[7];
    for (int q = 0; q < 8; ++q) {
      k[q] = q < a.nk ? a.k[q] : 0.0;
      for (int d = 0; d < 3; ++d) P[q][d] = N[q][d] = 0.0;
    }
    for (int q = 0; q < a.np; ++q) {
      const long long i = a.idx[(long long)s * a.np + q];
      for (int d = 0; d < 3; ++d) {
        P[q][d] = a.xyz64 ? a.xyz64[3 * i + d] : (double)__ldg(a.soa + d * a.n_pad + i);
        N[q][d] = a.xyz64 ? a.nrm64[3 * i + d] : (double)__ldg(a.soa + (3 + d) * a.n_pad + i);
      }
    }
    for (int j = 0; j < 7; ++j) p[j] = 0.0;
    int outw = 0;
    ok = rsc_user_fit(a.np, P, N, k, p, &outw);
    if (ok) {
      RscUserCand c;
      c.type = a.type;
      c.outwards = outw;
      for (int j = 0; j < 7; ++j) c.p[j] = p[j];
      a.dense[(long long)s * a.npos + a.pos] = c;
    }
  }
  const unsigned m = __ballot_sync(0xffffffffu, ok);
  if ((threadIdx.x & 31) == 0) a.okmask[((long long)blockIdx.x * a.npos + a.pos) * 4 + (threadIdx.x >> 5)] = m;
}
#endif  // RSC_USER_HAS_FIT

#endif  // __CUDACC_RTC__
