// rsc_cull.cu -- scoring with Morton-tile culling (extension; the same counts as rsc_score).
//
// The dense K2 kernel (rsc_score.cu) evaluates every (candidate, point) pair, like the reference's
// compatibles*.  Most of those pairs are far from the candidate's surface.  With the points in Morton
// order (rsc_octree.cu: the whole cloud after rsc_cloud_build_cells, or the Morton VIEW of a subset copy) a
// tile of consecutive points has a small bounding sphere (c, r), and every distance function of the path
// (plane.jl:82-103, sphere.jl:163-166, cylinder.jl:209-214, the cone's h sin - rho cos) is 1-Lipschitz in the
// point, so
//       |dist(c)| > eps + r   =>   no point of the tile is within eps   =>   the tile adds nothing
// to the candidate's count (cull_far; tests/test_cull_model.py).  7 % of the (candidate, 128-point tile) pairs of
// config c3 survive.
//
// Three sphere levels: 4096-point blocks (pre-pass cull_block_kernel: a bit per (block, candidate)), 512-point
// groups and 128-point tiles (inside cull_score_kernel: a CTA takes a group and a range of candidates, a thread
// tests one candidate).  Survivors of a tile are evaluated in the dense kernel's mapping -- lane = candidate,
// record in registers, the tile's points broadcast from shared memory, two points per packed FFMA2 -- in batches
// of 32 handed out to whichever warp is free; a lane counts for its own candidate, no reductions.  Same FP32
// forms and guard band as the dense kernel (evalp<T> in rsc_eval.cuh); a 32-point block that touches the band is
// redone by the warp with lane = point, its in-band pairs are decided in float64 in the reference's operation order
// by cull_pair_kernel (rsc_exact.cuh).  The records are sorted by column type first (cull_compile_kernel), so a
// warp runs one formula.  DESIGN.md section 3 has the measurements and the history.
// Counts only (masks would come out in Morton order).  Entry points: rsc_score_culled (whole cloud),
// rsc_score_culled_subset, and loop_score_new / K5 of rsc_ransac_run (cull_enqueue on device-resident candidates).
#include <math.h>
#include <stdlib.h>

#include <vector>

#include "rsc_eval.cuh"
#include "rsc_exact.cuh"

namespace rsc {

size_t cull_sphere_count(int64_t n_pad);
int32_t cull_tile_spheres(rsc_ctx* ctx, const PointSet& ps, float4* tiles, cudaStream_t st, const unsigned long long* d_n);

constexpr int kCullThreads = 128;
constexpr int kCullWarps = kCullThreads / 32;
constexpr int kCullTile = 128;                       // points of a warp's tile: one bounding sphere each
constexpr int kCullGroup = kCullTile * kCullWarps;   // points of a CTA's group of tiles (= kTile): one sphere too
constexpr int kCullBlockGroups = 8;                  // groups per block (4096 points): the coarsest sphere (pre-pass)
constexpr int kCullSuper = 2048;                     // most candidates of one work item (capacity of the tiles' survivor lists)
#ifndef RSC_CULL_MINB
#define RSC_CULL_MINB 4
#endif
#ifndef RSC_CULL_UNROLL
#define RSC_CULL_UNROLL 4  // point pairs in flight per lane in the narrow phase
#endif
constexpr int kCullUnroll = RSC_CULL_UNROLL;
constexpr int kCullMinB = RSC_CULL_MINB;  // CTAs per SM the kernel is compiled for (registers: 65536 / (128 kCullMinB))
static_assert(kCullGroup == kTile, "a group of tiles is one padding unit of the point sets");

struct CullArgs {
  PointSet ps;           // the points in Morton order (rows of n_pad floats; n_pad a multiple of 512)
  const float4* tiles;   // bounding sphere of every 128-point tile: centre, radius
  const float4* groups;  // bounding sphere of every 512-point group of four tiles
  const float4* blocks;  // bounding sphere of every 4096-point block of eight groups
  uint32_t* bbits;       // [nblocks][cwords] pre-pass: bit c = candidate c passes the block's sphere
  int nblocks, cwords;
  int ngroups;           // n_pad / 512: a CTA takes the four tiles of a group, one per warp
  int nranges;           // the candidates are split into nranges runs of cands_per_range (<= kCullSuper, multiple of 128)
  int cands_per_range;
  const float* rec;      // [C][kRecFields] compiled records, SORTED by column type
  const uint8_t* col;    // [C] column types (sorted)
  const int32_t* orig;   // [C] sorted slot -> index of the candidate
  const rsc_cand* cands;
  const int32_t* d_C;    // number of candidates on the device (nullptr: C)
  Thresh th;
  int C;
  int32_t* cv;  // [C] compatible real points
  int32_t* ce;  // [C] compatible enabled points
  unsigned long long* stats;  // [0] surviving (candidate, tile) pairs, [1] pairs decided in FP64
  uint32_t* work;             // dynamic work counter (items handed out)
  uint2* pairs;               // (slot, position) of the pairs inside the guard band: decided in float64 by cull_pair_kernel
  uint32_t pcap;
  uint32_t* pn;               // entries appended (beyond pcap: decided inline)
  int inline_fp64;            // != 0: no queue, every in-band pair is decided on the spot (RSC_CULL_INLINE=1)
};

__device__ __forceinline__ int cull_count(const CullArgs& a) { return a.d_C ? max(0, min(*a.d_C, a.C)) : a.C; }

// ---- candidate compiler: FP32 records sorted by column type (a warp of the scorer then runs one formula) ----
__global__ void cull_hist_kernel(const rsc_cand* __restrict__ cands, int C, const int32_t* __restrict__ d_C, uint32_t* __restrict__ hist) {
  __shared__ uint32_t h[kColTypes];
  if (threadIdx.x < kColTypes) h[threadIdx.x] = 0;
  __syncthreads();
  const int n = d_C ? max(0, min(*d_C, C)) : C;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicAdd(&h[col_type(cands[i])], 1u);
  __syncthreads();
  if (threadIdx.x < kColTypes && h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], h[threadIdx.x]);
}

__global__ void cull_compile_kernel(const rsc_cand* __restrict__ cands, int C, const int32_t* __restrict__ d_C, Thresh th, float pmax,
                                    float nmax, const uint32_t* __restrict__ hist, uint32_t* __restrict__ cursor,
                                    float* __restrict__ rec, uint8_t* __restrict__ col, int32_t* __restrict__ orig) {
  const int n = d_C ? max(0, min(*d_C, C)) : C;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const rsc_cand c = cands[i];
  const int ct = col_type(c);
  uint32_t base = 0;
  for (int t = 0; t < ct; ++t) base += hist[t];
  // one atomic per (warp, type): the lanes of a type take consecutive slots
  const uint32_t peers = __match_any_sync(__activemask(), ct);
  const int leader = __ffs(peers) - 1;
  uint32_t first = 0;
  if ((int)(threadIdx.x & 31) == leader) first = atomicAdd(&cursor[ct], (uint32_t)__popc(peers));
  first = __shfl_sync(peers, first, leader);
  const uint32_t slot = base + first + (uint32_t)__popc(peers & ((1u << (threadIdx.x & 31)) - 1u));
  float r[kRecFields];
  compile_record(c, ct, th, pmax, nmax, r);
  float4* out = reinterpret_cast<float4*>(rec + (size_t)slot * kRecFields);
  out[0] = make_float4(r[0], r[1], r[2], r[3]);
  out[1] = make_float4(r[4], r[5], r[6], r[7]);
  out[2] = make_float4(r[8], r[9], r[10], r[11]);
  col[slot] = (uint8_t)ct;
  orig[slot] = i;
}

__global__ void morton_gather_kernel(const float* __restrict__ soa, int64_t n_pad, const uint32_t* __restrict__ perm, int64_t n,
                                     float* __restrict__ msoa) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pad) return;
  const bool real = i < n;
  const int64_t j = real ? (int64_t)perm[i] : 0;
#pragma unroll
  for (int f = 0; f < 6; ++f) msoa[f * n_pad + i] = real ? soa[f * n_pad + j] : 0.f;
}

__global__ void widen_u32_kernel(const uint32_t* __restrict__ in, int64_t n, int64_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (int64_t)in[i];
}

// one warp per tile of `tile_pts` points: centre of the bounding box, radius = largest distance of a point to it
// (rounded up)
__global__ void __launch_bounds__(256) tile_sphere_kernel(const float* __restrict__ X, const float* __restrict__ Y,
                                                          const float* __restrict__ Z, int64_t n, int tile_pts, int ntiles,
                                                          float4* __restrict__ tiles, const unsigned long long* __restrict__ d_n) {
  if (d_n) n = min(n, (int64_t)*d_n);
  const int tile = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (tile >= ntiles) return;
  const int64_t base = (int64_t)tile * tile_pts;
  float lo[3] = {3.4e38f, 3.4e38f, 3.4e38f}, hi[3] = {-3.4e38f, -3.4e38f, -3.4e38f};
  for (int k = lane; k < tile_pts; k += 32) {
    const int64_t j = base + k;
    if (j < n) {
      const float p[3] = {X[j], Y[j], Z[j]};
#pragma unroll
      for (int d = 0; d < 3; ++d) lo[d] = fminf(lo[d], p[d]), hi[d] = fmaxf(hi[d], p[d]);
    }
  }
#pragma unroll
  for (int d = 0; d < 3; ++d)
#pragma unroll
    for (int s = 16; s; s >>= 1) {
      lo[d] = fminf(lo[d], __shfl_xor_sync(0xffffffffu, lo[d], s));
      hi[d] = fmaxf(hi[d], __shfl_xor_sync(0xffffffffu, hi[d], s));
    }
  const float cx = 0.5f * (lo[0] + hi[0]), cy = 0.5f * (lo[1] + hi[1]), cz = 0.5f * (lo[2] + hi[2]);
  float r2 = 0.f;
  for (int k = lane; k < tile_pts; k += 32) {
    const int64_t j = base + k;
    if (j < n) {
      const float dx = X[j] - cx, dy = Y[j] - cy, dz = Z[j] - cz;
      r2 = fmaxf(r2, dx * dx + dy * dy + dz * dz);
    }
  }
#pragma unroll
  for (int s = 16; s; s >>= 1) r2 = fmaxf(r2, __shfl_xor_sync(0xffffffffu, r2, s));
  if (lane == 0) {
    // NaN / Inf coordinates: an infinite radius, the tile is never culled; a tile of padding only: radius -1
    // (whether it is culled or not does not matter: its points are not valid)
    float r = sqrtf(r2) * 1.00001f + 1e-30f;
    if (!(r < 3.0e38f) || !(fabsf(cx) < 3.0e38f) || !(fabsf(cy) < 3.0e38f) || !(fabsf(cz) < 3.0e38f)) r = __int_as_float(0x7f800000);
    const bool empty = base >= n;
    tiles[tile] = make_float4(empty ? 0.f : cx, empty ? 0.f : cy, empty ? 0.f : cz, empty ? -1.f : r);
  }
}

// true: provably no point within eps of the candidate inside the sphere ts (NaN anywhere -> false)
__device__ __forceinline__ bool cull_far(int col, const float* r, float4 ts, float eps) {
  const float band = r[kBandField];
  const float rt = ts.w;
  float d, lim;
  if (col == RSC_PLANE) {
    d = fabsf(fmaf(r[0], ts.x, fmaf(r[1], ts.y, fmaf(r[2], ts.z, r[3]))));
    lim = eps + rt;
  } else {
    const float vx = fmaf(r[0], ts.x, r[1]), vy = fmaf(r[0], ts.y, r[2]), vz = fmaf(r[0], ts.z, r[3]);
    if (col == RSC_SPHERE) {
      d = fabsf(sqrtf(fmaf(vx, vx, fmaf(vy, vy, vz * vz))) + r[4]);
      lim = eps + rt;
    } else {
      const float h = fmaf(r[4], vx, fmaf(r[5], vy, r[6] * vz));
      const float wx = fmaf(-r[4], h, vx), wy = fmaf(-r[5], h, vy), wz = fmaf(-r[6], h, vz);
      const float rho = sqrtf(fmaf(wx, wx, fmaf(wy, wy, wz * wz)));
      if (col == RSC_CYLINDER) {
        // the reference uses the axis as given (Q8): p -> |v - a (a.v)| has Lipschitz constant
        // max(1, | |a|^2 - 1 |), which is 1 for the unit axes the fits produce
        const float a2 = fmaf(r[4], r[4], fmaf(r[5], r[5], r[6] * r[6]));
        d = fabsf(rho + r[7]);
        lim = eps + rt * fmaxf(1.f, fabsf(a2 - 1.f) * 1.0001f);
      } else {
        // the cone records are scaled by 1/cos (1/sin for wide cones) of the half angle: r8 = -eps/scale
        d = (col == kConeWide) ? fabsf(fmaf(-rho, r[7], h)) : fabsf(fmaf(h, r[7], -rho));
        lim = -r[8] * (1.f + rt / eps);
      }
    }
  }
  return d > lim * 1.0001f + 8.f * band;
}

__device__ __forceinline__ void load_rec(const float* __restrict__ rec, int slot, float* r) {
  const float4* g = reinterpret_cast<const float4*>(rec + (size_t)slot * kRecFields);
  const float4 r0 = g[0], r1 = g[1], r2 = g[2];
  r[0] = r0.x, r[1] = r0.y, r[2] = r0.z, r[3] = r0.w, r[4] = r1.x, r[5] = r1.y, r[6] = r1.z, r[7] = r1.w;
  r[8] = r2.x, r[9] = r2.y, r[10] = r2.z, r[11] = r2.w;
}

// the FP64 decision of one in-band pair; out of line so that its registers (and code) do not weigh on the FP32 loop
__device__ __noinline__ uint32_t cull_exact(const rsc_cand* __restrict__ cp, const Thresh* th, const PointSet* ps, int64_t j) {
  const rsc_cand c = *cp;
  ex::ConeTrig tr{1.0, 0.0};
  if (c.type == RSC_CONE) {
    tr.ct = cos(-c.p[6] / 2);
    tr.st = sin(-c.p[6] / 2);
  }
  ex::V3 p, n;
  ex::point64(*ps, j, &p, &n);
  return ex::compat(c, tr, *th, p, n) ? 1u : 0u;
}

// A batch of up to 32 surviving (candidate, tile) pairs: lane = candidate (its record in registers), the tile's 128
// points stream through as broadcast shared-memory reads, two points per packed operation.  No reduction: every
// lane counts for its own candidate.  wp: the tile's points, pair i at wp + 12 i as (x, x') (y, y') (z, z')
// (nx, nx') (ny, ny') (nz, nz').  ALL lanes run the formula of type T (the warp stays converged); `mine` marks the
// lanes whose candidate really is of that type -- only they count.
// A 32-point block with a margin inside the guard band (or NaN) is redone by the whole warp on the spot, lane =
// point, record of the owning lane by shuffles: sure points are counted from the FP32 sign, the in-band pairs go to
// the float64 pair queue (cull_pair_kernel adds their counts).
template <int T>
__device__ __forceinline__ void cull_narrow(const CullArgs& a, const float* __restrict__ wp, const float* r, bool mine, int slot,
                                            int64_t base, const uint32_t* __restrict__ wm, unsigned long long* n_exact) {
  constexpr int PT = public_type(T);
  const float eps = a.th.eps[PT], cosa = a.th.cosa[PT];
  const float band = r[kBandField];
  const int lane = threadIdx.x & 31;
  int cv = 0, ce = 0;
#pragma unroll 1
  for (int g = 0; g < kCullTile / 32; ++g) {
    uint32_t acc = 0;
    float amin = __int_as_float(0x7f800000);
    const float4* q = reinterpret_cast<const float4*>(wp + g * 16 * 12);
#pragma unroll kCullUnroll
    for (int i = 0; i < 16; ++i) {
      const float4 a0 = q[3 * i], a1 = q[3 * i + 1], a2 = q[3 * i + 2];
      const float2 m = evalp<T>(r, make_float2(a0.x, a0.y), make_float2(a0.z, a0.w), make_float2(a1.x, a1.y), make_float2(a1.z, a1.w),
                                make_float2(a2.x, a2.y), make_float2(a2.z, a2.w), eps, cosa);
      // the inlier bit is the sign of the margin: funnel-shifted into the block's word (point 0 ends up in bit 31)
      acc = __funnelshift_l(__float_as_uint(m.x), acc, 1);
      acc = __funnelshift_l(__float_as_uint(m.y), acc, 1);
      amin = fmin_nan(amin, fmin_nan(fabsf(m.x), fabsf(m.y)));
    }
    const uint32_t vmask = wm[g];  // the block's valid / enabled words in sign-word order (shared memory, broadcast)
    uint32_t ambm = __ballot_sync(0xffffffffu, mine && !(amin > band));
    while (ambm) {  // (uniform) some lane's block touches the guard band: the warp redoes it, lane = point
      const int src = __ffs(ambm) - 1;
      ambm &= ambm - 1;
      float rr[RecN<T>::n];
#pragma unroll
      for (int f = 0; f < RecN<T>::n; ++f) rr[f] = __shfl_sync(0xffffffffu, r[f], src);
      const float bb = __shfl_sync(0xffffffffu, band, src);
      const int sslot = __shfl_sync(0xffffffffu, slot, src);
      const float* pp = wp + ((g * 32 + lane) >> 1) * 12 + (lane & 1);
      const float px = pp[0], py = pp[2], pz = pp[4], nx = pp[6], ny = pp[8], nz = pp[10];
      const float m = eval<T>(rr, px, py, pz, nx, ny, nz, eps, cosa);
      const bool real = (vmask >> (31 - lane)) & 1u;
      const bool sure = fabsf(m) > bb;  // false for NaN
      uint32_t ok = (sure && m < 0.f) ? 1u : 0u;
      const uint32_t unsure = __ballot_sync(0xffffffffu, real && !sure);
      if (unsure) {
        uint32_t b0 = a.pcap;
        if (!a.inline_fp64) {
          if (lane == 0) b0 = atomicAdd(a.pn, (uint32_t)__popc(unsure));
          b0 = __shfl_sync(0xffffffffu, b0, 0);
        }
        if (real && !sure) {
          const uint32_t ps = a.inline_fp64 ? a.pcap : b0 + (uint32_t)__popc(unsure & ((1u << lane) - 1u));
          const int64_t j = base + g * 32 + lane;
          if (ps < a.pcap) {
            a.pairs[ps] = make_uint2((uint32_t)sslot, (uint32_t)j);
          } else {  // queue full or switched off: the reference's float64 decision right here
            ok = cull_exact(a.cands + a.orig[sslot], &a.th, &a.ps, j);
            ++*n_exact;
          }
        }
      }
      const uint32_t okm = __ballot_sync(0xffffffffu, ok != 0);
      if (lane == src) acc = __brev(okm);
    }
    cv += __popc(acc & vmask);
    ce += __popc(acc & wm[4 + g]);
  }
  if (mine) {
    const int o = a.orig[slot];
    if (cv) atomicAdd(a.cv + o, cv);
    if (ce) atomicAdd(a.ce + o, ce);
  }
}

// pre-pass: every candidate against every 4096-point block's sphere, a warp per (block, 32 candidates); the main
// kernel then only looks at the candidates whose bit is set (a fifth of them on c3)
__global__ void __launch_bounds__(256) cull_block_kernel(const __grid_constant__ CullArgs a) {
  const int C = cull_count(a);
  const int lane = threadIdx.x & 31;
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= (int64_t)a.nblocks * a.cwords) return;
  const int block = (int)(w / a.cwords), cw = (int)(w % a.cwords);
  const int c = cw * 32 + lane;
  bool keep = false;
  if (c < C) {
    float r[kRecFields];
    load_rec(a.rec, c, r);
    const int ct = a.col[c];
    keep = !cull_far(ct, r, a.blocks[block], a.th.eps[public_type(ct)]);
  }
  const uint32_t m = __ballot_sync(0xffffffffu, keep);
  if (lane == 0) a.bbits[w] = m;
}

__global__ void __launch_bounds__(kCullThreads, kCullMinB) cull_score_kernel(const __grid_constant__ CullArgs a) {
  __shared__ __align__(16) float wpts[kCullWarps][kCullTile / 2 * 12];  // the four tiles' points as packed pairs
  __shared__ uint32_t wmask[kCullWarps][2 * (kCullTile / 32)];          // their valid / enabled words in sign-word order
  __shared__ float4 wsph[kCullWarps];                                   // their bounding spheres
  __shared__ uint16_t slist[kCullSuper];              // the item's candidates (relative to its first) that pass the block's sphere
  __shared__ uint16_t wlist[kCullWarps][kCullSuper];  // per tile: those that pass the group's and the tile's sphere too
  __shared__ uint32_t wn[kCullWarps], bnext, sitem, swtot[kCullWarps];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int C = cull_count(a);
  unsigned long long n_surv = 0, n_exact = 0;
  const uint32_t nitems = (uint32_t)a.ngroups * (uint32_t)a.nranges;
  for (;;) {
    __syncthreads();  // everybody is done with the previous item's lists and points
    if (tid == 0) sitem = atomicAdd(a.work, 1u), bnext = 0;
    if (tid < kCullWarps) wn[tid] = 0;
    __syncthreads();
    const uint32_t item = sitem;
    if (item >= nitems) break;
    const int group = (int)(item % (uint32_t)a.ngroups), range = (int)(item / (uint32_t)a.ngroups);
    const int c_lo = range * a.cands_per_range;
    const int c_hi = min(C, c_lo + a.cands_per_range);
    if (c_lo >= c_hi) continue;  // uniform
    // ---- warp w: the 128 points of tile w -> shared memory as packed pairs ----
    {
      const int tile = group * kCullWarps + warp;
      const int64_t base = (int64_t)tile * kCullTile;
      float* wp = wpts[warp];
#pragma unroll
      for (int g = 0; g < kCullTile / 32; ++g) {
        const int64_t j = base + g * 32 + lane;
        const int pp = g * 32 + lane;
        float* dst = wp + (pp >> 1) * 12 + (pp & 1);
        dst[0] = a.ps.x[j], dst[2] = a.ps.y[j], dst[4] = a.ps.z[j], dst[6] = a.ps.nx[j], dst[8] = a.ps.ny[j], dst[10] = a.ps.nz[j];
        const uint32_t v = __ballot_sync(0xffffffffu, j < a.ps.n);
        if (lane == 0) wmask[warp][g] = __brev(v), wmask[warp][4 + g] = __brev(v & a.ps.enabled[(base >> 5) + g]);
      }
      if (lane == 0) wsph[warp] = a.tiles[tile];
    }
    __syncthreads();
    // ---- the item's candidates that passed the pre-pass (their block's sphere), in order: thread t expands the
    // bits of word t behind an exclusive scan of the words' bit counts ----
    int nlist = 0;
    {
      const int nw = (c_hi - c_lo + 31) >> 5;  // <= kCullSuper / 32 <= kCullThreads words (c_lo is a multiple of 128)
      const uint32_t* bw = a.bbits + (size_t)(group / kCullBlockGroups) * a.cwords + (c_lo >> 5);
      uint32_t word = tid < nw ? bw[tid] : 0u;
      if (tid < nw && (tid + 1) * 32 > c_hi - c_lo) word &= (1u << ((c_hi - c_lo) & 31)) - 1u;  // (bits beyond C are 0 anyway)
      const int cnt = __popc(word);
      int inc = cnt;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
      }
      if (lane == 31) swtot[warp] = (uint32_t)inc;
      __syncthreads();
      int off = inc - cnt;
#pragma unroll
      for (int w = 0; w < kCullWarps; ++w) {
        if (w < warp) off += (int)swtot[w];
        nlist += (int)swtot[w];
      }
      while (word) {
        const int b = __ffs(word) - 1;
        word &= word - 1;
        slist[off++] = (uint16_t)(tid * 32 + b);
      }
    }
    __syncthreads();
    // ---- broad phase, a listed candidate per thread: the group's sphere first, then the four tiles' spheres ----
    if (nlist > 0) {
      const float4 gs = a.groups[group];
      for (int e = tid; e < nlist; e += kCullThreads) {
        const int rel = (int)slist[e];
        const int c = c_lo + rel;
        float r[kRecFields];
        load_rec(a.rec, c, r);
        const int ct = a.col[c];
        const float eps = a.th.eps[public_type(ct)];
        if (!cull_far(ct, r, gs, eps)) {
#pragma unroll
          for (int w = 0; w < kCullWarps; ++w)
            if (!cull_far(ct, r, wsph[w], eps)) wlist[w][atomicAdd(&wn[w], 1u)] = (uint16_t)rel;
        }
      }
    }
    __syncthreads();
    // ---- narrow phase: batches of 32 (candidate, tile) pairs, handed out to whichever warp is free ----
    uint32_t nb[kCullWarps], total = 0;
#pragma unroll
    for (int w = 0; w < kCullWarps; ++w) {
      nb[w] = (wn[w] + 31u) >> 5;
      total += nb[w];
      if (warp == w) n_surv += wn[w];
    }
    for (;;) {
      uint32_t b = 0;
      if (lane == 0) b = atomicAdd(&bnext, 1u);
      b = __shfl_sync(0xffffffffu, b, 0);
      if (b >= total) break;
      int w = 0;
#pragma unroll
      for (int t = 0; t < kCullWarps - 1; ++t)
        if (w == t && b >= nb[t]) b -= nb[t], w = t + 1;
      const int e = (int)b * 32 + lane;
      const bool active = e < (int)wn[w];
      const int slot = c_lo + (int)wlist[w][active ? e : 0];  // idle lanes shadow entry 0 (and add nothing)
      float r[kRecFields];
      load_rec(a.rec, slot, r);
      const int ct = active ? (int)a.col[slot] : -1;
      const float* wp = wpts[w];
      const uint32_t* wm = wmask[w];
      const int64_t base = (int64_t)(group * kCullWarps + w) * kCullTile;
      // one formula at a time, all lanes in step (the candidates are sorted by type: a batch rarely holds more than one)
      if (__any_sync(0xffffffffu, ct == RSC_PLANE)) cull_narrow<RSC_PLANE>(a, wp, r, ct == RSC_PLANE, slot, base, wm, &n_exact);
      if (__any_sync(0xffffffffu, ct == RSC_SPHERE)) cull_narrow<RSC_SPHERE>(a, wp, r, ct == RSC_SPHERE, slot, base, wm, &n_exact);
      if (__any_sync(0xffffffffu, ct == RSC_CYLINDER)) cull_narrow<RSC_CYLINDER>(a, wp, r, ct == RSC_CYLINDER, slot, base, wm, &n_exact);
      if (__any_sync(0xffffffffu, ct == RSC_CONE)) cull_narrow<RSC_CONE>(a, wp, r, ct == RSC_CONE, slot, base, wm, &n_exact);
      if (__any_sync(0xffffffffu, ct == kConeWide)) cull_narrow<kConeWide>(a, wp, r, ct == kConeWide, slot, base, wm, &n_exact);
      __syncwarp();
    }
  }
  if (lane == 0 && n_surv) atomicAdd(a.stats, n_surv);
  n_exact = __reduce_add_sync(0xffffffffu, (unsigned)n_exact);
  if (lane == 0 && n_exact) atomicAdd(a.stats + 1, n_exact);
}

// float64 decisions of the in-band pairs: one thread per pair, all lanes busy
__global__ void __launch_bounds__(256) cull_pair_kernel(const __grid_constant__ CullArgs a) {
  const uint32_t n = *a.pn < a.pcap ? *a.pn : a.pcap;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint2 e = a.pairs[i];
    const int64_t j = (int64_t)e.y;
    if (cull_exact(a.cands + a.orig[e.x], &a.th, &a.ps, j)) {
      const int o = a.orig[e.x];
      atomicAdd(a.cv + o, 1);
      if ((a.ps.enabled[j >> 5] >> (j & 31)) & 1u) atomicAdd(a.ce + o, 1);
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && n) atomicAdd(a.stats + 1, (unsigned long long)n);
}

__global__ void cull_policy_kernel(const rsc_cand* __restrict__ cands, int C, const int32_t* __restrict__ cv,
                                   const int32_t* __restrict__ ce, uint32_t honour_enabled, int32_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= C) return;
  out[i] = ((honour_enabled >> cands[i].type) & 1u) ? ce[i] : cv[i];
}

// Morton-ordered copy of the cloud + tile spheres, kept with the flattened octree (dropped with it)
static int32_t cull_prepare(rsc_cloud* cloud, cudaStream_t st) {
  rsc_ctx* ctx = cloud->ctx;
  rsc_cells& c = cloud->cells;
  if (c.msoa) return RSC_OK;
  RSC_CUDA(ctx, cudaMalloc(&c.msoa, (size_t)6 * cloud->n_pad * sizeof(float)));
  cudaError_t e = cudaMalloc(&c.tiles, cull_sphere_count(cloud->n_pad) * sizeof(float4));
  if (e != cudaSuccess) {
    cudaFree(c.msoa);
    c.msoa = nullptr;
    return fail_cuda(ctx, e, "score_culled: cudaMalloc");
  }
  if (cloud->exact()) {  // the map of the Morton copy into the float64 coordinates
    e = cudaMalloc(&c.perm64, (size_t)cloud->n * sizeof(int64_t));
    if (e != cudaSuccess) {
      cudaFree(c.msoa), cudaFree(c.tiles);
      c.msoa = nullptr, c.tiles = nullptr;
      return fail_cuda(ctx, e, "score_culled: cudaMalloc");
    }
    widen_u32_kernel<<<(unsigned)((cloud->n + 255) / 256), 256, 0, st>>>(c.perm, cloud->n, c.perm64);
    RSC_CUDA(ctx, cudaGetLastError());
  }
  morton_gather_kernel<<<(unsigned)((cloud->n_pad + 255) / 256), 256, 0, st>>>(cloud->soa, cloud->n_pad, c.perm, cloud->n, c.msoa);
  RSC_CUDA(ctx, cudaGetLastError());
  PointSet ps;
  ps.x = c.msoa, ps.y = c.msoa + cloud->n_pad, ps.z = c.msoa + 2 * cloud->n_pad;
  ps.n = cloud->n, ps.n_pad = cloud->n_pad;
  return cull_tile_spheres(ctx, ps, reinterpret_cast<float4*>(c.tiles), st);
}

// bounding spheres of a point set that already is in a spatially coherent order: n_pad / 128 tile spheres, then
// n_pad / 512 group spheres, then ceil(n_pad / 4096) block spheres (`tiles` holds cull_sphere_count(n_pad) entries)
size_t cull_sphere_count(int64_t n_pad) {
  return (size_t)(n_pad / kCullTile + n_pad / kCullGroup + (n_pad / kCullGroup + kCullBlockGroups - 1) / kCullBlockGroups);
}

int32_t cull_tile_spheres(rsc_ctx* ctx, const PointSet& ps, float4* tiles, cudaStream_t st, const unsigned long long* d_n) {
  const int ntiles = (int)(ps.n_pad / kCullTile), ngroups = (int)(ps.n_pad / kCullGroup);
  const int nblocks = (ngroups + kCullBlockGroups - 1) / kCullBlockGroups;
  if (ntiles == 0) return RSC_OK;
  tile_sphere_kernel<<<(ntiles + 7) / 8, 256, 0, st>>>(ps.x, ps.y, ps.z, ps.n, kCullTile, ntiles, tiles, d_n);
  RSC_CUDA(ctx, cudaGetLastError());
  tile_sphere_kernel<<<(ngroups + 7) / 8, 256, 0, st>>>(ps.x, ps.y, ps.z, ps.n, kCullGroup, ngroups, tiles + ntiles, d_n);
  RSC_CUDA(ctx, cudaGetLastError());
  tile_sphere_kernel<<<(nblocks + 7) / 8, 256, 0, st>>>(ps.x, ps.y, ps.z, ps.n, kCullGroup * kCullBlockGroups, nblocks,
                                                        tiles + ntiles + ngroups, d_n);
  RSC_CUDA(ctx, cudaGetLastError());
  return RSC_OK;
}

// Enqueue the culled scoring of up to C_cap candidates on the device (their number may itself live on the
// device: d_C) against the Morton-ordered point set ps with the spheres of cull_tile_spheres.  cv / ce [C_cap]
// receive the compatible real / enabled points of every candidate.  No synchronisation; d_stats (2 x u64,
// optional) gets the surviving (candidate, tile) pairs and the pairs decided in float64.
int32_t cull_enqueue(rsc_ctx* ctx, const rsc_cloud* cloud, const PointSet& ps, const float4* tiles, const Thresh& th,
                     const rsc_cand* d_cands, int C_cap, const int32_t* d_C, int32_t* cv, int32_t* ce, unsigned long long* d_stats,
                     cudaStream_t st) {
  if (C_cap <= 0) return RSC_OK;
  RSC_CUDA(ctx, cudaMemsetAsync(cv, 0, (size_t)C_cap * sizeof(int32_t), st));
  RSC_CUDA(ctx, cudaMemsetAsync(ce, 0, (size_t)C_cap * sizeof(int32_t), st));
  if (ps.n_pad <= 0) return RSC_OK;
  if (C_cap >= (1 << 24)) return fail(ctx, RSC_E_ARG, "score_culled: too many candidates");
  // scratch: [rec][orig][col][stats 2 x u64 | pn, work | hist 5 | cursor 5][block bits][pair queue]
  const int ngroups = (int)(ps.n_pad / kCullGroup), nblocks = (ngroups + kCullBlockGroups - 1) / kCullBlockGroups;
  const int cwords = (C_cap + kCullThreads - 1) / kCullThreads * (kCullThreads / 32);  // whole 128-candidate ranges
  const size_t o_orig = (size_t)C_cap * kRecFields * sizeof(float);
  const size_t o_col = o_orig + (size_t)C_cap * sizeof(int32_t);
  const size_t o_ctr = (o_col + (size_t)C_cap + 15) / 16 * 16;
  const size_t o_bits = o_ctr + 96;
  const size_t o_queue = (o_bits + (size_t)nblocks * cwords * 4 + 15) / 16 * 16;
  int64_t qcap = (int64_t)((double)C_cap * (double)ps.n / 8192.0);
  qcap = qcap < (1 << 16) ? (1 << 16) : qcap > (8 << 20) ? (8 << 20) : qcap;
  RSC_CUDA(ctx, ctx->cullbuf.ensure(o_queue + (size_t)qcap * sizeof(uint2)));
  char* b = ctx->cullbuf.as<char>();
  float* d_rec = reinterpret_cast<float*>(b);
  int32_t* d_orig = reinterpret_cast<int32_t*>(b + o_orig);
  uint8_t* d_col = reinterpret_cast<uint8_t*>(b + o_col);
  unsigned long long* ctr = reinterpret_cast<unsigned long long*>(b + o_ctr);
  uint32_t* ctr32 = reinterpret_cast<uint32_t*>(ctr + 2);  // pn, work, hist[5], cursor[5]
  RSC_CUDA(ctx, cudaMemsetAsync(ctr, 0, 96, st));
  if (cloud->exact() && !ps.xyz64) return fail(ctx, RSC_E_STATE, "score_culled: a point set of an exact cloud lacks its float64 coordinates");
  Thresh thx = th;
  thx.exact_in = cloud->exact();
  cull_hist_kernel<<<(C_cap + 255) / 256, 256, 0, st>>>(d_cands, C_cap, d_C, ctr32 + 2);
  RSC_CUDA(ctx, cudaGetLastError());
  cull_compile_kernel<<<(C_cap + 127) / 128, 128, 0, st>>>(d_cands, C_cap, d_C, thx, cloud->pmax, cloud->nmax, ctr32 + 2, ctr32 + 7, d_rec,
                                                          d_col, d_orig);
  RSC_CUDA(ctx, cudaGetLastError());
  CullArgs a;
  a.ps = ps;
  a.tiles = tiles;
  a.groups = tiles + ps.n_pad / kCullTile;
  a.ngroups = ngroups;
  a.blocks = a.groups + ngroups;
  a.nblocks = nblocks, a.cwords = cwords;
  a.bbits = reinterpret_cast<uint32_t*>(b + o_bits);
  // work items = groups x candidate ranges: at most kCullSuper candidates each, fewer when the point set is small
  // (enough items to balance the persistent grid)
  const int cap = ctx->sm_count * kCullMinB;
  int per = kCullSuper;
  while (per > kCullThreads && (int64_t)a.ngroups * ((C_cap + per - 1) / per) < 8ll * cap) per /= 2;
  a.cands_per_range = per;
  a.nranges = (C_cap + per - 1) / per;
  a.rec = d_rec, a.col = d_col, a.orig = d_orig, a.cands = d_cands, a.d_C = d_C;
  a.th = thx;
  a.C = C_cap;
  a.cv = cv, a.ce = ce;
  a.stats = d_stats ? d_stats : ctr;
  a.pn = ctr32;
  a.work = ctr32 + 1;
  a.pairs = reinterpret_cast<uint2*>(b + o_queue);
  a.pcap = (uint32_t)qcap;
  // in-band pairs: queued for cull_pair_kernel (default) or decided on the spot (RSC_CULL_INLINE=1) -- both
  // validated against the dense path (tests/test_cull_gpu.py)
  a.inline_fp64 = getenv("RSC_CULL_INLINE") ? atoi(getenv("RSC_CULL_INLINE")) : 0;
  const int64_t items = (int64_t)a.ngroups * a.nranges;
  const int grid = (int)(items < cap ? items : cap);
  {
    const int64_t warps = (int64_t)nblocks * cwords;
    cull_block_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, st>>>(a);
    RSC_CUDA(ctx, cudaGetLastError());
  }
  cull_score_kernel<<<grid, kCullThreads, 0, st>>>(a);
  RSC_CUDA(ctx, cudaGetLastError());
  cull_pair_kernel<<<ctx->sm_count * 4, 256, 0, st>>>(a);
  RSC_CUDA(ctx, cudaGetLastError());
  return RSC_OK;
}

// did the dense path's guard-band queues overflow? (same test as rsc_loop.cuh::queue_overflow_kernel)
__global__ void dense_overflow_kernel(const uint32_t* __restrict__ wl_count, uint32_t cap, int32_t* __restrict__ out) {
  *out = (wl_count[0] > cap || wl_count[1] > cap) ? 1 : 0;
}

// K2 of the loops (see rsc_common.cuh).  Cross-over: the dense kernel scores ~1.6e12 pairs/s after ~40 us of fixed
// cost; the culled one pays ~25 us of fixed cost plus a broad phase per (candidate, 512-point group) -- it wins
// once a batch holds a few hundred candidates on a subset of a few hundred thousand points.
int32_t loop_score_new(rsc_ctx* ctx, rsc_cloud* cloud, rsc_subset& sub, const PointSet& ps, bool whole_subset, const Thresh& th,
                       const rsc_cand* d_cands, int n_new, int32_t* cv, int32_t* ce, int32_t* d_ovf, cudaStream_t st) {
  // (read per call: tests switch it between runs)
  const int mode = getenv("RSC_LOOP_CULL") ? atoi(getenv("RSC_LOOP_CULL")) : 1;  // 0: never, 1: when it pays, 2: always
  const double min_evals = getenv("RSC_LOOP_CULL_MIN") ? atof(getenv("RSC_LOOP_CULL_MIN")) : 4e8;
  // a subset without a Morton view yet: building one (a sort of the subset, four allocations) only pays for really
  // large batches -- the cell sampler's (>= 5e9 pairs each on c4); c5's root-cell batches of ~3e8-6e8 pairs stay dense
  const double need = sub.csoa ? min_evals : 10.0 * min_evals;
  const bool cull = mode != 0 && whole_subset && n_new > 0 && sub.m > 0 && (mode == 2 || (double)n_new * (double)sub.m >= need);
  if (!cull) {
    if (int32_t rc = score_enqueue(ctx, cloud, ps, th, d_cands, n_new, nullptr, false, st, cv, ce)) return rc;
    if (d_ovf) {
      dense_overflow_kernel<<<1, 1, 0, st>>>(ctx->wl_count.as<uint32_t>(), (uint32_t)ctx->wl_cap, d_ovf);
      RSC_CUDA(ctx, cudaGetLastError());
    }
    return RSC_OK;
  }
  if (int32_t rc = subset_cull_view(cloud, sub, st)) return rc;
  if (int32_t rc = cull_enqueue(ctx, cloud, view_subset_morton(&sub), reinterpret_cast<const float4*>(sub.ctiles), th, d_cands, n_new, nullptr, cv, ce, nullptr, st))
    return rc;
  if (d_ovf) RSC_CUDA(ctx, cudaMemsetAsync(d_ovf, 0, 4, st));  // nothing can overflow: pairs beyond the queue are decided inline
  ctx->stats.score_launches += 1;
  ctx->stats.evals += (int64_t)n_new * sub.m;
  ctx->stats.cands_scored += n_new;
  return RSC_OK;
}

}  // namespace rsc

using namespace rsc;

static int32_t score_culled_impl(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cands, int32_t C, int32_t subset_id,
                                 int32_t* counts, int64_t* pairs_total, int64_t* pairs_survived, double* kernel_ms) {
  rsc_ctx* ctx = cloud->ctx;
  if (!params) return fail(ctx, RSC_E_ARG, "score_culled: params is null");
  if (C < 0 || (C > 0 && (!cands || !counts))) return fail(ctx, RSC_E_ARG, "score_culled: null candidates/counts");
  for (int t = 0; t < RSC_NTYPES; ++t)
    if (!(params->eps[t] == params->eps[t]) || !(params->alpha[t] == params->alpha[t]))
      return fail(ctx, RSC_E_ARG, "params: NaN threshold");
  for (int i = 0; i < C; ++i)
    if (cands[i].type < 0 || cands[i].type >= RSC_NTYPES) return fail(ctx, RSC_E_ARG, "score_culled: unknown shape type");
  if (pairs_total) *pairs_total = 0;
  if (pairs_survived) *pairs_survived = 0;
  if (kernel_ms) *kernel_ms = 0.0;
  if (C == 0) return RSC_OK;
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if (int32_t rc = cloud_ready(cloud)) return rc;
  cudaStream_t st = ctx->stream;
  PointSet ps;
  const float4* tiles = nullptr;
  if (subset_id < 0) {
    if (cloud->cells.nlevels == 0) return fail(ctx, RSC_E_STATE, "score_culled: needs rsc_cloud_build_cells (Morton order) first");
    if (int32_t rc = cull_prepare(cloud, st)) return rc;
    if (int32_t rc = cells_refresh_enabled(cloud, st)) return rc;
    const float* m = cloud->cells.msoa;
    ps.x = m, ps.y = m + cloud->n_pad, ps.z = m + 2 * cloud->n_pad;
    ps.nx = m + 3 * cloud->n_pad, ps.ny = m + 4 * cloud->n_pad, ps.nz = m + 5 * cloud->n_pad;
    ps.enabled = cloud->cells.en_sorted, ps.valid = nullptr;
    ps.n = cloud->n, ps.n_pad = cloud->n_pad;
    ps.xyz64 = cloud->xyz64, ps.nrm64 = cloud->nrm64, ps.map = cloud->cells.perm64;
    tiles = reinterpret_cast<const float4*>(cloud->cells.tiles);
  } else {
    if ((size_t)subset_id >= cloud->subsets.size() || !cloud->subsets[subset_id].soa)
      return fail(ctx, RSC_E_ARG, "score_culled: subset has not been uploaded");
    rsc_subset& sub = cloud->subsets[subset_id];
    if (int32_t rc = subset_cull_view(cloud, sub, st)) return rc;
    ps = view_subset_morton(&sub);
    tiles = reinterpret_cast<const float4*>(sub.ctiles);
  }
  const Thresh th = make_thresh(params);
  // scratch: [cands][cv][ce][policy][stats]
  const size_t o_cv = (size_t)C * sizeof(rsc_cand);
  const size_t o_stats = (o_cv + (size_t)3 * C * sizeof(int32_t) + 15) / 16 * 16;
  RSC_CUDA(ctx, ctx->misc.ensure(o_stats + 16));
  char* b = ctx->misc.as<char>();
  rsc_cand* d_c = reinterpret_cast<rsc_cand*>(b);
  int32_t* d_cv = reinterpret_cast<int32_t*>(b + o_cv);
  unsigned long long* d_stats = reinterpret_cast<unsigned long long*>(b + o_stats);
  RSC_CUDA(ctx, cudaMemcpyAsync(d_c, cands, (size_t)C * sizeof(rsc_cand), cudaMemcpyHostToDevice, st));
  RSC_CUDA(ctx, cudaMemsetAsync(d_stats, 0, 16, st));
  RSC_CUDA(ctx, cudaEventRecord(ctx->evk0, st));
  if (int32_t rc = cull_enqueue(ctx, cloud, ps, tiles, th, d_c, C, nullptr, d_cv, d_cv + C, d_stats, st)) return rc;
  RSC_CUDA(ctx, cudaEventRecord(ctx->evk1, st));
  cull_policy_kernel<<<(C + 255) / 256, 256, 0, st>>>(d_c, C, d_cv, d_cv + C, th.honour_enabled, d_cv + 2 * (size_t)C);
  RSC_CUDA(ctx, cudaGetLastError());
  unsigned long long hs[2] = {0, 0};
  RSC_CUDA(ctx, cudaMemcpyAsync(counts, d_cv + 2 * (size_t)C, (size_t)C * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaMemcpyAsync(hs, d_stats, sizeof(hs), cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaStreamSynchronize(st));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, ctx->evk0, ctx->evk1);
  if (kernel_ms) *kernel_ms = ms;
  if (pairs_total) *pairs_total = (int64_t)C * (ps.n_pad / kCullTile);
  if (pairs_survived) *pairs_survived = (int64_t)hs[0];
  ctx->stats.evals += (int64_t)C * ps.n;
  ctx->stats.cands_scored += C;
  ctx->stats.exact_pairs += (int64_t)hs[1];
  return RSC_OK;
}

extern "C" int32_t rsc_score_culled(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cands, int32_t C, int32_t* counts,
                                    int64_t* pairs_total, int64_t* pairs_survived, double* kernel_ms) {
  if (!cloud) return RSC_E_ARG;
  return score_culled_impl(cloud, params, cands, C, -1, counts, pairs_total, pairs_survived, kernel_ms);
}

extern "C" int32_t rsc_score_culled_subset(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cands, int32_t C, int32_t subset_id,
                                           int32_t* counts, int64_t* pairs_total, int64_t* pairs_survived, double* kernel_ms) {
  if (!cloud) return RSC_E_ARG;
  if (subset_id < 0) return fail(cloud->ctx, RSC_E_ARG, "score_culled_subset: subset_id must be >= 0");
  return score_culled_impl(cloud, params, cands, C, subset_id, counts, pairs_total, pairs_survived, kernel_ms);
}
