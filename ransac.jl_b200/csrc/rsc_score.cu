// rsc_score.cu -- K2: candidate x point compatibility scoring (the hot kernel), the candidate
// compiler that feeds it, and the FP64 fix-up of guard-band pairs.
//
// Replaces scorecandidates!/scorecandidate/compatibles* (fitting.jl:181-190, plane.jl:61-130,
// sphere.jl:118-172, cylinder.jl:172-221, cone.jl:132-167).
//
// Mapping (B200-first, the path is FP32-issue bound):
//   * candidates are register resident: every thread owns K compiled candidates of ONE column type
//     (plane, sphere, cylinder, cone, wide cone; a CTA column = 128*K "slots" of one type, one kernel
//     per type, so no warp ever diverges on the type), evaluated as K/2 packed pairs (FFMA2);
//   * points stream HBM (SoA rows) -> warp-private shared-memory stages by TMA bulk copies
//     (cp.async.bulk + mbarrier, no CTA barrier in the loop) and are read back as warp-wide BROADCAST
//     128-bit loads: 6 LDS per 4 points feed K*32*4 evaluations per warp;
//   * the inlier bit of each evaluation (sign of its margin) is funnel-shifted into a per-candidate
//     register (one 32-bit mask word per 32 points), so counting is one POPC per 32 evaluations and
//     bitmasks come for free;
//   * per evaluation the kernel also tracks min|margin|; a 32-point group whose minimum falls inside
//     the FP32 guard band is queued, re-scanned (fixup_scan_kernel) and its ambiguous pairs are
//     decided in FP64 in the reference's operation order (fixup_pair_kernel).
// DESIGN.md section 3 has the measurements behind these choices and the register-bank analysis of
// what bounds the kernel.
#include <math.h>
#include <stdlib.h>

#include "rsc_eval.cuh"
#include "rsc_exact.cuh"

namespace rsc {

// a 32-point group of one candidate whose min|margin| fell inside the FP32 guard band: the fix-up
// kernel re-derives the reference's (float64) decision for its 32 points and corrects count/mask
struct GroupTask {
  uint32_t cand;   // original candidate index
  uint32_t group;  // 32-point group index in the point set
  uint32_t word;   // the FP32 decision bits the tiled kernel used (before enabled/valid gating)
  uint32_t slot_type;  // slot | (shape type << 28): saves the fix-up two dependent lookups
};

struct ScoreArgs {
  PointSet ps;
  Thresh th;
  const float* rec;        // [kRecFields][cslots]
  const int32_t* orig;     // [cslots] original candidate index, -1 for padding slots
  const BlockTab* tab;     // [gridDim.x]
  int32_t cslots;          // slot stride of rec / masks
  int32_t subs_per_chunk;  // 128-point sub-tiles per CTA row
  int32_t nsubs;
  int32_t* counts_valid;   // [C] compatible real points
  int32_t* counts_enabled; // [C] compatible enabled points
  uint32_t* masks;         // nullable, group-major [n_pad/32][cslots]
  GroupTask* wl;
  uint32_t* wl_count;
  uint32_t wl_cap;
};

constexpr int kSub = 128;                       // points per warp-private sub-tile
constexpr int kStages = 2;                      // sub-tiles in flight per warp
constexpr int kSubFloats = 6 * kSub;            // x|y|z|nx|ny|nz rows of one sub-tile
constexpr uint32_t kSubBytes = kSubFloats * 4;  // 3072

// ---- TMA bulk copy + mbarrier (sm_90+/sm_100 PTX) ---------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// one lane: fetch one sub-tile (6 SoA rows of 128 floats, `stride` floats apart) into a warp-private stage
__device__ __forceinline__ void issue_subtile(const float* src, int64_t stride, float* stage, uint64_t* bar) {
  mbar_expect_tx(bar, kSubBytes);
#pragma unroll
  for (int f = 0; f < 6; ++f) bulk_g2s(stage + f * kSub, src + f * stride, kSub * 4, bar);
}

// K candidates per thread; for even K they are evaluated as K/2 packed pairs (FFMA2 path).
// Every WARP streams the CTA row's points through its own double-buffered shared-memory stages
// (TMA bulk copies signalled on warp-private mbarriers): there is no CTA-wide barrier in the loop.
//
// Mask words are built MSB-first (the sign bit of each margin is funnel-shifted in from the right),
// so the first point of a 32-point group ends at bit 31: counts use the bit-reversed enabled/valid
// words, and only the words that leave the thread (mask store, fix-up queue) are reversed back.
template <int T, int K, int U, bool MASKS>
__device__ __forceinline__ void score_body(const ScoreArgs& a, int slot0, float* wstage, uint64_t* wbar) {
  constexpr int NR = RecN<T>::n;
  // U = 5 / 6: SCALAR evaluation (one FFMA per candidate and point; 5 = point-major, 6 = candidate-major source
  // order) -- three 32-bit sources per instruction instead of the packed forms' 64/32/64-bit, see DESIGN.md 3
  constexpr bool kPacked = (K % 2 == 0) && U < 5;
  constexpr int KP = kPacked ? K / 2 : 1;
  // U = 3: pair-major source order (all four points of a pair, then the next pair).  ptxas schedules the
  // block itself, but from this order it finds 1-5 % better operand reuse than from point-major (U = 1);
  // a lockstep order (every formula step for the four points back to back) and eight points per pair
  // were measured and are no better.
  constexpr bool kOrderJQ = (U == 3);
  float r[kPacked ? 1 : K][NR];  // scalar records (K odd, or the scalar tilings)
  float2 r2[KP][NR];             // packed records: .x = candidate 2j, .y = candidate 2j+1
  float band[K];
  int cnte[K], cntv[K];
  const int tid = threadIdx.x, lane = tid & 31;
  const float* recp = a.rec + slot0 + tid;
#pragma unroll
  for (int k = 0; k < K; ++k) {
#pragma unroll
    for (int f = 0; f < NR; ++f) {
      const float v = recp[(size_t)f * a.cslots + k * kThreads];
      if constexpr (kPacked) {
        if (k & 1)
          r2[k / 2][f].y = v;
        else
          r2[k / 2][f].x = v;
      } else {
        r[k][f] = v;
      }
    }
    band[k] = recp[(size_t)kBandField * a.cslots + k * kThreads];
    cnte[k] = 0;
    cntv[k] = 0;
  }
  constexpr int PT = public_type(T);
  const float eps = a.th.eps[PT], cosa = a.th.cosa[PT];
  // honour: the type ANDs pc.isenabled into its inliers; otherwise (sphere, Q4) the policy count is
  // the validity-gated one and the enabled-gated count is kept beside it (the loop's "tainted" flag)
  const bool honour = (a.th.honour_enabled >> PT) & 1u;

  const int sub0 = blockIdx.y * a.subs_per_chunk;
  const int nsub = min(a.subs_per_chunk, a.nsubs - sub0);
  const uint32_t* enp = a.ps.enabled + (size_t)sub0 * (kSub / 32);
  const uint32_t* vap = a.ps.valid + (size_t)sub0 * (kSub / 32);
  uint32_t* maskp = MASKS ? a.masks + (size_t)sub0 * (kSub / 32) * a.cslots + slot0 + tid : nullptr;
  const int64_t stride = a.ps.y - a.ps.x;  // the six SoA rows are equally spaced (host-checked)
  const float* src0 = a.ps.x + (int64_t)sub0 * kSub;
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < kStages; ++s)
      if (s < nsub) issue_subtile(src0 + s * kSub, stride, wstage + s * kSubFloats, wbar + s);
  }

  // four points (6 broadcast 128-bit loads) against the thread's K candidates
  auto body4 = [&](const float* gp, uint32_t (&mask)[K], float (&mabs)[K]) {
    const float4 X = *reinterpret_cast<const float4*>(gp);
    const float4 Y = *reinterpret_cast<const float4*>(gp + kSub);
    const float4 Z = *reinterpret_cast<const float4*>(gp + 2 * kSub);
    const float4 U4 = *reinterpret_cast<const float4*>(gp + 3 * kSub);
    const float4 V = *reinterpret_cast<const float4*>(gp + 4 * kSub);
    const float4 W = *reinterpret_cast<const float4*>(gp + 5 * kSub);
    const float px[4] = {X.x, X.y, X.z, X.w}, py[4] = {Y.x, Y.y, Y.z, Y.w}, pz[4] = {Z.x, Z.y, Z.z, Z.w};
    const float nx[4] = {U4.x, U4.y, U4.z, U4.w}, ny[4] = {V.x, V.y, V.z, V.w}, nz[4] = {W.x, W.y, W.z, W.w};
    if constexpr (kPacked && U == 4) {  // lockstep over the four points (eval2x4)
#pragma unroll
      for (int j = 0; j < KP; ++j) {
        float2 m[4];
        eval2x4<T>(r2[j], px, py, pz, nx, ny, nz, eps, cosa, m);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          mask[2 * j] = __funnelshift_l(__float_as_uint(m[q].x), mask[2 * j], 1);
          mask[2 * j + 1] = __funnelshift_l(__float_as_uint(m[q].y), mask[2 * j + 1], 1);
          mabs[2 * j] = fmin_nan(mabs[2 * j], fabsf(m[q].x));
          mabs[2 * j + 1] = fmin_nan(mabs[2 * j + 1], fabsf(m[q].y));
        }
      }
      return;
    }
    if constexpr (kPacked && kOrderJQ) {
#pragma unroll
      for (int j = 0; j < KP; ++j) {
        float2 m[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) m[q] = eval2<T>(r2[j], px[q], py[q], pz[q], nx[q], ny[q], nz[q], eps, cosa);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          mask[2 * j] = __funnelshift_l(__float_as_uint(m[q].x), mask[2 * j], 1);
          mask[2 * j + 1] = __funnelshift_l(__float_as_uint(m[q].y), mask[2 * j + 1], 1);
          mabs[2 * j] = fmin_nan(mabs[2 * j], fabsf(m[q].x));
          mabs[2 * j + 1] = fmin_nan(mabs[2 * j + 1], fabsf(m[q].y));
        }
      }
      return;
    }
    if constexpr (!kPacked && U == 6) {
#pragma unroll
      for (int k = 0; k < K; ++k) {
        float m[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) m[q] = eval<T>(r[k], px[q], py[q], pz[q], nx[q], ny[q], nz[q], eps, cosa);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          mask[k] = __funnelshift_l(__float_as_uint(m[q]), mask[k], 1);
          mabs[k] = fmin_nan(mabs[k], fabsf(m[q]));
        }
      }
      return;
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if constexpr (kPacked) {
#pragma unroll
        for (int j = 0; j < KP; ++j) {
          const float2 m = eval2<T>(r2[j], px[q], py[q], pz[q], nx[q], ny[q], nz[q], eps, cosa);
          mask[2 * j] = __funnelshift_l(__float_as_uint(m.x), mask[2 * j], 1);  // sign bit = compatible
          mask[2 * j + 1] = __funnelshift_l(__float_as_uint(m.y), mask[2 * j + 1], 1);
          mabs[2 * j] = fmin_nan(mabs[2 * j], fabsf(m.x));
          mabs[2 * j + 1] = fmin_nan(mabs[2 * j + 1], fabsf(m.y));
        }
      } else {
#pragma unroll
        for (int k = 0; k < K; ++k) {
          const float m = eval<T>(r[k], px[q], py[q], pz[q], nx[q], ny[q], nz[q], eps, cosa);
          mask[k] = __funnelshift_l(__float_as_uint(m), mask[k], 1);
          mabs[k] = fmin_nan(mabs[k], fabsf(m));
        }
      }
    }
  };

  // group epilogue: counts (+ mask words); the guard-band queue is the rare path
  auto epilogue = [&](const uint32_t (&mask)[K], const float (&mabs)[K], int gi, uint32_t en, uint32_t va) {
    const uint32_t ben = __brev(en), bva = __brev(va);
    bool amb = false;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      amb |= !(mabs[k] > band[k]);
      cnte[k] += __popc(mask[k] & ben);
    }
    if (!honour) {
#pragma unroll
      for (int k = 0; k < K; ++k) cntv[k] += __popc(mask[k] & bva);
    }
    if constexpr (MASKS) {
      const uint32_t gate = honour ? en : va;
#pragma unroll
      for (int k = 0; k < K; ++k) maskp[(size_t)gi * a.cslots + k * kThreads] = __brev(mask[k]) & gate;
    }
    if (amb && va) {  // rare: hand the group(s) to the FP64 fix-up kernels
      const int64_t gw = (int64_t)sub0 * (kSub / 32) + gi;
#pragma unroll
      for (int k = 0; k < K; ++k) {
        if (mabs[k] > band[k]) continue;
        const int slot = slot0 + k * kThreads + tid;
        const int o = a.orig[slot];
        if (o < 0) continue;
        const uint32_t pos = atomicAdd(a.wl_count, 1u);
        if (pos < a.wl_cap) a.wl[pos] = GroupTask{(uint32_t)o, (uint32_t)gw, __brev(mask[k]), (uint32_t)slot | ((uint32_t)T << 28)};
      }
    }
  };

  for (int it = 0; it < nsub; ++it) {
    const int st = it % kStages;
    mbar_wait(wbar + st, (it / kStages) & 1);
    const float* sx = wstage + st * kSubFloats;
#pragma unroll 1
    for (int g = 0; g < kSub / 32; ++g) {
      uint32_t mask[K];
      float mabs[K];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        mask[k] = 0u;
        mabs[k] = __int_as_float(0x7f800000);
      }
      const float* gx = sx + g * 32;
#pragma unroll(U >= 3 ? 1 : U)
      for (int i4 = 0; i4 < 32; i4 += 4) body4(gx + i4, mask, mabs);
      const int gi = it * (kSub / 32) + g;
      epilogue(mask, mabs, gi, __ldg(enp + gi), __ldg(vap + gi));
    }
    __syncwarp();
    if (lane == 0 && it + kStages < nsub) issue_subtile(src0 + (it + kStages) * kSub, stride, wstage + st * kSubFloats, wbar + st);
  }
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const int o = a.orig[slot0 + k * kThreads + tid];
    if (o >= 0) {
      if (cnte[k]) atomicAdd(a.counts_enabled + o, cnte[k]);
      if (!honour && cntv[k]) atomicAdd(a.counts_valid + o, cntv[k]);
    }
  }
}

// One kernel per shape type (and per tiling): register allocation, occupancy and the number of
// candidates per thread are chosen per type.  The grid spans ALL columns of the block table; CTAs of
// another type's columns leave at once (the host does not know the per-type candidate counts: the
// candidates may live on the device only).
template <int T, int K, int MINB, int U, bool MASKS>
__global__ void __launch_bounds__(kThreads, MINB) score_kernel(const __grid_constant__ ScoreArgs a) {
  __shared__ __align__(128) float stages[kThreads / 32][kStages * kSubFloats];
  __shared__ __align__(8) uint64_t bars[kThreads / 32][kStages];
  const BlockTab bt = a.tab[blockIdx.x];
  if (bt.type != T) return;
  const int warp = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int s = 0; s < kStages; ++s) mbar_init(&bars[warp][s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  score_body<T, K, U, MASKS>(a, bt.slot0, stages[warp], bars[warp]);
}

// All column types in ONE launch (runtime switch per CTA column): for small batches (the device loop
// scores a few hundred new candidates per iteration) five launches plus fork/join events cost more
// host time than the kernels run.  Registers = the maximum over the types, fine at K <= 2.
template <int K, int MINB, bool MASKS>
__global__ void __launch_bounds__(kThreads, MINB) score_kernel_any(const __grid_constant__ ScoreArgs a) {
  __shared__ __align__(128) float stages[kThreads / 32][kStages * kSubFloats];
  __shared__ __align__(8) uint64_t bars[kThreads / 32][kStages];
  const BlockTab bt = a.tab[blockIdx.x];
  if (bt.type < 0) return;
  const int warp = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int s = 0; s < kStages; ++s) mbar_init(&bars[warp][s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  switch (bt.type) {
    case RSC_PLANE:
      score_body<RSC_PLANE, K, 1, MASKS>(a, bt.slot0, stages[warp], bars[warp]);
      break;
    case RSC_SPHERE:
      score_body<RSC_SPHERE, K, 1, MASKS>(a, bt.slot0, stages[warp], bars[warp]);
      break;
    case RSC_CYLINDER:
      score_body<RSC_CYLINDER, K, 1, MASKS>(a, bt.slot0, stages[warp], bars[warp]);
      break;
    case RSC_CONE:
      score_body<RSC_CONE, K, 1, MASKS>(a, bt.slot0, stages[warp], bars[warp]);
      break;
    default:
      score_body<kConeWide, K, 1, MASKS>(a, bt.slot0, stages[warp], bars[warp]);
      break;
  }
}

// ---------------------------------------------------------------------------------------------
// FP64 fix-up, two launches.
//  1. fixup_scan_kernel: one warp per queued 32-point group, one lane per point.  The FP32 margin is
//     recomputed; outside the band its sign IS the float64 reference's decision (that is what the
//     band bounds), inside the band the (candidate, point) pair is queued.
//  2. fixup_pair_kernel: one thread per queued pair, evaluated in FP64 in the reference's operation
//     order (rsc_exact.cuh) -- all lanes busy, unlike a per-group FP64 branch.
//  Both correct counts / mask bits by the difference to the bits the tiled kernel used.
// ---------------------------------------------------------------------------------------------
struct AmbPair {
  uint32_t cand_bit;  // original candidate index | (bit the tiled kernel used << 31)
  uint32_t point;
};

__device__ __forceinline__ void apply_flip(const ScoreArgs& a, uint32_t cand, int type, int slot, uint32_t pt,
                                           bool now_ok) {
  const uint32_t word = pt >> 5, bit = 1u << (pt & 31);
  const bool va = a.ps.valid[word] & bit, en = a.ps.enabled[word] & bit;
  const int d = now_ok ? 1 : -1;
  if (va) atomicAdd(a.counts_valid + cand, d);
  if (en) atomicAdd(a.counts_enabled + cand, d);
  if (a.masks) {
    const bool honour = (a.th.honour_enabled >> type) & 1u;
    if (honour ? en : va) atomicXor(a.masks + (size_t)word * a.cslots + slot, bit);
  }
}

__global__ void __launch_bounds__(256) fixup_scan_kernel(const __grid_constant__ ScoreArgs a,
                                                         const rsc_cand* __restrict__ cands,
                                                         const int32_t* __restrict__ slot_of,
                                                         AmbPair* __restrict__ pairs, uint32_t* __restrict__ npairs,
                                                         uint32_t pair_cap) {
  // queued pairs are collected per CTA in shared memory and appended with ONE global atomic per
  // flush (a global atomic per pair on a single counter serialises in L2: 4 M pairs took 3 ms)
  constexpr int kBuf = 1024;
  __shared__ AmbPair sp[kBuf];
  __shared__ uint32_t scount, sbase;
  const uint32_t n = min(*a.wl_count, a.wl_cap);
  const int lane = threadIdx.x & 31;
  const uint32_t wpb = blockDim.x >> 5, warps = gridDim.x * wpb;
  const uint32_t rounds = (n + warps - 1) / warps;
  if (threadIdx.x == 0) scount = 0;
  __syncthreads();
  for (uint32_t rd = 0; rd < rounds; ++rd) {
    const uint32_t e = rd * warps + blockIdx.x * wpb + (threadIdx.x >> 5);
    if (e < n) {
      const GroupTask tk = a.wl[e];
      const int col = (int)(tk.slot_type >> 28);  // column type: selects the evaluation form
      const int type = public_type(col);
      const int slot = (int)(tk.slot_type & 0x0fffffffu);
      float r[kRecFields];
#pragma unroll
      for (int f = 0; f < kRecFields; ++f) r[f] = a.rec[(size_t)f * a.cslots + slot];
      const uint32_t pt = tk.group * 32u + lane;
      const float m = eval_any(col, r, a.ps.x[pt], a.ps.y[pt], a.ps.z[pt], a.ps.nx[pt], a.ps.ny[pt], a.ps.nz[pt],
                               a.th.eps[type], a.th.cosa[type]);
      const bool used = (tk.word >> lane) & 1u;
      if (!(fabsf(m) > r[kBandField])) {
        const uint32_t pos = atomicAdd(&scount, 1u);  // <= 256 per round, flushed below 768
        sp[pos] = AmbPair{tk.cand | ((uint32_t)used << 31), pt};
      } else if ((m < 0.f) != used) {
        apply_flip(a, tk.cand, type, slot, pt, m < 0.f);  // only if two FP32 evaluations straddled zero
      }
    }
    __syncthreads();
    if (scount > kBuf - 256 || rd + 1 == rounds) {
      if (threadIdx.x == 0) sbase = atomicAdd(npairs, scount);
      __syncthreads();
      for (uint32_t i = threadIdx.x; i < scount; i += blockDim.x)
        if (sbase + i < pair_cap) pairs[sbase + i] = sp[i];
      __syncthreads();
      if (threadIdx.x == 0) scount = 0;
      __syncthreads();
    }
  }
}

__global__ void __launch_bounds__(256) fixup_pair_kernel(const __grid_constant__ ScoreArgs a,
                                                         const rsc_cand* __restrict__ cands,
                                                         const ex::ConeTrig* __restrict__ trig,
                                                         const int32_t* __restrict__ slot_of,
                                                         const AmbPair* __restrict__ pairs,
                                                         const uint32_t* __restrict__ npairs, uint32_t pair_cap) {
  const uint32_t n = min(*npairs, pair_cap);
  for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
    const AmbPair pr = pairs[e];
    const uint32_t cand = pr.cand_bit & 0x7fffffffu;
    const bool used = pr.cand_bit >> 31;
    const rsc_cand c = cands[cand];
    ex::ConeTrig tr{1.0, 0.0};
    if (c.type == RSC_CONE) {
      if (trig) {
        tr = trig[cand];
      } else {
        tr.ct = cos(-c.p[6] / 2);
        tr.st = sin(-c.p[6] / 2);
      }
    }
    const uint32_t pt = pr.point;
    ex::V3 P, N;
    ex::point64(a.ps, pt, &P, &N);
    const bool ok = ex::compat(c, tr, a.th, P, N);
    if (ok != used) apply_flip(a, cand, c.type, slot_of[cand], pt, ok);
  }
}

// counts[c] = enabled-gated or validity-gated count, by the type's policy (Q4)
__global__ void select_counts_kernel(const rsc_cand* __restrict__ cands, int C,
                                     const int32_t* __restrict__ cv, const int32_t* __restrict__ ce,
                                     uint32_t honour_enabled, int32_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= C) return;
  const int t = cands[i].type;
  const bool honour = (t >= 0 && t < RSC_NTYPES) ? ((honour_enabled >> t) & 1u) : true;
  out[i] = honour ? ce[i] : cv[i];
}

// ---------------------------------------------------------------------------------------------
// candidate compiler: FP64 rsc_cand[C] -> type-segmented FP32 records + the CTA column table.
// One CTA; slots are assigned stably (candidate order within a type is kept).
// Column order is cone, cylinder, sphere, plane: the most expensive columns are scheduled first.
// ---------------------------------------------------------------------------------------------
struct ColSlots {
  int v[kColTypes];  // slots per CTA column (= 128 x candidates per thread) of each column type
};

__global__ void __launch_bounds__(1024) compile_kernel(const rsc_cand* __restrict__ cands, int C, const Thresh th,
                                                       const ColSlots spcs, int cslots,
                                                       int ncols, float pmax, float nmax,
                                                       const uint32_t* __restrict__ d_bounds,
                                                       float* __restrict__ rec, int32_t* __restrict__ orig,
                                                       int32_t* __restrict__ slot_of,
                                                       BlockTab* __restrict__ tab) {
  __shared__ int cnt[kColTypes], off[kColTypes], run[kColTypes], tot[kColTypes];
  __shared__ int wcnt[kColTypes][32], woff[kColTypes][32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (d_bounds) {  // scales of the chunk being scored, still on the device (chunked upload)
    pmax = sqrtf(__uint_as_float(d_bounds[0])) * 1.000001f;
    nmax = sqrtf(__uint_as_float(d_bounds[1])) * 1.000001f;
  }
  if (tid < kColTypes) {
    cnt[tid] = 0;
    run[tid] = 0;
  }
  __syncthreads();
  for (int i = tid; i < C; i += blockDim.x) {
    const int t = cands[i].type;
    if (t >= 0 && t < RSC_NTYPES) atomicAdd(&cnt[col_type(cands[i])], 1);
  }
  __syncthreads();
  if (tid == 0) {
    const int order[kColTypes] = {kConeWide, RSC_CONE, RSC_CYLINDER, RSC_SPHERE, RSC_PLANE};
    int s = 0, col = 0;
    for (int oi = 0; oi < kColTypes; ++oi) {
      const int t = order[oi];
      off[t] = s;
      const int spc = spcs.v[t];
      const int nb = (cnt[t] + spc - 1) / spc;
      for (int b = 0; b < nb && col < ncols; ++b) tab[col++] = BlockTab{t, s + b * spc};
      s += nb * spc;
    }
    for (; col < ncols; ++col) tab[col] = BlockTab{-1, 0};
  }
  __syncthreads();
  for (int base = 0; base < C; base += blockDim.x) {
    const int i = base + tid;
    int t = -1;
    if (i < C) {
      t = cands[i].type;
      t = (t < 0 || t >= RSC_NTYPES) ? -1 : col_type(cands[i]);
    }
    int myrank = 0;
#pragma unroll
    for (int tt = 0; tt < kColTypes; ++tt) {
      const unsigned b = __ballot_sync(0xffffffffu, t == tt);
      if (t == tt) myrank = __popc(b & ((1u << lane) - 1u));
      if (lane == 0) wcnt[tt][warp] = __popc(b);
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
      for (int tt = 0; tt < kColTypes; ++tt) {
        const int v = wcnt[tt][lane];
        int inc = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const int o = __shfl_up_sync(0xffffffffu, inc, d);
          if (lane >= d) inc += o;
        }
        woff[tt][lane] = inc - v;
        if (lane == 31) tot[tt] = inc;
      }
    }
    __syncthreads();
    if (i < C) {
      if (t >= 0) {
        const int slot = off[t] + run[t] + woff[t][warp] + myrank;
        float r[kRecFields];
        compile_record(cands[i], t, th, pmax, nmax, r);
#pragma unroll
        for (int f = 0; f < kRecFields; ++f) rec[(size_t)f * cslots + slot] = r[f];
        orig[slot] = i;
        slot_of[i] = slot;
      } else {
        slot_of[i] = -1;
      }
    }
    __syncthreads();
    if (tid < kColTypes) run[tid] += tot[tid];
    __syncthreads();
  }
  // padding slots replicate the last real candidate of their type (orig = -1: results dropped)
  for (int t = 0; t < kColTypes; ++t) {
    const int n = cnt[t];
    if (n == 0) continue;
    const int spc = spcs.v[t];
    const int padded = ((n + spc - 1) / spc) * spc;
    const int src = off[t] + n - 1;
    for (int s = n + tid; s < padded; s += blockDim.x) {
      const int dst = off[t] + s;
#pragma unroll
      for (int f = 0; f < kRecFields; ++f) rec[(size_t)f * cslots + dst] = rec[(size_t)f * cslots + src];
      orig[dst] = -1;
    }
  }
}

// group-major [G][cslots] -> candidate-major [C][words] (32x32 tiles through shared memory)
__global__ void __launch_bounds__(1024) masks_transpose_kernel(const uint32_t* __restrict__ gm,
                                                               const int32_t* __restrict__ slot_of,
                                                               int C, int cslots, int64_t words,
                                                               uint32_t* __restrict__ out) {
  __shared__ uint32_t t[32][33];
  const int c0 = blockIdx.x * 32;
  const int64_t g0 = (int64_t)blockIdx.y * 32;
  {  // read: lanes run over candidates (slots are near-contiguous), rows over groups
    const int c = c0 + threadIdx.x;
    const int64_t g = g0 + threadIdx.y;
    uint32_t v = 0;
    if (c < C && g < words) {
      const int s = slot_of[c];
      if (s >= 0) v = gm[(size_t)g * cslots + s];
    }
    t[threadIdx.y][threadIdx.x] = v;
  }
  __syncthreads();
  {
    const int c = c0 + threadIdx.y;
    const int64_t g = g0 + threadIdx.x;
    if (c < C && g < words) out[(size_t)c * words + g] = t[threadIdx.x][threadIdx.y];
  }
}

// ---------------------------------------------------------------------------------------------
// host-side launchers
// ---------------------------------------------------------------------------------------------
Thresh make_thresh(const rsc_params* p) {
  Thresh th;
  for (int t = 0; t < RSC_NTYPES; ++t) {
    th.eps_d[t] = p->eps[t];
    th.cosa_d[t] = cos(p->alpha[t]);
    th.eps[t] = (float)th.eps_d[t];
    th.cosa[t] = (float)th.cosa_d[t];
  }
  th.honour_enabled = 0xFu;
  if (p->compat_flags & RSC_COMPAT_SPHERE_IGNORES_ENABLED) th.honour_enabled &= ~(1u << RSC_SPHERE);
  return th;
}

// ---- tiling table -----------------------------------------------------------------------------
// (K candidates per thread, CTAs per SM, points unrolled x4) per shape type.  The defaults were
// picked on a B200 with tools/tune_score.py; RSC_CFG_<PLANE|SPHERE|CYLINDER|CONE>="K,MINB,U"
// overrides one type (tuning hook, read on every call).
using ScoreFn = void (*)(const ScoreArgs);
struct Tiling {
  int K, minb, U;
  ScoreFn fn[kColTypes];       // counts only
  ScoreFn fn_masks[kColTypes]; // counts + packed inlier bitmasks
};
#define RSC_TILING(K, MINB, U)                                                                          \
  Tiling {                                                                                              \
    K, MINB, U,                                                                                         \
        {score_kernel<RSC_PLANE, K, MINB, U, false>, score_kernel<RSC_SPHERE, K, MINB, U, false>,       \
         score_kernel<RSC_CYLINDER, K, MINB, U, false>, score_kernel<RSC_CONE, K, MINB, U, false>,      \
         score_kernel<kConeWide, K, MINB, U, false>},                                                   \
    {                                                                                                   \
      score_kernel<RSC_PLANE, K, MINB, U, true>, score_kernel<RSC_SPHERE, K, MINB, U, true>,            \
          score_kernel<RSC_CYLINDER, K, MINB, U, true>, score_kernel<RSC_CONE, K, MINB, U, true>,       \
          score_kernel<kConeWide, K, MINB, U, true>                                                     \
    }                                                                                                   \
  }
#ifdef RSC_EXP_K  // quick single-tiling builds for tools/sass_model.py: nvcc -DRSC_EXP_K=4 -DRSC_EXP_MINB=3 -DRSC_EXP_U=4
static const Tiling kTilings[] = {RSC_TILING(1, 4, 1), RSC_TILING(RSC_EXP_K, RSC_EXP_MINB, RSC_EXP_U)};
#else
static const Tiling kTilings[] = {
    RSC_TILING(1, 4, 1), RSC_TILING(2, 4, 1), RSC_TILING(4, 3, 1), RSC_TILING(4, 4, 1), RSC_TILING(8, 2, 1), RSC_TILING(4, 4, 3), RSC_TILING(4, 3, 3),
    RSC_TILING(4, 4, 5), RSC_TILING(4, 3, 5), RSC_TILING(4, 4, 6), RSC_TILING(4, 3, 6), RSC_TILING(8, 2, 5),
};
#endif
static const Tiling* find_tiling(int K, int minb, int U) {
  for (const Tiling& t : kTilings)
    if (t.K == K && t.minb == minb && t.U == U) return &t;
  return nullptr;
}

// K by problem size: few candidates -> fewer per thread, so that there are columns to spread over
static int cap_k(int C) { return C >= 3072 ? 8 : (C >= 768 ? 2 : 1); }

static const Tiling* pick_tiling(int type, int C) {
  static const char* names[kColTypes] = {"RSC_CFG_PLANE", "RSC_CFG_SPHERE", "RSC_CFG_CYLINDER", "RSC_CFG_CONE", "RSC_CFG_CONE"};
  static const int dflt[kColTypes][3] = {{4, 4, 3}, {4, 3, 3}, {4, 3, 3}, {4, 3, 3}, {4, 3, 3}};  // plane, sphere, cylinder, cone, wide cone
  int K = dflt[type][0], minb = dflt[type][1], U = dflt[type][2];
  if (const char* e = getenv(names[type])) {
    int a = 0, b = 0, c = 0;
    if (sscanf(e, "%d,%d,%d", &a, &b, &c) == 3 && find_tiling(a, b, c)) K = a, minb = b, U = c;
  }
  const int kc = cap_k(C);
  if (K > kc) {
    K = kc;
    minb = 4, U = 1;
  }
  return find_tiling(K, minb, U);
}

// layout of the compiled records for C candidates: per-type slots per column, total slot stride
struct SlotLayout {
  const Tiling* til[kColTypes];
  ColSlots spcs;
  int ncols, cslots;
};
static SlotLayout slot_layout(int C) {
  SlotLayout L;
  int min_spc = 1 << 30, sum_spc = 0;
  for (int t = 0; t < kColTypes; ++t) {
    L.til[t] = pick_tiling(t, C);
    L.spcs.v[t] = kThreads * L.til[t]->K;
    min_spc = min(min_spc, L.spcs.v[t]);
    sum_spc += L.spcs.v[t];
  }
  L.ncols = (C + min_spc - 1) / min_spc + kColTypes;
  L.cslots = ((C + sum_spc + 127) / 128) * 128;  // sum over types of ceil(cnt_t / spc_t) * spc_t <= C + sum spc_t
  return L;
}

int32_t score_enqueue(rsc_ctx* ctx, const rsc_cloud* cloud, const PointSet& ps, const Thresh& th,
                      const rsc_cand* d_cands, int32_t C, int32_t* d_counts_policy, bool want_masks,
                      cudaStream_t st, int32_t* d_counts_valid, int32_t* d_counts_enabled,
                      const double* d_trig, const uint32_t* d_bounds, bool accumulate) {
  if (C <= 0) return RSC_OK;
  if (ps.n_pad <= 0) {  // an empty slice (a rank without points of this set): zero counts, empty queues
    RSC_CUDA(ctx, ctx->counts.ensure((size_t)2 * C * sizeof(int32_t)));
    RSC_CUDA(ctx, ctx->wl_count.ensure(16));
    int32_t* cv0 = d_counts_valid ? d_counts_valid : ctx->counts.as<int32_t>();
    int32_t* ce0 = d_counts_enabled ? d_counts_enabled : ctx->counts.as<int32_t>() + C;
    if (!accumulate) {
      RSC_CUDA(ctx, cudaMemsetAsync(cv0, 0, (size_t)C * sizeof(int32_t), st));
      RSC_CUDA(ctx, cudaMemsetAsync(ce0, 0, (size_t)C * sizeof(int32_t), st));
    }
    RSC_CUDA(ctx, cudaMemsetAsync(ctx->wl_count.p, 0, 2 * sizeof(uint32_t), st));
    if (d_counts_policy) RSC_CUDA(ctx, cudaMemsetAsync(d_counts_policy, 0, (size_t)C * sizeof(int32_t), st));
    return RSC_OK;
  }
  if (ps.n_pad >= ((int64_t)1 << 32)) return fail(ctx, RSC_E_ARG, "point set too large for one shard (>= 2^32)");
  {
    const int64_t sd = ps.y - ps.x;
    if (ps.z - ps.y != sd || ps.nx - ps.z != sd || ps.ny - ps.nx != sd || ps.nz - ps.ny != sd)
      return fail(ctx, RSC_E_ARG, "score: the six SoA rows of the point set must be equally spaced");
  }
  const SlotLayout L = slot_layout(C);
  const int ncols = L.ncols, cslots = L.cslots;
  ctx->last_cslots = cslots;
  const int nsubs = (int)(ps.n_pad / kSub);
  const int64_t groups = ps.n_pad / 32;

  RSC_CUDA(ctx, ctx->rec.ensure((size_t)kRecFields * cslots * sizeof(float)));
  RSC_CUDA(ctx, ctx->orig.ensure((size_t)cslots * sizeof(int32_t)));
  RSC_CUDA(ctx, ctx->slot_of.ensure((size_t)C * sizeof(int32_t)));
  RSC_CUDA(ctx, ctx->blktab.ensure((size_t)ncols * sizeof(BlockTab)));
  RSC_CUDA(ctx, ctx->counts.ensure((size_t)2 * C * sizeof(int32_t)));
  RSC_CUDA(ctx, ctx->worklist.ensure(ctx->wl_cap * sizeof(GroupTask)));
  RSC_CUDA(ctx, ctx->wl_count.ensure(16));
  if (want_masks) RSC_CUDA(ctx, ctx->masks_gm.ensure((size_t)groups * cslots * sizeof(uint32_t)));

  int32_t* cv = d_counts_valid ? d_counts_valid : ctx->counts.as<int32_t>();
  int32_t* ce = d_counts_enabled ? d_counts_enabled : ctx->counts.as<int32_t>() + C;
  if (!accumulate) {
    RSC_CUDA(ctx, cudaMemsetAsync(cv, 0, (size_t)C * sizeof(int32_t), st));
    RSC_CUDA(ctx, cudaMemsetAsync(ce, 0, (size_t)C * sizeof(int32_t), st));
  }
  RSC_CUDA(ctx, ctx->pairs.ensure(ctx->wl_cap * 8));
  RSC_CUDA(ctx, cudaMemsetAsync(ctx->wl_count.p, 0, 2 * sizeof(uint32_t), st));

  if (cloud->exact() && !ps.xyz64) return fail(ctx, RSC_E_STATE, "score: a point set of an exact cloud lacks its float64 coordinates");
  Thresh thx = th;
  thx.exact_in = cloud->exact();
  compile_kernel<<<1, 1024, 0, st>>>(d_cands, C, thx, L.spcs, cslots, ncols, cloud->pmax, cloud->nmax, d_bounds,
                                     ctx->rec.as<float>(), ctx->orig.as<int32_t>(),
                                     ctx->slot_of.as<int32_t>(), ctx->blktab.as<BlockTab>());
  RSC_CUDA(ctx, cudaGetLastError());

  ScoreArgs a;
  a.ps = ps;
  a.th = thx;
  a.rec = ctx->rec.as<float>();
  a.orig = ctx->orig.as<int32_t>();
  a.tab = ctx->blktab.as<BlockTab>();
  a.cslots = cslots;
  a.nsubs = nsubs;
  a.counts_valid = cv;
  a.counts_enabled = ce;
  a.masks = want_masks ? ctx->masks_gm.as<uint32_t>() : nullptr;
  a.wl = ctx->worklist.as<GroupTask>();
  a.wl_count = ctx->wl_count.as<uint32_t>();
  a.wl_cap = (uint32_t)ctx->wl_cap;

  // grid: columns x point chunks; aim at `waves` waves of resident CTAs so the tail stays small.
  // The four per-type kernels are independent; on large problems they run on four streams (forked
  // from and joined back into `st`) so that one kernel's tail is filled by the next one's CTAs.
  const int waves = getenv("RSC_WAVES") ? atoi(getenv("RSC_WAVES")) : 32;
  const int est_cols = (C + kThreads * 4 - 1) / (kThreads * 4);
  const long target = (long)ctx->sm_count * 4 * waves;
  long chunks = (target + est_cols - 1) / est_cols;
  if (chunks > nsubs) chunks = nsubs;
  if (chunks < 1) chunks = 1;
  if (chunks > 65535) chunks = 65535;
  a.subs_per_chunk = (int)((nsubs + chunks - 1) / chunks);
  chunks = (nsubs + a.subs_per_chunk - 1) / a.subs_per_chunk;
  dim3 grid((unsigned)ncols, (unsigned)chunks);
  // (below ~1e9 evaluations the fused single-launch kernel or plain sequential launches are cheaper)
  static const double fork_min = getenv("RSC_FORK_MIN") ? atof(getenv("RSC_FORK_MIN")) : 1e9;
  const bool fork = (double)C * (double)ps.n_pad >= fork_min && !getenv("RSC_NOFORK");

  RSC_CUDA(ctx, cudaEventRecord(ctx->evk0, st));
  // small batches with one tiling for every type: a single launch with a per-column type switch
  const int K0 = L.til[0]->K;
  bool uniform_k = K0 <= 2;
  for (int t = 1; t < kColTypes; ++t) uniform_k = uniform_k && L.til[t]->K == K0;
  if (!fork && uniform_k && !getenv("RSC_NOFUSE")) {
    if (K0 == 1) {
      if (want_masks)
        score_kernel_any<1, 4, true><<<grid, kThreads, 0, st>>>(a);
      else
        score_kernel_any<1, 4, false><<<grid, kThreads, 0, st>>>(a);
    } else {
      if (want_masks)
        score_kernel_any<2, 4, true><<<grid, kThreads, 0, st>>>(a);
      else
        score_kernel_any<2, 4, false><<<grid, kThreads, 0, st>>>(a);
    }
    RSC_CUDA(ctx, cudaGetLastError());
  } else {
    if (fork) RSC_CUDA(ctx, cudaEventRecord(ctx->ev_fork, st));
    // most expensive type first
    const int order[kColTypes] = {RSC_CONE, kConeWide, RSC_CYLINDER, RSC_SPHERE, RSC_PLANE};
    for (int oi = 0; oi < kColTypes; ++oi) {
      const int t = order[oi];
      cudaStream_t s = st;
      if (fork && oi > 0) {
        s = ctx->sfork[oi - 1];
        RSC_CUDA(ctx, cudaStreamWaitEvent(s, ctx->ev_fork, 0));
      }
      (want_masks ? L.til[t]->fn_masks[t] : L.til[t]->fn[t])<<<grid, kThreads, 0, s>>>(a);
      RSC_CUDA(ctx, cudaGetLastError());
      if (fork && oi > 0) {
        RSC_CUDA(ctx, cudaEventRecord(ctx->ev_join[oi - 1], s));
        RSC_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev_join[oi - 1], 0));
      }
    }
  }
  RSC_CUDA(ctx, cudaGetLastError());
  RSC_CUDA(ctx, cudaEventRecord(ctx->evk1, st));
  ctx->stats.score_launches += 1;
  ctx->stats.evals += (int64_t)C * ps.n;
  ctx->stats.cands_scored += C;

  fixup_scan_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(a, d_cands, ctx->slot_of.as<int32_t>(), ctx->pairs.as<AmbPair>(),
                                                       ctx->wl_count.as<uint32_t>() + 1, (uint32_t)ctx->wl_cap);
  RSC_CUDA(ctx, cudaGetLastError());
  fixup_pair_kernel<<<ctx->sm_count * 4, 256, 0, st>>>(a, d_cands, reinterpret_cast<const ex::ConeTrig*>(d_trig),
                                                       ctx->slot_of.as<int32_t>(), ctx->pairs.as<AmbPair>(),
                                                       ctx->wl_count.as<uint32_t>() + 1, (uint32_t)ctx->wl_cap);
  RSC_CUDA(ctx, cudaGetLastError());
  if (d_counts_policy) {
    select_counts_kernel<<<(C + 255) / 256, 256, 0, st>>>(d_cands, C, cv, ce, th.honour_enabled, d_counts_policy);
    RSC_CUDA(ctx, cudaGetLastError());
  }
  return RSC_OK;
}

// ---- audit of the guard band on the real hardware (rsc_debug_margins) --------------------------------
__global__ void audit_compile_kernel(const rsc_cand* __restrict__ cands, int C, const Thresh th, float pmax, float nmax,
                                     float* __restrict__ rec /*[C][kRecFields]*/, int32_t* __restrict__ cols) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= C) return;
  const int col = (cands[i].type < 0 || cands[i].type >= RSC_NTYPES) ? RSC_PLANE : col_type(cands[i]);
  float r[kRecFields];
  compile_record(cands[i], col, th, pmax, nmax, r);
  for (int f = 0; f < kRecFields; ++f) rec[(size_t)i * kRecFields + f] = r[f];
  cols[i] = col;
}

// margins through the PACKED evaluation (eval2<T>, both halves hold the candidate: what score_kernel
// executes) and through the scalar one (eval<T>: the fix-up scan and K4); `diffs` counts pairs on which
// the two differ in any bit
template <int T>
__device__ __forceinline__ float audit_one(const float* r, float px, float py, float pz, float nx, float ny, float nz, float eps,
                                           float cosa, unsigned long long* diffs) {
  float2 r2[RecN<T>::n];
#pragma unroll
  for (int f = 0; f < RecN<T>::n; ++f) r2[f] = make_float2(r[f], r[f]);
  const float2 m2 = eval2<T>(r2, px, py, pz, nx, ny, nz, eps, cosa);
  const float m1 = eval<T>(r, px, py, pz, nx, ny, nz, eps, cosa);
  if (__float_as_uint(m2.x) != __float_as_uint(m1) || __float_as_uint(m2.y) != __float_as_uint(m1)) atomicAdd(diffs, 1ull);
  return m2.x;
}

__global__ void __launch_bounds__(256) audit_margin_kernel(PointSet ps, Thresh th, const float* __restrict__ rec,
                                                           const int32_t* __restrict__ cols, int64_t p0, int64_t np,
                                                           float* __restrict__ out, unsigned long long* __restrict__ diffs) {
  const int c = blockIdx.y;
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= np) return;
  float r[kRecFields];
#pragma unroll
  for (int f = 0; f < kRecFields; ++f) r[f] = rec[(size_t)c * kRecFields + f];
  const int col = cols[c], pt = public_type(col);
  const int64_t i = p0 + j;
  const float px = ps.x[i], py = ps.y[i], pz = ps.z[i], nx = ps.nx[i], ny = ps.ny[i], nz = ps.nz[i];
  const float eps = th.eps[pt], cosa = th.cosa[pt];
  float m;
  switch (col) {
    case RSC_PLANE:
      m = audit_one<RSC_PLANE>(r, px, py, pz, nx, ny, nz, eps, cosa, diffs);
      break;
    case RSC_SPHERE:
      m = audit_one<RSC_SPHERE>(r, px, py, pz, nx, ny, nz, eps, cosa, diffs);
      break;
    case RSC_CYLINDER:
      m = audit_one<RSC_CYLINDER>(r, px, py, pz, nx, ny, nz, eps, cosa, diffs);
      break;
    case kConeWide:
      m = audit_one<kConeWide>(r, px, py, pz, nx, ny, nz, eps, cosa, diffs);
      break;
    default:
      m = audit_one<RSC_CONE>(r, px, py, pz, nx, ny, nz, eps, cosa, diffs);
      break;
  }
  out[(size_t)c * np + j] = m;
}

int32_t audit_margins(rsc_ctx* ctx, const rsc_cloud* cloud, const PointSet& ps, const Thresh& th, const rsc_cand* d_cands, int32_t C,
                      int64_t p0, int64_t np, float* d_out, float* d_rec, int32_t* d_cols, unsigned long long* d_diffs, cudaStream_t st) {
  Thresh thx = th;
  thx.exact_in = cloud->exact();
  audit_compile_kernel<<<(C + 127) / 128, 128, 0, st>>>(d_cands, C, thx, cloud->pmax, cloud->nmax, d_rec, d_cols);
  RSC_CUDA(ctx, cudaGetLastError());
  audit_margin_kernel<<<dim3((unsigned)((np + 255) / 256), (unsigned)C), 256, 0, st>>>(ps, th, d_rec, d_cols, p0, np, d_out, d_diffs);
  RSC_CUDA(ctx, cudaGetLastError());
  return RSC_OK;
}

// after score_enqueue(want_masks=true): ctx->masks_cm = [C][ceil(m/32)] candidate-major masks
int32_t masks_to_candidate_major(rsc_ctx* ctx, int32_t C, int64_t m, cudaStream_t st, uint32_t* d_out) {
  const int cslots = ctx->last_cslots;
  const int64_t words = (m + 31) / 32;
  if (!d_out) {
    RSC_CUDA(ctx, ctx->masks_cm.ensure((size_t)C * words * sizeof(uint32_t)));
    d_out = ctx->masks_cm.as<uint32_t>();
  }
  dim3 grid((unsigned)((C + 31) / 32), (unsigned)((words + 31) / 32));
  masks_transpose_kernel<<<grid, dim3(32, 32), 0, st>>>(ctx->masks_gm.as<uint32_t>(), ctx->slot_of.as<int32_t>(),
                                                        C, cslots, words, d_out);
  RSC_CUDA(ctx, cudaGetLastError());
  return RSC_OK;
}

}  // namespace rsc
