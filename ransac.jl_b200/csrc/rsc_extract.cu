// rsc_extract.cu -- K4: refit + invalidate_indexes! for one shape over the whole cloud shard
// (plane.jl:137-143, sphere.jl:179-190, cylinder.jl:228-234, cone.jl:176-182, fitting.jl:197-202).
//
// HBM bound (24 B/point + 1/8 B of enabled mask).  Launches:
//   1. extract_mask_kernel<T>  four points per thread (128-bit loads of the six SoA rows, skipped for
//                              disabled points), FP32 margin -> inlier bitmask words; points whose
//                              margin is inside the guard band are queued
//   2. extract_fix_kernel      the queued points in FP64, in the reference's operation order
//                              (rsc_exact.cuh); patches their mask bits.  If the queue overflowed
//                              (flat cones: every point is "ambiguous") it re-scans the whole range.
//   3. block_count_kernel, scan_u32 (rsc_fit.cu)    exclusive scan of the per-CTA inlier counts
//   4. extract_write_kernel    ascending global indices by stream compaction (a warp per block); clears enabled bits
#include <stdlib.h>

#include "rsc_eval.cuh"
#include "rsc_exact.cuh"

namespace rsc {

constexpr int kExThreads = 256;
constexpr int kExPts = 2048;  // points per CTA (64 mask words)

struct ExtractArgs {
  PointSet ps;
  Thresh th;
  rsc_cand cand;
  ex::ConeTrig trig;
  float pmax, nmax;
  uint32_t* inl;    // [n_pad/32]
  int64_t block0;   // first CTA-sized block of this rank's point range
  int64_t nblocks;  // blocks of the range
  uint32_t* queue;  // local indices of points inside the guard band
  uint32_t* qn;     // queue fill
  uint32_t qcap;
  float* rec;       // [kRecFields] compiled record of the shape
  int col;          // column type (col_type(cand), decided on the host)
};

// the shape's FP32 record, compiled once (FP64 sqrt/sin/cos on one thread) ahead of the streaming kernel
__global__ void extract_compile_kernel(const __grid_constant__ ExtractArgs a) {
  float t[kRecFields];
  compile_record(a.cand, a.col, a.th, a.pmax, a.nmax, t);
  for (int f = 0; f < kRecFields; ++f) a.rec[f] = t[f];
}

template <int T>
__global__ void __launch_bounds__(kExThreads) extract_mask_kernel(const __grid_constant__ ExtractArgs a) {
  const float band = __ldg(a.rec + kBandField);
  const float eps = a.th.eps[public_type(T)], cosa = a.th.cosa[public_type(T)];
  float rr[RecN<T>::n];
#pragma unroll
  for (int f = 0; f < RecN<T>::n; ++f) rr[f] = __ldg(a.rec + f);
  const int64_t base = (a.block0 + blockIdx.x) * kExPts;
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int it = 0; it < kExPts / (kExThreads * 4); ++it) {
    const int64_t p = base + ((int64_t)it * kExThreads + threadIdx.x) * 4;  // n_pad is a multiple of 512
    uint32_t okb = 0;
    if (p < a.ps.n_pad) {
      const uint32_t nib = (__ldg(a.ps.enabled + (p >> 5)) >> (p & 31)) & 0xFu;
      if (nib) {
        const float4 X = __ldg(reinterpret_cast<const float4*>(a.ps.x + p));
        const float4 Y = __ldg(reinterpret_cast<const float4*>(a.ps.y + p));
        const float4 Z = __ldg(reinterpret_cast<const float4*>(a.ps.z + p));
        const float4 U = __ldg(reinterpret_cast<const float4*>(a.ps.nx + p));
        const float4 V = __ldg(reinterpret_cast<const float4*>(a.ps.ny + p));
        const float4 W = __ldg(reinterpret_cast<const float4*>(a.ps.nz + p));
        const float px[4] = {X.x, X.y, X.z, X.w}, py[4] = {Y.x, Y.y, Y.z, Y.w}, pz[4] = {Z.x, Z.y, Z.z, Z.w};
        const float nx[4] = {U.x, U.y, U.z, U.w}, ny[4] = {V.x, V.y, V.z, V.w}, nz[4] = {W.x, W.y, W.z, W.w};
        uint32_t amb = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float m = eval<T>(rr, px[q], py[q], pz[q], nx[q], ny[q], nz[q], eps, cosa);
          okb |= (m < 0.f ? 1u : 0u) << q;
          amb |= (!(fabsf(m) > band) ? 1u : 0u) << q;
        }
        okb &= nib;
        amb &= nib;
        if (amb) {  // rare
          const uint32_t cnt = __popc(amb);
          uint32_t pos = atomicAdd(a.qn, cnt);
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if ((amb >> q) & 1u) {
              if (pos < a.qcap) a.queue[pos] = (uint32_t)(p + q);
              ++pos;
            }
        }
      }
    }
    uint32_t v = okb << ((lane & 7) * 4);
    v |= __shfl_xor_sync(0xffffffffu, v, 1);
    v |= __shfl_xor_sync(0xffffffffu, v, 2);
    v |= __shfl_xor_sync(0xffffffffu, v, 4);
    if ((lane & 7) == 0 && p < a.ps.n_pad) a.inl[p >> 5] = v;
  }
}

// FP64 decisions for the queued points (or, after a queue overflow, for every enabled point of the
// range whose FP32 margin is inside the band)
__global__ void __launch_bounds__(256) extract_fix_kernel(const __grid_constant__ ExtractArgs a) {
  const uint32_t n = *a.qn;
  const int type = a.cand.type;  // public type: thresholds
  auto decide = [&](uint32_t pt) {
    ex::V3 P, N;
    ex::point64(a.ps, pt, &P, &N);
    const bool ok = ex::compat(a.cand, a.trig, a.th, P, N);
    const uint32_t bit = 1u << (pt & 31);
    if (ok)
      atomicOr(a.inl + (pt >> 5), bit);
    else
      atomicAnd(a.inl + (pt >> 5), ~bit);
  };
  if (n <= a.qcap) {
    for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) decide(a.queue[e]);
    return;
  }
  float rr[kRecFields];
#pragma unroll
  for (int f = 0; f < kRecFields; ++f) rr[f] = a.rec[f];
  const int64_t lo = a.block0 * kExPts;
  int64_t hi = (a.block0 + a.nblocks) * kExPts;
  if (hi > a.ps.n_pad) hi = a.ps.n_pad;
  for (int64_t p = lo + blockIdx.x * blockDim.x + threadIdx.x; p < hi; p += (int64_t)gridDim.x * blockDim.x) {
    if (!((a.ps.enabled[p >> 5] >> (p & 31)) & 1u)) continue;
    const float m = eval_any(a.col, rr, a.ps.x[p], a.ps.y[p], a.ps.z[p], a.ps.nx[p], a.ps.ny[p], a.ps.nz[p], a.th.eps[type],
                             a.th.cosa[type]);
    if (!(fabsf(m) > rr[kBandField])) decide((uint32_t)p);
  }
}

// inliers per CTA-sized block of the (all-reduced) inlier mask
// inliers per CTA-sized block of the mask (64 words): a WARP per block, two coalesced words per lane
// (a thread per block read the mask with a 256-byte stride: 12 us on 10 M points, 3 us now)
__global__ void __launch_bounds__(256) block_count_kernel(const uint32_t* __restrict__ inl, int64_t words, uint32_t* __restrict__ counts,
                                                          int nblocks) {
  const int b = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= nblocks) return;
  const int64_t i = (int64_t)b * (kExPts / 32) + lane;
  uint32_t s = 0;
  if (i < words) s += __popc(inl[i]);
  if (i + 32 < words) s += __popc(inl[i + 32]);
  s = __reduce_add_sync(0xffffffffu, s);
  if (lane == 0) counts[b] = s;
}


// a WARP per 2048-point block (64 mask words, two per lane): exclusive scan of the words' bit counts, then every lane
// writes the indices of its words' set bits (a thread per POINT spent 10 M threads on a mask with 2 % of its bits set)
__global__ void __launch_bounds__(kExThreads) extract_write_kernel(const uint32_t* __restrict__ inl,
                                                                   const unsigned long long* __restrict__ offsets,
                                                                   int64_t n_pad, int nblocks, int64_t global_offset,
                                                                   int64_t* __restrict__ out,
                                                                   uint32_t* __restrict__ enabled /*nullable*/) {
  const int b = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= nblocks) return;
  const int64_t nwords = n_pad >> 5;
  const int64_t wa = (int64_t)b * (kExPts / 32) + 2 * lane, wb = wa + 1;
  uint32_t ma = wa < nwords ? inl[wa] : 0u, mb = wb < nwords ? inl[wb] : 0u;
  const uint32_t a0 = __popc(ma), a1 = __popc(mb);
  uint32_t s = a0 + a1, inc = s;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += o;
  }
  if (enabled) {
    if (ma) enabled[wa] &= ~ma;
    if (mb) enabled[wb] &= ~mb;
  }
  if (!out) return;
  unsigned long long pos = offsets[b] + (inc - s);
  while (ma) {
    const int bit = __ffs(ma) - 1;
    ma &= ma - 1;
    out[pos++] = wa * 32 + bit + global_offset;
  }
  while (mb) {
    const int bit = __ffs(mb) - 1;
    mb &= mb - 1;
    out[pos++] = wb * 32 + bit + global_offset;
  }
}

// Enqueue steps 1+2; the caller reads the total (ctx->misc2[0]) and then calls refit_write_enqueue.
// Sharded: only this rank's point range is evaluated and the inlier-mask words are summed across
// ranks (disjoint ranges, so the sum is the union), after which every rank holds the full mask.
template <class F>
static void launch_mask(int col, F&& f) {
  switch (col) {
    case RSC_PLANE:
      f(extract_mask_kernel<RSC_PLANE>);
      break;
    case kConeWide:
      f(extract_mask_kernel<kConeWide>);
      break;
    case RSC_SPHERE:
      f(extract_mask_kernel<RSC_SPHERE>);
      break;
    case RSC_CYLINDER:
      f(extract_mask_kernel<RSC_CYLINDER>);
      break;
    case RSC_CONE:
      f(extract_mask_kernel<RSC_CONE>);
      break;
    default:
      break;
  }
}

int32_t refit_mask_enqueue(rsc_cloud* cloud, const Thresh& th, const rsc_cand& cand, cudaStream_t st, int timed_reps) {
  rsc_ctx* ctx = cloud->ctx;
  const int64_t n_pad = cloud->n_pad;
  const int64_t words = n_pad / 32;
  const int nblocks = (int)((n_pad + kExPts - 1) / kExPts);
  RSC_CUDA(ctx, ctx->idxbuf.ensure((size_t)words * 4 + (size_t)nblocks * (4 + 8) + 64));
  ExtractArgs a;
  a.ps = view_cloud(cloud);
  a.th = th;
  a.th.exact_in = cloud->exact();
  a.cand = cand;
  a.trig.ct = cos(-cand.p[6] / 2);
  a.trig.st = sin(-cand.p[6] / 2);
  a.pmax = cloud->pmax;
  a.nmax = cloud->nmax;
  char* b = ctx->idxbuf.as<char>();
  a.inl = reinterpret_cast<uint32_t*>(b);
  unsigned long long* offsets = reinterpret_cast<unsigned long long*>(b + ((size_t)words * 4 + 15) / 16 * 16);
  uint32_t* block_counts = reinterpret_cast<uint32_t*>(offsets + nblocks);
  RSC_CUDA(ctx, ctx->misc2.ensure(64));
  const bool sharded = ctx->allreduce && cloud->range_set;
  int64_t b0 = 0, b1 = nblocks;
  if (sharded) {
    b0 = cloud->range_lo / kExPts;
    b1 = (cloud->range_hi + kExPts - 1) / kExPts;
    if (b1 < b0) b1 = b0;  // an empty rank (range_lo == range_hi == n_pad) evaluates nothing
    RSC_CUDA(ctx, cudaMemsetAsync(a.inl, 0, (size_t)words * 4, st));
  }
  a.block0 = b0;
  a.nblocks = b1 - b0;
  size_t qcap = (size_t)1 << 20;
  if (const char* e = getenv("RSC_EXQ_CAP")) {  // test hook: force the queue-overflow path
    const long v = atol(e);
    if (v > 0) qcap = (size_t)v;
  }
  RSC_CUDA(ctx, ctx->exq.ensure(qcap * 4 + 16 + kRecFields * 4));
  a.qn = ctx->exq.as<uint32_t>();
  a.rec = reinterpret_cast<float*>(a.qn + 4);
  a.queue = a.qn + 4 + kRecFields;
  a.qcap = (uint32_t)qcap;
  RSC_CUDA(ctx, cudaMemsetAsync(a.qn, 0, 4, st));
  const unsigned grid = (unsigned)(b1 - b0);
  if (cand.type < 0 || cand.type >= RSC_NTYPES) return fail(ctx, RSC_E_ARG, "refit: unknown shape type");
  a.col = col_type(cand);
  extract_compile_kernel<<<1, 1, 0, st>>>(a);
  RSC_CUDA(ctx, cudaGetLastError());
  if (grid > 0 && timed_reps > 1) {  // measurement only: `timed_reps` launches between one event pair, then the real pass
    RSC_CUDA(ctx, cudaEventRecord(ctx->evr0, st));
    for (int r = 0; r < timed_reps; ++r) launch_mask(a.col, [&](auto k) { k<<<grid, kExThreads, 0, st>>>(a); });
    RSC_CUDA(ctx, cudaGetLastError());
    RSC_CUDA(ctx, cudaEventRecord(ctx->evr1, st));
    RSC_CUDA(ctx, cudaMemsetAsync(a.qn, 0, 4, st));
    launch_mask(a.col, [&](auto k) { k<<<grid, kExThreads, 0, st>>>(a); });
  } else {
    RSC_CUDA(ctx, cudaEventRecord(ctx->evr0, st));
    if (grid > 0) launch_mask(a.col, [&](auto k) { k<<<grid, kExThreads, 0, st>>>(a); });  // an empty rank only joins the all-reduce below
    RSC_CUDA(ctx, cudaGetLastError());
    RSC_CUDA(ctx, cudaEventRecord(ctx->evr1, st));
  }
  RSC_CUDA(ctx, cudaGetLastError());
  extract_fix_kernel<<<ctx->sm_count * 4, 256, 0, st>>>(a);
  RSC_CUDA(ctx, cudaGetLastError());
  if (sharded && ctx->allreduce(ctx->allreduce_user, a.inl, words, (void*)st))
    return fail(ctx, RSC_E_NCCL, "refit: all-reduce callback failed");
  block_count_kernel<<<(unsigned)(((int64_t)nblocks * 32 + 255) / 256), 256, 0, st>>>(a.inl, words, block_counts, nblocks);
  RSC_CUDA(ctx, cudaGetLastError());
  // (8 counts per thread and pass, tiled beyond 32 Ki blocks: c5's 48 828 blocks took one CTA 48 passes before)
  if (int32_t rcs = scan_u32(ctx, block_counts, nblocks, offsets, ctx->misc2.as<unsigned long long>(), st)) return rcs;
  ctx->stats.evals += (b1 - b0) * kExPts < cloud->n ? (b1 - b0) * kExPts : cloud->n;
  return RSC_OK;
}

__global__ void mask_from_list_kernel(const int64_t* __restrict__ list, int64_t n, int64_t global_offset, uint32_t* __restrict__ inl) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t p = list[i] - global_offset;
  atomicOr(inl + (p >> 5), 1u << (p & 31));
}

// Replace the inlier mask of the last refit_mask_enqueue by the points of `d_list` (n global indices, a subset
// of that mask: the parameter-space bitmap filter) and redo the per-CTA counts / offsets / total.
int32_t refit_mask_from_list(rsc_cloud* cloud, const int64_t* d_list, int64_t n, cudaStream_t st) {
  rsc_ctx* ctx = cloud->ctx;
  const int64_t n_pad = cloud->n_pad;
  const int64_t words = n_pad / 32;
  const int nblocks = (int)((n_pad + kExPts - 1) / kExPts);
  char* b = ctx->idxbuf.as<char>();
  uint32_t* inl = reinterpret_cast<uint32_t*>(b);
  unsigned long long* offsets = reinterpret_cast<unsigned long long*>(b + ((size_t)words * 4 + 15) / 16 * 16);
  uint32_t* block_counts = reinterpret_cast<uint32_t*>(offsets + nblocks);
  RSC_CUDA(ctx, cudaMemsetAsync(inl, 0, (size_t)words * 4, st));
  if (n > 0) {
    mask_from_list_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_list, n, cloud->global_offset, inl);
    RSC_CUDA(ctx, cudaGetLastError());
  }
  block_count_kernel<<<(unsigned)(((int64_t)nblocks * 32 + 255) / 256), 256, 0, st>>>(inl, words, block_counts, nblocks);
  RSC_CUDA(ctx, cudaGetLastError());
  return scan_u32(ctx, block_counts, nblocks, offsets, ctx->misc2.as<unsigned long long>(), st);
}

int32_t refit_mask_buffer(rsc_cloud* cloud, uint32_t** inl) {
  rsc_ctx* ctx = cloud->ctx;
  const int64_t words = cloud->n_pad / 32;
  const int nblocks = (int)((cloud->n_pad + kExPts - 1) / kExPts);
  RSC_CUDA(ctx, ctx->idxbuf.ensure((size_t)words * 4 + (size_t)nblocks * (4 + 8) + 64));
  RSC_CUDA(ctx, ctx->misc2.ensure(64));
  *inl = ctx->idxbuf.as<uint32_t>();
  return RSC_OK;
}

int32_t refit_scan_enqueue(rsc_cloud* cloud, cudaStream_t st) {
  rsc_ctx* ctx = cloud->ctx;
  const int64_t words = cloud->n_pad / 32;
  const int nblocks = (int)((cloud->n_pad + kExPts - 1) / kExPts);
  char* b = ctx->idxbuf.as<char>();
  const uint32_t* inl = reinterpret_cast<const uint32_t*>(b);
  unsigned long long* offsets = reinterpret_cast<unsigned long long*>(b + ((size_t)words * 4 + 15) / 16 * 16);
  uint32_t* block_counts = reinterpret_cast<uint32_t*>(offsets + nblocks);
  block_count_kernel<<<(unsigned)(((int64_t)nblocks * 32 + 255) / 256), 256, 0, st>>>(inl, words, block_counts, nblocks);
  RSC_CUDA(ctx, cudaGetLastError());
  return scan_u32(ctx, block_counts, nblocks, offsets, ctx->misc2.as<unsigned long long>(), st);
}

int32_t refit_write_enqueue(rsc_cloud* cloud, int64_t* d_out, bool disable, cudaStream_t st) {
  rsc_ctx* ctx = cloud->ctx;
  const int64_t n_pad = cloud->n_pad;
  const int nblocks = (int)((n_pad + kExPts - 1) / kExPts);
  char* b = ctx->idxbuf.as<char>();
  const uint32_t* inl = reinterpret_cast<const uint32_t*>(b);
  const unsigned long long* offsets =
      reinterpret_cast<const unsigned long long*>(b + ((size_t)(n_pad / 32) * 4 + 15) / 16 * 16);
  extract_write_kernel<<<(unsigned)(((int64_t)nblocks * 32 + kExThreads - 1) / kExThreads), kExThreads, 0, st>>>(
      inl, offsets, n_pad, nblocks, cloud->global_offset, d_out, disable ? cloud->enabled : nullptr);
  RSC_CUDA(ctx, cudaGetLastError());
  if (disable) {
    cloud->enabled_changed();
    return refresh_subsets_enabled(cloud, st);
  }
  return RSC_OK;
}

}  // namespace rsc
