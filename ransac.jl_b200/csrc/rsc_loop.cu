// rsc_loop.cu -- ransac(pc, params) (iterations.jl:35-162): the RANSAC loop behind rsc_ransac_run and
// rsc_ransac_run_user, with the candidate store, the scoring and the removal of invalid candidates on the device.
//
// Iterations run in SPECULATIVE BATCHES of nb: as long as nothing is extracted the enabled mask is unchanged,
// so iterations k..k+nb-1 sample (the same Philox set ids as separate iterations), fit and score together.  The
// decision then walks the batch with the reference's bookkeeping, iteration by iteration, and cuts it at the
// first extraction or at termination; the iterations behind the cut are discarded and redone (their sets
// sampled a stale mask).  Per batch:
//   K1  sample + fit                      rsc_fit.cu        -> candidates, per-iteration segment bounds (root-cell
//                                                            sampler; level-weighted cell sampler with RSC_SAMPLER_OCTREE)
//   K2  score the new candidates on subset 1 (iterations.jl:95), counts all-reduced when sharded
//   K3  finish_new / argmax / seg_argmax  -> best of the old store, best of every iteration's candidates
//       decide_kernel                     the reference's bookkeeping, iteration by iteration:
//                                         countcandidates (iterations.jl:94-102), findhighestscore
//                                         (fitting.jl:140-150), estimatescore (confidenceintervals.jl:
//                                         53-74, Int64 wrap included), prob / chooseS (utilities.jl:262,
//                                         :297-300), the extraction test (iterations.jl:113) and the
//                                         termination test (iterations.jl:151-156) -- it cuts the batch
//                                         at the first extraction / termination and leaves a 128-byte
//                                         record (iterations used, extract?, which candidate, its 64-byte
//                                         shape, counters) that the host reads with ONE synchronisation.
//       With RSC_SCORE_PROGRESSIVE, RSC_SAMPLER_OCTREE or RSC_LOOP_HOSTWALK the host takes that decision instead
//       (host_decide, rsc_run.cu), from the same segment bounds and keys read with one synchronisation.
//   on extraction:
//   K4  refit over the rank's points, ascending inlier indices by stream compaction, enabled bits
//       cleared (rsc_extract.cu)
//   K5  removeinvalidshapes! without stored inlier lists: every stored candidate's subset-1 inliers are enabled
//       at the time of an extraction (the reference removes any candidate with a disabled inlier at each
//       extraction, and new candidates only count enabled points), so "has a now-disabled inlier" == "is
//       compatible with one of the NEWLY disabled subset-1 points".  Those points are gathered into a scratch
//       point set and the store is re-scored against it, then invalidate + order-preserving compaction.
//       Spheres, whose reference scorer ignores `isenabled` (Q4), additionally die at the first extraction
//       after they were scored if they matched any already-disabled point.
// Host synchronisations: 1 per batch for a small batch (its K2 launch is sized by a prediction), else 2 (the
// number of new candidates sizes the K2 launch; the decision) + 1 per extraction (store size, inlier count).
//
// Multi-GPU, one process per GPU (include/rsc.h "point-range sharding"):
//   sharded storage  every rank holds its point range only; minimal sets are drawn from the replicated
//                    whole-cloud enabled mask (identical on all ranks), their coordinates gathered by one
//                    all-reduce per batch; counts / K5 hits all-reduced; the inlier list of a shape stays
//                    distributed (each rank holds the ascending indices of its range)
//   replicated       every rank holds the cloud and scores / refits its range (rsc_cloud_set_range)
// All ranks take identical decisions: decide_kernel runs replicated on identical (all-reduced) counts.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>

#include "rsc_loop.cuh"

namespace rsc {

struct DecideParams {
  long long N, M, tau;
  double prob_det;
  int S, drawN, extract_s, terminate_s;
};

struct K5Host {  // what the host reads after an extraction
  unsigned long long kept, total_local;
  int32_t ovf, tot_global;
};

// estimatescore(...).E with Julia's Int64 arithmetic (confidenceintervals.jl:53-74; the products wrap, Q9)
__device__ double estimate_E(long long M, long long N, long long count) {
  const long long Np = -2 - M, x = -2 - N, n = -1 - count;
  const long long xn = (long long)((unsigned long long)x * (unsigned long long)n);
  const long long prod =
      (long long)((unsigned long long)((long long)((unsigned long long)xn * (unsigned long long)(Np - x))) * (unsigned long long)(Np - n));
  const double sq_ = (double)prod / (double)(Np - 1);
  const double sq = sq_ < 0 ? 0.0 : sqrt(sq_);
  const double a = -1 - ((double)xn + sq) / (double)Np, b = -1 - ((double)xn - sq) / (double)Np;
  if (a != a || b != b) return NAN;
  const double lo = a < b ? a : b, hi = a < b ? b : a;
  return (lo + hi) / 2;
}

__device__ double prob_dev(double n, double s, double N, double k) { return 1 - pow(1 - pow(n / N, k), s); }  // utilities.jl:262

// K3: the bookkeeping of one batch.  The walk over the batch's iterations is sequential by nature (cut at the
// first extraction / termination), but what it compares is not: thread j evaluates iteration j's counters,
// running best (a prefix maximum of the per-iteration arg-max keys), estimatescore, and the two prob() tests
// (four FP64 pow calls); thread 0 then takes the first iteration that extracts or terminates.
__global__ void __launch_bounds__(kMaxBatch) decide_kernel(LoopDev* __restrict__ d, const int32_t* __restrict__ ovf, int store_n0,
                                                           int nb, int k0, DecideParams q, const rsc_cand* __restrict__ cands,
                                                           int cap_new) {
  __shared__ long long s_key[kMaxBatch];
  __shared__ int s_ext[kMaxBatch], s_term[kMaxBatch];
  const int j = threadIdx.x;
  const int over = ovf ? (*ovf ? 1 : 0) : 0;
  const int n_new = d->seg[nb];
  const bool redo = over || (cap_new >= 0 && n_new > cap_new);
  if (j < nb && !redo) {
    long long key = (store_n0 >= 1 && d->oldbest[0] >= 0) ? ((d->oldbest[1] << 32) | (long long)(0x7fffffff - d->oldbest[0])) : -1;
    for (int i = 0; i <= j; ++i)
      if (d->seg_keys[i] > key) key = d->seg_keys[i];  // strict >: the first maximum wins (the key carries the store index)
    const long long c0 = store_n0 + d->seg[j + 1];                 // iterations.jl:102
    const long long c1 = d->counters[1] + d->seg[j + 1];           // iterations.jl:94 (accumulated over the batch)
    const long long c2 = (long long)(k0 + j) * q.S;                // iterations.jl:99
    const long long cc[3] = {c0, c1, c2};
    int ext = 0;
    if (c0 >= 1 && key >= 0) {
      const double E = estimate_E(q.M, q.N, (long long)(key >> 32));
      ext = prob_dev(E, (double)cc[q.extract_s], (double)q.N, (double)q.drawN) > q.prob_det;  // iterations.jl:113
    }
    s_key[j] = key;
    s_ext[j] = ext;
    s_term[j] = prob_dev((double)q.tau, (double)cc[q.terminate_s], (double)q.N, (double)q.drawN) > q.prob_det;  // iterations.jl:151-156
  }
  __syncthreads();
  if (j != 0) return;
  BatchRec r;
  r.ovf = over ? 1 : ((cap_new >= 0 && n_new > cap_new) ? 2 : 0);  // 2: the sync-free launch was sized for fewer candidates
  r.n_new = n_new;
  r.pad = 0;
  r.used = 0, r.extract = 0, r.terminated = 0, r.iterations = k0 - 1, r.best_idx = -1, r.best_score = 0, r.store_n = store_n0;
  for (int i = 0; i < 3; ++i) r.counters[i] = d->counters[i];
  if (redo) {  // the counts are incomplete (queue overflow on some rank) or some candidates were not scored: the host repeats K2
    d->rec = r;
    return;
  }
  int last = nb - 1;
  for (int i = 0; i < nb; ++i)
    if (s_ext[i] || s_term[i]) {
      last = i;
      break;
    }
  if (nb > 0) {
    r.used = last + 1;
    r.iterations = k0 + last;
    r.store_n = store_n0 + d->seg[last + 1];
    r.counters[0] = r.store_n;
    r.counters[1] = d->counters[1] + d->seg[last + 1];
    r.counters[2] = (long long)(k0 + last) * q.S;
    r.extract = s_ext[last];
    r.terminated = s_term[last];
    if (r.extract) {
      r.best_idx = 0x7fffffff - (int)(s_key[last] & 0xffffffffll);
      r.best_score = (int)(s_key[last] >> 32);
      r.best = cands[r.best_idx];
    }
  }
  for (int i = 0; i < 3; ++i) d->counters[i] = r.counters[i];
  d->rec = r;
}

// the sync-free batch path: the number of new candidates stays on the device (the fit's compaction total)
__global__ void append_new_kernel(const rsc_cand* __restrict__ src, const unsigned long long* __restrict__ total, int cap,
                                  rsc_cand* __restrict__ dst) {
  const int n = (int)min(*total, (unsigned long long)cap);
  const uint4* s = reinterpret_cast<const uint4*>(src);
  uint4* d = reinterpret_cast<uint4*>(dst);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n * 4; i += gridDim.x * blockDim.x) d[i] = s[i];
}

// cell sampler, per batch iteration and octree level: number of new candidates and the sum of their scores
// (fitting.jl:184 adds E(score) per candidate; E is affine in the count, so the host adds the closed form of the sum)
__global__ void level_stats_kernel(const int32_t* __restrict__ out_set, const int32_t* __restrict__ set_level,
                                   const int32_t* __restrict__ score, int n, int S, long long (*__restrict__ lv)[22]) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int l = set_level[out_set[i]] - 1;
  if (l < 0 || l >= 11) return;
  long long* row = lv[out_set[i] / S];  // the batch iteration the candidate's minimal set belongs to
  atomicAdd((unsigned long long*)(row + l), 1ull);
  atomicAdd((unsigned long long*)(row + 11 + l), (unsigned long long)score[i]);
}

// K5: mask of the subset points the extraction just disabled, in place: old &= ~new
__global__ void newly_mask_kernel(uint32_t* __restrict__ old_en, const uint32_t* __restrict__ new_en, int64_t words) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w < words) old_en[w] &= ~new_en[w];
}

// K5, gathered form: the newly disabled subset points (old & ~new) into a compact SoA scratch set of
// `cap` points (the host sizes it by the extracted candidate's subset score, an upper bound of their
// number); *over = 1 if they do not fit (then the host repeats K5 in the masked form)
__global__ void newly_gather_capped_kernel(const uint32_t* __restrict__ old_en, const uint32_t* __restrict__ new_en, int64_t words,
                                           const unsigned long long* __restrict__ offs, const unsigned long long* __restrict__ total,
                                           const float* __restrict__ soa, int64_t m_pad, float* __restrict__ out, int64_t cap,
                                           int32_t* __restrict__ over, const int64_t* __restrict__ idx, int64_t* __restrict__ out_idx) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w == 0) *over = (*total > (unsigned long long)cap) ? 1 : 0;
  if (w >= words) return;
  uint32_t bits = old_en[w] & ~new_en[w];
  unsigned long long o = offs[w];
  while (bits) {
    const int b = __ffs(bits) - 1;
    bits &= bits - 1;
    const int64_t j = w * 32 + b;
    if (o < (unsigned long long)cap) {
#pragma unroll
      for (int f = 0; f < 6; ++f) out[f * cap + o] = soa[f * m_pad + j];
      if (out_idx) out_idx[o] = idx[j];  // exact clouds: the scratch set's map into the float64 coordinates
    }
    ++o;
  }
}

// valid (= enabled) words of the scratch set: the first *n points are real
__global__ void fill_valid_dev_kernel(uint32_t* __restrict__ valid, const unsigned long long* __restrict__ n, int64_t words) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= words) return;
  const long long nn = (long long)*n, lo = w * 32;
  valid[w] = lo + 32 <= nn ? 0xffffffffu : (lo < nn ? (1u << (nn - lo)) - 1u : 0u);
}

__global__ void k5_pack_kernel(LoopDev* __restrict__ d, const unsigned long long* __restrict__ ktot, const int32_t* __restrict__ ovf,
                               const int32_t* __restrict__ over, const unsigned long long* __restrict__ total_local,
                               K5Host* __restrict__ out) {
  out->kept = *ktot;
  out->total_local = *total_local;
  out->ovf = (*ovf ? 1 : 0) + (*over ? 2 : 0);  // bit 0: guard-band queue overflow, bit 1: scratch set too small (any rank)
  out->tot_global = d->tot_global[0];
}

// small-batch scorer (rsc_small.cu) limits: beyond them the tiled kernel is the faster one
// (measured on c4, profiles/r2h_launches_ransac_c4_summary.json: small kernel ~60 us at ~100 candidates x 312 k
// points and linear in the candidates, tiled path ~190 us flat at this size -> cross-over near 1e8 evaluations)
constexpr int kSmallMaxCands = 4096;
constexpr double kSmallMaxEvals = 1.2e8;

// K5's hits (rsc_loop.cuh).  Gathered form: the newly disabled points of the source go into a compact scratch set.
// Their number is only known on the device, but it cannot exceed the extracted candidate's subset-1 score in the
// store (every one of them was a compatible, enabled subset point when the candidate was scored; the enabled set
// only shrinks), which the host has from the decision record: that sizes the launch without a round trip.  If they
// do not fit, hit[nst + 1] says so and the caller repeats in the masked form.  Masked form (the least-squares refit
// moves the shape, so the bound does not hold; also the fallback): score against the whole source under the mask
// old & ~new.  The hits are enabled-gated counts over those points; with `coll` they are summed over the ranks,
// together with the two flags.
int32_t k5_hits(rsc_ctx* ctx, rsc_cloud* cloud, const K5In& in, const Thresh& th, K5Out* out, cudaStream_t st) {
  if (!ctx->loop_scratch) ctx->loop_scratch = new LoopScratch();
  LoopScratch& ls = *static_cast<LoopScratch*>(ctx->loop_scratch);
  const int nst = in.nst;
  const PointSet& src = in.src;
  const bool exact = src.xyz64 != nullptr;
  const uint32_t* old_src = in.olden + in.old_word0;
  int32_t rc = RSC_OK;
  PointSet dps = src;
  const float4* tiles = in.view ? in.view_tiles : nullptr;  // the culled scorer's spheres of dps
  // hit counts [nst] + two flags that ride with them through the all-reduce: guard-band queue overflow,
  // scratch set too small
  RSC_CUDA(ctx, ctx->counts.ensure(((size_t)3 * nst + 8) * 4));
  int32_t* hit = ctx->counts.as<int32_t>() + 2 * (size_t)nst;
  int32_t* d_over = hit + nst + 1;
  RSC_CUDA(ctx, cudaMemsetAsync(d_over, 0, 4, st));
  // scratch: [wcnt: sl_words u32][woff: sl_words + 1 u64][keep: nst u32][koff: nst + 1 u64]
  const int64_t sl_words = src.n_pad / 32;
  const size_t o_woff = ((size_t)sl_words * 4 + 255) / 256 * 256;
  const size_t o_keep = o_woff + ((size_t)(sl_words + 1) * 8 + 255) / 256 * 256;
  const size_t o_koff = o_keep + ((size_t)nst * 4 + 255) / 256 * 256;
  RSC_CUDA(ctx, ls.nmeta.ensure(o_koff + (size_t)(nst + 1) * 8));
  uint32_t* wcnt = ls.nmeta.as<uint32_t>();
  unsigned long long* woff = (unsigned long long*)(ls.nmeta.as<char>() + o_woff);
  unsigned long long* wtot = woff + sl_words;
  out->hit = hit;
  out->keep = (uint32_t*)(ls.nmeta.as<char>() + o_keep);
  out->koff = (unsigned long long*)(ls.nmeta.as<char>() + o_koff);
  out->ktot = out->koff + nst;
  // the culled scorer (built-in types only) on a view-ordered set when the store is large: most stored candidates
  // are then nowhere near the extracted shape, and the dense path's candidate compiler is ONE CTA (3 ms for a
  // store of a million candidates, the cell sampler's)
  auto culled = [&](int64_t npts) {
    return in.view && !in.uo && in.cull_mode != 0 && (in.cull_mode == 2 || nst >= 4096 || (double)nst * (double)npts >= 2e8);
  };
  if (in.masked) {
    newly_mask_kernel<<<(unsigned)((in.swords + 255) / 256), 256, 0, st>>>(in.olden, in.new_en, in.swords);
    RSC_CUDA(ctx, cudaGetLastError());
    dps.enabled = dps.valid = old_src;  // (only the enabled-gated counts are read)
  } else if (sl_words > 0) {
    const int64_t cap = ((int64_t)std::max(in.bound, 1) + kTile - 1) / kTile * kTile;
    newly_count_kernel<<<(unsigned)((sl_words + 255) / 256), 256, 0, st>>>(old_src, src.enabled, sl_words, wcnt);
    RSC_CUDA(ctx, cudaGetLastError());
    if ((rc = scan_u32(ctx, wcnt, (int)sl_words, woff, wtot, st))) return rc;
    RSC_CUDA(ctx, ls.nscratch.ensure((size_t)6 * cap * 4));
    RSC_CUDA(ctx, ls.nvalid.ensure((size_t)(cap / 32) * 4));
    RSC_CUDA(ctx, cudaMemsetAsync(ls.nscratch.p, 0, (size_t)6 * cap * 4, st));
    if (exact) {  // the scratch set's map into the float64 coordinates, the source's map gathered
      // (entries past the gathered count stay 0: padding lanes may still look their point up)
      RSC_CUDA(ctx, ls.nidx.ensure((size_t)cap * sizeof(int64_t)));
      RSC_CUDA(ctx, cudaMemsetAsync(ls.nidx.p, 0, (size_t)cap * sizeof(int64_t), st));
    }
    newly_gather_capped_kernel<<<(unsigned)((sl_words + 255) / 256), 256, 0, st>>>(
        old_src, src.enabled, sl_words, woff, wtot, src.x, src.y - src.x, ls.nscratch.as<float>(), cap, d_over, src.map,
        exact ? ls.nidx.as<int64_t>() : nullptr);
    RSC_CUDA(ctx, cudaGetLastError());
    fill_valid_dev_kernel<<<(unsigned)((cap / 32 + 255) / 256), 256, 0, st>>>(ls.nvalid.as<uint32_t>(), wtot, cap / 32);
    RSC_CUDA(ctx, cudaGetLastError());
    float* b = ls.nscratch.as<float>();
    dps.x = b, dps.y = b + cap, dps.z = b + 2 * cap, dps.nx = b + 3 * cap, dps.ny = b + 4 * cap, dps.nz = b + 5 * cap;
    dps.enabled = dps.valid = ls.nvalid.as<uint32_t>();
    dps.n = dps.n_pad = cap;
    dps.map = exact ? ls.nidx.as<int64_t>() : nullptr;
    if (culled(cap)) {  // spheres of the gathered points only: the zero padding stays out of them
      RSC_CUDA(ctx, ls.ntiles.ensure(cull_sphere_count(cap) * sizeof(float4)));
      if ((rc = cull_tile_spheres(ctx, dps, ls.ntiles.as<float4>(), st, wtot))) return rc;
      tiles = ls.ntiles.as<float4>();
    }
  }
  const rsc_cand* cands = in.cands;
  if (culled(dps.n)) {
    if ((rc = cull_enqueue(ctx, cloud, dps, tiles, th, cands, nst, nullptr, ctx->counts.as<int32_t>(), hit, nullptr, st))) return rc;
    RSC_CUDA(ctx, cudaMemsetAsync(hit + nst, 0, 4, st));  // nothing can overflow: pairs beyond the queue are decided inline
  } else if (in.use_small && nst <= kSmallMaxCands && (double)nst * (double)std::max<int64_t>(dps.n_pad, 1) <= kSmallMaxEvals) {
    if ((rc = score_small_enqueue(ctx, cloud, dps, th, cands, nst, nullptr, ctx->counts.as<int32_t>(), hit, st))) return rc;
    RSC_CUDA(ctx, cudaMemsetAsync(hit + nst, 0, 4, st));  // no guard-band queue on this path
  } else {
    if ((rc = score_enqueue(ctx, cloud, dps, th, cands, nst, nullptr, false, st, ctx->counts.as<int32_t>(), hit))) return rc;
    queue_overflow_kernel<<<1, 1, 0, st>>>(ctx->wl_count.as<uint32_t>(), (uint32_t)ctx->wl_cap, hit + nst);
    RSC_CUDA(ctx, cudaGetLastError());
  }
  // user records: the built-in scorers left their hits at 0 (enabled-gated counts, so the scratch bound holds)
  if (in.uo && (rc = user_score_enqueue(ctx, *in.uo, dps, cands, nst, nullptr, nullptr, hit, st))) return rc;
  if (in.coll && ctx->allreduce(ctx->allreduce_user, hit, (int64_t)nst + 2, (void*)st))
    return fail(ctx, RSC_E_NCCL, "ransac_run: all-reduce of the K5 hits failed");
  return RSC_OK;
}

int32_t k5_compact(const K5Out& o, int nst, int best, const rsc_cand* c0, const int32_t* s0, uint8_t* f0, rsc_cand* c1,
                   int32_t* s1, uint8_t* f1, rsc_ctx* ctx, cudaStream_t st) {
  invalidate_kernel<<<(nst + 255) / 256, 256, 0, st>>>(o.hit, f0, nst, best, o.keep);
  RSC_CUDA(ctx, cudaGetLastError());
  if (int32_t rc = scan_u32(ctx, o.keep, nst, o.koff, o.ktot, st)) return rc;
  compact_store_kernel<<<(nst + 255) / 256, 256, 0, st>>>(c0, s0, f0, o.keep, o.koff, nst, c1, s1, f1);
  RSC_CUDA(ctx, cudaGetLastError());
  return RSC_OK;
}

int32_t ransac_loop_device(rsc_cloud* cloud, const rsc_params* p, uint64_t seed, rsc_run* run, const FitOrder* order, HostWalk* host) {
  rsc_ctx* ctx = cloud->ctx;
  cudaStream_t st = ctx->stream;
  if (!ctx->loop_scratch) ctx->loop_scratch = new LoopScratch();
  LoopScratch& ls = *static_cast<LoopScratch*>(ctx->loop_scratch);
  Store& store = ls.store;
  store.n = 0, store.cur = 0;
  int32_t rc = RSC_OK;
  const Thresh th = make_thresh(p);
  rsc_subset& sub = cloud->subsets[0];
  const bool shard = cloud->is_shard();
  const bool ranged = !shard && ctx->allreduce != nullptr && cloud->range_set;
  const bool coll = shard || ranged;  // counts are summed over the ranks
  if (shard && !ctx->allreduce)
    return fail(ctx, RSC_E_STATE, "ransac_run: sharded storage needs a communicator (rsc_ctx_comm_init or rsc_ctx_set_allreduce)");
  if (shard && cloud->n_global >= 2147483647LL) return fail(ctx, RSC_E_ARG, "ransac_run: sharded storage supports clouds below 2^31 points");
  if (shard && (p->compat_flags & (RSC_REFIT_LSQ | RSC_EXTRACT_BITMAP)))
    return fail(ctx, RSC_E_STATE, "ransac_run: RSC_REFIT_LSQ / RSC_EXTRACT_BITMAP are not available on sharded storage");
  if ((p->compat_flags & RSC_EXTRACT_BITMAP) && !(ctx->bitmap_beta > 0.0))
    return fail(ctx, RSC_E_STATE, "ransac_run: RSC_EXTRACT_BITMAP needs rsc_ctx_set_bitmap(ctx, beta, eight) first");
  const bool cells = (p->compat_flags & RSC_SAMPLER_OCTREE) != 0;
  const bool prog = (p->compat_flags & RSC_SCORE_PROGRESSIVE) != 0;
  // cell sampler: the level weights are refreshed every `lw_period` iterations (params.lw_period; 1 = after every
  // iteration, the reference's schedule, iterations.jl:148); a batch never crosses a refresh, so the results for a
  // given period do not depend on the batch size
  const int lw_period = cells ? std::max(1, (int)p->lw_period) : 1;
  const int64_t N = cloud->n_global > 0 ? cloud->n_global : cloud->n;
  const int64_t M = sub.m_global > 0 ? sub.m_global : sub.m;
  const int S = p->minsubsetN;
  const int ntypes = order ? order->n : p->n_shape_types;
  const int maxnew = S * ntypes;
  // user shapes (rsc_ransac_run_user): their fit, score and mask kernels join K1, K2, K4 and K5; such runs never take
  // the culled scorer, which knows the built-in types only
  const FitOrder* uo = order && order->has_user ? order : nullptr;
  const PointSet sps = subset_slice(cloud, sub, ranged);
  const int64_t sps_word0 = sps.enabled - sub.enabled;
  // small-batch scorer (rsc_small.cu), within kSmallMaxCands / kSmallMaxEvals
  const bool use_small = getenv("RSC_NO_SMALL") == nullptr;
  // K5 on the subset's Morton view: the culled scorer (0: never, 1: for a large store, 2: always; read per run)
  const int k5_cull_mode = getenv("RSC_LOOP_CULL") ? atoi(getenv("RSC_LOOP_CULL")) : 1;
  long long rate_seen = -1;  // recent number of new candidates per iteration (-1: no batch yet)
  const int Bmax = getenv("RSC_BATCH") ? std::max(1, std::min(kMaxBatch, atoi(getenv("RSC_BATCH")))) : 16;
  const int Bmin = getenv("RSC_BATCH_MIN") ? std::max(1, std::min(Bmax, atoi(getenv("RSC_BATCH_MIN")))) : std::min(8, Bmax);
  // Unless RSC_BATCH / RSC_BATCH_MIN are set the batch sizes follow the run: a batch is cut at the first extraction and
  // the sets drawn behind the cut are fitted for nothing, so batches should not be much longer than the usual gap
  // between two extractions (c4: an extraction every ~11 iterations -> 6 rising to 12 measured best (13.7 ms of K1 + K2
  // against 15.0 at 8..16); c5: every ~17 -> 8..16).  `gap` = smoothed iterations per extraction; results do not
  // depend on any of this.  Host-decided runs follow the same policy: on c4 (B200, 1000 W) the cell sampler's loop
  // (lw_period 16) and progressive scoring's took the same time as under a doubling-to-16 / 8-after-an-extraction
  // rule, within the run-to-run spread.
  const bool adapt = !getenv("RSC_BATCH") && !getenv("RSC_BATCH_MIN");
  double gap = 16.0;
  int since_extract = 0;
  int B = 1;
  const bool trace = getenv("RSC_TRACE") != nullptr;
  double t_fit = 0, t_score = 0, t_extract = 0;
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto secs = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
    return std::chrono::duration<double>(b - a).count();
  };
  auto sync = [&]() {
    ++run->syncs;
    return cudaStreamSynchronize(st);
  };
#define RUN_CUDA(expr)                \
  do {                                \
    cudaError_t _e = (expr);          \
    if (_e != cudaSuccess) return fail_cuda(ctx, _e, #expr); \
  } while (0)

  // pinned mirror of what the host reads (seg bounds, decision record, K5 summary; the device state and the
  // overflow flag for the host decision)
  struct HostIo {
    int32_t seg[kMaxBatch + 2];
    BatchRec rec;
    K5Host k5;
    LoopDev dev;
    int32_t ovf;
  };
  if (ctx->pinned_cap < sizeof(HostIo)) {
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    ctx->pinned = nullptr, ctx->pinned_cap = 0;
    RUN_CUDA(cudaMallocHost(&ctx->pinned, sizeof(HostIo) + 256));
    ctx->pinned_cap = sizeof(HostIo) + 256;
  }
  HostIo* hio = static_cast<HostIo*>(ctx->pinned);
  RUN_CUDA(ls.hostio.ensure(sizeof(LoopDev) + sizeof(K5Host) + 64));
  LoopDev* dev = ls.hostio.as<LoopDev>();
  K5Host* dk5 = reinterpret_cast<K5Host*>(dev + 1);
  RUN_CUDA(cudaMemsetAsync(dev, 0, sizeof(LoopDev) + sizeof(K5Host), st));

  // sharded storage: whatever the ranks did to their local masks, the replicated one follows them
  if (shard && (rc = shard_sync_enabled(cloud, st))) return rc;
  int64_t n_enabled = 0, n_enabled_local = rsc_cloud_count_enabled(cloud);
  if (n_enabled_local < 0) return fail(ctx, RSC_E_CUDA, "ransac_run: counting the enabled points failed");
  ++run->syncs;
  if (shard) {
    n_enabled = count_mask_bits(ctx, cloud->g_enabled, cloud->g_words);
    if (n_enabled < 0) return fail(ctx, RSC_E_CUDA, "ransac_run: counting the enabled points failed");
    ++run->syncs;
  } else {
    n_enabled = n_enabled_local;
  }
  run->device = ctx->device;
  RUN_CUDA(cudaMalloc(&run->d_idx, (size_t)(n_enabled_local > 0 ? n_enabled_local : 1) * sizeof(int64_t)));  // a point is extracted at most once

  RUN_CUDA(ls.newcnt.ensure((size_t)2 * maxnew * Bmax * 4 + 64));
  if ((rc = fit_reserve(ctx, p, S * Bmax, ntypes))) return rc;
  RUN_CUDA(store.reserve((size_t)std::min<int64_t>((int64_t)maxnew * Bmax, 1 << 20), st));
  DecideParams q;
  q.N = N, q.M = M, q.tau = p->tau, q.prob_det = p->prob_det;
  q.S = S, q.drawN = p->drawN, q.extract_s = p->extract_s, q.terminate_s = p->terminate_s;
  bool terminated = false;
  std::vector<int32_t> newscore;  // progressive scoring: the new candidates' subset-1 scores, for the host decision
  std::vector<uint32_t> keep_h;   // progressive scoring: K5's survivors, to compact the host's mirror of the store

  for (int k = 1; k <= p->itermax && !terminated;) {
    if (n_enabled < p->tau) break;  // iterations.jl:75
    int nb = std::min(B, p->itermax - k + 1);
    if (cells) nb = std::min(nb, lw_period - (k - 1) % lw_period);  // up to the next refresh of the level weights
    const auto tk0 = now();
    ++run->batches;
    // ---- K1: nb * minsubsetN minimal sets -> candidates (device, compacted in reference order) ----
    FitScratch fs;
    double cum[11];
    if (cells) rsc_level_cumsum(run->levelweight, run->nlevels, cum);
    // (segment bounds of the batch's iterations: from the compaction itself when an iteration is whole groups of sets)
    const bool seg_fused = S % 128 == 0;
    if ((rc = fit_enqueue(ctx, cloud, cells ? 3 : 2, p, p->drawN, nullptr, nullptr, nullptr, S * nb, seed, (uint64_t)(k - 1) * S, st, &fs,
                          cells ? cum : nullptr, seg_fused ? dev->seg : nullptr, S, nb, order)))
      return rc;
    if (!seg_fused) {
      seg_bounds_kernel<<<1, 96, 0, st>>>(fs.out_set, fs.total, S, nb, dev->seg);
      RUN_CUDA(cudaGetLastError());
    }
    const int store_n0 = store.n;
    // ---- K2 on subset 1 + K3 for `n` new candidates: their number, or (d_total, the sync-free path) the size of a
    // launch whose true number of candidates stays on the device.  The dense scorer's overflow flag rides behind the
    // counts, so that a sharded run decides to repeat collectively.  (The cell sampler decides on the host, so its
    // batches never take the sync-free path: `n` is exact for its level statistics.)
    auto score_batch = [&](int n, const unsigned long long* d_total) -> int32_t {
      if (cells) RUN_CUDA(cudaMemsetAsync(dev->lv, 0, (size_t)nb * sizeof(dev->lv[0]), st));  // (an empty batch adds nothing)
      if (n > 0) {
        RUN_CUDA(store.reserve((size_t)store_n0 + n, st));
        RUN_CUDA(ls.newcnt.ensure((size_t)2 * n * 4 + 64));
        rsc_cand* dst = store.cands[store.cur].as<rsc_cand>() + store_n0;
        int32_t* cv = ls.newcnt.as<int32_t>();
        int32_t* ce = cv + n;
        if (d_total) {
          append_new_kernel<<<std::max(1, std::min(n * 4 / 256, 64)), 256, 0, st>>>(fs.out, d_total, n, dst);
          RUN_CUDA(cudaGetLastError());
          if ((rc = score_small_enqueue(ctx, cloud, sps, th, dst, n, d_total, cv, ce, st))) return rc;
        } else {
          RUN_CUDA(cudaMemcpyAsync(dst, fs.out, (size_t)n * sizeof(rsc_cand), cudaMemcpyDeviceToDevice, st));
          // (the culled scorer on the subset's Morton view when the batch is large: same counts)
          if ((rc = loop_score_new(ctx, cloud, sub, sps, !ranged && !uo, th, dst, n, cv, ce, cv + 2 * n, st))) return rc;
        }
        if (uo && (rc = user_score_enqueue(ctx, *uo, sps, dst, n, d_total, cv, ce, st))) return rc;
        if (coll && ctx->allreduce(ctx->allreduce_user, cv, (int64_t)2 * n + (d_total ? 0 : 1), (void*)st))
          return fail(ctx, RSC_E_NCCL, "ransac_run: all-reduce of the counts failed");
        int32_t* score = store.score[store.cur].as<int32_t>();
        uint8_t* flags = store.flags[store.cur].as<uint8_t>();
        finish_new_kernel<<<d_total ? std::max(1, std::min(n / 256, 64)) : (n + 255) / 256, 256, 0, st>>>(
            dst, fs.total, n, cv, ce, th.honour_enabled, score + store_n0, flags + store_n0);
        RUN_CUDA(cudaGetLastError());
        seg_argmax_kernel<<<nb, 256, 0, st>>>(score, flags, dev->seg, store_n0, dev->seg_keys, n);  // never reads past the launch
        RUN_CUDA(cudaGetLastError());
        if (cells) {
          level_stats_kernel<<<(n + 255) / 256, 256, 0, st>>>(fs.out_set, fs.level, score + store_n0, n, S, dev->lv);
          RUN_CUDA(cudaGetLastError());
        }
      } else {
        RUN_CUDA(cudaMemsetAsync(dev->seg_keys, 0xff, sizeof(dev->seg_keys), st));  // -1: no new candidate
      }
      if (store_n0 >= 1)
        RUN_CUDA(argmax_enqueue(store.score[store.cur].as<int32_t>(), store.flags[store.cur].as<uint8_t>(), store_n0, dev->oldbest,
                                ctx->sm_count, st));
      return RSC_OK;
    };
    // ---- the decision of the batch -> hio->rec, with one synchronisation: decide_kernel, or the host's ----
    auto decide = [&](const int32_t* d_ovf, int cap) -> int32_t {
      if (!host) {
        decide_kernel<<<1, kMaxBatch, 0, st>>>(dev, d_ovf, store_n0, nb, k, q, store.cands[store.cur].as<rsc_cand>(), cap);
        RUN_CUDA(cudaGetLastError());
        RUN_CUDA(cudaMemcpyAsync(&hio->rec, &dev->rec, sizeof(BatchRec), cudaMemcpyDeviceToHost, st));
        RUN_CUDA(sync());
        return RSC_OK;
      }
      const int n_new = hio->seg[nb];  // (host decisions never take the sync-free path: the bounds are on the host)
      // (what it reads leads the device state: the arg-maxes, the segment bounds and this batch's level rows)
      RUN_CUDA(cudaMemcpyAsync(&hio->dev, dev, offsetof(LoopDev, lv) + (cells ? nb : 0) * sizeof(dev->lv[0]), cudaMemcpyDeviceToHost, st));
      hio->ovf = 0;
      if (d_ovf) RUN_CUDA(cudaMemcpyAsync(&hio->ovf, d_ovf, 4, cudaMemcpyDeviceToHost, st));
      if (prog && n_new > 0) {
        newscore.resize(n_new);
        RUN_CUDA(cudaMemcpyAsync(newscore.data(), store.score[store.cur].as<int32_t>() + store_n0, (size_t)n_new * 4,
                                 cudaMemcpyDeviceToHost, st));
      }
      RUN_CUDA(sync());
      hio->rec.ovf = hio->ovf ? 1 : 0;
      return hio->ovf ? RSC_OK : host_decide(*host, hio->dev, newscore.data(), store_n0, nb, k, &hio->rec);
    };
    // ---- sync-free path: K2 for a small batch, sized by a PREDICTION of the number of new candidates ----
    // (4 x the largest per-iteration yield seen so far; the true number stays on the device.  If more turn up,
    // decide_kernel says so and the batch is scored again the classic way.)  The host decision needs the keys on
    // the host, so it always takes the classic path.
    int cap_new = -1;
    if (use_small && !host && rate_seen >= 0) {
      long long want = std::max<long long>(128, 4ll * rate_seen * nb + 64);
      if (const char* e = getenv("RSC_SMALL_CAP")) want = std::max(1, atoi(e));  // test hook: force undersized launches
      const long long cap = std::min<long long>((want + 127) / 128 * 128, (long long)maxnew * nb);
      // the launch is sized for `cap` but its cost follows the ACTUAL number (expected: cap / 4)
      if (cap <= kSmallMaxCands && (double)(cap / 4) * (double)std::max<int64_t>(sps.n_pad, 1) <= kSmallMaxEvals) cap_new = (int)cap;
    }
    bool scored = false;
    int n_new = 0;
    if (cap_new > 0) {
      if ((rc = score_batch(cap_new, fs.total)) || (rc = decide(nullptr, cap_new))) return rc;
      scored = hio->rec.ovf == 0;
      n_new = hio->rec.n_new;  // (also known from the record of an undersized attempt)
      if (scored) ctx->stats.evals += (int64_t)n_new * sps.n, ctx->stats.cands_scored += n_new;
    } else {
      RUN_CUDA(cudaMemcpyAsync(hio->seg, dev->seg, (size_t)(nb + 1) * 4, cudaMemcpyDeviceToHost, st));
      RUN_CUDA(sync());
      n_new = hio->seg[nb];
    }
    rate_seen = std::max<long long>((n_new + nb - 1) / nb, rate_seen / 2);  // the yield falls as shapes are extracted: follow it
    const auto tk1 = now();
    t_fit += secs(tk0, tk1);
    // ---- classic path: K2 (tiled or culled) + K3, repeated with a larger guard-band queue if that overflowed ----
    for (int attempt = 0; !scored; ++attempt) {
      if ((rc = score_batch(n_new, nullptr)) || (rc = decide(n_new > 0 ? ls.newcnt.as<int32_t>() + 2 * n_new : nullptr, -1))) return rc;
      if (!hio->rec.ovf) break;
      if (attempt >= 4) return fail(ctx, RSC_E_STATE, "ransac_run: guard-band queue kept overflowing");
      if ((rc = grow_guard_queue(ctx))) return rc;
    }
    const BatchRec rec = hio->rec;
    const auto tk2 = now();
    t_score += secs(tk1, tk2);
    run->iterations = rec.iterations;
    store.n = rec.store_n;
    terminated = rec.terminated != 0;
    if (rec.extract) {
      // K5's source of the newly disabled points: the subset's Morton view when it has one and the run scores the
      // whole subset (the points then come out spatially sorted, and the culled scorer can take them: the SET of
      // points is the same), else this rank's slice.  Its enabled words of before the extraction are kept.
      const bool view = sub.cen != nullptr && !coll;
      const PointSet src = view ? view_subset_morton(&sub) : sps;
      const int64_t swords = sub.m_pad / 32;
      RUN_CUDA(ls.olden.ensure((size_t)swords * 4));
      RUN_CUDA(cudaMemcpyAsync(ls.olden.p, view ? sub.cen : sub.enabled, (size_t)swords * 4, cudaMemcpyDeviceToDevice, st));
      // ---- K4: refit over this rank's points, invalidate them ----
      rsc_cand shape = rec.best;
      if (p->compat_flags & RSC_REFIT_LSQ) {  // extension: the paper's least-squares refit within 3 eps
        if ((rc = lsq_refine(cloud, p, 3.0, &shape, nullptr, nullptr, st))) return rc;
        ++run->syncs;
      }
      Thresh thr = th;
      thr.honour_enabled = 0xFu;
      if (shape.type >= RSC_USER_TYPE0) {
        if ((rc = user_refit_mask_enqueue(cloud, *uo, shape, st))) return rc;
      } else if ((rc = refit_mask_enqueue(cloud, thr, shape, st))) {
        return rc;
      }
      if (p->compat_flags & RSC_EXTRACT_BITMAP) {  // extension: only the largest connected component in parameter space
        unsigned long long tot = 0;
        RUN_CUDA(cudaMemcpyAsync(&tot, ctx->misc2.p, 8, cudaMemcpyDeviceToHost, st));
        RUN_CUDA(sync());
        if (tot > 0) {
          RUN_CUDA(ctx->misc.ensure((size_t)tot * 16));
          int64_t* lst = ctx->misc.as<int64_t>();
          if ((rc = refit_write_enqueue(cloud, lst, false, st))) return rc;  // the list, nothing disabled yet
          int64_t kept = 0;
          if ((rc = bitmap_filter_dev(cloud, shape, ctx->bitmap_beta, ctx->bitmap_eight != 0, lst, (int64_t)tot, lst + tot, &kept, nullptr, st)))
            return rc;
          ++run->syncs;
          if ((rc = refit_mask_from_list(cloud, lst + tot, kept, st))) return rc;
        }
      }
      // the inlier mask words (ctx->idxbuf) and this rank's inlier count (ctx->misc2) are on the device
      if ((rc = refit_write_enqueue(cloud, run->d_idx + run->off.back(), true, st))) return rc;
      if (shard) {  // the replicated whole-cloud mask follows; the ranks' inlier counts ride along
        RUN_CUDA(cudaMemcpyAsync(dev->tot_global, ctx->misc2.p, 8, cudaMemcpyDeviceToDevice, st));
        if ((rc = shard_clear_enabled(cloud, ctx->idxbuf.as<uint32_t>(), dev->tot_global, 1, dev->tot_global, st))) return rc;
      }
      // ---- K5: drop the best and every candidate compatible with a newly disabled subset point ----
      // (the bitmap filter only removes points from the list, so the gathered form's bound still holds with it)
      const int nst = store.n;
      K5In kin;
      kin.nst = nst;
      kin.src = src, kin.view = view, kin.view_tiles = static_cast<const float4*>(sub.ctiles);
      kin.olden = ls.olden.as<uint32_t>(), kin.old_word0 = view ? 0 : sps_word0;
      kin.new_en = view ? sub.cen : sub.enabled, kin.swords = swords;
      kin.bound = rec.best_score;
      kin.masked = (p->compat_flags & RSC_REFIT_LSQ) != 0 || getenv("RSC_K5_MASKED") != nullptr;
      kin.cull_mode = k5_cull_mode, kin.use_small = use_small, kin.uo = uo, kin.coll = coll;
      K5Out ko;
      int nxt = store.cur ^ 1;
      for (int attempt = 0;; ++attempt) {
        kin.cands = store.cands[store.cur].as<rsc_cand>();
        if ((rc = k5_hits(ctx, cloud, kin, th, &ko, st))) return rc;
        if ((rc = k5_compact(ko, nst, rec.best_idx, store.cands[store.cur].as<rsc_cand>(), store.score[store.cur].as<int32_t>(),
                             store.flags[store.cur].as<uint8_t>(), store.cands[nxt].as<rsc_cand>(), store.score[nxt].as<int32_t>(),
                             store.flags[nxt].as<uint8_t>(), ctx, st)))
          return rc;
        k5_pack_kernel<<<1, 1, 0, st>>>(dev, ko.ktot, ko.hit + nst, ko.hit + nst + 1, ctx->misc2.as<unsigned long long>(), dk5);
        RUN_CUDA(cudaGetLastError());
        RUN_CUDA(cudaMemcpyAsync(&hio->k5, dk5, sizeof(K5Host), cudaMemcpyDeviceToHost, st));
        if (host && prog) {
          keep_h.resize(nst);
          RUN_CUDA(cudaMemcpyAsync(keep_h.data(), ko.keep, (size_t)nst * 4, cudaMemcpyDeviceToHost, st));
        }
        RUN_CUDA(sync());
        if (!hio->k5.ovf) break;
        if (hio->k5.ovf & 2) {  // (not expected) more newly disabled points than the bound: masked form
          kin.masked = true;
          continue;
        }
        // invalidate_kernel marked flags of this attempt: they only ever go from alive to dead on hits that
        // can only grow with the complete counts, so repeating on the same flags is safe
        if (attempt >= 4) return fail(ctx, RSC_E_STATE, "ransac_run: guard-band queue kept overflowing");
        if ((rc = grow_guard_queue(ctx))) return rc;
      }
      if (host && prog) host_compacted(*host, keep_h);
      const int64_t total_local = (int64_t)hio->k5.total_local;
      const int64_t total = shard ? (int64_t)hio->k5.tot_global : total_local;
      run->shapes.push_back(shape);
      run->off.push_back(run->off.back() + total_local);
      run->total.push_back(total);
      n_enabled -= total;
      store.cur = nxt;
      store.n = (int)hio->k5.kept;
      t_extract += secs(tk2, now());
    }
    k += rec.used;
    since_extract += rec.used;
    if (rec.extract) {
      gap = 0.5 * gap + 0.5 * (double)since_extract;
      since_extract = 0;
    }
    if (adapt) {
      const int bmax = std::max(8, std::min(Bmax, (int)(gap + 1.5)));
      B = rec.extract ? std::max(4, std::min(bmax, (int)(0.5 * gap + 0.5))) : std::min(2 * B, bmax);
    } else {
      B = rec.extract ? Bmin : std::min(2 * B, Bmax);
    }
  }
  RUN_CUDA(sync());
  if (trace)
    fprintf(stderr,
            "[rsc_ransac_run] iterations %d shapes %zu batches %d syncs %d | sample+fit %.1f ms, score+decide %.1f ms, "
            "refit+invalidate %.1f ms | all-reduces %lld (%.1f MB)\n",
            run->iterations, run->shapes.size(), run->batches, run->syncs, 1e3 * t_fit, 1e3 * t_score, 1e3 * t_extract,
            (long long)ctx->allreduce_calls, ctx->allreduce_bytes / 1e6);
  return RSC_OK;
#undef RUN_CUDA
}

}  // namespace rsc

// Test hook: K5 on its own (include/rsc.h rsc_debug_k5_hits), through k5_hits and k5_compact as the loop calls them.
extern "C" int32_t rsc_debug_k5_hits(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cands, int32_t nst,
                                     const uint64_t* new_enabled, int32_t bound, int32_t form, int32_t best, int32_t* hit,
                                     int32_t* flags, int32_t* survivors, int32_t* n_survivors) {
  using namespace rsc;
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (nst <= 0 || !cands || !new_enabled || !hit || best < -1 || best >= nst || (form & ~3))
    return fail(ctx, RSC_E_ARG, "debug_k5_hits: bad arguments (nst >= 1, -1 <= best < nst, form in 0..3)");
  if (!params) return fail(ctx, RSC_E_ARG, "params is null");
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  int32_t rc = cloud_ready(cloud);
  if (rc) return rc;
  if (cloud->is_shard() || cloud->subsets.empty() || !cloud->subsets[0].soa)
    return fail(ctx, RSC_E_STATE, "debug_k5_hits: needs subset 0 uploaded (rsc_cloud_set_subset) on an unsharded cloud");
  cudaStream_t st = ctx->stream;
  rsc_subset& sub = cloud->subsets[0];
  const bool view = (form & 2) != 0;
  if (view && (rc = subset_cull_view(cloud, sub, st))) return rc;
  if (!ctx->loop_scratch) ctx->loop_scratch = new LoopScratch();
  LoopScratch& ls = *static_cast<LoopScratch*>(ctx->loop_scratch);
  const int64_t swords = sub.m_pad / 32;
  // the store: candidates, scores = their indices (so the compaction reports who survived), all alive
  RSC_CUDA(ctx, ls.store.reserve((size_t)nst, st));
  rsc_cand* c0 = ls.store.cands[0].as<rsc_cand>();
  int32_t* s0 = ls.store.score[0].as<int32_t>();
  std::vector<int32_t> iota(nst);
  for (int i = 0; i < nst; ++i) iota[i] = i;
  RSC_CUDA(ctx, cudaMemcpyAsync(c0, cands, (size_t)nst * sizeof(rsc_cand), cudaMemcpyHostToDevice, st));
  RSC_CUDA(ctx, cudaMemcpyAsync(s0, iota.data(), (size_t)nst * 4, cudaMemcpyHostToDevice, st));
  RSC_CUDA(ctx, cudaMemsetAsync(ls.store.flags[0].p, 1, (size_t)nst, st));
  // the enabled words of before, then the cloud's mask becomes new_enabled (the subset and its view follow)
  RSC_CUDA(ctx, ls.olden.ensure((size_t)swords * 4));
  RSC_CUDA(ctx, cudaMemcpyAsync(ls.olden.p, view ? sub.cen : sub.enabled, (size_t)swords * 4, cudaMemcpyDeviceToDevice, st));
  if ((rc = rsc_cloud_set_enabled(cloud, new_enabled))) return rc;
  K5In in;
  in.cands = c0, in.nst = nst;
  in.src = view ? view_subset_morton(&sub) : subset_slice(cloud, sub, false);
  in.view = view, in.view_tiles = static_cast<const float4*>(sub.ctiles);
  in.olden = ls.olden.as<uint32_t>(), in.old_word0 = 0;
  in.new_en = view ? sub.cen : sub.enabled, in.swords = swords;
  in.bound = bound;
  in.masked = (form & 1) != 0;
  in.cull_mode = getenv("RSC_LOOP_CULL") ? atoi(getenv("RSC_LOOP_CULL")) : 1;
  in.use_small = getenv("RSC_NO_SMALL") == nullptr;
  in.uo = nullptr, in.coll = false;
  const Thresh th = make_thresh(params);
  K5Out ko;
  int32_t fl[2] = {0, 0};
  for (int attempt = 0;; ++attempt) {  // the loop's repeats: the masked form when the scratch set is too small
    if ((rc = k5_hits(ctx, cloud, in, th, &ko, st))) return rc;
    int32_t f[2];
    RSC_CUDA(ctx, cudaMemcpyAsync(f, ko.hit + nst, 8, cudaMemcpyDeviceToHost, st));
    RSC_CUDA(ctx, cudaStreamSynchronize(st));
    if (attempt == 0) fl[0] = f[0], fl[1] = f[1];
    if (f[1] && !in.masked) {
      in.masked = true;
      continue;
    }
    if (f[0]) {
      if (attempt >= 4) return fail(ctx, RSC_E_STATE, "debug_k5_hits: guard-band queue kept overflowing");
      if ((rc = grow_guard_queue(ctx))) return rc;
      continue;
    }
    break;
  }
  if ((rc = k5_compact(ko, nst, best, c0, s0, ls.store.flags[0].as<uint8_t>(), ls.store.cands[1].as<rsc_cand>(),
                       ls.store.score[1].as<int32_t>(), ls.store.flags[1].as<uint8_t>(), ctx, st)))
    return rc;
  unsigned long long kept = 0;
  RSC_CUDA(ctx, cudaMemcpyAsync(hit, ko.hit, (size_t)nst * 4, cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaMemcpyAsync(&kept, ko.ktot, 8, cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaStreamSynchronize(st));
  if (survivors && kept)
    RSC_CUDA(ctx, cudaMemcpy(survivors, ls.store.score[1].p, (size_t)kept * 4, cudaMemcpyDeviceToHost));
  if (n_survivors) *n_survivors = (int32_t)kept;
  if (flags) flags[0] = fl[0], flags[1] = fl[1];
  return RSC_OK;
}
