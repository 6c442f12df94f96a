// rsc_run.cu -- the whole RANSAC loop for the built-in shapes behind one C-ABI call
// (ransac(pc, params; ...): iterations.jl:35-162), plus K3 (score bookkeeping: findhighestscore,
// fitting.jl:140-158) and K5 (removeinvalidshapes!, fitting.jl:209-221) on the device.
//
// Per iteration: K1 sample+fit (rsc_fit.cu) -> K2 score of the new candidates on subset 1
// (rsc_score.cu; iterations.jl:95 hard-wires subset 1) -> device arg-max over the candidate store
// -> host decides with prob() (utilities.jl:262) -> on extraction K4 refit over the whole cloud
// (rsc_extract.cu), enabled bits cleared, store invalidated and compacted.
//
// Iterations run in SPECULATIVE BATCHES of up to 16: as long as nothing is extracted the enabled mask
// is unchanged, so the iterations of a batch sample (same Philox set ids as separate iterations), fit
// and score together; the host then walks the batch with the reference's bookkeeping, iteration by
// iteration, and cuts it at the first extraction or at termination (see the loop below).
//
// K5 without stored inlier lists: every stored candidate's subset-1 inliers are enabled at the time
// of an extraction (the reference removes any candidate with a disabled inlier at each extraction,
// and new candidates only count enabled points), so "has a now-disabled inlier" == "is compatible
// with one of the NEWLY disabled subset-1 points".  Those few points are gathered into a scratch
// point set and all stored candidates are scored against it with the same K2 kernel.  Spheres,
// whose reference scorer ignores `isenabled` (Q4), additionally die at the first extraction after
// they were scored if they matched any already-disabled point.
//
// Sharding (one process per GPU): the cloud is replicated, every rank samples identically
// (counter-based Philox) and scores only its point range; per-candidate counts and the refit's
// inlier-mask words are summed across ranks through the all-reduce callback (NCCL on the host side).
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <vector>

#include "rsc_loop.cuh"

namespace rsc {

// from rsc_fit.cu
}  // namespace rsc
extern "C" void rsc_level_cumsum(const double* levelweight, int32_t nlevels, double* cum);
extern "C" void rsc_update_levelweight(double* levelweight, const double* levelscore, int32_t nlevels);
namespace rsc {
__global__ void scan_u32_kernel(const uint32_t* __restrict__ counts, int n, unsigned long long* __restrict__ offsets,
                                unsigned long long* __restrict__ out_total);

// ---- progressive subset scoring (extension, SURVEY 8(f)-2; iterations.jl:110 "TODO: refine if best.overlap") ----
__global__ void gather_cands_kernel(const rsc_cand* __restrict__ store, const int32_t* __restrict__ idx, int n,
                                    rsc_cand* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = store[idx[i]];
}

// Host mirror of the store's scores while refining: candidate i has been scored on subsets 1..lvl[i],
// sigma[i] compatible points among their M[i] points; interval from the union, in float64 without the
// reference's Int64 wrap (Q9) -- same operation order as oracle/ransac_oracle.py::estimatescore_f64.
struct ProgMirror {
  std::vector<int64_t> sigma, M, sigma1;  // sigma1: the subset-1 count (what a refined score falls back to after an extraction)
  std::vector<int32_t> lvl;
  std::vector<double> lo, hi, E;
  size_t size() const { return E.size(); }
  void clear() { sigma.clear(), M.clear(), sigma1.clear(), lvl.clear(), lo.clear(), hi.clear(), E.clear(); }
  static void interval(int64_t m, int64_t N, int64_t sg, double* lo, double* hi, double* E) {
    const double Np = (double)(-2 - m), x = (double)(-2 - N), n = (double)(-1 - sg);
    const double xn = x * n;
    const double sq_ = (xn * (Np - x)) * (Np - n) / (Np - 1.0);
    const double sq = sq_ < 0 ? 0.0 : sqrt(sq_);
    const double a = -1 - (xn + sq) / Np, b = -1 - (xn - sq) / Np;
    *lo = a < b ? a : b;
    *hi = a < b ? b : a;
    *E = (*lo + *hi) / 2;
  }
  void push(int64_t sg, int64_t m, int64_t N) {
    double a, b, e;
    interval(m, N, sg, &a, &b, &e);
    sigma.push_back(sg), M.push_back(m), sigma1.push_back(sg), lvl.push_back(1), lo.push_back(a), hi.push_back(b), E.push_back(e);
  }
  void add(size_t i, int64_t sg, int64_t m, int64_t N) {
    sigma[i] += sg, M[i] += m, lvl[i] += 1;
    interval(M[i], N, sigma[i], &lo[i], &hi[i], &E[i]);
  }
  int best() const {  // findhighestscore (fitting.jl:140-150): strict >, first wins
    if (E.empty()) return -1;
    int ind = 0;
    for (size_t i = 1; i < E.size(); ++i)
      if (E[i] > E[ind]) ind = (int)i;
    return ind;
  }
  bool overlap(size_t i, size_t j) const {  // isoverlap (confidenceintervals.jl:29-36)
    if (lo[i] == lo[j]) return true;
    return lo[i] < lo[j] ? lo[j] <= hi[i] : lo[i] <= hi[j];
  }
  void compact(const std::vector<uint32_t>& keep) {
    size_t o = 0;
    for (size_t i = 0; i < E.size(); ++i)
      if (keep[i]) sigma[o] = sigma[i], M[o] = M[i], sigma1[o] = sigma1[i], lvl[o] = lvl[i], lo[o] = lo[i], hi[o] = hi[i], E[o] = E[i], ++o;
    sigma.resize(o), M.resize(o), sigma1.resize(o), lvl.resize(o), lo.resize(o), hi.resize(o), E.resize(o);
  }
  // after an extraction: the survivors' subset-1 inliers are all still enabled, but their inliers in the subsets
  // 2..r may just have been extracted -- a refined score falls back to the (exact) subset-1 score
  void reset_refined(int64_t m1, int64_t N) {
    for (size_t i = 0; i < E.size(); ++i)
      if (lvl[i] > 1) {
        sigma[i] = sigma1[i], M[i] = m1, lvl[i] = 1;
        interval(m1, N, sigma1[i], &lo[i], &hi[i], &E[i]);
      }
  }
};

void loop_scratch_free(rsc_ctx* ctx) {
  LoopScratch* ls = static_cast<LoopScratch*>(ctx->loop_scratch);
  if (!ls) return;
  ls->store.release();
  ls->newcnt.release(), ls->hostio.release(), ls->olden.release(), ls->nscratch.release(), ls->nidx.release(), ls->nvalid.release(), ls->nmeta.release();
  ls->lvbuf.release(), ls->prog.release(), ls->ntiles.release();
  delete ls;
  ctx->loop_scratch = nullptr;
}

static double prob_(double n, double s, double N, double k) { return 1 - pow(1 - pow(n / N, k), s); }

}  // namespace rsc

using namespace rsc;

// Result of one run.  The inlier index lists stay in device memory (one arena, disjoint lists, in
// extraction order) until the caller fetches them with rsc_run_inpoints: no per-extraction host
// buffer, no device->host traffic inside the loop.
// per octree level: number of new candidates and the sum of their scores (fitting.jl:184 adds E(score)
// per candidate; E is affine in the count, so the host adds the closed form of the sum)
__global__ void level_stats_kernel(const int32_t* __restrict__ out_set, const int32_t* __restrict__ set_level,
                                   const int32_t* __restrict__ score, int n, int S, long long* __restrict__ lv /*[nb][2][11]*/) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int l = set_level[out_set[i]] - 1;
  if (l < 0 || l >= 11) return;
  long long* row = lv + (size_t)(out_set[i] / S) * 22;  // the batch iteration the candidate's minimal set belongs to
  atomicAdd((unsigned long long*)(row + l), 1ull);
  atomicAdd((unsigned long long*)(row + 11 + l), (unsigned long long)score[i]);
}

extern "C" {

int32_t rsc_ctx_set_allreduce(rsc_ctx* ctx, rsc_allreduce_fn fn, void* user) {
  if (!ctx) return RSC_E_ARG;
  ctx->allreduce = fn;
  ctx->allreduce_user = user;
  return RSC_OK;
}

int32_t rsc_cloud_set_range(rsc_cloud* cloud, int64_t lo, int64_t hi) {
  if (!cloud) return RSC_E_ARG;
  if (cloud->exact()) return fail(cloud->ctx, RSC_E_STATE, "set_range: ranged (replicated multi-GPU) runs do not support exact clouds yet");
  // 2048 = points per refit CTA (rsc_extract.cu); lo == hi is an empty rank (clouds smaller than 2048 x ranks)
  if (lo < 0 || hi > cloud->n_pad || lo > hi || (lo % 2048 && lo != cloud->n) || (hi % 2048 && hi != cloud->n_pad && hi != cloud->n))
    return fail(cloud->ctx, RSC_E_ARG, "set_range: range bounds must be multiples of 2048 points (or the cloud size)");
  cloud->range_lo = lo >= cloud->n ? cloud->n_pad : lo;
  cloud->range_hi = hi >= cloud->n ? cloud->n_pad : hi;
  cloud->range_set = true;
  return RSC_OK;
}

int32_t rsc_ransac_run_user(rsc_cloud* cloud, const rsc_params* p, const void* order, int32_t norder, uint64_t seed,
                            rsc_run** out) {
  if (!cloud || !out) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  *out = nullptr;
  if (!p) return fail(ctx, RSC_E_ARG, "ransac_run_user: params is null");
  FitOrder fo;
  if (int32_t rc = make_fit_order(ctx, static_cast<const rsc_shape_slot*>(order), norder, &fo, "ransac_run_user")) return rc;
  if (norder < 1) return fail(ctx, RSC_E_ARG, "ransac_run_user: an empty fit order");
  if (p->drawN < 3 || p->drawN > 8) return fail(ctx, RSC_E_ARG, "ransac_run_user: drawN must be 3..8");
  if (p->minsubsetN < 1) return fail(ctx, RSC_E_ARG, "ransac_run_user: nothing to sample/fit");
  if (p->extract_s < 0 || p->extract_s > 2 || p->terminate_s < 0 || p->terminate_s > 2)
    return fail(ctx, RSC_E_ARG, "ransac_run_user: extract_s/terminate_s must be RSC_S_*");
  if (cloud->is_shard() || cloud->range_set) return fail(ctx, RSC_E_STATE, "ransac_run_user: sharded or ranged clouds are not supported");
  if (p->compat_flags & (RSC_SAMPLER_OCTREE | RSC_SCORE_PROGRESSIVE | RSC_REFIT_LSQ | RSC_EXTRACT_BITMAP))
    return fail(ctx, RSC_E_STATE, "ransac_run_user: the extension switches are not available with a fit order");
  if (getenv("RSC_LOOP_HOSTWALK")) return fail(ctx, RSC_E_STATE, "ransac_run_user: runs the device loop only (RSC_LOOP_HOSTWALK is set)");
  if (cloud->subsets.empty() || !cloud->subsets[0].soa)
    return fail(ctx, RSC_E_STATE, "ransac_run_user: subset 1 is not uploaded (rsc_cloud_set_subset(cloud, 0, ...))");
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if (int32_t rcr = cloud_ready(cloud)) return rcr;
  const auto t0 = std::chrono::steady_clock::now();
  rsc_run* run = new rsc_run();
  run->ctx = ctx;
  const int32_t rcd = ransac_loop_device(cloud, p, seed, run, &fo);
  cudaStreamSynchronize(ctx->stream);
  if (rcd) {
    delete run;
    return rcd;
  }
  run->seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  *out = run;
  return RSC_OK;
}

int32_t rsc_ransac_run(rsc_cloud* cloud, const rsc_params* p, uint64_t seed, rsc_run** out) {
  if (!cloud || !out) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  *out = nullptr;
  if (!p) return fail(ctx, RSC_E_ARG, "ransac_run: params is null");
  if (p->drawN < 3 || p->drawN > 8) return fail(ctx, RSC_E_ARG, "ransac_run: drawN must be 3..8");
  if (p->minsubsetN < 1 || p->n_shape_types < 1) return fail(ctx, RSC_E_ARG, "ransac_run: nothing to sample/fit");
  if (p->extract_s < 0 || p->extract_s > 2 || p->terminate_s < 0 || p->terminate_s > 2)
    return fail(ctx, RSC_E_ARG, "ransac_run: extract_s/terminate_s must be RSC_S_*");
  if (cloud->subsets.empty() || !cloud->subsets[0].soa)
    return fail(ctx, RSC_E_STATE, "ransac_run: subset 1 is not uploaded (rsc_cloud_set_subset(cloud, 0, ...))");
  if (cloud->exact() && (p->compat_flags & (RSC_SAMPLER_OCTREE | RSC_SCORE_PROGRESSIVE | RSC_REFIT_LSQ | RSC_EXTRACT_BITMAP)))
    return fail(ctx, RSC_E_STATE,
                "ransac_run: RSC_SAMPLER_OCTREE / RSC_SCORE_PROGRESSIVE / RSC_REFIT_LSQ / RSC_EXTRACT_BITMAP do not support exact clouds yet");
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if (int32_t rcr = cloud_ready(cloud)) return rcr;
  cudaStream_t st = ctx->stream;
  const auto t0 = std::chrono::steady_clock::now();
  rsc_run* run = new rsc_run();
  run->ctx = ctx;
  // the reference's behaviour (no extension switch): the loop with the bookkeeping on the device (rsc_loop.cu)
  if (!(p->compat_flags & (RSC_SCORE_PROGRESSIVE | RSC_SAMPLER_OCTREE)) && !getenv("RSC_LOOP_HOSTWALK")) {
    const int32_t rcd = ransac_loop_device(cloud, p, seed, run);
    cudaStreamSynchronize(st);
    if (rcd) {
      delete run;
      return rcd;
    }
    run->seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    *out = run;
    return RSC_OK;
  }
  if (cloud->is_shard()) {
    delete run;
    return fail(ctx, RSC_E_STATE, "ransac_run: the extension switches are not available on sharded storage");
  }
  if (p->compat_flags & RSC_EXTRACT_BITMAP) {
    delete run;
    return fail(ctx, RSC_E_STATE, "ransac_run: RSC_EXTRACT_BITMAP cannot be combined with RSC_SCORE_PROGRESSIVE / RSC_SAMPLER_OCTREE");
  }
  if (!ctx->loop_scratch) ctx->loop_scratch = new LoopScratch();
  LoopScratch& ls = *static_cast<LoopScratch*>(ctx->loop_scratch);
  Store& store = ls.store;
  store.n = 0, store.cur = 0;
  int32_t rc = RSC_OK;
  const Thresh th = make_thresh(p);
  rsc_subset& sub = cloud->subsets[0];
  const int64_t N = cloud->n_global > 0 ? cloud->n_global : cloud->n;
  const int S = p->minsubsetN;
  const int maxnew = S * p->n_shape_types;
  const bool sharded = ctx->allreduce != nullptr;
  // this rank's slice of the subset copy (the whole of it when not sharded)
  int64_t slo = 0, shi = sub.m_pad;
  if (sharded && cloud->range_set && cloud->n_pad > 0) {
    slo = (int64_t)((double)cloud->range_lo / cloud->n_pad * sub.m_pad) / kTile * kTile;
    shi = cloud->range_hi >= cloud->n_pad ? sub.m_pad : (int64_t)((double)cloud->range_hi / cloud->n_pad * sub.m_pad) / kTile * kTile;
  }
  DevBuf &newcnt = ls.newcnt, &hostio = ls.hostio, &olden = ls.olden, &nscratch = ls.nscratch, &nvalid = ls.nvalid, &nmeta = ls.nmeta,
         &lvbuf = ls.lvbuf, &ntiles = ls.ntiles;
  const int k5_cull_mode = getenv("RSC_LOOP_CULL") ? atoi(getenv("RSC_LOOP_CULL")) : 1;
  const bool prog = (p->compat_flags & RSC_SCORE_PROGRESSIVE) != 0;
  const int nsub = (int)cloud->subsets.size();
  ProgMirror mirror;
  std::vector<int32_t> newscore, todo, todo_counts;
  std::vector<uint32_t> keep_h;
  // a rank's slice of a gathered subset copy: the same fraction of it as the rank's range of the cloud
  auto subset_view = [&](rsc_subset& sb) {
    PointSet v = view_subset(&sb);
    if (sharded && cloud->range_set && cloud->n_pad > 0) {
      const int64_t lo = (int64_t)((double)cloud->range_lo / cloud->n_pad * sb.m_pad) / kTile * kTile;
      const int64_t hi = cloud->range_hi >= cloud->n_pad ? sb.m_pad : (int64_t)((double)cloud->range_hi / cloud->n_pad * sb.m_pad) / kTile * kTile;
      v.x += lo, v.y += lo, v.z += lo, v.nx += lo, v.ny += lo, v.nz += lo;
      v.enabled += lo / 32, v.valid += lo / 32;
      v.n_pad = hi - lo;
      v.n = std::max<int64_t>(0, (sb.m < hi ? sb.m : hi) - lo);
    }
    return v;
  };
  // progressive scoring: policy counts of the store candidates `todo` on subset `sj` (0-based) -> todo_counts
  auto score_selected = [&](int sj) -> int32_t {
    const int n = (int)todo.size();
    todo_counts.assign(n, 0);
    const size_t o_c = ((size_t)n * 4 + 255) / 256 * 256, o_k = o_c + ((size_t)n * sizeof(rsc_cand) + 255) / 256 * 256;
    if (ls.prog.ensure(o_k + (size_t)(n + 1) * 4) != cudaSuccess) return fail(ctx, RSC_E_NOMEM, "ransac_run: progressive scratch");
    int32_t* d_idx = ls.prog.as<int32_t>();
    rsc_cand* d_c = (rsc_cand*)(ls.prog.as<char>() + o_c);
    int32_t* d_cnt = (int32_t*)(ls.prog.as<char>() + o_k);
    if (cudaMemcpyAsync(d_idx, todo.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st) != cudaSuccess)
      return fail(ctx, RSC_E_CUDA, "ransac_run: progressive upload");
    gather_cands_kernel<<<(n + 255) / 256, 256, 0, st>>>(store.cands[store.cur].as<rsc_cand>(), d_idx, n, d_c);
    for (int attempt = 0;; ++attempt) {
      int32_t r2 = score_enqueue(ctx, cloud, subset_view(cloud->subsets[sj]), th, d_c, n, d_cnt, false, st);
      if (r2) return r2;
      queue_overflow_kernel<<<1, 1, 0, st>>>(ctx->wl_count.as<uint32_t>(), (uint32_t)ctx->wl_cap, d_cnt + n);
      if (sharded && ctx->allreduce(ctx->allreduce_user, d_cnt, (int64_t)n + 1, (void*)st))
        return fail(ctx, RSC_E_NCCL, "ransac_run: all-reduce callback failed");
      int32_t ovf = 0;
      if (cudaMemcpyAsync(todo_counts.data(), d_cnt, (size_t)n * 4, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
          cudaMemcpyAsync(&ovf, d_cnt + n, 4, cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess)
        return fail(ctx, RSC_E_CUDA, "ransac_run: progressive scoring failed");
      if (ovf == 0) return RSC_OK;
      if (attempt >= 4) return fail(ctx, RSC_E_STATE, "ransac_run: guard-band queue kept overflowing");
      if ((r2 = grow_guard_queue(ctx))) return r2;
    }
  };
  const bool cells_mode = (p->compat_flags & RSC_SAMPLER_OCTREE) != 0;
  const int nlv = cloud->cells.nlevels;
  // cell sampler: the level weights are refreshed every `lw_period` iterations (params.lw_period; 1 = after every
  // iteration, the reference's schedule, iterations.jl:148); a speculative batch never crosses a refresh, so the
  // results for a given period do not depend on the batch size
  const int lw_period = cells_mode ? std::max(1, (int)p->lw_period) : 1;
  const int Bcap = getenv("RSC_BATCH") ? std::max(1, std::min(16, atoi(getenv("RSC_BATCH")))) : 16;
  const int Bmax = cells_mode ? std::min(Bcap, lw_period) : Bcap;
  const int Bmin = getenv("RSC_BATCH_MIN") ? std::max(1, atoi(getenv("RSC_BATCH_MIN"))) : 8;  // batch size after an extraction (swept on c2/c4: 8-16 best)
  int B = 1;  // iterations per speculative batch
  bool terminated = false;
  int64_t n_enabled = rsc_cloud_count_enabled(cloud);
  int64_t counters[3] = {0, 0, 0};  // lengthC, allcand, nofminset (iterations.jl:70)
  const bool trace = getenv("RSC_TRACE") != nullptr;
  double t_fit = 0, t_score = 0, t_extract = 0, t_k5 = 0, t_exa = 0, t_exb = 0;
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto secs = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
    return std::chrono::duration<double>(b - a).count();
  };

  auto cleanup = [&]() {};  // the scratch stays on the context (loop_scratch_free at rsc_ctx_destroy)
#define RUN_CUDA(expr)                                  \
  do {                                                  \
    cudaError_t _e = (expr);                            \
    if (_e != cudaSuccess) {                            \
      rc = fail_cuda(ctx, _e, #expr);                   \
      goto done;                                        \
    }                                                   \
  } while (0)

  RUN_CUDA(newcnt.ensure((size_t)2 * maxnew * 4 + 64));
  RUN_CUDA(hostio.ensure(64));
  run->device = ctx->device;
  RUN_CUDA(cudaMalloc(&run->d_idx, (size_t)(n_enabled > 0 ? n_enabled : 1) * sizeof(int64_t)));  // every point is extracted at most once

  // level-weighted cell sampler (extension, SURVEY 8(f)-1): un-swapped initial values (octree.jl:82-83)
  if (cells_mode) {
    if (nlv == 0) {
      rc = fail(ctx, RSC_E_STATE, "ransac_run: RSC_SAMPLER_OCTREE needs rsc_cloud_build_cells first");
      goto done;
    }
    run->nlevels = nlv;
    for (int l = 0; l < nlv; ++l) run->levelweight[l] = 1.0 / nlv, run->levelscore[l] = 0.0;
    RUN_CUDA(lvbuf.ensure((size_t)16 * 22 * 8));
  }

  if (prog)
    for (int j = 0; j < nsub; ++j)
      if (!cloud->subsets[j].soa) {
        rc = fail(ctx, RSC_E_STATE, "ransac_run: RSC_SCORE_PROGRESSIVE needs every subset uploaded (rsc_cloud_set_subset)");
        goto done;
      }

  // Iterations are run in speculative batches of nb: as long as nothing is extracted the enabled mask
  // does not change, so iterations k..k+nb-1 can sample, fit and score together (one K2 launch over
  // all their candidates, one or two host syncs per batch instead of per iteration).  The host then
  // walks the batch iteration by iteration with exactly the reference's bookkeeping and cuts it at
  // the first extraction or at termination; the later iterations of a cut batch are discarded and
  // redone (their sets sampled a stale mask).  The cell sampler updates its level weights every
  // iteration (iterations.jl:148), so it runs with nb = 1.
  RUN_CUDA(newcnt.ensure((size_t)2 * maxnew * Bmax * 4 + 64));
  RUN_CUDA(hostio.ensure(64 + (size_t)(Bmax + 2) * 8 + (size_t)(Bmax + 2) * 4));
  if ((rc = fit_reserve(ctx, p, S * Bmax))) goto done;
  RUN_CUDA(store.reserve((size_t)maxnew * Bmax, st));  // room for the first batches without re-allocations
  for (int k = 1; k <= p->itermax && !terminated;) {
    if (n_enabled < p->tau) break;  // iterations.jl:75
    int nb = std::min(B, p->itermax - k + 1);
    if (cells_mode) nb = std::min(nb, lw_period - (k - 1) % lw_period);  // up to the next refresh of the level weights
    const auto tk0 = now();
    // ---- K1: nb * minsubsetN minimal sets -> candidates (device, compacted in reference order) ----
    FitScratch fs;
    double cum[11];
    if (cells_mode) rsc_level_cumsum(run->levelweight, nlv, cum);
    if ((rc = fit_enqueue(ctx, cloud, cells_mode ? 3 : 2, p, p->drawN, nullptr, nullptr, nullptr, S * nb, seed, (uint64_t)(k - 1) * S,
                          st, &fs, cells_mode ? cum : nullptr)))
      goto done;
    long long* d_keys = hostio.as<long long>() + 8;         // [nb] segment arg-max keys
    int32_t* d_seg = (int32_t*)(d_keys + Bmax + 2);           // [nb + 1] segment bounds
    int32_t seg_h[18] = {0};
    seg_bounds_kernel<<<1, 32, 0, st>>>(fs.out_set, fs.total, S, nb, d_seg);
    RUN_CUDA(cudaGetLastError());
    RUN_CUDA(cudaMemcpyAsync(seg_h, d_seg, (size_t)(nb + 1) * 4, cudaMemcpyDeviceToHost, st));
    RUN_CUDA(cudaStreamSynchronize(st));
    const int n_new = seg_h[nb];
    const auto tk1 = now();
    t_fit += secs(tk0, tk1);
    // ---- K2 on subset 1 + K3 ----  (repeated with a larger guard-band queue if that overflowed:
    // dropped queue entries would leave FP32 decisions in the counts)
    const int store_n0 = store.n;
    int64_t best[2] = {-1, 0};
    long long seg_keys[18];
    for (int j = 0; j < 18; ++j) seg_keys[j] = -1;
    long long lv_host[16 * 22] = {0};
    for (int attempt = 0;; ++attempt) {
      store.n = store_n0;
      int32_t ovf = 0;
      if (n_new > 0) {
        RUN_CUDA(store.reserve((size_t)store.n + n_new, st));
        rsc_cand* dst = store.cands[store.cur].as<rsc_cand>() + store.n;
        RUN_CUDA(cudaMemcpyAsync(dst, fs.out, (size_t)n_new * sizeof(rsc_cand), cudaMemcpyDeviceToDevice, st));
        int32_t* cv = newcnt.as<int32_t>();
        int32_t* ce = cv + n_new;
        PointSet ps = view_subset(&sub);
        if (sharded) {
          ps.x += slo, ps.y += slo, ps.z += slo, ps.nx += slo, ps.ny += slo, ps.nz += slo;
          ps.enabled += slo / 32, ps.valid += slo / 32;
          ps.n_pad = shi - slo;
          ps.n = std::max<int64_t>(0, (sub.m < shi ? sub.m : shi) - slo);
        }
        // (the culled scorer on the subset's Morton view when the batch is large: same counts)
        // overflow flag rides behind the counts, so that a sharded run decides to repeat collectively
        if ((rc = loop_score_new(ctx, cloud, sub, ps, !sharded, th, dst, n_new, cv, ce, cv + 2 * n_new, st))) goto done;
        if (sharded && (rc = ctx->allreduce(ctx->allreduce_user, cv, (int64_t)2 * n_new + 1, (void*)st))) {
          rc = fail(ctx, RSC_E_NCCL, "ransac_run: all-reduce callback failed");
          goto done;
        }
        finish_new_kernel<<<(n_new + 255) / 256, 256, 0, st>>>(dst, n_new, cv, ce, th.honour_enabled,
                                                               store.score[store.cur].as<int32_t>() + store.n,
                                                               store.flags[store.cur].as<uint8_t>() + store.n);
        RUN_CUDA(cudaGetLastError());
        RUN_CUDA(cudaMemcpyAsync(&ovf, cv + 2 * n_new, 4, cudaMemcpyDeviceToHost, st));
        if (cells_mode) {
          RUN_CUDA(cudaMemsetAsync(lvbuf.p, 0, (size_t)nb * 22 * 8, st));
          level_stats_kernel<<<(n_new + 255) / 256, 256, 0, st>>>(fs.out_set, fs.level, store.score[store.cur].as<int32_t>() + store.n,
                                                                  n_new, S, lvbuf.as<long long>());
          RUN_CUDA(cudaGetLastError());
          RUN_CUDA(cudaMemcpyAsync(lv_host, lvbuf.p, (size_t)nb * 22 * 8, cudaMemcpyDeviceToHost, st));
        }
        store.n += n_new;
      }
      if (store_n0 >= 1) {  // best of the candidates stored before this batch
        RUN_CUDA(argmax_enqueue(store.score[store.cur].as<int32_t>(), store.flags[store.cur].as<uint8_t>(), store_n0,
                                          hostio.as<int64_t>(), ctx->sm_count, st));
        RUN_CUDA(cudaMemcpyAsync(best, hostio.p, 16, cudaMemcpyDeviceToHost, st));
      }
      if (n_new > 0) {  // and of every iteration's new candidates
        seg_argmax_kernel<<<nb, 256, 0, st>>>(store.score[store.cur].as<int32_t>(), store.flags[store.cur].as<uint8_t>(), d_seg,
                                               store_n0, d_keys);
        RUN_CUDA(cudaGetLastError());
        RUN_CUDA(cudaMemcpyAsync(seg_keys, d_keys, (size_t)nb * 8, cudaMemcpyDeviceToHost, st));
      }
      if (prog && n_new > 0) {
        newscore.resize(n_new);
        RUN_CUDA(cudaMemcpyAsync(newscore.data(), store.score[store.cur].as<int32_t>() + store_n0, (size_t)n_new * 4,
                                 cudaMemcpyDeviceToHost, st));
      }
      RUN_CUDA(cudaStreamSynchronize(st));
      if (ovf == 0) break;
      if (attempt >= 4) {
        rc = fail(ctx, RSC_E_STATE, "ransac_run: guard-band queue kept overflowing");
        goto done;
      }
      if ((rc = grow_guard_queue(ctx))) goto done;
    }
    const auto tk2 = now();
    t_score += secs(tk1, tk2);
    // ---- walk the iterations of the batch with the reference's bookkeeping ----
    long long bestkey = (store_n0 >= 1 && best[0] >= 0) ? (((long long)best[1] << 32) | (long long)(0x7fffffff - best[0])) : -1;
    bool extracted_now = false;
    int used = 0;
    for (int j = 0; j < nb && !extracted_now && !terminated; ++j) {
    const int kk = k + j;
    run->iterations = kk;
    used = j + 1;
    counters[1] += seg_h[j + 1] - seg_h[j];
    store.n = store_n0 + seg_h[j + 1];
    counters[2] = (int64_t)kk * S;
    counters[0] = store.n;
    if (cells_mode && n_new > 0) {  // levelscore[level] += sum of E = -n + (N+2)/(M+2) (sum sigma + n)
      const long long* lvj = lv_host + (size_t)j * 22;
      for (int l = 0; l < nlv; ++l)
        if (lvj[l])
          run->levelscore[l] += (-(double)lvj[l]) + ((double)(N + 2) / (double)(sub.m + 2)) * (double)(lvj[11 + l] + lvj[l]);
    }
    if (seg_keys[j] > bestkey) bestkey = seg_keys[j];  // first maximum wins: the key carries the store index
    best[0] = bestkey >= 0 ? (int64_t)(0x7fffffff - (bestkey & 0xffffffffll)) : -1;
    best[1] = bestkey >= 0 ? (int64_t)(bestkey >> 32) : 0;
    if (prog) {
      // refine while the best interval overlaps another one: the least-evaluated candidates among the best
      // and its overlappers are scored on their next subset (one K2 launch per round), re-estimated
      // from the union; stops when the best stands alone or those candidates have seen every subset
      for (int i = seg_h[j]; i < seg_h[j + 1]; ++i) mirror.push(newscore[i], sub.m, N);
      while (mirror.size() > 1) {
        const int b = mirror.best();
        int lmin = 1 << 30;
        bool any = false;
        for (size_t i = 0; i < mirror.size(); ++i)
          if ((int)i == b || mirror.overlap(i, b)) {
            any = any || (int)i != b;
            lmin = mirror.lvl[i] < lmin ? mirror.lvl[i] : lmin;
          }
        if (!any || lmin >= nsub) break;
        todo.clear();
        for (size_t i = 0; i < mirror.size(); ++i)
          if (((int)i == b || mirror.overlap(i, b)) && mirror.lvl[i] == lmin) todo.push_back((int32_t)i);
        if ((rc = score_selected(lmin))) goto done;
        for (size_t t = 0; t < todo.size(); ++t) mirror.add(todo[t], todo_counts[t], cloud->subsets[lmin].m, N);
        run->refined += (int64_t)todo.size();
      }
      best[0] = mirror.best();
    }
    if (store.n >= 1) {
      if (best[0] >= 0) {
        double E;
        if (prog)
          E = mirror.E[best[0]];
        else
          rsc_estimate_score(sub.m, N, best[1], nullptr, nullptr, &E);
        const double s_ex = (double)counters[p->extract_s];
        if (prob_(E, s_ex, (double)N, (double)p->drawN) > p->prob_det) {
          // ---- K4: refit over the whole cloud, invalidate its points ----
          const auto tkx = now();
          rsc_cand shape;
          RUN_CUDA(cudaMemcpyAsync(&shape, store.cands[store.cur].as<rsc_cand>() + best[0], sizeof(shape),
                                   cudaMemcpyDeviceToHost, st));
          RUN_CUDA(cudaStreamSynchronize(st));
          const auto tka = now();
          t_exa += secs(tkx, tka);
          if (p->compat_flags & RSC_REFIT_LSQ) {  // extension: the paper's least-squares refit within 3 eps
            if ((rc = lsq_refine(cloud, p, 3.0, &shape, nullptr, nullptr, st))) goto done;
          }
          Thresh thr = th;
          thr.honour_enabled = 0xFu;
          if ((rc = refit_mask_enqueue(cloud, thr, shape, st))) goto done;
          unsigned long long total = 0;
          RUN_CUDA(cudaMemcpyAsync(&total, ctx->misc2.p, 8, cudaMemcpyDeviceToHost, st));
          RUN_CUDA(cudaStreamSynchronize(st));
          t_exb += secs(tka, now());
          // keep the subset's enabled words of before the extraction.  When the subset has a Morton view (the culled
          // scorer ran on it) K5 works on the view: the newly disabled points then come out spatially sorted and the
          // store can be re-scored against them by the culled scorer too (the SET of points is the same)
          const int64_t swords = sub.m_pad / 32;
          const bool k5_view = sub.cen != nullptr && !sharded;
          const uint32_t* sub_en = k5_view ? sub.cen : sub.enabled;
          const float* sub_soa = k5_view ? sub.csoa : sub.soa;
          RUN_CUDA(olden.ensure((size_t)swords * 4));
          RUN_CUDA(cudaMemcpyAsync(olden.p, sub_en, (size_t)swords * 4, cudaMemcpyDeviceToDevice, st));
          int64_t* d_out = run->d_idx + run->off.back();
          if ((rc = refit_write_enqueue(cloud, total ? d_out : nullptr, true, st))) goto done;
          run->shapes.push_back(shape);
          run->off.push_back(run->off.back() + (int64_t)total);
          run->total.push_back((int64_t)total);
          n_enabled -= (int64_t)total;
          const auto tk3 = now();
          t_extract += secs(tkx, tk3);
          // ---- K5: drop the best and every candidate compatible with a newly disabled subset point ----
          const int nst = store.n;
          // scratch layout: [wcnt: swords u32][woff: swords u64][wtot u64][keep: nst u32][koff: nst u64][ktot u64]
          const size_t o_woff = ((size_t)swords * 4 + 255) / 256 * 256;
          const size_t o_keep = o_woff + (size_t)(swords + 1) * 8;
          const size_t o_koff = (o_keep + (size_t)nst * 4 + 255) / 256 * 256;
          RUN_CUDA(nmeta.ensure(o_koff + (size_t)(nst + 1) * 8));
          uint32_t* wcnt = nmeta.as<uint32_t>();
          unsigned long long* woff = (unsigned long long*)(nmeta.as<char>() + o_woff);
          unsigned long long* wtot = woff + swords;
          uint32_t* keep = (uint32_t*)(nmeta.as<char>() + o_keep);
          unsigned long long* koff = (unsigned long long*)(nmeta.as<char>() + o_koff);
          newly_count_kernel<<<(unsigned)((swords + 255) / 256), 256, 0, st>>>(olden.as<uint32_t>(), sub_en, swords, wcnt);
          RUN_CUDA(cudaGetLastError());
          if ((rc = scan_u32(ctx, wcnt, (int)swords, woff, wtot, st))) goto done;
          unsigned long long nnew_dis = 0;
          RUN_CUDA(cudaMemcpyAsync(&nnew_dis, wtot, 8, cudaMemcpyDeviceToHost, st));
          RUN_CUDA(cudaStreamSynchronize(st));
          int32_t* hit = nullptr;
          RUN_CUDA(ctx->counts.ensure((size_t)3 * nst * 4));
          hit = ctx->counts.as<int32_t>() + 2 * (size_t)nst;
          unsigned long long kept = 0;
          bool k5_culled = false;
          int nxt = store.cur ^ 1;
          for (int attempt = 0;; ++attempt) {  // repeated if the guard-band queue overflowed
          if (nnew_dis > 0) {
            const int64_t sp = ((int64_t)nnew_dis + kTile - 1) / kTile * kTile;
            RUN_CUDA(nscratch.ensure((size_t)6 * sp * 4));
            RUN_CUDA(nvalid.ensure((size_t)(sp / 32) * 4));
            RUN_CUDA(cudaMemsetAsync(nscratch.p, 0, (size_t)6 * sp * 4, st));
            if (cloud->exact()) RUN_CUDA(ls.nidx.ensure((size_t)sp * sizeof(int64_t)));
            newly_gather_kernel<<<(unsigned)((swords + 255) / 256), 256, 0, st>>>(olden.as<uint32_t>(), sub_en, swords, woff, sub_soa,
                                                                                   sub.m_pad, nscratch.as<float>(), sp, sub.idx,
                                                                                   cloud->exact() ? ls.nidx.as<int64_t>() : nullptr);
            RUN_CUDA(cudaGetLastError());
            fill_valid_words_kernel<<<(unsigned)((sp / 32 + 255) / 256), 256, 0, st>>>(nvalid.as<uint32_t>(), (int64_t)nnew_dis, sp / 32);
            RUN_CUDA(cudaGetLastError());
            PointSet ps;
            float* b = nscratch.as<float>();
            ps.x = b, ps.y = b + sp, ps.z = b + 2 * sp, ps.nx = b + 3 * sp, ps.ny = b + 4 * sp, ps.nz = b + 5 * sp;
            ps.enabled = nvalid.as<uint32_t>();
            ps.valid = nvalid.as<uint32_t>();
            ps.n = (int64_t)nnew_dis;
            ps.n_pad = sp;
            if (cloud->exact()) ps.xyz64 = cloud->xyz64, ps.nrm64 = cloud->nrm64, ps.map = ls.nidx.as<int64_t>();
            // replicated on every rank (the scratch set is tiny): no all-reduce needed
            // enabled == valid on the scratch set: the enabled-gated count (kept for every type) is the hit count
            // a large store (cell sampler): most stored candidates are nowhere near the extracted shape -- and the dense
            // path's candidate compiler is ONE CTA (3 ms for a store of a million candidates)
            k5_culled = k5_view && k5_cull_mode != 0 && (k5_cull_mode == 2 || nst >= 4096 || (double)nst * (double)nnew_dis >= 2e8);
            if (k5_culled) {
              RUN_CUDA(ntiles.ensure(cull_sphere_count(sp) * sizeof(float4)));
              if ((rc = cull_tile_spheres(ctx, ps, ntiles.as<float4>(), st))) goto done;
              if ((rc = cull_enqueue(ctx, cloud, ps, ntiles.as<float4>(), th, store.cands[store.cur].as<rsc_cand>(), nst, nullptr,
                                     ctx->counts.as<int32_t>(), hit, nullptr, st)))
                goto done;
            } else if ((rc = score_enqueue(ctx, cloud, ps, th, store.cands[store.cur].as<rsc_cand>(), nst, nullptr, false, st,
                                           ctx->counts.as<int32_t>(), hit))) {
              goto done;
            }
          } else {
            RUN_CUDA(cudaMemsetAsync(hit, 0, (size_t)nst * 4, st));
          }
          unsigned long long* ktot = koff + nst;
          invalidate_kernel<<<(nst + 255) / 256, 256, 0, st>>>(hit, store.flags[store.cur].as<uint8_t>(), nst, (int)best[0], keep);
          RUN_CUDA(cudaGetLastError());
          if ((rc = scan_u32(ctx, keep, nst, koff, ktot, st))) goto done;
          nxt = store.cur ^ 1;
          compact_store_kernel<<<(nst + 255) / 256, 256, 0, st>>>(
              store.cands[store.cur].as<rsc_cand>(), store.score[store.cur].as<int32_t>(), store.flags[store.cur].as<uint8_t>(),
              keep, koff, nst, store.cands[nxt].as<rsc_cand>(), store.score[nxt].as<int32_t>(), store.flags[nxt].as<uint8_t>());
          RUN_CUDA(cudaGetLastError());
          uint32_t wln[2] = {0, 0};
          if (nnew_dis > 0 && !k5_culled) RUN_CUDA(cudaMemcpyAsync(wln, ctx->wl_count.p, 8, cudaMemcpyDeviceToHost, st));
          RUN_CUDA(cudaMemcpyAsync(&kept, ktot, 8, cudaMemcpyDeviceToHost, st));
          RUN_CUDA(cudaStreamSynchronize(st));
          if (wln[0] <= ctx->wl_cap && wln[1] <= ctx->wl_cap) break;
          if (attempt >= 4) {
            rc = fail(ctx, RSC_E_STATE, "ransac_run: guard-band queue kept overflowing");
            goto done;
          }
          if ((rc = grow_guard_queue(ctx))) goto done;
          }
          if (prog) {
            keep_h.resize(nst);
            RUN_CUDA(cudaMemcpyAsync(keep_h.data(), keep, (size_t)nst * 4, cudaMemcpyDeviceToHost, st));
            RUN_CUDA(cudaStreamSynchronize(st));
            mirror.compact(keep_h);
            mirror.reset_refined(sub.m, N);
          }
          store.cur = nxt;
          store.n = (int)kept;
          t_k5 += secs(tk3, now());
          extracted_now = true;  // the rest of the batch sampled the mask of before this extraction
        }
      }
    }
    if (cells_mode && kk % lw_period == 0) rsc_update_levelweight(run->levelweight, run->levelscore, nlv);  // iterations.jl:148
    // iterations.jl:151-156
    if (prob_((double)p->tau, (double)counters[p->terminate_s], (double)N, (double)p->drawN) > p->prob_det) terminated = true;
    }  // iterations of the batch
    k += used;
    B = extracted_now ? std::min(Bmin, Bmax) : std::min(2 * B, Bmax);
    if (B > Bmax) B = Bmax;
  }
done:
  cudaStreamSynchronize(st);
  if (trace)
    fprintf(stderr, "[rsc_ransac_run] iterations %d shapes %zu | sample+fit %.1f ms, score+argmax %.1f ms, refit+extract %.1f ms (shape fetch %.1f, mask+count %.1f), invalidate+compact %.1f ms\n",
            run->iterations, run->shapes.size(), 1e3 * t_fit, 1e3 * t_score, 1e3 * t_extract, 1e3 * t_exa, 1e3 * t_exb, 1e3 * t_k5);
  cleanup();
  if (rc) {
    delete run;
    return rc;
  }
  run->seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  *out = run;
  return RSC_OK;
#undef RUN_CUDA
}

int32_t rsc_run_nshapes(const rsc_run* r) { return r ? (int32_t)r->shapes.size() : 0; }
int32_t rsc_run_iterations(const rsc_run* r) { return r ? r->iterations : 0; }
int64_t rsc_run_refined(const rsc_run* r) { return r ? r->refined : 0; }
double rsc_run_seconds(const rsc_run* r) { return r ? r->seconds : 0.0; }

int32_t rsc_run_levelweight(const rsc_run* r, double* levelweight, double* levelscore) {
  if (!r) return 0;
  for (int l = 0; l < r->nlevels; ++l) {
    if (levelweight) levelweight[l] = r->levelweight[l];
    if (levelscore) levelscore[l] = r->levelscore[l];
  }
  return r->nlevels;
}

int32_t rsc_run_shape(const rsc_run* r, int32_t i, rsc_cand* shape, int64_t* n_inpoints) {
  if (!r || i < 0 || (size_t)i >= r->shapes.size()) return RSC_E_ARG;
  if (shape) *shape = r->shapes[i];
  if (n_inpoints) *n_inpoints = r->off[i + 1] - r->off[i];
  return RSC_OK;
}

int64_t rsc_run_shape_total(const rsc_run* r, int32_t i) {
  if (!r || i < 0 || (size_t)i >= r->total.size()) return -1;
  return r->total[i];
}

int32_t rsc_run_syncs(const rsc_run* r, int32_t* batches) {
  if (!r) return 0;
  if (batches) *batches = r->batches;
  return r->syncs;
}

int32_t rsc_run_inpoints(const rsc_run* r, int32_t i, int64_t* out_idx) {
  if (!r || i < 0 || (size_t)i >= r->shapes.size() || !out_idx) return RSC_E_ARG;
  const int64_t n = r->off[i + 1] - r->off[i];
  if (n == 0) return RSC_OK;
  if (cudaSetDevice(r->device) != cudaSuccess) return RSC_E_CUDA;
  if (r->ctx) return staged_d2h(r->ctx, out_idx, r->d_idx + r->off[i], (size_t)n * sizeof(int64_t), r->ctx->stream);
  return cudaMemcpy(out_idx, r->d_idx + r->off[i], (size_t)n * sizeof(int64_t), cudaMemcpyDeviceToHost) == cudaSuccess ? RSC_OK
                                                                                                                        : RSC_E_CUDA;
}

void rsc_run_destroy(rsc_run* r) { delete r; }

}  // extern "C"
