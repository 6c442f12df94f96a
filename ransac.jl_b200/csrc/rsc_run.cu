// rsc_run.cu -- the C-ABI entry points of the RANSAC loop (ransac(pc, params; ...): iterations.jl:35-162):
// rsc_ransac_run and rsc_ransac_run_user check their arguments and run the loop of rsc_loop.cu; the accessors
// of a run's results; and the host decision of the extension switches.
//
// The host decision (RSC_SCORE_PROGRESSIVE, RSC_SAMPLER_OCTREE, or RSC_LOOP_HOSTWALK set) replaces decide_kernel:
// after a batch's K2 + K3 the host reads the segment bounds, the segment keys and the old store's arg-max (plus
// the new candidates' scores for progressive scoring and the level statistics for the cell sampler) with one
// synchronisation and walks the batch's iterations with the reference's bookkeeping.  What the device does not:
//   progressive scoring (SURVEY 8(f)-2; iterations.jl:110 "TODO: refine if best.overlap") refines overlapping score
//     intervals on the subsets 2..r before each extraction test (ProgMirror);
//   the cell sampler accumulates the level scores and refreshes the level weights (octree.jl:198-205,
//     iterations.jl:148).  Its tests stay on the host's pow(): the device's can differ in the last ulp at the
//     prob_det threshold.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <string>
#include <vector>

#include "rsc_loop.cuh"

namespace rsc {

__global__ void gather_cands_kernel(const rsc_cand* __restrict__ store, const int32_t* __restrict__ idx, int n,
                                    rsc_cand* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = store[idx[i]];
}

// progressive scoring: host mirror of the store's scores while refining: candidate i has been scored on subsets 1..lvl[i],
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

static double prob_(double n, double s, double N, double k) { return 1 - pow(1 - pow(n / N, k), s); }  // utilities.jl:262

struct HostWalk {  // what the host decision keeps over a run
  rsc_cloud* cloud;
  const rsc_params* p;
  rsc_run* run;
  Thresh th;
  bool prog, cells, ranged;  // ranged: counts are summed over the ranks of a replicated cloud
  int64_t N;
  long long counters[3] = {0, 0, 0};  // lengthC, allcand, nofminset (iterations.jl:70)
  ProgMirror mirror;
  std::vector<int32_t> todo, todo_counts;
};

// progressive scoring: policy counts of the store candidates `todo` on subset `sj` (0-based) -> todo_counts
static int32_t score_selected(HostWalk& w, int sj) {
  rsc_ctx* ctx = w.cloud->ctx;
  cudaStream_t st = ctx->stream;
  LoopScratch& ls = *static_cast<LoopScratch*>(ctx->loop_scratch);
  const int n = (int)w.todo.size();
  w.todo_counts.assign(n, 0);
  const size_t o_c = ((size_t)n * 4 + 255) / 256 * 256, o_k = o_c + ((size_t)n * sizeof(rsc_cand) + 255) / 256 * 256;
  if (ls.prog.ensure(o_k + (size_t)(n + 1) * 4) != cudaSuccess) return fail(ctx, RSC_E_NOMEM, "ransac_run: progressive scratch");
  int32_t* d_idx = ls.prog.as<int32_t>();
  rsc_cand* d_c = (rsc_cand*)(ls.prog.as<char>() + o_c);
  int32_t* d_cnt = (int32_t*)(ls.prog.as<char>() + o_k);
  if (cudaMemcpyAsync(d_idx, w.todo.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st) != cudaSuccess)
    return fail(ctx, RSC_E_CUDA, "ransac_run: progressive upload");
  gather_cands_kernel<<<(n + 255) / 256, 256, 0, st>>>(ls.store.cands[ls.store.cur].as<rsc_cand>(), d_idx, n, d_c);
  for (int attempt = 0;; ++attempt) {
    int32_t r2 = score_enqueue(ctx, w.cloud, subset_slice(w.cloud, w.cloud->subsets[sj], w.ranged), w.th, d_c, n, d_cnt, false, st);
    if (r2) return r2;
    queue_overflow_kernel<<<1, 1, 0, st>>>(ctx->wl_count.as<uint32_t>(), (uint32_t)ctx->wl_cap, d_cnt + n);
    if (w.ranged && ctx->allreduce(ctx->allreduce_user, d_cnt, (int64_t)n + 1, (void*)st))
      return fail(ctx, RSC_E_NCCL, "ransac_run: all-reduce callback failed");
    int32_t ovf = 0;
    if (cudaMemcpyAsync(w.todo_counts.data(), d_cnt, (size_t)n * 4, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaMemcpyAsync(&ovf, d_cnt + n, 4, cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess)
      return fail(ctx, RSC_E_CUDA, "ransac_run: progressive scoring failed");
    ++w.run->syncs;
    if (ovf == 0) return RSC_OK;
    if (attempt >= 4) return fail(ctx, RSC_E_STATE, "ransac_run: guard-band queue kept overflowing");
    if ((r2 = grow_guard_queue(ctx))) return r2;
  }
}

int32_t host_decide(HostWalk& w, const LoopDev& d, const int32_t* newscore, int store_n0, int nb, int k0, BatchRec* rec) {
  rsc_ctx* ctx = w.cloud->ctx;
  const rsc_params* p = w.p;
  rsc_run* run = w.run;
  const rsc_subset& sub = w.cloud->subsets[0];
  const int S = p->minsubsetN;
  const int nlv = run->nlevels, nsub = (int)w.cloud->subsets.size();
  long long* counters = w.counters;
  BatchRec r{};
  r.iterations = k0 - 1, r.best_idx = -1, r.store_n = store_n0;
  long long bestkey = (store_n0 >= 1 && d.oldbest[0] >= 0) ? ((d.oldbest[1] << 32) | (long long)(0x7fffffff - d.oldbest[0])) : -1;
  int64_t best = -1;
  for (int j = 0; j < nb && !r.extract && !r.terminated; ++j) {
    const int kk = k0 + j;
    r.used = j + 1;
    r.iterations = kk;
    counters[1] += d.seg[j + 1] - d.seg[j];
    r.store_n = store_n0 + d.seg[j + 1];
    counters[2] = (int64_t)kk * S;
    counters[0] = r.store_n;
    if (w.cells) {  // levelscore[level] += sum of E = -n + (N+2)/(M+2) (sum sigma + n)
      const long long* lvj = d.lv[j];
      for (int l = 0; l < nlv; ++l)
        if (lvj[l]) run->levelscore[l] += (-(double)lvj[l]) + ((double)(w.N + 2) / (double)(sub.m + 2)) * (double)(lvj[11 + l] + lvj[l]);
    }
    if (d.seg_keys[j] > bestkey) bestkey = d.seg_keys[j];  // first maximum wins: the key carries the store index
    best = bestkey >= 0 ? (int64_t)(0x7fffffff - (bestkey & 0xffffffffll)) : -1;
    if (w.prog) {
      // refine while the best interval overlaps another one: the least-evaluated candidates among the best
      // and its overlappers are scored on their next subset (one K2 launch per round), re-estimated
      // from the union; stops when the best stands alone or those candidates have seen every subset
      ProgMirror& mirror = w.mirror;
      for (int i = d.seg[j]; i < d.seg[j + 1]; ++i) mirror.push(newscore[i], sub.m, w.N);
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
        w.todo.clear();
        for (size_t i = 0; i < mirror.size(); ++i)
          if (((int)i == b || mirror.overlap(i, b)) && mirror.lvl[i] == lmin) w.todo.push_back((int32_t)i);
        if (int32_t rc = score_selected(w, lmin)) return rc;
        for (size_t t = 0; t < w.todo.size(); ++t) mirror.add(w.todo[t], w.todo_counts[t], w.cloud->subsets[lmin].m, w.N);
        run->refined += (int64_t)w.todo.size();
      }
      best = mirror.best();
    }
    if (r.store_n >= 1 && best >= 0) {
      double E;
      if (w.prog)
        E = w.mirror.E[best];
      else
        rsc_estimate_score(sub.m, w.N, bestkey >> 32, nullptr, nullptr, &E);
      r.extract = prob_(E, (double)counters[p->extract_s], (double)w.N, (double)p->drawN) > p->prob_det;
    }
    if (w.cells && kk % std::max(1, (int)p->lw_period) == 0) rsc_update_levelweight(run->levelweight, run->levelscore, nlv);  // iterations.jl:148
    // iterations.jl:151-156
    r.terminated = prob_((double)p->tau, (double)counters[p->terminate_s], (double)w.N, (double)p->drawN) > p->prob_det;
  }
  for (int i = 0; i < 3; ++i) r.counters[i] = counters[i];
  if (r.extract) {  // the chosen candidate and its subset-1 score (the bound of K5's gather) from the store
    const Store& store = static_cast<LoopScratch*>(ctx->loop_scratch)->store;
    r.best_idx = (int32_t)best;
    RSC_CUDA(ctx, cudaMemcpyAsync(&r.best, store.cands[store.cur].as<rsc_cand>() + best, sizeof(rsc_cand), cudaMemcpyDeviceToHost, ctx->stream));
    RSC_CUDA(ctx, cudaMemcpyAsync(&r.best_score, store.score[store.cur].as<int32_t>() + best, 4, cudaMemcpyDeviceToHost, ctx->stream));
    RSC_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ++run->syncs;
  }
  *rec = r;
  return RSC_OK;
}

void host_compacted(HostWalk& w, const std::vector<uint32_t>& keep) {
  w.mirror.compact(keep);
  w.mirror.reset_refined(w.cloud->subsets[0].m, w.N);
}

void loop_scratch_free(rsc_ctx* ctx) {
  LoopScratch* ls = static_cast<LoopScratch*>(ctx->loop_scratch);
  if (!ls) return;
  ls->store.release();
  ls->newcnt.release(), ls->hostio.release(), ls->olden.release(), ls->nscratch.release(), ls->nidx.release(), ls->nvalid.release();
  ls->nmeta.release(), ls->prog.release(), ls->ntiles.release();
  delete ls;
  ctx->loop_scratch = nullptr;
}

// the checks on the parameters both entry points share (`who`: the entry point, for the messages)
static int32_t check_params(rsc_ctx* ctx, const rsc_params* p, const char* who) {
  auto bad = [&](const char* what) { return fail(ctx, RSC_E_ARG, (std::string(who) + ": " + what).c_str()); };
  if (!p) return bad("params is null");
  if (p->drawN < 3 || p->drawN > 8) return bad("drawN must be 3..8");
  if (p->minsubsetN < 1) return bad("nothing to sample/fit");
  if (p->extract_s < 0 || p->extract_s > 2 || p->terminate_s < 0 || p->terminate_s > 2) return bad("extract_s/terminate_s must be RSC_S_*");
  return RSC_OK;
}

// the state both entry points need, then the loop; *out = the run, timed
static int32_t run_loop(rsc_cloud* cloud, const rsc_params* p, uint64_t seed, const FitOrder* order, bool host_decides, const char* who,
                        rsc_run** out) {
  rsc_ctx* ctx = cloud->ctx;
  if (cloud->subsets.empty() || !cloud->subsets[0].soa)
    return fail(ctx, RSC_E_STATE, (std::string(who) + ": subset 1 is not uploaded (rsc_cloud_set_subset(cloud, 0, ...))").c_str());
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if (int32_t rcr = cloud_ready(cloud)) return rcr;
  const auto t0 = std::chrono::steady_clock::now();
  rsc_run* run = new rsc_run();
  run->ctx = ctx;
  HostWalk w{cloud, p, run, make_thresh(p)};
  w.prog = (p->compat_flags & RSC_SCORE_PROGRESSIVE) != 0;
  w.cells = (p->compat_flags & RSC_SAMPLER_OCTREE) != 0;
  w.ranged = ctx->allreduce != nullptr && cloud->range_set;
  w.N = cloud->n_global > 0 ? cloud->n_global : cloud->n;
  if (w.cells) {  // level-weighted cell sampler (extension, SURVEY 8(f)-1): un-swapped initial values (octree.jl:82-83)
    run->nlevels = cloud->cells.nlevels;
    for (int l = 0; l < run->nlevels; ++l) run->levelweight[l] = 1.0 / run->nlevels, run->levelscore[l] = 0.0;
  }
  const int32_t rc = ransac_loop_device(cloud, p, seed, run, order, host_decides ? &w : nullptr);
  cudaStreamSynchronize(ctx->stream);
  if (rc) {
    delete run;
    return rc;
  }
  run->seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  *out = run;
  return RSC_OK;
}

}  // namespace rsc

using namespace rsc;

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
  FitOrder fo;
  if (int32_t rc = check_params(ctx, p, "ransac_run_user")) return rc;
  if (int32_t rc = make_fit_order(ctx, static_cast<const rsc_shape_slot*>(order), norder, &fo, "ransac_run_user")) return rc;
  if (norder < 1) return fail(ctx, RSC_E_ARG, "ransac_run_user: an empty fit order");
  if (cloud->is_shard() || cloud->range_set) return fail(ctx, RSC_E_STATE, "ransac_run_user: sharded or ranged clouds are not supported");
  if (p->compat_flags & (RSC_SAMPLER_OCTREE | RSC_SCORE_PROGRESSIVE | RSC_REFIT_LSQ | RSC_EXTRACT_BITMAP))
    return fail(ctx, RSC_E_STATE, "ransac_run_user: the extension switches are not available with a fit order");
  if (getenv("RSC_LOOP_HOSTWALK")) return fail(ctx, RSC_E_STATE, "ransac_run_user: runs the device loop only (RSC_LOOP_HOSTWALK is set)");
  return run_loop(cloud, p, seed, &fo, false, "ransac_run_user", out);
}

int32_t rsc_ransac_run(rsc_cloud* cloud, const rsc_params* p, uint64_t seed, rsc_run** out) {
  if (!cloud || !out) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  *out = nullptr;
  if (int32_t rc = check_params(ctx, p, "ransac_run")) return rc;
  if (p->n_shape_types < 1) return fail(ctx, RSC_E_ARG, "ransac_run: nothing to sample/fit");
  const uint32_t ext = p->compat_flags & (RSC_SAMPLER_OCTREE | RSC_SCORE_PROGRESSIVE | RSC_REFIT_LSQ | RSC_EXTRACT_BITMAP);
  if (cloud->exact() && ext)
    return fail(ctx, RSC_E_STATE,
                "ransac_run: RSC_SAMPLER_OCTREE / RSC_SCORE_PROGRESSIVE / RSC_REFIT_LSQ / RSC_EXTRACT_BITMAP do not support exact clouds yet");
  // the host decides the batches of progressive scoring and of the cell sampler (and, for comparison, of any run with
  // RSC_LOOP_HOSTWALK set)
  const bool host_decides = (ext & (RSC_SCORE_PROGRESSIVE | RSC_SAMPLER_OCTREE)) || getenv("RSC_LOOP_HOSTWALK");
  if (host_decides) {
    if (cloud->is_shard()) return fail(ctx, RSC_E_STATE, "ransac_run: the extension switches are not available on sharded storage");
    if (ext & RSC_EXTRACT_BITMAP)
      return fail(ctx, RSC_E_STATE, "ransac_run: RSC_EXTRACT_BITMAP cannot be combined with RSC_SCORE_PROGRESSIVE / RSC_SAMPLER_OCTREE");
    if ((ext & RSC_SAMPLER_OCTREE) && cloud->cells.nlevels == 0)
      return fail(ctx, RSC_E_STATE, "ransac_run: RSC_SAMPLER_OCTREE needs rsc_cloud_build_cells first");
    if (ext & RSC_SCORE_PROGRESSIVE)
      for (const rsc_subset& s : cloud->subsets)
        if (!s.soa) return fail(ctx, RSC_E_STATE, "ransac_run: RSC_SCORE_PROGRESSIVE needs every subset uploaded (rsc_cloud_set_subset)");
  }
  return run_loop(cloud, p, seed, nullptr, host_decides, "ransac_run", out);
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
