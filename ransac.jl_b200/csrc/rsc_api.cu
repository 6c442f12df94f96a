// rsc_api.cu -- extern "C" entry points of libransac_b200 (include/rsc.h): context, scoring,
// refit/extract, score statistics.  Host-side glue only; the kernels live in rsc_score.cu,
// rsc_extract.cu, rsc_fit.cu, rsc_cloud.cu.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "rsc_common.cuh"

namespace rsc {

int32_t fail(rsc_ctx* ctx, int32_t code, const char* what) {
  if (ctx) ctx->err = what ? what : "error";
  return code;
}

int32_t fail_cuda(rsc_ctx* ctx, cudaError_t e, const char* where) {
  if (ctx) {
    ctx->err = std::string(where ? where : "cuda") + ": " + cudaGetErrorString(e);
  }
  return e == cudaErrorMemoryAllocation ? RSC_E_NOMEM : RSC_E_CUDA;
}

static int32_t check_params(rsc_ctx* ctx, const rsc_params* p) {
  if (!p) return fail(ctx, RSC_E_ARG, "params is null");
  for (int t = 0; t < RSC_NTYPES; ++t)
    if (!(p->eps[t] == p->eps[t]) || !(p->alpha[t] == p->alpha[t])) return fail(ctx, RSC_E_ARG, "params: NaN threshold");
  return RSC_OK;
}

static int32_t pick_pointset(rsc_cloud* cloud, int32_t subset_id, PointSet* ps) {
  rsc_ctx* ctx = cloud->ctx;
  if (subset_id < 0) {
    *ps = view_cloud(cloud);
    return RSC_OK;
  }
  if ((size_t)subset_id >= cloud->subsets.size() || !cloud->subsets[subset_id].soa)
    return fail(ctx, RSC_E_STATE, "score: subset not uploaded (rsc_cloud_set_subset)");
  *ps = view_subset(&cloud->subsets[subset_id]);
  return RSC_OK;
}

// chunked scoring: every per-chunk score_enqueue resets the guard-band queue fill, so a chunk's overflow
// is latched here (wl_count[2] = largest fill that exceeded the capacity) before the next chunk runs
__global__ void latch_overflow_kernel(uint32_t* __restrict__ wl_count, uint32_t cap) {
  const uint32_t m = wl_count[0] > wl_count[1] ? wl_count[0] : wl_count[1];
  if (m > cap && m > wl_count[2]) wl_count[2] = m;
}

}  // namespace rsc

using namespace rsc;

extern "C" {

int32_t rsc_version(void) { return RSC_VERSION; }

void rsc_params_default(rsc_params* p) {
  if (!p) return;
  memset(p, 0, sizeof(*p));
  // utilities.jl:345,371; plane.jl:22; sphere.jl:25; cylinder.jl:27; cone.jl:30; RANSAC.jl:94
  p->drawN = 3;
  p->minsubsetN = 15;
  p->prob_det = 0.9;
  p->tau = 900;
  p->itermax = 1000;
  p->extract_s = RSC_S_NOFMINSET;
  p->terminate_s = RSC_S_NOFMINSET;
  p->n_shape_types = 4;
  p->shape_types[0] = RSC_PLANE;
  p->shape_types[1] = RSC_CONE;
  p->shape_types[2] = RSC_CYLINDER;
  p->shape_types[3] = RSC_SPHERE;
  p->collin_threshold = 0.2;
  p->parallelthrdeg = 1.0;
  const double five_deg = 5.0 * 3.14159265358979323846 / 180.0;
  for (int t = 0; t < RSC_NTYPES; ++t) {
    p->eps[t] = 0.3;
    p->alpha[t] = five_deg;
  }
  p->sphere_par = 0.02;
  p->minconeopang = 2.0 * 3.14159265358979323846 / 180.0;
  p->compat_flags = RSC_COMPAT_DEFAULT;
}

int32_t rsc_ctx_create(int32_t device, rsc_ctx** out) {
  if (!out) return RSC_E_ARG;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return RSC_E_NODEVICE;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return RSC_E_NODEVICE;
  if (prop.major != 10) return RSC_E_NODEVICE;  // built for sm_100a only; there is no fallback
  if (cudaSetDevice(device) != cudaSuccess) return RSC_E_CUDA;
  rsc_ctx* ctx = new rsc_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  if (const char* e = getenv("RSC_WL_CAP")) {  // test hook: start with a tiny guard-band queue
    const long v = atol(e);
    if (v > 0) ctx->wl_cap = (size_t)v;
  }
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess ||
      cudaEventCreate(&ctx->evk0) != cudaSuccess || cudaEventCreate(&ctx->evk1) != cudaSuccess ||
      cudaEventCreate(&ctx->evr0) != cudaSuccess || cudaEventCreate(&ctx->evr1) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) != cudaSuccess) {
    rsc_ctx_destroy(ctx);  // releases whatever was created (handles start out null)
    return RSC_E_CUDA;
  }
  for (int i = 0; i < 4; ++i)
    if (cudaStreamCreateWithFlags(&ctx->sfork[i], cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming) != cudaSuccess) {
      rsc_ctx_destroy(ctx);
      return RSC_E_CUDA;
    }
  *out = ctx;
  return RSC_OK;
}

void rsc_ctx_destroy(rsc_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  rsc::DevBuf* bufs[] = {&ctx->cands,    &ctx->rec,      &ctx->orig,     &ctx->slot_of, &ctx->blktab,
                         &ctx->counts,   &ctx->masks_gm, &ctx->masks_cm, &ctx->worklist, &ctx->wl_count, &ctx->pairs,
                         &ctx->aux,      &ctx->misc,     &ctx->misc2,    &ctx->idxbuf,  &ctx->fitbuf, &ctx->selbuf, &ctx->exq, &ctx->scanbuf, &ctx->lsqbuf, &ctx->cullbuf, &ctx->shardbuf, &ctx->gselbuf, &ctx->smallbuf, &ctx->viewtmp};
  for (auto* b : bufs) b->release();
  rsc::loop_scratch_free(ctx);
  rsc::user_shapes_free(ctx);
  if (ctx->comm) rsc_ctx_comm_destroy(ctx);
  ctx->stage[0].release(), ctx->stage[1].release();
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  for (int i = 0; i < 4; ++i) {
    if (ctx->sfork[i]) cudaStreamSynchronize(ctx->sfork[i]), cudaStreamDestroy(ctx->sfork[i]);
    if (ctx->ev_join[i]) cudaEventDestroy(ctx->ev_join[i]);
  }
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  for (int b = 0; b < 2; ++b) {
    if (ctx->hstage[b]) cudaFreeHost(ctx->hstage[b]);
    if (ctx->hstage_free[b]) cudaEventDestroy(ctx->hstage_free[b]);
  }
  for (cudaEvent_t e : {ctx->ev0, ctx->ev1, ctx->evk0, ctx->evk1, ctx->evr0, ctx->evr1})
    if (e) cudaEventDestroy(e);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  cudaGetLastError();  // a failed create leaves nothing sticky behind
  delete ctx;
}

const char* rsc_last_error(const rsc_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int32_t rsc_ctx_stats(rsc_ctx* ctx, rsc_stats* out) {
  if (!ctx || !out) return RSC_E_ARG;
  *out = ctx->stats;
  return RSC_OK;
}

void* rsc_ctx_stream(rsc_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int32_t rsc_ctx_last_kernel(rsc_ctx* ctx, double* kernel_ms, int64_t* guard_pairs) {
  if (!ctx) return RSC_E_ARG;
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  RSC_CUDA(ctx, cudaDeviceSynchronize());
  if (kernel_ms) {
    float ms = 0.f;
    RSC_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->evk0, ctx->evk1));
    *kernel_ms = ms;
    ctx->stats.last_kernel_ms = ms;
  }
  if (guard_pairs) {
    uint32_t n[2] = {0, 0};
    if (ctx->wl_count.p) RSC_CUDA(ctx, cudaMemcpy(n, ctx->wl_count.p, sizeof(n), cudaMemcpyDeviceToHost));
    if (n[0] > ctx->wl_cap || n[1] > ctx->wl_cap) {
      const size_t need = n[0] > n[1] ? n[0] : n[1];
      ctx->wl_cap = need + need / 4 + 1024;  // the next call has room; this one's counts are incomplete
      return fail(ctx, RSC_E_STATE, "guard-band queue overflowed in a *_dev call: repeat the call");
    }
    *guard_pairs = n[1];
  }
  return RSC_OK;
}

// ---------------------------------------------------------------------------------------------
// scoring
// ---------------------------------------------------------------------------------------------
int32_t rsc_score(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cands, int32_t C,
                  int32_t subset_id, int32_t* counts, uint32_t* masks) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (C < 0 || (C > 0 && (!cands || !counts))) return fail(ctx, RSC_E_ARG, "score: null candidates/counts");
  int32_t rc = check_params(ctx, params);
  if (rc) return rc;
  if (C == 0) return RSC_OK;
  for (int i = 0; i < C; ++i)
    if (cands[i].type < 0 || cands[i].type >= RSC_NTYPES) return fail(ctx, RSC_E_ARG, "score: unknown shape type");
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  // a chunked upload still in flight: whole-cloud, counts-only scoring follows it chunk by chunk
  const bool chunked = cloud->pending && subset_id < 0 && !masks;
  if (!chunked && (rc = cloud_ready(cloud))) return rc;
  PointSet ps;
  if ((rc = pick_pointset(cloud, subset_id, &ps))) return rc;
  const Thresh th = make_thresh(params);
  cudaStream_t st = ctx->stream;

  // candidates + host-libm cos/sin(-opang/2) for the FP64 path (cone.jl:78)
  std::vector<double> trig((size_t)2 * C, 0.0);
  for (int i = 0; i < C; ++i)
    if (cands[i].type == RSC_CONE) {
      trig[2 * i] = cos(-cands[i].p[6] / 2);
      trig[2 * i + 1] = sin(-cands[i].p[6] / 2);
    }
  RSC_CUDA(ctx, ctx->cands.ensure((size_t)C * sizeof(rsc_cand)));
  RSC_CUDA(ctx, ctx->aux.ensure((size_t)2 * C * sizeof(double)));
  RSC_CUDA(ctx, ctx->counts.ensure((size_t)3 * C * sizeof(int32_t)));
  RSC_CUDA(ctx, cudaMemcpyAsync(ctx->cands.p, cands, (size_t)C * sizeof(rsc_cand), cudaMemcpyHostToDevice, st));
  RSC_CUDA(ctx, cudaMemcpyAsync(ctx->aux.p, trig.data(), (size_t)2 * C * sizeof(double), cudaMemcpyHostToDevice, st));

  for (int attempt = 0; attempt < 3; ++attempt) {
    RSC_CUDA(ctx, cudaEventRecord(ctx->ev0, st));
    int32_t* d_policy = ctx->counts.as<int32_t>() + 2 * (size_t)C;
    if (chunked && attempt == 0) {
      const int nchunks = cloud->n_chunks();
      RSC_CUDA(ctx, ctx->wl_count.ensure(16));
      RSC_CUDA(ctx, cudaMemsetAsync(ctx->wl_count.as<uint32_t>() + 2, 0, sizeof(uint32_t), st));
      for (int i = 0; i < nchunks && !rc; ++i) {
        const int64_t off = cloud->chunk_begin(i);
        PointSet sl = ps;
        sl.x += off, sl.y += off, sl.z += off, sl.nx += off, sl.ny += off, sl.nz += off;
        sl.enabled += off / 32, sl.valid += off / 32;
        if (sl.xyz64) sl.xyz64 += 3 * off, sl.nrm64 += 3 * off;  // (the whole cloud: no map)
        sl.n = cloud->chunk_begin(i + 1) - off;
        sl.n_pad = (i == nchunks - 1) ? cloud->n_pad - off : sl.n;
        RSC_CUDA(ctx, cudaStreamWaitEvent(st, cloud->chunk_ev[i], 0));
        rc = score_enqueue(ctx, cloud, sl, th, ctx->cands.as<rsc_cand>(), C, i == nchunks - 1 ? d_policy : nullptr, false, st,
                           ctx->counts.as<int32_t>(), ctx->counts.as<int32_t>() + C, ctx->aux.as<double>(),
                           cloud->d_bounds + 2 * i, i > 0);
        if (!rc) {
          latch_overflow_kernel<<<1, 1, 0, st>>>(ctx->wl_count.as<uint32_t>(), (uint32_t)ctx->wl_cap);
          RSC_CUDA(ctx, cudaGetLastError());
        }
      }
      if (rc) return rc;
      if ((rc = cloud_ready(cloud))) return rc;
    } else {
      rc = score_enqueue(ctx, cloud, ps, th, ctx->cands.as<rsc_cand>(), C, d_policy, masks != nullptr, st,
                         ctx->counts.as<int32_t>(), ctx->counts.as<int32_t>() + C, ctx->aux.as<double>());
      if (rc) return rc;
    }
    RSC_CUDA(ctx, cudaEventRecord(ctx->ev1, st));
    uint32_t nq[3] = {0, 0, 0};  // queued groups, queued pairs, latched overflow of an earlier chunk
    const bool latched = chunked && attempt == 0;
    RSC_CUDA(ctx, cudaMemcpyAsync(counts, d_policy, (size_t)C * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    RSC_CUDA(ctx, cudaMemcpyAsync(nq, ctx->wl_count.p, (latched ? 3 : 2) * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    RSC_CUDA(ctx, cudaStreamSynchronize(st));
    const uint32_t namb = nq[1];
    if ((size_t)nq[0] > ctx->wl_cap || (size_t)nq[1] > ctx->wl_cap || nq[2] != 0) {  // a guard-band queue overflowed: grow, redo
      size_t need = nq[0] > nq[1] ? nq[0] : nq[1];
      if (nq[2] > need) need = nq[2];
      ctx->wl_cap = need + need / 4 + 1024;
      ctx->stats.evals -= (int64_t)C * ps.n;
      ctx->stats.cands_scored -= C;
      continue;
    }
    ctx->stats.exact_pairs += namb;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
    ctx->stats.score_ms = ms;
    cudaEventElapsedTime(&ms, ctx->evk0, ctx->evk1);
    ctx->stats.last_kernel_ms = ms;
    if (masks) {
      if ((rc = masks_to_candidate_major(ctx, C, ps.n, st))) return rc;
      const size_t words = (size_t)((ps.n + 31) / 32);
      RSC_CUDA(ctx, cudaMemcpyAsync(masks, ctx->masks_cm.p, (size_t)C * words * 4, cudaMemcpyDeviceToHost, st));
      RSC_CUDA(ctx, cudaStreamSynchronize(st));
    }
    return RSC_OK;
  }
  return fail(ctx, RSC_E_STATE, "score: guard-band queue kept overflowing");
}

int32_t rsc_score_dev(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* d_cands, int32_t C,
                      int32_t subset_id, int32_t* d_counts, void* stream) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (C < 0 || (C > 0 && (!d_cands || !d_counts))) return fail(ctx, RSC_E_ARG, "score_dev: null device pointers");
  int32_t rc = check_params(ctx, params);
  if (rc) return rc;
  if (C == 0) return RSC_OK;
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if ((rc = cloud_ready(cloud))) return rc;
  PointSet ps;
  if ((rc = pick_pointset(cloud, subset_id, &ps))) return rc;
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  return score_enqueue(ctx, cloud, ps, make_thresh(params), d_cands, C, d_counts, false, st);
}

int32_t rsc_score_dev_masks(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* d_cands, int32_t C,
                            int32_t subset_id, int32_t* d_counts, uint32_t* d_masks, void* stream) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (C < 0 || (C > 0 && (!d_cands || !d_counts || !d_masks))) return fail(ctx, RSC_E_ARG, "score_dev_masks: null device pointers");
  int32_t rc = check_params(ctx, params);
  if (rc) return rc;
  if (C == 0) return RSC_OK;
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if ((rc = cloud_ready(cloud))) return rc;
  PointSet ps;
  if ((rc = pick_pointset(cloud, subset_id, &ps))) return rc;
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  if ((rc = score_enqueue(ctx, cloud, ps, make_thresh(params), d_cands, C, d_counts, true, st))) return rc;
  return masks_to_candidate_major(ctx, C, ps.n, st, d_masks);
}

// Measurement hook: average duration of K4's mask kernel over `reps` back-to-back launches (one CUDA-event pair)
int32_t rsc_debug_refit_mask_ms(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cand, int32_t reps, double* ms_per_launch,
                                int64_t* n_inliers) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (!cand || !ms_per_launch || reps < 2 || reps > 1000) return fail(ctx, RSC_E_ARG, "debug_refit_mask_ms: bad arguments (2 <= reps <= 1000)");
  if (cand->type < 0 || cand->type >= RSC_NTYPES) return fail(ctx, RSC_E_ARG, "debug_refit_mask_ms: unknown shape type");
  int32_t rc = check_params(ctx, params);
  if (rc) return rc;
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if ((rc = cloud_ready(cloud))) return rc;
  Thresh th = make_thresh(params);
  th.honour_enabled = 0xFu;
  if ((rc = refit_mask_enqueue(cloud, th, *cand, ctx->stream, reps))) return rc;
  unsigned long long total = 0;
  RSC_CUDA(ctx, cudaMemcpyAsync(&total, ctx->misc2.p, sizeof(total), cudaMemcpyDeviceToHost, ctx->stream));
  RSC_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  float ms = 0.f;
  RSC_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->evr0, ctx->evr1));
  *ms_per_launch = (double)ms / reps;
  if (n_inliers) *n_inliers = (int64_t)total;
  return RSC_OK;
}

// Audit of the FP32 guard band on the real hardware: the margins the tiled kernels compute.
int32_t rsc_debug_margins(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cands, int32_t C, int64_t point0,
                          int64_t npoints, float* margins, float* bands, int32_t* col_types, int64_t* packed_vs_scalar_diffs) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (C <= 0 || C > 65535 || !cands || !margins || npoints <= 0 || point0 < 0 || point0 + npoints > cloud->n)
    return fail(ctx, RSC_E_ARG, "debug_margins: bad arguments (1 <= C <= 65535, point range inside the cloud)");
  int32_t rc = check_params(ctx, params);
  if (rc) return rc;
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if ((rc = cloud_ready(cloud))) return rc;
  cudaStream_t st = ctx->stream;
  const size_t o_rec = ((size_t)C * sizeof(rsc_cand) + 255) / 256 * 256, o_col = o_rec + ((size_t)C * kRecFields * 4 + 255) / 256 * 256;
  const size_t o_diff = o_col + ((size_t)C * 4 + 255) / 256 * 256, o_out = o_diff + 256;
  RSC_CUDA(ctx, ctx->cullbuf.ensure(o_out + (size_t)C * npoints * 4));
  char* b = ctx->cullbuf.as<char>();
  rsc_cand* d_c = (rsc_cand*)b;
  float* d_rec = (float*)(b + o_rec);
  int32_t* d_col = (int32_t*)(b + o_col);
  unsigned long long* d_diff = (unsigned long long*)(b + o_diff);
  float* d_out = (float*)(b + o_out);
  RSC_CUDA(ctx, cudaMemcpyAsync(d_c, cands, (size_t)C * sizeof(rsc_cand), cudaMemcpyHostToDevice, st));
  RSC_CUDA(ctx, cudaMemsetAsync(d_diff, 0, 8, st));
  if ((rc = audit_margins(ctx, cloud, view_cloud(cloud), make_thresh(params), d_c, C, point0, npoints, d_out, d_rec, d_col, d_diff, st)))
    return rc;
  RSC_CUDA(ctx, cudaMemcpyAsync(margins, d_out, (size_t)C * npoints * 4, cudaMemcpyDeviceToHost, st));
  std::vector<float> rec((size_t)C * kRecFields);
  RSC_CUDA(ctx, cudaMemcpyAsync(rec.data(), d_rec, rec.size() * 4, cudaMemcpyDeviceToHost, st));
  if (col_types) RSC_CUDA(ctx, cudaMemcpyAsync(col_types, d_col, (size_t)C * 4, cudaMemcpyDeviceToHost, st));
  unsigned long long diffs = 0;
  RSC_CUDA(ctx, cudaMemcpyAsync(&diffs, d_diff, 8, cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaStreamSynchronize(st));
  if (bands)
    for (int i = 0; i < C; ++i) bands[i] = rec[(size_t)i * kRecFields + kBandField];
  if (packed_vs_scalar_diffs) *packed_vs_scalar_diffs = (int64_t)diffs;
  return RSC_OK;
}

// Test hook: the small-batch scorer (rsc_small.cu) as the device loop launches it, on a cloud or a subset.
int32_t rsc_debug_score_small(rsc_cloud* cloud, const rsc_params* params, int32_t subset_id, const rsc_cand* cands, int32_t C,
                              int64_t count, int32_t* cv, int32_t* ce) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (C <= 0 || !cands || !cv || !ce) return fail(ctx, RSC_E_ARG, "debug_score_small: bad arguments (C >= 1, non-null buffers)");
  int32_t rc = check_params(ctx, params);
  if (rc) return rc;
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if ((rc = cloud_ready(cloud))) return rc;
  PointSet ps;
  if ((rc = pick_pointset(cloud, subset_id, &ps))) return rc;
  cudaStream_t st = ctx->stream;
  // [candidates][cv: C][ce: C][count: u64]
  const size_t o_cnt = ((size_t)C * sizeof(rsc_cand) + 255) / 256 * 256, o_n = o_cnt + ((size_t)2 * C * 4 + 255) / 256 * 256;
  RSC_CUDA(ctx, ctx->cullbuf.ensure(o_n + 8));
  char* b = ctx->cullbuf.as<char>();
  int32_t* d_cv = (int32_t*)(b + o_cnt);
  unsigned long long* d_n = (unsigned long long*)(b + o_n);
  const unsigned long long n = count >= 0 ? (unsigned long long)count : 0ull;
  RSC_CUDA(ctx, cudaMemcpyAsync(b, cands, (size_t)C * sizeof(rsc_cand), cudaMemcpyHostToDevice, st));
  RSC_CUDA(ctx, cudaMemcpyAsync(d_n, &n, 8, cudaMemcpyHostToDevice, st));
  if ((rc = score_small_enqueue(ctx, cloud, ps, make_thresh(params), (const rsc_cand*)b, C, count >= 0 ? d_n : nullptr, d_cv, d_cv + C, st)))
    return rc;
  RSC_CUDA(ctx, cudaMemcpyAsync(cv, d_cv, (size_t)C * 4, cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaMemcpyAsync(ce, d_cv + C, (size_t)C * 4, cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaStreamSynchronize(st));
  return RSC_OK;
}

static inline int64_t wrapmul(int64_t a, int64_t b) { return (int64_t)((uint64_t)a * (uint64_t)b); }

void rsc_estimate_score(int64_t subset_len, int64_t cloud_len, int64_t count, double* out_min, double* out_max,
                        double* out_E) {
  // confidenceintervals.jl:53-74 with Julia's Int64 wrap-around (Q9)
  const int64_t N = -2 - subset_len, x = -2 - cloud_len, n = -1 - count;
  const int64_t xn = wrapmul(x, n);
  const int64_t prod = wrapmul(wrapmul(xn, N - x), N - n);
  const double sq_ = (double)prod / (double)(N - 1);
  const double sq = sq_ < 0 ? 0.0 : sqrt(sq_);
  const double a = -1 - ((double)xn + sq) / (double)N;
  const double b = -1 - ((double)xn - sq) / (double)N;
  double lo, hi;
  if (a != a || b != b) {
    lo = hi = NAN;
  } else {
    lo = a < b ? a : b;
    hi = a < b ? b : a;
  }
  if (out_min) *out_min = lo;
  if (out_max) *out_max = hi;
  if (out_E) *out_E = (lo + hi) / 2;
}

// ---------------------------------------------------------------------------------------------
// refit + invalidate
// ---------------------------------------------------------------------------------------------
int32_t rsc_refit_extract(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cand, int64_t* out_idx,
                          int64_t* out_n, int32_t disable) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (!cand || !out_n) return fail(ctx, RSC_E_ARG, "refit_extract: null candidate/out_n");
  if (cand->type < 0 || cand->type >= RSC_NTYPES) return fail(ctx, RSC_E_ARG, "refit_extract: unknown shape type");
  int32_t rc = check_params(ctx, params);
  if (rc) return rc;
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if ((rc = cloud_ready(cloud))) return rc;
  cudaStream_t st = ctx->stream;
  Thresh th = make_thresh(params);
  th.honour_enabled = 0xFu;  // refit always works on the enabled points (e.g. sphere.jl:181-185)
  if ((rc = refit_mask_enqueue(cloud, th, *cand, st))) return rc;
  unsigned long long total = 0;
  RSC_CUDA(ctx, cudaMemcpyAsync(&total, ctx->misc2.p, sizeof(total), cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaStreamSynchronize(st));
  {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->evr0, ctx->evr1) == cudaSuccess) ctx->stats.refit_mask_ms = ms;
  }
  *out_n = (int64_t)total;
  int64_t* d_out = nullptr;
  if (out_idx && total) {
    RSC_CUDA(ctx, ctx->misc.ensure((size_t)total * sizeof(int64_t)));
    d_out = ctx->misc.as<int64_t>();
  }
  if (d_out || disable) {
    if ((rc = refit_write_enqueue(cloud, d_out, disable != 0, st))) return rc;
    if (d_out)
      RSC_CUDA(ctx, cudaMemcpyAsync(out_idx, d_out, (size_t)total * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    RSC_CUDA(ctx, cudaStreamSynchronize(st));
  }
  return RSC_OK;
}

}  // extern "C"
