/*
 * rsc.h -- C ABI of libransac_b200: the B200 (sm_100a) hot path of efficient-RANSAC shape
 * detection, built to sit underneath cserteGT3/RANSAC.jl's public surface.
 *
 * The reference has no FFI; its extension boundary is Julia multiple dispatch
 * (docs/src/newprimitive.md:12-18).  Each entry point below replaces the body of one group of
 * reference methods for the four built-in shapes, and is what a `ccall` from those methods binds
 * (see INTEGRATION.md for the Julia stubs).  Citations are relative to the reference root.
 *
 * Conventions
 *   - every function returns 0 on success, a negative RSC_E_* on failure; the message of the last
 *     failure on a context is rsc_last_error(ctx).  No exception crosses the boundary.
 *   - indices are 0-based on this side (Julia adds/subtracts 1).
 *   - host buffers are copied during the call, never retained; outputs go to caller-owned buffers.
 *   - a context (and its clouds) is bound to one CUDA device and is not thread-safe.
 *   - there is NO CPU fallback: without a usable sm_100 device rsc_ctx_create fails.
 *   - `*_dev` variants take DEVICE pointers and a cudaStream_t (as void*) and do not synchronise;
 *     they are what a multi-GPU host (one process per GPU) chains with its NCCL collectives.
 */
#ifndef RSC_H
#define RSC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RSC_VERSION 100

/* shape kinds (src/shapes/{plane,sphere,cylinder,cone}.jl) */
#define RSC_PLANE 0
#define RSC_SPHERE 1
#define RSC_CYLINDER 2
#define RSC_CONE 3
#define RSC_NTYPES 4

/* error codes */
#define RSC_OK 0
#define RSC_E_ARG (-1)      /* bad argument (the reference's @assert failures map here) */
#define RSC_E_CUDA (-2)     /* CUDA runtime error */
#define RSC_E_NODEVICE (-3) /* no sm_100 device: there is no fallback path */
#define RSC_E_NOMEM (-4)
#define RSC_E_STATE (-5)    /* e.g. subset not uploaded */
#define RSC_E_NCCL (-6)

/* compat_flags: reference behaviours that can be switched off (SURVEY.md 8a' quirk numbers) */
#define RSC_COMPAT_SPHERE_IGNORES_ENABLED 1u /* Q4: sphere.jl:121,131 */
#define RSC_COMPAT_DEFAULT (RSC_COMPAT_SPHERE_IGNORES_ENABLED)
/* extension switch (off by default): draw minimal sets with the level-weighted octree-cell sampler the
 * reference is written for (fitting.jl:383-430, octree.jl:198-205) instead of from the root cell, which
 * is what its shipped code always does (Q1: levelweight/levelscore swapped, octree.jl:82-84).
 * Needs rsc_cloud_build_cells. */
#define RSC_SAMPLER_OCTREE 2u
/* extension switch (off by default): rsc_ransac_run refits the best candidate by least squares to the
 * compatible points within 3 eps (rsc_refit_lsq) before it extracts it -- the paper's refit, which the
 * reference leaves out (docs/src/ransac.md:163-169). */
#define RSC_REFIT_LSQ 8u
/* extension switch (off by default): progressive subset scoring inside rsc_ransac_run -- what the
 * reference leaves as "TODO: refine if best.overlap" (iterations.jl:110; docs/src/ransac.md:137-141).
 * While the confidence interval of the best candidate overlaps another one (isoverlap,
 * confidenceintervals.jl:29-36) the least-evaluated candidates among the best and its overlappers are
 * scored on their next subset and re-estimated from the union; intervals are the float64 ones (no
 * Int64 wrap, Q9).  Needs every subset uploaded with rsc_cloud_set_subset. */
#define RSC_SCORE_PROGRESSIVE 16u

/* extension switch (off by default): rsc_ransac_run keeps, of every extracted shape's compatible points, only
 * those in the largest connected component of its parameter-space bitmap (rsc_bitmap_filter) -- the paper's
 * third compatibility criterion, which the reference documents and leaves out (docs/src/ransac.md:106-112).
 * Cell size / connectivity: rsc_ctx_set_bitmap.  Not with sharded storage. */
#define RSC_EXTRACT_BITMAP 32u

/* which counter plays `s` in prob(n,s,N,k): utilities.jl:297-300 */
#define RSC_S_LENGTHC 0
#define RSC_S_ALLCAND 1
#define RSC_S_NOFMINSET 2

typedef struct rsc_ctx rsc_ctx;
typedef struct rsc_cloud rsc_cloud;
typedef struct rsc_run rsc_run;

/*
 * One shape candidate, 64 bytes.  Mirrors the Fitted* structs (float64 like the reference):
 *   plane    p = point[3], normal[3], -        (plane.jl:8-11)
 *   sphere   p = center[3], radius, -,-,-      (sphere.jl:9-13)
 *   cylinder p = axis[3], center[3], radius    (cylinder.jl:11-16)
 *   cone     p = apex[3], axis[3], opang       (cone.jl:11-19; opang = FULL opening angle, rad)
 */
typedef struct rsc_cand {
  int32_t type;
  int32_t outwards; /* 0/1; ignored for planes */
  double p[7];
} rsc_cand;

/*
 * Flat mirror of the nested NamedTuple built by ransacparameters (utilities.jl:332-433).
 * Defaults (rsc_params_default) are the values pinned by test/utilitytests.jl:41-82.
 * eps/alpha are indexed by RSC_PLANE..RSC_CONE.
 */
typedef struct rsc_params {
  int32_t drawN;       /* iteration.drawN: 3..8 (the fits use the first three points, the rest only validate) */
  int32_t minsubsetN;  /* iteration.minsubsetN */
  double prob_det;     /* iteration.prob_det */
  int64_t tau;         /* iteration.tau */
  int32_t itermax;     /* iteration.itermax */
  int32_t extract_s;   /* RSC_S_* */
  int32_t terminate_s; /* RSC_S_* */
  int32_t n_shape_types;
  int32_t shape_types[RSC_NTYPES]; /* fit order, e.g. {PLANE, CONE, CYLINDER, SPHERE} (RANSAC.jl:94) */
  double collin_threshold;         /* common.collin_threshold (ineffective, Q3) */
  double parallelthrdeg;           /* common.parallelthrdeg, degrees */
  double eps[RSC_NTYPES];
  double alpha[RSC_NTYPES];
  double sphere_par;   /* sphere.sphere_par */
  double minconeopang; /* cone.minconeopang */
  uint32_t compat_flags;
  uint32_t lw_period; /* RSC_SAMPLER_OCTREE: the level weights are refreshed every lw_period iterations (0 or 1 = after
                         every iteration, the reference's schedule, iterations.jl:148); larger periods let the loop
                         batch its iterations -- the results depend on the period, not on the batching */
} rsc_params;

/* cumulative counters / device timers of a context */
typedef struct rsc_stats {
  int64_t evals;          /* candidate x point pairs evaluated by the score/refit kernels */
  int64_t exact_pairs;    /* pairs inside the FP32 guard band, re-evaluated in FP64 */
  int64_t sets_drawn;     /* minimal sets attempted */
  int64_t cands_scored;
  int64_t score_launches; /* launches of the tiled score kernel */
  double score_ms;        /* CUDA-event time of the last score call's kernels */
  double last_kernel_ms;  /* CUDA-event time of the last tiled score kernel launch alone */
  double refit_mask_ms;   /* CUDA-event time of the last refit's compatibility-mask kernel (K4, HBM bound) */
} rsc_stats;

/* ---- context ----------------------------------------------------------------------- */
int32_t rsc_version(void);
void rsc_params_default(rsc_params* p);
int32_t rsc_ctx_create(int32_t device, rsc_ctx** out);
void rsc_ctx_destroy(rsc_ctx* ctx);
const char* rsc_last_error(const rsc_ctx* ctx);
int32_t rsc_ctx_stats(rsc_ctx* ctx, rsc_stats* out);
void* rsc_ctx_stream(rsc_ctx* ctx); /* the cudaStream_t all work of this context is ordered on */
/* After a *_dev call: waits for the device, then reports the CUDA-event duration of the last tiled
 * score kernel launch alone (ms) and how many guard-band pairs it sent to FP64 (nullable outs). */
int32_t rsc_ctx_last_kernel(rsc_ctx* ctx, double* kernel_ms, int64_t* guard_pairs);

/* ---- cloud: RANSACCloud (octree.jl:37-59, ctors :78-138) ------------------------------ */
/* xyz/nrm are AoS (N x 3), bit-compatible with Vector{SVector{3,Float32}}; stored on device as
 * SoA float32.  `_f64` down-converts Vector{SVector{3,Float64}} (the device computes on the float32
 * roundings: decisions are the float64 ones OF THE ROUNDED coordinates; `_f64_exact` below keeps the
 * float64 coordinates too).  `_shard` uploads the point
 * range [global_offset, global_offset+n) of a cloud of n_global points (one shard per GPU/process,
 * sharded storage): global_offset must be a multiple of 2048 and n a multiple of 2048 unless the range
 * ends the cloud; indices the library returns or takes (subsets, inlier lists) are GLOBAL.
 * The upload is enqueued in 2 Mi-point chunks and the call returns; the next call on the cloud waits
 * for it (rsc_score on the whole cloud even follows it chunk by chunk).  From pageable arrays (a
 * Julia Vector, a NumPy array) CUDA has staged the data when the call returns and the host arrays
 * are not needed any more; PAGE-LOCKED arrays are read by DMA after the return and must stay valid
 * and unchanged until the next call on this cloud has returned. */
int32_t rsc_cloud_create(rsc_ctx* ctx, const float* xyz, const float* nrm, int64_t n, rsc_cloud** out);
int32_t rsc_cloud_create_f64(rsc_ctx* ctx, const double* xyz, const double* nrm, int64_t n, rsc_cloud** out);
int32_t rsc_cloud_create_shard(rsc_ctx* ctx, const float* xyz, const float* nrm, int64_t n,
                               int64_t global_offset, int64_t n_global, rsc_cloud** out);
/* Like rsc_cloud_create_f64, but the device also keeps the caller's float64 coordinates: every
 * decision (scoring, refit/extraction, the loops) is the float64 one of the UNROUNDED points and
 * every fit runs on them.  +48 B/point of HBM.  Refused later on: rsc_cloud_update, rsc_cloud_set_range.
 * Not yet available on an exact cloud (RSC_E_STATE): the cell sampler (rsc_sample_fit_cells,
 * RSC_SAMPLER_OCTREE), RSC_SCORE_PROGRESSIVE, RSC_REFIT_LSQ / rsc_refit_lsq and RSC_EXTRACT_BITMAP /
 * rsc_bitmap_filter.  rsc_cloud_build_cells quantises the float32 roundings; on an exact cloud its
 * cells only order the culled scorer (rsc_score_culled), whose counts do not depend on the order. */
int32_t rsc_cloud_create_f64_exact(rsc_ctx* ctx, const double* xyz, const double* nrm, int64_t n, rsc_cloud** out);
int32_t rsc_cloud_is_exact(const rsc_cloud* cloud); /* 1 / 0 */
/* Re-upload new coordinates (same n) into the device buffers of an existing cloud: all points
 * enabled again, subset copies re-gathered, the flattened octree (rsc_cloud_build_cells) dropped.
 * A re-scan of the same scene, no re-allocation. */
int32_t rsc_cloud_update(rsc_cloud* cloud, const float* xyz, const float* nrm, int64_t n);
void rsc_cloud_destroy(rsc_cloud* cloud);
int64_t rsc_cloud_size(const rsc_cloud* cloud);
/* pc.subsets (octree.jl:129-135): `idx` holds subset `subset_id`'s local point indices in subset
 * order; the device keeps a gathered contiguous copy so that scoring streams it linearly. */
/* On a shard (rsc_cloud_create_shard) `idx` holds the GLOBAL indices of the whole subset (the same array
 * on every rank); the rank keeps the entries of its own range, in subset order. */
int32_t rsc_cloud_set_subset(rsc_cloud* cloud, int32_t subset_id, const int64_t* idx, int64_t m);
int64_t rsc_cloud_subset_size(const rsc_cloud* cloud, int32_t subset_id);
/* pc.isenabled in BitArray.chunks layout: ceil(n/64) UInt64 words, bit i%64 of word i/64 */
int32_t rsc_cloud_get_enabled(rsc_cloud* cloud, uint64_t* words);
int32_t rsc_cloud_set_enabled(rsc_cloud* cloud, const uint64_t* words);
int32_t rsc_cloud_enable_all(rsc_cloud* cloud); /* ransac(pc, params, true): iterations.jl:15-19 */
int64_t rsc_cloud_count_enabled(rsc_cloud* cloud);

/* ---- scoring: scorecandidates!/scorecandidate/compatibles* ---------------------------- */
/* (fitting.jl:181-190; plane.jl:61-71,114-130; sphere.jl:118-172; cylinder.jl:172-221;
 *  cone.jl:132-167)
 * Scores C candidates against subset `subset_id` (>= 0) or the whole cloud (-1).
 *   counts[c]  = number of compatible (and enabled, except Q4) points;
 *   masks      = NULL, or C x ceil(M/32) words, row c = inlier bitmask of candidate c in subset
 *                order (bit j%32 of word j/32 = point j): inpoints = subset[mask]. */
int32_t rsc_score(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cands, int32_t C,
                  int32_t subset_id, int32_t* counts, uint32_t* masks);
/* Extension: the same counts as rsc_score(cloud, params, cands, C, -1, counts, NULL) -- whole cloud,
 * counts only -- without evaluating the pairs that cannot match.  Needs rsc_cloud_build_cells (Morton
 * order): every 128-point tile of the Morton-ordered cloud has a bounding sphere (c, r); the distance
 * functions of compatibles* are 1-Lipschitz in the point, so |dist(c)| > eps + r proves that no point
 * of the tile is compatible and the (candidate, tile) pair is skipped.  The surviving pairs go through
 * the same FP32 forms, guard band and float64 decisions as rsc_score: the counts are identical.
 * Optional outs: (candidate, tile) pairs in total / surviving the test, CUDA-event time of the kernel. */
int32_t rsc_score_culled(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cands, int32_t C,
                         int32_t* counts, int64_t* pairs_total, int64_t* pairs_survived, double* kernel_ms);
/* The same against an uploaded subset (counts == rsc_score(..., subset_id, counts, NULL)).  Needs no
 * rsc_cloud_build_cells: the first call sorts a copy of the subset into Morton order (kept with the subset, its
 * isenabled bits follow every change).  rsc_ransac_run uses this path by itself for large candidate batches
 * (environment RSC_LOOP_CULL = 0 switches that off, 2 forces it for every batch). */
int32_t rsc_score_culled_subset(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cands, int32_t C,
                                int32_t subset_id, int32_t* counts, int64_t* pairs_total, int64_t* pairs_survived,
                                double* kernel_ms);
/* device-pointer variant: d_cands/d_counts live on the context's device; enqueues on `stream`
 * (NULL = the context stream) and returns without synchronising. */
int32_t rsc_score_dev(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* d_cands, int32_t C,
                      int32_t subset_id, int32_t* d_counts, void* stream);
/* same, plus the packed inlier bitmasks, candidate-major [C][ceil(m/32)] uint32 words (LSB = first point of the
 * set; gated like the counts), written to DEVICE memory -- the counts+masks variant without a host round trip. */
int32_t rsc_score_dev_masks(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* d_cands, int32_t C,
                            int32_t subset_id, int32_t* d_counts, uint32_t* d_masks, void* stream);
/* Audit hook for the exactness argument (DESIGN.md section 4): the FP32 MARGINS the tiled kernels compute
 * for C candidates x the points [point0, point0+npoints) of the whole cloud -- the packed FFMA2 evaluation
 * of score_kernel with the hardware's MUFU.RSQ and contraction -- candidate-major into margins[C][npoints];
 * bands[C] = each candidate's guard band (a pair is decided in FP32 only if |margin| > band), col_types[C] =
 * the evaluation form (0..3, 4 = wide cone: the margin is in units of 1/cos or 1/sin of the half angle),
 * *packed_vs_scalar_diffs = pairs on which the packed and the scalar evaluation differ in any bit.
 * tests/test_guard_band_gpu.py checks |margin - float64 margin| < band / 2 on 10^8 pairs.  All outs but
 * margins are nullable. */
int32_t rsc_debug_margins(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cands, int32_t C, int64_t point0,
                          int64_t npoints, float* margins, float* bands, int32_t* col_types, int64_t* packed_vs_scalar_diffs);
/* Test hook for the device loop's small-batch scorer (the one it uses for a batch of new candidates and for
 * re-scoring a small store after an extraction): the same launch, on the whole cloud (subset_id = -1) or an
 * uploaded subset.  cv[C] = compatible real points, ce[C] = compatible enabled points, whatever the shape type
 * (the sphere quirk Q4 picks between them later).  Type ids outside 0..3 compile to no column and count 0.
 * count >= 0: the number of candidates is read from device memory and C is the capacity, as in the loop's
 * synchronisation-free path (entries count..C-1 come back 0; count > C scores C). */
int32_t rsc_debug_score_small(rsc_cloud* cloud, const rsc_params* params, int32_t subset_id, const rsc_cand* cands, int32_t C,
                              int64_t count, int32_t* cv, int32_t* ce);
/* Test hook for K5, the device loop's re-scoring of its candidate store after an extraction.  cands[nst] = the
 * store; the cloud's current enabled mask is the one of before the extraction, new_enabled (packed like
 * rsc_cloud_set_enabled) the one after, which the cloud keeps.  hit[i] = the number of subset-0 points that were
 * enabled before and are not after and are compatible with candidate i (all of them counted as enabled).  The
 * source of those points is subset 0 itself or (form bit 1) its Morton view, built if needed; the form is the
 * gathered one, in a scratch set sized by `bound` (in the loop: the extracted candidate's subset score), or (form
 * bit 0) the masked one.  A gathered attempt whose points do not fit is repeated in the masked form, as the loop
 * does.  The scorer follows RSC_LOOP_CULL and RSC_NO_SMALL like the loop's.  flags[2] (nullable) = the first
 * attempt's guard-band queue overflow and scratch overflow; survivors[nst] (nullable) = the indices of the candidates
 * that stay in the store, in order (not `best`, no hit), *n_survivors their number (nullable). */
int32_t rsc_debug_k5_hits(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cands, int32_t nst, const uint64_t* new_enabled,
                          int32_t bound, int32_t form, int32_t best, int32_t* hit, int32_t* flags, int32_t* survivors,
                          int32_t* n_survivors);
/* Measurement hook for K4 (HBM bound): average duration (ms) of the refit's compatibility-mask kernel over
 * `reps` back-to-back launches between ONE CUDA-event pair (an event pair around a single ~70 us launch
 * over-reads it by the event latency).  Nothing is extracted or disabled. */
int32_t rsc_debug_refit_mask_ms(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cand, int32_t reps,
                                double* ms_per_launch, int64_t* n_inliers);
/* estimatescore (confidenceintervals.jl:53-74), Int64 wrap-around included (Q9). */
void rsc_estimate_score(int64_t subset_len, int64_t cloud_len, int64_t count, double* out_min,
                        double* out_max, double* out_E);

/* ---- fitting: forcefitshapes!/fit x4 (fitting.jl:165-173; plane.jl:33-57; sphere.jl:29-114;
 *      cylinder.jl:34-168; cone.jl:39-128) -------------------------------------------------- */
/* idx = S x drawN local point indices.  Output candidates are compacted in (set, shape_types)
 * order (Q16); out_set[i] = source set of candidate i.  Capacity of out/out_set: S*n_shape_types. */
int32_t rsc_fit_batch(rsc_cloud* cloud, const rsc_params* params, const int64_t* idx, int32_t S,
                      rsc_cand* out, int32_t* out_set, int32_t* out_n);
/* Same fits on explicit coordinates: p, n = S x k x 3 doubles (k >= 3 points per set; points beyond
 * the minimal set only validate, like the 4-point sets of test/dummyspheretest.jl).  This is the
 * direct counterpart of fit(::Type{S}, p, n, pc, params) and needs no cloud. */
int32_t rsc_fit_points(rsc_ctx* ctx, const rsc_params* params, const double* p, const double* n,
                       int32_t S, int32_t k, rsc_cand* out, int32_t* out_set, int32_t* out_n);
/* samplepointcloud4! (fitting.jl:383-430, root cell only -- Q1) fused with the fits: minimal set
 * `set0+i` draws from Philox4x32-10 keyed by `seed`.  out_idx (S x drawN) receives the drawn
 * indices, -1 rows for failed samples (nullable). */
int32_t rsc_sample_fit(rsc_cloud* cloud, const rsc_params* params, uint64_t seed, uint64_t set0,
                       int32_t S, rsc_cand* out, int32_t* out_set, int64_t* out_idx, int32_t* out_n);

/* ---- refit + invalidate_indexes! (plane.jl:137-143; sphere.jl:179-190; cylinder.jl:228-234;
 *      cone.jl:176-182; fitting.jl:197-202) ------------------------------------------------- */
/* Compatible points among the ENABLED points of the whole cloud, ascending global indices into
 * out_idx (nullable; capacity = cloud size); *out_n = how many.  disable != 0 also clears their
 * enabled bits (and those of the uploaded subsets). */
int32_t rsc_refit_extract(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cand,
                          int64_t* out_idx, int64_t* out_n, int32_t disable);
/* Extension (SURVEY 8(f)-4; the reference's refit keeps the candidate unchanged, docs/src/ransac.md:
 * 163-169): least-squares refit of `cand` to the enabled points compatible with it inside band * eps
 * (the paper uses band = 3).  The point set is selected once, with the exact float64 decisions of
 * rsc_refit_extract; planes get the total-least-squares plane, the other shapes a Levenberg-Marquardt
 * minimisation of the squared point-to-surface distances (normal equations accumulated on the device
 * in float64, one streaming pass per step).  *out = refined shape (= *cand if fewer than 2 x #parameters
 * points are selected or the minimisation fails), *n_used = selected points, *rms = root mean square
 * distance after the refit (NaN if unchanged); n_used and rms may be NULL.  Nothing is disabled:
 * call rsc_refit_extract with *out afterwards. */
int32_t rsc_refit_lsq(rsc_cloud* cloud, const rsc_params* params, const rsc_cand* cand, double band,
                      rsc_cand* out, int64_t* n_used, double* rms);

/* Extension (SURVEY 8(f)-4, second half): the paper's third compatibility criterion, which the reference
 * documents and leaves out (docs/src/ransac.md:106-112; src/parameterspacebitmap.jl is dead code there) --
 * keep, of the points idx[0..n) (local indices, e.g. an inlier list of rsc_refit_extract(..., disable = 0)),
 * those whose cell in the shape's 2-D parameter-space bitmap (cell size ~ beta) belongs to the LARGEST
 * connected component (4-connected, or 8-connected with eight != 0; the azimuth axis of spheres, cylinders
 * and cones wraps).  out_idx (capacity n) receives them in input order, *out_n their number; info[4]
 * (nullable) = cells along u, cells along v, number of components, cells of the largest.  Definition:
 * oracle/ransac_oracle.py::bitmap_filter. */
int32_t rsc_ctx_set_bitmap(rsc_ctx* ctx, double beta, int32_t eight); /* parameters of RSC_EXTRACT_BITMAP */
int32_t rsc_bitmap_filter(rsc_cloud* cloud, const rsc_cand* cand, double beta, int32_t eight, const int64_t* idx, int64_t n,
                          int64_t* out_idx, int64_t* out_n, int32_t* info);

/* ---- point-range sharding over the GPUs of one box (one process per GPU) ----------------------
 * The path shards by point range (SURVEY.md 8e): every rank scores/refits the points it owns and the
 * per-candidate counts are summed with an int32 all-reduce.  Two layouts:
 *   (1) SHARDED STORAGE (the default for multi-GPU runs): every rank uploads only its own range with
 *       rsc_cloud_create_shard -- 24 B/point and the host->device copy scale with 1/ranks.  The enabled
 *       mask of the WHOLE cloud (1 bit/point) is replicated so that every rank draws the same Philox
 *       minimal sets; the 3 x 24 B of coordinates a set needs are gathered from their owners with one
 *       all-reduce per batch of sets; subset copies, refit, inlier lists and K5 stay local to the range.
 *       Needs a communicator (rsc_ctx_comm_init or rsc_ctx_set_allreduce).  rsc_ransac_run supports the
 *       reference behaviour in this layout (not the extension switches).
 *   (2) REPLICATED STORAGE: every rank holds the whole cloud (rsc_cloud_create) and is given a range
 *       with rsc_cloud_set_range; also works with the extension switches.
 * The all-reduce is NCCL inside the library (rsc_ctx_comm_init: libnccl.so.2 is dlopen-ed, so the
 * library itself loads without NCCL) or a host callback (rsc_ctx_set_allreduce). */
#define RSC_UNIQUE_ID_BYTES 128
/* rank 0: ncclGetUniqueId into out[128]; the host passes the bytes to the other ranks (MPI, sockets, ...) */
int32_t rsc_comm_unique_id(void* out);
/* every rank: ncclCommInitRank on the context's device; all later sharded calls on this context
 * all-reduce on the context stream with ncclAllReduce(int32, sum).  Collective. */
int32_t rsc_ctx_comm_init(rsc_ctx* ctx, const void* unique_id, int32_t rank, int32_t nranks);
int32_t rsc_ctx_comm_destroy(rsc_ctx* ctx);
/* all-reduces the library has issued through its own communicator on this context, and their payload */
int32_t rsc_ctx_comm_stats(rsc_ctx* ctx, int64_t* calls, int64_t* bytes);
/* sums `count` int32 elements at DEVICE pointer d_buf over the ranks (in place) with the context's
 * communicator or callback, enqueued on `stream` (NULL = the context stream); no synchronisation.  This is
 * what follows rsc_score_dev on a shard: per-candidate counts of the ranks' point ranges -> counts of the cloud. */
int32_t rsc_ctx_allreduce(rsc_ctx* ctx, int32_t* d_buf, int64_t count, void* stream);
/* alternative: the host sums `count` int32 elements at device pointer d_buf over the ranks, enqueued on
 * `stream` (non-zero return = failure) */
typedef int32_t (*rsc_allreduce_fn)(void* user, void* d_buf, int64_t count, void* stream);
int32_t rsc_ctx_set_allreduce(rsc_ctx* ctx, rsc_allreduce_fn fn, void* user);
/* layout (2): this rank's range [lo, hi) of a replicated cloud -- multiples of 2048 points (hi may also
 * be the cloud size); lo == hi is an empty rank, which still joins every all-reduce */
int32_t rsc_cloud_set_range(rsc_cloud* cloud, int64_t lo, int64_t hi);

/* ---- flattened octree + level-weighted cell sampler (extension; SURVEY.md 8(f)-1) -------------
 * Replaces the RegionTrees octree (octree.jl:158-244) by Morton-sorted cells: level 1 = the bounding
 * box, every level halves each axis, a cell "splits" while it holds more than 8 points
 * (octree.jl:163-165).  nlevels <= 11.  rsc_sample_fit_cells is rsc_sample_fit with the cell of a
 * level drawn from `levelweight` (restricted to the levels above the first point's leaf);
 * out_level[S] receives the level of every set.  rsc_update_levelweight is octree.jl:198-205. */
int32_t rsc_cloud_build_cells(rsc_cloud* cloud, int32_t nlevels);
int32_t rsc_cloud_cells_levels(const rsc_cloud* cloud);
int32_t rsc_cloud_get_cells(rsc_cloud* cloud, uint32_t* codes_sorted, uint32_t* perm, uint8_t* leafdepth);
int32_t rsc_sample_fit_cells(rsc_cloud* cloud, const rsc_params* params, uint64_t seed, uint64_t set0, int32_t S,
                             const double* levelweight, int32_t nlevels, rsc_cand* out, int32_t* out_set,
                             int64_t* out_idx, int32_t* out_level, int32_t* out_n);
void rsc_level_cumsum(const double* levelweight, int32_t nlevels, double* cum);
void rsc_update_levelweight(double* levelweight, const double* levelscore, int32_t nlevels);

/* ---- the whole loop: ransac(pc, params; ...) iterations.jl:35-162 for built-in shapes ------- */
int32_t rsc_ransac_run(rsc_cloud* cloud, const rsc_params* params, uint64_t seed, rsc_run** out);
int32_t rsc_run_nshapes(const rsc_run* run);
int32_t rsc_run_iterations(const rsc_run* run);
int64_t rsc_run_refined(const rsc_run* run); /* RSC_SCORE_PROGRESSIVE: (candidate, subset) evaluations beyond subset 1 */
double rsc_run_seconds(const rsc_run* run);
/* cell sampler runs: final level weights and accumulated level scores; returns the number of levels (0: root-cell run) */
int32_t rsc_run_levelweight(const rsc_run* run, double* levelweight, double* levelscore);
int32_t rsc_run_shape(const rsc_run* run, int32_t i, rsc_cand* shape, int64_t* n_inpoints);
/* sharded storage: n_inpoints above counts the indices THIS rank holds (its range's part of the list;
 * concatenated in rank order the parts are the ascending global list); this is the size of the whole list */
int64_t rsc_run_shape_total(const rsc_run* run, int32_t i);
/* host synchronisations (cudaStreamSynchronize) the loop needed, and speculative batches it ran */
int32_t rsc_run_syncs(const rsc_run* run, int32_t* batches);
/* The inlier index lists of a run stay in device memory until they are asked for: this call copies
 * list i (ascending 0-based global indices, n_inpoints of rsc_run_shape) into the caller's buffer. */
int32_t rsc_run_inpoints(const rsc_run* run, int32_t i, int64_t* out_idx);
void rsc_run_destroy(rsc_run* run);

/* ---- user-defined shapes on the device (docs/src/newprimitive.md:12-18) ------------------------
 * A user shape brings its compatibility test as CUDA C source defining
 *   __device__ bool rsc_user_compatible(const double p[7], int outwards, const double k[8],
 *                                       double x, double y, double z, double nx, double ny, double nz);
 * p / outwards are the candidate's rsc_cand fields (cand.type = the id returned below), k the constants
 * passed with each call (nk <= 8, e.g. eps and cos(alpha), computed on the host), x..nz the point's float32
 * coordinates and normal widened to double.  The library gates every point on its enabled bit itself.
 * libnvrtc.so.12 (dlopen-ed on first use) compiles the source with the library's kernel template for sm_100a,
 * --fmad=false and no fast-math: float64 + - * / sqrt round to nearest, so a host restatement in the same
 * operation order makes the same decisions (DESIGN.md section 8).  Fitting stays with the caller unless the
 * source also defines rsc_user_fit (below).  Not for
 * sharded or ranged clouds (RSC_E_STATE).  The source is passed as bytes + length. */
#define RSC_USER_TYPE0 16
/* compile only, no device needed: RSC_OK or RSC_E_ARG (RSC_E_STATE: NVRTC cannot be loaded); NVRTC's log
 * (ptxas -v included), NUL-terminated, into log[0..log_cap) (nullable) */
int32_t rsc_user_shape_check(const void* src, int64_t nbytes, void* log, int64_t log_cap);
/* compile + load on ctx, cached by the source bytes (the same source gives the same id);
 * *type_id >= RSC_USER_TYPE0.  Failure: RSC_E_ARG with NVRTC's log in rsc_last_error. */
int32_t rsc_user_shape_compile(rsc_ctx* ctx, const void* src, int64_t nbytes, int32_t* type_id);
/* rsc_score for C candidates of ONE compiled user type: counts[c] = compatible enabled points of subset
 * subset_id (-1 = the whole cloud); masks = NULL or C x ceil(M/32) words in rsc_score's layout */
int32_t rsc_user_score(rsc_cloud* cloud, const double* k, int32_t nk, const rsc_cand* cands, int32_t C,
                       int32_t subset_id, int32_t* counts, uint32_t* masks);
/* rsc_refit_extract for one user-shape candidate: ascending global indices of its compatible enabled
 * points into out_idx (nullable), *out_n how many; disable != 0 clears their enabled bits (and those of
 * the uploaded subsets) */
int32_t rsc_user_refit_extract(rsc_cloud* cloud, const double* k, int32_t nk, const rsc_cand* cand,
                               int64_t* out_idx, int64_t* out_n, int32_t disable);

/* ---- user shapes inside the sampler and the device loop ------------------------------------------
 * A user source that also defines
 *   __device__ bool rsc_user_fit(int np, const double P[8][3], const double N[8][3], const double k[8],
 *                                double p[7], int* outwards);
 * fits on the device: np = drawN (3..8), P / N the minimal set's points and normals in draw order (float32
 * widened to double), k the type's constants.  It returns true when the set yields a candidate, whose record
 * is then (type id, *outwards, p); p and *outwards are zeroed before the call.  At most one candidate per
 * (set, type), like every built-in fit.  Sources without rsc_user_fit compile as before and cannot be used
 * in a fit order.  The library looks for the token `rsc_user_fit` anywhere in the source, comments included:
 * a scoring-only source must not mention it, or its compile fails for want of the definition. */
#define RSC_MAX_ORDER 8 /* positions of a fit order: the 4 built-ins plus up to 4 user types */
/* one entry of the fit order: a built-in kind (RSC_PLANE..RSC_CONE; k ignored, eps/alpha from rsc_params) or a
 * compiled user type id (>= RSC_USER_TYPE0) with its nk <= 8 constants.  The calls below take the order as
 * `const void* order` pointing at rsc_shape_slot[norder] (an rsc_shape_slot array converts implicitly). */
typedef struct rsc_shape_slot {
  int32_t type;
  int32_t nk;
  double k[8];
} rsc_shape_slot; /* 72 bytes */
/* rsc_sample_fit with a mixed fit order (replaces params->shape_types): the same Philox sets, candidates
 * merged in (set, position in order) order.  norder = 0 only draws (out_idx).  Each type at most once,
 * norder <= 8, every user type compiled on the cloud's context with a fit (else RSC_E_ARG). */
int32_t rsc_sample_fit_user(rsc_cloud* cloud, const rsc_params* params, const void* order, int32_t norder,
                            uint64_t seed, uint64_t set0, int32_t S, rsc_cand* out, int32_t* out_set,
                            int64_t* out_idx, int32_t* out_n);
/* rsc_ransac_run with a mixed fit order: the device loop scores, refits and invalidates user candidates with
 * their compiled kernels.  Built-ins only: exactly rsc_ransac_run with that shape_types.  RSC_E_STATE on
 * sharded or ranged clouds, with RSC_SAMPLER_OCTREE / RSC_SCORE_PROGRESSIVE / RSC_REFIT_LSQ /
 * RSC_EXTRACT_BITMAP, and with RSC_LOOP_HOSTWALK set. */
int32_t rsc_ransac_run_user(rsc_cloud* cloud, const rsc_params* params, const void* order, int32_t norder,
                            uint64_t seed, rsc_run** out);

/* ---- normal estimation: oriented PCA normals of the k nearest neighbours (DESIGN.md section 8) ----------
 * For float32 AoS coordinates xyz[3 n] (the layout rsc_cloud_create takes), N(i) is the k_eff = min(k, finite
 * points) finite points j smallest in (d2(i, j), j) order, d2 = ((xj-xi)^2 + (yj-yi)^2) + (zj-zi)^2 in float64 of
 * the float32 values, every operation rounded, no FMA; i itself is included.  The normal is the unit eigenvector of
 * the smallest eigenvalue of the float64 covariance of N(i) (mean and sums in list order, divided by k_eff), or
 * (0,0,0) when k_eff < 3, when the middle eigenvalue is <= 2^-40 times the largest (collinear or coincident
 * neighbours), or when point i has a non-finite coordinate (such points appear in no list).  Sign: with a viewpoint v,
 * n . (v - p_i) >= 0 (normals face the sensor); without one, the component of largest magnitude is positive (the
 * first axis on ties).  The normalised float64 vector is rounded to float32 into nrm[3 n], ready for rsc_cloud_create.
 * 3 <= k <= 32, 1 <= n < 2^31; host in / host out, synchronising.  Device memory: about 60 B per point, plus
 * 8 n k bytes when nbr is asked for.  Cost: every point of the cells searched around a query is evaluated, so m
 * coincident points (e.g. the (0,0,0) rows of missing depth) cost O(m^2) distances, and a lone outlier, whose search
 * covers the whole box, costs n; results stay exact.
 *   viewpoint: NULL or 3 doubles.  nbr: NULL or n x k int64, row i = N(i) in (d2, index) order, -1 beyond k_eff.
 *   pairs: NULL or the number of (query, candidate) distances evaluated (for the benchmark). */
int32_t rsc_estimate_normals(rsc_ctx* ctx, const float* xyz, int64_t n, int32_t k, const double* viewpoint,
                             float* nrm, int64_t* nbr, int64_t* pairs);

/* ---- normal orientation without a viewpoint: minimum spanning forest of the k-NN graph (DESIGN.md section 8) ---
 * Makes the signs of the normals consistent over each connected piece of the cloud, for clouds with no single sensor
 * position (CAD or mesh samples, merged scans, photogrammetry, files with arbitrary signs).  Deterministic; the
 * definition, restated in oracle/orient_oracle.py orient_mst:
 *   1. point i is a vertex when its float32 coordinates are finite and its normal is finite with (x^2 + y^2) + z^2 > 0
 *      in float64; every other point is returned unchanged (a zero normal stays zero, a NaN normal is copied);
 *   2. u_i = n_i / sqrt((x^2 + y^2) + z^2) in float64 of the float32 values, every operation rounded, no FMA;
 *   3. the undirected edges are {i, j}, i != j, j in N(i) (the k-NN lists of rsc_estimate_normals, same k), both
 *      vertices; the symmetric union, duplicates merged;
 *   4. d(i, j) = (u_i.x u_j.x + u_i.y u_j.y) + u_i.z u_j.z and w = 1 - |d| in float64; edges are ordered by
 *      (w, lo, hi), lo < hi the two indices, so the minimum spanning forest F is unique;
 *   5. each tree of F is rooted at its vertex of largest float32 z (lowest index on ties); the root's sign s is +1 when
 *      u_r.z > 0, -1 when u_r.z < 0, and when u_r.z == 0 the sign that makes its largest-magnitude component positive
 *      (the first axis on ties);
 *   6. along a tree edge from parent p to child c, s(c) = s(p) when d(p, c) >= 0, else -s(p);
 *   7. nrm_out[i] = s(i) * nrm_in[i]: the input float32 normal with its sign bit flipped or not, not renormalised.
 * nrm_in NULL: the normals are first estimated exactly as rsc_estimate_normals does without a viewpoint, from the
 * same k-NN search.  nrm_in == nrm_out is allowed.  Each connected component of the graph is oriented on its own.
 *   edges: NULL or int64[2 n]: F's edges as (lo, hi) pairs in ascending order, stats[1] of them.
 *   stats: NULL or int64[4]: {vertices, edges of F, trees of F, Boruvka rounds}.
 * 3 <= k <= 32, 1 <= n < 2^31; host in / host out, synchronising.  Device memory: about (130 + 4 k) B per point plus
 * 32 B per graph edge (at most n k edges; about 0.6 n k on surface samples). */
int32_t rsc_orient_normals(rsc_ctx* ctx, const float* xyz, int64_t n, int32_t k, const float* nrm_in, float* nrm_out,
                           int64_t* edges, int64_t* stats);

/* ---- the same two on a cloud sharded by point range over the ranks of the context's communicator ----------------
 * Collective: every rank calls with its own rows [global_offset, global_offset + n) of a cloud of n_global points
 * (1 <= n_global < 2^31), the layout rsc_cloud_create_shard takes.  xyz, nrm, nbr, nrm_in and nrm_out hold this rank's
 * rows; nbr holds global indices.  The ranges must tile [0, n_global) (any order of ranks, no alignment); a rank may be
 * empty (n = 0, its row pointers may be NULL).  The concatenation of the ranks' outputs in range order is bit for bit
 * the single call's on the whole cloud: normals and lists, and the sum of the ranks' `pairs` (each rank counts its own
 * distances).  edges (capacity 2 n_global values) and stats describe the whole forest and are identical on every rank.
 * Protocol (DESIGN.md section 8):
 *   1. argument check, two all-reduces (104 B and 4 B): k, n_global, the viewpoint and whether it is given must agree,
 *      the n must sum to n_global, nbr / nrm_in must be given on all non-empty ranks or on none, and every rank must
 *      allocate the device buffers of the later steps (between the two all-reduces).  Otherwise every rank returns
 *      RSC_E_ARG; without a communicator, RSC_E_STATE at once.  After the check a rank leaves early only on a CUDA
 *      error (a device fault, a failed launch), which can leave the other ranks blocked in the next all-reduce, as in
 *      every collective of the library;
 *   2. gather: every rank's rows into a zero-filled n_global record buffer (coordinates + a coverage word: 16 B per
 *      point; 28 B with nrm_in, whose normals travel along), one all-reduce; overlapping or missing rows: RSC_E_ARG on
 *      every rank;
 *   3. every rank sorts the whole cloud as rsc_estimate_normals does and searches one contiguous run of the sorted
 *      queries; the non-empty ranks share the finite points equally;
 *   4. the rows (normals 12 B, int64 lists 8 k B / int32 lists 4 k B per point) return to their owners through one
 *      zero-filled n_global buffer and one all-reduce; orientation then builds the forest on every rank.
 * All-reduces per call: 4.  Volume: estimation 104 + 4 + (16 + 12) n_global B, plus 8 k n_global with nbr;
 * orientation 104 + 4 + (28 + 4 k) n_global B.  Device memory per rank: the single call's on n_global points, plus
 * the record and row buffers (16 + 12 B per point, + 8 k / 4 k).  The search divides over the ranks; the gather, the
 * sort, the exchanges and orientation's forest are replicated. */
int32_t rsc_estimate_normals_shard(rsc_ctx* ctx, const float* xyz, int64_t n, int64_t global_offset, int64_t n_global,
                                   int32_t k, const double* viewpoint, float* nrm, int64_t* nbr, int64_t* pairs);
int32_t rsc_orient_normals_shard(rsc_ctx* ctx, const float* xyz, int64_t n, int64_t global_offset, int64_t n_global,
                                 int32_t k, const float* nrm_in, float* nrm_out, int64_t* edges, int64_t* stats);

#ifdef __cplusplus
}
#endif
#endif /* RSC_H */
