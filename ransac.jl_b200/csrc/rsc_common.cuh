// rsc_common.cuh -- internal structures shared by the kernels of libransac_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <string>
#include <vector>

#include "rsc.h"

namespace rsc {

// ---- tiling constants of the score kernel (K2) ------------------------------------------------
constexpr int kThreads = 128;      // threads per CTA: one candidate "slot" column per thread
constexpr int kTile = 512;         // points staged in shared memory per tile
constexpr int kGroupsPerTile = kTile / 32;
constexpr int kRecFields = 12;     // floats per compiled candidate record (SoA over slots)
constexpr int kBandField = 11;     // record field holding the FP32 guard band
// Column (kernel) types of the tiled scorer: the four public shape types plus wide cones (opening
// angle > 120 deg), which are evaluated in a form scaled by 1/sin(opang/2) instead of 1/cos(opang/2).
constexpr int kColTypes = 5;
constexpr int kConeWide = 4;
__host__ __device__ constexpr int public_type(int col_type) { return col_type == kConeWide ? RSC_CONE : col_type; }

// SoA float32 view of a set of points resident in HBM (the whole cloud shard or a gathered subset).
// All arrays have n_pad (multiple of kTile) elements; padding points are zero with enabled=valid=0.
struct PointSet {
  const float* x;
  const float* y;
  const float* z;
  const float* nx;
  const float* ny;
  const float* nz;
  const uint32_t* enabled;  // bit j%32 of word j/32 = pc.isenabled of point j
  const uint32_t* valid;    // 1 for real points, 0 for padding
  int64_t n;
  int64_t n_pad;
  // exact clouds (rsc_cloud_create_f64_exact): the caller's float64 coordinates, AoS [3 n] in the cloud's point
  // order; real point j of the set is cloud point map[j] (map == nullptr: j).  Null for every other cloud.
  const double* xyz64 = nullptr;
  const double* nrm64 = nullptr;
  const int64_t* map = nullptr;
};

// per-type thresholds, FP32 for the tiled kernel and FP64 for the exact re-evaluation
struct Thresh {
  float eps[RSC_NTYPES];
  float cosa[RSC_NTYPES];
  double eps_d[RSC_NTYPES];
  double cosa_d[RSC_NTYPES];
  uint32_t honour_enabled;  // bit t set: type t ANDs pc.isenabled into its inliers (Q4 clears SPHERE)
  uint32_t exact_in = 0;    // 1: the points are the float32 roundings of float64 ones and every decision is the float64
                            // one of the unrounded point: the guard bands carry the input-rounding term (kappa_in)
};

// block table written by the candidate compiler: which slots/type each CTA column covers
struct BlockTab {
  int32_t type;   // -1: empty column
  int32_t slot0;  // first slot of the column
};

// growable device buffer
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const {
    return reinterpret_cast<T*>(p);
  }
};

}  // namespace rsc

struct rsc_ctx {
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;  // host->device uploads, overlapped with scoring of earlier chunks
  rsc::DevBuf stage[2];                // double-buffered AoS staging of one upload chunk
  // page-locked host staging for PAGEABLE caller arrays (rsc_cloud.cu): worker threads copy the caller's data
  // into it, the DMA engine takes it from there -- 2-3 x the rate of cudaMemcpy from pageable memory
  void* hstage[2] = {nullptr, nullptr};
  size_t hstage_cap = 0;
  cudaEvent_t hstage_free[2] = {nullptr, nullptr};
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evk0 = nullptr, evk1 = nullptr, evr0 = nullptr, evr1 = nullptr;
  cudaStream_t sfork[4] = {nullptr, nullptr, nullptr, nullptr};  // the per-type score kernels of one call run side by side
  cudaEvent_t ev_fork = nullptr, ev_join[4] = {nullptr, nullptr, nullptr, nullptr};
  void* loop_scratch = nullptr;        // rsc::LoopScratch of rsc_ransac_run, kept between runs (rsc_run.cu)
  int last_cslots = 0;                 // slot stride of the last compiled candidate records / masks
  std::string err;
  rsc_stats stats{};
  // scratch of the score path
  rsc::DevBuf cands, rec, orig, slot_of, blktab, counts, masks_gm, masks_cm, worklist, pairs, wl_count, aux;
  rsc::DevBuf misc, misc2, idxbuf, fitbuf, selbuf, exq, scanbuf, lsqbuf, cullbuf, shardbuf, gselbuf, smallbuf, viewtmp;
  size_t wl_cap = 1u << 22;  // guard-band queue capacity (groups / pairs), grows on overflow
  rsc_allreduce_fn allreduce = nullptr;  // sums int32 device buffers across the ranks of a sharded run
  void* allreduce_user = nullptr;
  void* comm = nullptr;                  // ncclComm_t of rsc_ctx_comm_init (rsc_comm.cu); allreduce then points into the library
  int rank = 0, nranks = 1;
  int64_t allreduce_calls = 0, allreduce_bytes = 0;
  double bitmap_beta = 0.0;  // RSC_EXTRACT_BITMAP: cell size of the parameter-space bitmap (rsc_ctx_set_bitmap)
  int bitmap_eight = 0;
  void* pinned = nullptr;    // small pinned staging area
  size_t pinned_cap = 0;
  void* user_shapes = nullptr;  // rsc::UserShapes of rsc_user.cu: the NVRTC-compiled programs of user-defined shapes
};

struct rsc_subset {
  int64_t m = 0, m_pad = 0;
  int64_t m_global = 0;        // size of the whole subset (= m unless the cloud is a shard: then m counts this rank's entries)
  float* soa = nullptr;        // 6 * m_pad floats
  uint32_t* enabled = nullptr; // m_pad/32 words
  uint32_t* valid = nullptr;
  int64_t* idx = nullptr;      // m local point indices (device)
  const double* xyz64 = nullptr, *nrm64 = nullptr;  // the cloud's float64 coordinates (exact clouds; idx maps into them)
  // Morton-ordered view for the culled scorer (rsc_cull.cu), built on first use by subset_cull_view():
  // the same m points in a spatially coherent order + bounding spheres of their 128 / 512-point tiles
  float* csoa = nullptr;       // 6 * m_pad floats
  uint32_t* cen = nullptr;     // m_pad/32 words: pc.isenabled in that order (kept current with `enabled`)
  int64_t* cidx = nullptr;     // m local point indices in that order
  void* ctiles = nullptr;      // float4 [cull_sphere_count(m_pad)]: spheres of the 128 / 512 / 4096-point tiles
  void release_cull_view() {
    if (csoa) cudaFree(csoa);
    if (cen) cudaFree(cen);
    if (cidx) cudaFree(cidx);
    if (ctiles) cudaFree(ctiles);
    csoa = nullptr, cen = nullptr, cidx = nullptr, ctiles = nullptr;
  }
};

// flattened octree of a cloud (rsc_octree.cu): Morton-sorted codes, cells = contiguous code ranges
struct rsc_cells {
  int nlevels = 0;               // 0: not built
  uint32_t* codes = nullptr;     // [n] sorted Morton codes (3 (nlevels-1) bits)
  uint32_t* perm = nullptr;      // [n] sorted position -> point index
  int64_t* perm64 = nullptr;     // [n] the same, widened: the map of msoa into an exact cloud's float64 coordinates
  uint32_t* inv = nullptr;       // [n] point index -> sorted position
  uint8_t* leafdepth = nullptr;  // [n] by point index: first level whose cell holds <= 8 points
  uint32_t* en_sorted = nullptr; // [n_pad/32] pc.isenabled in Morton order
  float* msoa = nullptr;         // [6 n_pad] Morton-ordered SoA copy of the cloud (rsc_cull.cu, built on first use)
  void* tiles = nullptr;         // float4 [cull_sphere_count(n_pad)]: spheres of the 128 / 512 / 4096-point tiles of msoa
  bool en_valid = false;         // en_sorted matches the cloud's enabled mask
  rsc::DevBuf selbuf;            // rank/select index over en_sorted
  bool sel_valid = false;
  double lo[3] = {0, 0, 0}, w[3] = {1, 1, 1};  // bounding box used for the quantisation
};

struct rsc_cloud {
  rsc_ctx* ctx = nullptr;
  int64_t n = 0, n_pad = 0;
  int64_t global_offset = 0, n_global = 0;
  int64_t range_lo = 0, range_hi = 0;  // this rank's point range of a replicated cloud
  bool range_set = false;              // false: the whole cloud; true with lo == hi: an empty rank (joins every all-reduce with zeros)
  float* soa = nullptr;        // 6 * n_pad floats: x | y | z | nx | ny | nz
  uint32_t* enabled = nullptr; // n_pad/32 words
  uint32_t* valid = nullptr;
  // exact clouds only (rsc_cloud_create_f64_exact): the caller's float64 coordinates in the caller's AoS layout [3 n];
  // every float64 decision and fit reads them, the float32 SoA above is their rounding
  double* xyz64 = nullptr;
  double* nrm64 = nullptr;
  bool exact() const { return xyz64 != nullptr; }
  float pmax = 0.f;            // max |p| over the cloud (guard-band scale)
  float nmax = 1.f;            // max |n| over the cloud
  // chunked upload in flight: chunk i is usable once chunk_ev[i] has fired on the copy stream
  bool pending = false;
  int64_t chunk_pts = 0;
  int64_t chunk_first = 0;  // the first chunk is smaller: whatever follows the upload can start sooner
  std::vector<cudaEvent_t> chunk_ev;
  int n_chunks() const { return n <= chunk_first ? 1 : 1 + (int)((n - chunk_first + chunk_pts - 1) / chunk_pts); }
  int64_t chunk_begin(int i) const { return i == 0 ? 0 : std::min<int64_t>(n, chunk_first + (int64_t)(i - 1) * chunk_pts); }
  uint32_t* d_bounds = nullptr;  // per chunk: max |p|^2, max |n|^2 (float bits); last pair = whole cloud
  std::vector<rsc_subset> subsets;
  // rank/select index over `enabled` for the sampler (rsc_fit.cu); rebuilt lazily after any change
  rsc::DevBuf selbuf;
  bool sel_valid = false;
  // sharded storage (rsc_cloud_create_shard with n_global > n): isenabled of the WHOLE cloud, replicated on
  // every rank (1 bit/point) so that all ranks draw the same minimal sets; kept equal by all-reducing
  // the cleared words after every extraction.  g_words is a multiple of 16 (512 points).
  uint32_t* g_enabled = nullptr;
  int64_t g_words = 0;
  bool is_shard() const { return g_enabled != nullptr; }
  rsc_cells cells;
  // every change of `enabled` goes through here: the cached sampler indices are rebuilt lazily
  void enabled_changed() {
    sel_valid = false;
    cells.en_valid = false;
    cells.sel_valid = false;
  }
};

namespace rsc {

int32_t cells_refresh_enabled(rsc_cloud* cloud, cudaStream_t st);
void cells_release(rsc_cloud* cloud);

inline PointSet view_cloud(const rsc_cloud* c) {
  PointSet ps;
  ps.x = c->soa;
  ps.y = c->soa + c->n_pad;
  ps.z = c->soa + 2 * c->n_pad;
  ps.nx = c->soa + 3 * c->n_pad;
  ps.ny = c->soa + 4 * c->n_pad;
  ps.nz = c->soa + 5 * c->n_pad;
  ps.enabled = c->enabled;
  ps.valid = c->valid;
  ps.n = c->n;
  ps.n_pad = c->n_pad;
  ps.xyz64 = c->xyz64;
  ps.nrm64 = c->nrm64;
  return ps;
}

inline PointSet view_subset(const rsc_subset* s) {
  PointSet ps;
  ps.x = s->soa;
  ps.y = s->soa + s->m_pad;
  ps.z = s->soa + 2 * s->m_pad;
  ps.nx = s->soa + 3 * s->m_pad;
  ps.ny = s->soa + 4 * s->m_pad;
  ps.nz = s->soa + 5 * s->m_pad;
  ps.enabled = s->enabled;
  ps.valid = s->valid;
  ps.n = s->m;
  ps.n_pad = s->m_pad;
  ps.xyz64 = s->xyz64;
  ps.nrm64 = s->nrm64;
  if (s->xyz64) ps.map = s->idx;
  return ps;
}

// the subset's Morton-ordered view (subset_cull_view), as the culled scorer reads it: no valid words (the first m
// points are the real ones)
inline PointSet view_subset_morton(const rsc_subset* s) {
  PointSet ps;
  ps.x = s->csoa, ps.y = s->csoa + s->m_pad, ps.z = s->csoa + 2 * s->m_pad;
  ps.nx = s->csoa + 3 * s->m_pad, ps.ny = s->csoa + 4 * s->m_pad, ps.nz = s->csoa + 5 * s->m_pad;
  ps.enabled = s->cen, ps.valid = nullptr;
  ps.n = s->m, ps.n_pad = s->m_pad;
  ps.xyz64 = s->xyz64, ps.nrm64 = s->nrm64, ps.map = s->cidx;
  return ps;
}

// error plumbing
int32_t fail(rsc_ctx* ctx, int32_t code, const char* what);
int32_t fail_cuda(rsc_ctx* ctx, cudaError_t e, const char* where);

#define RSC_CUDA(ctx, expr)                                        \
  do {                                                             \
    cudaError_t _e = (expr);                                       \
    if (_e != cudaSuccess) return rsc::fail_cuda((ctx), _e, #expr); \
  } while (0)

Thresh make_thresh(const rsc_params* p);

// internal launchers (all enqueue on `st`, none synchronise)
int32_t score_enqueue(rsc_ctx* ctx, const rsc_cloud* cloud, const PointSet& ps, const Thresh& th,
                      const rsc_cand* d_cands, int32_t C, int32_t* d_counts_policy, bool want_masks,
                      cudaStream_t st, int32_t* d_counts_valid = nullptr,
                      int32_t* d_counts_enabled = nullptr, const double* d_trig = nullptr,
                      const uint32_t* d_bounds = nullptr, bool accumulate = false);
// K2 for small candidate batches (rsc_small.cu): thread = point, candidates from shared memory, FP64 decisions
// inline; the candidate count may live on the device (d_count), c_cap bounds it.  Zeroes d_cv / d_ce [c_cap].
int32_t score_small_enqueue(rsc_ctx* ctx, const rsc_cloud* cloud, const PointSet& ps, const Thresh& th, const rsc_cand* d_cands,
                            int32_t c_cap, const unsigned long long* d_count, int32_t* d_cv, int32_t* d_ce, cudaStream_t st);
int32_t audit_margins(rsc_ctx* ctx, const rsc_cloud* cloud, const PointSet& ps, const Thresh& th, const rsc_cand* d_cands, int32_t C,
                      int64_t p0, int64_t np, float* d_out, float* d_rec, int32_t* d_cols, unsigned long long* d_diffs, cudaStream_t st);
// waits for a chunked upload to land and finalises the cloud's guard-band scales
int32_t cloud_ready(rsc_cloud* cloud);
// refresh the gathered enabled bits of every uploaded subset from the cloud's enabled mask
int32_t refresh_subsets_enabled(rsc_cloud* cloud, cudaStream_t st);
// culled scorer (rsc_cull.cu) and the Morton view of a subset it runs on (rsc_octree.cu)
int32_t subset_cull_view(rsc_cloud* cloud, rsc_subset& s, cudaStream_t st);
size_t cull_sphere_count(int64_t n_pad);  // float4 entries cull_tile_spheres writes (tiles, groups, blocks)
// (d_n, nullable: the number of real points lives on the device, at most ps.n -- the spheres leave the rest out)
int32_t cull_tile_spheres(rsc_ctx* ctx, const PointSet& ps, float4* tiles, cudaStream_t st, const unsigned long long* d_n = nullptr);
int32_t cull_enqueue(rsc_ctx* ctx, const rsc_cloud* cloud, const PointSet& ps, const float4* tiles, const Thresh& th,
                     const rsc_cand* d_cands, int C_cap, const int32_t* d_C, int32_t* cv, int32_t* ce, unsigned long long* d_stats,
                     cudaStream_t st);
// K2 of the loops for `n_new` new candidates on a subset (or this rank's slice `ps` of it): the culled scorer on
// the subset's Morton view when the slice is the whole subset and the batch is large enough to pay, else the dense
// tiled kernel.  *d_ovf (device, optional) receives the dense path's guard-band queue overflow flag (0 when culled).
int32_t loop_score_new(rsc_ctx* ctx, rsc_cloud* cloud, rsc_subset& sub, const PointSet& ps, bool whole_subset, const Thresh& th,
                       const rsc_cand* d_cands, int n_new, int32_t* cv, int32_t* ce, int32_t* d_ovf, cudaStream_t st);

// group-major masks of the last score_enqueue(want_masks) -> candidate-major [C][ceil(m/32)] (d_out, or ctx->masks_cm)
int32_t masks_to_candidate_major(rsc_ctx* ctx, int32_t C, int64_t m, cudaStream_t st, uint32_t* d_out = nullptr);

}  // namespace rsc

namespace rsc {
// scratch of one sample/fit batch inside ctx->fitbuf (rsc_fit.cu)
struct FitScratch {
  rsc_cand* dense;
  rsc_cand* out;
  uint32_t* okmask;  // ballot word per (group of 128 sets, type, warp): which sets gave a candidate
  uint32_t* base;    // per group: candidates before it
  unsigned long long* total;
  int32_t* out_set;
  int64_t* idx;
  int32_t* level;  // per set: octree level its cell came from (cell sampler only)
  float* gath;     // sharded storage: [S][k][6] coordinates + normals of the drawn points, gathered from their owners
};
// a validated fit order of built-in kinds and compiled user types (rsc_shape_slot[], make_fit_order in rsc_user.cu)
struct FitOrder {
  int n = 0;
  bool has_user = false;
  int32_t type[RSC_MAX_ORDER];
  int32_t nk[RSC_MAX_ORDER];
  double k[RSC_MAX_ORDER][8];
};
// order: nullptr = params->shape_types (built-ins); else the mixed order, whose user positions are fitted by their
// compiled rsc_user_fit_kernel into the same dense slots / ballot words
int32_t fit_enqueue(rsc_ctx* ctx, rsc_cloud* cloud, int mode, const rsc_params* params, int k, const double* dP,
                    const double* dN, const int64_t* d_idx, int S, uint64_t seed, uint64_t set0, cudaStream_t st,
                    FitScratch* fs, const double* cum = nullptr, int32_t* d_seg = nullptr, int sets_per_iter = 0, int nb = 0,
                    const FitOrder* order = nullptr);
// user shapes of a fit order (rsc_user.cu).  RSC_E_ARG (reason in rsc_last_error) for a duplicate or unknown type,
// a user type without a compiled fit, norder outside 0..RSC_MAX_ORDER or nk outside 0..8
int32_t make_fit_order(rsc_ctx* ctx, const rsc_shape_slot* order, int32_t norder, FitOrder* fo, const char* who);
// K1: the fit kernel of user position `pos` over the S sets of `idx` (cloud coordinates)
int32_t user_fit_enqueue(rsc_ctx* ctx, const FitOrder& fo, int pos, const rsc_cloud* cloud, const int64_t* idx, int S, int np,
                         rsc_cand* dense, uint32_t* okmask, cudaStream_t st);
// K2 / K5: for every user type of the order, ADD the counts of its records among d_cands[0..min(*d_count, c_cap))
// (d_count nullable: c_cap candidates) on `ps` to ce (and cv, nullable); other records are left as they are
int32_t user_score_enqueue(rsc_ctx* ctx, const FitOrder& fo, const PointSet& ps, const rsc_cand* d_cands, int c_cap,
                           const unsigned long long* d_count, int32_t* cv, int32_t* ce, cudaStream_t st);
// K4 for a user candidate: the inlier-mask words + their count / scan (what refit_mask_enqueue does for a built-in)
int32_t user_refit_mask_enqueue(rsc_cloud* cloud, const FitOrder& fo, const rsc_cand& cand, cudaStream_t st);
int64_t count_mask_bits(rsc_ctx* ctx, const uint32_t* words, int64_t nwords);
// device -> (pageable) host through page-locked staging and worker threads; synchronises `st`
int32_t staged_d2h(rsc_ctx* ctx, void* h_dst, const void* d_src, size_t bytes, cudaStream_t st);
// sharded storage: (re)build the replicated whole-cloud enabled mask from the ranks' local masks (collective)
int32_t shard_sync_enabled(rsc_cloud* cloud, cudaStream_t st);
// sharded storage, after an extraction: clear the bits of the ranks' local inlier-mask words `inl_local`
// (n_pad/32 words) in the replicated mask; the int32 behind the words carries `extra` values summed over
// the ranks too (returned in d_extra_out[0..n_extra), device) -- collective
int32_t shard_clear_enabled(rsc_cloud* cloud, const uint32_t* inl_local, const int32_t* d_extra_in, int n_extra,
                            int32_t* d_extra_out, cudaStream_t st);
void loop_scratch_free(rsc_ctx* ctx);
int32_t fit_reserve(rsc_ctx* ctx, const rsc_params* params, int S, int ntypes = -1);
// exclusive scan of n uint32 counts into 64-bit offsets (+ total) on `st` (rsc_fit.cu)
int32_t scan_u32(rsc_ctx* ctx, const uint32_t* counts, int n, unsigned long long* offsets, unsigned long long* total,
                 cudaStream_t st);
// timed_reps > 1 (measurement only): the mask kernel runs that many times back to back between the evr0/evr1
// events before the real pass, so that its duration is not an event pair around one ~70 us launch
int32_t refit_mask_enqueue(rsc_cloud* cloud, const Thresh& th, const rsc_cand& cand, cudaStream_t st, int timed_reps = 1);
int32_t refit_write_enqueue(rsc_cloud* cloud, int64_t* d_out, bool disable, cudaStream_t st);
int32_t refit_mask_from_list(rsc_cloud* cloud, const int64_t* d_list, int64_t n, cudaStream_t st);
// for a mask written by another kernel (user shapes, rsc_user.cu): *inl = the n_pad/32 inlier-mask words refit_mask_enqueue
// would write; refit_scan_enqueue then counts and scans them for refit_write_enqueue (total in ctx->misc2[0])
int32_t refit_mask_buffer(rsc_cloud* cloud, uint32_t** inl);
int32_t refit_scan_enqueue(rsc_cloud* cloud, cudaStream_t st);
// unloads the user-shape programs of a context (rsc_ctx_destroy)
void user_shapes_free(rsc_ctx* ctx);
// parameter-space bitmap filter (rsc_bitmap.cu): the points of d_idx whose cell lies in the largest connected
// component -> d_out (capacity n); synchronises `st`
int32_t bitmap_filter_dev(rsc_cloud* cloud, const rsc_cand& cand, double beta, bool eight, const int64_t* d_idx, int64_t n,
                          int64_t* d_out, int64_t* out_n, int32_t* info, cudaStream_t st);
// least-squares refit of *cand in place (rsc_lsq.cu); synchronises `st`
int32_t lsq_refine(rsc_cloud* cloud, const rsc_params* params, double band, rsc_cand* cand, int64_t* n_used, double* rms,
                   cudaStream_t st);
}  // namespace rsc
