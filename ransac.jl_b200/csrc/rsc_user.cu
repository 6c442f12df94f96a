// rsc_user.cu -- user-defined shapes on the device: the plug-in boundary of the reference
// (docs/src/newprimitive.md:12-18) with the candidate x point work in CUDA.
//
// A user shape brings its compatibility test as a short piece of CUDA C (rsc_user_compatible, see
// rsc_user_kernels.cuh).  NVRTC compiles it together with the embedded kernel template for sm_100a with
// --fmad=false and no fast-math; the CUBIN is loaded with cudaLibraryLoadData, so the library links neither
// libnvrtc nor libcuda.  libnvrtc.so.12 is dlopen-ed on first use (like NCCL in rsc_comm.cu): the library loads
// and every built-in entry point works without it.  Programs are cached per context, keyed by the source bytes;
// type ids start at RSC_USER_TYPE0.
//   rsc_user_score          rsc_user_score_kernel: counts (+ masks) over a subset copy or the whole cloud
//   rsc_user_refit_extract  rsc_user_mask_kernel writes K4's inlier-mask words; the count, scan and compaction of
//                           rsc_extract.cu follow (ascending lists, cleared enabled bits, refreshed subset copies)
// A source that also defines rsc_user_fit gets rsc_user_fit_kernel (K1 of the sampler and of the device loop,
// rsc_fit.cu); the device loop (rsc_loop.cu) scores its mixed batches with rsc_user_score_kernel too.
// Sharded and ranged clouds are out of scope (RSC_E_STATE).
#include <dlfcn.h>
#include <nvrtc.h>
#include <string.h>

#include "rsc_common.cuh"
#include "rsc_user_kernels.cuh"

namespace rsc {

static const char kUserTemplate[] =
#include "rsc_user_kernels.inc"
    ;

static_assert(sizeof(RscUserCand) == sizeof(rsc_cand), "RscUserCand mirrors rsc_cand");
static_assert(sizeof(RscUserPoints) == sizeof(PointSet), "RscUserPoints mirrors PointSet");

struct NvrtcApi {
  void* h = nullptr;
  nvrtcResult (*CreateProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
  nvrtcResult (*CompileProgram)(nvrtcProgram, int, const char* const*) = nullptr;
  nvrtcResult (*GetProgramLogSize)(nvrtcProgram, size_t*) = nullptr;
  nvrtcResult (*GetProgramLog)(nvrtcProgram, char*) = nullptr;
  nvrtcResult (*GetCUBINSize)(nvrtcProgram, size_t*) = nullptr;
  nvrtcResult (*GetCUBIN)(nvrtcProgram, char*) = nullptr;
  nvrtcResult (*DestroyProgram)(nvrtcProgram*) = nullptr;
  const char* (*GetErrorString)(nvrtcResult) = nullptr;
  std::string err;
};

static NvrtcApi* nvrtc_api() {
  static NvrtcApi api;
  if (api.h || !api.err.empty()) return &api;
  const char* names[] = {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12"};
  for (const char* n : names)
    if ((api.h = dlopen(n, RTLD_NOW | RTLD_LOCAL))) break;
  if (!api.h) {
    const char* e = dlerror();
    api.err = std::string("cannot load libnvrtc.so.12: ") + (e ? e : "?");
    return &api;
  }
  auto sym = [&](const char* s) {
    void* p = dlsym(api.h, s);
    if (!p && api.err.empty()) api.err = std::string("libnvrtc lacks ") + s;
    return p;
  };
  api.CreateProgram = reinterpret_cast<decltype(api.CreateProgram)>(sym("nvrtcCreateProgram"));
  api.CompileProgram = reinterpret_cast<decltype(api.CompileProgram)>(sym("nvrtcCompileProgram"));
  api.GetProgramLogSize = reinterpret_cast<decltype(api.GetProgramLogSize)>(sym("nvrtcGetProgramLogSize"));
  api.GetProgramLog = reinterpret_cast<decltype(api.GetProgramLog)>(sym("nvrtcGetProgramLog"));
  api.GetCUBINSize = reinterpret_cast<decltype(api.GetCUBINSize)>(sym("nvrtcGetCUBINSize"));
  api.GetCUBIN = reinterpret_cast<decltype(api.GetCUBIN)>(sym("nvrtcGetCUBIN"));
  api.DestroyProgram = reinterpret_cast<decltype(api.DestroyProgram)>(sym("nvrtcDestroyProgram"));
  api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("nvrtcGetErrorString"));
  if (!api.err.empty()) {
    dlclose(api.h);
    api.h = nullptr;
  }
  return &api;
}

// Compiles template + user source to a CUBIN.  Returns RSC_OK, RSC_E_ARG (the source does not compile, or defines
// no rsc_user_compatible) or RSC_E_STATE (NVRTC not available); *log receives NVRTC's log in every case.
// *has_fit (nullable): the source defines rsc_user_fit, and the program holds rsc_user_fit_kernel.
static int32_t user_compile(const char* src, size_t nbytes, std::string* cubin, std::string* log, bool* has_fit = nullptr) {
  log->clear();
  const std::string user(src, nbytes);
  const bool fit = user.find("rsc_user_fit") != std::string::npos;
  if (has_fit) *has_fit = fit;
  if (user.find("rsc_user_compatible") == std::string::npos) {
    *log = "user shape source defines no rsc_user_compatible(const double p[7], int outwards, const double k[8], double x, "
           "double y, double z, double nx, double ny, double nz)";
    return RSC_E_ARG;
  }
  NvrtcApi* a = nvrtc_api();
  if (!a->h) {
    *log = a->err;
    return RSC_E_STATE;
  }
  // the user's lines keep their own numbers in the diagnostics
  const std::string prog = std::string(kUserTemplate) + "\n#line 1 \"rsc_user_shape.cu\"\n" + user + "\n";
  nvrtcProgram p = nullptr;
  nvrtcResult r = a->CreateProgram(&p, prog.c_str(), "rsc_user_shape.cu", 0, nullptr, nullptr);
  if (r != NVRTC_SUCCESS) {
    *log = std::string("nvrtcCreateProgram: ") + a->GetErrorString(r);
    return RSC_E_ARG;
  }
  // IEEE float64 + - * / sqrt, no contraction: a host restatement in the same operation order decides alike
  const char* opts[] = {"--gpu-architecture=sm_100a", "--fmad=false", "--std=c++17", "--ptxas-options=-v", "-DRSC_USER_HAS_FIT"};
  const int nopts = (int)(sizeof(opts) / sizeof(opts[0])) - (fit ? 0 : 1);
  r = a->CompileProgram(p, nopts, opts);
  size_t ls = 0;
  if (a->GetProgramLogSize(p, &ls) == NVRTC_SUCCESS && ls > 1) {
    log->resize(ls);
    a->GetProgramLog(p, &(*log)[0]);
    while (!log->empty() && log->back() == '\0') log->pop_back();
  }
  int32_t rc = RSC_OK;
  size_t cs = 0;
  if (r != NVRTC_SUCCESS || a->GetCUBINSize(p, &cs) != NVRTC_SUCCESS || cs == 0) {
    if (log->empty()) *log = std::string("nvrtcCompileProgram: ") + a->GetErrorString(r);
    rc = RSC_E_ARG;
  } else {
    cubin->resize(cs);
    if (a->GetCUBIN(p, &(*cubin)[0]) != NVRTC_SUCCESS) rc = RSC_E_ARG;
  }
  a->DestroyProgram(&p);
  return rc;
}

struct UserProgram {
  std::string src;
  cudaLibrary_t lib = nullptr;
  cudaKernel_t score = nullptr, mask = nullptr;
  cudaKernel_t fit = nullptr;  // null: the source defines no rsc_user_fit
};

struct UserShapes {
  std::vector<UserProgram> progs;  // type id = RSC_USER_TYPE0 + position
};

static UserShapes* user_shapes(rsc_ctx* ctx) {
  if (!ctx->user_shapes) ctx->user_shapes = new UserShapes();
  return static_cast<UserShapes*>(ctx->user_shapes);
}

static const UserProgram* user_program(rsc_ctx* ctx, int32_t type) {
  if (!ctx->user_shapes || type < RSC_USER_TYPE0) return nullptr;
  const UserShapes* us = static_cast<const UserShapes*>(ctx->user_shapes);
  const size_t i = (size_t)(type - RSC_USER_TYPE0);
  return i < us->progs.size() ? &us->progs[i] : nullptr;
}

void user_shapes_free(rsc_ctx* ctx) {
  if (!ctx->user_shapes) return;
  UserShapes* us = static_cast<UserShapes*>(ctx->user_shapes);
  for (UserProgram& p : us->progs)
    if (p.lib) cudaLibraryUnload(p.lib);
  delete us;
  ctx->user_shapes = nullptr;
}

static int32_t user_common_checks(rsc_cloud* cloud, const double* k, int32_t nk) {
  rsc_ctx* ctx = cloud->ctx;
  if (nk < 0 || nk > 8 || (nk > 0 && !k)) return fail(ctx, RSC_E_ARG, "user shape: 0 <= nk <= 8 constants");
  if (cloud->is_shard() || cloud->range_set) return fail(ctx, RSC_E_STATE, "user shape: sharded or ranged clouds are not supported");
  return RSC_OK;
}

static PointSet user_pointset(rsc_cloud* cloud, int32_t subset_id) {
  return subset_id < 0 ? view_cloud(cloud) : view_subset(&cloud->subsets[subset_id]);
}

static RscUserPoints to_user_points(const PointSet& ps) {
  RscUserPoints u;
  u.x = ps.x, u.y = ps.y, u.z = ps.z, u.nx = ps.nx, u.ny = ps.ny, u.nz = ps.nz;
  u.enabled = ps.enabled, u.valid = ps.valid, u.n = ps.n, u.n_pad = ps.n_pad;
  u.xyz64 = ps.xyz64, u.nrm64 = ps.nrm64, u.map = reinterpret_cast<const long long*>(ps.map);
  return u;
}

int32_t make_fit_order(rsc_ctx* ctx, const rsc_shape_slot* order, int32_t norder, FitOrder* fo, const char* who) {
  const std::string w(who);
  if (norder < 0 || norder > RSC_MAX_ORDER || (norder > 0 && !order)) return fail(ctx, RSC_E_ARG, (w + ": 0 <= norder <= 8").c_str());
  fo->n = norder;
  fo->has_user = false;
  for (int i = 0; i < norder; ++i) {
    const rsc_shape_slot& sl = order[i];
    for (int j = 0; j < i; ++j)
      if (order[j].type == sl.type) return fail(ctx, RSC_E_ARG, (w + ": a type appears twice in the fit order").c_str());
    fo->type[i] = sl.type;
    fo->nk[i] = 0;
    for (int q = 0; q < 8; ++q) fo->k[i][q] = 0.0;
    if (sl.type >= 0 && sl.type < RSC_NTYPES) continue;  // built-in: eps / alpha come from rsc_params
    const UserProgram* prog = user_program(ctx, sl.type);
    if (!prog) return fail(ctx, RSC_E_ARG, (w + ": type " + std::to_string(sl.type) + " is neither built-in nor a compiled user shape of this context").c_str());
    if (!prog->fit) return fail(ctx, RSC_E_ARG, (w + ": user type " + std::to_string(sl.type) + " has no rsc_user_fit").c_str());
    if (sl.nk < 0 || sl.nk > 8) return fail(ctx, RSC_E_ARG, (w + ": 0 <= nk <= 8 constants").c_str());
    fo->nk[i] = sl.nk;
    for (int q = 0; q < sl.nk; ++q) fo->k[i][q] = sl.k[q];
    fo->has_user = true;
  }
  return RSC_OK;
}

int32_t user_fit_enqueue(rsc_ctx* ctx, const FitOrder& fo, int pos, const rsc_cloud* cloud, const int64_t* idx, int S, int np,
                         rsc_cand* dense, uint32_t* okmask, cudaStream_t st) {
  const UserProgram* prog = user_program(ctx, fo.type[pos]);
  if (!prog || !prog->fit) return fail(ctx, RSC_E_ARG, "fit: user type without a compiled rsc_user_fit");
  if (S <= 0) return RSC_OK;
  RscUserFitArgs a;
  memset(&a, 0, sizeof(a));
  a.soa = cloud->soa;
  a.n_pad = cloud->n_pad;
  a.xyz64 = cloud->xyz64;
  a.nrm64 = cloud->nrm64;
  a.idx = reinterpret_cast<const long long*>(idx);
  a.S = S, a.np = np, a.npos = fo.n, a.pos = pos, a.type = fo.type[pos], a.nk = fo.nk[pos];
  for (int q = 0; q < 8; ++q) a.k[q] = fo.k[pos][q];
  a.dense = reinterpret_cast<RscUserCand*>(dense);
  a.okmask = okmask;
  void* args[] = {&a};
  RSC_CUDA(ctx, cudaLaunchKernel((const void*)prog->fit, dim3((unsigned)((S + 127) / 128)), dim3(128), args, 0, st));
  return RSC_OK;
}

int32_t user_score_enqueue(rsc_ctx* ctx, const FitOrder& fo, const PointSet& ps, const rsc_cand* d_cands, int c_cap,
                           const unsigned long long* d_count, int32_t* cv, int32_t* ce, cudaStream_t st) {
  const int64_t ntiles = ps.n_pad / RSC_USER_THREADS;
  if (c_cap <= 0 || ntiles <= 0) return RSC_OK;
  for (int t = 0; t < fo.n; ++t) {
    if (fo.type[t] < RSC_NTYPES) continue;
    const UserProgram* prog = user_program(ctx, fo.type[t]);
    if (!prog) return fail(ctx, RSC_E_ARG, "score: user type is not compiled on this context");
    RscUserScoreArgs a;
    memset(&a, 0, sizeof(a));
    a.ps = to_user_points(ps);
    a.cands = reinterpret_cast<const RscUserCand*>(d_cands);
    a.C = c_cap;
    a.nk = fo.nk[t];
    for (int q = 0; q < 8; ++q) a.k[q] = fo.k[t][q];
    a.counts = ce;
    a.counts2 = cv;
    a.d_count = d_count;
    a.type = fo.type[t];
    const int gx = (int)std::min<int64_t>(ntiles, (int64_t)ctx->sm_count * 8);
    // (a launch sized by a capacity expects a quarter of it, like the small-batch scorer's)
    const int chunks = ((d_count ? (c_cap + 3) / 4 : c_cap) + RSC_USER_TILE - 1) / RSC_USER_TILE;
    const int gy = std::max(1, std::min(chunks, ctx->sm_count * 16 / gx));
    void* args[] = {&a};
    RSC_CUDA(ctx, cudaLaunchKernel((const void*)prog->score, dim3((unsigned)gx, (unsigned)gy), dim3(RSC_USER_THREADS), args, 0, st));
    ctx->stats.score_launches += 1;
  }
  return RSC_OK;
}

int32_t user_refit_mask_enqueue(rsc_cloud* cloud, const FitOrder& fo, const rsc_cand& cand, cudaStream_t st) {
  rsc_ctx* ctx = cloud->ctx;
  int pos = -1;
  for (int t = 0; t < fo.n; ++t)
    if (fo.type[t] == cand.type) pos = t;
  const UserProgram* prog = user_program(ctx, cand.type);
  if (pos < 0 || !prog) return fail(ctx, RSC_E_ARG, "refit: user type is not part of the fit order");
  uint32_t* inl = nullptr;
  if (int32_t rc = refit_mask_buffer(cloud, &inl)) return rc;
  RscUserMaskArgs a;
  memset(&a, 0, sizeof(a));
  a.ps = to_user_points(view_cloud(cloud));
  memcpy(&a.cand, &cand, sizeof(rsc_cand));
  a.nk = fo.nk[pos];
  for (int q = 0; q < 8; ++q) a.k[q] = fo.k[pos][q];
  a.inl = inl;
  const int64_t nblk = cloud->n_pad / RSC_USER_THREADS;
  if (nblk > 0) {
    const unsigned grid = (unsigned)std::min<int64_t>(nblk, (int64_t)ctx->sm_count * 16);
    void* args[] = {&a};
    RSC_CUDA(ctx, cudaLaunchKernel((const void*)prog->mask, dim3(grid), dim3(RSC_USER_THREADS), args, 0, st));
  }
  ctx->stats.evals += cloud->n;
  return refit_scan_enqueue(cloud, st);
}

}  // namespace rsc

using namespace rsc;

extern "C" {

int32_t rsc_user_shape_check(const void* src, int64_t nbytes, void* log, int64_t log_cap) {
  if (!src || nbytes <= 0) return RSC_E_ARG;
  std::string cubin, msg;
  const int32_t rc = user_compile(static_cast<const char*>(src), (size_t)nbytes, &cubin, &msg);
  if (log && log_cap > 0) {
    const size_t n = std::min<size_t>(msg.size(), (size_t)log_cap - 1);
    memcpy(log, msg.data(), n);
    static_cast<char*>(log)[n] = '\0';
  }
  return rc;
}

int32_t rsc_user_shape_compile(rsc_ctx* ctx, const void* src, int64_t nbytes, int32_t* type_id) {
  if (!ctx) return RSC_E_ARG;
  if (!src || nbytes <= 0 || !type_id) return fail(ctx, RSC_E_ARG, "user_shape_compile: null source / type_id");
  UserShapes* us = user_shapes(ctx);
  const std::string key(static_cast<const char*>(src), (size_t)nbytes);
  for (size_t i = 0; i < us->progs.size(); ++i)
    if (us->progs[i].src == key) {
      *type_id = RSC_USER_TYPE0 + (int32_t)i;
      return RSC_OK;
    }
  std::string cubin, log;
  bool has_fit = false;
  const int32_t rc = user_compile(key.data(), key.size(), &cubin, &log, &has_fit);
  if (rc) return fail(ctx, rc, ("user_shape_compile: " + log).c_str());
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  UserProgram p;
  p.src = key;
  RSC_CUDA(ctx, cudaLibraryLoadData(&p.lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0));
  if (cudaLibraryGetKernel(&p.score, p.lib, "rsc_user_score_kernel") != cudaSuccess ||
      cudaLibraryGetKernel(&p.mask, p.lib, "rsc_user_mask_kernel") != cudaSuccess ||
      (has_fit && cudaLibraryGetKernel(&p.fit, p.lib, "rsc_user_fit_kernel") != cudaSuccess)) {
    cudaLibraryUnload(p.lib);
    cudaGetLastError();
    return fail(ctx, RSC_E_CUDA, "user_shape_compile: kernels missing from the compiled program");
  }
  us->progs.push_back(p);
  *type_id = RSC_USER_TYPE0 + (int32_t)(us->progs.size() - 1);
  return RSC_OK;
}

int32_t rsc_user_score(rsc_cloud* cloud, const double* k, int32_t nk, const rsc_cand* cands, int32_t C, int32_t subset_id,
                       int32_t* counts, uint32_t* masks) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (C < 0 || (C > 0 && (!cands || !counts))) return fail(ctx, RSC_E_ARG, "user_score: null candidates/counts");
  int32_t rc = user_common_checks(cloud, k, nk);
  if (rc) return rc;
  if (C == 0) return RSC_OK;
  const UserProgram* prog = user_program(ctx, cands[0].type);
  if (!prog) return fail(ctx, RSC_E_ARG, "user_score: candidate type is not a compiled user shape of this context");
  for (int i = 1; i < C; ++i)
    if (cands[i].type != cands[0].type) return fail(ctx, RSC_E_ARG, "user_score: all candidates must have the same type");
  if (subset_id >= 0 && ((size_t)subset_id >= cloud->subsets.size() || !cloud->subsets[subset_id].soa))
    return fail(ctx, RSC_E_STATE, "user_score: subset not uploaded (rsc_cloud_set_subset)");
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if ((rc = cloud_ready(cloud))) return rc;
  const PointSet ps = user_pointset(cloud, subset_id);
  cudaStream_t st = ctx->stream;
  const int64_t words = (ps.n + 31) / 32;
  RSC_CUDA(ctx, ctx->cands.ensure((size_t)C * sizeof(rsc_cand)));
  RSC_CUDA(ctx, ctx->counts.ensure((size_t)C * sizeof(int32_t)));
  if (masks) RSC_CUDA(ctx, ctx->masks_cm.ensure((size_t)C * words * 4 + 4));
  RSC_CUDA(ctx, cudaMemcpyAsync(ctx->cands.p, cands, (size_t)C * sizeof(rsc_cand), cudaMemcpyHostToDevice, st));
  RSC_CUDA(ctx, cudaMemsetAsync(ctx->counts.p, 0, (size_t)C * sizeof(int32_t), st));
  if (masks) RSC_CUDA(ctx, cudaMemsetAsync(ctx->masks_cm.p, 0, (size_t)C * words * 4, st));
  RscUserScoreArgs a;
  memset(&a, 0, sizeof(a));
  a.ps = to_user_points(ps);
  a.cands = ctx->cands.as<RscUserCand>();
  a.C = C;
  a.type = cands[0].type;
  a.nk = nk;
  for (int i = 0; i < nk; ++i) a.k[i] = k[i];
  a.counts = ctx->counts.as<int32_t>();
  a.masks = masks ? ctx->masks_cm.as<uint32_t>() : nullptr;
  a.words = words;
  RSC_CUDA(ctx, cudaEventRecord(ctx->ev0, st));
  const int64_t ntiles = ps.n_pad / RSC_USER_THREADS;
  if (ntiles > 0) {
    const int gx = (int)std::min<int64_t>(ntiles, (int64_t)ctx->sm_count * 8);
    const int chunks = (C + RSC_USER_TILE - 1) / RSC_USER_TILE;
    const int gy = std::max(1, std::min(chunks, ctx->sm_count * 16 / gx));
    void* args[] = {&a};
    RSC_CUDA(ctx, cudaLaunchKernel((const void*)prog->score, dim3((unsigned)gx, (unsigned)gy), dim3(RSC_USER_THREADS), args, 0, st));
  }
  RSC_CUDA(ctx, cudaEventRecord(ctx->ev1, st));
  RSC_CUDA(ctx, cudaMemcpyAsync(counts, ctx->counts.p, (size_t)C * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (masks) RSC_CUDA(ctx, cudaMemcpyAsync(masks, ctx->masks_cm.p, (size_t)C * words * 4, cudaMemcpyDeviceToHost, st));
  RSC_CUDA(ctx, cudaStreamSynchronize(st));
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->stats.score_ms = ms;
  ctx->stats.evals += (int64_t)C * ps.n;
  ctx->stats.cands_scored += C;
  ctx->stats.score_launches += 1;
  return RSC_OK;
}

int32_t rsc_user_refit_extract(rsc_cloud* cloud, const double* k, int32_t nk, const rsc_cand* cand, int64_t* out_idx,
                               int64_t* out_n, int32_t disable) {
  if (!cloud) return RSC_E_ARG;
  rsc_ctx* ctx = cloud->ctx;
  if (!cand || !out_n) return fail(ctx, RSC_E_ARG, "user_refit_extract: null candidate/out_n");
  int32_t rc = user_common_checks(cloud, k, nk);
  if (rc) return rc;
  const UserProgram* prog = user_program(ctx, cand->type);
  if (!prog) return fail(ctx, RSC_E_ARG, "user_refit_extract: candidate type is not a compiled user shape of this context");
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if ((rc = cloud_ready(cloud))) return rc;
  cudaStream_t st = ctx->stream;
  uint32_t* inl = nullptr;
  if ((rc = refit_mask_buffer(cloud, &inl))) return rc;
  RscUserMaskArgs a;
  memset(&a, 0, sizeof(a));
  a.ps = to_user_points(view_cloud(cloud));
  memcpy(&a.cand, cand, sizeof(rsc_cand));
  a.nk = nk;
  for (int i = 0; i < nk; ++i) a.k[i] = k[i];
  a.inl = inl;
  RSC_CUDA(ctx, cudaEventRecord(ctx->evr0, st));
  const int64_t nblk = cloud->n_pad / RSC_USER_THREADS;
  if (nblk > 0) {
    const unsigned grid = (unsigned)std::min<int64_t>(nblk, (int64_t)ctx->sm_count * 16);
    void* args[] = {&a};
    RSC_CUDA(ctx, cudaLaunchKernel((const void*)prog->mask, dim3(grid), dim3(RSC_USER_THREADS), args, 0, st));
  }
  RSC_CUDA(ctx, cudaEventRecord(ctx->evr1, st));
  if ((rc = refit_scan_enqueue(cloud, st))) return rc;
  ctx->stats.evals += cloud->n;
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
    if (d_out) RSC_CUDA(ctx, cudaMemcpyAsync(out_idx, d_out, (size_t)total * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    RSC_CUDA(ctx, cudaStreamSynchronize(st));
  }
  return RSC_OK;
}

}  // extern "C"
