// rsc_small.cu -- K2 for SMALL candidate batches (the device loop's per-batch scoring and K5).
//
// The tiled scorer (rsc_score.cu) keeps candidates in registers and streams points past them: at
// 4096 candidates it runs at the FP32-issue limit, but the device loop scores a few dozen new
// candidates per batch of iterations (config c4: ~60), and at that size the tiled path is all fixed
// cost -- a one-CTA candidate compiler, a 128-slot column that is mostly padding, two fix-up launches,
// and a launch shape the HOST must size from the candidate count, which costs a synchronisation.
// Here the mapping is transposed: a thread owns a POINT, the CTA walks the candidates, whose compiled
// FP32 records sit in shared memory and are read as broadcasts; the inlier bits of a (candidate,
// 32 points) group are one warp ballot + POPC into a shared-memory counter.  Pairs inside the FP32
// guard band are decided on the spot in FP64 in the reference's operation order (rsc_exact.cuh), so
// there are no queues, no overflow, no repeat.  The candidate COUNT is read from device memory
// (the fit kernel's compaction total), so nothing has to come back to the host before the launch.
// Same FP32 forms, same bands, same FP64 decisions as the tiled path: identical counts.
#include "rsc_eval.cuh"
#include "rsc_exact.cuh"

namespace rsc {

constexpr int kSmallThreads = 256;
constexpr int kSmallTile = 128;  // candidates staged in shared memory per pass

struct SmallArgs {
  PointSet ps;
  Thresh th;
  const rsc_cand* cands;
  const unsigned long long* d_count;  // nullable: number of candidates on the device
  int c_host;                         // number of candidates (capacity when d_count is given)
  float* rec;                         // [c_host][kRecFields]
  int32_t* cols;                      // [c_host] column type
  int32_t* cv;                        // [c_host] compatible real points
  int32_t* ce;                        // [c_host] compatible enabled points
  float pmax, nmax;
};

__device__ __forceinline__ int small_count(const SmallArgs& a) {
  if (!a.d_count) return a.c_host;
  const unsigned long long n = *a.d_count;
  return n < (unsigned long long)a.c_host ? (int)n : a.c_host;
}

__global__ void small_compile_kernel(const __grid_constant__ SmallArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= small_count(a)) return;
  const rsc_cand c = a.cands[i];
  const int col = (c.type < 0 || c.type >= RSC_NTYPES) ? -1 : col_type(c);
  float r[kRecFields];
  if (col >= 0) {
    compile_record(c, col, a.th, a.pmax, a.nmax, r);
  } else {
    for (int f = 0; f < kRecFields; ++f) r[f] = 0.f;
  }
#pragma unroll
  for (int f = 0; f < kRecFields; ++f) a.rec[(size_t)i * kRecFields + f] = r[f];
  a.cols[i] = col;
}

// the rare path, out of line so that it does not cost the streaming loop registers
__device__ __noinline__ bool small_exact(const rsc_cand* c, const Thresh& th, const PointSet& ps, int64_t p) {
  ex::ConeTrig tr{1.0, 0.0};
  if (c->type == RSC_CONE) {
    tr.ct = cos(-c->p[6] / 2);
    tr.st = sin(-c->p[6] / 2);
  }
  ex::V3 P, N;
  ex::point64(ps, p, &P, &N);
  return ex::compat(*c, tr, th, P, N);
}

__global__ void __launch_bounds__(kSmallThreads) small_score_kernel(const __grid_constant__ SmallArgs a) {
  __shared__ __align__(16) float srec[kSmallTile][kRecFields];
  __shared__ int scol[kSmallTile];
  __shared__ int sce[kSmallTile], scv[kSmallTile];
  const int C = small_count(a);
  const int lane = threadIdx.x & 31;
  const int64_t ntiles = a.ps.n_pad / kSmallThreads;  // n_pad is a multiple of 512
  // the candidate chunks are spread over gridDim.y (K5: a large store against few points would otherwise be one long
  // serial walk in a handful of CTAs)
  for (int c0 = blockIdx.y * kSmallTile; c0 < C; c0 += gridDim.y * kSmallTile) {
    const int ct = min(kSmallTile, C - c0);
    for (int i = threadIdx.x; i < ct * kRecFields; i += kSmallThreads) (&srec[0][0])[i] = a.rec[(size_t)c0 * kRecFields + i];
    for (int i = threadIdx.x; i < ct; i += kSmallThreads) {
      scol[i] = a.cols[c0 + i];
      sce[i] = 0;
      scv[i] = 0;
    }
    __syncthreads();
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
      const int64_t p = t * kSmallThreads + threadIdx.x;
      const uint32_t wen = __ldg(a.ps.enabled + (p >> 5)), wva = __ldg(a.ps.valid + (p >> 5));
      if (wva == 0u) continue;  // a whole group of padding (warp-uniform)
      const bool en = (wen >> lane) & 1u, va = (wva >> lane) & 1u;
      const float px = __ldg(a.ps.x + p), py = __ldg(a.ps.y + p), pz = __ldg(a.ps.z + p);
      const float nx = __ldg(a.ps.nx + p), ny = __ldg(a.ps.ny + p), nz = __ldg(a.ps.nz + p);
      for (int c = 0; c < ct; ++c) {
        const int col = scol[c];
        if (col < 0) continue;
        float r[kRecFields];
        const float4* rp = reinterpret_cast<const float4*>(srec[c]);
        const float4 r0 = rp[0], r1 = rp[1], r2 = rp[2];
        r[0] = r0.x, r[1] = r0.y, r[2] = r0.z, r[3] = r0.w, r[4] = r1.x, r[5] = r1.y, r[6] = r1.z, r[7] = r1.w;
        r[8] = r2.x, r[9] = r2.y, r[10] = r2.z, r[11] = r2.w;
        const int pt = public_type(col);
        const float m = eval_any(col, r, px, py, pz, nx, ny, nz, a.th.eps[pt], a.th.cosa[pt]);
        bool ok = m < 0.f;
        if (va && !(fabsf(m) > r[kBandField])) ok = small_exact(a.cands + c0 + c, a.th, a.ps, p);
        const unsigned be = __ballot_sync(0xffffffffu, ok && en);
        const unsigned bv = __ballot_sync(0xffffffffu, ok && va);
        if (lane == 0) {
          if (be) atomicAdd(&sce[c], __popc(be));
          if (bv) atomicAdd(&scv[c], __popc(bv));
        }
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < ct; i += kSmallThreads) {
      if (sce[i]) atomicAdd(a.ce + c0 + i, sce[i]);
      if (scv[i]) atomicAdd(a.cv + c0 + i, scv[i]);
    }
    __syncthreads();
  }
}

// d_cv / d_ce [c_cap] are zeroed here.  d_count (nullable) = the number of candidates, on the device.
int32_t score_small_enqueue(rsc_ctx* ctx, const rsc_cloud* cloud, const PointSet& ps, const Thresh& th, const rsc_cand* d_cands,
                            int32_t c_cap, const unsigned long long* d_count, int32_t* d_cv, int32_t* d_ce, cudaStream_t st) {
  if (c_cap <= 0) return RSC_OK;
  RSC_CUDA(ctx, cudaMemsetAsync(d_cv, 0, (size_t)c_cap * 4, st));
  RSC_CUDA(ctx, cudaMemsetAsync(d_ce, 0, (size_t)c_cap * 4, st));
  if (ps.n_pad <= 0) return RSC_OK;
  if (cloud->exact() && !ps.xyz64) return fail(ctx, RSC_E_STATE, "score: a point set of an exact cloud lacks its float64 coordinates");
  const size_t o_col = ((size_t)c_cap * kRecFields * 4 + 255) / 256 * 256;
  RSC_CUDA(ctx, ctx->smallbuf.ensure(o_col + (size_t)c_cap * 4));
  SmallArgs a;
  a.ps = ps;
  a.th = th;
  a.th.exact_in = cloud->exact();
  a.cands = d_cands;
  a.d_count = d_count;
  a.c_host = c_cap;
  a.rec = ctx->smallbuf.as<float>();
  a.cols = reinterpret_cast<int32_t*>(ctx->smallbuf.as<char>() + o_col);
  a.cv = d_cv;
  a.ce = d_ce;
  a.pmax = cloud->pmax;
  a.nmax = cloud->nmax;
  small_compile_kernel<<<(c_cap + 127) / 128, 128, 0, st>>>(a);
  RSC_CUDA(ctx, cudaGetLastError());
  const int64_t ntiles = ps.n_pad / kSmallThreads;
  const int gx = (int)std::min<int64_t>(ntiles, (int64_t)ctx->sm_count * 8);
  // rows of candidate chunks: as many as there is room for beside the point tiles (a launch sized by a capacity
  // expects a quarter of it, see the device loop)
  const int chunks = ((d_count ? (c_cap + 3) / 4 : c_cap) + kSmallTile - 1) / kSmallTile;
  const int gy = std::max(1, std::min(chunks, ctx->sm_count * 16 / gx));
  small_score_kernel<<<dim3((unsigned)gx, (unsigned)gy), kSmallThreads, 0, st>>>(a);
  RSC_CUDA(ctx, cudaGetLastError());
  ctx->stats.score_launches += 1;
  return RSC_OK;
}

}  // namespace rsc
