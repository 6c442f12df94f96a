// rsc_cloud.cu -- the device-resident RANSACCloud (octree.jl:37-59, constructors :78-138):
// AoS host arrays -> SoA float32 in HBM, the enabled bitmask (BitArray.chunks layout), and the
// gathered contiguous copies of the random subsets (octree.jl:129-135) that scoring streams.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <thread>

#include "rsc_common.cuh"

namespace rsc {

// xyz/nrm: AoS staging of the points [off, off+cnt); soa: the whole cloud's SoA arrays
template <class T>
__global__ void aos_to_soa_kernel(const T* __restrict__ xyz, const T* __restrict__ nrm, int64_t off, int64_t cnt,
                                  int64_t n_pad, float* __restrict__ soa, uint32_t* __restrict__ bounds,
                                  uint32_t* __restrict__ gbounds) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t i = off + j;
  float p2 = 0.f, n2 = 0.f;
  if (j < cnt) {
    const float x = (float)xyz[3 * j], y = (float)xyz[3 * j + 1], z = (float)xyz[3 * j + 2];
    const float a = (float)nrm[3 * j], b = (float)nrm[3 * j + 1], c = (float)nrm[3 * j + 2];
    soa[i] = x;
    soa[n_pad + i] = y;
    soa[2 * n_pad + i] = z;
    soa[3 * n_pad + i] = a;
    soa[4 * n_pad + i] = b;
    soa[5 * n_pad + i] = c;
    p2 = x * x + y * y + z * z;
    n2 = a * a + b * b + c * c;
    if (!(p2 == p2)) p2 = 0.f;  // NaN points do not widen the band
    if (!(n2 == n2)) n2 = 0.f;
  }
#pragma unroll
  for (int d = 16; d; d >>= 1) {
    p2 = fmaxf(p2, __shfl_xor_sync(0xffffffffu, p2, d));
    n2 = fmaxf(n2, __shfl_xor_sync(0xffffffffu, n2, d));
  }
  if ((threadIdx.x & 31) == 0) {  // non-negative floats order like their bit patterns
    atomicMax(bounds, __float_as_uint(p2));
    atomicMax(bounds + 1, __float_as_uint(n2));
    atomicMax(gbounds, __float_as_uint(p2));  // running maximum over the whole cloud
    atomicMax(gbounds + 1, __float_as_uint(n2));
  }
}

__global__ void fill_valid_kernel(uint32_t* __restrict__ valid, uint32_t* __restrict__ enabled,
                                  int64_t n, int64_t words) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= words) return;
  const int64_t lo = w * 32;
  uint32_t v = 0;
  if (lo + 32 <= n)
    v = 0xffffffffu;
  else if (lo < n)
    v = (1u << (n - lo)) - 1u;
  valid[w] = v;
  if (enabled) enabled[w] = v;
}

__global__ void and_words_kernel(uint32_t* __restrict__ dst, const uint32_t* __restrict__ m, int64_t words) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w < words) dst[w] &= m[w];
}

__global__ void gather_subset_kernel(const float* __restrict__ soa, int64_t n_pad, const int64_t* __restrict__ idx,
                                     int64_t m, int64_t m_pad, float* __restrict__ out) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  const int64_t i = idx[j];
#pragma unroll
  for (int f = 0; f < 6; ++f) out[f * m_pad + j] = soa[f * n_pad + i];
}

// one warp per subset word: bit j = enabled[idx[j]]
__global__ void gather_enabled_kernel(const uint32_t* __restrict__ enabled, const int64_t* __restrict__ idx,
                                      int64_t m, int64_t words, uint32_t* __restrict__ out) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool b = false;
  if (j < m) {
    const int64_t i = idx[j];
    b = (enabled[i >> 5] >> (i & 31)) & 1u;
  }
  const unsigned bal = __ballot_sync(0xffffffffu, b);
  if ((threadIdx.x & 31) == 0 && (j >> 5) < words) out[j >> 5] = bal;
}

__global__ void popc_words_kernel(const uint32_t* __restrict__ w, int64_t words, unsigned long long* __restrict__ out) {
  unsigned long long s = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < words; i += (int64_t)gridDim.x * blockDim.x)
    s += __popc(w[i]);
#pragma unroll
  for (int d = 16; d; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
  if ((threadIdx.x & 31) == 0 && s) atomicAdd(out, s);
}

__global__ void andnot_words_kernel(uint32_t* __restrict__ dst, const uint32_t* __restrict__ m, int64_t words) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w < words) dst[w] &= ~m[w];
}

// ---- sharded storage: the replicated whole-cloud enabled mask ---------------------------------------
// Ranges are disjoint and start at multiples of 2048 points, so every rank's local words land in their own
// slots of a zeroed whole-cloud buffer and an int32 sum over the ranks is the union.
static int32_t shard_exchange(rsc_cloud* c, const uint32_t* local_words, const int32_t* d_extra_in, int n_extra, cudaStream_t st,
                              uint32_t** out) {
  rsc_ctx* ctx = c->ctx;
  if (!ctx->allreduce) return fail(ctx, RSC_E_STATE, "sharded storage needs a communicator (rsc_ctx_comm_init or rsc_ctx_set_allreduce)");
  RSC_CUDA(ctx, ctx->shardbuf.ensure((size_t)(c->g_words + n_extra + 4) * 4));
  uint32_t* tmp = ctx->shardbuf.as<uint32_t>();
  RSC_CUDA(ctx, cudaMemsetAsync(tmp, 0, (size_t)(c->g_words + n_extra) * 4, st));
  RSC_CUDA(ctx, cudaMemcpyAsync(tmp + c->global_offset / 32, local_words, (size_t)(c->n_pad / 32) * 4, cudaMemcpyDeviceToDevice, st));
  if (n_extra) RSC_CUDA(ctx, cudaMemcpyAsync(tmp + c->g_words, d_extra_in, (size_t)n_extra * 4, cudaMemcpyDeviceToDevice, st));
  if (ctx->allreduce(ctx->allreduce_user, tmp, c->g_words + n_extra, (void*)st)) return fail(ctx, RSC_E_NCCL, "sharded storage: all-reduce failed");
  *out = tmp;
  return RSC_OK;
}

int32_t shard_sync_enabled(rsc_cloud* c, cudaStream_t st) {
  uint32_t* tmp = nullptr;
  if (int32_t rc = shard_exchange(c, c->enabled, nullptr, 0, st, &tmp)) return rc;
  RSC_CUDA(c->ctx, cudaMemcpyAsync(c->g_enabled, tmp, (size_t)c->g_words * 4, cudaMemcpyDeviceToDevice, st));
  c->enabled_changed();
  return RSC_OK;
}

int32_t shard_clear_enabled(rsc_cloud* c, const uint32_t* inl_local, const int32_t* d_extra_in, int n_extra, int32_t* d_extra_out,
                            cudaStream_t st) {
  uint32_t* tmp = nullptr;
  if (int32_t rc = shard_exchange(c, inl_local, d_extra_in, n_extra, st, &tmp)) return rc;
  andnot_words_kernel<<<(unsigned)((c->g_words + 255) / 256), 256, 0, st>>>(c->g_enabled, tmp, c->g_words);
  RSC_CUDA(c->ctx, cudaGetLastError());
  if (n_extra) RSC_CUDA(c->ctx, cudaMemcpyAsync(d_extra_out, tmp + c->g_words, (size_t)n_extra * 4, cudaMemcpyDeviceToDevice, st));
  c->enabled_changed();
  return RSC_OK;
}

// set bits of a mask (synchronises the context stream); -1 on failure
int64_t count_mask_bits(rsc_ctx* ctx, const uint32_t* words, int64_t nwords) {
  if (ctx->misc.ensure(16) != cudaSuccess) return -1;
  unsigned long long* d = ctx->misc.as<unsigned long long>();
  cudaMemsetAsync(d, 0, 8, ctx->stream);
  popc_words_kernel<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(words, nwords, d);
  unsigned long long h = 0;
  cudaMemcpyAsync(&h, d, 8, cudaMemcpyDeviceToHost, ctx->stream);
  if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return -1;
  return (int64_t)h;
}

int32_t refresh_subsets_enabled(rsc_cloud* cloud, cudaStream_t st) {
  rsc_ctx* ctx = cloud->ctx;
  for (auto& s : cloud->subsets) {
    if (!s.soa) continue;
    const int64_t words = s.m_pad / 32;
    const int64_t threads = words * 32;
    gather_enabled_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(cloud->enabled, s.idx, s.m, words, s.enabled);
    RSC_CUDA(ctx, cudaGetLastError());
    if (s.cen) {  // the Morton view of the culled scorer follows
      gather_enabled_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(cloud->enabled, s.cidx, s.m, words, s.cen);
      RSC_CUDA(ctx, cudaGetLastError());
    }
  }
  return RSC_OK;
}

// Upload granularity.  Through page-locked staging (pageable caller arrays): 2 Mi points (48 MB of float32 AoS), the
// host copy of chunk i + 1 overlaps the DMA of chunk i.  Straight from the caller's page-locked arrays: 4 Mi points --
// rsc_score follows the upload chunk by chunk and every chunk costs it a compile + two fix-up launches (c3 e2e step
// 46.7 ms at 2 Mi / 2 Mi first, 45.7 ms at 4 Mi / 1 Mi first; tools/e2e_first_chunk.sh).  The FIRST chunk is a
// quarter of that: its arrival is pure latency for whatever follows the upload.
static int64_t chunk_points(bool staged) {
  if (const char* e = getenv("RSC_CHUNK_PTS")) return std::max<int64_t>(1 << 16, std::min<int64_t>(16 << 20, atoll(e) / kTile * kTile));
  return staged ? (2 << 20) : (4 << 20);
}

// ---- pageable host memory <-> device through page-locked staging filled by worker threads ----------------
static int host_copy_threads() {
  if (const char* e = getenv("RSC_COPY_THREADS")) return std::max(1, std::min(32, atoi(e)));
  const unsigned hw = std::thread::hardware_concurrency();
  return (int)std::max(1u, std::min(8u, hw / 2));  // c5 upload on a 16-thread host: 2 / 4 / 8 / 12 threads -> 0.17 / 0.11 / 0.08 / 0.085 s
}

static void par_memcpy(void* dst, const void* src, size_t bytes, int nthreads) {
  if (nthreads <= 1 || bytes < ((size_t)4 << 20)) {
    memcpy(dst, src, bytes);
    return;
  }
  const size_t per = (bytes / nthreads + 4095) / 4096 * 4096;
  std::vector<std::thread> th;
  for (int t = 1; t < nthreads; ++t) {
    const size_t off = (size_t)t * per;
    if (off >= bytes) break;
    const size_t len = std::min(per, bytes - off);
    th.emplace_back([=] { memcpy((char*)dst + off, (const char*)src + off, len); });
  }
  memcpy(dst, src, std::min(per, bytes));
  for (auto& x : th) x.join();
}

static bool is_pageable(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return true;
  }
  return at.type == cudaMemoryTypeUnregistered;
}

static int32_t ensure_hstage(rsc_ctx* ctx, size_t bytes) {
  if (ctx->hstage_cap >= bytes) return RSC_OK;
  for (int b = 0; b < 2; ++b) {
    if (ctx->hstage[b]) cudaFreeHost(ctx->hstage[b]);
    ctx->hstage[b] = nullptr;
    if (!ctx->hstage_free[b]) RSC_CUDA(ctx, cudaEventCreateWithFlags(&ctx->hstage_free[b], cudaEventDisableTiming));
  }
  ctx->hstage_cap = 0;
  for (int b = 0; b < 2; ++b) RSC_CUDA(ctx, cudaMallocHost(&ctx->hstage[b], bytes));
  ctx->hstage_cap = bytes;
  return RSC_OK;
}

// device -> pageable host, `bytes` from d_src: DMA into the page-locked staging, worker threads copy out
int32_t staged_d2h(rsc_ctx* ctx, void* h_dst, const void* d_src, size_t bytes, cudaStream_t st) {
  if (bytes == 0) return RSC_OK;
  if (bytes < ((size_t)8 << 20) || !is_pageable(h_dst)) {
    RSC_CUDA(ctx, cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, st));
    RSC_CUDA(ctx, cudaStreamSynchronize(st));
    return RSC_OK;
  }
  const size_t piece = (size_t)32 << 20;
  if (int32_t rc = ensure_hstage(ctx, std::max(piece, ctx->hstage_cap))) return rc;
  const int nt = host_copy_threads();
  const size_t np = (bytes + piece - 1) / piece;
  for (size_t i = 0; i <= np; ++i) {
    if (i < np) {  // DMA piece i into buffer i & 1
      const size_t off = i * piece, len = std::min(piece, bytes - off);
      RSC_CUDA(ctx, cudaMemcpyAsync(ctx->hstage[i & 1], (const char*)d_src + off, len, cudaMemcpyDeviceToHost, st));
      RSC_CUDA(ctx, cudaEventRecord(ctx->hstage_free[i & 1], st));
    }
    if (i > 0) {  // copy piece i - 1 out while piece i is in flight
      const size_t off = (i - 1) * piece, len = std::min(piece, bytes - off);
      RSC_CUDA(ctx, cudaEventSynchronize(ctx->hstage_free[(i - 1) & 1]));
      par_memcpy((char*)h_dst + off, ctx->hstage[(i - 1) & 1], len, nt);
    }
  }
  return RSC_OK;
}

// host AoS -> device SoA into the cloud's existing buffers, in chunks on the copy stream:
// H2D of chunk i+1 overlaps the transposition of chunk i and -- because the call returns as soon as
// everything is enqueued -- whatever scoring the caller launches next (rsc_score walks the chunks
// as their events fire).  Other entry points first wait for the upload (cloud_ready).
template <class T>
static int32_t cloud_upload(rsc_cloud* c, const T* xyz, const T* nrm) {
  rsc_ctx* ctx = c->ctx;
  cudaStream_t cs = ctx->copy_stream;
  const int64_t n = c->n;
  const int64_t words = c->n_pad / 32;
  // pageable caller arrays of a large cloud: worker threads copy each chunk into page-locked staging and the DMA
  // engine takes it from there (cudaMemcpy from pageable memory is a single-threaded staged copy, ~10 GB/s)
  const bool staged = n >= ((int64_t)1 << 20) && !getenv("RSC_NO_STAGED_UPLOAD") && is_pageable(xyz) && is_pageable(nrm);
  const int64_t kChunkPts = chunk_points(staged);
  c->chunk_pts = kChunkPts;
  c->chunk_first = getenv("RSC_FIRST_CHUNK_PTS") ? std::max<int64_t>(kTile, std::min<int64_t>(kChunkPts, atoll(getenv("RSC_FIRST_CHUNK_PTS")) / kTile * kTile))
                                                 : kChunkPts / 4;
  const int nchunks = c->n_chunks();
  // previous work on the compute stream may still read the old coordinates
  RSC_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (!c->d_bounds || (int)c->chunk_ev.size() < nchunks) {
    if (c->d_bounds) cudaFree(c->d_bounds);
    RSC_CUDA(ctx, cudaMalloc(&c->d_bounds, (size_t)(2 * nchunks + 2) * sizeof(uint32_t)));
    while ((int)c->chunk_ev.size() < nchunks) {
      cudaEvent_t e;
      RSC_CUDA(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      c->chunk_ev.push_back(e);
    }
  }
  RSC_CUDA(ctx, cudaMemsetAsync(c->d_bounds, 0, (size_t)(2 * nchunks + 2) * sizeof(uint32_t), cs));
  fill_valid_kernel<<<(unsigned)((words + 255) / 256), 256, 0, cs>>>(c->valid, c->enabled, n, words);
  RSC_CUDA(ctx, cudaGetLastError());
  const size_t cbytes = (size_t)3 * kChunkPts * sizeof(T);
  if (!c->xyz64)
    for (int b = 0; b < 2; ++b) RSC_CUDA(ctx, ctx->stage[b].ensure(2 * cbytes));
  const int nt = staged ? host_copy_threads() : 1;
  if (staged)
    if (int32_t rcs = ensure_hstage(ctx, 2 * cbytes)) return rcs;
  for (int i = 0; i < nchunks; ++i) {
    const int64_t off = c->chunk_begin(i);
    const int64_t cnt = c->chunk_begin(i + 1) - off;
    T* sx = ctx->stage[i & 1].as<T>();
    T* sn = sx + 3 * kChunkPts;
    if constexpr (sizeof(T) == sizeof(double)) {
      if (c->xyz64) {  // exact cloud: the chunk lands in the persistent float64 arrays, the transposition reads it there
        sx = c->xyz64 + 3 * off;
        sn = c->nrm64 + 3 * off;
      }
    }
    if (staged) {
      const size_t half = (size_t)3 * cnt * sizeof(T);
      char* hs = static_cast<char*>(ctx->hstage[i & 1]);
      if (i >= 2) RSC_CUDA(ctx, cudaEventSynchronize(ctx->hstage_free[i & 1]));  // the DMA of chunk i - 2 has left this buffer
      par_memcpy(hs, xyz + 3 * off, half, nt);
      par_memcpy(hs + cbytes, nrm + 3 * off, half, nt);
      RSC_CUDA(ctx, cudaMemcpyAsync(sx, hs, half, cudaMemcpyHostToDevice, cs));
      RSC_CUDA(ctx, cudaMemcpyAsync(sn, hs + cbytes, half, cudaMemcpyHostToDevice, cs));
      RSC_CUDA(ctx, cudaEventRecord(ctx->hstage_free[i & 1], cs));
    } else {
      RSC_CUDA(ctx, cudaMemcpyAsync(sx, xyz + 3 * off, (size_t)3 * cnt * sizeof(T), cudaMemcpyHostToDevice, cs));
      RSC_CUDA(ctx, cudaMemcpyAsync(sn, nrm + 3 * off, (size_t)3 * cnt * sizeof(T), cudaMemcpyHostToDevice, cs));
    }
    // bounds layout: [2i, 2i+1] this chunk, [2*nchunks, 2*nchunks+1] whole cloud
    aos_to_soa_kernel<T><<<(unsigned)((cnt + 255) / 256), 256, 0, cs>>>(sx, sn, off, cnt, c->n_pad, c->soa,
                                                                        c->d_bounds + 2 * i, c->d_bounds + 2 * nchunks);
    RSC_CUDA(ctx, cudaGetLastError());
    RSC_CUDA(ctx, cudaEventRecord(c->chunk_ev[i], cs));
  }
  c->pending = true;
  c->enabled_changed();
  if (c->cells.nlevels) cells_release(c);  // the octree was built for the old coordinates
  return RSC_OK;
}

}  // namespace rsc

namespace rsc {
int32_t cloud_ready(rsc_cloud* c) {
  if (!c || !c->pending) return RSC_OK;
  rsc_ctx* ctx = c->ctx;
  const int nchunks = c->n_chunks();
  uint32_t hb[2];
  RSC_CUDA(ctx, cudaMemcpyAsync(hb, c->d_bounds + 2 * nchunks, sizeof(hb), cudaMemcpyDeviceToHost, ctx->copy_stream));
  RSC_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
  float p2, n2;
  memcpy(&p2, &hb[0], 4);
  memcpy(&n2, &hb[1], 4);
  c->pmax = sqrtf(p2) * 1.000001f;
  c->nmax = sqrtf(n2) * 1.000001f;
  c->pending = false;
  return RSC_OK;
}

template <class T>
static int32_t cloud_create_impl(rsc_ctx* ctx, const T* xyz, const T* nrm, int64_t n, int64_t global_offset,
                                 int64_t n_global, rsc_cloud** out, bool exact = false) {
  if (!ctx || !out) return RSC_E_ARG;
  *out = nullptr;
  if (!xyz || !nrm || n <= 0) return fail(ctx, RSC_E_ARG, "cloud_create: empty cloud or null arrays");
  if (n >= ((int64_t)1 << 32) - kTile) return fail(ctx, RSC_E_ARG, "cloud_create: shard too large (>= 2^32 points)");
  const bool shard = n_global > n;
  if (shard && (global_offset % 2048 || (n % 2048 && global_offset + n != n_global)))
    return fail(ctx, RSC_E_ARG, "cloud_create_shard: a range must start at a multiple of 2048 points and hold a multiple of 2048 points unless it ends the cloud");
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  rsc_cloud* c = new rsc_cloud();
  c->ctx = ctx;
  c->n = n;
  c->n_pad = (n + kTile - 1) / kTile * kTile;
  c->global_offset = global_offset;
  c->n_global = n_global;
  cudaStream_t st = ctx->stream;
  const int64_t words = c->n_pad / 32;
  cudaError_t e;
  if ((e = cudaMalloc(&c->soa, (size_t)6 * c->n_pad * sizeof(float))) != cudaSuccess ||
      (e = cudaMalloc(&c->enabled, (size_t)words * 4)) != cudaSuccess ||
      (e = cudaMalloc(&c->valid, (size_t)words * 4)) != cudaSuccess) {
    rsc_cloud_destroy(c);
    return fail_cuda(ctx, e, "cloud_create: cudaMalloc");
  }
  RSC_CUDA(ctx, cudaMemsetAsync(c->soa, 0, (size_t)6 * c->n_pad * sizeof(float), st));
  if (exact && ((e = cudaMalloc(&c->xyz64, (size_t)3 * n * sizeof(double))) != cudaSuccess ||
                (e = cudaMalloc(&c->nrm64, (size_t)3 * n * sizeof(double))) != cudaSuccess)) {
    rsc_cloud_destroy(c);
    return fail_cuda(ctx, e, "cloud_create_f64_exact: cudaMalloc");
  }
  if (shard) {  // replicated whole-cloud enabled mask, all points enabled (like every rank's local mask)
    c->g_words = (n_global + kTile - 1) / kTile * (kTile / 32);
    if ((e = cudaMalloc(&c->g_enabled, (size_t)c->g_words * 4)) != cudaSuccess) {
      rsc_cloud_destroy(c);
      return fail_cuda(ctx, e, "cloud_create_shard: cudaMalloc");
    }
    fill_valid_kernel<<<(unsigned)((c->g_words + 255) / 256), 256, 0, st>>>(c->g_enabled, nullptr, n_global, c->g_words);
  }
  RSC_CUDA(ctx, cudaStreamSynchronize(st));
  int32_t rc = cloud_upload<T>(c, xyz, nrm);
  if (rc) {
    rsc_cloud_destroy(c);
    return rc;
  }
  *out = c;
  return RSC_OK;
}

}  // namespace rsc

using namespace rsc;

extern "C" {

int32_t rsc_cloud_create(rsc_ctx* ctx, const float* xyz, const float* nrm, int64_t n, rsc_cloud** out) {
  return cloud_create_impl<float>(ctx, xyz, nrm, n, 0, n, out);
}

int32_t rsc_cloud_create_f64(rsc_ctx* ctx, const double* xyz, const double* nrm, int64_t n, rsc_cloud** out) {
  return cloud_create_impl<double>(ctx, xyz, nrm, n, 0, n, out);
}

int32_t rsc_cloud_create_f64_exact(rsc_ctx* ctx, const double* xyz, const double* nrm, int64_t n, rsc_cloud** out) {
  return cloud_create_impl<double>(ctx, xyz, nrm, n, 0, n, out, true);
}

int32_t rsc_cloud_is_exact(const rsc_cloud* c) { return c && c->exact() ? 1 : 0; }

int32_t rsc_cloud_create_shard(rsc_ctx* ctx, const float* xyz, const float* nrm, int64_t n, int64_t global_offset,
                               int64_t n_global, rsc_cloud** out) {
  if (global_offset < 0 || n_global < global_offset + n) return fail(ctx, RSC_E_ARG, "cloud_create_shard: bad range");
  return cloud_create_impl<float>(ctx, xyz, nrm, n, global_offset, n_global, out);
}

int32_t rsc_cloud_update(rsc_cloud* c, const float* xyz, const float* nrm, int64_t n) {
  if (!c) return RSC_E_ARG;
  if (c->exact()) return fail(c->ctx, RSC_E_STATE, "cloud_update: an exact cloud keeps the float64 coordinates it was created from (create a new one)");
  if (!xyz || !nrm || n != c->n) return fail(c->ctx, RSC_E_ARG, "cloud_update: the cloud size cannot change");
  RSC_CUDA(c->ctx, cudaSetDevice(c->ctx->device));
  int32_t rc = cloud_ready(c);  // an earlier upload may still be in flight
  if (rc) return rc;
  if ((rc = cloud_upload<float>(c, xyz, nrm))) return rc;
  bool has_subsets = false;
  for (auto& s : c->subsets) has_subsets = has_subsets || s.soa;
  if (!has_subsets) return RSC_OK;  // stays asynchronous: the next rsc_score overlaps with the upload
  if ((rc = cloud_ready(c))) return rc;
  for (size_t i = 0; i < c->subsets.size(); ++i) {  // gathered subset copies follow the new coordinates
    rsc_subset& s = c->subsets[i];
    if (!s.soa) continue;
    s.release_cull_view();  // new coordinates: the Morton view is rebuilt when it is next needed
    if (s.m > 0) {
      gather_subset_kernel<<<(unsigned)((s.m + 255) / 256), 256, 0, c->ctx->stream>>>(c->soa, c->n_pad, s.idx, s.m, s.m_pad, s.soa);
      RSC_CUDA(c->ctx, cudaGetLastError());
    }
    RSC_CUDA(c->ctx, cudaMemcpyAsync(s.enabled, s.valid, (size_t)(s.m_pad / 32) * 4, cudaMemcpyDeviceToDevice, c->ctx->stream));
  }
  RSC_CUDA(c->ctx, cudaStreamSynchronize(c->ctx->stream));
  return RSC_OK;
}

void rsc_cloud_destroy(rsc_cloud* c) {
  if (!c) return;
  if (c->ctx) {
    cudaSetDevice(c->ctx->device);
    cudaStreamSynchronize(c->ctx->copy_stream);
    cudaStreamSynchronize(c->ctx->stream);
  }
  c->selbuf.release();
  cells_release(c);
  for (auto e : c->chunk_ev) cudaEventDestroy(e);
  if (c->d_bounds) cudaFree(c->d_bounds);
  for (auto& s : c->subsets) {
    if (s.soa) cudaFree(s.soa);
    if (s.enabled) cudaFree(s.enabled);
    if (s.valid) cudaFree(s.valid);
    if (s.idx) cudaFree(s.idx);
    s.release_cull_view();
  }
  if (c->soa) cudaFree(c->soa);
  if (c->xyz64) cudaFree(c->xyz64);
  if (c->nrm64) cudaFree(c->nrm64);
  if (c->g_enabled) cudaFree(c->g_enabled);
  if (c->enabled) cudaFree(c->enabled);
  if (c->valid) cudaFree(c->valid);
  delete c;
}

int64_t rsc_cloud_size(const rsc_cloud* c) { return c ? c->n : 0; }

int32_t rsc_cloud_set_subset(rsc_cloud* c, int32_t subset_id, const int64_t* idx, int64_t m) {
  if (!c) return RSC_E_ARG;
  if (int32_t rcr = cloud_ready(c)) return rcr;
  rsc_ctx* ctx = c->ctx;
  if (subset_id < 0 || subset_id > 4095 || !idx || m <= 0) return fail(ctx, RSC_E_ARG, "set_subset: bad arguments");
  const int64_t m_global = m;
  std::vector<int64_t> local;  // shard: the entries of this rank's range, as local indices, in subset order
  if (c->is_shard()) {
    for (int64_t j = 0; j < m; ++j) {
      if (idx[j] < 0 || idx[j] >= c->n_global) return fail(ctx, RSC_E_ARG, "set_subset: index out of range");
      if (idx[j] >= c->global_offset && idx[j] < c->global_offset + c->n) local.push_back(idx[j] - c->global_offset);
    }
    idx = local.data();
    m = (int64_t)local.size();
  } else {
    for (int64_t j = 0; j < m; ++j)
      if (idx[j] < 0 || idx[j] >= c->n) return fail(ctx, RSC_E_ARG, "set_subset: index out of range");
  }
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  if ((size_t)subset_id >= c->subsets.size()) c->subsets.resize(subset_id + 1);
  rsc_subset& s = c->subsets[subset_id];
  if (s.soa) {
    cudaFree(s.soa), cudaFree(s.enabled), cudaFree(s.valid), cudaFree(s.idx);
    s.release_cull_view();
    s = rsc_subset();
  }
  s.m = m;
  s.m_global = m_global;
  s.xyz64 = c->xyz64;
  s.nrm64 = c->nrm64;
  s.m_pad = (m + kTile - 1) / kTile * kTile;
  if (s.m_pad == 0) s.m_pad = kTile;  // a rank may own no point of the subset: one all-padding tile
  const int64_t words = s.m_pad / 32;
  cudaStream_t st = ctx->stream;
  cudaError_t e;
  if ((e = cudaMalloc(&s.soa, (size_t)6 * s.m_pad * sizeof(float))) != cudaSuccess ||
      (e = cudaMalloc(&s.enabled, (size_t)words * 4)) != cudaSuccess ||
      (e = cudaMalloc(&s.valid, (size_t)words * 4)) != cudaSuccess ||
      (e = cudaMalloc(&s.idx, (size_t)(m > 0 ? m : 1) * sizeof(int64_t))) != cudaSuccess) {
    cudaFree(s.soa), cudaFree(s.enabled), cudaFree(s.valid), cudaFree(s.idx);  // cudaFree(nullptr) is a no-op
    s = rsc_subset();  // not uploaded
    return fail_cuda(ctx, e, "set_subset: cudaMalloc");
  }
  RSC_CUDA(ctx, cudaMemsetAsync(s.soa, 0, (size_t)6 * s.m_pad * sizeof(float), st));
  if (m > 0) {
    RSC_CUDA(ctx, cudaMemcpyAsync(s.idx, idx, (size_t)m * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    gather_subset_kernel<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(c->soa, c->n_pad, s.idx, m, s.m_pad, s.soa);
    RSC_CUDA(ctx, cudaGetLastError());
  }
  fill_valid_kernel<<<(unsigned)((words + 255) / 256), 256, 0, st>>>(s.valid, nullptr, m, words);
  RSC_CUDA(ctx, cudaGetLastError());
  gather_enabled_kernel<<<(unsigned)((words * 32 + 255) / 256), 256, 0, st>>>(c->enabled, s.idx, m, words, s.enabled);
  RSC_CUDA(ctx, cudaGetLastError());
  RSC_CUDA(ctx, cudaStreamSynchronize(st));
  return RSC_OK;
}

int64_t rsc_cloud_subset_size(const rsc_cloud* c, int32_t subset_id) {
  if (!c || subset_id < 0 || (size_t)subset_id >= c->subsets.size()) return -1;
  return c->subsets[subset_id].soa ? c->subsets[subset_id].m : -1;
}

int32_t rsc_cloud_get_enabled(rsc_cloud* c, uint64_t* words) {
  if (!c || !words) return RSC_E_ARG;
  if (int32_t rcr = cloud_ready(c)) return rcr;
  rsc_ctx* ctx = c->ctx;
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t bytes = (size_t)((c->n + 63) / 64) * 8;
  RSC_CUDA(ctx, cudaMemcpyAsync(words, c->enabled, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  RSC_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return RSC_OK;
}

int32_t rsc_cloud_set_enabled(rsc_cloud* c, const uint64_t* words) {
  if (!c || !words) return RSC_E_ARG;
  if (int32_t rcr = cloud_ready(c)) return rcr;
  rsc_ctx* ctx = c->ctx;
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t bytes = (size_t)((c->n + 63) / 64) * 8;
  const int64_t w = c->n_pad / 32;
  c->enabled_changed();
  RSC_CUDA(ctx, cudaMemcpyAsync(c->enabled, words, bytes, cudaMemcpyHostToDevice, ctx->stream));
  and_words_kernel<<<(unsigned)((w + 255) / 256), 256, 0, ctx->stream>>>(c->enabled, c->valid, w);
  RSC_CUDA(ctx, cudaGetLastError());
  int32_t rc = refresh_subsets_enabled(c, ctx->stream);
  if (rc) return rc;
  RSC_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return RSC_OK;
}

int32_t rsc_cloud_enable_all(rsc_cloud* c) {
  if (!c) return RSC_E_ARG;
  if (int32_t rcr = cloud_ready(c)) return rcr;
  rsc_ctx* ctx = c->ctx;
  RSC_CUDA(ctx, cudaSetDevice(ctx->device));
  c->enabled_changed();
  RSC_CUDA(ctx, cudaMemcpyAsync(c->enabled, c->valid, (size_t)(c->n_pad / 32) * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  if (c->is_shard()) {  // every rank enables all of its points: so does the replicated mask
    fill_valid_kernel<<<(unsigned)((c->g_words + 255) / 256), 256, 0, ctx->stream>>>(c->g_enabled, nullptr, c->n_global, c->g_words);
    RSC_CUDA(ctx, cudaGetLastError());
  }
  for (auto& s : c->subsets) {
    if (!s.soa) continue;
    RSC_CUDA(ctx, cudaMemcpyAsync(s.enabled, s.valid, (size_t)(s.m_pad / 32) * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    // (the Morton view of the culled scorer has its real points in front too: the same words)
    if (s.cen) RSC_CUDA(ctx, cudaMemcpyAsync(s.cen, s.valid, (size_t)(s.m_pad / 32) * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  }
  RSC_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return RSC_OK;
}

int64_t rsc_cloud_count_enabled(rsc_cloud* c) {
  if (!c) return -1;
  if (cloud_ready(c)) return -1;
  rsc_ctx* ctx = c->ctx;
  if (cudaSetDevice(ctx->device) != cudaSuccess) return -1;
  return count_mask_bits(ctx, c->enabled, c->n_pad / 32);
}

}  // extern "C"
