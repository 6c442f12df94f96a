// rsc_loop.cuh -- kernels and device-side structures shared by the two loops behind rsc_ransac_run
// (rsc_loop.cu: the reference behaviour with the bookkeeping decided on the device; rsc_run.cu: the
// host-walked loop of the extension switches).  Included by both translation units (static kernels).
#pragma once
#include <vector>

#include "rsc_common.cuh"

namespace rsc {

// ---- K3: scores of the freshly scored candidates, arg-max over the store -------------------------
// score = policy count; tainted = sphere whose count includes a disabled point (Q4)
static __global__ void finish_new_kernel(const rsc_cand* __restrict__ cands, int n, const int32_t* __restrict__ cv,
                                  const int32_t* __restrict__ ce, uint32_t honour_enabled, int32_t* __restrict__ score,
                                  uint8_t* __restrict__ flags) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int t = cands[i].type;
  const bool honour = t >= RSC_NTYPES || ((honour_enabled >> t) & 1u);  // user shapes honour the enabled mask
  score[i] = honour ? ce[i] : cv[i];
  flags[i] = (uint8_t)(1u | ((!honour && cv[i] != ce[i]) ? 2u : 0u));  // bit0 alive, bit1 tainted
}

// first index of the maximum score among alive candidates (ties: first wins, Q16)
static __global__ void __launch_bounds__(1024) argmax_kernel(const int32_t* __restrict__ score, const uint8_t* __restrict__ flags,
                                                      int n, int64_t* __restrict__ out /*[2]: index, score*/) {
  __shared__ long long best[32];
  long long b = -1;  // key = score << 32 | (0x7fffffff - index): larger key = better
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    if (flags[i] & 1u) {
      const long long key = ((long long)score[i] << 32) | (long long)(0x7fffffff - i);
      b = key > b ? key : b;
    }
#pragma unroll
  for (int d = 16; d; d >>= 1) {
    const long long o = __shfl_xor_sync(0xffffffffu, b, d);
    b = o > b ? o : b;
  }
  if ((threadIdx.x & 31) == 0) best[threadIdx.x >> 5] = b;
  __syncthreads();
  if (threadIdx.x < 32) {
    b = best[threadIdx.x];
#pragma unroll
    for (int d = 16; d; d >>= 1) {
      const long long o = __shfl_xor_sync(0xffffffffu, b, d);
      b = o > b ? o : b;
    }
    if (threadIdx.x == 0) {
      if (b < 0) {
        out[0] = -1, out[1] = 0;
      } else {
        out[0] = 0x7fffffff - (int)(b & 0xffffffffll);
        out[1] = (int)(b >> 32);
      }
    }
  }
}

// the same over a large store (cell sampler: millions of candidates) by many CTAs: partial maxima meet in
// out[0] (as a key, by atomicMax), a one-thread kernel decodes it in place
static __global__ void __launch_bounds__(256) argmax_part_kernel(const int32_t* __restrict__ score, const uint8_t* __restrict__ flags,
                                                                  int n, long long* __restrict__ key_out) {
  __shared__ long long best[8];
  long long b = -1;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    if (flags[i] & 1u) {
      const long long key = ((long long)score[i] << 32) | (long long)(0x7fffffff - i);
      b = key > b ? key : b;
    }
#pragma unroll
  for (int d = 16; d; d >>= 1) {
    const long long o = __shfl_xor_sync(0xffffffffu, b, d);
    b = o > b ? o : b;
  }
  if ((threadIdx.x & 31) == 0) best[threadIdx.x >> 5] = b;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) b = best[w] > b ? best[w] : b;
    if (b >= 0) atomicMax(key_out, b);
  }
}

static __global__ void argmax_decode_kernel(int64_t* __restrict__ out) {
  const long long b = (long long)out[0];
  if (b < 0) {
    out[0] = -1, out[1] = 0;
  } else {
    out[0] = 0x7fffffff - (int)(b & 0xffffffffll);
    out[1] = (int)(b >> 32);
  }
}

static cudaError_t argmax_enqueue(const int32_t* score, const uint8_t* flags, int n, int64_t* out, int sm_count, cudaStream_t st) {
  if (n <= (1 << 16)) {
    argmax_kernel<<<1, 1024, 0, st>>>(score, flags, n, out);
    return cudaGetLastError();
  }
  cudaError_t e = cudaMemsetAsync(out, 0xff, 8, st);  // key -1
  if (e != cudaSuccess) return e;
  const int grid = std::min(sm_count * 4, (n + 2047) / 2048);
  argmax_part_kernel<<<grid, 256, 0, st>>>(score, flags, n, reinterpret_cast<long long*>(out));
  argmax_decode_kernel<<<1, 1, 0, st>>>(out);
  return cudaGetLastError();
}

// ---- K5 helpers -----------------------------------------------------------------------------------
// per word of the subset mask: how many bits were cleared by the extraction
static __global__ void newly_count_kernel(const uint32_t* __restrict__ old_en, const uint32_t* __restrict__ new_en, int64_t words,
                                   uint32_t* __restrict__ cnt) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w < words) cnt[w] = __popc(old_en[w] & ~new_en[w]);
}

// gather the newly disabled subset points into a compact SoA scratch set
// (exact clouds: idx / out_idx non-null, the cloud index of every gathered point, the map of the scratch set)
static __global__ void newly_gather_kernel(const uint32_t* __restrict__ old_en, const uint32_t* __restrict__ new_en, int64_t words,
                                    const unsigned long long* __restrict__ offs, const float* __restrict__ soa, int64_t m_pad,
                                    float* __restrict__ out, int64_t out_pad, const int64_t* __restrict__ idx,
                                    int64_t* __restrict__ out_idx) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= words) return;
  uint32_t bits = old_en[w] & ~new_en[w];
  unsigned long long o = offs[w];
  while (bits) {
    const int b = __ffs(bits) - 1;
    bits &= bits - 1;
    const int64_t j = w * 32 + b;
#pragma unroll
    for (int f = 0; f < 6; ++f) out[f * out_pad + o] = soa[f * m_pad + j];
    if (out_idx) out_idx[o] = idx[j];
    ++o;
  }
}

static __global__ void fill_valid_words_kernel(uint32_t* __restrict__ valid, int64_t n, int64_t words) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= words) return;
  const int64_t lo = w * 32;
  valid[w] = lo + 32 <= n ? 0xffffffffu : (lo < n ? (1u << (n - lo)) - 1u : 0u);
}

// alive &= no newly disabled compatible point; tainted spheres die; keep[] = alive as 0/1 words
static __global__ void invalidate_kernel(const int32_t* __restrict__ hit, uint8_t* __restrict__ flags, int n, int best,
                                  uint32_t* __restrict__ keep) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint8_t f = flags[i];
  if (i == best || hit[i] > 0 || (f & 2u)) f = 0;
  flags[i] = f;
  keep[i] = f & 1u;
}

static __global__ void compact_store_kernel(const rsc_cand* __restrict__ c0, const int32_t* __restrict__ s0,
                                     const uint8_t* __restrict__ f0, const uint32_t* __restrict__ keep,
                                     const unsigned long long* __restrict__ offs, int n, rsc_cand* __restrict__ c1,
                                     int32_t* __restrict__ s1, uint8_t* __restrict__ f1) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !keep[i]) return;
  const unsigned long long o = offs[i];
  c1[o] = c0[i];
  s1[o] = s0[i];
  f1[o] = f0[i];
}

// the candidate store (device), ping-pong buffers for order-preserving compaction
struct Store {
  DevBuf cands[2], score[2], flags[2];
  int cur = 0;
  int n = 0;
  size_t cap = 0;
  cudaError_t reserve(size_t want, cudaStream_t st) {
    if (want <= cap) return cudaSuccess;
    size_t ncap = cap ? cap : 4096;
    while (ncap < want) ncap *= 2;
    for (int b = 0; b < 2; ++b) {
      DevBuf nc, ns, nf;
      cudaError_t e;
      if ((e = nc.ensure(ncap * sizeof(rsc_cand))) != cudaSuccess) return e;
      if ((e = ns.ensure(ncap * 4)) != cudaSuccess) return e;
      if ((e = nf.ensure(ncap)) != cudaSuccess) return e;
      if (b == cur && n) {
        cudaMemcpyAsync(nc.p, cands[b].p, (size_t)n * sizeof(rsc_cand), cudaMemcpyDeviceToDevice, st);
        cudaMemcpyAsync(ns.p, score[b].p, (size_t)n * 4, cudaMemcpyDeviceToDevice, st);
        cudaMemcpyAsync(nf.p, flags[b].p, (size_t)n, cudaMemcpyDeviceToDevice, st);
        cudaStreamSynchronize(st);
      }
      cands[b].release(), score[b].release(), flags[b].release();
      cands[b] = nc, score[b] = ns, flags[b] = nf;
    }
    cap = ncap;
    return cudaSuccess;
  }
  void release() {
    for (int b = 0; b < 2; ++b) cands[b].release(), score[b].release(), flags[b].release();
  }
};

// scratch of the device loop, kept on the context between runs (allocating and freeing ~100 MB of
// device buffers per run cost 10-25 ms of a 40 ms loop)
struct LoopScratch {
  Store store;
  DevBuf newcnt, hostio, olden, nscratch, nidx, nvalid, nmeta, lvbuf, prog, ntiles;
};

}  // namespace rsc

// The loop runs `nb` iterations speculatively as one batch (same Philox set ids as nb separate
// iterations).  seg[j] = first compacted candidate that belongs to iteration j of the batch
// (candidates are in set order), seg[nb] = their number.
static __global__ void seg_bounds_kernel(const int32_t* __restrict__ out_set, const unsigned long long* __restrict__ total, int S, int nb,
                                  int32_t* __restrict__ seg) {
  const int j = threadIdx.x;
  if (j > nb) return;
  const int n = (int)*total;
  int lo = 0, hi = n;
  const int key = j * S;  // first set of iteration j
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (out_set[mid] < key)
      lo = mid + 1;
    else
      hi = mid;
  }
  seg[j] = (j == nb) ? n : lo;
}

// per batch iteration: arg-max key (score << 32 | 0x7fffffff - store index; -1 if empty) over its new candidates
static __global__ void __launch_bounds__(256) seg_argmax_kernel(const int32_t* __restrict__ score, const uint8_t* __restrict__ flags,
                                                         const int32_t* __restrict__ seg, int store_n0, long long* __restrict__ keys,
                                                         int limit = 0x7fffffff /* candidates actually scored (sync-free path) */) {
  __shared__ long long best[8];
  const int j = blockIdx.x;
  long long b = -1;
  const int hi = min(seg[j + 1], limit);
  for (int i = seg[j] + threadIdx.x; i < hi; i += blockDim.x) {
    const int g = store_n0 + i;
    if (flags[g] & 1u) {
      const long long key = ((long long)score[g] << 32) | (long long)(0x7fffffff - g);
      b = key > b ? key : b;
    }
  }
#pragma unroll
  for (int d = 16; d; d >>= 1) {
    const long long o = __shfl_xor_sync(0xffffffffu, b, d);
    b = o > b ? o : b;
  }
  if ((threadIdx.x & 31) == 0) best[threadIdx.x >> 5] = b;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) b = best[w] > b ? best[w] : b;
    keys[j] = b;
  }
}

// 1 if either guard-band queue (groups, pairs) of the last score call overflowed
static __global__ void queue_overflow_kernel(const uint32_t* __restrict__ wl_count, uint32_t cap, int32_t* __restrict__ out) {
  *out = (wl_count[0] > cap || wl_count[1] > cap) ? 1 : 0;
}

// after an overflow: size the queues for what the last call wanted (+25 %); the buffers themselves
// are re-allocated by the next score_enqueue
static int32_t grow_guard_queue(rsc_ctx* ctx) {
  uint32_t n[2] = {0, 0};
  if (cudaMemcpy(n, ctx->wl_count.p, sizeof(n), cudaMemcpyDeviceToHost) != cudaSuccess)
    return rsc::fail(ctx, RSC_E_CUDA, "ransac_run: reading the guard-band queue fill failed");
  const size_t need = (size_t)(n[0] > n[1] ? n[0] : n[1]);
  if (need > ctx->wl_cap) ctx->wl_cap = need + need / 4 + 1024;
  else ctx->wl_cap = ctx->wl_cap * 2;  // another rank overflowed: keep the sizes moving together
  return RSC_OK;
}

struct rsc_run {
  std::vector<rsc_cand> shapes;
  std::vector<int64_t> off{0};  // off[i]..off[i+1]: list of shape i inside d_idx
  int64_t* d_idx = nullptr;
  rsc_ctx* ctx = nullptr;  // the context the run was made on (must outlive the run)
  int device = 0;
  int iterations = 0;
  int64_t refined = 0;  // progressive scoring: (candidate, subset) evaluations beyond subset 1
  double seconds = 0.0;
  int nlevels = 0;  // cell sampler: final level weights / accumulated level scores
  double levelweight[11] = {0}, levelscore[11] = {0};
  std::vector<int64_t> total;  // whole-list sizes (sharded storage: off[] then counts this rank's part only)
  int syncs = 0, batches = 0;  // host synchronisations / speculative batches of the loop
  ~rsc_run() {
    if (d_idx) {
      cudaSetDevice(device);
      cudaFree(d_idx);
    }
  }
};

