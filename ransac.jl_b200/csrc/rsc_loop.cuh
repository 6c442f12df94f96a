// rsc_loop.cuh -- kernels and structures of the RANSAC loop (rsc_loop.cu) and what the host decision of the
// extension switches (rsc_run.cu) shares with it: the candidate store, the loop's device state and decision
// record, the slice of a subset a rank scores, the guard-band queue retry and the run object.
#pragma once
#include <vector>

#include "rsc_common.cuh"

namespace rsc {

// ---- K3: scores of the freshly scored candidates, arg-max over the store -------------------------
// score = policy count; tainted = sphere whose count includes a disabled point (Q4).  The candidates are the
// first min(*total, cap) of the launch (the sync-free path sizes it by a prediction, the classic one exactly).
static __global__ void finish_new_kernel(const rsc_cand* __restrict__ cands, const unsigned long long* __restrict__ total, int cap,
                                         const int32_t* __restrict__ cv, const int32_t* __restrict__ ce, uint32_t honour_enabled,
                                         int32_t* __restrict__ score, uint8_t* __restrict__ flags) {
  const int n = (int)min(*total, (unsigned long long)cap);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int t = cands[i].type;
    const bool honour = t >= RSC_NTYPES || ((honour_enabled >> t) & 1u);  // user shapes honour the enabled mask
    score[i] = honour ? ce[i] : cv[i];
    flags[i] = (uint8_t)(1u | ((!honour && cv[i] != ce[i]) ? 2u : 0u));  // bit0 alive, bit1 tainted
  }
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
  DevBuf newcnt, hostio, olden, nscratch, nidx, nvalid, nmeta, prog, ntiles;
};

constexpr int kMaxBatch = 64;  // most iterations of one speculative batch

struct BatchRec {  // the decision of one batch (decide_kernel's record, or the host's): device -> host, once per batch
  long long counters[3];
  int32_t used, extract, terminated, iterations;
  int32_t best_idx, best_score, store_n, ovf;  // ovf: 1 = a guard-band queue overflowed, 2 = more new candidates than the launch was sized for
  int32_t n_new, pad;
  rsc_cand best;
};

struct LoopDev {  // device-resident scratch + state of one run
  int64_t oldbest[2];             // arg-max over the store as it was before the batch: index, score
  long long seg_keys[kMaxBatch];  // per batch iteration: arg-max key over its new candidates
  int32_t seg[kMaxBatch + 2];     // per batch iteration: first new candidate
  long long lv[kMaxBatch][22];    // cell sampler, per batch iteration and octree level: new candidates, sum of their scores
  // (the host decision reads the fields above, up to this batch's rows of lv)
  long long counters[3];          // countcandidates: lengthC, allcand, nofminset (iterations.jl:70)
  BatchRec rec;
  int32_t tot_global[2];          // sharded storage: inliers of the extraction summed over the ranks
};

// This rank's slice of a subset copy: all of it (single GPU, or a shard's local entries) or, on replicated storage
// with a point range (`ranged`), the same fraction of it as the rank's range of the cloud.
inline PointSet subset_slice(const rsc_cloud* cloud, const rsc_subset& sb, bool ranged) {
  PointSet v = view_subset(&sb);
  if (!ranged || cloud->n_pad <= 0) return v;
  const int64_t lo = (int64_t)((double)cloud->range_lo / cloud->n_pad * sb.m_pad) / kTile * kTile;
  const int64_t hi = cloud->range_hi >= cloud->n_pad ? sb.m_pad : (int64_t)((double)cloud->range_hi / cloud->n_pad * sb.m_pad) / kTile * kTile;
  v.x += lo, v.y += lo, v.z += lo, v.nx += lo, v.ny += lo, v.nz += lo;
  v.enabled += lo / 32, v.valid += lo / 32;
  if (v.map) v.map += lo;
  v.n_pad = std::max<int64_t>(0, hi - lo);
  v.n = std::max<int64_t>(0, std::min(sb.m, hi) - lo);
  return v;
}

// K5, the re-scoring of the store after an extraction: for each stored candidate, its compatible points among the
// subset points the extraction just disabled (old & ~new words of the source).
struct K5In {
  const rsc_cand* cands;     // the store [nst]
  int nst;
  PointSet src;              // the source of the newly disabled points: the subset's Morton view or the rank's slice
  bool view;                 // src is the Morton view (sub.ctiles are its spheres)
  const float4* view_tiles;  // sub.ctiles
  uint32_t* olden;           // the source's whole-subset enabled words before the extraction (the masked form clears
                             // the still-enabled ones in place: old &= ~new)
  int64_t old_word0;         // the first word of src within olden
  const uint32_t* new_en;    // the whole-subset enabled words after the extraction (sub.cen for the view)
  int64_t swords;            // words of olden / new_en
  int bound;                 // scratch bound of the gathered form: the extracted candidate's subset-1 score
  bool masked;               // masked form: score the whole source under old & ~new instead of gathering
  int cull_mode;             // RSC_LOOP_CULL: 0 never, 1 for a large store, 2 always (view only)
  bool use_small;            // the small-batch scorer may be taken
  const FitOrder* uo;        // user shapes (nullable)
  bool coll;                 // hits summed over the ranks
};
struct K5Out {
  int32_t* hit;              // [nst] hits, then [nst] guard-band queue overflow, [nst + 1] scratch set too small
  uint32_t* keep;            // [nst] scratch for k5_compact
  unsigned long long *koff, *ktot;
};
int32_t k5_hits(rsc_ctx* ctx, rsc_cloud* cloud, const K5In& in, const Thresh& th, K5Out* out, cudaStream_t st);
// removeinvalidshapes!: drop the best, every candidate with a hit and the tainted spheres, order-preserving
// compaction of (cands, score, flags)[0 .. nst) into the *1 arrays; *ktot = survivors
int32_t k5_compact(const K5Out& o, int nst, int best, const rsc_cand* c0, const int32_t* s0, uint8_t* f0, rsc_cand* c1,
                       int32_t* s1, uint8_t* f1, rsc_ctx* ctx, cudaStream_t st);

// The host decision of a batch (rsc_run.cu), taken instead of decide_kernel's when RSC_SCORE_PROGRESSIVE,
// RSC_SAMPLER_OCTREE or RSC_LOOP_HOSTWALK is set.  `d` is the host copy of the device state after K2 + K3,
// `newscore` the new candidates' subset-1 scores (progressive scoring).  Fills *rec like decide_kernel does.
struct HostWalk;
int32_t host_decide(HostWalk& w, const LoopDev& d, const int32_t* newscore, int store_n0, int nb, int k0, BatchRec* rec);
// after K5: keep[i] = 1 for the store entries that survived (progressive scoring compacts its host mirror with it)
void host_compacted(HostWalk& w, const std::vector<uint32_t>& keep);
// the loop behind rsc_ransac_run / rsc_ransac_run_user.  order (nullable): a mixed fit order in place of
// p->shape_types; host (nullable): the host decision, else decide_kernel's
int32_t ransac_loop_device(rsc_cloud* cloud, const rsc_params* p, uint64_t seed, rsc_run* run, const FitOrder* order, HostWalk* host);

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

