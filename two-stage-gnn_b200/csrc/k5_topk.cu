// K5 -- SAGPooling selection: per-graph top-k, filter_adj edge compaction, gated gather.
//
// Replaces PyG 1.6.3 `topk` / `filter_adj` (called from Code/sag/layers.py:20,23) and the gate
// x[perm] * tanh(score[perm]) (Code/sag/layers.py:21).  Integer outputs are deterministic and
// bit-exact: the ordering is a strict total order on (score descending, node id ascending), NaN
// first, -0.0 == +0.0, i.e. what torch's stable CPU sort produces.
//
// top-k = rank selection, one CTA per graph: the graph's keys are staged in shared memory as
// order-preserving 64-bit composites (score key, ~index), every thread owns a node and counts the keys that precede its own
// (broadcast shared-memory reads, no barriers in the hot loop, no atomics).  n_g is ~10^2..10^3,
// so the O(n^2) compares (72k for a DD graph) cost less than the barriers of a sorting network.
#include "common.cuh"
#include <stdlib.h>

namespace tsg {

// order-preserving map: larger key <=> earlier in a descending sort. NaN -> max, -0 -> +0.
__device__ __forceinline__ uint32_t score_key(float s) {
  if (s != s) return 0xFFFFFFFFu;
  if (s == 0.f) s = 0.f;                       // canonicalise -0.0
  uint32_t b = __float_as_uint(s);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

struct KofN {
  const int64_t* gptr; float ratio;
  __device__ int operator()(int64_t g) const {
    float n = (float)(gptr[g + 1] - gptr[g]);
    return (int)ceilf(__fmul_rn(ratio, n));
  }
};

constexpr int TOPK_THREADS = 128;
constexpr int TOPK_SMEM_KEYS = 4096;   // 32 KB of 64-bit keys; larger graphs keep their keys in global memory

// Composite 64-bit key = (order-preserving score key << 32) | ~local index: one unsigned compare implements the
// strict total order (score descending, node id ascending), all keys of a graph are distinct, and
// rank(i) = #{j : key_j > key_i}.
__global__ void __launch_bounds__(TOPK_THREADS)
k_topk_rank(const float* __restrict__ score, const int64_t* __restrict__ gptr,
            const int64_t* __restrict__ kptr, int64_t* __restrict__ perm, unsigned long long* __restrict__ gkeys,
            int skip_upto) {
  pdl_wait();
  pdl_launch_dependents();
  __shared__ __align__(16) unsigned long long skeys[TOPK_SMEM_KEYS];
  const int g = blockIdx.x;
  const int64_t base = gptr[g];
  const int n = (int)(gptr[g + 1] - base);
  const int64_t obase = kptr[g];
  const int k = (int)(kptr[g + 1] - obase);
  if (n == 0 || k == 0) return;
  if (n <= skip_upto) return;                      // sorted by k_topk_sort
  const bool in_smem = n <= TOPK_SMEM_KEYS;
  unsigned long long* keys = in_smem ? skeys : (gkeys + base);
  for (int i = threadIdx.x; i < n; i += TOPK_THREADS)
    keys[i] = ((unsigned long long)score_key(score[base + i]) << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)i);
  __syncthreads();    // (global path: writes by this block, read by this block after the barrier)
  for (int i = threadIdx.x; i < n; i += TOPK_THREADS) {
    const unsigned long long ki = keys[i];
    int rank = 0;
    int j = 0;
    for (; j + 4 <= n; j += 4) {
      const unsigned long long a = keys[j], b = keys[j + 1], c = keys[j + 2], d = keys[j + 3];
      rank += (a > ki) + (b > ki) + (c > ki) + (d > ki);
    }
    for (; j < n; ++j) rank += keys[j] > ki;
    if (rank < k) perm[obase + rank] = base + i;
  }
}

// (Measured and dropped, profiles/r01c_step_kernels.md: one WARP per graph with the keys in registers -- shuffles for
// strides < 32, register exchanges above, no barriers: 95 us instead of 69 for the 0.97 M-node level; 24 serial
// warps per SM lose to 8-warp CTAs at the same compare-exchange count.)
// Sorting variant for graphs that fit shared memory (n <= TOPK_SMEM_KEYS): bitonic sort of the composite keys in
// DESCENDING order -- n log^2 n compare-exchanges instead of n^2 compares (10x fewer at n = 512; the rank kernel
// took 135 us on the 0.97 M-node level).  Keys are distinct, so the network's output is THE total order the rank
// kernel computes: identical perm.  Padding keys are 0 (smaller than every real key: score_key >= 1 << 31 or the
// index part is non-zero) and sort to the tail.
constexpr int TOPK_SORT_THREADS = 256;
__global__ void __launch_bounds__(TOPK_SORT_THREADS)
k_topk_sort(const float* __restrict__ score, const int64_t* __restrict__ gptr, const int64_t* __restrict__ kptr,
            int64_t* __restrict__ perm, int max_pad, int min_n) {
  pdl_wait();
  pdl_launch_dependents();
  extern __shared__ __align__(16) unsigned long long sk[];
  {
    const int g = blockIdx.x;
    const int64_t base = gptr[g];
    const int n = (int)(gptr[g + 1] - base);
    const int64_t obase = kptr[g];
    const int k = (int)(kptr[g + 1] - obase);
    if (n == 0 || k == 0) return;
    if (n > max_pad) return;                       // handled by k_topk_rank (second launch skips the rest)
    if (n <= min_n) return;                        // handled by k_topk_runs
    int npad = 32; while (npad < n) npad <<= 1;
    for (int i = threadIdx.x; i < npad; i += TOPK_SORT_THREADS)
      sk[i] = i < n ? (((unsigned long long)score_key(score[base + i]) << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)i)) : 0ull;
    __syncthreads();
    for (int kk = 2; kk <= npad; kk <<= 1) {
      for (int j = kk >> 1; j > 0; j >>= 1) {
        for (int t = threadIdx.x; t < (npad >> 1); t += TOPK_SORT_THREADS) {
          const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
          const int l = i | j;
          const unsigned long long a = sk[i], b = sk[l];
          const bool desc = (i & kk) == 0;
          if ((a < b) == desc) { sk[i] = b; sk[l] = a; }
        }
        __syncthreads();
      }
    }
    for (int i = threadIdx.x; i < k; i += TOPK_SORT_THREADS)
      perm[obase + i] = base + (int64_t)(0xFFFFFFFFu - (unsigned)(sk[i] & 0xFFFFFFFFull));
  }
}


// Register-run top-k (round 2): graphs of n <= TOPK_RUN_THREADS * 4 keys.  Every warp sorts its own run of 32 * KPT
// composite keys in REGISTERS (element e = slot * 32 + lane: strides < 32 are shuffles, strides >= 32 register swaps,
// no barrier), the runs go to shared memory, and a key's rank in the union is its position in its own run plus, for
// every other run, the number of keys greater than it (binary search; keys are distinct).  Two CTA barriers instead of
// the 45 of the 512-key network above; identical perm (the order is the same strict total order).
constexpr int TOPK_RUN_THREADS = 256;
template <int KPT>
__device__ __forceinline__ void topk_runs_body(const float* __restrict__ score, int64_t base, int n, int k,
                                               int64_t obase, int64_t* __restrict__ perm, unsigned long long* runs) {
  constexpr int NW = TOPK_RUN_THREADS / 32, RL = 32 * KPT;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  unsigned long long key[KPT];
#pragma unroll
  for (int s = 0; s < KPT; ++s) {
    const int i = w * RL + s * 32 + lane;
    key[s] = i < n ? (((unsigned long long)score_key(score[base + i]) << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)i)) : 0ull;
  }
#pragma unroll
  for (int kk = 2; kk <= RL; kk <<= 1) {
#pragma unroll
    for (int j = kk >> 1; j > 0; j >>= 1) {
      if (j >= 32) {
        const int js = j >> 5;
#pragma unroll
        for (int s = 0; s < KPT; ++s) {
          if ((s & js) == 0) {
            const bool desc = ((s * 32 + lane) & kk) == 0;
            const unsigned long long x = key[s], y = key[s | js];
            if ((x < y) == desc) { key[s] = y; key[s | js] = x; }
          }
        }
      } else {
#pragma unroll
        for (int s = 0; s < KPT; ++s) {
          const unsigned long long x = key[s];
          const unsigned long long y = __shfl_xor_sync(0xffffffffu, x, j);
          const bool keep_max = ((lane & j) == 0) == ((((s * 32 + lane) & kk)) == 0);
          key[s] = keep_max ? (x > y ? x : y) : (x < y ? x : y);
        }
      }
    }
  }
#pragma unroll
  for (int s = 0; s < KPT; ++s) runs[w * RL + s * 32 + lane] = key[s];
  __syncthreads();
#pragma unroll
  for (int s = 0; s < KPT; ++s) {
    const unsigned long long x = key[s];
    if (x == 0ull) continue;                                // padding
    int rank = s * 32 + lane;
    for (int r = 0; r < NW && r * RL < n; ++r) {
      if (r == w) continue;
      const unsigned long long* run = runs + r * RL;
      int lo = 0, hi = RL;                                  // first position whose key is < x (descending run)
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (run[mid] > x) lo = mid + 1; else hi = mid;
      }
      rank += lo;
    }
    if (rank < k) perm[obase + rank] = base + (int64_t)(0xFFFFFFFFu - (unsigned)(x & 0xFFFFFFFFull));
  }
}

// A graph of at most 32 * KPT <= 128 keys is ONE run: a warp sorts it in registers and the rank is the position, no
// shared memory and no CTA barrier -- the pooled levels of a DD-shape batch average 139 and 69 nodes, and a 256-thread CTA
// per such graph left most of its warps without keys and only G / 8 graphs in flight per wave.
template <int KPT>
__device__ __forceinline__ void topk_warp_body(const float* __restrict__ score, int64_t base, int n, int k,
                                               int64_t obase, int64_t* __restrict__ perm) {
  constexpr int RL = 32 * KPT;
  const int lane = threadIdx.x & 31;
  unsigned long long key[KPT];
#pragma unroll
  for (int s = 0; s < KPT; ++s) {
    const int i = s * 32 + lane;
    key[s] = i < n ? (((unsigned long long)score_key(score[base + i]) << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)i)) : 0ull;
  }
#pragma unroll
  for (int kk = 2; kk <= RL; kk <<= 1) {
#pragma unroll
    for (int j = kk >> 1; j > 0; j >>= 1) {
      if (j >= 32) {
        const int js = j >> 5;
#pragma unroll
        for (int s = 0; s < KPT; ++s) {
          if ((s & js) == 0) {
            const bool desc = ((s * 32 + lane) & kk) == 0;
            const unsigned long long x = key[s], y = key[s | js];
            if ((x < y) == desc) { key[s] = y; key[s | js] = x; }
          }
        }
      } else {
#pragma unroll
        for (int s = 0; s < KPT; ++s) {
          const unsigned long long x = key[s];
          const unsigned long long y = __shfl_xor_sync(0xffffffffu, x, j);
          const bool keep_max = ((lane & j) == 0) == ((((s * 32 + lane) & kk)) == 0);
          key[s] = keep_max ? (x > y ? x : y) : (x < y ? x : y);
        }
      }
    }
  }
#pragma unroll
  for (int s = 0; s < KPT; ++s) {
    const int rank = s * 32 + lane;
    if (key[s] != 0ull && rank < k) perm[obase + rank] = base + (int64_t)(0xFFFFFFFFu - (unsigned)(key[s] & 0xFFFFFFFFull));
  }
}

constexpr int TOPK_WARP_KEYS = 128;

__global__ void __launch_bounds__(TOPK_RUN_THREADS)
k_topk_runs(const float* __restrict__ score, const int64_t* __restrict__ gptr, const int64_t* __restrict__ kptr,
            int64_t* __restrict__ perm, int G, int cta_blocks) {
  pdl_wait();
  pdl_launch_dependents();
  __shared__ __align__(16) unsigned long long runs[TOPK_RUN_THREADS * 4];
  constexpr int NW = TOPK_RUN_THREADS / 32;
  if ((int)blockIdx.x >= cta_blocks) {
    // warp role: blocks behind the first cta_blocks give every warp one SMALL graph
    const int nwarps = ((int)gridDim.x - cta_blocks) * NW;
    for (int g = ((int)blockIdx.x - cta_blocks) * NW + (threadIdx.x >> 5); g < G; g += nwarps) {
      const int64_t base = gptr[g];
      const int n = (int)(gptr[g + 1] - base);
      if (n <= 0 || n > TOPK_WARP_KEYS) continue;
      const int64_t obase = kptr[g];
      const int k = (int)(kptr[g + 1] - obase);
      if (k <= 0) continue;
      if (n <= 32) topk_warp_body<1>(score, base, n, k, obase, perm);
      else if (n <= 64) topk_warp_body<2>(score, base, n, k, obase, perm);
      else topk_warp_body<4>(score, base, n, k, obase, perm);
    }
    return;
  }
  // CTA role: a graph of 129 .. 1,024 keys per block iteration
  for (int g = blockIdx.x; g < G; g += cta_blocks) {
    const int64_t base = gptr[g];
    const int n = (int)(gptr[g + 1] - base);
    if (n <= TOPK_WARP_KEYS || n > TOPK_RUN_THREADS * 4) continue;     // CTA-uniform
    const int64_t obase = kptr[g];
    const int k = (int)(kptr[g + 1] - obase);
    if (k > 0) {
      if (n <= TOPK_RUN_THREADS) topk_runs_body<1>(score, base, n, k, obase, perm, runs);
      else if (n <= 2 * TOPK_RUN_THREADS) topk_runs_body<2>(score, base, n, k, obase, perm, runs);
      else topk_runs_body<4>(score, base, n, k, obase, perm, runs);
    }
    __syncthreads();                                        // runs[] is reused by the next graph
  }
}

__global__ void k_batch_to_ptr(const int64_t* __restrict__ batch, int64_t n, int64_t G, int64_t* __restrict__ gptr) {
  // graph_ptr[g] = first i with batch[i] >= g ; batch sorted ascending
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= n;
       i += (int64_t)gridDim.x * blockDim.x) {
    int64_t prev = i == 0 ? -1 : batch[i - 1];
    int64_t cur = i == n ? G : batch[i];
    if (cur > G) cur = G;
    for (int64_t g = prev + 1; g <= cur; ++g) gptr[g] = i;
  }
}

// ---------------------------------- filter_adj -------------------------------------------
constexpr int FA_THREADS = 256;
constexpr int FA_ITEMS = 8;
constexpr int FA_TILE = FA_THREADS * FA_ITEMS;

__global__ void k_inv_perm(const int64_t* __restrict__ perm, int64_t k, int* __restrict__ inv) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < k;
       i += (int64_t)gridDim.x * blockDim.x)
    inv[perm[i]] = (int)i;
}

// pass 1: per-tile survivor count.  pass 2 (WRITE): order-preserving compaction.
template <bool WRITE>
__global__ void __launch_bounds__(FA_THREADS)
k_filter_adj(const int64_t* __restrict__ row, const int64_t* __restrict__ col, int64_t E_cap,
             const int64_t* __restrict__ E_dev, const int* __restrict__ inv,
             int* __restrict__ tile_cnt, const int* __restrict__ tile_off,
             int64_t* __restrict__ out_row, int64_t* __restrict__ out_col) {
  __shared__ int wcnt[FA_ITEMS][FA_THREADS / 32];
  __shared__ int woff[FA_ITEMS][FA_THREADS / 32];
  const int64_t E = dev_count(E_cap, E_dev);
  const int64_t base = (int64_t)blockIdx.x * FA_TILE;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int nr[FA_ITEMS], nc[FA_ITEMS];
  unsigned ball[FA_ITEMS];
#pragma unroll
  for (int k = 0; k < FA_ITEMS; ++k) {
    int64_t e = base + k * FA_THREADS + threadIdx.x;
    int r = -1, c = -1;
    if (e < E) { r = inv[row[e]]; c = inv[col[e]]; }
    bool keep = (r >= 0) && (c >= 0);
    nr[k] = r; nc[k] = c;
    ball[k] = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) wcnt[k][w] = __popc(ball[k]);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0;
    for (int k = 0; k < FA_ITEMS; ++k)
      for (int ww = 0; ww < FA_THREADS / 32; ++ww) { woff[k][ww] = s; s += wcnt[k][ww]; }
    if (!WRITE) tile_cnt[blockIdx.x] = s;
  }
  if (!WRITE) return;
  __syncthreads();
  const int toff = tile_off[blockIdx.x];
#pragma unroll
  for (int k = 0; k < FA_ITEMS; ++k) {
    if ((ball[k] >> lane) & 1u) {
      int p = toff + woff[k][w] + __popc(ball[k] & ((1u << lane) - 1u));
      out_row[p] = nr[k];
      out_col[p] = nc[k];
    }
  }
}

struct TileCnt {
  const int* c;
  __device__ int operator()(int64_t i) const { return c[i]; }
};

__global__ void k_store_count(const int* src, int64_t* dst) { *dst = (int64_t)*src; }

// ---------------------------------- gated gather -----------------------------------------
template <int VEC>
__global__ void __launch_bounds__(256)
k_gate_gather_fwd(const float* __restrict__ x, const float* __restrict__ score,
                  const int64_t* __restrict__ perm, const int64_t* __restrict__ batch,
                  float* __restrict__ xo, int64_t* __restrict__ batch_out, int64_t K, int F) {
  const int FV = F / VEC;
  const int64_t total = K * FV;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int64_t i = idx / FV; int f = (int)(idx - i * FV);
    int64_t j = perm[i];
    float t = tanhf(score[j]);
    if (VEC == 4) {
      float4 v = __ldg(reinterpret_cast<const float4*>(x) + j * FV + f);
      v.x *= t; v.y *= t; v.z *= t; v.w *= t;
      reinterpret_cast<float4*>(xo)[i * FV + f] = v;
    } else {
      xo[i * FV + f] = x[j * FV + f] * t;
    }
    if (f == 0 && batch != nullptr) batch_out[i] = batch[j];
  }
}

// float4 variant: LPR = F/4 lanes per node (8 lanes at F = 32 => 4 nodes per warp, 128-bit accesses)
template <int LPR>
__global__ void __launch_bounds__(256)
k_gate_gather_bwd_v4(const float4* __restrict__ dxo, const float4* __restrict__ x,
                     const float* __restrict__ score, const int* __restrict__ inv,
                     float4* __restrict__ dx, float* __restrict__ dscore, int64_t N, int F4) {
  const int l = threadIdx.x % LPR;
  const int64_t groups = ((int64_t)gridDim.x * blockDim.x) / LPR;
  const int64_t first = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPR;
  const int64_t iters = (N + groups - 1) / groups;                  // uniform trip count (shuffles below)
  for (int64_t it = 0; it < iters; ++it) {
    const int64_t j = first + it * groups;
    const bool ok = j < N;
    const int m = ok ? inv[j] : -1;
    float t = 0.f, dot = 0.f;
    if (m >= 0) t = tanhf(score[j]);
    for (int f = l; f < F4; f += LPR) {
      float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m >= 0) {
        const float4 go = __ldg(dxo + (int64_t)m * F4 + f);
        const float4 xv = __ldg(x + j * F4 + f);
        dot += go.x * xv.x + go.y * xv.y + go.z * xv.z + go.w * xv.w;
        g = make_float4(go.x * t, go.y * t, go.z * t, go.w * t);
      }
      if (ok && dx) dx[j * F4 + f] = g;
    }
#pragma unroll
    for (int d = LPR / 2; d > 0; d >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, d, LPR);
    if (ok && l == 0) dscore[j] = m >= 0 ? dot * (1.f - t * t) : 0.f;
  }
}

// one group of LPR lanes per source node j; writes every row of dx (zeros for dropped nodes)
template <int LPR>
__global__ void __launch_bounds__(256)
k_gate_gather_bwd(const float* __restrict__ dxo, const float* __restrict__ x,
                  const float* __restrict__ score, const int* __restrict__ inv,
                  float* __restrict__ dx, float* __restrict__ dscore, int64_t N, int F) {
  const int l = threadIdx.x % LPR;
  const int64_t group = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPR;
  const int64_t ngroups = ((int64_t)gridDim.x * blockDim.x) / LPR;
  // shuffles name only the LPR lanes of this group, which always iterate together
  const unsigned gmask = LPR == 32 ? 0xffffffffu
                                   : (((1u << LPR) - 1u) << (((threadIdx.x & 31) / LPR) * LPR));
  for (int64_t j = group; j < N; j += ngroups) {
    int m = inv[j];
    float dot = 0.f;
    float t = 0.f;
    if (m >= 0) t = tanhf(score[j]);
    for (int f = l; f < F; f += LPR) {
      float g = 0.f;
      if (m >= 0) {
        float go = dxo[(int64_t)m * F + f];
        dot += go * x[j * F + f];
        g = go * t;
      }
      if (dx) dx[j * F + f] = g;
    }
#pragma unroll
    for (int d = LPR / 2; d > 0; d >>= 1) dot += __shfl_xor_sync(gmask, dot, d);
    if (l == 0) dscore[j] = m >= 0 ? dot * (1.f - t * t) : 0.f;
  }
}

// Score-side half of the gate backward, driven by perm instead of inv (K10 fused backward; the x-side half lives in
// k_sag_conv_bwd_v4): for the i-th kept node j = perm[i]
//     dscore[j] = (dxo[i, :] . x[j, :]) * (1 - tanh(score[j])^2)            layers.py:21 backward w.r.t. score
// (dropped nodes keep the zero the caller memset), and the kernel also returns sum_j dscore[j] = the score layer's
// bias gradient.  Same per-lane products and butterfly as k_gate_gather_bwd_v4, so dscore is bit-identical to it; every
// lane group works on a kept row (the inv-driven kernel idled on the dropped half) and dxo is read sequentially.
constexpr int GSB_THREADS = 256;
constexpr int GSB_GRID = TSG_NUM_SMS * 4;
constexpr int GSB_ROWS = 4;

template <int LPR>
__global__ void __launch_bounds__(GSB_THREADS)
k_gate_score_bwd(const float4* __restrict__ dxo, const float4* __restrict__ x, const float* __restrict__ score,
                 const int64_t* __restrict__ perm, float* __restrict__ dscore, float* __restrict__ part,
                 int64_t K, int F4, float* __restrict__ dbs, unsigned* ticket) {
  pdl_wait();
  pdl_launch_dependents();
  constexpr int GROUPS = GSB_THREADS / LPR;
  __shared__ float s_sum[GSB_THREADS / 32];
  const int l = threadIdx.x % LPR, grp = threadIdx.x / LPR;
  const int64_t per_cta = (K + gridDim.x - 1) / gridDim.x;
  const int64_t i0 = (int64_t)blockIdx.x * per_cta;
  const int64_t i1 = i0 + per_cta < K ? i0 + per_cta : K;
  const int64_t iters = (per_cta + GROUPS * GSB_ROWS - 1) / (GROUPS * GSB_ROWS);      // uniform trip count (shuffles below)
  float local = 0.f;                                                    // this group's dscore sum (lane 0 holds it)
  for (int64_t it = 0; it < iters; ++it) {
    // GSB_ROWS kept rows per lane group in flight: perm first, then the dependent score / x gathers
    int64_t i[GSB_ROWS], j[GSB_ROWS];
    bool ok[GSB_ROWS];
    float t[GSB_ROWS], dot[GSB_ROWS];
#pragma unroll
    for (int u = 0; u < GSB_ROWS; ++u) {
      i[u] = i0 + (it * GSB_ROWS + u) * GROUPS + grp;
      ok[u] = i[u] < i1;
      j[u] = ok[u] ? __ldg(perm + i[u]) : 0;
    }
#pragma unroll
    for (int u = 0; u < GSB_ROWS; ++u) {
      t[u] = ok[u] ? __ldg(score + j[u]) : 0.f;
      dot[u] = 0.f;
      for (int f = l; f < F4; f += LPR) {
        if (ok[u]) {
          const float4 go = __ldg(dxo + i[u] * F4 + f);
          const float4 xv = __ldg(x + j[u] * F4 + f);
          dot[u] += go.x * xv.x + go.y * xv.y + go.z * xv.z + go.w * xv.w;
        }
      }
    }
#pragma unroll
    for (int u = 0; u < GSB_ROWS; ++u) {
#pragma unroll
      for (int d = LPR / 2; d > 0; d >>= 1) dot[u] += __shfl_xor_sync(0xffffffffu, dot[u], d, LPR);
      if (ok[u] && l == 0) {
        const float th = tanhf(t[u]);
        const float ds = dot[u] * (1.f - th * th);
        dscore[j[u]] = ds;
        local += ds;
      }
    }
  }
  // block sum in a fixed order: lanes (butterfly over the warp; non-leader lanes hold 0), then warps in index order
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) local += __shfl_xor_sync(0xffffffffu, local, d);
  if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tsum = s_sum[0];
    for (int w = 1; w < GSB_THREADS / 32; ++w) tsum += s_sum[w];
    part[blockIdx.x] = tsum;
  }
  partial_sum_tail(part, dbs, 1, nullptr, gridDim.x, 1, ticket);
}

}  // namespace tsg

using namespace tsg;

extern "C" size_t tsg_topk_workspace_bytes(int64_t N, int64_t G) {
  return ws_bytes(scan_ws_ints(G), 4) + ws_bytes((size_t)N + 1, 8) + 512;
}

extern "C" int tsg_topk_sizes(const int64_t* gptr, int64_t G, float ratio, int64_t* kptr,
                              void* workspace, size_t workspace_bytes, void* stream) {
  TSG_REQUIRE(G >= 0 && gptr && kptr, "topk_sizes: bad arguments");
  if (workspace_bytes < tsg_topk_workspace_bytes(0, G)) { set_error("topk_sizes: workspace too small"); return TSG_EWORKSPACE; }
  return exclusive_scan(KofN{gptr, ratio}, G, kptr, (int*)workspace, (cudaStream_t)stream);
}

extern "C" int tsg_topk(const float* score, const int64_t* gptr, const int64_t* kptr, int64_t G,
                        int64_t N, int64_t* perm, void* workspace, size_t workspace_bytes, void* stream) {
  return tsg_topk_bounded(score, gptr, kptr, G, N, N, perm, workspace, workspace_bytes, stream);
}

extern "C" int tsg_topk_bounded(const float* score, const int64_t* gptr, const int64_t* kptr, int64_t G, int64_t N,
                                int64_t max_graph_nodes, int64_t* perm, void* workspace, size_t workspace_bytes,
                                void* stream) {
  TSG_REQUIRE(G >= 0 && N >= 0, "topk: bad sizes");
  if (G == 0 || N == 0) return TSG_OK;
  TSG_REQUIRE(score && gptr && kptr && perm, "topk: null pointer");
  if (workspace_bytes < tsg_topk_workspace_bytes(N, G)) { set_error("topk: workspace too small"); return TSG_EWORKSPACE; }
  Workspace ws(workspace, workspace_bytes);
  ws.take<int>(scan_ws_ints(G));
  unsigned long long* gkeys = ws.take<unsigned long long>(N + 1);
  TSG_REQUIRE(G < (int64_t)0x7fffffff, "topk: too many graphs");
  static const bool no_sort = getenv("TSG_TOPK_NOSORT") != nullptr;
  static const bool no_runs = getenv("TSG_TOPK_NORUNS") != nullptr;      // A/B: round 1's shared-memory bitonic network only
  const int max_pad = no_sort ? 0 : TOPK_SMEM_KEYS;
  const int runs_upto = (no_sort || no_runs) ? 0 : TOPK_RUN_THREADS * 4;
  if (runs_upto > 0) {
    // CTA-per-graph blocks for graphs of 129 .. 1,024 keys, then warp-per-graph blocks for the smaller ones
    const int cta_blocks = (int)(G < (int64_t)TSG_NUM_SMS * 8 ? G : (int64_t)TSG_NUM_SMS * 8);
    const int64_t groups = (G + TOPK_RUN_THREADS / 32 - 1) / (TOPK_RUN_THREADS / 32);
    const int warp_blocks = (int)(groups < (int64_t)TSG_NUM_SMS * 4 ? groups : (int64_t)TSG_NUM_SMS * 4);
    TSG_LAUNCH_PDL("topk(runs)", k_topk_runs, cta_blocks + warp_blocks, TOPK_RUN_THREADS, 0, (cudaStream_t)stream, score, gptr, kptr, perm, (int)G, cta_blocks);
  }
  // the caller's bound on the largest graph decides which of the three size ranges can be populated at all
  if (!no_sort && max_graph_nodes > runs_upto)
    TSG_LAUNCH_PDL("topk(sort)", k_topk_sort, (int)G, TOPK_SORT_THREADS, (size_t)TOPK_SMEM_KEYS * 8, (cudaStream_t)stream, score, gptr, kptr, perm, max_pad, runs_upto);
  // graphs larger than the sort's shared-memory budget (and everything when the sort is disabled)
  if (max_graph_nodes > max_pad)
    TSG_LAUNCH_PDL("topk(rank)", k_topk_rank, (int)G, TOPK_THREADS, 0, (cudaStream_t)stream, score, gptr, kptr, perm, gkeys, max_pad);
  return check_launch("topk");
}

extern "C" int tsg_batch_to_ptr(const int64_t* batch, int64_t N, int64_t G, int64_t* gptr, void* stream) {
  TSG_REQUIRE(N >= 0 && G >= 0 && gptr && (N == 0 || batch), "batch_to_ptr: bad arguments");
  k_batch_to_ptr<<<grid_for(N + 1, 256), 256, 0, (cudaStream_t)stream>>>(batch, N, G, gptr);
  return check_launch("batch_to_ptr");
}

extern "C" size_t tsg_filter_adj_workspace_bytes(int64_t E) {
  size_t tiles = (size_t)((E + FA_TILE - 1) / FA_TILE) + 1;
  return 2 * ws_bytes(tiles + 1, 4) + ws_bytes(scan_ws_ints((int64_t)tiles), 4) + 512;
}

extern "C" int tsg_filter_adj(const int64_t* row, const int64_t* col, int64_t E, const int64_t* E_dev,
                              const int64_t* perm, int64_t K, int64_t N, int32_t* inv,
                              int64_t* out_row, int64_t* out_col, int64_t* out_E_dev,
                              void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TSG_REQUIRE(E >= 0 && K >= 0 && N >= 0 && inv && out_E_dev, "filter_adj: bad arguments");
  TSG_REQUIRE(E < (int64_t)0x7fffffff && N < (int64_t)0x7fffffff, "filter_adj: sizes must stay below 2^31");
  if (workspace_bytes < tsg_filter_adj_workspace_bytes(E)) { set_error("filter_adj: workspace too small"); return TSG_EWORKSPACE; }
  int tiles = (int)((E + FA_TILE - 1) / FA_TILE);
  Workspace ws(workspace, workspace_bytes);
  int* tile_cnt = ws.take<int>(tiles + 2);
  int* tile_off = ws.take<int>(tiles + 2);
  int* scan_ws = ws.take<int>(scan_ws_ints(tiles + 1));
  if (N > 0) cudaMemsetAsync(inv, 0xFF, (size_t)N * 4, st);
  if (K > 0) k_inv_perm<<<grid_for(K, 256), 256, 0, st>>>(perm, K, inv);
  if (tiles == 0) { cudaMemsetAsync(out_E_dev, 0, 8, st); return check_launch("filter_adj(empty)"); }
  k_filter_adj<false><<<tiles, FA_THREADS, 0, st>>>(row, col, E, E_dev, inv, tile_cnt, nullptr, nullptr, nullptr);
  int rc = exclusive_scan(TileCnt{tile_cnt}, tiles, tile_off, scan_ws, st);
  if (rc) return rc;
  k_store_count<<<1, 1, 0, st>>>(tile_off + tiles, out_E_dev);
  k_filter_adj<true><<<tiles, FA_THREADS, 0, st>>>(row, col, E, E_dev, inv, nullptr, tile_off, out_row, out_col);
  return check_launch("filter_adj");
}

extern "C" int tsg_gate_gather_fwd(const float* x, const float* score, const int64_t* perm,
                                   const int64_t* batch, float* xo, int64_t* batch_out,
                                   int64_t K, int64_t F, void* stream) {
  TSG_REQUIRE(K >= 0 && F > 0, "gate_gather_fwd: bad shape");
  if (K == 0) return TSG_OK;
  TSG_REQUIRE(x && score && perm && xo, "gate_gather_fwd: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  bool vec = F % 4 == 0 && (((uintptr_t)x | (uintptr_t)xo) & 15) == 0;
  if (vec) k_gate_gather_fwd<4><<<grid_for(K * (F / 4), 256), 256, 0, st>>>(x, score, perm, batch, xo, batch_out, K, (int)F);
  else k_gate_gather_fwd<1><<<grid_for(K * F, 256), 256, 0, st>>>(x, score, perm, batch, xo, batch_out, K, (int)F);
  return check_launch("gate_gather_fwd");
}

extern "C" int tsg_gate_gather_bwd(const float* dxo, const float* x, const float* score,
                                   const int32_t* inv, float* dx, float* dscore,
                                   int64_t N, int64_t F, void* stream) {
  TSG_REQUIRE(N >= 0 && F > 0, "gate_gather_bwd: bad shape");
  if (N == 0) return TSG_OK;
  TSG_REQUIRE(dxo && x && score && inv && dscore, "gate_gather_bwd: null pointer");     // dx nullable: dscore only
  cudaStream_t st = (cudaStream_t)stream;
  if (F % 4 == 0 && ((((uintptr_t)dxo) | ((uintptr_t)x) | ((uintptr_t)dx)) & 15) == 0) {
    int F4 = (int)(F / 4);
    int lp = 1; while (lp < F4 && lp < 32) lp <<= 1;
    int gr = grid_for(N, 256 / lp, 16);
#define TSG_GV(L) k_gate_gather_bwd_v4<L><<<gr, 256, 0, st>>>((const float4*)dxo, (const float4*)x, score, inv, (float4*)dx, dscore, N, F4)
    switch (lp) {
      case 1: TSG_GV(1); break; case 2: TSG_GV(2); break; case 4: TSG_GV(4); break;
      case 8: TSG_GV(8); break; case 16: TSG_GV(16); break; default: TSG_GV(32); break;
    }
#undef TSG_GV
    return check_launch("gate_gather_bwd");
  }
  int lpr = 1; while (lpr < F && lpr < 32) lpr <<= 1;
  int grid = grid_for(N, 256 / lpr);
#define TSG_GO(L) k_gate_gather_bwd<L><<<grid, 256, 0, st>>>(dxo, x, score, inv, dx, dscore, N, (int)F)
  switch (lpr) {
    case 1: TSG_GO(1); break; case 2: TSG_GO(2); break; case 4: TSG_GO(4); break;
    case 8: TSG_GO(8); break; case 16: TSG_GO(16); break; default: TSG_GO(32); break;
  }
#undef TSG_GO
  return check_launch("gate_gather_bwd");
}

/* workspace: GSB_GRID floats */
extern "C" size_t tsg_gate_score_bwd_workspace_bytes(void) { return ws_bytes((size_t)GSB_GRID, 4) + 256; }

extern "C" int tsg_gate_score_bwd(const float* dxo, const float* x, const float* score, const int64_t* perm,
                                  int64_t num_perm, int64_t num_nodes, int64_t F, float* dscore, float* dbias_score,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  TSG_REQUIRE(num_perm > 0 && num_nodes > 0 && F > 0 && F % 4 == 0, "gate_score_bwd: bad shape");
  TSG_REQUIRE(dxo && x && score && perm && dscore && dbias_score && workspace, "gate_score_bwd: null pointer");
  TSG_REQUIRE(((((uintptr_t)dxo) | ((uintptr_t)x)) & 15) == 0, "gate_score_bwd: operands must be 16-byte aligned");
  if (workspace_bytes < tsg_gate_score_bwd_workspace_bytes()) { set_error("gate_score_bwd: workspace too small"); return TSG_EWORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  unsigned* ticket = ticket_next();
  TSG_REQUIRE(ticket != nullptr, "gate_score_bwd: call tsg_init_device() once per device first (no counter pool)");
  cudaMemsetAsync(dscore, 0, (size_t)num_nodes * sizeof(float), st);      // dropped nodes
  const int F4 = (int)(F / 4);
  int lp = 1; while (lp < F4 && lp < 32) lp <<= 1;
  int grid = (int)((num_perm + (GSB_THREADS / lp) - 1) / (GSB_THREADS / lp));
  if (grid > GSB_GRID) grid = GSB_GRID;
#define TSG_GS(L) TSG_LAUNCH_PDL("gate_score_bwd", k_gate_score_bwd<L>, grid, GSB_THREADS, 0, st, (const float4*)dxo, (const float4*)x, score, perm, dscore, \
                                                                    (float*)workspace, num_perm, F4, dbias_score, ticket)
  switch (lp) {
    case 1: TSG_GS(1); break; case 2: TSG_GS(2); break; case 4: TSG_GS(4); break;
    case 8: TSG_GS(8); break; case 16: TSG_GS(16); break; default: TSG_GS(32); break;
  }
#undef TSG_GS
  return check_launch("gate_score_bwd");
}
