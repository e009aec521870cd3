// common.cuh -- shared device/host helpers for libtsg (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <stdlib.h>
#include <utility>
#include "../../include/tsg.h"

#ifndef TSG_NUM_SMS
#define TSG_NUM_SMS 148   // B200: 2 dies x 74 SMs; grids are sized in multiples of this
#endif

namespace tsg {

void set_error(const char* fmt, ...);

inline int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return TSG_ELAUNCH;
  }
  return TSG_OK;
}

#define TSG_REQUIRE(cond, ...)            \
  do {                                    \
    if (!(cond)) {                        \
      ::tsg::set_error(__VA_ARGS__);      \
      return TSG_EINVAL;                  \
    }                                     \
  } while (0)

#define TSG_LAUNCH_CHECK(what)                       \
  do {                                               \
    int _rc = ::tsg::check_launch(what);             \
    if (_rc != TSG_OK) return _rc;                   \
  } while (0)

// ------------------------------------------------------------------------------------------
// Programmatic dependent launch (PDL).  A kernel launched by launch_pdl may be scheduled while its predecessor in
// the stream is still draining, so the launch, the drain and the ramp-up of consecutive kernels overlap.  The rule
// that keeps this as safe as plain stream order: every CTA of such a kernel calls pdl_wait() unconditionally, before
// its first global load or store and before any early return, then pdl_launch_dependents().  pdl_wait() returns once
// the predecessor grid has completed and its memory is visible; since every kernel of the chain waits, completion is
// transitive and kernel i + 2 also sees kernel i's writes.  Launched with <<<>>> (other paths, graph capture), the
// two instructions do nothing.  Memsets, copies and library kernels between two launches stay ordinary stream order.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
static inline int launch_pdl(const char* what, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                             cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return TSG_ELAUNCH;
  }
  return TSG_OK;
}

#define TSG_LAUNCH_PDL(...)                          \
  do {                                               \
    int _rc = ::tsg::launch_pdl(__VA_ARGS__);        \
    if (_rc != TSG_OK) return _rc;                   \
  } while (0)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// bump allocator over the caller-provided workspace
struct Workspace {
  char* base; size_t size; size_t off;
  Workspace(void* p, size_t n) : base((char*)p), size(n), off(0) {}
  template <typename T> T* take(size_t count) {
    size_t bytes = align_up(count * sizeof(T), 256);
    if (off + bytes > size) { off = size + 1; return nullptr; }
    T* r = (T*)(base + off); off += bytes; return r;
  }
  bool ok() const { return off <= size; }
};
static inline size_t ws_bytes(size_t count, size_t elem) { return align_up(count * elem, 256); }

static inline int grid_for(int64_t work_items, int per_block, int max_waves = 64) {
  int64_t b = (work_items + per_block - 1) / per_block;
  int64_t cap = (int64_t)TSG_NUM_SMS * max_waves;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

__device__ __forceinline__ int64_t dev_count(int64_t cap, const int64_t* dev) {
  if (dev == nullptr) return cap;
  int64_t v = *dev;
  return v < cap ? (v < 0 ? 0 : v) : cap;
}

__device__ __forceinline__ int warp_incl_scan(int v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v += t;
  }
  return v;
}

// Block-wide exclusive scan of one int per thread (blockDim.x <= 1024, multiple of 32).
// Returns the exclusive prefix; *total receives the block sum.  smem: 33 ints.
__device__ __forceinline__ int block_excl_scan(int v, int* smem, int* total) {
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int inc = warp_incl_scan(v, lane);
  if (lane == 31) smem[w] = inc;
  __syncthreads();
  if (w == 0) {
    int s = lane < nw ? smem[lane] : 0;
    int si = warp_incl_scan(s, lane);
    smem[lane] = si - s;
    if (lane == 31) smem[32] = si;
  }
  __syncthreads();
  int r = inc - v + smem[w];
  *total = smem[32];
  __syncthreads();
  return r;
}

// ------------------------------------------------------------------------------------------
// Device-wide exclusive scan (reduce-then-scan, 3 launches, deterministic).
//   out[i] = sum_{j<i} f(j), i in [0, n];  out has n+1 entries.  f is a functor int(int64 j).
//   tile_ws: ceil(n / SCAN_TILE) + 1 ints.   OutT is int32_t or int64_t.
// ------------------------------------------------------------------------------------------
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

template <typename F>
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_tile_reduce(F f, int64_t n, int* tile_sum) {
  pdl_wait();
  pdl_launch_dependents();
  __shared__ int sm[33];
  int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
  int s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    int64_t i = base + k * SCAN_THREADS + threadIdx.x;
    if (i < n) s += f(i);
  }
  int tot;
  block_excl_scan(s, sm, &tot);
  if (threadIdx.x == 0) tile_sum[blockIdx.x] = tot;
}

template <typename OutT>
__global__ void __launch_bounds__(1024) k_scan_tile_sums(int* tile_sum, int num_tiles, OutT* out_total) {
  pdl_wait();
  pdl_launch_dependents();
  __shared__ int sm[33];
  long long carry = 0;
  for (int base = 0; base < num_tiles; base += 1024) {
    int i = base + threadIdx.x;
    int v = i < num_tiles ? tile_sum[i] : 0;
    int tot;
    int ex = block_excl_scan(v, sm, &tot);
    if (i < num_tiles) tile_sum[i] = (int)(carry + ex);
    carry += tot;
  }
  if (threadIdx.x == 0) *out_total = (OutT)carry;
}

template <typename F, typename OutT>
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_tile_scan(F f, int64_t n, const int* tile_off, OutT* out) {
  pdl_wait();
  pdl_launch_dependents();
  __shared__ int sm[33];
  __shared__ int vals[SCAN_TILE];
  int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    int j = k * SCAN_THREADS + threadIdx.x;
    int64_t i = base + j;
    vals[j] = i < n ? f(i) : 0;
  }
  __syncthreads();
  int loc[SCAN_ITEMS];
  int s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) { loc[k] = s; s += vals[threadIdx.x * SCAN_ITEMS + k]; }
  int tot;
  int ex = block_excl_scan(s, sm, &tot);
  int off = tile_off[blockIdx.x] + ex;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) vals[threadIdx.x * SCAN_ITEMS + k] = off + loc[k];
  __syncthreads();
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    int j = k * SCAN_THREADS + threadIdx.x;
    int64_t i = base + j;
    if (i < n) out[i] = (OutT)vals[j];
  }
}

static inline size_t scan_ws_ints(int64_t n) { return (size_t)((n + SCAN_TILE - 1) / SCAN_TILE + 1); }

template <typename F, typename OutT>
int exclusive_scan(F f, int64_t n, OutT* out, int* tile_ws, cudaStream_t st) {
  int num_tiles = (int)((n + SCAN_TILE - 1) / SCAN_TILE);
  if (num_tiles == 0) return launch_pdl("scan(empty)", k_scan_tile_sums<OutT>, 1, 1024, 0, st, tile_ws, 0, out);
  TSG_LAUNCH_PDL("scan(reduce)", k_scan_tile_reduce<F>, num_tiles, SCAN_THREADS, 0, st, f, n, tile_ws);
  TSG_LAUNCH_PDL("scan(tile sums)", k_scan_tile_sums<OutT>, 1, 1024, 0, st, tile_ws, num_tiles, out + n);
  return launch_pdl("scan", k_scan_tile_scan<F, OutT>, num_tiles, SCAN_THREADS, 0, st, f, n, (const int*)tile_ws, out);
}

// ------------------------------------------------------------------------------------------
// Second stage of every deterministic two-stage reduction: out[i] = sum_b part[b][i], b ascending
// inside 32 fixed slices (4 independent accumulators each, so the loads overlap) that are then combined
// in slice order.  Block = 32 entries x 32 slices; the order never depends on the grid or the device.
// ------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(1024)
k_partial_sum_final(const float* __restrict__ part, float* __restrict__ out0, int n0,
                    float* __restrict__ out1, int nb, int total) {
  pdl_wait();
  pdl_launch_dependents();
  __shared__ float sm[32][33];
  const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + x;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  if (i < total) {
    int b = y;
    for (; b + 96 < nb; b += 128) {
      s0 += part[(size_t)b * total + i];
      s1 += part[(size_t)(b + 32) * total + i];
      s2 += part[(size_t)(b + 64) * total + i];
      s3 += part[(size_t)(b + 96) * total + i];
    }
    for (; b < nb; b += 32) s0 += part[(size_t)b * total + i];
  }
  sm[y][x] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  if (y == 0 && i < total) {
    float t = sm[0][x];
#pragma unroll
    for (int k = 1; k < 32; ++k) t += sm[k][x];
    if (i < n0) { if (out0) out0[i] = t; }
    else if (out1) out1[i - n0] = t;
  }
}

// Same second stage fused into the producing kernel: every CTA calls this (all threads, no early exits) after it
// wrote its partial row; the CTA that draws the last ticket folds the rows in EXACTLY k_partial_sum_final's order, so
// the result does not depend on which CTA that is.  Saves one launch per reduction, but ONE CTA folding the partials
// is latency bound: measured 40 us for 1,184 x 64 partials (the stand-alone kernel: 5 us), so fused_tail_ok only
// admits reductions of at most 2,048 partial values (column sums of narrow matrices, scalar sums).  The ticket is a
// zero-initialised counter from ticket_next(); atomicInc wraps it back to zero for its next user.
__device__ __forceinline__ void partial_sum_tail(const float* part, float* out0, int n0, float* out1, int nb,
                                                 int total, unsigned* ticket) {
  __shared__ float t_sm[32][33];
  __shared__ int t_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) t_last = atomicInc(ticket, gridDim.x - 1) == gridDim.x - 1;
  __syncthreads();
  if (!t_last) return;
  __threadfence();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int cb = 0; cb < total; cb += 32) {
    const int i = cb + lane;
    for (int y = w; y < 32; y += nw) {
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
      if (i < total) {
        int b = y;
#pragma unroll 4
        for (; b + 96 < nb; b += 128) {
          s0 += __ldcg(part + (size_t)b * total + i);
          s1 += __ldcg(part + (size_t)(b + 32) * total + i);
          s2 += __ldcg(part + (size_t)(b + 64) * total + i);
          s3 += __ldcg(part + (size_t)(b + 96) * total + i);
        }
        for (; b < nb; b += 32) s0 += __ldcg(part + (size_t)b * total + i);
      }
      t_sm[y][lane] = (s0 + s1) + (s2 + s3);
    }
    __syncthreads();
    if (w == 0 && i < total) {
      float t = t_sm[0][lane];
#pragma unroll
      for (int k = 1; k < 32; ++k) t += t_sm[k][lane];
      if (i < n0) { if (out0) out0[i] = t; }
      else if (out1) out1[i - n0] = t;
    }
    __syncthreads();
  }
}

static inline bool fused_tail_ok(int64_t nb, int64_t total) {
  static const bool off = getenv("TSG_NO_FUSED_TAIL") != nullptr;
  return !off && nb * total <= 2048;
}

// A graph label read for a C-class head: outside [0, C) it is clamped for the read and sets TSG_SAG_LABEL_RANGE in `bad`
// (the caller ORs that into its status word).
__device__ __forceinline__ int clamp_label(int64_t y, int C, int& bad) {
  if (y < 0 || y >= C) { bad = TSG_SAG_LABEL_RANGE; return y < 0 ? 0 : C - 1; }
  return (int)y;
}

// Fixed-order totals over n rows on one CTA: thread t adds rows t, t + 1024, ... in order, then a fixed tree.
// sum_out = (sum v) / div; count_out = sum hit (int64).  Either output may be NULL.  (The losses and evaluation totals of
// K14 and K16.)
constexpr int SUM_THREADS = 1024;
static __global__ void __launch_bounds__(SUM_THREADS)
k_sum_fixed(const float* __restrict__ v, const int* __restrict__ hit, int n, float div, float* sum_out, int64_t* count_out) {
  pdl_wait();
  pdl_launch_dependents();
  __shared__ float sv[SUM_THREADS];
  __shared__ long long sc[SUM_THREADS];
  float s = 0.f;
  long long c = 0;
  for (int i = threadIdx.x; i < n; i += SUM_THREADS) {
    if (sum_out) s += v[i];
    if (count_out) c += hit[i];
  }
  sv[threadIdx.x] = s; sc[threadIdx.x] = c;
  __syncthreads();
  for (int o = SUM_THREADS / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) { sv[threadIdx.x] += sv[threadIdx.x + o]; sc[threadIdx.x] += sc[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    if (sum_out) *sum_out = sv[0] / div;
    if (count_out) *count_out = sc[0];
  }
}

unsigned* ticket_next();      // api.cu: a zeroed device counter from a per-device pool (nullptr if the pool cannot be made)

// k9_triplet.cu: tsg_triplet_fwd that also stores 1.0 to *dloss_seed (if given) from its last kernel
int triplet_fwd(const float* emb, const int64_t* trip, int64_t T, int64_t M, int64_t D, float margin, float eps,
                float* dpos, float* dneg, float* loss, float* dloss_seed, void* workspace, size_t workspace_bytes,
                void* stream);

static inline int launch_partial_sum_final(const float* part, float* out0, int n0, float* out1, int nb,
                                           int total, cudaStream_t st) {
  return launch_pdl("partial_sum_final", k_partial_sum_final, (total + 31) / 32, 1024, 0, st, part, out0, n0, out1, nb, total);
}

}  // namespace tsg
