// K2 -- CSR segment-sum SpMM   Y[r,:] = sum_p val[p] * H[colidx[p],:] (+bias) (ReLU)
//
// Replaces the gather -> mul -> scatter_add of PyG GCNConv.propagate (Code/sag/network.py:34,
// 38,42; Code/sag/layers.py:18) and torch.matmul(adj, x) of the dense GraphConv
// (Code/sage+gat+diffpool/encoders.py:33; Code/eigengcn/encoders.py:31) on a block-diagonal CSR.
//
// Gather kernel, no tensor cores (AI ~ 0.5 flop/B).  Common design of every variant below:
//   * a group of LPR lanes owns one destination row; each lane carries 4 consecutive features in
//     a float4 (128-bit loads/stores); LPR = F/4 rounded up to a power of two (8 lanes at F=32, 32
//     lanes at F=128) so one warp covers 32/LPR rows and every gathered row is one or more
//     fully-used 128-byte lines;
//   * the per-row loop is sequential in CSR order: deterministic, independent of the launch geometry;
//     with TSG_SPMM_EXACT the product is rounded before the add (__fmul_rn / __fadd_rn), which is
//     bit-identical to index_add_ in COO order;
//   * neighbours of a row live in the same small graph block, so the gathers hit L1/L2 and DRAM
//     sees ~compulsory traffic (H once, Y once, CSR once).
// k_spmm_g is the production kernel; k_spmm_vec4 (round-1 first cut) stays as the legacy baseline the
// profiles compare against (TSG_SPMM_LEGACY=1); k_spmm_scalar serves widths that are not multiples of 4.
#include "common.cuh"
#include <stdlib.h>

namespace tsg {

constexpr int SPMM_THREADS = 256;

template <int LPR, bool HAS_VAL>
__global__ void __launch_bounds__(SPMM_THREADS)
k_spmm_vec4(const int* __restrict__ rowptr, const int* __restrict__ colidx,
            const float* __restrict__ val, const float4* __restrict__ H,
            const float4* __restrict__ bias, float4* __restrict__ Y,
            int num_rows, int F4, int relu) {
  pdl_wait();
  pdl_launch_dependents();
  const int lane_in_row = threadIdx.x % LPR;
  // blocked assignment: CTA b owns rows [b*rpc, (b+1)*rpc) so the rows of one small graph (whose
  // neighbours are each other) are gathered through the same SM's L1
  const int rpc = (num_rows + gridDim.x - 1) / gridDim.x;
  const int r_begin = blockIdx.x * rpc;
  const int r_end = min(num_rows, r_begin + rpc);
  for (int r = r_begin + threadIdx.x / LPR; r < r_end; r += SPMM_THREADS / LPR) {
    const int s = __ldg(rowptr + r), t = __ldg(rowptr + r + 1);
    for (int f = lane_in_row; f < F4; f += LPR) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      int p = s;
      for (; p + 4 <= t; p += 4) {
        int c0 = __ldg(colidx + p), c1 = __ldg(colidx + p + 1);
        int c2 = __ldg(colidx + p + 2), c3 = __ldg(colidx + p + 3);
        float v0 = 1.f, v1 = 1.f, v2 = 1.f, v3 = 1.f;
        if (HAS_VAL) { v0 = __ldg(val + p); v1 = __ldg(val + p + 1); v2 = __ldg(val + p + 2); v3 = __ldg(val + p + 3); }
        float4 h0 = __ldg(H + (int64_t)c0 * F4 + f);
        float4 h1 = __ldg(H + (int64_t)c1 * F4 + f);
        float4 h2 = __ldg(H + (int64_t)c2 * F4 + f);
        float4 h3 = __ldg(H + (int64_t)c3 * F4 + f);
#define TSG_ACC(h, v)                                   \
        acc.x = __fadd_rn(acc.x, __fmul_rn(v, h.x));    \
        acc.y = __fadd_rn(acc.y, __fmul_rn(v, h.y));    \
        acc.z = __fadd_rn(acc.z, __fmul_rn(v, h.z));    \
        acc.w = __fadd_rn(acc.w, __fmul_rn(v, h.w));
        TSG_ACC(h0, v0) TSG_ACC(h1, v1) TSG_ACC(h2, v2) TSG_ACC(h3, v3)
      }
      for (; p < t; ++p) {
        int c0 = __ldg(colidx + p);
        float v0 = HAS_VAL ? __ldg(val + p) : 1.f;
        float4 h0 = __ldg(H + (int64_t)c0 * F4 + f);
        TSG_ACC(h0, v0)
      }
#undef TSG_ACC
      if (bias != nullptr) {
        float4 b = __ldg(bias + f);
        acc.x = __fadd_rn(acc.x, b.x); acc.y = __fadd_rn(acc.y, b.y);
        acc.z = __fadd_rn(acc.z, b.z); acc.w = __fadd_rn(acc.w, b.w);
      }
      if (relu) {
        acc.x = fmaxf(acc.x, 0.f); acc.y = fmaxf(acc.y, 0.f);
        acc.z = fmaxf(acc.z, 0.f); acc.w = fmaxf(acc.w, 0.f);
      }
      Y[(int64_t)r * F4 + f] = acc;
    }
  }
}

// scalar-feature variant (F not a multiple of 4, or F == 1 where LPR == 1 => thread per row)
template <int LPR, bool HAS_VAL>
__global__ void __launch_bounds__(SPMM_THREADS)
k_spmm_scalar(const int* __restrict__ rowptr, const int* __restrict__ colidx,
              const float* __restrict__ val, const float* __restrict__ H,
              const float* __restrict__ bias, float* __restrict__ Y,
              int num_rows, int F, int relu) {
  pdl_wait();
  pdl_launch_dependents();
  const int lane_in_row = threadIdx.x % LPR;
  // blocked assignment: CTA b owns rows [b*rpc, (b+1)*rpc) so the rows of one small graph (whose
  // neighbours are each other) are gathered through the same SM's L1
  const int rpc = (num_rows + gridDim.x - 1) / gridDim.x;
  const int r_begin = blockIdx.x * rpc;
  const int r_end = min(num_rows, r_begin + rpc);
  for (int r = r_begin + threadIdx.x / LPR; r < r_end; r += SPMM_THREADS / LPR) {
    const int s = __ldg(rowptr + r), t = __ldg(rowptr + r + 1);
    for (int f = lane_in_row; f < F; f += LPR) {
      float acc = 0.f;
      int p = s;
      for (; p + 4 <= t; p += 4) {
        int c0 = __ldg(colidx + p), c1 = __ldg(colidx + p + 1);
        int c2 = __ldg(colidx + p + 2), c3 = __ldg(colidx + p + 3);
        float v0 = 1.f, v1 = 1.f, v2 = 1.f, v3 = 1.f;
        if (HAS_VAL) { v0 = __ldg(val + p); v1 = __ldg(val + p + 1); v2 = __ldg(val + p + 2); v3 = __ldg(val + p + 3); }
        float h0 = __ldg(H + (int64_t)c0 * F + f), h1 = __ldg(H + (int64_t)c1 * F + f);
        float h2 = __ldg(H + (int64_t)c2 * F + f), h3 = __ldg(H + (int64_t)c3 * F + f);
        acc = __fadd_rn(acc, __fmul_rn(v0, h0));
        acc = __fadd_rn(acc, __fmul_rn(v1, h1));
        acc = __fadd_rn(acc, __fmul_rn(v2, h2));
        acc = __fadd_rn(acc, __fmul_rn(v3, h3));
      }
      for (; p < t; ++p) {
        float v0 = HAS_VAL ? __ldg(val + p) : 1.f;
        acc = __fadd_rn(acc, __fmul_rn(v0, __ldg(H + (int64_t)__ldg(colidx + p) * F + f)));
      }
      if (bias != nullptr) acc = __fadd_rn(acc, __ldg(bias + f));
      if (relu) acc = fmaxf(acc, 0.f);
      Y[(int64_t)r * F + f] = acc;
    }
  }
}

// ------------------------------------------------------------------------------------------
// Tiled variant: shared-memory staging of the small per-graph blocks (north-star design).
// A tile is a run of consecutive rows [tile_ptr[t], tile_ptr[t+1]) whose neighbours all lie inside
// the same run (a packed batch is block diagonal: tiles = whole graphs).  The CTA bulk-copies the
// tile's H rows (contiguous in memory: one coalesced cp.async stream), its CSR slice and rowptr
// slice into shared memory, then every gather is a 30-cycle LDS instead of a dependent global load.
// DRAM sees exactly the compulsory traffic; L2 sees H once.  The kernel VERIFIES containment
// (min / max of the staged column ids); a tile that is too large for the staging buffers or not
// self-contained takes the global-gather path, so correctness never depends on the caller's promise.
// Accumulation order per row is unchanged => still bit-identical to index_add_ order.
// ------------------------------------------------------------------------------------------
constexpr int TILED_SMEM_BYTES = 112 * 1024;      // 2 CTAs / SM
constexpr int TILED_MAX_NNZ = 3840;               // 30 KB of (colidx, val)
constexpr int TILED_MAX_ROWS_RP = 704;            // rowptr slice entries

__device__ __forceinline__ void cp_async_4(void* sdst, const void* gsrc) {
  unsigned a = (unsigned)__cvta_generic_to_shared(sdst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(a), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_16(void* sdst, const void* gsrc) {
  unsigned a = (unsigned)__cvta_generic_to_shared(sdst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(a), "l"(gsrc) : "memory");
}

constexpr int TILED_THREADS = 512;

template <int LPR, bool HAS_VAL>
__global__ void __launch_bounds__(TILED_THREADS, 2)
k_spmm_tiled(const int* __restrict__ rowptr, const int* __restrict__ colidx, const float* __restrict__ val,
             const float4* __restrict__ H, const float4* __restrict__ bias, float4* __restrict__ Y,
             const int64_t* __restrict__ tile_ptr, int num_tiles, int F4, int max_rows, int relu) {
  extern __shared__ __align__(16) unsigned char tsm[];
  int* s_off = reinterpret_cast<int*>(tsm);                         // (col - r0) * F4, pre-scaled
  float* s_val = reinterpret_cast<float*>(tsm + TILED_MAX_NNZ * 4);
  int* s_rp = reinterpret_cast<int*>(tsm + TILED_MAX_NNZ * 8);
  float4* s_H = reinterpret_cast<float4*>(tsm + TILED_MAX_NNZ * 8 + (TILED_MAX_ROWS_RP + 32) * 4);
  __shared__ int s_flag;
  const int lane_in_row = threadIdx.x % LPR;
  // this lane's bias columns stay in registers for the whole kernel (F4 <= 2*LPR is the common case)
  for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
    const int r0 = (int)tile_ptr[t], r1 = (int)tile_ptr[t + 1];
    const int rows = r1 - r0;
    if (rows <= 0) continue;
    const int p0 = __ldg(rowptr + r0), p1 = __ldg(rowptr + r1);
    const int nnz = p1 - p0;
    const bool fits = rows <= max_rows && rows <= TILED_MAX_ROWS_RP && nnz <= TILED_MAX_NNZ;
    if (threadIdx.x == 0) s_flag = 1;
    __syncthreads();                           // previous tile fully consumed; flag reset
    if (fits) {
      const float4* src = H + (size_t)r0 * F4;
      for (int i = threadIdx.x; i < rows * F4; i += TILED_THREADS) cp_async_16(s_H + i, src + i);
      if (HAS_VAL) for (int i = threadIdx.x; i < nnz; i += TILED_THREADS) cp_async_4(s_val + i, val + p0 + i);
      asm volatile("cp.async.commit_group;" ::: "memory");
      int bad = 0;
      for (int i = threadIdx.x; i < nnz; i += TILED_THREADS) {
        const int c = __ldg(colidx + p0 + i);
        bad |= (c < r0) | (c >= r1);
        s_off[i] = (c - r0) * F4;
      }
      for (int i = threadIdx.x; i <= rows; i += TILED_THREADS) s_rp[i] = __ldg(rowptr + r0 + i) - p0;
      if (bad) s_flag = 0;
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      __syncthreads();
    }
    const bool staged = fits && s_flag;
    if (staged) {
      for (int r = threadIdx.x / LPR; r < rows; r += TILED_THREADS / LPR) {
        const int s = s_rp[r], e = s_rp[r + 1];
        for (int f = lane_in_row; f < F4; f += LPR) {
          float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
          const float4* hb = s_H + f;
          int p = s;
#define TSG_TACC(h, v)                                                                          \
          acc.x = __fadd_rn(acc.x, __fmul_rn(v, h.x)); acc.y = __fadd_rn(acc.y, __fmul_rn(v, h.y)); \
          acc.z = __fadd_rn(acc.z, __fmul_rn(v, h.z)); acc.w = __fadd_rn(acc.w, __fmul_rn(v, h.w));
          for (; p + 2 <= e; p += 2) {
            const int o0 = s_off[p], o1 = s_off[p + 1];
            const float v0 = HAS_VAL ? s_val[p] : 1.f, v1 = HAS_VAL ? s_val[p + 1] : 1.f;
            const float4 h0 = hb[o0], h1 = hb[o1];
            TSG_TACC(h0, v0) TSG_TACC(h1, v1)
          }
          if (p < e) {
            const float v0 = HAS_VAL ? s_val[p] : 1.f;
            const float4 h0 = hb[s_off[p]];
            TSG_TACC(h0, v0)
          }
#undef TSG_TACC
          if (bias != nullptr) {
            float4 b = __ldg(bias + f);
            acc.x = __fadd_rn(acc.x, b.x); acc.y = __fadd_rn(acc.y, b.y);
            acc.z = __fadd_rn(acc.z, b.z); acc.w = __fadd_rn(acc.w, b.w);
          }
          if (relu) { acc.x = fmaxf(acc.x, 0.f); acc.y = fmaxf(acc.y, 0.f); acc.z = fmaxf(acc.z, 0.f); acc.w = fmaxf(acc.w, 0.f); }
          Y[(size_t)(r0 + r) * F4 + f] = acc;
        }
      }
    } else {                                   // global-gather path (same arithmetic, same order)
      for (int r = r0 + threadIdx.x / LPR; r < r1; r += TILED_THREADS / LPR) {
        const int s = __ldg(rowptr + r), e = __ldg(rowptr + r + 1);
        for (int f = lane_in_row; f < F4; f += LPR) {
          float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
          for (int p = s; p < e; ++p) {
            const float v = HAS_VAL ? __ldg(val + p) : 1.f;
            const float4 h = __ldg(H + (size_t)__ldg(colidx + p) * F4 + f);
            acc.x = __fadd_rn(acc.x, __fmul_rn(v, h.x)); acc.y = __fadd_rn(acc.y, __fmul_rn(v, h.y));
            acc.z = __fadd_rn(acc.z, __fmul_rn(v, h.z)); acc.w = __fadd_rn(acc.w, __fmul_rn(v, h.w));
          }
          if (bias != nullptr) {
            float4 b = __ldg(bias + f);
            acc.x = __fadd_rn(acc.x, b.x); acc.y = __fadd_rn(acc.y, b.y);
            acc.z = __fadd_rn(acc.z, b.z); acc.w = __fadd_rn(acc.w, b.w);
          }
          if (relu) { acc.x = fmaxf(acc.x, 0.f); acc.y = fmaxf(acc.y, 0.f); acc.z = fmaxf(acc.z, 0.f); acc.w = fmaxf(acc.w, 0.f); }
          Y[(size_t)r * F4 + f] = acc;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// k_spmm_g (default for 16-byte aligned widths): what the ncu captures of round 1 taught
// (profiles/r01b_spmm_variants.md):
//   * k_spmm_vec4 is NOT DRAM bound: an L2-resident problem runs no faster per row.  It is bound by
//     the L2 -> L1 fill traffic of gathers that miss L1 (487 MB for 175 MB of compulsory reads, L1 hit
//     rate 51 %).  Every H row is gathered ~6 times, always from rows of the same graph, so it should
//     miss once and hit five times; it does not because 8 small CTAs per SM walk 8 different graphs.
//     => 1024-thread CTAs: all 32 warps of a CTA sweep the SAME graph at the same time, an SM holds two
//     graph windows instead of eight (L1 hit rate 74 %, L2 -> L1 traffic halved);
//   * after that the L1 misses are the compulsory DRAM stream.  One thread per CTA asks the TMA engine
//     (`cp.async.bulk.prefetch.L2`) for the contiguous ranges the CTA is about to read: the H rows
//     `hdist` rows ahead and the colidx / val slices ~2 iterations ahead (position extrapolated from
//     the CTA's average row length: no dependent load).  Per-lane `prefetch.global.L2` did cut the
//     long-scoreboard stalls too but cost more issue slots / LSU queue than it won;
//   * lean loop: one IMAD.WIDE.U32 per gathered address (lane base + col * row_bytes), batches of 4
//     neighbours + ONE predicated batch for the 1..3 left over (no serial remainder chain).
// Accumulation is sequential in CSR order in every mode: run-to-run deterministic and independent of
// the launch geometry.  FMA = false rounds the product before the add (bit-identical to index_add_
// in COO order: flag TSG_SPMM_EXACT); FMA = true (default) fuses it: <= 1 ulp per term.
// Negative results kept out of the tree: warp-private cp.async staging of the CSR slice (153-200 us),
// a producer warp issuing per-line L2 prefetches (126 us), L1 evict_first / evict_last hints (+10 %),
// two float4 per lane with 4 lanes per row (fewer instructions, less memory parallelism: 123-160 us).
// ------------------------------------------------------------------------------------------
// TMA bulk prefetch into L2 of [p, p + bytes): start aligned down (stays inside the array: allocations are at least
// 16-byte aligned), end aligned DOWN too, so the request never reaches past the array's last byte and tsg_spmm needs no
// slack behind rowptr / colidx / val (a trailing partial 16 bytes is simply not prefetched)
__device__ __forceinline__ void bulk_prefetch_l2(const void* p, size_t bytes) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)15;
  const uintptr_t e = (reinterpret_cast<uintptr_t>(p) + bytes) & ~(uintptr_t)15;
  if (e <= a) return;
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" :: "l"(a), "r"((unsigned)(e - a)) : "memory");
}

// MODE bit 0: y . dot_vec epilogue; bit 1: H is a table indexed by row_label (compile-time: the plain kernel runs at its
// 32-register budget and the extra operands cost it 10 % when they were run-time branches)
template <int LPR, bool HAS_VAL, bool FMA, int THREADS, int MODE>
__global__ void __launch_bounds__(THREADS, 2048 / THREADS)
k_spmm_g(const int* __restrict__ rowptr, const int* __restrict__ colidx,
         const float* __restrict__ val, const float4* __restrict__ H,
         const float4* __restrict__ bias, float4* __restrict__ Y,
         int num_rows, int F4, int relu, int hdist,
         const float4* __restrict__ dot_vec, float* __restrict__ dot_out,
         const int* __restrict__ row_label = nullptr, int num_labels = 0) {
  pdl_wait();
  pdl_launch_dependents();
  // (MODE & 2): H is a [num_labels, F] TABLE and neighbour c contributes H[row_label[c]] -- conv1 on one-hot
  // node-label features (x W = W[label]) without ever materialising x W: the gathers hit an L1-resident table.
  constexpr int RPI = THREADS / LPR;              // rows per CTA iteration
  const int l = threadIdx.x % LPR;
  const int rpc = (num_rows + gridDim.x - 1) / gridDim.x;
  const int r_begin = blockIdx.x * rpc;
  const int r_end = min(num_rows, r_begin + rpc);
  const unsigned row_bytes = (unsigned)F4 * 16u;
  __shared__ int s_pf[2];                         // [0] CSR entries per CTA iteration (estimate), [1] nnz
  if (hdist > 0 && threadIdx.x == 0 && r_begin < r_end) {
    const int p_b = __ldg(rowptr + r_begin), p_e = __ldg(rowptr + r_end);
    const int nnz_end = __ldg(rowptr + num_rows);
    const int epi = (int)(((long long)(p_e - p_b) * RPI) / (r_end - r_begin)) + 1;
    s_pf[0] = epi; s_pf[1] = nnz_end;
    // head of this CTA's H window and CSR slice
    if (!(MODE & 2))
      bulk_prefetch_l2(reinterpret_cast<const char*>(H) + (size_t)r_begin * row_bytes,
                       (size_t)min(hdist, num_rows - r_begin) * row_bytes);
    const size_t n0 = (size_t)min(2 * epi, nnz_end - p_b) * 4;
    bulk_prefetch_l2(colidx + p_b, n0);
    if (HAS_VAL) bulk_prefetch_l2(val + p_b, n0);
  }
  for (int r = r_begin + threadIdx.x / LPR; r < r_end; r += RPI) {
    const int s = __ldg(rowptr + r), t = __ldg(rowptr + r + 1);
    if (hdist > 0 && threadIdx.x == 0) {
      const int hr = r + hdist;                                       // H rows [hr, hr + RPI)
      if (hr < num_rows && !(MODE & 2))
        bulk_prefetch_l2(reinterpret_cast<const char*>(H) + (size_t)hr * row_bytes,
                         (size_t)min(RPI, num_rows - hr) * row_bytes);
      const int epi = s_pf[0], nnz_end = s_pf[1];
      const long long q = (long long)s + 2LL * epi - (epi >> 2);      // CSR entries ~2 iterations ahead
      if (q < (long long)nnz_end) {
        const size_t n = (size_t)min((long long)epi + (epi >> 1), (long long)nnz_end - q) * 4;
        bulk_prefetch_l2(colidx + q, n);
        if (HAS_VAL) bulk_prefetch_l2(val + q, n);
      }
    }
    float dot = 0.f;                     // fused y[r, :] . dot_vec (host guarantees F4 <= LPR: one f per lane)
    for (int f = l; f < F4; f += LPR) {
      const char* Hl = reinterpret_cast<const char*>(H + f);
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#define TSG_LD(c) __ldg(reinterpret_cast<const float4*>(Hl + (size_t)(unsigned)(c) * row_bytes))
#define TSG_ACC(h, v)                                                                                   \
      if (FMA) { acc.x = fmaf(v, h.x, acc.x); acc.y = fmaf(v, h.y, acc.y);                              \
                 acc.z = fmaf(v, h.z, acc.z); acc.w = fmaf(v, h.w, acc.w); }                            \
      else { acc.x = __fadd_rn(acc.x, __fmul_rn(v, h.x)); acc.y = __fadd_rn(acc.y, __fmul_rn(v, h.y));  \
             acc.z = __fadd_rn(acc.z, __fmul_rn(v, h.z)); acc.w = __fadd_rn(acc.w, __fmul_rn(v, h.w)); }
      int p = s;
      for (; p + 4 <= t; p += 4) {
        int c0 = __ldg(colidx + p), c1 = __ldg(colidx + p + 1);
        int c2 = __ldg(colidx + p + 2), c3 = __ldg(colidx + p + 3);
        float v0 = 1.f, v1 = 1.f, v2 = 1.f, v3 = 1.f;
        if (HAS_VAL) { v0 = __ldg(val + p); v1 = __ldg(val + p + 1); v2 = __ldg(val + p + 2); v3 = __ldg(val + p + 3); }
        if ((MODE & 2)) {
          c0 = __ldg(row_label + c0); c1 = __ldg(row_label + c1); c2 = __ldg(row_label + c2); c3 = __ldg(row_label + c3);
          // a label outside the table is the all-zero one-hot row: contributes nothing
          if ((unsigned)c0 >= (unsigned)num_labels) { c0 = 0; v0 = 0.f; }
          if ((unsigned)c1 >= (unsigned)num_labels) { c1 = 0; v1 = 0.f; }
          if ((unsigned)c2 >= (unsigned)num_labels) { c2 = 0; v2 = 0.f; }
          if ((unsigned)c3 >= (unsigned)num_labels) { c3 = 0; v3 = 0.f; }
        }
        const float4 h0 = TSG_LD(c0), h1 = TSG_LD(c1), h2 = TSG_LD(c2), h3 = TSG_LD(c3);
        TSG_ACC(h0, v0) TSG_ACC(h1, v1) TSG_ACC(h2, v2) TSG_ACC(h3, v3)
      }
      const int rem = t - p;
      if (rem > 0) {                     // 1..3 left: one predicated batch
        int c0 = __ldg(colidx + p), c1 = 0, c2 = 0;
        float v0 = 1.f, v1 = 1.f, v2 = 1.f;
        if (HAS_VAL) v0 = __ldg(val + p);
        if (rem > 1) { c1 = __ldg(colidx + p + 1); if (HAS_VAL) v1 = __ldg(val + p + 1); }
        if (rem > 2) { c2 = __ldg(colidx + p + 2); if (HAS_VAL) v2 = __ldg(val + p + 2); }
        if ((MODE & 2)) {
          c0 = __ldg(row_label + c0);
          if ((unsigned)c0 >= (unsigned)num_labels) { c0 = 0; v0 = 0.f; }
          if (rem > 1) { c1 = __ldg(row_label + c1); if ((unsigned)c1 >= (unsigned)num_labels) { c1 = 0; v1 = 0.f; } }
          if (rem > 2) { c2 = __ldg(row_label + c2); if ((unsigned)c2 >= (unsigned)num_labels) { c2 = 0; v2 = 0.f; } }
        }
        const float4 h0 = TSG_LD(c0);
        float4 h1 = h0, h2 = h0;
        if (rem > 1) h1 = TSG_LD(c1);
        if (rem > 2) h2 = TSG_LD(c2);
        TSG_ACC(h0, v0)
        if (rem > 1) { TSG_ACC(h1, v1) }
        if (rem > 2) { TSG_ACC(h2, v2) }
      }
#undef TSG_ACC
#undef TSG_LD
      if (bias != nullptr) {
        const float4 b = __ldg(bias + f);
        acc.x = __fadd_rn(acc.x, b.x); acc.y = __fadd_rn(acc.y, b.y);
        acc.z = __fadd_rn(acc.z, b.z); acc.w = __fadd_rn(acc.w, b.w);
      }
      if (relu) {
        acc.x = fmaxf(acc.x, 0.f); acc.y = fmaxf(acc.y, 0.f);
        acc.z = fmaxf(acc.z, 0.f); acc.w = fmaxf(acc.w, 0.f);
      }
      Y[(size_t)r * F4 + f] = acc;
      if ((MODE & 1)) {          // same per-lane FMA chain and butterfly as k_linear_fwd_small: bit-identical
        const float4 w = __ldg(dot_vec + f);
        dot = fmaf(acc.x, w.x, dot); dot = fmaf(acc.y, w.y, dot);
        dot = fmaf(acc.z, w.z, dot); dot = fmaf(acc.w, w.w, dot);
      }
    }
    if ((MODE & 1)) {
      // the LPR lanes of a row leave the row loop together, so the group is converged here
      const unsigned gmask = LPR == 32 ? 0xffffffffu : (((1u << LPR) - 1u) << (((threadIdx.x & 31) / LPR) * LPR));
#pragma unroll
      for (int d = LPR / 2; d > 0; d >>= 1) dot += __shfl_xor_sync(gmask, dot, d, LPR);
      if (l == 0) dot_out[r] = dot;
    }
  }
}

// ------------------------------------------------------------------------------------------
// k_spmm_tma: whole-graph tiles staged in shared memory by the TMA engine, double buffered.
//
// k_spmm_g is bound by the latency of gathers that go through L1 tags / L2 (long_scoreboard 18 warp-cycles per
// issue; fewer instructions per neighbour made it SLOWER, more memory parallelism is what it lacks).  A packed
// batch is block diagonal, so a graph's rows only gather rows of the same graph: one CTA per SM keeps TWO tile
// stages (H rows, colidx / val slice, rowptr slice of one graph each) in shared memory; a producer warp
// fills stage i+1 with four `cp.async.bulk` copies on a tx-count mbarrier while 31 consumer warps compute
// stage i with every index load an LDS and every gather an LDS.128 (no tags, no first-touch stall);
// consumers release a stage by arriving on its `empty` mbarrier.  Graphs that do not fit a stage
// (rows > cap or nnz > cap) are processed by the same consumers straight from global memory.
// Arithmetic and order identical to k_spmm_g.  Requires 16 readable bytes of slack behind rowptr / colidx /
// val (the copies are rounded to 16 bytes) and tiles that are self-contained (guaranteed for CSRs built by
// K1b / K1c from a packed batch, which trap on an edge that leaves its graph).
// ------------------------------------------------------------------------------------------
constexpr int TT_THREADS = 1024;
constexpr int TT_CWARPS = TT_THREADS / 32 - 1;          // 31 consumer warps + 1 producer warp
constexpr int TT_STAGE_BYTES = 104 * 1024;
constexpr int TT_SPIN = 1 << 22;

__device__ __forceinline__ uint32_t tt_smem(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ bool tt_wait(uint32_t bar, uint32_t parity) {
  for (int spin = 0; spin < TT_SPIN; ++spin) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}\n" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (ok) return true;
  }
  __trap();        // hang guard: never continue on shared memory the copy has not filled
  return false;
}
__device__ __forceinline__ void tt_tma(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

struct TileHdr { int r0, rows, p0a, dr, staged; };     // dr = r0 - (r0 & ~3): offset of the tile's first rowptr entry

template <int LPR, bool HAS_VAL, bool FMA>
__global__ void __launch_bounds__(TT_THREADS, 1)
k_spmm_tma(const int* __restrict__ rowptr, const int* __restrict__ colidx, const float* __restrict__ val,
           const float4* __restrict__ H, const float4* __restrict__ bias, float4* __restrict__ Y,
           const int64_t* __restrict__ tile_ptr, int num_tiles, int F4, int row_cap, int nnz_cap, int relu,
           int* __restrict__ err) {
  extern __shared__ __align__(128) char tt_smem_buf[];
  __shared__ __align__(8) uint64_t bar_full[2], bar_empty[2];
  __shared__ TileHdr hdr[2];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned row_bytes = (unsigned)F4 * 16u;
  // stage layout: H rows | colidx | val | rowptr
  const int h_bytes = row_cap * (int)row_bytes;
  const int c_bytes = (nnz_cap + 8) * 4;
  const int r_off = h_bytes + 2 * c_bytes;
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(tt_smem(&bar_full[i])), "r"(1u) : "memory");
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(tt_smem(&bar_empty[i])), "r"((uint32_t)TT_CWARPS) : "memory");
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const int my_tiles = blockIdx.x < num_tiles ? (num_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  bool ok = true;
  if (warp == TT_CWARPS) {
    // ---------------- producer
    if (lane == 0) {
      // tile metadata (tile_ptr pair -> rowptr pair: two dependent global loads) is fetched one tile ahead so
      // its latency hides behind the wait for the stage
      auto meta = [&](int i, int& r0, int& r1, int& p0, int& p1) {
        r0 = r1 = p0 = p1 = 0;
        if (i < my_tiles) {
          const int t = blockIdx.x + i * gridDim.x;
          r0 = (int)tile_ptr[t]; r1 = (int)tile_ptr[t + 1];
          if (r1 > r0) { p0 = __ldg(rowptr + r0); p1 = __ldg(rowptr + r1); }
        }
      };
      int nr0, nr1, np0, np1;
      meta(0, nr0, nr1, np0, np1);
      for (int i = 0; i < my_tiles && ok; ++i) {
        const int s = i & 1;
        const int r0 = nr0, r1 = nr1, p0 = np0, p1 = np1;
        meta(i + 1, nr0, nr1, np0, np1);
        if (i >= 2) ok = tt_wait(tt_smem(&bar_empty[s]), (uint32_t)(((i >> 1) - 1) & 1));   // consumers left stage s
        const int rows = r1 - r0;
        const int p0a = p0 & ~3, r0a = r0 & ~3;
        const bool fits = rows > 0 && rows <= row_cap && (p1 - p0a) <= nnz_cap;
        hdr[s].r0 = r0; hdr[s].rows = rows; hdr[s].p0a = p0a; hdr[s].dr = r0 - r0a; hdr[s].staged = fits ? 1 : 0;
        const uint32_t bar = tt_smem(&bar_full[s]);
        if (fits) {
          char* st = tt_smem_buf + (size_t)s * TT_STAGE_BYTES;
          const uint32_t bh = (uint32_t)rows * row_bytes;
          const uint32_t bc = (uint32_t)(((p1 - p0a) * 4 + 15) & ~15);
          const uint32_t br = (uint32_t)(((r1 - r0a + 1) * 4 + 15) & ~15);
          asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                       :: "r"(bar), "r"(bh + bc * (HAS_VAL ? 2u : 1u) + br) : "memory");
          tt_tma(tt_smem(st), reinterpret_cast<const char*>(H) + (size_t)r0 * row_bytes, bh, bar);
          tt_tma(tt_smem(st + h_bytes), colidx + p0a, bc, bar);
          if (HAS_VAL) tt_tma(tt_smem(st + h_bytes + c_bytes), val + p0a, bc, bar);
          tt_tma(tt_smem(st + r_off), rowptr + r0a, br, bar);
        } else {
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");   // header only
        }
      }
    }
  } else {
    // ---------------- consumers: LPR lanes x float4 per row, 32 / LPR rows per warp
    const int l = lane % LPR, sub = lane / LPR;
    constexpr int RPW = 32 / LPR;
    const bool fok = l < F4;
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 b4 = zero4;
    if (bias != nullptr && fok) b4 = __ldg(bias + l);
    for (int i = 0; i < my_tiles && ok; ++i) {
      const int s = i & 1;
      ok = tt_wait(tt_smem(&bar_full[s]), (uint32_t)((i >> 1) & 1));
      const TileHdr h = hdr[s];
      const char* st = tt_smem_buf + (size_t)s * TT_STAGE_BYTES;
      const float4* sH = reinterpret_cast<const float4*>(st);
      const int* sC = reinterpret_cast<const int*>(st + h_bytes);
      const float* sV = reinterpret_cast<const float*>(st + h_bytes + c_bytes);
      const int* sR = reinterpret_cast<const int*>(st + r_off) + h.dr;
#define TSG_ACC(hh, v)                                                                                    \
      if (FMA) { acc.x = fmaf(v, hh.x, acc.x); acc.y = fmaf(v, hh.y, acc.y);                              \
                 acc.z = fmaf(v, hh.z, acc.z); acc.w = fmaf(v, hh.w, acc.w); }                            \
      else { acc.x = __fadd_rn(acc.x, __fmul_rn(v, hh.x)); acc.y = __fadd_rn(acc.y, __fmul_rn(v, hh.y));  \
             acc.z = __fadd_rn(acc.z, __fmul_rn(v, hh.z)); acc.w = __fadd_rn(acc.w, __fmul_rn(v, hh.w)); }
      for (int rl = warp * RPW + sub; rl < h.rows; rl += TT_CWARPS * RPW) {
        float4 acc = zero4;
        if (h.staged) {
          const int ps = sR[rl] - h.p0a, pe = sR[rl + 1] - h.p0a;
          const float4* Hl = sH + l - (size_t)h.r0 * F4;                  // gathers index by GLOBAL column id
          int p = ps;
          for (; p + 4 <= pe; p += 4) {
            const int c0 = sC[p], c1 = sC[p + 1], c2 = sC[p + 2], c3 = sC[p + 3];
            float v0 = 1.f, v1 = 1.f, v2 = 1.f, v3 = 1.f;
            if (HAS_VAL) { v0 = sV[p]; v1 = sV[p + 1]; v2 = sV[p + 2]; v3 = sV[p + 3]; }
            if (fok) {
              const float4 h0 = Hl[(size_t)c0 * F4], h1 = Hl[(size_t)c1 * F4], h2 = Hl[(size_t)c2 * F4], h3 = Hl[(size_t)c3 * F4];
              TSG_ACC(h0, v0) TSG_ACC(h1, v1) TSG_ACC(h2, v2) TSG_ACC(h3, v3)
            }
          }
          for (; p < pe; ++p) {
            const int c0 = sC[p];
            const float v0 = HAS_VAL ? sV[p] : 1.f;
            if (fok) { const float4 h0 = Hl[(size_t)c0 * F4]; TSG_ACC(h0, v0) }
          }
        } else {                                                            // oversize graph: global gathers
          const int r = h.r0 + rl;
          const int ps = __ldg(rowptr + r), pe = __ldg(rowptr + r + 1);
          for (int p = ps; p < pe; ++p) {
            const float v0 = HAS_VAL ? __ldg(val + p) : 1.f;
            if (fok) { const float4 h0 = __ldg(H + (size_t)__ldg(colidx + p) * F4 + l); TSG_ACC(h0, v0) }
          }
        }
#undef TSG_ACC
        if (bias != nullptr) {
          acc.x = __fadd_rn(acc.x, b4.x); acc.y = __fadd_rn(acc.y, b4.y);
          acc.z = __fadd_rn(acc.z, b4.z); acc.w = __fadd_rn(acc.w, b4.w);
        }
        if (relu) { acc.x = fmaxf(acc.x, 0.f); acc.y = fmaxf(acc.y, 0.f); acc.z = fmaxf(acc.z, 0.f); acc.w = fmaxf(acc.w, 0.f); }
        if (fok) Y[(size_t)(h.r0 + rl) * F4 + l] = acc;
      }
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(tt_smem(&bar_empty[s])) : "memory");
    }
  }
  if (!ok) atomicExch(err, 1);
}

static int env_int(const char* name, int dflt) {
  const char* s = getenv(name);
  return s ? atoi(s) : dflt;
}

template <bool HAS_VAL>
static int launch_spmm(const int* rowptr, const int* colidx, const float* val, const float* H,
                       const float* bias, float* Y, int64_t N, int64_t F, int relu, bool exact, cudaStream_t st,
                       const float* dot_vec = nullptr, float* dot_out = nullptr, bool* dot_done = nullptr,
                       const int* row_label = nullptr, int num_labels = 0) {
  if (dot_done) *dot_done = false;
  bool vec = (F % 4 == 0) && (((uintptr_t)H & 15) == 0) && (((uintptr_t)Y & 15) == 0) &&
             (bias == nullptr || ((uintptr_t)bias & 15) == 0);
  if (vec) {
    int F4 = (int)(F / 4);
    int lpr = 1; while (lpr < F4 && lpr < 32) lpr <<= 1;
    // tuning knobs (defaults = measured best on B200, DD-shape level 1): TSG_SPMM_LEGACY=1 selects k_spmm_vec4
    static const bool legacy = env_int("TSG_SPMM_LEGACY", 0) != 0;
    static const int hdist = env_int("TSG_SPMM_HDIST", 128);
    static const int ctas_per_sm_1024 = env_int("TSG_SPMM_CTAS", 2);
    if (legacy && row_label == nullptr) {
      int grid = grid_for(N, SPMM_THREADS / lpr, 32);
#define TSG_GO(L) TSG_LAUNCH_PDL("spmm", k_spmm_vec4<L, HAS_VAL>, grid, SPMM_THREADS, 0, st, rowptr, colidx, val, (const float4*)H, (const float4*)bias, (float4*)Y, (int)N, F4, relu)
      switch (lpr) {
        case 1: TSG_GO(1); break; case 2: TSG_GO(2); break; case 4: TSG_GO(4); break;
        case 8: TSG_GO(8); break; case 16: TSG_GO(16); break; default: TSG_GO(32); break;
      }
#undef TSG_GO
    } else {
      // 1024-thread CTAs once every SM gets two of them; smaller problems use 256-thread CTAs so the
      // grid still covers the machine
      const bool big = N >= (int64_t)TSG_NUM_SMS * 2 * (1024 / lpr) * 2;
      const int threads = big ? 1024 : 256;
      const int rpi = threads / lpr;
      int g = (int)((N + rpi - 1) / rpi);
      const int cap = big ? TSG_NUM_SMS * ctas_per_sm_1024 : TSG_NUM_SMS * 32;
      if (g > cap) g = cap;
      // y . dot_vec in the epilogue when one lane owns one float4 of the row (F <= 128) -- the shape k_linear_fwd_small
      // would take; otherwise the caller runs K3 afterwards
      const bool fuse_dot = dot_vec && dot_out && F4 <= lpr && (((uintptr_t)dot_vec) & 15) == 0;
      const float4* dv = fuse_dot ? (const float4*)dot_vec : nullptr;
      if (dot_done) *dot_done = fuse_dot;
      const int mode = (dv ? 1 : 0) | (row_label ? 2 : 0);
#define TSG_GM(L, FM, T, M) TSG_LAUNCH_PDL("spmm", k_spmm_g<L, HAS_VAL, FM, T, M>, g, T, 0, st, rowptr, colidx, val, (const float4*)H, (const float4*)bias, (float4*)Y, (int)N, F4, relu, big ? hdist : 0, dv, dot_out, row_label, num_labels)
#define TSG_G(L, FM, T) { if (mode == 0) TSG_GM(L, FM, T, 0); else if (mode == 1) TSG_GM(L, FM, T, 1); else if (mode == 2) TSG_GM(L, FM, T, 2); else TSG_GM(L, FM, T, 3); }
#define TSG_GT(L, FM) if (big) TSG_G(L, FM, 1024) else TSG_G(L, FM, 256)
#define TSG_GV(L) if (exact) { TSG_GT(L, false) } else { TSG_GT(L, true) }
      switch (lpr) {
        case 1: TSG_GV(1) break; case 2: TSG_GV(2) break; case 4: TSG_GV(4) break;
        case 8: TSG_GV(8) break; case 16: TSG_GV(16) break; default: TSG_GV(32) break;
      }
#undef TSG_GV
#undef TSG_GT
#undef TSG_G
#undef TSG_GM
    }
  } else {
    int lpr = 1; while (lpr < F && lpr < 32) lpr <<= 1;
    int rows_per_block = SPMM_THREADS / lpr;
    int grid = grid_for(N, rows_per_block, 32);
#define TSG_GO(L) TSG_LAUNCH_PDL("spmm", k_spmm_scalar<L, HAS_VAL>, grid, SPMM_THREADS, 0, st, rowptr, colidx, val, H, bias, Y, (int)N, (int)F, relu)
    switch (lpr) {
      case 1: TSG_GO(1); break; case 2: TSG_GO(2); break; case 4: TSG_GO(4); break;
      case 8: TSG_GO(8); break; case 16: TSG_GO(16); break; default: TSG_GO(32); break;
    }
#undef TSG_GO
  }
  return check_launch("spmm");
}

// ------------------------------------------------------------------------------------------
// ReLU backward + bias gradient (column sum), deterministic two-stage reduction.
//   stage 1: block b sums rows [b*RPB, (b+1)*RPB) per feature column into part[b, F]
//   stage 2: one block sums part[:, f] sequentially in block order.
// ------------------------------------------------------------------------------------------
constexpr int CS_THREADS = 256;
constexpr int CS_MAX_BLOCKS = TSG_NUM_SMS * 8;

__global__ void __launch_bounds__(CS_THREADS)
k_relu_bwd_colsum(const float* __restrict__ dY, const float* __restrict__ Y, float* __restrict__ dYm,
                  float* __restrict__ part, int64_t N, int F, int64_t rows_per_block,
                  const float* __restrict__ row_scale, const float* __restrict__ col_vec,
                  float* __restrict__ dbias, unsigned* ticket) {
  // thread layout: column f = threadIdx.x % Fp, row lane = threadIdx.x / Fp  (Fp = cols per pass)
  extern __shared__ float sm[];
  int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  int64_t r1 = r0 + rows_per_block; if (r1 > N) r1 = N;
  int cols = F < CS_THREADS ? F : CS_THREADS;
  int rl = CS_THREADS / cols;             // row lanes
  for (int fb = 0; fb < F; fb += cols) {
    int f = fb + threadIdx.x % cols;
    int lane_r = threadIdx.x / cols;
    float acc = 0.f;
    if (lane_r < rl && f < F) {
      const float cv = col_vec ? col_vec[f] : 0.f;
      for (int64_t r = r0 + lane_r; r < r1; r += rl) {
        float g = dY[r * F + f];
        if (row_scale) g = __fadd_rn(g, __fmul_rn(row_scale[r], cv));
        if (Y != nullptr && !(Y[r * F + f] > 0.f)) g = 0.f;
        if (dYm != nullptr) dYm[r * F + f] = g;
        acc += g;
      }
    }
    sm[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x < cols && fb + threadIdx.x < F) {
      float s = 0.f;
      for (int k = 0; k < rl; ++k) s += sm[k * cols + threadIdx.x];
      part[(int64_t)blockIdx.x * F + fb + threadIdx.x] = s;
    }
    __syncthreads();
  }
  if (ticket) partial_sum_tail(part, dbias, F, nullptr, gridDim.x, F, ticket);
}

// float4 variant for F % 4 == 0 (the scalar kernel above ran at 2.8 TB/s): thread = (row lane, group of 4
// columns), two rows in flight per iteration; same two-stage reduction (per-thread partial -> fixed-order sum over
// the row lanes of the block -> k_partial_sum_final over blocks).
__global__ void __launch_bounds__(CS_THREADS)
k_relu_bwd_colsum_v4(const float4* __restrict__ dY, const float4* __restrict__ Y, float4* __restrict__ dYm,
                     float* __restrict__ part, int64_t N, int F4, int64_t rows_per_block,
                     const float* __restrict__ row_scale, const float4* __restrict__ col_vec,
                     float* __restrict__ dbias, unsigned* ticket) {
  extern __shared__ float4 sm4[];
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  int64_t r1 = r0 + rows_per_block; if (r1 > N) r1 = N;
  const int cols = F4 < CS_THREADS ? F4 : CS_THREADS;
  const int rl = CS_THREADS / cols;
  for (int fb = 0; fb < F4; fb += cols) {
    const int f = fb + threadIdx.x % cols;
    const int lane_r = threadIdx.x / cols;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (lane_r < rl && f < F4) {
      const float4 cv = col_vec ? col_vec[f] : make_float4(0.f, 0.f, 0.f, 0.f);
      auto one = [&](int64_t r) {
        float4 g = dY[r * F4 + f];
        if (row_scale) {
          const float rs = row_scale[r];
          g.x = __fadd_rn(g.x, __fmul_rn(rs, cv.x)); g.y = __fadd_rn(g.y, __fmul_rn(rs, cv.y));
          g.z = __fadd_rn(g.z, __fmul_rn(rs, cv.z)); g.w = __fadd_rn(g.w, __fmul_rn(rs, cv.w));
        }
        if (Y != nullptr) {
          const float4 y = Y[r * F4 + f];
          if (!(y.x > 0.f)) g.x = 0.f;
          if (!(y.y > 0.f)) g.y = 0.f;
          if (!(y.z > 0.f)) g.z = 0.f;
          if (!(y.w > 0.f)) g.w = 0.f;
        }
        if (dYm != nullptr) dYm[r * F4 + f] = g;
        acc.x += g.x; acc.y += g.y; acc.z += g.z; acc.w += g.w;
      };
      int64_t r = r0 + lane_r;
      for (; r + rl < r1; r += 2 * rl) { one(r); one(r + rl); }
      if (r < r1) one(r);
    }
    sm4[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x < cols && fb + threadIdx.x < F4) {
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int k = 0; k < rl; ++k) { const float4 v = sm4[k * cols + threadIdx.x]; t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w; }
      reinterpret_cast<float4*>(part + (int64_t)blockIdx.x * F4 * 4)[fb + threadIdx.x] = t;
    }
    __syncthreads();
  }
  if (ticket) partial_sum_tail(part, dbias, F4 * 4, nullptr, gridDim.x, F4 * 4, ticket);
}

// Backward of one SAGPool level's conv output h, fused (K10 executor, F % 4 == 0):
//   dh[r]   = inv[r] >= 0 ? dxo[inv[r]] * tanh(score[r]) : 0        (gate backward, layers.py:21 -- never written)
//   g       = dh + dsw[r] * ws                                      (score layer's x-gradient, rank 1)
//   dhm     = g where h > 0 else 0                                  (ReLU backward; the only big write)
//   dbias   = column sum of dhm                                     (conv bias gradient)
//   dws     = column sum of h * dsw[r]                              (score layer's weight gradient h^T dsw)
// Same per-element arithmetic as k_gate_gather_bwd_v4 followed by k_relu_bwd_colsum_v4 (dhm and dbias are
// bit-identical to that sequence); dws replaces a separate pass over h (k_linear_bwd_weight_small) and is summed in
// this kernel's fixed row order.  Saves, per level, one write + one read of dh and one read of h.
template <int CB_ROWS>
__global__ void __launch_bounds__(CS_THREADS)
k_sag_conv_bwd_v4(const float4* __restrict__ dxo, const int* __restrict__ inv, const float* __restrict__ score,
                  const float4* __restrict__ Y, const float* __restrict__ dsw, const float4* __restrict__ ws4,
                  float4* __restrict__ dYm, float* __restrict__ part, int64_t N, int F4, int64_t rows_per_block,
                  float* __restrict__ dbias, float* __restrict__ dws, unsigned* ticket) {
  pdl_wait();
  pdl_launch_dependents();
  extern __shared__ float4 sm4[];                       // [2][CS_THREADS]
  int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  int64_t r1 = r0 + rows_per_block; if (r1 > N) r1 = N;
  const int cols = F4 < CS_THREADS ? F4 : CS_THREADS;
  const int rl = CS_THREADS / cols;
  const int F = F4 * 4;
  for (int fb = 0; fb < F4; fb += cols) {
    const int f = fb + threadIdx.x % cols;
    const int lane_r = threadIdx.x / cols;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), acw = make_float4(0.f, 0.f, 0.f, 0.f);
    if (lane_r < rl && f < F4) {
      const float4 cv = ws4[f];
      // CB_ROWS rows per thread in flight: all index / scale / h loads first, then the dependent score -> tanh and
      // inv -> dxo gathers, then the arithmetic (rows are still accumulated in increasing order)
      for (int64_t rb = r0 + lane_r; rb < r1; rb += (int64_t)CB_ROWS * rl) {
        int m[CB_ROWS]; float rs[CB_ROWS], t[CB_ROWS]; float4 y[CB_ROWS], go[CB_ROWS];
#pragma unroll
        for (int u = 0; u < CB_ROWS; ++u) {
          const int64_t r = rb + (int64_t)u * rl;
          const bool ok = r < r1;
          m[u] = ok ? __ldg(inv + r) : -2;
          rs[u] = ok ? __ldg(dsw + r) : 0.f;
          y[u] = ok ? Y[r * F4 + f] : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < CB_ROWS; ++u) {
          const int64_t r = rb + (int64_t)u * rl;
          t[u] = 0.f; go[u] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (m[u] >= 0) { t[u] = __ldg(score + r); go[u] = __ldg(dxo + (int64_t)m[u] * F4 + f); }
        }
#pragma unroll
        for (int u = 0; u < CB_ROWS; ++u) {
          if (m[u] == -2) continue;
          const int64_t r = rb + (int64_t)u * rl;
          float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
          if (m[u] >= 0) {
            const float th = tanhf(t[u]);
            g = make_float4(go[u].x * th, go[u].y * th, go[u].z * th, go[u].w * th);
          }
          g.x = __fadd_rn(g.x, __fmul_rn(rs[u], cv.x)); g.y = __fadd_rn(g.y, __fmul_rn(rs[u], cv.y));
          g.z = __fadd_rn(g.z, __fmul_rn(rs[u], cv.z)); g.w = __fadd_rn(g.w, __fmul_rn(rs[u], cv.w));
          if (!(y[u].x > 0.f)) g.x = 0.f;
          if (!(y[u].y > 0.f)) g.y = 0.f;
          if (!(y[u].z > 0.f)) g.z = 0.f;
          if (!(y[u].w > 0.f)) g.w = 0.f;
          __stcs(dYm + r * F4 + f, g);
          acc.x += g.x; acc.y += g.y; acc.z += g.z; acc.w += g.w;
          acw.x = fmaf(y[u].x, rs[u], acw.x); acw.y = fmaf(y[u].y, rs[u], acw.y);
          acw.z = fmaf(y[u].z, rs[u], acw.z); acw.w = fmaf(y[u].w, rs[u], acw.w);
        }
      }
    }
    sm4[threadIdx.x] = acc;
    sm4[CS_THREADS + threadIdx.x] = acw;
    __syncthreads();
    if (threadIdx.x < 2 * cols && fb + threadIdx.x % cols < F4) {
      const int which = threadIdx.x / cols, c = threadIdx.x % cols;       // 0: dbias partial, 1: dws partial
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int k = 0; k < rl; ++k) { const float4 v = sm4[which * CS_THREADS + k * cols + c]; t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w; }
      reinterpret_cast<float4*>(part + (int64_t)blockIdx.x * 2 * F + (int64_t)which * F)[fb + c] = t;
    }
    __syncthreads();
  }
  if (ticket) partial_sum_tail(part, dbias, F, dws, gridDim.x, 2 * F, ticket);
}

}  // namespace tsg

using namespace tsg;

extern "C" int tsg_spmm(const int32_t* rowptr, const int32_t* colidx, const float* val,
                        const float* H, const float* bias, float* Y,
                        int64_t num_rows, int64_t feat, int flags, void* stream) {
  TSG_REQUIRE(num_rows >= 0 && feat > 0, "spmm: bad shape rows=%lld feat=%lld", (long long)num_rows, (long long)feat);
  TSG_REQUIRE(num_rows < (int64_t)0x7fffffff, "spmm: too many rows");
  if (num_rows == 0) return TSG_OK;
  TSG_REQUIRE(rowptr && colidx && H && Y, "spmm: null pointer");
  int relu = (flags & TSG_SPMM_RELU) ? 1 : 0;
  const bool exact = (flags & TSG_SPMM_EXACT) != 0;
  cudaStream_t st = (cudaStream_t)stream;
  return val ? launch_spmm<true>(rowptr, colidx, val, H, bias, Y, num_rows, feat, relu, exact, st)
             : launch_spmm<false>(rowptr, colidx, val, H, bias, Y, num_rows, feat, relu, exact, st);
}


extern "C" int tsg_spmm_tiled(const int32_t* rowptr, const int32_t* colidx, const float* val,
                              const float* H, const float* bias, float* Y, const int64_t* tile_ptr,
                              int64_t num_tiles, int64_t num_rows, int64_t feat, int flags, void* stream) {
  TSG_REQUIRE(num_rows >= 0 && feat > 0 && num_tiles >= 0, "spmm_tiled: bad shape");
  TSG_REQUIRE(num_rows < (int64_t)0x7fffffff && num_tiles < (int64_t)0x7fffffff, "spmm_tiled: too large");
  if (num_rows == 0 || num_tiles == 0) return TSG_OK;
  TSG_REQUIRE(rowptr && colidx && H && Y && tile_ptr, "spmm_tiled: null pointer");
  bool vec = (feat % 4 == 0) && (((uintptr_t)H & 15) == 0) && (((uintptr_t)Y & 15) == 0) &&
             (bias == nullptr || ((uintptr_t)bias & 15) == 0);
  if (!vec) return tsg_spmm(rowptr, colidx, val, H, bias, Y, num_rows, feat, flags, stream);   // scalar widths: untiled kernel
  cudaStream_t st = (cudaStream_t)stream;
  int relu = (flags & TSG_SPMM_RELU) ? 1 : 0;
  int F4 = (int)(feat / 4);
  int lpr = 1; while (lpr < F4 && lpr < 32) lpr <<= 1;
  size_t h_bytes = TILED_SMEM_BYTES - (size_t)TILED_MAX_NNZ * 8 - (TILED_MAX_ROWS_RP + 32) * 4;
  int max_rows = (int)(h_bytes / ((size_t)F4 * 16));
  int grid = (int)(num_tiles < TSG_NUM_SMS * 2 ? num_tiles : TSG_NUM_SMS * 2);
#define TSG_GO(L, V)                                                                                         \
  { cudaFuncSetAttribute(k_spmm_tiled<L, V>, cudaFuncAttributeMaxDynamicSharedMemorySize, TILED_SMEM_BYTES);   \
    k_spmm_tiled<L, V><<<grid, TILED_THREADS, TILED_SMEM_BYTES, st>>>(rowptr, colidx, val, (const float4*)H,    \
        (const float4*)bias, (float4*)Y, tile_ptr, (int)num_tiles, F4, max_rows, relu); }
#define TSG_SW(V) switch (lpr) { case 1: TSG_GO(1, V) break; case 2: TSG_GO(2, V) break; case 4: TSG_GO(4, V) break; \
                                 case 8: TSG_GO(8, V) break; case 16: TSG_GO(16, V) break; default: TSG_GO(32, V) break; }
  if (val) { TSG_SW(true) } else { TSG_SW(false) }
#undef TSG_SW
#undef TSG_GO
  return check_launch("spmm_tiled");
}

extern "C" int tsg_spmm_tma(const int32_t* rowptr, const int32_t* colidx, const float* val,
                            const float* H, const float* bias, float* Y, const int64_t* tile_ptr,
                            int64_t num_tiles, int64_t num_rows, int64_t feat, int flags, int32_t* status_dev,
                            void* stream) {
  TSG_REQUIRE(num_rows >= 0 && feat > 0 && num_tiles >= 0, "spmm_tma: bad shape");
  TSG_REQUIRE(num_rows < (int64_t)0x7fffffff && num_tiles < (int64_t)0x7fffffff, "spmm_tma: too large");
  if (num_rows == 0 || num_tiles == 0) return TSG_OK;
  TSG_REQUIRE(rowptr && colidx && H && Y && tile_ptr && status_dev, "spmm_tma: null pointer");
  const bool ok_shape = (feat % 4 == 0) && feat <= 32 &&
                        ((((uintptr_t)H) | ((uintptr_t)Y) | ((uintptr_t)rowptr) | ((uintptr_t)colidx) | ((uintptr_t)val) |
                          ((uintptr_t)bias)) & 15) == 0;
  if (!ok_shape) return tsg_spmm(rowptr, colidx, val, H, bias, Y, num_rows, feat, flags, stream);
  cudaStream_t st = (cudaStream_t)stream;
  const int relu = (flags & TSG_SPMM_RELU) ? 1 : 0;
  const bool exact = (flags & TSG_SPMM_EXACT) != 0;
  const int F4 = (int)(feat / 4);
  int lpr = 1; while (lpr < F4) lpr <<= 1;
  // stage budget: H rows + (colidx, val) + rowptr; ~6.5 entries per row => split the budget accordingly
  const int row_bytes = F4 * 16;
  const int row_cap = (TT_STAGE_BYTES - 4096) / (row_bytes + 7 * 8 + 4) & ~3;
  const int nnz_cap = ((TT_STAGE_BYTES - 1024 - row_cap * (row_bytes + 4)) / 8 - 8) & ~3;
  const size_t smem = 2 * (size_t)TT_STAGE_BYTES;
  int grid = (int)(num_tiles < TSG_NUM_SMS ? num_tiles : TSG_NUM_SMS);
#define TSG_TT(L, V, FM)                                                                                          \
  { cudaFuncSetAttribute(k_spmm_tma<L, V, FM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);              \
    k_spmm_tma<L, V, FM><<<grid, TT_THREADS, smem, st>>>(rowptr, colidx, val, (const float4*)H, (const float4*)bias, \
        (float4*)Y, tile_ptr, (int)num_tiles, F4, row_cap, nnz_cap, relu, status_dev); }
#define TSG_TTF(L, V) if (exact) TSG_TT(L, V, false) else TSG_TT(L, V, true)
#define TSG_TTV(L) if (val) { TSG_TTF(L, true) } else { TSG_TTF(L, false) }
  switch (lpr) { case 1: TSG_TTV(1) break; case 2: TSG_TTV(2) break; case 4: TSG_TTV(4) break; default: TSG_TTV(8) break; }
#undef TSG_TTV
#undef TSG_TTF
#undef TSG_TT
  return check_launch("spmm_tma");
}

static int colsum_blocks(int64_t N) {
  int64_t nb = (N + 255) / 256;
  if (nb > CS_MAX_BLOCKS) nb = CS_MAX_BLOCKS;
  if (nb < 1) nb = 1;
  return (int)nb;
}

extern "C" size_t tsg_colsum_workspace_bytes(int64_t N, int64_t F) {
  return ws_bytes((size_t)colsum_blocks(N) * (size_t)F, 4) + 256;
}

extern "C" int tsg_relu_bwd_colsum_rank1(const float* dY, const float* Y, const float* row_scale, const float* col_vec,
                                         float* dYm, float* dbias, int64_t N, int64_t F,
                                         void* workspace, size_t workspace_bytes, void* stream);

extern "C" int tsg_relu_bwd_colsum(const float* dY, const float* Y, float* dYm, float* dbias,
                                   int64_t N, int64_t F, void* workspace, size_t workspace_bytes,
                                   void* stream) {
  return tsg_relu_bwd_colsum_rank1(dY, Y, nullptr, nullptr, dYm, dbias, N, F, workspace, workspace_bytes, stream);
}

extern "C" int tsg_relu_bwd_colsum_rank1(const float* dY, const float* Y, const float* row_scale, const float* col_vec,
                                         float* dYm, float* dbias, int64_t N, int64_t F,
                                         void* workspace, size_t workspace_bytes, void* stream) {
  TSG_REQUIRE(N >= 0 && F > 0 && dY && dbias, "relu_bwd_colsum: bad arguments");
  TSG_REQUIRE((row_scale == nullptr) == (col_vec == nullptr), "relu_bwd_colsum: row_scale and col_vec go together");
  cudaStream_t st = (cudaStream_t)stream;
  if (workspace_bytes < tsg_colsum_workspace_bytes(N, F)) { set_error("relu_bwd_colsum: workspace too small"); return TSG_EWORKSPACE; }
  float* part = (float*)workspace;
  int nb = colsum_blocks(N);
  int64_t rpb = (N + nb - 1) / nb; if (rpb < 1) rpb = 1;
  const bool v4 = (F % 4 == 0) && ((((uintptr_t)dY) | ((uintptr_t)Y) | ((uintptr_t)dYm) | ((uintptr_t)col_vec) | ((uintptr_t)part)) & 15) == 0;
  unsigned* ticket = fused_tail_ok(nb, F) ? ticket_next() : nullptr;      // second stage inside the kernel when small
  if (v4)
    k_relu_bwd_colsum_v4<<<nb, CS_THREADS, CS_THREADS * sizeof(float4), st>>>((const float4*)dY, (const float4*)Y, (float4*)dYm, part,
                                                                            N, (int)(F / 4), rpb, row_scale, (const float4*)col_vec,
                                                                            dbias, ticket);
  else
    k_relu_bwd_colsum<<<nb, CS_THREADS, CS_THREADS * sizeof(float), st>>>(dY, Y, dYm, part, N, (int)F, rpb, row_scale, col_vec,
                                                                        dbias, ticket);
  if (!ticket) { int rc = launch_partial_sum_final(part, dbias, (int)F, nullptr, nb, (int)F, st); if (rc) return rc; }
  return check_launch("relu_bwd_colsum");
}

/* K10's fused level backward (see k_sag_conv_bwd_v4).  Requires F % 4 == 0 and 16-byte aligned matrices; the caller
 * (k10_sag_exec.cu) uses the unfused sequence otherwise.  Workspace: 2 * tsg_colsum_workspace_bytes(N, F). */
extern "C" int tsg_sag_conv_bwd_fused(const float* dxo, const int32_t* inv, const float* score, const float* h,
                                      const float* dsw, const float* ws_vec, float* dhm, float* dbias, float* dws,
                                      int64_t N, int64_t F, void* workspace, size_t workspace_bytes, void* stream) {
  TSG_REQUIRE(N > 0 && F > 0 && F % 4 == 0 && 2 * (F / 4) <= CS_THREADS, "sag_conv_bwd_fused: bad shape");
  TSG_REQUIRE(dxo && inv && score && h && dsw && ws_vec && dhm && dbias && dws, "sag_conv_bwd_fused: null pointer");
  TSG_REQUIRE(((((uintptr_t)dxo) | ((uintptr_t)h) | ((uintptr_t)dhm) | ((uintptr_t)ws_vec) | ((uintptr_t)workspace)) & 15) == 0,
              "sag_conv_bwd_fused: operands must be 16-byte aligned");
  if (workspace_bytes < 2 * tsg_colsum_workspace_bytes(N, F)) { set_error("sag_conv_bwd_fused: workspace too small"); return TSG_EWORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  float* part = (float*)workspace;
  const int nb = colsum_blocks(N);
  int64_t rpb = (N + nb - 1) / nb; if (rpb < 1) rpb = 1;
  unsigned* ticket = fused_tail_ok(nb, 2 * F) ? ticket_next() : nullptr;
  static const int cbr = env_int("TSG_CONV_BWD_ROWS", 2);      // measured at the level-0 shape: 1: 99 us, 2: 79, 4: 83, 8: 99
#define TSG_CB(R) TSG_LAUNCH_PDL("sag_conv_bwd_fused", k_sag_conv_bwd_v4<R>, nb, CS_THREADS, 2 * CS_THREADS * sizeof(float4), st, \
      (const float4*)dxo, inv, score, (const float4*)h, dsw, (const float4*)ws_vec, (float4*)dhm, part, N, (int)(F / 4), rpb, \
      dbias, dws, ticket)
  if (cbr == 1) TSG_CB(1); else if (cbr == 4) TSG_CB(4); else if (cbr == 8) TSG_CB(8); else TSG_CB(2);
#undef TSG_CB
  if (!ticket) { int rc = launch_partial_sum_final(part, dbias, (int)F, dws, nb, (int)(2 * F), st); if (rc) return rc; }
  return check_launch("sag_conv_bwd_fused");
}

/* tsg_spmm + the row-wise product Y @ dot_vec (the score layer's h @ ws of Code/sag/layers.py:18 right behind
 * conv's ReLU(A_hat (xW) + b)): computed in K2's epilogue while the row is in registers -- bit-identical to
 * tsg_linear_fwd(Y, dot_vec, M = 1) -- or, for shapes the epilogue does not cover, by that call. */
extern "C" int tsg_linear_fwd(const float* X, const float* W, const float* bias, float* Y, int64_t N, int64_t K, int64_t M,
                              int w_transposed, int flags, void* stream);
extern "C" int tsg_spmm_dot(const int32_t* rowptr, const int32_t* colidx, const float* val, const float* H,
                            const float* bias, float* Y, const float* dot_vec, float* dot_out,
                            int64_t num_rows, int64_t feat, int flags, void* stream) {
  TSG_REQUIRE(num_rows >= 0 && feat > 0, "spmm_dot: bad shape rows=%lld feat=%lld", (long long)num_rows, (long long)feat);
  TSG_REQUIRE(num_rows < (int64_t)0x7fffffff, "spmm_dot: too many rows");
  if (num_rows == 0) return TSG_OK;
  TSG_REQUIRE(rowptr && colidx && H && Y && dot_vec && dot_out, "spmm_dot: null pointer");
  const int relu = (flags & TSG_SPMM_RELU) ? 1 : 0;
  const bool exact = (flags & TSG_SPMM_EXACT) != 0;
  cudaStream_t st = (cudaStream_t)stream;
  static const bool off = getenv("TSG_NO_SPMM_DOT") != nullptr;
  bool done = false;
  int rc = val ? launch_spmm<true>(rowptr, colidx, val, H, bias, Y, num_rows, feat, relu, exact, st, off ? nullptr : dot_vec, dot_out, &done)
               : launch_spmm<false>(rowptr, colidx, val, H, bias, Y, num_rows, feat, relu, exact, st, off ? nullptr : dot_vec, dot_out, &done);
  if (rc != TSG_OK || done) return rc;
  return tsg_linear_fwd(Y, dot_vec, nullptr, dot_out, num_rows, feat, 1, 0, 0, stream);
}

/* conv1 on one-hot node-label features without x W: Y = act(A_hat * W[label] + bias), and optionally the score
 * layer's Y @ dot_vec from the same epilogue (dot_vec / dot_out may both be null).  Bit-identical to tsg_embed_fwd ->
 * tsg_spmm_dot.  Needs the float4 path (feat % 4 == 0, 16-byte aligned W / Y / bias); returns TSG_EINVAL otherwise and
 * the caller runs the two-call sequence. */
extern "C" int tsg_spmm_label_dot(const int32_t* rowptr, const int32_t* colidx, const float* val, const float* W,
                                  const int32_t* label, int64_t num_labels, const float* bias, float* Y,
                                  const float* dot_vec, float* dot_out, int64_t num_rows, int64_t feat, int flags,
                                  void* stream) {
  TSG_REQUIRE(num_rows > 0 && feat > 0 && num_labels > 0 && num_rows < (int64_t)0x7fffffff && num_labels < (int64_t)0x7fffffff,
              "spmm_label_dot: bad shape");
  TSG_REQUIRE(rowptr && colidx && W && label && Y && ((dot_vec == nullptr) == (dot_out == nullptr)), "spmm_label_dot: null pointer");
  const bool vec = (feat % 4 == 0) && (((uintptr_t)W & 15) == 0) && (((uintptr_t)Y & 15) == 0) &&
                   (bias == nullptr || ((uintptr_t)bias & 15) == 0) && (dot_vec == nullptr || (((uintptr_t)dot_vec & 15) == 0 && feat <= 128));
  TSG_REQUIRE(vec, "spmm_label_dot: needs feat %% 4 == 0 (<= 128 with dot_vec) and 16-byte aligned operands");
  const int relu = (flags & TSG_SPMM_RELU) ? 1 : 0;
  const bool exact = (flags & TSG_SPMM_EXACT) != 0;
  cudaStream_t st = (cudaStream_t)stream;
  bool done = false;
  int rc = val ? launch_spmm<true>(rowptr, colidx, val, W, bias, Y, num_rows, feat, relu, exact, st, dot_vec, dot_out, &done, label, (int)num_labels)
               : launch_spmm<false>(rowptr, colidx, val, W, bias, Y, num_rows, feat, relu, exact, st, dot_vec, dot_out, &done, label, (int)num_labels);
  if (rc == TSG_OK && dot_vec && !done) { set_error("spmm_label_dot: dot epilogue not taken"); return TSG_EINVAL; }
  return rc;
}
