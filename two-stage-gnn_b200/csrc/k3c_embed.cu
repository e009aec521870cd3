// K3c -- the level-0 products when the node features are one-hot node labels.
//
// Every TU dataset the reference trains on gives a node ONE categorical label; the loaders expand it to a one-hot
// row (Code/sag/train.py:34 TUDataset -> data.x; Code/sage+gat+diffpool/load_data.py:74-87 `node_label_one_hot`),
// and conv1 multiplies that [N, L] matrix by W1 [L, H] (Code/sag/network.py:34).  With x = onehot(label):
//     x @ W        = W[label, :]                 (a row gather: every other term of the dot product is 0 * w)
//     x^T @ dY     = segment-sum of dY rows by label
// so the 89-column fp32 matrix (345 MB for the bench batch, read twice per step) never has to exist: the forward
// is a pure 124 MB write stream, the weight gradient a pure 124 MB read stream.  Forward results are bit-identical
// to the dense K3 product (adding +-0 products never changes an fp32 sum; tests/test_compact_gpu.py); the
// gradient is summed in a fixed order (row -> warp table -> CTA -> slice), deterministic run to run, and agrees with
// the dense K3 dW to fp32 summation-order tolerance.
// A label outside [0, L) is the all-zero row of one-hot (what k_pack_batch writes for it): zero output, no gradient.
#include <stdlib.h>
#include "common.cuh"

namespace tsg {

constexpr int EMB_THREADS = 256;

constexpr int EMB_FWD_ILP = 4;

template <bool VEC4>
__global__ void __launch_bounds__(EMB_THREADS)
k_embed_fwd(const float* __restrict__ W, const int* __restrict__ label, float* __restrict__ out,
            int64_t N, int K, int M) {
  pdl_wait();
  pdl_launch_dependents();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  if (VEC4) {
    const int m4 = M >> 2;
    const int64_t total = N * m4;
    const float4* W4 = reinterpret_cast<const float4*>(W);
    float4* o4 = reinterpret_cast<float4*>(out);
    // label -> W row -> store is a dependent chain of two loads: EMB_FWD_ILP independent chains per thread
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < total; i0 += stride * EMB_FWD_ILP) {
      int l[EMB_FWD_ILP], c[EMB_FWD_ILP];
      float4 v[EMB_FWD_ILP];
#pragma unroll
      for (int u = 0; u < EMB_FWD_ILP; ++u) {
        const int64_t i = i0 + u * stride;
        const int64_t r = i / m4;
        c[u] = (int)(i - r * m4);
        l[u] = i < total ? __ldg(label + r) : -1;
      }
#pragma unroll
      for (int u = 0; u < EMB_FWD_ILP; ++u) {
        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if ((unsigned)l[u] < (unsigned)K) v[u] = __ldg(W4 + (size_t)l[u] * m4 + c[u]);
      }
#pragma unroll
      for (int u = 0; u < EMB_FWD_ILP; ++u) {
        const int64_t i = i0 + u * stride;
        if (i < total) __stcs(o4 + i, v[u]);
      }
    }
  } else {
    const int64_t total = N * M;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
      const int64_t r = i / M; const int c = (int)(i - r * M);
      const int l = __ldg(label + r);
      out[i] = (unsigned)l < (unsigned)K ? __ldg(W + (size_t)l * M + c) : 0.f;
    }
  }
}

// dW[k, :] = sum of dY rows whose label is k.  One private [K, M] table per warp in shared memory (lane = column,
// so a row's update is conflict free and the warp applies its rows in row order), EMB_UNROLL rows of loads in
// flight per warp; the CTA then folds its warps' tables in warp order into one partial, and
// k_partial_sum_final folds the CTAs.  The row -> (CTA, warp) map depends on N only.
constexpr int EMB_BWD_GRID = 148;

template <int EMB_UNROLL, bool PIPE>
__global__ void __launch_bounds__(512)
k_embed_bwd_weight(const int* __restrict__ label, const float* __restrict__ dY, float* __restrict__ part,
                   int64_t N, int K, int M, int64_t rows_per_cta) {
  pdl_wait();
  pdl_launch_dependents();
  extern __shared__ float tab[];
  const int nw = blockDim.x >> 5, w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int KM = K * M;
  for (int i = threadIdx.x; i < nw * KM; i += blockDim.x) tab[i] = 0.f;
  __syncthreads();
  float* mine = tab + (size_t)w * KM;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_cta;
  const int64_t r1 = r0 + rows_per_cta < N ? r0 + rows_per_cta : N;
  for (int m0 = 0; m0 < M; m0 += 32) {
    const int m = m0 + lane;
    const bool col_ok = m < M;
    auto load = [&](int64_t r, int (&l)[EMB_UNROLL], float (&v)[EMB_UNROLL]) {
#pragma unroll
      for (int u = 0; u < EMB_UNROLL; ++u) {
        const int64_t rr = r + (int64_t)u * nw;
        const bool ok = rr < r1;
        l[u] = ok ? __ldg(label + rr) : -1;
        v[u] = (ok && col_ok) ? __ldcs(dY + (size_t)rr * M + m) : 0.f;
      }
    };
    auto apply = [&](const int (&l)[EMB_UNROLL], const float (&v)[EMB_UNROLL]) {
#pragma unroll
      for (int u = 0; u < EMB_UNROLL; ++u)
        if ((unsigned)l[u] < (unsigned)K && col_ok) mine[l[u] * M + m] += v[u];
    };
    // two register batches: the loads of batch i+1 are in flight while batch i's (serial: two rows may share a
    // label) read-modify-write chain runs
    const int64_t step = (int64_t)nw * EMB_UNROLL;
    int la[EMB_UNROLL], lb[EMB_UNROLL];
    float va[EMB_UNROLL], vb[EMB_UNROLL];
    int64_t r = r0 + w;
    if (PIPE) {
      load(r, la, va);
      for (; r < r1; r += 2 * step) {
        load(r + step, lb, vb);
        apply(la, va);
        load(r + 2 * step, la, va);
        apply(lb, vb);
      }
    } else {
      for (; r < r1; r += step) { load(r, la, va); apply(la, va); }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < KM; i += blockDim.x) {
    float s = tab[i];
    for (int q = 1; q < nw; ++q) s += tab[(size_t)q * KM + i];
    part[(size_t)blockIdx.x * KM + i] = s;
  }
}

static int embed_bwd_warps(int64_t K, int64_t M) {
  const size_t table = (size_t)K * M * 4;
  if (table == 0 || table > 200 * 1024) return 0;
  size_t nw = (200 * 1024) / table;
  return (int)(nw > 16 ? 16 : nw);
}

}  // namespace tsg

using namespace tsg;

extern "C" int tsg_embed_fwd(const float* W, const int32_t* label, float* out, int64_t N, int64_t K, int64_t M, void* stream) {
  TSG_REQUIRE(N >= 0 && K > 0 && M > 0 && K < (1 << 24) && M < (1 << 24), "embed_fwd: bad shape");
  if (N == 0) return TSG_OK;
  TSG_REQUIRE(W && label && out, "embed_fwd: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const bool v4 = (M % 4 == 0) && (((uintptr_t)W | (uintptr_t)out) % 16 == 0);
  const int64_t total = v4 ? N * (M / 4) : N * M;
  const int grid = grid_for((total + EMB_FWD_ILP - 1) / EMB_FWD_ILP, EMB_THREADS, 8);
  if (v4) return launch_pdl("embed_fwd", k_embed_fwd<true>, grid, EMB_THREADS, 0, st, W, label, out, N, (int)K, (int)M);
  return launch_pdl("embed_fwd", k_embed_fwd<false>, grid, EMB_THREADS, 0, st, W, label, out, N, (int)K, (int)M);
}

/* 0 when the [K, M] table does not fit one warp's share of shared memory (use the dense K3 product instead) */
extern "C" size_t tsg_embed_bwd_weight_workspace_bytes(int64_t K, int64_t M) {
  if (K <= 0 || M <= 0 || embed_bwd_warps(K, M) == 0) return 0;
  return ws_bytes((size_t)EMB_BWD_GRID * K * M, 4) + 256;
}

extern "C" int tsg_embed_bwd_weight(const int32_t* label, const float* dY, float* dW, int64_t N, int64_t K, int64_t M,
                                    void* workspace, size_t workspace_bytes, void* stream) {
  TSG_REQUIRE(N >= 0 && K > 0 && M > 0, "embed_bwd_weight: bad shape");
  const int nw = embed_bwd_warps(K, M);
  TSG_REQUIRE(nw > 0, "embed_bwd_weight: a %lld x %lld table does not fit shared memory", (long long)K, (long long)M);
  TSG_REQUIRE(dW && (N == 0 || (label && dY)), "embed_bwd_weight: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (N == 0) { cudaMemsetAsync(dW, 0, (size_t)K * M * 4, st); return check_launch("embed_bwd_weight"); }
  if (workspace_bytes < tsg_embed_bwd_weight_workspace_bytes(K, M)) { set_error("embed_bwd_weight: workspace too small"); return TSG_EWORKSPACE; }
  Workspace ws(workspace, workspace_bytes);
  float* part = ws.take<float>((size_t)EMB_BWD_GRID * K * M);
  const size_t smem = (size_t)nw * K * M * 4;
  const int64_t rows_per_cta = (N + EMB_BWD_GRID - 1) / EMB_BWD_GRID;
  static const int variant = [] { const char* e = getenv("TSG_EMB_VARIANT"); return e ? atoi(e) : 0; }();
  auto launch = [&](auto kern) {
    if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    return launch_pdl("embed_bwd_weight", kern, EMB_BWD_GRID, nw * 32, smem, st, label, dY, part, N, (int)K, (int)M, rows_per_cta);
  };
  int rc;
  if (variant == 1) rc = launch(k_embed_bwd_weight<8, true>);          // A/B variants (TSG_EMB_VARIANT), measured in
  else if (variant == 2) rc = launch(k_embed_bwd_weight<16, false>);   // profiles/r01c_compact_input.md
  else rc = launch(k_embed_bwd_weight<16, true>);
  if (rc) return rc;
  rc = launch_partial_sum_final(part, dW, (int)(K * M), nullptr, EMB_BWD_GRID, (int)(K * M), st);
  if (rc) return rc;
  return check_launch("embed_bwd_weight");
}
