// K15 -- DiffPool's auxiliary link-prediction loss (SURVEY 8f n4; Code/sage+gat+diffpool/encoders.py:409-441, reached
// with --linkpred in the original setting, train.py:121-126):
//     P_g = S_g S_g^T (clamped at 1),   L = sum_g sum_{i,j < n_g} [ -A_ij log(P_ij + eps) - (1 - A_ij) log(1 - P_ij + eps) ]
//         / sum_g n_g^2,   eps = 1e-7
// on the PACKED layout: S [sum n, K] are the assignment rows (softmax: padded rows do not exist here, the reference masks
// them to zero and drops their entries from the sum), A the 0/1 adjacency as RAW CSR.  The reference materialises the dense
// [N, N] P per graph; here a CTA walks 32 x 32 tiles of (i, j) pairs with both row tiles of S in shared memory, looks A_ij
// up in row i's sorted column list, and never writes P.  Backward: dS_i = dL * sum_j (G_ij + G_ji) S_j with
// G_ij = dL/dP_ij recomputed per tile; rows of dS are owned by one CTA each and accumulated in a fixed order.
// Upstream defect kept out: the reference clamps with `torch.min(pred_adj, torch.Tensor(1).cuda())`, an UNINITIALISED
// one-element tensor; the intended clamp at 1 is what is implemented (a no-op for softmax rows: s_i . s_j <= 1).
#include "common.cuh"

namespace tsg {

constexpr int LP_T = 256, LP_TILE = 32;

__device__ __forceinline__ float lp_adj(const int* __restrict__ rowptr, const int* __restrict__ colidx, int64_t gi, int64_t gj) {
  for (int p = rowptr[gi]; p < rowptr[gi + 1]; ++p) if (colidx[p] == (int)gj) return 1.f;
  return 0.f;
}

// MODE 0: loss partial per graph.  MODE 1: dS rows.
template <int MODE>
__global__ void __launch_bounds__(LP_T)
k_linkpred(const float* __restrict__ S, const int64_t* __restrict__ gptr, const int* __restrict__ rowptr,
           const int* __restrict__ colidx, int K, float eps, float* __restrict__ loss_part, const float* __restrict__ dloss,
           float inv_entries, float* __restrict__ dS) {
  extern __shared__ __align__(16) float lsm[];
  const int pitch = K + 1;
  float* Si = lsm;                       // [32][K+1]
  float* Sj = lsm + LP_TILE * pitch;     // [32][K+1]
  float* Gt = Sj + LP_TILE * pitch;      // [32][33]   G_ij + G_ji for the tile (MODE 1)
  __shared__ float red[LP_T / 32];
  const int g = blockIdx.x;
  const int64_t lo = gptr[g];
  const int n = (int)(gptr[g + 1] - lo);
  const int tid = threadIdx.x;
  float acc_loss = 0.f;
  const float scale = MODE == 1 ? (*dloss) * inv_entries : 0.f;
  for (int i0 = 0; i0 < n; i0 += LP_TILE) {
    const int ni = min(LP_TILE, n - i0);
    __syncthreads();
    for (int t = tid; t < LP_TILE * K; t += LP_T) {
      const int r = t / K, k = t - r * K;
      Si[r * pitch + k] = r < ni ? S[(lo + i0 + r) * K + k] : 0.f;
    }
    // MODE 1: this CTA's dS rows i0..i0+31: thread (r = tid / 8, lane8 = tid % 8) owns columns k = lane8, lane8 + 8, ...
    float dacc[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) dacc[q] = 0.f;
    for (int j0 = 0; j0 < n; j0 += LP_TILE) {
      const int nj = min(LP_TILE, n - j0);
      __syncthreads();
      for (int t = tid; t < LP_TILE * K; t += LP_T) {
        const int r = t / K, k = t - r * K;
        Sj[r * pitch + k] = r < nj ? S[(lo + j0 + r) * K + k] : 0.f;
      }
      __syncthreads();
      // 1,024 pairs of the tile, 4 per thread: pair (i = t / 32, j = t % 32)
      for (int t = tid; t < LP_TILE * LP_TILE; t += LP_T) {
        const int i = t >> 5, j = t & 31;
        float gsum = 0.f;
        if (i < ni && j < nj) {
          float p = 0.f;
          for (int k = 0; k < K; ++k) p = fmaf(Si[i * pitch + k], Sj[j * pitch + k], p);
          const bool clamped = p > 1.f;
          p = fminf(p, 1.f);
          const int64_t gi = lo + i0 + i, gj = lo + j0 + j;
          const float a_ij = lp_adj(rowptr, colidx, gi, gj);
          if (MODE == 0) {
            acc_loss += -a_ij * logf(p + eps) - (1.f - a_ij) * logf(1.f - p + eps);
          } else {
            // P is symmetric, A may not be: G_ij + G_ji with the transposed entry looked up as well
            const float a_ji = lp_adj(rowptr, colidx, gj, gi);
            if (!clamped) {
              gsum = (-a_ij / (p + eps) + (1.f - a_ij) / (1.f - p + eps)) + (-a_ji / (p + eps) + (1.f - a_ji) / (1.f - p + eps));
            }
          }
        }
        if (MODE == 1) Gt[i * 33 + j] = gsum;
      }
      if (MODE == 1) {
        __syncthreads();
        const int r = tid >> 3, l8 = tid & 7;
        if (r < ni) {
          for (int j = 0; j < nj; ++j) {
            const float gv = Gt[r * 33 + j];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              const int k = l8 + 8 * q;
              if (k < K) dacc[q] = fmaf(gv, Sj[j * pitch + k], dacc[q]);
            }
          }
        }
      }
    }
    if (MODE == 1) {
      const int r = tid >> 3, l8 = tid & 7;
      if (r < ni) {
#pragma unroll
        for (int q = 0; q < 16; ++q) {
          const int k = l8 + 8 * q;
          if (k < K) dS[(lo + i0 + r) * K + k] = dacc[q] * scale;
        }
      }
    }
  }
  if (MODE == 0) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc_loss += __shfl_xor_sync(0xffffffffu, acc_loss, o);
    if ((tid & 31) == 0) red[tid >> 5] = acc_loss;
    __syncthreads();
    if (tid == 0) {
      float t = 0.f;
      for (int w = 0; w < LP_T / 32; ++w) t += red[w];
      loss_part[g] = t;
    }
  }
}

__global__ void k_lp_finish(const float* __restrict__ total, float inv_entries, float* __restrict__ loss) { *loss = *total * inv_entries; }

}  // namespace tsg

using namespace tsg;

extern "C" size_t tsg_linkpred_workspace_bytes(int64_t G) { return align_up((size_t)(G + 1) * 4, 256) + 256; }

static int lp_common(int64_t G, int64_t K, size_t* smem) {
  TSG_REQUIRE(G >= 0 && K > 0 && K <= 128, "linkpred: needs 1 <= assign_dim <= 128 (got %lld)", (long long)K);
  *smem = ((size_t)2 * LP_TILE * (K + 1) + LP_TILE * 33) * 4;
  return TSG_OK;
}

extern "C" int tsg_linkpred_loss_fwd(const float* S, const int64_t* graph_ptr, const int32_t* rowptr, const int32_t* colidx,
                                     int64_t G, int64_t K, double num_entries, float eps, float* loss, void* workspace,
                                     size_t workspace_bytes, void* stream) {
  size_t smem;
  int rc = lp_common(G, K, &smem);
  if (rc) return rc;
  TSG_REQUIRE(S && graph_ptr && rowptr && colidx && loss && workspace && num_entries > 0, "linkpred_loss_fwd: bad arguments");
  if (workspace_bytes < tsg_linkpred_workspace_bytes(G)) { set_error("linkpred_loss_fwd: workspace too small"); return TSG_EWORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  float* part = (float*)workspace;
  float* total = part + G;
  if (G == 0) { cudaMemsetAsync(loss, 0, 4, st); return TSG_OK; }
  k_linkpred<0><<<(int)G, LP_T, smem, st>>>(S, graph_ptr, rowptr, colidx, (int)K, eps, part, nullptr, 0.f, nullptr);
  rc = launch_partial_sum_final(part, total, 1, nullptr, (int)G, 1, st);
  if (rc) return rc;
  k_lp_finish<<<1, 1, 0, st>>>(total, (float)(1.0 / num_entries), loss);
  return check_launch("linkpred_loss_fwd");
}

extern "C" int tsg_linkpred_loss_bwd(const float* S, const int64_t* graph_ptr, const int32_t* rowptr, const int32_t* colidx,
                                     int64_t G, int64_t K, double num_entries, float eps, const float* dloss, float* dS,
                                     void* stream) {
  size_t smem;
  int rc = lp_common(G, K, &smem);
  if (rc) return rc;
  TSG_REQUIRE(S && graph_ptr && rowptr && colidx && dloss && dS && num_entries > 0, "linkpred_loss_bwd: bad arguments");
  if (G == 0) return TSG_OK;
  k_linkpred<1><<<(int)G, LP_T, smem, (cudaStream_t)stream>>>(S, graph_ptr, rowptr, colidx, (int)K, eps, nullptr, dloss,
                                                               (float)(1.0 / num_entries), dS);
  return check_launch("linkpred_loss_bwd");
}
