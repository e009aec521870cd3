// K11 -- EigenPooling preprocessing on the GPU (SURVEY 8f n2).
//
// Replaces the per-graph CPU work of Code/eigengcn/coarsen_pooling_with_last_eigen_padding.py:121-182
// (`_coarserning_pooling_`) AFTER the clustering step: for every cluster, the Laplacian of the induced
// subgraph (graph.laplacian(adj, normalize=False): L = D - W, graph.py:116-126), its full eigendecomposition
// (graph.fourier -> numpy.linalg.eigh, graph.py:147-163: ascending eigenvalues), the sign rule "first entry
// of the eigenvector >= 0" (coarsen...py:165-168), "repeat the last eigenvector when the cluster is smaller
// than j+1" (:169-173), and the coarsened adjacency Omega^T A_ext Omega (:135-149).  The reference does this
// with scipy / numpy per graph at load time (plus SpectralClustering, which stays outside: cluster labels are
// an INPUT here); at the 1 M-graph corpus of BASELINE config 5 that is ~27 M small eigenproblems.
//
// One warp per cluster, cluster size <= 32.  The dense Laplacian and the eigenvector matrix live in shared
// memory in double precision; cyclic Jacobi: for every pair (p, q) all lanes compute the same rotation from
// A[p][p], A[q][q], A[p][q]; lane k updates row/column k of A and row k of V; sweeps stop when the
// off-diagonal mass is below 1e-22 * trace-scale or after 30 sweeps.  Eigenpairs are then ranked by
// (eigenvalue, original column) -- a stable ascending sort like LAPACK's output order for distinct
// eigenvalues.  Degenerate eigenvalues: any orthonormal basis of the eigenspace is a valid answer and
// LAPACK's choice is not reproducible by another algorithm; parity is therefore stated on eigenvalues and on
// the projector of every eigenspace (tests/test_eigpool_gpu.py), and exactly on non-degenerate vectors.
#include "common.cuh"

namespace tsg {

constexpr int EIG_MAX = TSG_EIG_MAX;          // 32
constexpr int EIG_WARPS = 2;                  // clusters per CTA (2 x 2 x 32 x 33 doubles = 33 KB static smem)

__global__ void __launch_bounds__(EIG_WARPS * 32)
k_cluster_eig(const int* __restrict__ rowptr, const int* __restrict__ colidx, const float* __restrict__ val,
              const int* __restrict__ cluster_of, const int* __restrict__ member_ptr, const int* __restrict__ member,
              int num_clusters, int num_nodes, int num_vec,
              float* __restrict__ pool_val, float* __restrict__ pool_val_nodes, float* __restrict__ eigvals,
              int* __restrict__ status) {
  __shared__ double sA[EIG_WARPS][EIG_MAX][EIG_MAX + 1];
  __shared__ double sV[EIG_WARPS][EIG_MAX][EIG_MAX + 1];
  __shared__ int sNode[EIG_WARPS][EIG_MAX];
  __shared__ int sRank[EIG_WARPS][EIG_MAX];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x * EIG_WARPS + w;
  if (c >= num_clusters) return;
  const int m0 = member_ptr[c], n = member_ptr[c + 1] - m0;
  if (n > EIG_MAX) { if (lane == 0) atomicExch(status, 1); return; }     // caller falls back to the host path
  if (n == 0) return;                           // an empty cluster has no vector (its rank lookup would read sRank[-1])
  double (*A)[EIG_MAX + 1] = sA[w];
  double (*V)[EIG_MAX + 1] = sV[w];
  if (lane < n) sNode[w][lane] = member[m0 + lane];
  for (int i = 0; i < n; ++i) { A[i][lane] = 0.0; V[i][lane] = (i == lane) ? 1.0 : 0.0; }
  __syncwarp();
  // induced weight matrix: lane k scans the adjacency row of its node; members are few, so a linear search
  // over the (<= 32) member ids via the cluster label + a rank lookup is enough
  if (lane < n) {
    const int u = sNode[w][lane];
    double deg = 0.0;
    for (int p = rowptr[u]; p < rowptr[u + 1]; ++p) {
      const int v = colidx[p];
      if (v == u || cluster_of[v] != c) continue;
      int kq = -1;
      for (int q = 0; q < n; ++q) if (sNode[w][q] == v) { kq = q; break; }
      if (kq < 0) continue;
      const double wv = val ? (double)val[p] : 1.0;
      A[lane][kq] -= wv;                        // L = D - W  (W summed over duplicate entries)
      deg += wv;
    }
    A[lane][lane] += deg;                       // d = W.sum(axis=0) on a symmetric W (graph.py:120)
  }
  __syncwarp();
  // cyclic Jacobi
  for (int sweep = 0; sweep < 30; ++sweep) {
    double off = 0.0, diag = 0.0;
    if (lane < n) {
      for (int q = 0; q < n; ++q) { const double a = A[lane][q]; if (q == lane) diag += a * a; else off += a * a; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { off += __shfl_xor_sync(0xffffffffu, off, o); diag += __shfl_xor_sync(0xffffffffu, diag, o); }
    if (off <= 1e-26 * (diag + 1e-300) || off == 0.0) break;
    for (int p = 0; p < n - 1; ++p) {
      for (int q = p + 1; q < n; ++q) {
        const double apq = A[p][q];
        if (fabs(apq) > 1e-300) {
          const double app = A[p][p], aqq = A[q][q];
          const double theta = (aqq - app) / (2.0 * apq);
          const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
          const double cs = 1.0 / sqrt(t * t + 1.0), sn = t * cs;
          __syncwarp();
          if (lane < n) {
            const int k = lane;
            // rows/columns p and q of the symmetric A (lane k owns element k of each)
            if (k != p && k != q) {
              const double akp = A[k][p], akq = A[k][q];
              const double nkp = cs * akp - sn * akq, nkq = sn * akp + cs * akq;
              A[k][p] = nkp; A[p][k] = nkp; A[k][q] = nkq; A[q][k] = nkq;
            }
            const double vkp = V[k][p], vkq = V[k][q];
            V[k][p] = cs * vkp - sn * vkq; V[k][q] = sn * vkp + cs * vkq;
          }
          __syncwarp();
          if (lane == 0) {
            A[p][p] = app - t * apq; A[q][q] = aqq + t * apq; A[p][q] = 0.0; A[q][p] = 0.0;
          }
          __syncwarp();
        }
      }
    }
  }
  __syncwarp();
  // rank of eigenpair `lane` in ascending (eigenvalue, column) order
  if (lane < n) {
    const double lam = A[lane][lane];
    int r = 0;
    for (int q = 0; q < n; ++q) { const double lq = A[q][q]; r += (lq < lam) || (lq == lam && q < lane); }
    sRank[w][r] = lane;
    if (eigvals) eigvals[(int64_t)c * EIG_MAX + r] = (float)lam;
  }
  if (eigvals && lane >= n) eigvals[(int64_t)c * EIG_MAX + lane] = 0.f;
  __syncwarp();
  // pooling weights: vector j = eigenvector of rank min(j, n-1), sign-fixed on its first entry (member 0)
  for (int j = 0; j < num_vec; ++j) {
    const int col = sRank[w][min(j, n - 1)];
    const double sgn = V[0][col] < 0.0 ? -1.0 : 1.0;
    if (lane < n) {
      const float v = (float)(sgn * V[lane][col]);
      pool_val[(int64_t)j * num_nodes + m0 + lane] = v;
      pool_val_nodes[(int64_t)j * num_nodes + sNode[w][lane]] = v;
    }
  }
}

// inter-cluster edges: keep[e] = cluster_of[row] != cluster_of[col]; order-preserving compaction
constexpr int CO_TILE = 1024;
struct KeepCount { const int* v; __device__ int operator()(int64_t i) const { return v[i]; } };

template <bool WRITE>
__global__ void __launch_bounds__(256)
k_coarsen_edges(const int64_t* __restrict__ row, const int64_t* __restrict__ col, const float* __restrict__ w,
                int64_t E, const int* __restrict__ cluster_of, int* __restrict__ tile_cnt,
                const int* __restrict__ tile_off, int64_t* __restrict__ orow, int64_t* __restrict__ ocol,
                float* __restrict__ ow) {
  __shared__ int sm[33];
  const int64_t base = (int64_t)blockIdx.x * CO_TILE;
  int keep[4], cnt = 0;
  int64_t cr[4], cc[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int64_t e = base + (int64_t)threadIdx.x * 4 + k;          // 4 consecutive edges per thread: order kept
    keep[k] = 0;
    if (e < E) {
      cr[k] = cluster_of[row[e]]; cc[k] = cluster_of[col[e]];
      keep[k] = cr[k] != cc[k];
    }
    cnt += keep[k];
  }
  int tot;
  const int ex = block_excl_scan(cnt, sm, &tot);
  if (!WRITE) { if (threadIdx.x == 0) tile_cnt[blockIdx.x] = tot; return; }
  int64_t o = (int64_t)tile_off[blockIdx.x] + ex;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (keep[k]) {
      const int64_t e = base + (int64_t)threadIdx.x * 4 + k;
      orow[o] = cr[k]; ocol[o] = cc[k]; ow[o] = w ? w[e] : 1.f; ++o;
    }
  }
}

__global__ void k_store_count64(const int* src, int64_t* dst) { *dst = (int64_t)*src; }

}  // namespace tsg

using namespace tsg;

extern "C" int tsg_eigpool_build(const int32_t* adj_rowptr, const int32_t* adj_colidx, const float* adj_val,
                                 const int32_t* cluster_of, const int32_t* member_ptr, const int32_t* member,
                                 int64_t num_nodes, int64_t num_clusters, int num_vectors,
                                 float* pool_val, float* pool_val_nodes, float* eigvals, int32_t* status_dev,
                                 void* stream) {
  TSG_REQUIRE(num_nodes >= 0 && num_clusters >= 0 && num_vectors > 0, "eigpool_build: bad shape");
  TSG_REQUIRE(num_nodes < (int64_t)0x7fffffff && num_clusters < (int64_t)0x7fffffff, "eigpool_build: too large");
  if (num_clusters == 0 || num_nodes == 0) return TSG_OK;
  TSG_REQUIRE(adj_rowptr && adj_colidx && cluster_of && member_ptr && member && pool_val && pool_val_nodes && status_dev,
              "eigpool_build: null pointer");
  const int grid = (int)((num_clusters + EIG_WARPS - 1) / EIG_WARPS);
  k_cluster_eig<<<grid, EIG_WARPS * 32, 0, (cudaStream_t)stream>>>(adj_rowptr, adj_colidx, adj_val, cluster_of, member_ptr,
                                                                  member, (int)num_clusters, (int)num_nodes, num_vectors,
                                                                  pool_val, pool_val_nodes, eigvals, status_dev);
  return check_launch("eigpool_build");
}

extern "C" size_t tsg_coarsen_edges_workspace_bytes(int64_t num_edges) {
  const size_t tiles = (size_t)((num_edges + CO_TILE - 1) / CO_TILE);
  return 2 * ws_bytes(tiles + 2, 4) + ws_bytes(scan_ws_ints((int64_t)tiles + 1), 4) + 512;
}

extern "C" int tsg_coarsen_edges(const int64_t* row, const int64_t* col, const float* weight, int64_t num_edges,
                                 const int32_t* cluster_of, int64_t* out_row, int64_t* out_col, float* out_weight,
                                 int64_t* out_count_dev, void* workspace, size_t workspace_bytes, void* stream) {
  TSG_REQUIRE(num_edges >= 0 && out_count_dev, "coarsen_edges: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (num_edges == 0) { cudaMemsetAsync(out_count_dev, 0, 8, st); return check_launch("coarsen_edges(empty)"); }
  TSG_REQUIRE(row && col && cluster_of && out_row && out_col && out_weight, "coarsen_edges: null pointer");
  if (workspace_bytes < tsg_coarsen_edges_workspace_bytes(num_edges)) { set_error("coarsen_edges: workspace too small"); return TSG_EWORKSPACE; }
  const int tiles = (int)((num_edges + CO_TILE - 1) / CO_TILE);
  Workspace ws(workspace, workspace_bytes);
  int* tile_cnt = ws.take<int>(tiles + 2);
  int* tile_off = ws.take<int>(tiles + 2);
  int* scan_ws = ws.take<int>(scan_ws_ints(tiles + 1));
  k_coarsen_edges<false><<<tiles, 256, 0, st>>>(row, col, weight, num_edges, cluster_of, tile_cnt, nullptr, nullptr, nullptr, nullptr);
  int rc = exclusive_scan(KeepCount{tile_cnt}, tiles, tile_off, scan_ws, st);
  if (rc) return rc;
  k_store_count64<<<1, 1, 0, st>>>(tile_off + tiles, out_count_dev);
  k_coarsen_edges<true><<<tiles, 256, 0, st>>>(row, col, weight, num_edges, cluster_of, nullptr, tile_off, out_row, out_col, out_weight);
  return check_launch("coarsen_edges");
}
