// K1c -- the pooled level's CSR straight from the previous level's CSR (no COO round trip).
//
// Code/sag/layers.py:20-23 selects nodes (`perm`) and filters the edge list (`filter_adj`); the next
// GCNConv (network.py:38,42) then renormalises it.  Going through the COO list costs K5b (two passes over
// int64 edges + scans) and a full K1b rebuild per level.  But the result is a pure function of the old CSR:
//   * new row i is old row perm[i] with the entries whose column survives (inv >= 0), in the SAME order
//     (filter_adj keeps the COO order and K1's rows are in COO order, so "filter then sort" == "sort then
//     filter"); the appended self loop (last entry of every old row) survives with its row and stays last;
//   * columns are relabelled by inv; deg' = surviving entries of the dst-major row (self loop included);
//     val = (deg'^-1/2[src] * 1) * deg'^-1/2[dst] with the same IEEE div / sqrt as K1.
// Three steps: count the survivors of both orientations (thread per new row), ONE scan over the concatenated
// counters, write.  Bit-identical to K1b(filter_adj(edges, perm)) -- tests/test_sag_exec_gpu.py compares the
// executor (which uses this) with the op-by-op path (which does not).
#include "common.cuh"

namespace tsg {

__global__ void k_inv_perm32(const int64_t* __restrict__ perm, int64_t k, int* __restrict__ inv) {
  pdl_wait();
  pdl_launch_dependents();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < k; i += (int64_t)gridDim.x * blockDim.x)
    inv[perm[i]] = (int)i;
}

// cnt[i] (i < k): dst-major survivors of new row i;  cnt[k + i]: src-major survivors
__global__ void __launch_bounds__(256)
k_csrf_count(const int* __restrict__ rowptr, const int* __restrict__ colidx, const int* __restrict__ t_rowptr,
             const int* __restrict__ t_colidx, const int64_t* __restrict__ perm, const int* __restrict__ inv,
             int k, int* __restrict__ cnt, int halves) {
  pdl_wait();
  pdl_launch_dependents();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < halves * k; i += gridDim.x * blockDim.x) {
    const bool tr = i >= k;
    const int r = (int)perm[tr ? i - k : i];
    const int* rp = tr ? t_rowptr : rowptr;
    const int* ci = tr ? t_colidx : colidx;
    int c = 0;
    for (int p = rp[r]; p < rp[r + 1]; ++p) c += inv[ci[p]] >= 0;
    cnt[i] = c;
  }
}

struct CsrfCnt { const int* v; __device__ int operator()(int64_t i) const { return v[i]; } };

// off = exclusive scan of cnt over [0, 2k]; the src-major half is rebased by off[k]
__global__ void __launch_bounds__(256)
k_csrf_write(const int* __restrict__ rowptr, const int* __restrict__ colidx, const int* __restrict__ t_rowptr,
             const int* __restrict__ t_colidx, const int64_t* __restrict__ perm, const int* __restrict__ inv,
             int k, const int* __restrict__ cnt, const int* __restrict__ off,
             int* __restrict__ n_rowptr, int* __restrict__ n_colidx, float* __restrict__ n_val,
             int* __restrict__ nt_rowptr, int* __restrict__ nt_colidx, float* __restrict__ nt_val, int halves) {
  pdl_wait();
  pdl_launch_dependents();
  const int half = off[k];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < halves * k; i += gridDim.x * blockDim.x) {
    const bool tr = i >= k;
    const int row = tr ? i - k : i;
    const int r = (int)perm[row];
    const int* rp = tr ? t_rowptr : rowptr;
    const int* ci = tr ? t_colidx : colidx;
    int o = off[i] - (tr ? half : 0);
    (tr ? nt_rowptr : n_rowptr)[row] = o;
    if (row == k - 1) (tr ? nt_rowptr : n_rowptr)[k] = o + cnt[i];
    // deg' of a node = its dst-major survivor count (self loop included)
    const float dis_row = __fdiv_rn(1.0f, __fsqrt_rn((float)cnt[row]));
    int* oc = tr ? nt_colidx : n_colidx;
    float* ov = tr ? nt_val : n_val;
    for (int p = rp[r]; p < rp[r + 1]; ++p) {
      const int j = inv[ci[p]];
      if (j < 0) continue;
      const float dis_j = __fdiv_rn(1.0f, __fsqrt_rn((float)cnt[j]));
      // K1: val = (dis[src] * w) * dis[dst], w = 1.  dst-major row: dst = row, src = j; src-major: src = row, dst = j
      const float v = tr ? __fmul_rn(__fmul_rn(dis_row, 1.0f), dis_j) : __fmul_rn(__fmul_rn(dis_j, 1.0f), dis_row);
      oc[o] = j; ov[o] = v; ++o;
    }
  }
}

}  // namespace tsg

using namespace tsg;

extern "C" int tsg_inv_perm(const int64_t* perm, int64_t num_perm, int64_t num_nodes, int32_t* inv_perm, void* stream) {
  TSG_REQUIRE(num_perm >= 0 && num_nodes >= 0 && (num_nodes == 0 || inv_perm) && (num_perm == 0 || perm), "inv_perm: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (num_nodes > 0) cudaMemsetAsync(inv_perm, 0xFF, (size_t)num_nodes * 4, st);
  if (num_perm > 0) TSG_LAUNCH_PDL("inv_perm", k_inv_perm32, grid_for(num_perm, 256), 256, 0, st, perm, num_perm, inv_perm);
  return TSG_OK;
}

extern "C" size_t tsg_csr_filter_workspace_bytes(int64_t num_perm) {
  return 2 * ws_bytes((size_t)(2 * num_perm + 2), 4) + ws_bytes(scan_ws_ints(2 * num_perm + 1), 4) + 512;
}

extern "C" int tsg_csr_filter(const int32_t* rowptr, const int32_t* colidx, const int32_t* t_rowptr,
                              const int32_t* t_colidx, const int64_t* perm, const int32_t* inv_perm, int64_t num_perm,
                              int32_t* out_rowptr, int32_t* out_colidx, float* out_val,
                              int32_t* out_t_rowptr, int32_t* out_t_colidx, float* out_t_val,
                              void* workspace, size_t workspace_bytes, void* stream) {
  TSG_REQUIRE(num_perm > 0 && num_perm < (int64_t)0x3fffffff, "csr_filter: bad row count");
  // symmetric operators (the src-major CSR is the same arrays as the dst-major one: K1d): pass NULL for every
  // transposed pointer and only one orientation is counted, scanned and written
  const bool sym = !t_rowptr && !t_colidx && !out_t_rowptr && !out_t_colidx && !out_t_val;
  TSG_REQUIRE(rowptr && colidx && perm && inv_perm && out_rowptr && out_colidx && out_val &&
              (sym || (t_rowptr && t_colidx && out_t_rowptr && out_t_colidx && out_t_val)), "csr_filter: null pointer");
  const int halves = sym ? 1 : 2;
  if (workspace_bytes < tsg_csr_filter_workspace_bytes(num_perm)) { set_error("csr_filter: workspace too small"); return TSG_EWORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  const int k = (int)num_perm;
  int* cnt = ws.take<int>(2 * num_perm + 2);
  int* off = ws.take<int>(2 * num_perm + 2);
  int* scan_ws = ws.take<int>(scan_ws_ints(2 * num_perm + 1));
  const int grid = grid_for(halves * num_perm, 256);
  TSG_LAUNCH_PDL("csr_filter(count)", k_csrf_count, grid, 256, 0, st, rowptr, colidx, t_rowptr, t_colidx, perm, inv_perm, k, cnt, halves);
  int rc = exclusive_scan(CsrfCnt{cnt}, halves * num_perm, off, scan_ws, st);
  if (rc) return rc;
  return launch_pdl("csr_filter", k_csrf_write, grid, 256, 0, st, rowptr, colidx, t_rowptr, t_colidx, perm, inv_perm, k, (const int*)cnt,
                    (const int*)off, out_rowptr, out_colidx, out_val, out_t_rowptr, out_t_colidx, out_t_val, halves);
}
