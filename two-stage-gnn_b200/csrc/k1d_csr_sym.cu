// K1d -- CSR of A_hat for packed batches whose per-graph edge lists are COALESCED and SYMMETRIC (sorted by (row, col),
// loop free, (r, c) listed <=> (c, r) listed): what TUDataset, the TU loader (H1) and tsg.synth produce.  One kernel, no
// counting pass, no atomics, no device-wide scan, ONE orientation:
//   * row r's edges are the run of lrow == r, so row starts fall out of the run boundaries;
//   * every node adds exactly one self loop, so graph g's entries start at edge_ptr[g] + node_ptr[g]: global offsets are
//     known without a scan;
//   * symmetric => the dst-major CSR and the src-major CSR are the SAME arrays (row r = its neighbours in ascending
//     order, self loop last: PyG's add_remaining_self_loops order), so the transposed orientation is an alias, not a copy.
// Replaces K1b (k1b_csr_graphs.cu: 5 launches, shared-memory atomics, both orientations written -- 170 us = 10 % of the
// round-1 step at 13 % of the HBM roofline) on this input class; values and indices are bit-identical to K1b's (same
// formulas: dis = 1 / sqrt(deg + 1) with IEEE div / sqrt, val = dis[src] * dis[dst]).  The kernel VERIFIES the promise
// per graph (range, order, symmetry by binary search) and ORs TSG_FUSED_* bits into *status: the host raises, nothing
// falls back silently.
// Reference: PyG gcn_norm via Code/sag/network.py:34 (GCNConv), SURVEY A.1.1 / A.1.6.
#include "common.cuh"
#include "sag_fused.cuh"

namespace tsg {

constexpr int CSYM_THREADS = 256;

__global__ void __launch_bounds__(CSYM_THREADS)
k_csr_sym(const int32_t* __restrict__ lrow, const int32_t* __restrict__ lcol, const int64_t* __restrict__ edge_ptr,
          const int64_t* __restrict__ node_ptr, int G, int nmax, int32_t* __restrict__ rowptr, int32_t* __restrict__ colidx,
          float* __restrict__ val, int* __restrict__ status) {
  pdl_wait();
  pdl_launch_dependents();
  extern __shared__ __align__(16) unsigned char sm[];
  int* rs = reinterpret_cast<int*>(sm);                       // [nmax + 2] first edge of every row
  float* dis = reinterpret_cast<float*>(sm + (size_t)(nmax + 2) * 4);
  __shared__ int s_bad;
  const int tid = threadIdx.x;
  for (int g = blockIdx.x; g < G; g += gridDim.x) {
    const int64_t eb = edge_ptr[g], nb = node_ptr[g];
    const int e = (int)(edge_ptr[g + 1] - eb), n = (int)(node_ptr[g + 1] - nb);
    if (tid == 0) s_bad = 0;
    __syncthreads();
    int bad = 0;
    for (int p = tid; p <= e; p += CSYM_THREADS) {
      const int r = p < e ? lrow[eb + p] : n;
      const int r0 = p > 0 ? lrow[eb + p - 1] : -1;
      if (p < e) {
        const int q = lcol[eb + p];
        if ((unsigned)r >= (unsigned)n || (unsigned)q >= (unsigned)n || r == q) { bad |= TSG_FUSED_BAD_EDGE; continue; }
        if (p > 0 && !(r0 < r || (r0 == r && lcol[eb + p - 1] < q))) { bad |= TSG_FUSED_UNSORTED; continue; }
      }
      if (r0 != -1 && (unsigned)r0 >= (unsigned)n) continue;
      for (int rr = r0 + 1; rr <= r; ++rr) rs[rr] = p;
    }
    if (bad) atomicOr(&s_bad, bad);
    __syncthreads();
    if (s_bad) {                                              // uniform: skip the graph, report
      if (tid == 0) atomicOr(status, s_bad);
      __syncthreads();
      continue;
    }
    const int64_t ob = eb + nb;                               // first CSR entry of this graph
    for (int r = tid; r <= n; r += CSYM_THREADS) {
      rowptr[nb + r] = (int32_t)(ob + rs[r] + r);
      if (r < n) dis[r] = __fdiv_rn(1.0f, __fsqrt_rn((float)(rs[r + 1] - rs[r] + 1)));
    }
    __syncthreads();
    bad = 0;
    for (int p = tid; p < e; p += CSYM_THREADS) {
      const int r = lrow[eb + p], q = lcol[eb + p];
      const int64_t o = ob + p + r;
      colidx[o] = (int32_t)(nb + q);
      val[o] = __fmul_rn(__fmul_rn(dis[q], 1.0f), dis[r]);
      // symmetry: (q, r) must be listed in row q
      int lo = rs[q], hi = rs[q + 1];
      bool found = false;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const int v = lcol[eb + mid];
        if (v == r) { found = true; break; }
        if (v < r) lo = mid + 1; else hi = mid;
      }
      if (!found) bad |= TSG_FUSED_ASYMMETRIC;
    }
    for (int r = tid; r < n; r += CSYM_THREADS) {             // self loop closes the row
      const int64_t o = ob + rs[r + 1] + r;
      colidx[o] = (int32_t)(nb + r);
      val[o] = __fmul_rn(__fmul_rn(dis[r], 1.0f), dis[r]);
    }
    if (bad) atomicOr(status, bad);
    __syncthreads();                                          // rs / dis are reused by the next graph
  }
}

}  // namespace tsg

using namespace tsg;

extern "C" int tsg_csr_build_graphs_sym_local(const int32_t* local_row, const int32_t* local_col, const int64_t* edge_ptr,
                                              const int64_t* node_ptr, int64_t G, int64_t N, int64_t E,
                                              int64_t max_graph_nodes, int32_t* rowptr, int32_t* colidx, float* val,
                                              int32_t* status, void* stream) {
  TSG_REQUIRE(G > 0 && N > 0 && E >= 0 && max_graph_nodes > 0 && N + E < (int64_t)0x7fffffff, "csr_build_graphs_sym: bad sizes");
  TSG_REQUIRE(edge_ptr && node_ptr && rowptr && colidx && val && status && (E == 0 || (local_row && local_col)),
              "csr_build_graphs_sym: null pointer");
  const size_t smem = (size_t)(max_graph_nodes + 2) * 4 + (size_t)max_graph_nodes * 4 + 16;
  TSG_REQUIRE(smem <= 200 * 1024, "csr_build_graphs_sym: a graph of %lld nodes exceeds the shared-memory budget", (long long)max_graph_nodes);
  static size_t configured = 0;
  if (smem > 48 * 1024 && smem > configured) {
    cudaFuncSetAttribute(k_csr_sym, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    configured = 200 * 1024;
  }
  const int grid = (int)(G < (int64_t)TSG_NUM_SMS * 8 ? G : (int64_t)TSG_NUM_SMS * 8);
  return launch_pdl("csr_build_graphs_sym", k_csr_sym, grid, CSYM_THREADS, smem, (cudaStream_t)stream, local_row, local_col, edge_ptr,
                    node_ptr, (int)G, (int)max_graph_nodes, rowptr, colidx, val, status);
}
