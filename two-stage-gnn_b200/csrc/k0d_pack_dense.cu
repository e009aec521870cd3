// K0d -- device-side assembly of a DENSE-encoder batch (GraphSAGE / GAT / DiffPool, Code/sage+gat+diffpool) from an
// HBM-resident corpus whose per-graph edge lists are COALESCED and SYMMETRIC (sorted by (row, col), loop free,
// (r, c) listed <=> (c, r) listed: TUDataset / the TU loader / tsg.synth).  One launch writes everything the packed
// dense encoders take for the chosen graphs:
//   * x [N, F]: row out_node_ptr[b] + i = table[i] (the shared N(0, 2^2) feature table indexed by node position,
//     Code/sage+gat+diffpool/train_triplet.py:379-385), float4 stores where F % 4 == 0;
//   * has_pad [B] = n_b < max_nodes (the virtual zero-padded row of the reference's max_nodes padding);
//   * the RAW 0/1 CSR of the packed adjacency, equal to tsg_csr_build(TSG_CSR_RAW) on the expanded edge_index:
//       - row r's edges are the run of lrow == r, so row starts fall out of the run boundaries (as in K1d): no counting
//         pass, no scan, no atomics; rows without edges (isolated nodes, trailing ones, edge-free graphs) point at the
//         next run;
//       - symmetric => the dst-major and src-major orientations have the same rowptr / colidx / val, written once;
//       - src-major t_eid is the identity (slot = edge position); dst-major eid is the position of the REVERSE edge,
//         found by a binary search in the target's row -- the same search verifies symmetry.
// The kernel VERIFIES the promise per graph and ORs TSG_FUSED_* bits (1 range / self loop, 2 order, 4 symmetry) into
// *status; the host raises (tsg.nn.check_fused_status).  A graph that breaks it gets a CSR whose indices all stay inside
// the batch (every edge in the graph's last row), so nothing downstream reads out of bounds before the check.
// Replaces bench.py's host path for these configs (synth.select + synth.pack on the CPU, an int64 edge_index H2D copy,
// K1 tsg_csr_build(CSR_RAW): three passes with global atomics) and the reference's per-graph padded numpy tensors
// (Code/sage+gat+diffpool/tripletnet.py:18-33).
#include "pack_csr.cuh"

namespace tsg {

constexpr int PDENSE_THREADS = 256;

__global__ void __launch_bounds__(PDENSE_THREADS)
k_pack_dense(const int64_t* __restrict__ ids, const int64_t* __restrict__ out_node_ptr,
             const int64_t* __restrict__ out_edge_ptr, int B, int N, int E, const int64_t* __restrict__ c_node_ptr,
             const int64_t* __restrict__ c_edge_ptr, const int32_t* __restrict__ lrow, const int32_t* __restrict__ lcol,
             const float* __restrict__ table, int nmax, int F, bool vec4, float* __restrict__ x_out,
             uint8_t* __restrict__ has_pad, int32_t* __restrict__ rowptr, int32_t* __restrict__ colidx,
             float* __restrict__ val, int32_t* __restrict__ eid, int32_t* __restrict__ t_eid, int* __restrict__ status) {
  extern __shared__ __align__(16) unsigned char sm[];
  int* rs = reinterpret_cast<int*>(sm);                       // [nmax + 2] first edge of every row
  __shared__ int s_bad;
  const int tid = threadIdx.x;
  if (rowptr != nullptr && blockIdx.x == 0 && tid == 0) rowptr[N] = E;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const int64_t g = ids[b];
    const int64_t cn = c_node_ptr[g], ce = c_edge_ptr[g];
    const int n = (int)(c_node_ptr[g + 1] - cn), e = (int)(c_edge_ptr[g + 1] - ce);
    const int64_t nb = out_node_ptr[b], ob = out_edge_ptr[b];
    if (tid == 0) has_pad[b] = n < nmax ? 1 : 0;
    // features: rows 0..n-1 of the table (a row past the table, which the host rules out, is written as zeros)
    if (vec4) {
      const int F4 = F >> 2;
      const float4* t4 = reinterpret_cast<const float4*>(table);
      float4* x4 = reinterpret_cast<float4*>(x_out) + nb * F4;
      const int64_t total = (int64_t)n * F4;
      for (int64_t i = tid; i < total; i += PDENSE_THREADS) {
        const int64_t v = i / F4;
        x4[i] = v < nmax ? __ldg(t4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    } else {
      float* xo = x_out + nb * F;
      const int64_t total = (int64_t)n * F;
      for (int64_t i = tid; i < total; i += PDENSE_THREADS) xo[i] = i / F < nmax ? __ldg(table + i) : 0.f;
    }
    if (rowptr == nullptr) continue;                          // features and pad flags only (general-path callers)

    if (tid == 0) s_bad = n > nmax ? TSG_FUSED_BAD_EDGE : 0;
    __syncthreads();
    int bad = 0;
    if (n <= nmax) bad = coalesced_row_starts(lrow + ce, lcol + ce, n, e, rs, tid, PDENSE_THREADS);
    if (bad) atomicOr(&s_bad, bad);
    __syncthreads();
    const int sb = s_bad;
    if (sb) {                                                 // uniform: report, keep every index inside the batch
      if (tid == 0) atomicOr(status, sb);
      for (int r = tid; r < n; r += PDENSE_THREADS) rowptr[nb + r] = (int32_t)ob;
      const int32_t last = (int32_t)(n > 0 ? nb + n - 1 : (nb < N ? nb : N - 1));
      for (int p = tid; p < e; p += PDENSE_THREADS) {
        const int64_t o = ob + p;
        colidx[o] = last < 0 ? 0 : last;
        val[o] = 1.0f;
        if (eid) eid[o] = (int32_t)o;
        if (t_eid) t_eid[o] = (int32_t)o;
      }
      __syncthreads();
      continue;
    }
    // row starts: the graph's rows 0..n-1 (row n is the next graph's row 0, or rowptr[N] written above)
    for (int r = tid; r < n; r += PDENSE_THREADS) rowptr[nb + r] = (int32_t)(ob + rs[r]);
    bad = 0;
    for (int p = tid; p < e; p += PDENSE_THREADS) {
      const int r = lrow[ce + p], q = lcol[ce + p];
      const int64_t o = ob + p;
      colidx[o] = (int32_t)(nb + q);
      val[o] = 1.0f;
      if (t_eid) t_eid[o] = (int32_t)o;                        // src-major: slot o holds edge o itself
      // dst-major: slot o is row r's entry q, i.e. the edge (q -> r); its position is r's place in row q
      int at = coalesced_find(lcol + ce, rs, q, r);
      if (at < 0) { bad |= TSG_FUSED_ASYMMETRIC; at = p; }
      if (eid) eid[o] = (int32_t)(ob + at);
    }
    if (bad) atomicOr(status, bad);
    __syncthreads();                                          // rs is reused by the next graph
  }
}

}  // namespace tsg

using namespace tsg;

extern "C" int tsg_pack_dense_batch(const int64_t* ids, const int64_t* out_node_ptr, const int64_t* out_edge_ptr,
                                    int64_t B, int64_t N, int64_t E, const int64_t* c_node_ptr,
                                    const int64_t* c_edge_ptr, const int32_t* c_row, const int32_t* c_col,
                                    const float* table, int64_t max_nodes, int64_t F, float* x_out, uint8_t* has_pad,
                                    int32_t* rowptr, int32_t* colidx, float* val, int32_t* eid, int32_t* t_eid,
                                    int32_t* status, void* stream) {
  const int64_t lim = (int64_t)0x7fffffff;
  TSG_REQUIRE(B > 0 && B < lim && N >= 0 && E >= 0 && N + E < lim, "pack_dense_batch: bad sizes (B %lld, N %lld, E %lld)",
              (long long)B, (long long)N, (long long)E);
  TSG_REQUIRE(F > 0 && F < lim && max_nodes > 0 && max_nodes < lim && N * F < ((int64_t)1 << 62),
              "pack_dense_batch: bad feature table shape [%lld, %lld]", (long long)max_nodes, (long long)F);
  TSG_REQUIRE(ids && out_node_ptr && out_edge_ptr && c_node_ptr && c_edge_ptr && table && has_pad &&
              (N == 0 || x_out), "pack_dense_batch: null pointer");
  TSG_REQUIRE(!rowptr || (status && (E == 0 || (c_row && c_col && colidx && val))),
              "pack_dense_batch: null CSR pointer");
  const size_t smem = rowptr ? (size_t)(max_nodes + 2) * 4 : 0;     // rs[]: one run start per row
  TSG_REQUIRE(smem <= 48 * 1024, "pack_dense_batch: a graph of %lld nodes exceeds the shared-memory budget (%d nodes)",
              (long long)max_nodes, 48 * 1024 / 4 - 2);
  const bool vec4 = F % 4 == 0 && ((reinterpret_cast<uintptr_t>(table) | reinterpret_cast<uintptr_t>(x_out)) & 15) == 0;
  const int grid = (int)(B < (int64_t)TSG_NUM_SMS * 8 ? B : (int64_t)TSG_NUM_SMS * 8);
  k_pack_dense<<<grid, PDENSE_THREADS, smem, (cudaStream_t)stream>>>(
      ids, out_node_ptr, out_edge_ptr, (int)B, (int)N, (int)E, c_node_ptr, c_edge_ptr, c_row, c_col, table,
      (int)max_nodes, (int)F, vec4, x_out, has_pad, rowptr, colidx, val, eid, t_eid, status);
  return check_launch("pack_dense_batch");
}
