// K0e -- device-side assembly of an EigenGCN batch (WavePoolingGcnEncoder + Pool, Code/eigengcn) from an HBM-resident
// corpus and its resident per-graph EigenPooling operands (cluster label and pooling weights per node, coarsened
// adjacency entries and final-pooling weights per graph; tsg.feeder.DeviceCorpus.attach_eigen).  One launch writes
// everything tsg.dense.PackedWaveEncoder takes for the chosen graphs, each array equal to the host path it replaces:
//   * x [N, F]: one-hot of the node labels (what K0 tsg_pack_batch writes);
//   * the RAW 0/1 CSR of the packed adjacency (= tsg_csr_build(TSG_CSR_RAW) on the expanded edge_index), one
//     orientation serving as its own transpose, row starts from run boundaries (pack_csr.cuh, shared with K0d);
//   * P_j^T for j < J (= dense.build_rect_csr on the (node -> cluster, pool_w[j]) list): rows = batch-global clusters
//     whose members are listed in ascending node order; transposed side = one entry per node (arange(N+1), its global
//     cluster, pool_w[j] in node order).  The members are placed by a per-graph counting sort in shared memory whose
//     slot claims (atomics) are then ranked by node id, so the order does not depend on which atomic came first;
//   * the coarsened adjacency (= tsg_csr_build(TSG_CSR_RAW, edge_weight) on the relabelled (cluster, cluster, count)
//     entries), one orientation serving as its own transpose, row starts from run boundaries;
//   * the final pooling for j < Jf (= build_rect_csr on (cluster -> graph, final_w[j])): G rows over the batch's clusters;
//   * has_pad [3, B]: n_b < max_nodes, nc_b < max_nodes, 1 < max_nodes -- whether the reference's max_nodes padding
//     leaves a zero row at level 0, at the pooled level and after the final pooling (one real row per graph).
// The kernel VERIFIES what it relies on per graph and ORs bits into *status (tsg.nn.check_fused_status raises): the
// adjacency promise as in K0d (1 range / self loop, 2 order, 4 symmetry) and TSG_EIGEN_BAD_OPERANDS (16) for a cluster
// id outside [0, nc), a graph with more clusters than max_nodes (or none while it has nodes), or a coarse entry list
// that is out of range, unsorted, has a self loop or is asymmetric (in position or in weight).  A graph that breaks a
// promise still gets in-range indices (bad cluster ids are clamped; a broken list is put in the graph's last row), so
// nothing downstream reads out of bounds before the check.
// Replaces bench.Config5.assemble + eigenpool.build: K0 + K1 (three atomic passes) for the adjacency, two DeviceRagged
// gathers, repeat_interleave, build_rect_csr for the final pooling, and K11's two K1 builds + tsg_coarsen_edges.
#include "pack_csr.cuh"

namespace tsg {

constexpr int PEIGEN_THREADS = 256;
constexpr int TSG_EIGEN_BAD_OPERANDS = 16;
constexpr size_t PEIGEN_MAX_SMEM = 227 * 1024;               // sm_100 opt-in limit per block

struct EigenPackArgs {
  const int64_t *ids, *out_node_ptr, *out_edge_ptr, *out_cluster_ptr, *out_coarse_ptr;
  int B, N, E, NC, EC, F, nmax, J, Jf;
  const int64_t *c_node_ptr, *c_edge_ptr, *c_cluster_ptr, *c_coarse_ptr;
  const int32_t *c_label, *c_row, *c_col, *cluster_of, *coarse_row, *coarse_col;
  const float *pool_w, *coarse_w, *final_w;
  int64_t pool_stride, final_stride;
  float* x;
  uint8_t* has_pad;
  int32_t *rowptr, *colidx;
  float* val;
  int32_t *member_ptr, *member, *node_iota, *node_cluster;
  float *pool_val, *pool_val_nodes;
  int32_t *coarse_rowptr, *coarse_colidx;
  float* coarse_val;
  int32_t *final_rowptr, *cluster_iota, *cluster_graph;
  float* final_val;
  int64_t* graph_iota;
  int* status;
};

__global__ void __launch_bounds__(PEIGEN_THREADS) k_pack_eigen(const EigenPackArgs a) {
  extern __shared__ __align__(16) int sm[];                  // 3 * nmax + 2 ints, reused by the three phases
  __shared__ int s_scan[33];
  __shared__ int s_bad;
  const int tid = threadIdx.x;
  const int B = a.B, N = a.N, NC = a.NC, nmax = a.nmax;
  if (blockIdx.x == 0 && tid == 0) {                          // the trailing entries of every pointer array
    if (a.rowptr) a.rowptr[N] = a.E;
    a.member_ptr[NC] = N; a.node_iota[N] = N; a.coarse_rowptr[NC] = a.EC; a.graph_iota[B] = B;
    if (a.Jf > 0) { a.final_rowptr[B] = NC; a.cluster_iota[NC] = NC; }
  }
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const int64_t g = a.ids[b];
    const int64_t cn = a.c_node_ptr[g], ce = a.c_edge_ptr[g], gc = a.c_cluster_ptr[g], gq = a.c_coarse_ptr[g];
    const int n = (int)(a.c_node_ptr[g + 1] - cn), e = (int)(a.c_edge_ptr[g + 1] - ce);
    const int nb = (int)a.out_node_ptr[b], ob = (int)a.out_edge_ptr[b];
    const int cb = (int)a.out_cluster_ptr[b], nc = (int)(a.out_cluster_ptr[b + 1] - cb);
    const int qb = (int)a.out_coarse_ptr[b], ec = (int)(a.out_coarse_ptr[b + 1] - qb);
    if (tid == 0) {
      a.has_pad[b] = n < nmax; a.has_pad[B + b] = nc < nmax; a.has_pad[2 * B + b] = 1 < nmax;
      a.graph_iota[b] = b;
      if (a.Jf > 0) a.final_rowptr[b] = cb;
    }
    // x: one-hot of the labels; the transposed side of P_j^T (one entry per node, weights in node order)
    for (int64_t i = tid; i < (int64_t)n * a.F; i += PEIGEN_THREADS) {
      const int v = (int)(i / a.F);
      a.x[(int64_t)nb * a.F + i] = a.c_label[cn + v] == (int)(i - (int64_t)v * a.F) ? 1.f : 0.f;
    }
    for (int i = tid; i < n; i += PEIGEN_THREADS) {
      a.node_iota[nb + i] = nb + i;
      for (int j = 0; j < a.J; ++j) a.pool_val_nodes[(int64_t)j * N + nb + i] = a.pool_w[j * a.pool_stride + cn + i];
    }
    // final pooling: cluster c of this graph is column c of row b
    for (int c = tid; c < nc && a.Jf > 0; c += PEIGEN_THREADS) {
      a.cluster_iota[cb + c] = cb + c;
      a.cluster_graph[cb + c] = b;
      for (int j = 0; j < a.Jf; ++j) a.final_val[(int64_t)j * NC + cb + c] = a.final_w[j * a.final_stride + gc + c];
    }

    // ---- adjacency (K0d's construction without eids); skipped when the caller builds it with K0 + K1
    if (a.rowptr != nullptr) {
      int* rs = sm;                                           // [nmax + 2]
      if (tid == 0) s_bad = n > nmax ? TSG_FUSED_BAD_EDGE : 0;
      __syncthreads();
      int bad = n <= nmax ? coalesced_row_starts(a.c_row + ce, a.c_col + ce, n, e, rs, tid, PEIGEN_THREADS) : 0;
      if (bad) atomicOr(&s_bad, bad);
      __syncthreads();
      const int sb = s_bad;
      if (sb) {                                               // uniform: report, keep every index inside the batch
        if (tid == 0) atomicOr(a.status, sb);
        for (int r = tid; r < n; r += PEIGEN_THREADS) a.rowptr[nb + r] = ob;
        const int last = n > 0 ? nb + n - 1 : (nb < N ? nb : N - 1);
        for (int p = tid; p < e; p += PEIGEN_THREADS) { a.colidx[ob + p] = last < 0 ? 0 : last; a.val[ob + p] = 1.0f; }
      } else {
        for (int r = tid; r < n; r += PEIGEN_THREADS) a.rowptr[nb + r] = ob + rs[r];
        bad = 0;
        for (int p = tid; p < e; p += PEIGEN_THREADS) {
          const int r = a.c_row[ce + p], q = a.c_col[ce + p];
          a.colidx[ob + p] = nb + q;
          a.val[ob + p] = 1.0f;
          if (coalesced_find(a.c_col + ce, rs, q, r) < 0) bad |= TSG_FUSED_ASYMMETRIC;
        }
        if (bad) atomicOr(a.status, bad);
      }
      __syncthreads();                                        // sm is reused below
    }

    // ---- P_j^T: stable counting sort of the nodes by cluster (cs = cluster starts, fill = claims, tmp = slots)
    const bool ops_fit = nc <= nmax && n <= nmax && (nc > 0 || n == 0);
    const int lastc = nc > 0 ? cb + nc - 1 : (cb > 0 ? cb - 1 : 0);
    if (!ops_fit) {                                           // uniform: every node in the graph's last cluster row
      if (tid == 0) atomicOr(a.status, TSG_EIGEN_BAD_OPERANDS);
      for (int c = tid; c < nc; c += PEIGEN_THREADS) a.member_ptr[cb + c] = nb;
      for (int i = tid; i < n; i += PEIGEN_THREADS) {
        a.member[nb + i] = nb + i;
        a.node_cluster[nb + i] = lastc;
        for (int j = 0; j < a.J; ++j) a.pool_val[(int64_t)j * N + nb + i] = a.pool_w[j * a.pool_stride + cn + i];
      }
      for (int r = tid; r < nc; r += PEIGEN_THREADS) a.coarse_rowptr[cb + r] = qb;
      for (int p = tid; p < ec; p += PEIGEN_THREADS) { a.coarse_colidx[qb + p] = lastc; a.coarse_val[qb + p] = a.coarse_w[gq + p]; }
      continue;
    }
    int* cs = sm;                                             // [nc + 1]
    int* fill = sm + nc + 1;                                  // [nc]
    int* tmp = sm + 2 * nc + 1;                               // [n]
    for (int c = tid; c < 2 * nc + 1; c += PEIGEN_THREADS) sm[c] = 0;
    __syncthreads();
    int obad = 0;
    for (int i = tid; i < n; i += PEIGEN_THREADS) {
      int c = a.cluster_of[cn + i];
      if ((unsigned)c >= (unsigned)nc) { obad = TSG_EIGEN_BAD_OPERANDS; c = c < 0 ? 0 : nc - 1; }
      atomicAdd(&cs[c], 1);
    }
    __syncthreads();
    {                                                         // exclusive scan of the counts, chunk per thread
      const int per = (nc + PEIGEN_THREADS - 1) / PEIGEN_THREADS;
      const int c0 = min(tid * per, nc), c1 = min(c0 + per, nc);
      int s = 0;
      for (int c = c0; c < c1; ++c) s += cs[c];
      int tot;
      int run = block_excl_scan(s, s_scan, &tot);
      for (int c = c0; c < c1; ++c) { const int v = cs[c]; cs[c] = run; run += v; }
      if (tid == 0) cs[nc] = n;
    }
    __syncthreads();
    for (int i = tid; i < n; i += PEIGEN_THREADS) {
      const int c = min(max(a.cluster_of[cn + i], 0), nc - 1);
      tmp[cs[c] + atomicAdd(&fill[c], 1)] = i;
    }
    for (int c = tid; c < nc; c += PEIGEN_THREADS) a.member_ptr[cb + c] = nb + cs[c];
    __syncthreads();
    for (int p = tid; p < n; p += PEIGEN_THREADS) {           // rank the claims by node id: ascending node order
      const int i = tmp[p];
      const int c = min(max(a.cluster_of[cn + i], 0), nc - 1);
      const int s = cs[c], t = cs[c + 1];
      int rank = 0;
      for (int q = s; q < t; ++q) rank += tmp[q] < i;
      const int o = nb + s + rank;
      a.member[o] = nb + i;
      a.node_cluster[nb + i] = cb + c;
      for (int j = 0; j < a.J; ++j) a.pool_val[(int64_t)j * N + o] = a.pool_w[j * a.pool_stride + cn + i];
    }
    __syncthreads();                                          // sm is reused below

    // ---- coarsened adjacency: the (cluster, cluster, count) list, verified like the adjacency plus weight symmetry
    const int32_t* qrow = a.coarse_row + gq;
    const int32_t* qcol = a.coarse_col + gq;
    const float* qw = a.coarse_w + gq;
    int* rs = sm;                                             // [nc + 1]
    if (tid == 0) s_bad = 0;
    __syncthreads();
    int lbad = coalesced_row_starts(qrow, qcol, nc, ec, rs, tid, PEIGEN_THREADS) ? 1 : 0;
    if (lbad | obad) atomicOr(&s_bad, lbad | (obad ? 2 : 0));   // 1: the list is broken, 2: a cluster id was clamped
    __syncthreads();
    if (tid == 0 && s_bad) atomicOr(a.status, TSG_EIGEN_BAD_OPERANDS);
    if (s_bad & 1) {                                          // uniform: the whole list goes to the graph's last row
      for (int r = tid; r < nc; r += PEIGEN_THREADS) a.coarse_rowptr[cb + r] = qb;
      for (int p = tid; p < ec; p += PEIGEN_THREADS) { a.coarse_colidx[qb + p] = lastc; a.coarse_val[qb + p] = qw[p]; }
      __syncthreads();
      continue;
    }
    for (int r = tid; r < nc; r += PEIGEN_THREADS) a.coarse_rowptr[cb + r] = qb + rs[r];
    obad = 0;
    for (int p = tid; p < ec; p += PEIGEN_THREADS) {
      const int r = qrow[p], q = qcol[p];
      const float w = qw[p];
      a.coarse_colidx[qb + p] = cb + q;
      a.coarse_val[qb + p] = w;
      const int at = coalesced_find(qcol, rs, q, r);
      if (at < 0 || qw[at] != w) obad = TSG_EIGEN_BAD_OPERANDS;
    }
    if (obad) atomicOr(a.status, obad);
    __syncthreads();                                          // rs is reused by the next graph
  }
}

}  // namespace tsg

using namespace tsg;

extern "C" int tsg_pack_eigen_batch(
    const int64_t* ids, const int64_t* out_node_ptr, const int64_t* out_edge_ptr, const int64_t* out_cluster_ptr,
    const int64_t* out_coarse_ptr, int64_t B, int64_t N, int64_t E, int64_t NC, int64_t EC,
    const int64_t* c_node_ptr, const int64_t* c_edge_ptr, const int32_t* c_label, const int32_t* c_row,
    const int32_t* c_col, int64_t F, const int64_t* c_cluster_ptr, const int64_t* c_coarse_ptr,
    const int32_t* cluster_of, const float* pool_w, int64_t pool_stride, int64_t J, const int32_t* coarse_row,
    const int32_t* coarse_col, const float* coarse_w, const float* final_w, int64_t final_stride, int64_t Jf,
    int64_t max_nodes, float* x_out, uint8_t* has_pad, int32_t* rowptr, int32_t* colidx, float* val,
    int32_t* member_ptr, int32_t* member, float* pool_val, int32_t* node_iota, int32_t* node_cluster,
    float* pool_val_nodes, int32_t* coarse_rowptr, int32_t* coarse_colidx, float* coarse_val, int32_t* final_rowptr,
    int32_t* cluster_iota, int32_t* cluster_graph, float* final_val, int64_t* graph_iota, int32_t* status,
    void* stream) {
  const int64_t lim = (int64_t)0x7fffffff;
  TSG_REQUIRE(B > 0 && B < lim && N >= 0 && E >= 0 && NC >= 0 && EC >= 0 && N + E < lim && NC + EC < lim,
              "pack_eigen_batch: bad sizes (B %lld, N %lld, E %lld, NC %lld, EC %lld)", (long long)B, (long long)N,
              (long long)E, (long long)NC, (long long)EC);
  TSG_REQUIRE(F > 0 && F < lim && N * F < ((int64_t)1 << 62) && max_nodes > 0 && max_nodes < lim,
              "pack_eigen_batch: bad feature width %lld or max_nodes %lld", (long long)F, (long long)max_nodes);
  TSG_REQUIRE(J > 0 && J < 256 && Jf >= 0 && Jf < 256 && pool_stride >= 0 && pool_stride < lim && final_stride >= 0 &&
              final_stride < lim, "pack_eigen_batch: bad operand counts (J %lld, Jf %lld)", (long long)J, (long long)Jf);
  TSG_REQUIRE(N == 0 || NC > 0, "pack_eigen_batch: %lld nodes but no clusters", (long long)N);
  // arrays with nothing to read or write may be NULL (an empty tensor's data pointer): node-sized ones when N = 0,
  // the coarse entries when EC = 0 (a batch of single-cluster graphs), the adjacency's when E = 0
  TSG_REQUIRE(ids && out_node_ptr && out_edge_ptr && out_cluster_ptr && out_coarse_ptr && c_node_ptr && c_edge_ptr &&
              c_cluster_ptr && c_coarse_ptr && has_pad && member_ptr && node_iota && coarse_rowptr && graph_iota &&
              status, "pack_eigen_batch: null pointer");
  TSG_REQUIRE(N == 0 || (c_label && cluster_of && pool_w && x_out && member && pool_val && node_cluster &&
                         pool_val_nodes), "pack_eigen_batch: null node-sized pointer");
  TSG_REQUIRE(EC == 0 || (coarse_row && coarse_col && coarse_w && coarse_colidx && coarse_val),
              "pack_eigen_batch: null coarse-entry pointer");
  TSG_REQUIRE(Jf == 0 || (final_rowptr && cluster_iota && (NC == 0 || (final_w && cluster_graph && final_val))),
              "pack_eigen_batch: null final-pooling pointer");
  TSG_REQUIRE(!rowptr || E == 0 || (c_row && c_col && colidx && val), "pack_eigen_batch: null adjacency pointer");
  const size_t smem = (size_t)(3 * max_nodes + 2) * 4;
  TSG_REQUIRE(smem <= PEIGEN_MAX_SMEM, "pack_eigen_batch: a graph of %lld nodes exceeds the shared-memory budget (%d nodes)",
              (long long)max_nodes, (int)((PEIGEN_MAX_SMEM / 4 - 2) / 3));
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(k_pack_eigen, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return check_launch("pack_eigen_batch (shared-memory opt-in)");
  EigenPackArgs a{ids, out_node_ptr, out_edge_ptr, out_cluster_ptr, out_coarse_ptr, (int)B, (int)N, (int)E, (int)NC,
                  (int)EC, (int)F, (int)max_nodes, (int)J, (int)Jf, c_node_ptr, c_edge_ptr, c_cluster_ptr, c_coarse_ptr,
                  c_label, c_row, c_col, cluster_of, coarse_row, coarse_col, pool_w, coarse_w, final_w, pool_stride,
                  final_stride, x_out, has_pad, rowptr, colidx, val, member_ptr, member, node_iota, node_cluster, pool_val,
                  pool_val_nodes, coarse_rowptr, coarse_colidx, coarse_val, final_rowptr, cluster_iota, cluster_graph,
                  final_val, graph_iota, status};
  const int grid = (int)(B < (int64_t)TSG_NUM_SMS * 8 ? B : (int64_t)TSG_NUM_SMS * 8);
  k_pack_eigen<<<grid, PEIGEN_THREADS, smem, (cudaStream_t)stream>>>(a);
  return check_launch("pack_eigen_batch");
}
