// K17 -- a resident corpus's EigenPooling operands built on the GPU (tsg.feeder.DeviceCorpus.build_eigen), in the
// layout DeviceCorpus.attach_eigen uploads.  Replaces the per-graph numpy / scipy loop of tsg.eigen_synth
// (make_operands / operands_from_clusters), i.e. the work of Code/eigengcn/coarsen_pooling_with_last_eigen_padding.py
// :121-182 with the clustering of :125-126 replaced by eigen_synth's BFS chunks or by labels the caller supplies.
// The host drives it over chunks of consecutive graphs; in a chunk, graph g's nodes sit at chunk offset nb (its corpus
// node offset minus the chunk's) and its edges at ob, and its clusters take the ids nb + local id.  A graph has at most
// as many clusters as nodes, so these ids need no scan: cluster rows nb + nc .. nb + n - 1 are simply empty.
//   k_eigen_bfs     the synthetic clustering (eigen_synth.bfs_clusters): queue BFS from node 0 over ascending
//                   neighbour lists, unreached nodes appended in ascending order, chunks of pool_size in that order;
//   k_eigen_group   the clusters of given labels, members in ascending node order (operands_from_clusters);
//   k_eigen_coarse  per graph, the sorted, merged (cl[row], cl[col], count) list of the inter-cluster edges
//                   (np.nonzero of Omega^T A_ext Omega, coarsen...py:135-149): a counting pass and a writing pass;
//   k_eigen_final   the final pooling: first eigenvectors of the Laplacian of the binary coarse adjacency over all of
//                   a graph's clusters (:150-182 with one cluster holding every coarse node), the sign and repeat
//                   rules of K11.  One CTA per graph, fp64 cyclic Jacobi; graphs above TSG_EIGEN_FINAL_MAX clusters
//                   are left to the host.
// The per-cluster eigenvectors are K11's k_cluster_eig (tsg_eigpool_build), fed with the chunk CSR, cluster ids and
// member lists the first two kernels write.
#include "pack_csr.cuh"

#include <limits.h>

namespace tsg {

constexpr int EB_THREADS = 256;
constexpr int EF_THREADS = 128;
constexpr int EB_MAX_NODES = TSG_EIGEN_BUILD_MAX_NODES;
constexpr int EF_MAX = TSG_EIGEN_FINAL_MAX;
constexpr size_t EB_MAX_SMEM = 227 * 1024;                   // sm_100 opt-in limit per block
static_assert((3 * (size_t)EB_MAX_NODES + 2) * 4 <= EB_MAX_SMEM, "node cap exceeds the shared-memory budget");
static_assert(2 * (size_t)EF_MAX * (EF_MAX + 1) * 8 + EF_MAX * 4 <= EB_MAX_SMEM, "final cap exceeds shared memory");
static_assert(EF_MAX <= EF_THREADS, "one thread per coarse node");

// Graph g's rows of the chunk CSR (rowptr [nb + u] = ob + start of row u, colidx = nb + local column; val = 1 is
// implied), verified like K0d: range / self loop, order and symmetry.  rs [n + 1] (shared) receives the row starts.
// A graph that breaks the promise is recorded in *bad_graph and gets empty rows, so nothing reads out of bounds.
__device__ void graph_csr(const int32_t* __restrict__ lrow, const int32_t* __restrict__ lcol, int n, int e, int nb,
                          int ob, int64_t g, int* rs, int* s_bad, int32_t* __restrict__ rowptr,
                          int32_t* __restrict__ colidx, int* bad_graph) {
  const int tid = threadIdx.x;
  if (tid == 0) *s_bad = 0;
  __syncthreads();
  int bad = coalesced_row_starts(lrow, lcol, n, e, rs, tid, EB_THREADS);
  if (bad) atomicOr(s_bad, bad);
  __syncthreads();
  if (*s_bad == 0) {
    for (int p = tid; p < e; p += EB_THREADS)
      if (coalesced_find(lcol, rs, lcol[p], lrow[p]) < 0) { atomicOr(s_bad, TSG_FUSED_ASYMMETRIC); break; }
  }
  __syncthreads();
  if (*s_bad) {
    if (tid == 0) atomicMin(bad_graph, (int)g);
    for (int r = tid; r <= n; r += EB_THREADS) rs[r] = 0;
  }
  __syncthreads();
  for (int u = tid; u < n; u += EB_THREADS) rowptr[nb + u] = ob + rs[u];
  for (int p = tid; p < e; p += EB_THREADS) colidx[ob + p] = nb + min(max(lcol[p], 0), max(n - 1, 0));
}

struct ChunkArgs {
  const int64_t *node_ptr, *edge_ptr;
  const int32_t *row, *col;
  int64_t g0;
  int B, N, E, pool_size;
  int32_t* cluster_of;                                        // corpus, graph-local ids (BFS: out, labels: in)
  int32_t* num_clusters;                                      // corpus [G] (nullable for labels)
  int32_t *rowptr, *colidx, *cluster_g, *member_ptr, *member; // chunk
  int* status;                                                // [0] bad edge list, [1] cluster > 32, [2] id >= n
};

__device__ __forceinline__ void chunk_tail(const ChunkArgs& a) {
  if (blockIdx.x == 0 && threadIdx.x == 0) { a.rowptr[a.N] = a.E; a.member_ptr[a.N] = a.N; }
}

// BFS order of every graph (eigen_synth._bfs_order) and its chunks of pool_size.  Level-synchronous: every frontier
// node claims its unvisited neighbours with atomicMax on st = -2 - (its queue position), so each node ends with its
// FIRST discoverer; the frontier then writes its claimed neighbours in queue order, each in its ascending neighbour
// order -- the order a FIFO queue visits them.  st[v] >= 0: v's queue position; INT_MIN: not reached yet.
// Shared memory: rs [n + 1], queue [n], st [n].
__global__ void __launch_bounds__(EB_THREADS) k_eigen_bfs(const ChunkArgs a) {
  extern __shared__ __align__(16) int sm[];
  __shared__ int s_scan[33];
  __shared__ int s_bad;
  const int tid = threadIdx.x;
  chunk_tail(a);
  const int64_t n0 = a.node_ptr[a.g0], e0 = a.edge_ptr[a.g0];
  for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
    const int64_t g = a.g0 + b;
    const int64_t cn = a.node_ptr[g], ce = a.edge_ptr[g];
    const int n = (int)(a.node_ptr[g + 1] - cn), e = (int)(a.edge_ptr[g + 1] - ce);
    const int nb = (int)(cn - n0), ob = (int)(ce - e0);
    int* rs = sm;
    int* queue = sm + n + 1;
    int* st = queue + n;
    graph_csr(a.row + ce, a.col + ce, n, e, nb, ob, g, rs, &s_bad, a.rowptr, a.colidx, &a.status[0]);
    const int32_t* lcol = a.col + ce;
    for (int i = tid; i < n; i += EB_THREADS) st[i] = INT_MIN;
    __syncthreads();
    if (tid == 0 && n > 0) { queue[0] = 0; st[0] = 0; }
    __syncthreads();
    int lo = 0, hi = n > 0 ? 1 : 0;
    while (lo < hi) {
      for (int i = lo + tid; i < hi; i += EB_THREADS) {
        const int u = queue[i];
        for (int p = rs[u]; p < rs[u + 1]; ++p) atomicMax(&st[lcol[p]], -2 - i);   // no effect on visited nodes
      }
      __syncthreads();
      int tail = hi;
      for (int base = lo; base < hi; base += EB_THREADS) {
        const int i = base + tid;
        int cnt = 0;
        if (i < hi) {
          const int u = queue[i];
          for (int p = rs[u]; p < rs[u + 1]; ++p) cnt += st[lcol[p]] == -2 - i;
        }
        int tot;
        int o = tail + block_excl_scan(cnt, s_scan, &tot);
        if (i < hi) {
          const int u = queue[i];
          for (int p = rs[u]; p < rs[u + 1]; ++p) {
            const int v = lcol[p];
            if (st[v] == -2 - i) { queue[o] = v; st[v] = o; ++o; }
          }
        }
        tail += tot;
        __syncthreads();
      }
      lo = hi; hi = tail;
    }
    for (int base = 0; base < n && hi < n; base += EB_THREADS) {   // unreached nodes, ascending
      const int i = base + tid;
      const int un = i < n && st[i] < 0;
      int tot;
      const int o = hi + block_excl_scan(un, s_scan, &tot);
      if (un) queue[o] = i;
      hi += tot;
    }
    __syncthreads();
    const int ps = a.pool_size;
    for (int p = tid; p < n; p += EB_THREADS) {
      const int v = queue[p];
      a.cluster_of[cn + v] = p / ps;
      a.cluster_g[nb + v] = nb + p / ps;
      a.member[nb + p] = nb + v;
      a.member_ptr[nb + p] = nb + min(p * ps, n);
    }
    if (tid == 0) a.num_clusters[g] = (n + ps - 1) / ps;
    __syncthreads();                                          // sm is reused by the next graph
  }
}

// Clusters of given graph-local labels: member lists in ascending node order by a counting sort whose claims are
// ranked by node id (as K0e does), nc = max label + 1.  A label outside [0, n) is recorded in status[2] (and clamped),
// a cluster of more than TSG_EIG_MAX members in status[1].  Shared memory: cs [n + 1], fill [n], tmp [n].
__global__ void __launch_bounds__(EB_THREADS) k_eigen_group(const ChunkArgs a) {
  extern __shared__ __align__(16) int sm[];
  __shared__ int s_scan[33];
  __shared__ int s_bad, s_max;
  const int tid = threadIdx.x;
  chunk_tail(a);
  const int64_t n0 = a.node_ptr[a.g0], e0 = a.edge_ptr[a.g0];
  for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
    const int64_t g = a.g0 + b;
    const int64_t cn = a.node_ptr[g], ce = a.edge_ptr[g];
    const int n = (int)(a.node_ptr[g + 1] - cn), e = (int)(a.edge_ptr[g + 1] - ce);
    const int nb = (int)(cn - n0), ob = (int)(ce - e0);
    graph_csr(a.row + ce, a.col + ce, n, e, nb, ob, g, sm, &s_bad, a.rowptr, a.colidx, &a.status[0]);
    __syncthreads();                                          // sm is reused below
    int* cs = sm;
    int* fill = sm + n + 1;
    int* tmp = sm + 2 * n + 1;
    for (int c = tid; c < 2 * n + 1; c += EB_THREADS) sm[c] = 0;
    if (tid == 0) s_max = -1;
    __syncthreads();
    const int32_t* cl = a.cluster_of + cn;
    for (int i = tid; i < n; i += EB_THREADS) {
      int c = cl[i];
      if ((unsigned)c >= (unsigned)n) { atomicMin(&a.status[2], (int)g); c = c < 0 ? 0 : n - 1; }
      atomicAdd(&cs[c], 1);
      atomicMax(&s_max, c);
    }
    __syncthreads();
    {                                                         // exclusive scan of the counts, chunk per thread
      const int per = (n + EB_THREADS - 1) / EB_THREADS;
      const int c0 = min(tid * per, n), c1 = min(c0 + per, n);
      int s = 0, big = 0;
      for (int c = c0; c < c1; ++c) { s += cs[c]; big |= cs[c] > TSG_EIG_MAX; }
      if (big) atomicMin(&a.status[1], (int)g);
      int tot;
      int run = block_excl_scan(s, s_scan, &tot);
      for (int c = c0; c < c1; ++c) { const int v = cs[c]; cs[c] = run; run += v; }
      if (tid == 0) cs[n] = n;
    }
    __syncthreads();
    for (int i = tid; i < n; i += EB_THREADS) {
      const int c = min(max(cl[i], 0), n - 1);
      tmp[cs[c] + atomicAdd(&fill[c], 1)] = i;
    }
    for (int c = tid; c < n; c += EB_THREADS) a.member_ptr[nb + c] = nb + cs[c];   // rows past nc: empty
    __syncthreads();
    for (int p = tid; p < n; p += EB_THREADS) {
      const int i = tmp[p];
      const int c = min(max(cl[i], 0), n - 1);
      const int s = cs[c], t = cs[c + 1];
      int rank = 0;
      for (int q = s; q < t; ++q) rank += tmp[q] < i;
      a.member[nb + s + rank] = nb + i;
      a.cluster_g[nb + i] = nb + c;
    }
    if (tid == 0 && a.num_clusters) a.num_clusters[g] = s_max + 1;
    __syncthreads();                                          // sm is reused by the next graph
  }
}

// One warp: the coarse entries of cluster row r = (nb + r): the distinct clusters c != r that its members' edges
// reach, ascending, each with its edge count, found one value per pass (a warp-wide min over the values above the
// last one).  Writes them at out[o..] when out_row is given; returns their number.
__device__ int coarse_row(int r, int nb, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                          const int32_t* __restrict__ cluster_g, const int32_t* __restrict__ member_ptr,
                          const int32_t* __restrict__ member, int32_t* out_row, int32_t* out_col, float* out_w,
                          int64_t o) {
  const int lane = threadIdx.x & 31;
  const int rg = nb + r, m0 = member_ptr[rg], m1 = member_ptr[rg + 1];
  int cur = -1, count = 0;
  while (true) {
    int best = INT_MAX, hits = 0;
    for (int m = m0; m < m1; ++m) {
      const int u = member[m];
      for (int p = rowptr[u] + lane; p < rowptr[u + 1]; p += 32) {
        const int c = cluster_g[colidx[p]];
        if (c == rg || c <= cur) continue;
        if (c < best) { best = c; hits = 1; } else if (c == best) ++hits;
      }
    }
    int wbest = best;
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) wbest = min(wbest, __shfl_xor_sync(0xffffffffu, wbest, s));
    if (wbest == INT_MAX) break;
    hits = best == wbest ? hits : 0;
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) hits += __shfl_xor_sync(0xffffffffu, hits, s);
    if (out_row && lane == 0) { out_row[o + count] = r; out_col[o + count] = wbest - nb; out_w[o + count] = (float)hits; }
    ++count;
    cur = wbest;
  }
  return count;
}

struct CoarseArgs {
  const int64_t* node_ptr;
  int64_t g0;
  int B;
  const int32_t *num_clusters, *rowptr, *colidx, *cluster_g, *member_ptr, *member;
  int32_t* row_off;                                           // chunk [N]: per-row counts, then offsets
  int32_t* num_coarse;                                        // corpus [G] (counting pass)
  const int64_t* coarse_ptr;                                  // corpus [G + 1] (writing pass)
  int32_t *coarse_row, *coarse_col;
  float* coarse_w;
};

template <bool WRITE>
__global__ void __launch_bounds__(EB_THREADS) k_eigen_coarse(const CoarseArgs a) {
  __shared__ int s_scan[33];
  __shared__ int s_tot;
  const int tid = threadIdx.x, warp = tid >> 5;
  constexpr int WARPS = EB_THREADS / 32;
  const int64_t n0 = a.node_ptr[a.g0];
  for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
    const int64_t g = a.g0 + b;
    const int nb = (int)(a.node_ptr[g] - n0), nc = a.num_clusters[g];
    if (tid == 0) s_tot = 0;
    __syncthreads();
    for (int r = warp; r < nc; r += WARPS) {
      const int cnt = coarse_row(r, nb, a.rowptr, a.colidx, a.cluster_g, a.member_ptr, a.member, nullptr, nullptr,
                                 nullptr, 0);
      if ((tid & 31) == 0) { if (WRITE) a.row_off[nb + r] = cnt; else atomicAdd(&s_tot, cnt); }
    }
    __syncthreads();
    if (!WRITE) {
      if (tid == 0) a.num_coarse[g] = s_tot;
      continue;
    }
    int carry = 0;                                            // row counts -> row offsets, in rounds of the block
    for (int base = 0; base < nc; base += EB_THREADS) {
      const int r = base + tid;
      const int v = r < nc ? a.row_off[nb + r] : 0;
      int tot;
      const int ex = block_excl_scan(v, s_scan, &tot);
      if (r < nc) a.row_off[nb + r] = carry + ex;
      carry += tot;
    }
    __syncthreads();
    const int64_t q0 = a.coarse_ptr[g];
    for (int r = warp; r < nc; r += WARPS)
      coarse_row(r, nb, a.rowptr, a.colidx, a.cluster_g, a.member_ptr, a.member, a.coarse_row, a.coarse_col,
                 a.coarse_w, q0 + a.row_off[nb + r]);
    __syncthreads();                                          // row_off of this graph is read before the next
  }
}

// Final pooling of graphs with lo < nc <= ld - 1 clusters (others are skipped: another size class, or the host).  A = D - W of the binary coarse
// adjacency, V = I; cyclic Jacobi as K11's k_cluster_eig with thread k owning row / column k; eigenpairs ranked by
// (eigenvalue, column); vector j = rank min(j, nc - 1), sign fixed on its first entry.
__global__ void __launch_bounds__(EF_THREADS)
k_eigen_final(const int64_t* __restrict__ cluster_ptr, const int64_t* __restrict__ coarse_ptr,
              const int32_t* __restrict__ crow, const int32_t* __restrict__ ccol, int64_t g0, int B, int lo, int ld,
              int num_vec, float* __restrict__ final_w, int64_t stride) {
  extern __shared__ __align__(16) double dsm[];
  __shared__ double s_red[2][EF_THREADS / 32];
  double* A = dsm;
  double* V = dsm + (size_t)(ld - 1) * ld;
  int* rank = (int*)(V + (size_t)(ld - 1) * ld);
  const int k = threadIdx.x, lane = k & 31, w = k >> 5;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const int64_t g = g0 + b;
    const int64_t c0 = cluster_ptr[g];
    const int nc = (int)(cluster_ptr[g + 1] - c0);
    if (nc > ld - 1 || nc <= lo || nc == 0) continue;        // uniform
    for (int i = 0; i < nc; ++i) if (k < nc) { A[i * ld + k] = 0.0; V[i * ld + k] = i == k ? 1.0 : 0.0; }
    __syncthreads();
    const int64_t q0 = coarse_ptr[g], q1 = coarse_ptr[g + 1];
    for (int64_t q = q0 + k; q < q1; q += EF_THREADS) {
      const int r = crow[q], c = ccol[q];
      if ((unsigned)r < (unsigned)nc && (unsigned)c < (unsigned)nc && r != c) A[r * ld + c] = -1.0;
    }
    __syncthreads();
    if (k < nc) {
      double deg = 0.0;
      for (int c = 0; c < nc; ++c) deg -= A[k * ld + c];
      A[k * ld + k] = deg;
    }
    __syncthreads();
    for (int sweep = 0; sweep < 30; ++sweep) {
      double off = 0.0, diag = 0.0;
      if (k < nc)
        for (int q = 0; q < nc; ++q) { const double v = A[k * ld + q]; if (q == k) diag += v * v; else off += v * v; }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) { off += __shfl_xor_sync(0xffffffffu, off, o); diag += __shfl_xor_sync(0xffffffffu, diag, o); }
      if (lane == 0) { s_red[0][w] = off; s_red[1][w] = diag; }
      __syncthreads();
      off = 0.0; diag = 0.0;
#pragma unroll
      for (int i = 0; i < EF_THREADS / 32; ++i) { off += s_red[0][i]; diag += s_red[1][i]; }
      __syncthreads();
      if (off <= 1e-26 * (diag + 1e-300) || off == 0.0) break;
      for (int p = 0; p < nc - 1; ++p) {
        for (int q = p + 1; q < nc; ++q) {
          const double apq = A[p * ld + q];
          if (fabs(apq) > 1e-300) {
            const double app = A[p * ld + p], aqq = A[q * ld + q];
            const double theta = (aqq - app) / (2.0 * apq);
            const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
            const double cs = 1.0 / sqrt(t * t + 1.0), sn = t * cs;
            __syncthreads();
            if (k < nc) {
              if (k != p && k != q) {
                const double akp = A[k * ld + p], akq = A[k * ld + q];
                const double nkp = cs * akp - sn * akq, nkq = sn * akp + cs * akq;
                A[k * ld + p] = nkp; A[p * ld + k] = nkp; A[k * ld + q] = nkq; A[q * ld + k] = nkq;
              }
              const double vkp = V[k * ld + p], vkq = V[k * ld + q];
              V[k * ld + p] = cs * vkp - sn * vkq; V[k * ld + q] = sn * vkp + cs * vkq;
            }
            __syncthreads();
            if (k == 0) { A[p * ld + p] = app - t * apq; A[q * ld + q] = aqq + t * apq; A[p * ld + q] = 0.0; A[q * ld + p] = 0.0; }
            __syncthreads();
          }
        }
      }
    }
    if (k < nc) {
      const double lam = A[k * ld + k];
      int r = 0;
      for (int q = 0; q < nc; ++q) { const double lq = A[q * ld + q]; r += (lq < lam) || (lq == lam && q < k); }
      rank[r] = k;
    }
    __syncthreads();
    for (int j = 0; j < num_vec; ++j) {
      const int col = rank[min(j, nc - 1)];
      const double sgn = V[col] < 0.0 ? -1.0 : 1.0;           // V[0][col]
      if (k < nc) final_w[(int64_t)j * stride + c0 + k] = (float)(sgn * V[k * ld + col]);
    }
    __syncthreads();                                          // shared memory is reused by the next graph
  }
}

static inline int eb_grid(int64_t B) { return (int)(B < (int64_t)TSG_NUM_SMS * 8 ? B : (int64_t)TSG_NUM_SMS * 8); }

template <typename K>
static int set_smem(K kernel, size_t smem, const char* what) {
  if (smem > 48 * 1024 && cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return check_launch(what);
  return TSG_OK;
}

static int chunk_checks(const int64_t* node_ptr, const int64_t* edge_ptr, const int32_t* row, const int32_t* col,
                        int64_t g0, int64_t B, int64_t N, int64_t E, int64_t max_nodes, int32_t* rowptr,
                        int32_t* colidx, int32_t* cluster_g, int32_t* member_ptr, int32_t* member, int32_t* status) {
  const int64_t lim = (int64_t)0x7fffffff;
  TSG_REQUIRE(g0 >= 0 && B > 0 && B < lim && N >= 0 && E >= 0 && N + E < lim,
              "eigen build: bad chunk (first graph %lld, %lld graphs, %lld nodes, %lld edges)", (long long)g0,
              (long long)B, (long long)N, (long long)E);
  TSG_REQUIRE(max_nodes >= 0 && max_nodes <= EB_MAX_NODES, "eigen build: a graph of %lld nodes exceeds the cap (%d)",
              (long long)max_nodes, EB_MAX_NODES);
  TSG_REQUIRE(node_ptr && edge_ptr && rowptr && member_ptr && status, "eigen build: null pointer");
  TSG_REQUIRE(N == 0 || (cluster_g && member), "eigen build: null node-sized pointer");
  TSG_REQUIRE(E == 0 || (row && col && colidx), "eigen build: null edge-sized pointer");
  return TSG_OK;
}

}  // namespace tsg

using namespace tsg;

extern "C" int tsg_eigen_bfs_clusters(const int64_t* node_ptr, const int64_t* edge_ptr, const int32_t* row,
                                      const int32_t* col, int64_t first_graph, int64_t num_graphs, int64_t num_nodes,
                                      int64_t num_edges, int64_t max_nodes, int64_t pool_size, int32_t* cluster_of,
                                      int32_t* num_clusters, int32_t* rowptr, int32_t* colidx, int32_t* cluster_g,
                                      int32_t* member_ptr, int32_t* member, int32_t* status, void* stream) {
  int rc = chunk_checks(node_ptr, edge_ptr, row, col, first_graph, num_graphs, num_nodes, num_edges, max_nodes, rowptr,
                        colidx, cluster_g, member_ptr, member, status);
  if (rc) return rc;
  TSG_REQUIRE(pool_size >= 1 && pool_size <= TSG_EIG_MAX, "eigen_bfs_clusters: pool_size %lld outside [1, %d]",
              (long long)pool_size, TSG_EIG_MAX);
  TSG_REQUIRE(num_clusters && (num_nodes == 0 || cluster_of), "eigen_bfs_clusters: null pointer");
  const size_t smem = (size_t)(3 * max_nodes + 2) * 4;
  if ((rc = set_smem(k_eigen_bfs, smem, "eigen_bfs_clusters (shared-memory opt-in)"))) return rc;
  ChunkArgs a{node_ptr, edge_ptr, row, col, first_graph, (int)num_graphs, (int)num_nodes, (int)num_edges,
              (int)pool_size, cluster_of, num_clusters, rowptr, colidx, cluster_g, member_ptr, member, status};
  k_eigen_bfs<<<eb_grid(num_graphs), EB_THREADS, smem, (cudaStream_t)stream>>>(a);
  return check_launch("eigen_bfs_clusters");
}

extern "C" int tsg_eigen_group_clusters(const int64_t* node_ptr, const int64_t* edge_ptr, const int32_t* row,
                                        const int32_t* col, int64_t first_graph, int64_t num_graphs, int64_t num_nodes,
                                        int64_t num_edges, int64_t max_nodes, const int32_t* cluster_of,
                                        int32_t* num_clusters, int32_t* rowptr, int32_t* colidx, int32_t* cluster_g,
                                        int32_t* member_ptr, int32_t* member, int32_t* status, void* stream) {
  int rc = chunk_checks(node_ptr, edge_ptr, row, col, first_graph, num_graphs, num_nodes, num_edges, max_nodes, rowptr,
                        colidx, cluster_g, member_ptr, member, status);
  if (rc) return rc;
  TSG_REQUIRE(num_nodes == 0 || cluster_of, "eigen_group_clusters: null cluster_of");
  const size_t smem = (size_t)(3 * max_nodes + 2) * 4;
  if ((rc = set_smem(k_eigen_group, smem, "eigen_group_clusters (shared-memory opt-in)"))) return rc;
  ChunkArgs a{node_ptr, edge_ptr, row, col, first_graph, (int)num_graphs, (int)num_nodes, (int)num_edges, 0,
              const_cast<int32_t*>(cluster_of), num_clusters, rowptr, colidx, cluster_g, member_ptr, member, status};
  k_eigen_group<<<eb_grid(num_graphs), EB_THREADS, smem, (cudaStream_t)stream>>>(a);
  return check_launch("eigen_group_clusters");
}

extern "C" int tsg_eigen_coarse(const int64_t* node_ptr, int64_t first_graph, int64_t num_graphs,
                                const int32_t* num_clusters, const int32_t* rowptr, const int32_t* colidx,
                                const int32_t* cluster_g, const int32_t* member_ptr, const int32_t* member,
                                int32_t* row_scratch, int32_t* num_coarse, const int64_t* coarse_ptr,
                                int32_t* coarse_row, int32_t* coarse_col, float* coarse_w, void* stream) {
  TSG_REQUIRE(first_graph >= 0 && num_graphs > 0 && num_graphs < (int64_t)0x7fffffff, "eigen_coarse: bad chunk");
  TSG_REQUIRE(node_ptr && num_clusters && rowptr && member_ptr, "eigen_coarse: null pointer");
  const bool write = coarse_row != nullptr;
  TSG_REQUIRE(write ? (coarse_ptr && coarse_col && coarse_w && row_scratch) : num_coarse != nullptr,
              "eigen_coarse: give num_coarse (counting) or coarse_ptr, row_scratch and the three outputs (writing)");
  CoarseArgs a{node_ptr, first_graph, (int)num_graphs, num_clusters, rowptr, colidx, cluster_g, member_ptr, member,
               row_scratch, num_coarse, coarse_ptr, coarse_row, coarse_col, coarse_w};
  if (write) k_eigen_coarse<true><<<eb_grid(num_graphs), EB_THREADS, 0, (cudaStream_t)stream>>>(a);
  else k_eigen_coarse<false><<<eb_grid(num_graphs), EB_THREADS, 0, (cudaStream_t)stream>>>(a);
  return check_launch("eigen_coarse");
}

extern "C" int tsg_eigen_final(const int64_t* cluster_ptr, const int64_t* coarse_ptr, const int32_t* coarse_row,
                               const int32_t* coarse_col, int64_t first_graph, int64_t num_graphs, int64_t min_clusters,
                               int64_t max_clusters, int64_t num_vectors, float* final_w, int64_t final_stride,
                               void* stream) {
  TSG_REQUIRE(first_graph >= 0 && num_graphs > 0 && num_graphs < (int64_t)0x7fffffff, "eigen_final: bad chunk");
  TSG_REQUIRE(max_clusters >= 1 && max_clusters <= EF_MAX && min_clusters >= 0 && min_clusters < max_clusters,
              "eigen_final: cluster range (%lld, %lld] outside (0, %d]", (long long)min_clusters, (long long)max_clusters,
              EF_MAX);
  TSG_REQUIRE(num_vectors >= 1 && final_stride >= 0, "eigen_final: bad num_vectors %lld", (long long)num_vectors);
  TSG_REQUIRE(cluster_ptr && coarse_ptr && final_w, "eigen_final: null pointer");
  const int ld = (int)max_clusters + 1;
  const size_t smem = 2 * (size_t)max_clusters * ld * 8 + (size_t)max_clusters * 4;
  int rc = set_smem(k_eigen_final, smem, "eigen_final (shared-memory opt-in)");
  if (rc) return rc;
  k_eigen_final<<<eb_grid(num_graphs), EF_THREADS, smem, (cudaStream_t)stream>>>(
      cluster_ptr, coarse_ptr, coarse_row, coarse_col, first_graph, (int)num_graphs, (int)min_clusters, ld,
      (int)num_vectors, final_w,
      final_stride);
  return check_launch("eigen_final");
}
