/*
 * tsg.h -- C ABI of libtsg.so: the B200 (sm_100a) hot path of two-stage-gnn graph-classification
 * training (batched message passing + pooling forward/backward).
 *
 * Every entry point replaces a reference-side operator; the citation on each declaration is the
 * reference file:line (relative to the upstream repo root) whose arithmetic it implements.  The
 * reference reaches these operators through PyTorch-Geometric 1.6.3 / ATen library calls; this
 * library is what a maintainer would bind instead (ctypes stub in INTEGRATION.md).
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host; caller allocates everything
 *     (inputs, outputs, workspace); the compute entry points never allocate, never retain pointers
 *     past return, never synchronise the stream, and are CUDA-graph-capture safe.  The ONE exception
 *     is tsg_init_device(): call it once per device before the first compute call and outside any
 *     stream capture (it cudaMalloc's 16 KB of zeroed counters the fused reduction tails draw from);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*);
 *   - return value: 0 on success, negative TSG_E* on failure; tsg_last_error() gives the message
 *     (thread local).  No exceptions cross the ABI.  There is no CPU fallback.
 *   - features are fp32 row-major; node / edge indices arriving from the PyG surface are int64,
 *     internal CSR indices are int32 (sum n + sum E must stay below 2^31).
 *   - `*_dev` count pointers are optional device-side scalars: when non-NULL the kernels use
 *     min(*ptr, capacity) as the element count, so data-dependent sizes (edges surviving
 *     filter_adj) never need a host synchronisation.
 */
#ifndef TSG_H_
#define TSG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TSG_ABI_VERSION 1

enum {
  TSG_OK = 0,
  TSG_EINVAL = -1,     /* bad shape / null pointer / unsupported size            */
  TSG_EWORKSPACE = -2, /* workspace too small                                    */
  TSG_ELAUNCH = -3,    /* CUDA launch error (message carries cudaGetErrorString) */
  TSG_EARCH = -4       /* device is not sm_100                                   */
};

int tsg_abi_version(void);
const char* tsg_last_error(void);
/* 0 if the current device can run this library (compute capability 10.x), else TSG_EARCH. */
int tsg_check_device(void);
/* One-time, per-device set-up (the only entry point that allocates / synchronises): creates the 4,096-counter pool
 * used by kernels that finish their second-stage reduction in the last CTA.  Idempotent, thread safe.  Entry points
 * that have a separate-launch second stage fall back to it when the pool is missing; tsg_gate_score_bwd and the
 * executor entries return TSG_EINVAL. */
int tsg_init_device(void);

/* ------------------------------------------------------------------------------------------
 * K0  device-side batch assembly from an HBM-resident corpus (SURVEY 8f n1)
 *   replaces PyG Batch.from_data_list (Code/sag/train.py:181) + the per-graph `.to(device)` /
 *   `torch.Tensor([ndarray]).cuda()` marshaling of the triplet loops (Code/sag/train_triplet.py:207;
 *   Code/sage+gat+diffpool/tripletnet.py:18-33).  Graph b of the batch is corpus graph ids[b]; its nodes
 *   land at rows out_node_ptr[b].. of x_out (one-hot of c_label when given, else rows of c_x) and its
 *   edges at out_edge_ptr[b].. of row_out/col_out with global (batch) node ids.  Offsets are computed by
 *   the host from the graph sizes it already knows (no device round trip).
 * ------------------------------------------------------------------------------------------ */
int tsg_pack_batch(const int64_t* ids, const int64_t* out_node_ptr, const int64_t* out_edge_ptr,
                   int64_t batch_graphs, const int64_t* corpus_node_ptr, const int64_t* corpus_edge_ptr,
                   const int32_t* corpus_row, const int32_t* corpus_col,
                   const int32_t* corpus_label /*nullable*/, const float* corpus_x /*nullable*/,
                   int64_t feat, float* x_out, int64_t* row_out, int64_t* col_out, void* stream);
/* Same gather in the compact form the executor's *_compact entries consume: labels and graph-LOCAL int32 endpoints
 * (out_edge_ptr doubles as their per-graph edge offsets); 4N + 8E bytes written instead of 4NL + 16E. */
int tsg_pack_batch_compact(const int64_t* ids, const int64_t* out_node_ptr, const int64_t* out_edge_ptr,
                           int64_t batch_graphs, const int64_t* corpus_node_ptr, const int64_t* corpus_edge_ptr,
                           const int32_t* corpus_row, const int32_t* corpus_col, const int32_t* corpus_label,
                           int32_t* label_out, int32_t* row_out, int32_t* col_out, void* stream);
/* K0d: a dense-encoder batch (GraphSAGE / GAT / DiffPool) in ONE launch, for a corpus whose per-graph edge lists are
 * coalesced and symmetric (sorted by (row, col), loop free, (r, c) <=> (c, r); graph-local int32 endpoints).
 *   replaces: the reference's per-graph padded numpy adjacency / feature tensors and their `torch.Tensor([ndarray])`
 *   marshaling (Code/sage+gat+diffpool/tripletnet.py:18-33, load_data.py:74-87 padding to max_nodes), with the node
 *   features = rows of the shared feature table by node position (train_triplet.py:379-385).
 *   Writes for graph b = corpus graph ids[b]: x_out rows out_node_ptr[b] + i = table[i] (table [max_nodes, feat] fp32),
 *   has_pad[b] = (n_b < max_nodes), and -- when rowptr is given -- the RAW 0/1 CSR of the packed adjacency exactly as
 *   tsg_csr_build(TSG_CSR_RAW) builds it from the expanded edge_index: rowptr [num_nodes + 1], colidx / val
 *   [num_edges] serve BOTH orientations (symmetric), t_eid (nullable) = the src-major eid = identity, eid (nullable) =
 *   the dst-major eid = position of the reverse edge.  Row starts come from run boundaries: no scan, no atomics.
 *   The promise is verified per graph; violations OR TSG_FUSED_* bits (1 range / self loop, 2 order, 4 symmetry) into
 *   *status (int32, device) and that graph's CSR is replaced by one whose indices stay in range.  rowptr == NULL:
 *   x_out and has_pad only (callers that build the CSR with tsg_csr_build).  Sizes below 2^31 (num_nodes + num_edges);
 *   max_nodes + 2 ints of shared memory per CTA (graphs of up to 12,286 nodes); TSG_EINVAL otherwise. */
int tsg_pack_dense_batch(const int64_t* ids, const int64_t* out_node_ptr, const int64_t* out_edge_ptr,
                         int64_t batch_graphs, int64_t num_nodes, int64_t num_edges, const int64_t* corpus_node_ptr,
                         const int64_t* corpus_edge_ptr, const int32_t* corpus_row, const int32_t* corpus_col,
                         const float* table, int64_t max_nodes, int64_t feat, float* x_out, uint8_t* has_pad,
                         int32_t* rowptr /*nullable*/, int32_t* colidx, float* val, int32_t* eid /*nullable*/,
                         int32_t* t_eid /*nullable*/, int32_t* status, void* stream);
/* K0e: an EigenGCN batch (WavePoolingGcnEncoder + Pool, Code/eigengcn) in ONE launch, from the corpus (coalesced,
 * symmetric graph-local lists as for K0d; int32 node labels, F classes) and its resident EigenPooling operands:
 * cluster_of [sum n] graph-local cluster ids, pool_w [J, pool_stride] (P_j[node, cluster_of[node]]), c_cluster_ptr /
 * c_coarse_ptr [G+1], coarse_row / coarse_col graph-local cluster ids with coarse_w (the coarsened adjacency, coalesced
 * and symmetric in position and weight, no self loops), final_w [Jf, final_stride] (one weight per cluster).
 *   replaces: the reference's per-graph spectral pooling operands padded to max_nodes and marshaled per graph
 *   (Code/eigengcn/tripletnet.py:19-56, coarsen_pooling_with_last_eigen_padding.py:121-182), and bench.Config5's
 *   K0 + K1 + gathers + repeat_interleave + build_rect_csr + K11 (tsg_eigpool_build is not needed: pool_w is resident).
 *   Writes for graph b = ids[b] at the packed offsets out_*_ptr (nodes, edges, clusters, coarse entries):
 *   x_out [N, F] one-hot; has_pad [3, B] = (n_b < max_nodes, nc_b < max_nodes, 1 < max_nodes); when rowptr is given the
 *   RAW 0/1 adjacency CSR (rowptr [N+1], colidx / val [E], one orientation = its own transpose; NULL: built elsewhere);
 *   P_j^T: member_ptr [NC+1] / member [N] (cluster rows, members in ascending node order) / pool_val [J, N] and its
 *   transpose node_iota [N+1] (= arange) / node_cluster [N] (batch-global cluster) / pool_val_nodes [J, N];
 *   the coarsened adjacency coarse_rowptr [NC+1] / coarse_colidx / coarse_val [EC] (RAW, its own transpose);
 *   when Jf > 0 the final pooling final_rowptr [B+1] / cluster_iota [NC+1] (its [:NC] = colidx, all of it = the
 *   transposed rowptr) / cluster_graph [NC] / final_val [Jf, NC]; graph_iota [B+1] int64 = arange (the final level's
 *   row offsets).  Violations OR into *status: TSG_FUSED_* 1 / 2 / 4 for the adjacency as in K0d, 16 for the operands
 *   (cluster id outside [0, nc_b), nc_b > max_nodes, no cluster for a graph with nodes, a coarse list out of range,
 *   unsorted, with a self loop or asymmetric); indices stay in range either way.  TSG_EINVAL: sizes of 2^31 or more,
 *   null pointers (an array with nothing to read or write may be NULL: node arrays when N = 0, coarse-entry arrays
 *   when EC = 0, adjacency arrays when E = 0), J = 0, N > 0 with NC = 0, or max_nodes above the shared-memory budget
 *   (3 max_nodes + 2 ints per CTA: 19,370 nodes). */
int tsg_pack_eigen_batch(const int64_t* ids, const int64_t* out_node_ptr, const int64_t* out_edge_ptr,
                         const int64_t* out_cluster_ptr, const int64_t* out_coarse_ptr, int64_t batch_graphs,
                         int64_t num_nodes, int64_t num_edges, int64_t num_clusters, int64_t num_coarse,
                         const int64_t* corpus_node_ptr, const int64_t* corpus_edge_ptr, const int32_t* corpus_label,
                         const int32_t* corpus_row, const int32_t* corpus_col, int64_t feat,
                         const int64_t* corpus_cluster_ptr, const int64_t* corpus_coarse_ptr, const int32_t* cluster_of,
                         const float* pool_w, int64_t pool_stride, int64_t num_pool, const int32_t* coarse_row,
                         const int32_t* coarse_col, const float* coarse_w, const float* final_w /*nullable if Jf = 0*/,
                         int64_t final_stride, int64_t num_final, int64_t max_nodes, float* x_out, uint8_t* has_pad,
                         int32_t* rowptr /*nullable*/, int32_t* colidx, float* val, int32_t* member_ptr,
                         int32_t* member, float* pool_val, int32_t* node_iota, int32_t* node_cluster,
                         float* pool_val_nodes, int32_t* coarse_rowptr, int32_t* coarse_colidx, float* coarse_val,
                         int32_t* final_rowptr, int32_t* cluster_iota, int32_t* cluster_graph, float* final_val,
                         int64_t* graph_iota, int32_t* status, void* stream);

/* ------------------------------------------------------------------------------------------
 * K1  CSR construction + GCN normalisation
 *   replaces: PyG GCNConv.norm / gcn_norm (add_remaining_self_loops, scatter_add degree,
 *   deg^-1/2 A deg^-1/2) as called from Code/sag/network.py:34,38,42 and Code/sag/layers.py:18.
 *   mode TSG_CSR_GCN : drop input self loops, append one loop per node LAST in its row, weight 1
 *                      (or the last listed loop's weight when edge_weight is given), val = norm.
 *   mode TSG_CSR_RAW : keep the edge list as is, val = edge_weight or 1 (the dense directories'
 *                      0/1 adjacency, Code/sage+gat+diffpool/encoders.py:33).
 *   Output is the stable counting sort of the (augmented) COO list: within a row entries keep COO
 *   order.  The dst-major CSR (rows = targets, colidx = sources) drives the forward aggregation,
 *   the src-major one (rows = sources, colidx = targets) the backward; pass NULL t_* to skip it.
 *   eid = original edge position (< num_edges) or num_edges + node for an appended self loop.
 *   Capacity of colidx/val/eid: num_edges + num_nodes (GCN) or num_edges (RAW).
 * ------------------------------------------------------------------------------------------ */
#define TSG_CSR_GCN 0
#define TSG_CSR_RAW 1
size_t tsg_csr_build_workspace_bytes(int64_t num_edges, int64_t num_nodes);
int tsg_csr_build(const int64_t* row, const int64_t* col, const float* edge_weight /*nullable*/,
                  int64_t num_edges, const int64_t* num_edges_dev /*nullable*/, int64_t num_nodes,
                  int mode,
                  int32_t* rowptr, int32_t* colidx, float* val, int32_t* eid /*nullable*/,
                  int32_t* t_rowptr /*nullable*/, int32_t* t_colidx, float* t_val,
                  int32_t* t_eid /*nullable*/,
                  void* workspace, size_t workspace_bytes, void* stream);

/* K1b: the same CSR (TSG_CSR_GCN, unit weights, both orientations) for a block-diagonal packed batch
 * whose edge list keeps every graph's edges contiguous (PyG Batch.from_data_list, SURVEY A.1.5; the
 * order-preserving filter_adj keeps it true at every pooling level).  One CTA per graph, counting /
 * slot claim / rank-in-row placement in shared memory: bit-identical to tsg_csr_build.
 *   tsg_edge_ptr: edge_ptr[g] = first edge whose source row >= node_ptr[g] (int64 [G+1], device).
 *   max_graph_nodes: host-side upper bound over the graphs of the batch (sizes the shared-memory
 *   arrays; TSG_EINVAL if a graph cannot fit, caller then uses tsg_csr_build).  The bound is the
 *   caller's contract (the packer knows every graph's size; pooling only shrinks graphs); a graph that
 *   violates it at run time traps the kernel (loud failure, no corruption). */
int tsg_edge_ptr(const int64_t* row, int64_t num_edges, const int64_t* num_edges_dev /*nullable*/,
                 const int64_t* node_ptr, int64_t num_graphs, int64_t* edge_ptr, void* stream);
size_t tsg_csr_build_graphs_workspace_bytes(int64_t num_graphs, int64_t num_edges_cap);
int tsg_csr_build_graphs(const int64_t* row, const int64_t* col, const int64_t* edge_ptr,
                         const int64_t* node_ptr, int64_t num_graphs, int64_t num_nodes,
                         int64_t num_edges_cap, int64_t max_graph_nodes,
                         int32_t* rowptr, int32_t* colidx, float* val, int32_t* eid /*nullable*/,
                         int32_t* t_rowptr /*nullable*/, int32_t* t_colidx, float* t_val,
                         int32_t* t_eid /*nullable*/,
                         void* workspace, size_t workspace_bytes, void* stream);
/* Same result from graph-LOCAL int32 endpoints (ids in [0, n_g), the form the TU files and the compact feeder
 * hold) with the per-graph edge offsets given: no int64 edge_index has to be materialised. */
int tsg_csr_build_graphs_local(const int32_t* local_row, const int32_t* local_col, const int64_t* edge_ptr,
                         const int64_t* node_ptr, int64_t num_graphs, int64_t num_nodes,
                         int64_t num_edges_cap, int64_t max_graph_nodes,
                         int32_t* rowptr, int32_t* colidx, float* val, int32_t* eid /*nullable*/,
                         int32_t* t_rowptr /*nullable*/, int32_t* t_colidx, float* t_val,
                         int32_t* t_eid /*nullable*/,
                         void* workspace, size_t workspace_bytes, void* stream);

/* K1c: the GCN CSR of a pooled level directly from the previous level's CSR: new row i = old row perm[i]
 * restricted to surviving columns (inv_perm >= 0), relabelled, same order, renormalised -- bit-identical to
 * tsg_csr_build_graphs(tsg_filter_adj(edges, perm)) (Code/sag/layers.py:20-23 followed by the next GCNConv's
 * gcn_norm) without touching the edge list.  Output capacity: the old nnz.  tsg_inv_perm is filter_adj's
 * relabelling table alone (inv_perm[v] = position of v in perm, or -1). */
int tsg_inv_perm(const int64_t* perm, int64_t num_perm, int64_t num_nodes, int32_t* inv_perm, void* stream);
size_t tsg_csr_filter_workspace_bytes(int64_t num_perm);
int tsg_csr_filter(const int32_t* rowptr, const int32_t* colidx, const int32_t* t_rowptr, const int32_t* t_colidx,
                   const int64_t* perm, const int32_t* inv_perm, int64_t num_perm,
                   int32_t* out_rowptr, int32_t* out_colidx, float* out_val,
                   int32_t* out_t_rowptr, int32_t* out_t_colidx, float* out_t_val,
                   void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * K2  CSR segment-sum SpMM:  Y[r,:] = sum_p val[p] * H[colidx[p],:]  (+ bias) (ReLU optional)
 *   replaces: the gather / mul / scatter_add of PyG GCNConv.propagate (Code/sag/network.py:34)
 *   and `torch.matmul(adj, x)` of the dense GraphConv (Code/sage+gat+diffpool/encoders.py:33,
 *   Code/eigengcn/encoders.py:31).  Per-row accumulation is sequential in CSR order (deterministic,
 *   launch-geometry independent); with TSG_SPMM_EXACT the product is rounded before the add, which
 *   is bit-identical to index_add_ in COO order; without it the product is fused (FFMA).
 *   The backward (dH = A^T dY) is the same call on the src-major CSR.
 *   flags: TSG_SPMM_RELU applies max(.,0) after the bias; relu_mask (nullable, uint8 [N,F]) is
 *   not needed because ReLU's backward is recomputed from Y > 0.
 * ------------------------------------------------------------------------------------------ */
#define TSG_SPMM_RELU 1
#define TSG_SPMM_EXACT 2 /* round every product before the add: bit-identical to index_add_ in COO order (default fuses: <= 1 ulp/term) */
int tsg_spmm(const int32_t* rowptr, const int32_t* colidx, const float* val /*nullable => 1*/,
             const float* H, const float* bias /*nullable*/, float* Y,
             int64_t num_rows, int64_t feat, int flags, void* stream);

/* Tiled K2: `tile_ptr[T+1]` (int64, device) cuts the rows into runs whose neighbours all lie inside the
 * same run (a packed batch is block diagonal: a tile = one or several whole graphs).  Each CTA stages
 * its tile's H rows, CSR slice and rowptr slice in shared memory with bulk async copies and gathers
 * from there; tiles that do not fit the staging buffers or are not self-contained (verified in the
 * kernel) use the global-gather path.  Same arithmetic and order as tsg_spmm (bit-identical). */
int tsg_spmm_tiled(const int32_t* rowptr, const int32_t* colidx, const float* val /*nullable => 1*/,
                   const float* H, const float* bias /*nullable*/, float* Y, const int64_t* tile_ptr,
                   int64_t num_tiles, int64_t num_rows, int64_t feat, int flags, void* stream);

/* TMA-staged K2 for packed batches: tile_ptr[T+1] (int64, device) = graph boundaries; every tile (one graph)
 * is copied into shared memory by `cp.async.bulk` (H rows, colidx / val slice, rowptr slice; two stages per
 * CTA, producer warp + 31 consumer warps, mbarriers) and gathered from there; graphs that do not fit a stage are
 * gathered from global memory by the same kernel.  Same arithmetic and order as tsg_spmm.  Needs feat % 4 == 0,
 * feat <= 32, 16-byte aligned arrays with 16 readable bytes behind rowptr / colidx / val, and self-contained
 * tiles (CSRs from tsg_csr_build_graphs / tsg_csr_filter).  Other shapes are forwarded to tsg_spmm.
 * status_dev (int32, device, caller-zeroed) is set to 1 if a pipeline wait ever times out (hang guard). */
int tsg_spmm_tma(const int32_t* rowptr, const int32_t* colidx, const float* val /*nullable => 1*/,
                 const float* H, const float* bias /*nullable*/, float* Y, const int64_t* tile_ptr,
                 int64_t num_tiles, int64_t num_rows, int64_t feat, int flags, int32_t* status_dev, void* stream);

/* dY_masked = dY * (Y > 0): ReLU backward fused with the column sum that gives the bias gradient:
 * dbias[f] = sum_r dY_masked[r,f]  (deterministic two-stage reduction).  Y may be NULL (no ReLU).
 * workspace: tsg_colsum_workspace_bytes(num_rows, feat). */
size_t tsg_colsum_workspace_bytes(int64_t num_rows, int64_t feat);
int tsg_relu_bwd_colsum(const float* dY, const float* Y /*nullable*/, float* dY_masked /*nullable*/,
                        float* dbias, int64_t num_rows, int64_t feat,
                        void* workspace, size_t workspace_bytes, void* stream);
/* Same with the gradient of a rank-1 branch added on the fly: g[r,f] = dY[r,f] + row_scale[r] * col_vec[f]
 * before the mask (the score layer's  d h += d(h ws) ws^T  of Code/sag/layers.py:18 without materialising
 * the [N,F] outer product or a separate add pass).  Product rounded before the add (== the unfused path). */
int tsg_relu_bwd_colsum_rank1(const float* dY, const float* Y /*nullable*/, const float* row_scale,
                              const float* col_vec, float* dY_masked /*nullable*/, float* dbias,
                              int64_t num_rows, int64_t feat,
                              void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * K3  tall-skinny row-local dense products (N ~ 10^6 rows, K and M <= 128 columns), fp32 FFMA,
 *     exact zeros of X skipped (one-hot node-label features).
 *   tsg_linear_fwd: Y = epilogue(X[N,K] . Wop + bias), Wop = W[K,M] (w_transposed=0) or W[M,K]^T.
 *     replaces `x @ weight` of PyG GCNConv (Code/sag/network.py:34) and, with the epilogue flags,
 *     `torch.matmul(y, self.weight) + self.bias` -> F.normalize(dim=2) (Code/sage+gat+diffpool/
 *     encoders.py:36-40) -> self.act (ReLU, :177) -> apply_bn (:134-138: fresh BatchNorm1d(N) =
 *     per-node statistics over the feature axis, biased variance, eps 1e-5, no affine).
 *     The input gradient dX = dY . W^T is the same call with w_transposed=1.
 *   tsg_dense_epilogue_bwd: dU (gradient at X.W+b) from dO, recomputing the forward from X.
 *   tsg_linear_bwd_weight: dW[K,M] = X^T . dY and db[M] = colsum(dY), deterministic two-stage.
 * ------------------------------------------------------------------------------------------ */
#define TSG_LIN_NORMALIZE 1
#define TSG_LIN_RELU 2
#define TSG_LIN_NODEBN 4
#define TSG_LIN_SOFTMAX 8    /* row softmax of the product (DiffPool assignment, encoders.py:369); not combined with the others */
int tsg_linear_fwd(const float* X, const float* W, const float* bias /*nullable*/, float* Y,
                   int64_t num_rows, int64_t in_feat, int64_t out_feat, int w_transposed, int flags,
                   void* stream);
int tsg_dense_epilogue_bwd(const float* X, const float* W, const float* bias /*nullable*/,
                           const float* dO, float* dU, int64_t num_rows, int64_t in_feat,
                           int64_t out_feat, int flags, void* stream);
size_t tsg_linear_bwd_weight_workspace_bytes(int64_t in_feat, int64_t out_feat);
int tsg_linear_bwd_weight(const float* X, const float* dY, float* dW /*nullable*/,
                          float* db /*nullable*/, int64_t num_rows, int64_t in_feat, int64_t out_feat,
                          void* workspace, size_t workspace_bytes, void* stream);
/* SAGPool level boundary of the encoder backward (levels 2 and 1) in one pass over the rows:
 *   dxg = readout_bwd(dz) + dxw . W^T and dW = x^T . dxw,
 * with dxw [N,H] (= A_hat^T dhm of conv_l), x [N,H] (conv_l's input), W [H,H] (conv_l's weight, read as
 * tsg_linear_fwd(..., w_transposed=1) reads it), dz [G, >= 2H] (row stride dz_stride; [max || mean] gradient of the
 * readout below) with argmax [G,H] and graph_ptr [G+1] of those N rows.  Bit-identical to tsg_linear_fwd(dxw, W,
 * NULL, dxg, N, H, H, 1, 0) -> tsg_readout_bwd(dz, dz_stride, argmax, graph_ptr, G, N, H, MAX|MEAN|ACCUM, dxg) and
 * tsg_linear_bwd_weight(x, dxw, dW, NULL, N, H, H):
 *   dX[r,m]  = (sum_k dxw[r,k] W[m,k], one fmaf per term, k ascending from 0.f) + 0.f
 *   dxg[r,m] = (dz[g,H+m] / (float)max(n_g,1) + (argmax[g,m] == r ? dz[g,m] : 0.f)) + dX[r,m]   (g: graph of row r;
 *              a row outside graph_ptr's graphs gets dX[r,m])
 *   dW       = tsg_linear_bwd_weight's dense partition: 2 x 148 CTAs of ceil(N / 296) rows, 128-row tiles from each
 *              CTA's first row, row i of a tile to group i mod (256 / (H/4)^2), groups then CTAs summed in index order.
 * hidden % 4 == 0 and 8 <= hidden <= 64; dxw, x, dxg, dz, argmax 16-byte aligned; dz_stride % 4 == 0;
 * workspace >= tsg_linear_bwd_weight_workspace_bytes(hidden, hidden).  Two kernels (the pass + the partials' fold). */
int tsg_sag_boundary_bwd(const float* dxw, const float* x, const float* W, const float* dz, int64_t dz_stride,
                         const int32_t* argmax, const int64_t* graph_ptr, int64_t num_graphs, int64_t num_rows,
                         int64_t hidden, float* dxg, float* dW, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Dense wire-format adapters (dense directories)
 *   tsg_dense_to_coo: non-zeros of zero-padded dense matrices M[B,R,C] (adjacency
 *     Code/sage+gat+diffpool/cross_val.py:163-184; pooled adjacency / eigen-pooling operators
 *     Code/eigengcn/graph_sampler.py:185-241) in row-major order as COO triplets
 *     (row_off[b] + r, col_off[b] + c, M[b,r,c]) for r < nrows[b], c < ncols[b]; feed to
 *     tsg_csr_build(TSG_CSR_RAW).  capacity >= number of non-zeros; count returned on the device.
 *   tsg_nodebn_{fwd,bwd}: `apply_bn` (encoders.py:134-138) on x[B,N,F]: statistics per node over
 *     (B,F), biased variance, eps 1e-5, no affine.  fwd also returns mean[N], rstd[N].
 * ------------------------------------------------------------------------------------------ */
size_t tsg_dense_to_coo_workspace_bytes(int64_t B, int64_t R);
int tsg_dense_to_coo(const float* M, int64_t B, int64_t R, int64_t C,
                     const int64_t* nrows, const int64_t* ncols,
                     const int64_t* row_off, const int64_t* col_off,
                     int64_t* out_r, int64_t* out_c, float* out_w, int64_t capacity,
                     int64_t* out_count_dev, void* workspace, size_t workspace_bytes, void* stream);
int tsg_nodebn_fwd(const float* x, float* y, float* mean, float* rstd,
                   int64_t B, int64_t N, int64_t F, void* stream);
int tsg_nodebn_bwd(const float* dy, const float* y, const float* rstd, float* dx,
                   int64_t B, int64_t N, int64_t F, void* stream);

/* ------------------------------------------------------------------------------------------
 * K4  dense-GAT head on the packed CSR (all heads of a layer at once)
 *   replaces DGATHead.forward (Code/sage+gat+diffpool/encoders_GAT.py:29-49):
 *     e_ij = LeakyReLU(s1_i + s2_j) on edges adj[i,j] > 0, softmax over i for every column j
 *     (dim=1 of the broadcast [1,N,N] tensor), h'_i = sum_j att_ij h_j.
 *   h [n, heads*F], s1 = h.a[:F], s2 = h.a[F:] as [n, heads].  (rowptr, colidx, eid) is the
 *   dst-major CSR (row i lists its columns j), t_* the src-major one (column j lists its rows i);
 *   both from tsg_csr_build(TSG_CSR_RAW) with eids.  fwd also returns the per-column softmax
 *   statistics mx, zs [n, heads].  Columns without any edge are not touched (host-side correction).
 * ------------------------------------------------------------------------------------------ */
int tsg_gat_fwd(const int32_t* rowptr, const int32_t* colidx, const int32_t* t_rowptr,
                const int32_t* t_colidx, const float* h, const float* s1, const float* s2,
                int64_t num_nodes, int64_t heads, int64_t feat, float slope,
                float* mx, float* zs, float* hp, void* stream);
size_t tsg_gat_bwd_workspace_bytes(int64_t nnz, int64_t heads);
int tsg_gat_bwd(const int32_t* rowptr, const int32_t* eid, const int32_t* t_rowptr,
                const int32_t* t_colidx, const int32_t* t_eid, const float* h, const float* s1,
                const float* s2, const float* mx, const float* zs, const float* dhp,
                int64_t num_nodes, int64_t nnz, int64_t heads, int64_t feat, float slope,
                float* dh, float* ds1, float* ds2,
                void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * K7  DiffPool per-graph dense contractions (packed layout)
 *   replaces the batched dense matmuls of SoftPoolingGcnEncoder.forward
 *   (Code/sage+gat+diffpool/encoders.py:374-375: x = S^T Z, adj = S^T adj S) and of the post-pool
 *   tower on the dense K x K pooled adjacency (encoders.py:378).
 *   tsg_seg_contract: C[g] (Kx x Ky) = sum_{r in graph g} X[r,:]^T Y[r,:], g = 0..G-1.
 *     With Y = [Z | A.S] and X = S this is both products at once.  use_tensor_cores = 1 runs the
 *     tcgen05 kernel (kind::tf32, 3xTF32 error-compensated split, TMEM accumulators; needs
 *     Kx <= 128, Ky <= 256); 0 runs the fp32 SIMT kernel.  status_dev (int32, device, caller-zeroed)
 *     is set to 1 if an MMA completion wait ever times out (hang guard; required for tcgen05).
 *   tsg_seg_linear: Y[r,:] = X[r,:] . W[g] (Kin x M) (or W[g]^T stored M x Kin) for r in graph g.
 * ------------------------------------------------------------------------------------------ */
int tsg_seg_contract(const float* X, const float* Y, const int64_t* graph_ptr, int64_t num_graphs,
                     int64_t Kx, int64_t Ky, float* C, int use_tensor_cores,
                     int32_t* status_dev /*nullable unless tensor cores*/, void* stream);
int tsg_seg_linear(const float* X, const float* W, const int64_t* graph_ptr, int64_t num_graphs,
                   int64_t in_feat, int64_t out_feat, int w_transposed, float* Y, void* stream);
/* tsg_seg_linear on tcgen05 (kind::tf32, 3xTF32 split, TMEM accumulators; the rows of a graph are the MMA's M dimension,
 * 128 at a time, the contraction runs over Kin in chunks of 32).  Needs M <= 256, M % 4 == 0, Kin % 4 == 0 and 16-byte
 * aligned operands (TSG_EINVAL otherwise: call tsg_seg_linear); status_dev as for tsg_seg_contract. */
int tsg_seg_linear_tc(const float* X, const float* W, const int64_t* graph_ptr, int64_t num_graphs, int64_t Kin, int64_t M,
                      int w_transposed, float* Y, int32_t* status_dev, void* stream);
/* Y = X . W (W [Kin, M], or W stored [M, Kin] with w_transposed) for ONE shared weight on the same tcgen05 kernel (a CTA per
 * 128 rows), then, if softmax != 0, Y = softmax(Y + bias) per row in place: DiffPool's assignment Linear + softmax
 * (Code/sage+gat+diffpool/encoders.py:366-369).  Same shape limits as tsg_seg_linear_tc; bias only with softmax. */
int tsg_linear_tc(const float* X, const float* W, const float* bias /*nullable*/, int64_t num_rows, int64_t Kin, int64_t M,
                  int w_transposed, int softmax, float* Y, int32_t* status_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * K5a  per-graph top-k (deterministic: descending score, ties -> lower node id, NaN first)
 *   replaces: PyG topk_pool.topk as called from Code/sag/layers.py:20.
 *   graph_ptr[G+1] are node offsets of the (sorted) batch vector; k_g = ceil(ratio * n_g) in
 *   fp32.  tsg_topk_sizes writes k_ptr[G+1] (exclusive scan of k_g); tsg_topk writes
 *   perm[k_ptr[G]] (global node ids, graph-major, score-descending) as int64.
 * ------------------------------------------------------------------------------------------ */
size_t tsg_topk_workspace_bytes(int64_t num_nodes, int64_t num_graphs);
int tsg_topk_sizes(const int64_t* graph_ptr, int64_t num_graphs, float ratio, int64_t* k_ptr,
                   void* workspace, size_t workspace_bytes, void* stream);
int tsg_topk(const float* score, const int64_t* graph_ptr, const int64_t* k_ptr,
             int64_t num_graphs, int64_t num_nodes, int64_t* perm,
             void* workspace, size_t workspace_bytes, void* stream);
/* tsg_topk with the caller's bound on the largest graph (host side, e.g. from the packer): size ranges that cannot be
 * populated are not launched (n <= 1,024: register-run kernel; <= 4,096: shared-memory bitonic network; larger: rank
 * selection).  tsg_topk == tsg_topk_bounded(..., max_graph_nodes = num_nodes). */
int tsg_topk_bounded(const float* score, const int64_t* graph_ptr, const int64_t* k_ptr, int64_t num_graphs,
                     int64_t num_nodes, int64_t max_graph_nodes, int64_t* perm, void* workspace, size_t workspace_bytes,
                     void* stream);

/* node offsets from a sorted batch vector: graph_ptr[g] = first i with batch[i] >= g. */
int tsg_batch_to_ptr(const int64_t* batch, int64_t num_nodes, int64_t num_graphs,
                     int64_t* graph_ptr, void* stream);

/* ------------------------------------------------------------------------------------------
 * K5b  filter_adj: relabel by perm, keep edges whose both ends survive, order preserving.
 *   replaces: PyG topk_pool.filter_adj as called from Code/sag/layers.py:23.
 *   inv_perm[num_nodes] (int32 out): position of node in perm or -1.  Survivors are written to
 *   out_row/out_col (capacity num_edges); *out_num_edges_dev receives the count.
 * ------------------------------------------------------------------------------------------ */
size_t tsg_filter_adj_workspace_bytes(int64_t num_edges);
int tsg_filter_adj(const int64_t* row, const int64_t* col, int64_t num_edges,
                   const int64_t* num_edges_dev /*nullable*/,
                   const int64_t* perm, int64_t num_perm, int64_t num_nodes,
                   int32_t* inv_perm, int64_t* out_row, int64_t* out_col,
                   int64_t* out_num_edges_dev,
                   void* workspace, size_t workspace_bytes, void* stream);

/* gated gather  xo[i,:] = x[perm[i],:] * tanh(score[perm[i]])   (Code/sag/layers.py:21)
 * also emits batch_out[i] = batch[perm[i]] (layers.py:22) when batch != NULL. */
int tsg_gate_gather_fwd(const float* x, const float* score, const int64_t* perm,
                        const int64_t* batch /*nullable*/, float* xo, int64_t* batch_out,
                        int64_t num_perm, int64_t feat, void* stream);
/* dx[j,:] = inv_perm[j] >= 0 ? dxo[inv_perm[j],:] * tanh(score[j]) : 0
 * dscore[j] = inv_perm[j] >= 0 ? sum_f(dxo[m,f] * x[j,f]) * (1 - tanh^2(score[j])) : 0 */
int tsg_gate_gather_bwd(const float* dxo, const float* x, const float* score,
                        const int32_t* inv_perm, float* dx, float* dscore,
                        int64_t num_nodes, int64_t feat, void* stream);

/* ------------------------------------------------------------------------------------------
 * K6  per-graph readout: out[g, 0:F] = max_i x[i,:], out[g, F:2F] = mean_i x[i,:]
 *   replaces: torch.cat([gmp(x,batch), gap(x,batch)],1) of Code/sag/network.py:36,40,44 and the
 *   `torch.max(x, dim=1)` readouts of the dense directories (encoders.py:183,190,197).
 *   argmax[g,f] (int32) = global row of the FIRST maximum (-1 for an empty graph => output 0).
 *   mode bit0: emit max, bit1: emit mean, bit2: emit sum instead of mean.
 * ------------------------------------------------------------------------------------------ */
#define TSG_READOUT_MAX 1
#define TSG_READOUT_MEAN 2
#define TSG_READOUT_SUM 4
#define TSG_READOUT_ACCUM 8 /* tsg_readout_bwd only: dx += (instead of dx =), fusing the add of a second gradient */
int tsg_readout_fwd(const float* x, const int64_t* graph_ptr, int64_t num_graphs, int64_t feat,
                    int mode, float* out, int64_t out_stride, int32_t* argmax, void* stream);
/* dx[i,f] = (argmax[g,f]==i) * dout[g,f] + dout[g,F+f]/n_g ; g found from graph_ptr. */
int tsg_readout_bwd(const float* dout, int64_t dout_stride, const int32_t* argmax,
                    const int64_t* graph_ptr, int64_t num_graphs, int64_t num_nodes, int64_t feat,
                    int mode, float* dx, void* stream);

/* ------------------------------------------------------------------------------------------
 * K9  triplet distances + margin ranking loss
 *   replaces: F.pairwise_distance x2 (Code/sag/tripletnet.py:21-22) + MarginRankingLoss with
 *   target -1 (Code/sag/train_triplet.py:196,208-211):
 *   d(a,b) = || e_a - e_b + 1e-6 ||_2 ; loss = mean_t max(0, d_ap - d_an + margin).
 *   triplets[T,3] int64 index rows of emb[M,D].  bwd is deterministic: per embedding row the
 *   contributions are summed in triplet order via an inverted index built on the device.
 *   tsg_pairdist_matrix writes the full [M,M] matrix (hard-negative mining / kNN evaluation).
 * ------------------------------------------------------------------------------------------ */
size_t tsg_triplet_workspace_bytes(int64_t num_triplets, int64_t num_rows, int64_t dim);
int tsg_triplet_fwd(const float* emb, const int64_t* triplets, int64_t num_triplets,
                    int64_t num_rows, int64_t dim, float margin, float eps,
                    float* dist_pos, float* dist_neg, float* loss,
                    void* workspace, size_t workspace_bytes, void* stream);
int tsg_triplet_bwd(const float* emb, const int64_t* triplets, int64_t num_triplets,
                    int64_t num_rows, int64_t dim, float margin, float eps,
                    const float* dist_pos, const float* dist_neg, const float* dloss,
                    float* demb, void* workspace, size_t workspace_bytes, void* stream);
int tsg_pairdist_matrix(const float* emb, int64_t num_rows, int64_t dim, float eps,
                        float* dist, void* stream);

/* ------------------------------------------------------------------------------------------
 * K11  EigenPooling preprocessing (SURVEY 8f n2)
 *   replaces the post-clustering half of `_coarserning_pooling_`
 *   (Code/eigengcn/coarsen_pooling_with_last_eigen_padding.py:121-182): per cluster the unnormalised
 *   Laplacian L = D - W of the induced subgraph (graph.py:116-126), its eigendecomposition in ascending
 *   order (graph.py:147-163), sign rule "first entry >= 0" (:165-168), last vector repeated for j >= size
 *   (:169-173); and A_coarse = Omega^T A_ext Omega (:135-149).  Cluster labels are an input (the reference
 *   gets them from sklearn SpectralClustering, :125-126).
 *   tsg_eigpool_build: adjacency as RAW CSR (any orientation: symmetric); cluster_of[N] = global cluster id
 *     of every node; (member_ptr[C+1], member[N]) = nodes of every cluster in ascending node order (K1 RAW
 *     on the (node -> cluster) list).  pool_val[j, p] = P_j[member[p], cluster] (CSR value order of P_j^T),
 *     pool_val_nodes[j, v] = the same value in node order (the transposed operator).  eigvals (nullable):
 *     [C, TSG_EIG_MAX] ascending, zero padded.  Clusters larger than TSG_EIG_MAX set *status_dev = 1 and are
 *     left untouched (host fallback).  Warp per cluster, double-precision cyclic Jacobi in shared memory.
 *   tsg_coarsen_edges: the inter-cluster edges relabelled to cluster ids, original order kept; duplicates
 *     are NOT merged (K2 sums them), count on the device.
 * ------------------------------------------------------------------------------------------ */
#define TSG_EIG_MAX 32
int tsg_eigpool_build(const int32_t* adj_rowptr, const int32_t* adj_colidx, const float* adj_val /*nullable => 1*/,
                      const int32_t* cluster_of, const int32_t* member_ptr, const int32_t* member,
                      int64_t num_nodes, int64_t num_clusters, int num_vectors,
                      float* pool_val, float* pool_val_nodes, float* eigvals /*nullable*/,
                      int32_t* status_dev, void* stream);
size_t tsg_coarsen_edges_workspace_bytes(int64_t num_edges);
int tsg_coarsen_edges(const int64_t* row, const int64_t* col, const float* weight /*nullable => 1*/,
                      int64_t num_edges, const int32_t* cluster_of, int64_t* out_row, int64_t* out_col,
                      float* out_weight, int64_t* out_count_dev,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * K17  a resident corpus's EigenPooling operands (tsg.feeder.DeviceCorpus.build_eigen), in attach_eigen's layout
 *   replaces the per-graph host loop of tsg.eigen_synth (make_operands = bfs_clusters + operands_from_clusters), i.e.
 *   Code/eigengcn/coarsen_pooling_with_last_eigen_padding.py:121-182 with the clustering input of :125-126 (sklearn
 *   SpectralClustering there) replaced by eigen_synth's BFS chunks or by labels the caller gives.
 *   The corpus is coalesced and symmetric (as for K0d; graph-local int32 row / col, int64 node_ptr / edge_ptr [G+1]).
 *   The entries work on a CHUNK of graphs first_graph .. first_graph + num_graphs - 1 holding num_nodes nodes and
 *   num_edges edges (each below 2^31 together), graphs of at most max_nodes <= TSG_EIGEN_BUILD_MAX_NODES nodes
 *   (3 max_nodes + 2 ints of shared memory per CTA).  In the chunk, graph g's nodes start at nb = node_ptr[g] -
 *   node_ptr[first_graph], its edges at ob, and its cluster k has the chunk id nb + k (a graph has no more clusters
 *   than nodes; rows nb + nc .. nb + n - 1 stay empty), so the chunk arrays are:
 *     rowptr [num_nodes + 1] / colidx [num_edges]: the RAW adjacency CSR with chunk node ids (val = 1 implied);
 *     cluster_g [num_nodes]: chunk cluster id of every node; member_ptr [num_nodes + 1] / member [num_nodes]: the
 *     members of every chunk cluster row -- together exactly what tsg_eigpool_build takes (num_clusters = num_nodes).
 *   status int32 [4], initialised by the caller to INT32_MAX: [0] = least graph whose edge list breaks the promise
 *   (range, self loop, order or symmetry; its rows are left empty), [1] = least graph with a cluster of more than
 *   TSG_EIG_MAX members, [2] = least graph with a label outside [0, n); [3] is free for tsg_eigpool_build's status.
 *   tsg_eigen_bfs_clusters: eigen_synth.bfs_clusters -- the queue BFS from node 0 over ascending neighbour lists
 *     (scipy breadth_first_order on the symmetric list), unreached nodes appended in ascending order, clusters =
 *     chunks of pool_size (1 .. TSG_EIG_MAX) in that order.  Writes cluster_of [sum n] (corpus, graph-local ids),
 *     num_clusters [G] (corpus, ceil(n / pool_size)) and the chunk arrays, members in BFS order.  Level-synchronous,
 *     one CTA per graph: every node takes its first discoverer, and a level is ordered by (discoverer, node id).
 *   tsg_eigen_group_clusters: the chunk arrays for the graph-local labels cluster_of (corpus, input), members in
 *     ascending node order; num_clusters (nullable) [G] = max label + 1.
 *   tsg_eigen_coarse: per graph, the entries of Omega^T A_ext Omega (coarsen...py:135-149): the (cl[row], cl[col])
 *     pairs of the inter-cluster edges, merged, sorted row-major (np.nonzero's order), count = weight.  Counting pass
 *     (coarse_row NULL): num_coarse [G] (corpus).  Writing pass: coarse_row / coarse_col (graph-local cluster ids) /
 *     coarse_w at the corpus offsets coarse_ptr [G+1]; row_scratch [num_nodes].  Any member order works.
 *   tsg_eigen_final: the final pooling (:150-182 with one cluster holding every coarse node): the first num_vectors
 *     eigenvectors of D - A of the binary coarse adjacency of every graph with min_clusters < nc <= max_clusters (<=
 *     TSG_EIGEN_FINAL_MAX) clusters, with K11's ordering, sign and repeat rules, to final_w [num_vectors, final_stride]
 *     at the corpus offsets cluster_ptr [G+1]; other graphs are not written (another size class, or the caller
 *     computes them).  One CTA per graph, fp64 cyclic Jacobi in 2 max_clusters (max_clusters + 1) doubles of shared
 *     memory, so a launch per size class keeps small graphs many to an SM.
 * ------------------------------------------------------------------------------------------ */
#define TSG_EIGEN_BUILD_MAX_NODES 19370
#define TSG_EIGEN_FINAL_MAX 112
int tsg_eigen_bfs_clusters(const int64_t* corpus_node_ptr, const int64_t* corpus_edge_ptr, const int32_t* corpus_row,
                           const int32_t* corpus_col, int64_t first_graph, int64_t num_graphs, int64_t num_nodes,
                           int64_t num_edges, int64_t max_nodes, int64_t pool_size, int32_t* cluster_of,
                           int32_t* num_clusters, int32_t* rowptr, int32_t* colidx, int32_t* cluster_g,
                           int32_t* member_ptr, int32_t* member, int32_t* status, void* stream);
int tsg_eigen_group_clusters(const int64_t* corpus_node_ptr, const int64_t* corpus_edge_ptr,
                             const int32_t* corpus_row, const int32_t* corpus_col, int64_t first_graph,
                             int64_t num_graphs, int64_t num_nodes, int64_t num_edges, int64_t max_nodes,
                             const int32_t* cluster_of, int32_t* num_clusters /*nullable*/, int32_t* rowptr,
                             int32_t* colidx, int32_t* cluster_g, int32_t* member_ptr, int32_t* member,
                             int32_t* status, void* stream);
int tsg_eigen_coarse(const int64_t* corpus_node_ptr, int64_t first_graph, int64_t num_graphs,
                     const int32_t* num_clusters, const int32_t* rowptr, const int32_t* colidx,
                     const int32_t* cluster_g, const int32_t* member_ptr, const int32_t* member,
                     int32_t* row_scratch, int32_t* num_coarse, const int64_t* coarse_ptr, int32_t* coarse_row,
                     int32_t* coarse_col, float* coarse_w, void* stream);
int tsg_eigen_final(const int64_t* cluster_ptr, const int64_t* coarse_ptr, const int32_t* coarse_row,
                    const int32_t* coarse_col, int64_t first_graph, int64_t num_graphs, int64_t min_clusters,
                    int64_t max_clusters, int64_t num_vectors, float* final_w, int64_t final_stride, void* stream);

/* ------------------------------------------------------------------------------------------
 * K12  stage-2 evaluation heads on graph embeddings (SURVEY 8f n4)
 *   tsg_knn_classify replaces KNeighborsClassifier(n_neighbors=k).fit(train).predict(query) of `evaluate`
 *     (Code/sage+gat+diffpool/train_triplet.py:80-85): Euclidean, uniform weights; distance ties -> lower
 *     train index, vote ties -> lower class id.  1 <= k <= 32 (fewer than k train rows: all of them vote),
 *     1 <= num_classes <= 1024.  pred int64 [num_query]; with query_labels, *correct (int64, device) = #(pred ==
 *     label), an integer reduction (correct NULL: not written; with num_query > 0 correct needs query_labels).  A train or query label
 *     outside [0, num_classes) is clamped for the read and ORs TSG_SAG_LABEL_RANGE into *status (nullable: not
 *     reported).  tsg_knn_predict is tsg_knn_classify(query_labels = correct = status = NULL).
 *   tsg_mlp1_predict is that MLP's forward over num_rows rows (params as for tsg_mlp1_train): pred int64 [num_rows] =
 *     first-index argmax of the logits; logits (nullable) [num_rows, classes]; labels / correct / status as for
 *     tsg_knn_classify.  Every unit is the trainer's own fmaf chain over its input index ascending, so the logits
 *     equal those the trainer's forward computes for the same parameters, bit for bit.
 *   tsg_mlp1_train replaces the stage-2 classifier loop of `evaluate_mlp` (train_triplet.py:148-165):
 *     MLP dim -> hidden1 -> hidden2 -> classes with LeakyReLU(slope), Adam, ONE sample per step in the given
 *     order; all num_samples steps run inside one CTA with weights and moments in shared memory.
 *     params / adam_m / adam_v: flat fp32 [W1 (hidden1 x dim), b1, W2 (hidden2 x hidden1), b2, W3 (classes x
 *     hidden2), b3] (torch nn.Linear layout), updated in place; step0 = Adam steps already taken;
 *     losses (nullable) [num_samples] = the per-step cross-entropy.
 * ------------------------------------------------------------------------------------------ */
int tsg_knn_predict(const float* train, const int64_t* train_labels, const float* query,
                    int64_t num_train, int64_t num_query, int64_t dim, int k, int num_classes,
                    int64_t* pred, void* stream);
int tsg_knn_classify(const float* train, const int64_t* train_labels, const float* query,
                     const int64_t* query_labels /*nullable*/, int64_t num_train, int64_t num_query, int64_t dim, int k,
                     int num_classes, int64_t* pred, int64_t* correct /*nullable*/, int32_t* status /*nullable*/,
                     void* stream);
int tsg_mlp1_predict(const float* emb, const int64_t* labels /*nullable*/, int64_t num_rows, int64_t dim,
                     int64_t hidden1, int64_t hidden2, int64_t num_classes, const float* params, float slope,
                     int64_t* pred, float* logits /*nullable*/, int64_t* correct /*nullable*/,
                     int32_t* status /*nullable*/, void* stream);
int tsg_mlp1_train(const float* emb, const int64_t* labels, int64_t num_samples, int64_t dim,
                   int64_t hidden1, int64_t hidden2, int64_t num_classes,
                   float* params, float* adam_m, float* adam_v, int64_t step0,
                   float lr, float beta1, float beta2, float eps, float slope,
                   float* losses /*nullable*/, void* stream);

/* ------------------------------------------------------------------------------------------
 * K15  DiffPool link-prediction loss (SURVEY 8f n4)
 *   replaces the `self.linkpred` branch of SoftPoolingGcnEncoder.loss (Code/sage+gat+diffpool/encoders.py:416-440):
 *   L = sum_g sum_{i,j<n_g} [-A_ij log(P_ij + eps) - (1 - A_ij) log(1 - P_ij + eps)] / num_entries, P = min(S S^T, 1),
 *   num_entries = sum_g n_g^2 (host), on packed assignment rows S [sum n, K] (K <= 128) and the RAW CSR of the 0/1
 *   adjacency (column ids global, as built by tsg_csr_build(TSG_CSR_RAW)).  P is never materialised.  bwd writes dS.
 * ------------------------------------------------------------------------------------------ */
size_t tsg_linkpred_workspace_bytes(int64_t num_graphs);
int tsg_linkpred_loss_fwd(const float* S, const int64_t* graph_ptr, const int32_t* rowptr, const int32_t* colidx,
                          int64_t num_graphs, int64_t assign_dim, double num_entries, float eps, float* loss,
                          void* workspace, size_t workspace_bytes, void* stream);
int tsg_linkpred_loss_bwd(const float* S, const int64_t* graph_ptr, const int32_t* rowptr, const int32_t* colidx,
                          int64_t num_graphs, int64_t assign_dim, double num_entries, float eps, const float* dloss,
                          float* dS, void* stream);

/* ------------------------------------------------------------------------------------------
 * K16  prediction head + cross-entropy of the dense encoders' supervised settings (original and 2stg+)
 *   replaces the chain of nn.Linear / ReLU layers over the graph readouts r [G, in_dim] and F.cross_entropy of
 *   Code/sage+gat+diffpool/train.py:85-152 (and the stage-2 loop of train_triplet_pre_train.py:249-256).
 *   Layer l maps in_l (in_dim for l = 0, else out_dim[l-1]) to out_dim[l] with weight [out_l, in_l] (nn.Linear layout)
 *   and an optional bias; bit l of relu_mask puts a ReLU after it.  Every unit is ONE fmaf chain over the input index
 *   ascending from 0.f, then + bias (the chain of tsg_linear_fwd(..., w_transposed = 1, flags = 0)'s row kernels), so a
 *   row's logits do not depend on the other rows of the batch or on num_rows.  num_layers = 0: the logits are r.
 *   C = the last width.  softmax_first: the loss is the cross-entropy of softmax(logits) (the reference's 2stg+ stage 2).
 *   Limits: 0 <= num_layers <= 8, every width in [1, 256]; TSG_EINVAL otherwise (and 0 from the workspace queries,
 *   which are pure host code).  A label outside [0, C) is read clamped and ORs TSG_SAG_LABEL_RANGE into *status
 *   (nullable: not reported).  No floating-point atomics: every sum has a fixed order.
 *   tsg_pred_ce_fwd: *loss = mean over the rows of logsumexp(q) - q_y (q = logits, or their softmax), summed in a fixed
 *     order; logits_out (nullable) [G, C]; saves the activations in the workspace for tsg_pred_ce_bwd (same workspace,
 *     same arguments).
 *   tsg_pred_ce_bwd: from *dloss (nullable => 1): dr [G, in_dim] (nullable), dweight[l] [out_l, in_l] and dbias[l]
 *     [out_l] (nullable per layer) WRITTEN, not accumulated; the parameter gradients are K3's fixed-order reductions
 *     (tsg_linear_bwd_weight, tsg_relu_bwd_colsum) over the per-row deltas.
 *   tsg_pred_classify: the eval-mode forward: pred int64 [G] = first-index argmax of the logits (out.max(dim=1)[1]);
 *     logits_out (nullable); with labels y, *correct (int64) = #(pred == y) and *ce_sum = the fixed-order sum of the
 *     per-row loss (softmax_first included); both nullable.
 * ------------------------------------------------------------------------------------------ */
#define TSG_PRED_MAX_LAYERS 8
#define TSG_PRED_MAX_WIDTH 256
typedef struct tsg_pred_head {
  int64_t num_layers;
  int64_t in_dim;
  int64_t out_dim[TSG_PRED_MAX_LAYERS];
  int64_t relu_mask;
  int64_t softmax_first;
  const float* weight[TSG_PRED_MAX_LAYERS];
  const float* bias[TSG_PRED_MAX_LAYERS];      /* nullable */
} tsg_pred_head;
size_t tsg_pred_ce_workspace_bytes(const tsg_pred_head* head, int64_t num_rows);
int tsg_pred_ce_fwd(const tsg_pred_head* head, const float* r, const int64_t* y, int64_t num_rows, float* loss,
                    float* logits_out /*nullable*/, int32_t* status /*nullable*/, void* workspace, size_t workspace_bytes,
                    void* stream);
int tsg_pred_ce_bwd(const tsg_pred_head* head, const float* r, const int64_t* y, int64_t num_rows,
                    const float* dloss /*nullable*/, float* dr /*nullable*/, float* const* dweight,
                    float* const* dbias, void* workspace, size_t workspace_bytes, void* stream);
size_t tsg_pred_classify_workspace_bytes(const tsg_pred_head* head, int64_t num_rows);
int tsg_pred_classify(const tsg_pred_head* head, const float* r, const int64_t* y /*nullable*/, int64_t num_rows,
                      int64_t* pred, float* logits_out /*nullable*/, int64_t* correct /*nullable*/,
                      float* ce_sum /*nullable*/, int32_t* status /*nullable*/, void* workspace, size_t workspace_bytes,
                      void* stream);

/* ------------------------------------------------------------------------------------------
 * H1  TU-format dataset loader -> packed corpus arrays (SURVEY 8f n3).  HOST pointers throughout.
 *   replaces `read_graphfile` (Code/sage+gat+diffpool/load_data.py:12-126, Code/eigengcn/load_data.py) in
 *   TSG_TU_NETWORKX mode (node set / order / labels exactly as the networkx graphs the reference builds) and
 *   PyG's TUDataset reader (Code/sag/train*.py:161-163) in TSG_TU_PYG mode.  `prefix` = <datadir>/<NAME>/<NAME>
 *   (files <prefix>_A.txt, _graph_indicator.txt, _graph_labels.txt, optional _node_labels.txt /
 *   _node_attributes.txt).  sizes[6] = {graphs, nodes, directed edges, node-label classes, attribute width,
 *   graph classes}; tsg_tu_fill copies node_ptr[G+1], edge_ptr[G+1], local row/col[E] (sorted by (row, col)
 *   inside a graph), node_label[N], y[G], attr[N, width] (nullable) into caller-allocated host arrays.
 * ------------------------------------------------------------------------------------------ */
#define TSG_TU_NETWORKX 0
#define TSG_TU_PYG 1
typedef struct tsg_tu_handle tsg_tu_handle;
int tsg_tu_load(const char* prefix, int mode, int64_t max_nodes /*0 = no limit*/, tsg_tu_handle** out);
int tsg_tu_sizes(const tsg_tu_handle* h, int64_t* sizes);
int tsg_tu_fill(const tsg_tu_handle* h, int64_t* node_ptr, int64_t* edge_ptr, int64_t* row, int64_t* col,
                int32_t* node_label, int64_t* y, float* attr /*nullable*/);
void tsg_tu_free(tsg_tu_handle* h);

/* K1d: K1b for packed batches whose per-graph edge lists are coalesced and symmetric (sorted by (row, col), loop free,
 * (r, c) listed <=> (c, r) listed).  One launch, no atomics, no scan, ONE orientation -- the src-major CSR of a symmetric
 * operator is the same arrays.  rowptr [N+1], colidx / val [E+N]; bit-identical to tsg_csr_build_graphs_local's dst-major
 * output.  The promise is verified per graph; violations OR TSG_FUSED_* bits (1 range / self loop, 2 order, 4 symmetry)
 * into *status (device int32, zeroed by the caller) and leave that graph's rows unwritten. */
int tsg_csr_build_graphs_sym_local(const int32_t* local_row, const int32_t* local_col, const int64_t* edge_ptr,
                                   const int64_t* node_ptr, int64_t num_graphs, int64_t num_nodes, int64_t num_edges,
                                   int64_t max_graph_nodes, int32_t* rowptr, int32_t* colidx, float* val,
                                   int32_t* status, void* stream);

/* ------------------------------------------------------------------------------------------
 * K10  native step executor for the SAGPool encoder
 *   replaces the Python-level sequencing of Code/sag/network.py:33-46 (`Net.forward` up to the sum
 *   of the three readouts) and Code/sag/layers.py:14-26 (`SAGPool.forward`) over a packed batch: ONE
 *   call enqueues K1b, K3, K2, K5a, K5b, gate and K6 of all three levels (same kernels, same order as
 *   the per-kernel entry points above), ONE call the whole backward.  All intermediates live in the
 *   caller's arena (tsg_sag_arena_bytes); the forward leaves its saved tensors there for the backward.
 *   n[l] = packed node count of level l (n[0] = input rows, n[l+1] = sum_g ceil(ratio * n_g) computed
 *   on the host exactly as PyG's topk does); level_ptr = device int64 [4, G+1] node offsets per level;
 *   params / grads = 12 device pointers: for l = 0..2 { conv_l.weight [in,H], conv_l.bias [H],
 *   pool_l.score_layer.weight [H,1], pool_l.score_layer.bias [1] }.  z, dz: [G, 2H].
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int64_t num_graphs, in_feat, hidden, num_edges;
  int64_t n[4];
  int64_t max_graph_nodes[3];
  int64_t max_graph_edges;   /* max directed edges of one graph (host knows it from edge_ptr); 0 = unknown: the
                                graph-resident kernels (K13) are not used */
  double pooling_ratio;      /* SAGPool ratio (sizes the shared-memory classes of K13; level sizes themselves come from
                                level_ptr) */
  int64_t flags;             /* TSG_SAG_COALESCED: the caller promises that every graph's edge list is sorted by (row, col),
                                loop free and symmetric (TUDataset / TU loader / tsg.synth form).  The compact entries then
                                build ONE CSR orientation per level (K1d, single-orientation K1c) and use it for both A_hat
                                and its transpose.  The promise is VERIFIED on the device: a violation sets the arena's
                                TSG_SAG_STATUS word (the caller must look at it where it synchronises) */
  int32_t* status;           /* optional DEVICE int32 the verification bits are OR-ed into instead of the arena's own
                                TSG_SAG_STATUS word (never cleared by the library: one persistent word can collect many
                                steps and be read once); NULL = the arena's word, zeroed by every forward */
} tsg_sag_shape;
#define TSG_SAG_COALESCED 1
size_t tsg_sag_arena_bytes(const tsg_sag_shape* shape);
/* tsg_sag_encoder_embed_compact (below) is the FORWARD-ONLY form of tsg_sag_encoder_fwd_compact: embeddings for the
 * reference's evaluation loops (Code/sag/train_triplet.py:36-58,86-99 embed every graph without a backward).  It runs the
 * graph-resident kernels (K13, k13_sag_fused.cu: one CTA carries one graph through all three levels in shared memory, one
 * launch per size class instead of 36) when the shape allows it -- hidden in {32, 64, 128}, max_graph_edges given, per-graph
 * working set within 227 KB of shared memory -- else the kernel-per-operator sequence.  z, and the perm / score / h the
 * forward leaves in the arena, are bit-identical either way.  tsg_sag_set_fused(0) forces the operator sequence (A/B
 * measurements, parity tests); returns the previous setting.  Initial value: environment TSG_SAG_FUSED (default 1). */
int tsg_sag_set_fused(int on);
/* Where the forward leaves a saved tensor inside the arena (a pure function of the shape): byte offset and size of
 * `field` of pooling level `level` (0..2).  What a caller needs to read back SAGPool.forward's other return values
 * (Code/sag/layers.py:26 returns perm; the parity tests assert it level by level).  perm: int64 [n[level+1]];
 * score / h / xg: fp32 [n], [n, hidden], [n[level+1], hidden]; CSR arrays: int32 / fp32 of the level's A_hat. */
enum { TSG_SAG_PERM = 0, TSG_SAG_SCORE = 1, TSG_SAG_H = 2, TSG_SAG_XG = 3, TSG_SAG_ROWPTR = 4, TSG_SAG_COLIDX = 5,
       TSG_SAG_VAL = 6, TSG_SAG_INV = 7, TSG_SAG_STATUS = 8 /* int32: 0, or TSG_FUSED_* bits set by the graph-resident
       kernels when a graph's edge list is not coalesced + symmetric (any level; XG / CSR fields are only filled by the
       kernel-per-operator executor, TSG_SAG_FUSED=0) */ };
int tsg_sag_arena_locate(const tsg_sag_shape* shape, int level, int field, size_t* offset, size_t* bytes);
int tsg_sag_encoder_fwd(const tsg_sag_shape* shape, const float* x, const int64_t* row, const int64_t* col,
                        const int64_t* level_ptr, const float* const* params, float* z,
                        void* arena, size_t arena_bytes, void* stream);
int tsg_sag_encoder_bwd(const tsg_sag_shape* shape, const float* x, const int64_t* level_ptr,
                        const float* const* params, const float* dz, float* const* grads,
                        void* arena, size_t arena_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * K14  the whole 2stg SAGPool training step in one call
 *   replaces the body of the stage-1 loop of Code/sag/train_triplet.py:203-212 for a packed batch: TNet forward
 *   (tripletnet.py:14-24 -> network.py:30-53, head included: lin1 / ReLU / dropout / lin2 / ReLU / lin3 / log_softmax),
 *   MarginRankingLoss(margin)(d_p, d_n, -1) (train_triplet.py:196,208-211) and loss.backward().  Enqueues: K10 forward,
 *   head forward, K9 forward + backward, head backward (fixed-order gradient reduction), K10 backward -- without
 *   returning to the interpreter in between (round 1: 1.46 ms of Python per 1.69 ms step).
 *   params / grads: 18 device pointers = the 12 of K10, then lin1.weight [H, 2H], lin1.bias [H], lin2.weight [H/2, H],
 *   lin2.bias, lin3.weight [C, H/2], lin3.bias (torch.nn.Linear layout).  triplets int64 [T, 3] rows of the batch.
 *   dropout_mask: NULL, or a [G, H] keep-multiplier matrix (0 or 1/(1-p): what parity tests inject); with NULL and
 *   dropout_p > 0 a counter-based hash of (seed, graph, column) draws the mask.  loss: device float (mean over T);
 *   emb_out: optional [G, C] embeddings (log-softmax vectors).  Gradients are WRITTEN (not accumulated).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int64_t num_classes;       /* C = final_dim */
  int64_t num_triplets;      /* T */
  float margin, eps, dropout_p;
  uint64_t seed;
} tsg_sag_head;
size_t tsg_sag_triplet_step_workspace_bytes(const tsg_sag_shape* shape, const tsg_sag_head* head);
int tsg_sag_triplet_step_compact(const tsg_sag_shape* shape, const tsg_sag_head* head, const int32_t* label,
                                 const int32_t* local_row, const int32_t* local_col, const int64_t* edge_ptr,
                                 const int64_t* level_ptr, const float* const* params, const int64_t* triplets,
                                 const float* dropout_mask /*nullable*/, float* const* grads, float* loss,
                                 float* emb_out /*nullable*/, void* arena, size_t arena_bytes, void* workspace,
                                 size_t workspace_bytes, void* stream);

/* The two halves of K14 for a loss evaluated outside the call (all-gather formulation: embeddings of every rank are
 * gathered, the global triplet loss is evaluated on the gathered matrix, this rank's slice of d(loss)/d(emb) comes back):
 * fwd = encoder + head -> emb [G, C]; bwd = head backward + encoder backward from demb [G, C].  Same arena and workspace
 * (tsg_sag_triplet_step_workspace_bytes) in both calls. */
int tsg_sag_step_fwd_compact(const tsg_sag_shape* shape, const tsg_sag_head* head, const int32_t* label,
                             const int32_t* local_row, const int32_t* local_col, const int64_t* edge_ptr,
                             const int64_t* level_ptr, const float* const* params, const float* dropout_mask /*nullable*/,
                             float* emb, void* arena, size_t arena_bytes, void* workspace, size_t workspace_bytes,
                             void* stream);
int tsg_sag_step_bwd_compact(const tsg_sag_shape* shape, const tsg_sag_head* head, const int32_t* label,
                             const int64_t* level_ptr, const float* const* params, const float* emb, const float* demb,
                             float* const* grads, void* arena, size_t arena_bytes, void* workspace,
                             size_t workspace_bytes, void* stream);

/* The supervised ("original") setting of the same model.  num_triplets / margin / eps of `head` are not used here.
 * The head backward of K14 takes every even hidden width whose head forward fits shared memory (H = 128 with C <= 64
 * included): where its per-CTA gradient row does not fit, per-graph deltas go to the workspace and the parameter
 * gradients come from K3's fixed-order reductions (tsg_linear_bwd_weight / tsg_relu_bwd_colsum).
 *   tsg_sag_nll_step_compact replaces the body of the loop of Code/sag/train.py:194: out = model(data);
 *     F.nll_loss(out, data.y) (mean over the G graphs); loss.backward().  y int64 [G] graph labels; loss: device float;
 *     emb_out optional [G, C] log-probabilities; gradients WRITTEN into the 18 grads as in K14.  The gradients are
 *     bit-identical to tsg_sag_step_fwd_compact + autograd F.nll_loss + tsg_sag_step_bwd_compact.
 *   tsg_sag_classify_compact replaces `test()` of Code/sag/train.py:19-29 on a packed batch: model.eval() forward
 *     (tsg_sag_encoder_embed_compact, then the head with dropout off), pred int64 [G] = out.max(dim=1)[1] (first index
 *     on ties), optional logp_out [G, C]; with y: *correct (int64) = #(pred == y) and *nll_sum (float) =
 *     F.nll_loss(out, y, reduction='sum'), both reduced in a fixed order (y NULL: both must be NULL).
 * A label outside [0, C) is clamped for the read and sets bit TSG_SAG_LABEL_RANGE in shape->status (or, when that is
 * NULL, in the arena's TSG_SAG_STATUS word).  Workspace queries return 0 exactly when the call cannot run the shape. */
#define TSG_SAG_LABEL_RANGE 8
size_t tsg_sag_nll_step_workspace_bytes(const tsg_sag_shape* shape, const tsg_sag_head* head);
int tsg_sag_nll_step_compact(const tsg_sag_shape* shape, const tsg_sag_head* head, const int32_t* label,
                             const int32_t* local_row, const int32_t* local_col, const int64_t* edge_ptr,
                             const int64_t* level_ptr, const float* const* params, const int64_t* y,
                             const float* dropout_mask /*nullable*/, float* const* grads, float* loss,
                             float* emb_out /*nullable*/, void* arena, size_t arena_bytes, void* workspace,
                             size_t workspace_bytes, void* stream);
size_t tsg_sag_classify_workspace_bytes(const tsg_sag_shape* shape, const tsg_sag_head* head);
int tsg_sag_classify_compact(const tsg_sag_shape* shape, const tsg_sag_head* head, const int32_t* label,
                             const int32_t* local_row, const int32_t* local_col, const int64_t* edge_ptr,
                             const int64_t* level_ptr, const float* const* params, const int64_t* y /*nullable*/,
                             int64_t* pred, float* logp_out /*nullable*/, int64_t* correct /*nullable*/,
                             float* nll_sum /*nullable*/, void* arena, size_t arena_bytes, void* workspace,
                             size_t workspace_bytes, void* stream);

/* Row-softmax backward from the saved output of tsg_linear_fwd(..., TSG_LIN_SOFTMAX): dL = S * (dS - rowsum(S * dS))
 * (SoftPoolingGcnEncoder's assignment, encoders.py:369; SURVEY A.4 K7). */
int tsg_softmax_bwd(const float* S, const float* dS, float* dL, int64_t num_rows, int64_t num_cols, void* stream);

/* tsg_spmm plus dot_out[r] = Y[r, :] . dot_vec from K2's epilogue (conv + the score layer's h @ ws of
 * Code/sag/layers.py:18 in one pass); bit-identical to tsg_spmm followed by tsg_linear_fwd(Y, dot_vec, out_feat = 1),
 * which is what runs for shapes the epilogue does not cover (feat > 128 or not a multiple of 4). */
int tsg_spmm_dot(const int32_t* rowptr, const int32_t* colidx, const float* val /*nullable*/, const float* H,
                 const float* bias /*nullable*/, float* Y, const float* dot_vec, float* dot_out,
                 int64_t num_rows, int64_t feat, int flags, void* stream);

/* SAGPool gate + readout in one pass (used by tsg_sag_encoder_fwd when hidden % 4 == 0): xo[i] = x[perm[i]] *
 * tanh(score[perm[i]]) (Code/sag/layers.py:21) and out[g] = [max || mean] over graph g's rows of xo
 * (network.py:36,40,44), argmax as tsg_readout_fwd.  Bit-identical to tsg_gate_gather_fwd + tsg_readout_fwd. */
int tsg_gate_readout_fwd(const float* x, const float* score, const int64_t* perm, const int64_t* graph_ptr_out,
                         int64_t num_graphs, int64_t feat, float* xo, float* out, int64_t out_stride,
                         int32_t* argmax, void* stream);

/* Gate + readout plus the NEXT GCNConv's feature transform (Code/sag/network.py:38,42 -> PyG GCNConv: x W before the
 * propagation): xw_next[i] = xo[i] @ w_next, w_next [feat, feat] row-major as [in, out].  feat = 32 / 64: one flat pass
 * gates the rows and multiplies them by w_next while they are on chip (the pooled rows are not read back from HBM for
 * the product), then the readout runs on xo.  xo, out, argmax and xw_next are bit-identical to tsg_gate_gather_fwd,
 * tsg_readout_fwd and tsg_linear_fwd(xo, w_next); other widths, or w_next / xw_next NULL, run tsg_gate_readout_fwd
 * (+ tsg_linear_fwd).  num_rows_out = graph_ptr_out[G] (known on the host). */
int tsg_gate_readout_linear_fwd(const float* x, const float* score, const int64_t* perm, const int64_t* graph_ptr_out,
                                int64_t num_graphs, int64_t num_rows_out, int64_t feat, float* xo, float* out,
                                int64_t out_stride, int32_t* argmax, const float* w_next /*nullable*/,
                                float* xw_next /*nullable*/, void* stream);

/* Score-side gate backward driven by perm (the other half of tsg_sag_conv_bwd_fused): dscore[perm[i]] =
 * (dxo[i] . x[perm[i]]) * (1 - tanh(score)^2), zero for dropped nodes, and dbias_score = sum(dscore) (the score
 * GCNConv's bias gradient).  dscore bit-identical to tsg_gate_gather_bwd; feat % 4 == 0. */
/* (draws a counter from the per-device pool created by tsg_init_device) */
size_t tsg_gate_score_bwd_workspace_bytes(void);
int tsg_gate_score_bwd(const float* dxo, const float* x, const float* score, const int64_t* perm,
                       int64_t num_perm, int64_t num_nodes, int64_t feat, float* dscore, float* dbias_score,
                       void* workspace, size_t workspace_bytes, void* stream);

/* conv1 on one-hot node-label features: Y = act(A_hat * W[label] + bias) with the table gathered inside K2 (x W is
 * never materialised), plus the optional Y @ dot_vec epilogue of tsg_spmm_dot.  Bit-identical to tsg_embed_fwd followed
 * by tsg_spmm_dot.  feat % 4 == 0 (<= 128 with dot_vec), 16-byte aligned W / bias / Y; TSG_EINVAL otherwise. */
int tsg_spmm_label_dot(const int32_t* rowptr, const int32_t* colidx, const float* val /*nullable*/, const float* W,
                       const int32_t* label, int64_t num_labels, const float* bias /*nullable*/, float* Y,
                       const float* dot_vec /*nullable*/, float* dot_out /*nullable*/, int64_t num_rows, int64_t feat,
                       int flags, void* stream);

/* One level's conv-output backward, fused (used by tsg_sag_encoder_bwd when hidden % 4 == 0): with
 * dh = inv >= 0 ? dxo[inv] * tanh(score) : 0 (gate backward of Code/sag/layers.py:21, never materialised),
 * dhm = ReLU'(h) * (dh + dsw ws^T), dbias = colsum(dhm), dws = h^T dsw (score_layer.weight gradient).
 * dhm / dbias bit-identical to tsg_gate_gather_bwd + tsg_relu_bwd_colsum_rank1; dws to fp32 summation order of
 * tsg_linear_bwd_weight.  workspace >= 2 * tsg_colsum_workspace_bytes(N, F). */
int tsg_sag_conv_bwd_fused(const float* dxo, const int32_t* inv, const float* score, const float* h,
                           const float* dsw, const float* ws_vec, float* dhm, float* dbias, float* dws,
                           int64_t N, int64_t F, void* workspace, size_t workspace_bytes, void* stream);

/* Compact level-0 input (SURVEY 8f n1 feeder): the batch as the dataset stores it -- one categorical label per node
 * (the one-hot x of Code/sag/train.py:34 / load_data.py:74-87 is onehot(label), in_feat = number of labels) and
 * graph-local int32 edge endpoints with per-graph offsets edge_ptr [G+1] (device).  conv1's x @ W becomes a row gather
 * of W (K3c), its dW a segment sum, K1b reads the local endpoints: z is bit-identical to tsg_sag_encoder_fwd on the
 * expanded batch (tsg_pack_batch), gradients agree to fp32 summation order (level-0 dW only; all others bit-identical).
 * Same arena (tsg_sag_arena_bytes) and the same level_ptr / params / grads as above. */
int tsg_sag_encoder_fwd_compact(const tsg_sag_shape* shape, const int32_t* label, const int32_t* local_row,
                                const int32_t* local_col, const int64_t* edge_ptr, const int64_t* level_ptr,
                                const float* const* params, float* z, void* arena, size_t arena_bytes, void* stream);
int tsg_sag_encoder_embed_compact(const tsg_sag_shape* shape, const int32_t* label, const int32_t* local_row,
                                  const int32_t* local_col, const int64_t* edge_ptr, const int64_t* level_ptr,
                                  const float* const* params, float* z, void* arena, size_t arena_bytes, void* stream);
int tsg_sag_encoder_bwd_compact(const tsg_sag_shape* shape, const int32_t* label, const int64_t* level_ptr,
                                const float* const* params, const float* dz, float* const* grads,
                                void* arena, size_t arena_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * K3c  level-0 products for one-hot node-label features (x = onehot(label), never materialised)
 *   replaces x @ W1 / x^T dY of Code/sag/network.py:34 (GCNConv.lin on data.x) for label-featured datasets.
 *   out[i, :] = W[label[i], :] (zero row for a label outside [0, K));  dW[k, :] = sum_{label[i] == k} dY[i, :],
 *   fixed summation order.  tsg_embed_bwd_weight_workspace_bytes returns 0 when a K x M table does not fit
 *   shared memory (use tsg_pack_batch + the dense K3 entries then).
 * ------------------------------------------------------------------------------------------ */
int tsg_embed_fwd(const float* W, const int32_t* label, float* out, int64_t N, int64_t K, int64_t M, void* stream);
size_t tsg_embed_bwd_weight_workspace_bytes(int64_t K, int64_t M);
int tsg_embed_bwd_weight(const int32_t* label, const float* dY, float* dW, int64_t N, int64_t K, int64_t M,
                         void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TSG_H_ */
