// K10 -- native step executor for the SAGPool encoder (Code/sag/network.py:33-46 + layers.py:14-26).
//
// The per-kernel entry points of this library are driven from Python one ctypes call at a time; with
// ~110 launches per training step that costs 3.3 ms of host time for 2.9 ms of kernels (measured,
// profiles/r01b_bench_breakdown.txt): the step was launch bound.  This file sequences the SAME entry
// points (same kernels, same order, same arithmetic as tsg/nn.py PackedSAGNet drives them) from C++:
// one call enqueues the whole encoder forward, one call the whole backward.  Every intermediate lives
// in a caller-provided arena whose layout is a pure function of the shape, so the forward leaves its
// saved tensors where the backward finds them; nothing is allocated, nothing synchronises.
//
//   per level l = 0..2 (n = n[l] rows in, k = n[l+1] rows out):
//     CSR   = K1b(edges, level_ptr[0]) at l = 0; K1c(CSR_{l-1}, perm, inv) below -- conv_l and score_l share it
//     h     = ReLU(A_hat (x_l W_l) + b_l)                     network.py:34,38,42
//     score = A_hat (h ws_l) + bs_l                           layers.py:18
//     perm  = topk(score)                                     layers.py:20
//     inv   = filter_adj's relabelling table                  layers.py:23 (the filtered list itself is never built)
//     x_{l+1} = h[perm] * tanh(score[perm])                   layers.py:21
//     out_l = [gmp(x_{l+1}) || gap(x_{l+1})]                  network.py:36,40,44
//   z = out_0 + out_1 + out_2                                 network.py:46
#include "common.cuh"
#include "sag_fused.cuh"

namespace tsg {

struct LevelBuf {
  int64_t* eptr;
  int32_t *rowptr, *colidx, *t_rowptr, *t_colidx;
  float *val, *t_val;
  float *xw, *h, *sw, *score, *xg, *out;
  int64_t* perm;
  int32_t* inv;
  int32_t* argmax;
};

struct SagArena {
  LevelBuf lv[3];
  // backward temporaries, sized for level 0 and reused by every level
  float *dxg, *dh, *dhm, *dxw, *dscore, *dsw;
  void* scratch; size_t scratch_bytes;
  // graph-resident forward (k13_sag_fused.cu): scheduling counters + status word
  unsigned* sched; int* status;
  size_t total;
};

static size_t scratch_need(const tsg_sag_shape* sh) {
  size_t m = 0;
  auto up = [&](size_t v) { if (v > m) m = v; };
  for (int l = 0; l < 3; ++l) {
    up(tsg_csr_build_graphs_workspace_bytes(sh->num_graphs, sh->num_edges));
    up(tsg_topk_workspace_bytes(sh->n[l], sh->num_graphs));
    up(tsg_csr_filter_workspace_bytes(sh->n[l + 1]));
    up(2 * tsg_colsum_workspace_bytes(sh->n[l], sh->hidden));
    up(tsg_linear_bwd_weight_workspace_bytes(l == 0 ? sh->in_feat : sh->hidden, sh->hidden));
    up(tsg_linear_bwd_weight_workspace_bytes(sh->hidden, 1));
  }
  up(tsg_embed_bwd_weight_workspace_bytes(sh->in_feat, sh->hidden));
  up(tsg_gate_score_bwd_workspace_bytes());
  return align_up(m, 256) + 256;
}

// layout(arena == nullptr) only measures
static void layout(const tsg_sag_shape* sh, void* arena, SagArena* a) {
  char* base = (char*)arena;
  size_t off = 0;
  auto take = [&](size_t bytes) -> void* {
    void* p = base ? (void*)(base + off) : nullptr;
    off += align_up(bytes, 256);
    return p;
  };
  const int64_t G = sh->num_graphs, H = sh->hidden, E = sh->num_edges;
  for (int l = 0; l < 3; ++l) {
    LevelBuf& b = a->lv[l];
    const int64_t n = sh->n[l], k = sh->n[l + 1], cap = E + n;
    b.eptr = (int64_t*)take((G + 1) * 8);
    b.rowptr = (int32_t*)take((n + 1) * 4); b.t_rowptr = (int32_t*)take((n + 1) * 4);
    b.colidx = (int32_t*)take(cap * 4); b.t_colidx = (int32_t*)take(cap * 4);
    b.val = (float*)take(cap * 4); b.t_val = (float*)take(cap * 4);
    b.xw = (float*)take(n * H * 4); b.h = (float*)take(n * H * 4);
    b.sw = (float*)take(n * 4); b.score = (float*)take(n * 4);
    b.perm = (int64_t*)take((k > 0 ? k : 1) * 8);
    b.inv = (int32_t*)take((n > 0 ? n : 1) * 4);
    b.xg = (float*)take((k > 0 ? k : 1) * H * 4);
    b.out = (float*)take(G * 2 * H * 4);
    b.argmax = (int32_t*)take(G * H * 4);
  }
  const int64_t n0 = sh->n[0] > 0 ? sh->n[0] : 1;
  a->dxg = (float*)take(n0 * H * 4); a->dh = (float*)take(n0 * H * 4);
  a->dhm = (float*)take(n0 * H * 4); a->dxw = (float*)take(n0 * H * 4);
  a->dscore = (float*)take(n0 * 4); a->dsw = (float*)take(n0 * 4);
  a->scratch_bytes = scratch_need(sh);
  a->scratch = take(a->scratch_bytes);
  a->sched = (unsigned*)take(256);
  a->status = (int*)((char*)a->sched + 128);
  if (sh->status && base) a->status = sh->status;      // caller-owned persistent status word
  a->total = off;
  if (sh->flags & TSG_SAG_COALESCED)          // symmetric operators: the transposed CSR is the same arrays
    for (int l = 0; l < 3; ++l) {
      LevelBuf& b = a->lv[l];
      b.t_rowptr = b.rowptr; b.t_colidx = b.colidx; b.t_val = b.val;
    }
}

__global__ void __launch_bounds__(256)
k_add3(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ c, float* __restrict__ o, int64_t n) {
  pdl_wait();
  pdl_launch_dependents();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    o[i] = (a[i] + b[i]) + c[i];
}

// Level-0 input: either the PyG wire format (dense x [n0, in_feat] fp32 + global int64 edge_index) or the compact
// one (one categorical label per node = the one-hot x, graph-local int32 endpoints + per-graph edge offsets).
struct SagInput {
  const float* x;
  const int64_t *row, *col;
  const int32_t* label;
  const int32_t *lrow, *lcol;
  const int64_t* edge_ptr;
};

static bool sag_unfused_env() {        // TSG_SAG_UNFUSED=1: the kernel-per-op backward (A/B measurements, parity tests)
  static const bool v = getenv("TSG_SAG_UNFUSED") != nullptr;
  return v;
}

// TSG_SAG_FUSED=0 (or tsg_sag_set_fused(0)): the kernel-per-operator executor of round 1 (A/B runs, parity tests)
static int g_sag_fused = -1;
static bool sag_fused_env() {
  if (g_sag_fused < 0) g_sag_fused = !(getenv("TSG_SAG_FUSED") && getenv("TSG_SAG_FUSED")[0] == '0');
  return g_sag_fused != 0;
}

static bool use_fused(const tsg_sag_shape* sh, bool compact) {
  if (!compact || !sag_fused_env() || sh->max_graph_edges <= 0) return false;
  for (int l = 0; l < 3; ++l) if (sh->max_graph_nodes[l] > 32767) return false;
  return fused_supported((int)sh->hidden, (int)sh->in_feat, (int)sh->max_graph_nodes[0], (int)sh->max_graph_nodes[1],
                         (int)sh->max_graph_edges);
}

static void fill_fused(FusedArgs& f, const tsg_sag_shape* sh, const SagArena& a, const int32_t* label, const int32_t* lrow,
                       const int32_t* lcol, const int64_t* edge_ptr, const int64_t* level_ptr, const float* const* params) {
  f.G = (int)sh->num_graphs; f.L = (int)sh->in_feat; f.H = (int)sh->hidden;
  for (int l = 0; l < 3; ++l) f.nmax[l] = (int)sh->max_graph_nodes[l];
  f.emax = (int)sh->max_graph_edges;
  f.ratio = (float)sh->pooling_ratio; f.avg_degree = (double)sh->num_edges / (double)(sh->n[0] > 0 ? sh->n[0] : 1);
  f.cls = 0; f.cls_nlo = 0; f.cls_elo = -1;
  f.label = label; f.lrow = lrow; f.lcol = lcol; f.edge_ptr = edge_ptr; f.level_ptr = level_ptr;
  for (int i = 0; i < 12; ++i) f.params[i] = params[i];
  for (int l = 0; l < 3; ++l) {
    f.h[l] = a.lv[l].h; f.score[l] = a.lv[l].score; f.perm[l] = a.lv[l].perm; f.argmax[l] = a.lv[l].argmax;
  }
  f.z = nullptr;
  f.sched = a.sched; f.status = a.status;
}

static bool shape_ok(const tsg_sag_shape* sh) {
  if (!sh || sh->num_graphs <= 0 || sh->in_feat <= 0 || sh->hidden <= 0 || sh->num_edges < 0) return false;
  for (int l = 0; l < 4; ++l) if (sh->n[l] <= 0) return false;
  for (int l = 0; l < 3; ++l) if (sh->max_graph_nodes[l] <= 0) return false;
  return true;
}

}  // namespace tsg

using namespace tsg;

#define TSG_TRY(call)                 \
  do {                                \
    int _rc = (call);                 \
    if (_rc != TSG_OK) return _rc;    \
  } while (0)

extern "C" int tsg_sag_set_fused(int on) {
  const int prev = sag_fused_env() ? 1 : 0;
  g_sag_fused = on ? 1 : 0;
  return prev;
}

extern "C" size_t tsg_sag_arena_bytes(const tsg_sag_shape* shape) {
  if (!shape_ok(shape)) return 0;
  SagArena a;
  layout(shape, nullptr, &a);
  return a.total;
}

extern "C" int tsg_sag_arena_locate(const tsg_sag_shape* sh, int level, int field, size_t* offset, size_t* bytes) {
  TSG_REQUIRE(shape_ok(sh) && level >= 0 && level < 3 && offset && bytes, "sag_arena_locate: bad argument");
  SagArena a;
  char* const base = (char*)256;            // any non-null base: only differences are used
  tsg_sag_shape own = *sh;
  own.status = nullptr;                     // the arena's own word, not the caller's
  layout(&own, base, &a);
  const LevelBuf& b = a.lv[level];
  const int64_t n = sh->n[level], k = sh->n[level + 1], H = sh->hidden;
  const void* p = nullptr; size_t sz = 0;
  switch (field) {
    case TSG_SAG_PERM: p = b.perm; sz = (size_t)k * 8; break;
    case TSG_SAG_SCORE: p = b.score; sz = (size_t)n * 4; break;
    case TSG_SAG_H: p = b.h; sz = (size_t)n * H * 4; break;
    case TSG_SAG_XG: p = b.xg; sz = (size_t)k * H * 4; break;
    case TSG_SAG_ROWPTR: p = b.rowptr; sz = (size_t)(n + 1) * 4; break;
    case TSG_SAG_COLIDX: p = b.colidx; sz = (size_t)(sh->num_edges + n) * 4; break;
    case TSG_SAG_VAL: p = b.val; sz = (size_t)(sh->num_edges + n) * 4; break;
    case TSG_SAG_INV: p = b.inv; sz = (size_t)n * 4; break;
    case TSG_SAG_STATUS: p = a.status; sz = 4; break;
    default: set_error("sag_arena_locate: unknown field %d", field); return TSG_EINVAL;
  }
  *offset = (size_t)((const char*)p - base);
  *bytes = sz;
  return TSG_OK;
}

static int sag_fwd(const tsg_sag_shape* sh, const SagInput& in, const int64_t* level_ptr, const float* const* params,
                   float* z, void* arena, size_t arena_bytes, void* stream, bool forward_only = false) {
  SagArena a;
  layout(sh, arena, &a);
  if (arena_bytes < a.total) { set_error("sag_encoder_fwd: arena too small (%zu < %zu)", arena_bytes, a.total); return TSG_EWORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t G = sh->num_graphs, H = sh->hidden, E = sh->num_edges;
  if (!sh->status) cudaMemsetAsync(a.status, 0, sizeof(int), st);       // every path leaves a defined status word
  // graph-resident path (K13): the whole encoder forward in one kernel per size class.  Forward only: it keeps every
  // intermediate in shared memory, while the backward below consumes the per-level CSRs / gated rows from the arena.
  if (forward_only && use_fused(sh, in.label != nullptr)) {
    FusedArgs f;
    fill_fused(f, sh, a, in.label, in.lrow, in.lcol, in.edge_ptr, level_ptr, params);
    f.z = z;
    return launch_sag_fused_fwd(f, st);
  }
  const float* xin = in.x;
  bool xw_ready = false;         // b.xw already written by the previous level's gate kernel
  for (int l = 0; l < 3; ++l) {
    LevelBuf& b = a.lv[l];
    const int64_t n = sh->n[l], k = sh->n[l + 1], fin = l == 0 ? sh->in_feat : H;
    const float *W = params[4 * l], *bias = params[4 * l + 1], *ws = params[4 * l + 2], *bs = params[4 * l + 3];
    const int64_t* ptr_l = level_ptr + (size_t)l * (G + 1);
    const int64_t* ptr_n = level_ptr + (size_t)(l + 1) * (G + 1);
    const bool sym = in.label && (sh->flags & TSG_SAG_COALESCED);
    if (l == 0 && sym) {
      TSG_TRY(tsg_csr_build_graphs_sym_local(in.lrow, in.lcol, in.edge_ptr, ptr_l, G, n, E, sh->max_graph_nodes[l], b.rowptr,
                                             b.colidx, b.val, a.status, stream));
    } else if (l == 0 && in.label) {
      TSG_TRY(tsg_csr_build_graphs_local(in.lrow, in.lcol, in.edge_ptr, ptr_l, G, n, E, sh->max_graph_nodes[l], b.rowptr,
                                         b.colidx, b.val, nullptr, b.t_rowptr, b.t_colidx, b.t_val, nullptr, a.scratch,
                                         a.scratch_bytes, stream));
    } else if (l == 0) {
      TSG_TRY(tsg_edge_ptr(in.row, E, nullptr, ptr_l, G, b.eptr, stream));
      TSG_TRY(tsg_csr_build_graphs(in.row, in.col, b.eptr, ptr_l, G, n, E, sh->max_graph_nodes[l], b.rowptr, b.colidx, b.val,
                                   nullptr, b.t_rowptr, b.t_colidx, b.t_val, nullptr, a.scratch, a.scratch_bytes, stream));
    } else {        // K1c: the pooled level's CSR straight from the previous level's CSR, perm and inv
      const LevelBuf& pb = a.lv[l - 1];
      if (sym) TSG_TRY(tsg_csr_filter(pb.rowptr, pb.colidx, nullptr, nullptr, pb.perm, pb.inv, n, b.rowptr, b.colidx, b.val,
                                      nullptr, nullptr, nullptr, a.scratch, a.scratch_bytes, stream));
      else TSG_TRY(tsg_csr_filter(pb.rowptr, pb.colidx, pb.t_rowptr, pb.t_colidx, pb.perm, pb.inv, n, b.rowptr, b.colidx, b.val,
                                  b.t_rowptr, b.t_colidx, b.t_val, a.scratch, a.scratch_bytes, stream));
    }
    static const bool no_label_spmm = getenv("TSG_NO_LABEL_SPMM") != nullptr;
    const bool label_spmm = l == 0 && in.label && H % 4 == 0 && H <= 128 && !no_label_spmm &&
                            ((((uintptr_t)W) | ((uintptr_t)bias) | ((uintptr_t)ws)) & 15) == 0;
    if (label_spmm) {
      // conv1 on one-hot labels: x W = W[label] is gathered from the 11 KB table inside K2, never written
      TSG_TRY(tsg_spmm_label_dot(b.rowptr, b.colidx, b.val, W, in.label, fin, bias, b.h, ws, b.sw, n, H, TSG_SPMM_RELU, stream));
    } else {
      if (l == 0 && in.label) TSG_TRY(tsg_embed_fwd(W, in.label, b.xw, n, fin, H, stream));     // onehot(label) @ W
      else if (!xw_ready) TSG_TRY(tsg_linear_fwd(xin, W, nullptr, b.xw, n, fin, H, 0, 0, stream));
      // h = ReLU(A_hat xw + b) and, from the same registers, sw = h ws (the score layer's product)
      TSG_TRY(tsg_spmm_dot(b.rowptr, b.colidx, b.val, b.xw, bias, b.h, ws, b.sw, n, H, TSG_SPMM_RELU, stream));
    }
    TSG_TRY(tsg_spmm(b.rowptr, b.colidx, b.val, b.sw, bs, b.score, n, 1, 0, stream));
    TSG_TRY(tsg_topk_bounded(b.score, ptr_l, ptr_n, G, n, sh->max_graph_nodes[l], b.perm, a.scratch, a.scratch_bytes, stream));
    TSG_TRY(tsg_inv_perm(b.perm, k, n, b.inv, stream));            // filter_adj's relabelling table (layers.py:23)
    static const bool no_gr = getenv("TSG_NO_GATE_READOUT") != nullptr;
    if (H % 4 == 0 && !sag_unfused_env() && !no_gr) {
      // gate + readout in one pass (the gated rows are not read back), and the next level's x W from the same rows
      const bool next_xw = l < 2 && (((uintptr_t)params[4 * (l + 1)]) & 15) == 0;
      TSG_TRY(tsg_gate_readout_linear_fwd(b.h, b.score, b.perm, ptr_n, G, k, H, b.xg, b.out, 2 * H, b.argmax,
                                          next_xw ? params[4 * (l + 1)] : nullptr, next_xw ? a.lv[l + 1].xw : nullptr, stream));
      xw_ready = next_xw;
    } else {
      xw_ready = false;
      TSG_TRY(tsg_gate_gather_fwd(b.h, b.score, b.perm, nullptr, b.xg, nullptr, k, H, stream));
      TSG_TRY(tsg_readout_fwd(b.xg, ptr_n, G, H, TSG_READOUT_MAX | TSG_READOUT_MEAN, b.out, 2 * H, b.argmax, stream));
    }
    xin = b.xg;
  }
  const int64_t tot = G * 2 * H;
  return launch_pdl("sag_encoder_fwd", k_add3, grid_for(tot, 256, 8), 256, 0, st, (const float*)a.lv[0].out, (const float*)a.lv[1].out,
                    (const float*)a.lv[2].out, z, tot);
}

extern "C" int tsg_sag_encoder_fwd(const tsg_sag_shape* sh, const float* x, const int64_t* row, const int64_t* col,
                                   const int64_t* level_ptr, const float* const* params, float* z,
                                   void* arena, size_t arena_bytes, void* stream) {
  TSG_REQUIRE(shape_ok(sh), "sag_encoder_fwd: bad shape");
  TSG_REQUIRE(x && level_ptr && params && z && arena && (sh->num_edges == 0 || (row && col)), "sag_encoder_fwd: null pointer");
  const SagInput in{x, row, col, nullptr, nullptr, nullptr, nullptr};
  return sag_fwd(sh, in, level_ptr, params, z, arena, arena_bytes, stream);
}

extern "C" int tsg_sag_encoder_fwd_compact(const tsg_sag_shape* sh, const int32_t* label, const int32_t* local_row,
                                           const int32_t* local_col, const int64_t* edge_ptr, const int64_t* level_ptr,
                                           const float* const* params, float* z, void* arena, size_t arena_bytes,
                                           void* stream) {
  TSG_REQUIRE(shape_ok(sh), "sag_encoder_fwd_compact: bad shape");
  TSG_REQUIRE(label && edge_ptr && level_ptr && params && z && arena && (sh->num_edges == 0 || (local_row && local_col)),
              "sag_encoder_fwd_compact: null pointer");
  TSG_REQUIRE(tsg_embed_bwd_weight_workspace_bytes(sh->in_feat, sh->hidden) > 0,
              "sag_encoder_fwd_compact: %lld labels x %lld hidden does not fit the label-table kernels; expand with tsg_pack_batch",
              (long long)sh->in_feat, (long long)sh->hidden);
  const SagInput in{nullptr, nullptr, nullptr, label, local_row, local_col, edge_ptr};
  return sag_fwd(sh, in, level_ptr, params, z, arena, arena_bytes, stream);
}

extern "C" int tsg_sag_encoder_embed_compact(const tsg_sag_shape* sh, const int32_t* label, const int32_t* local_row,
                                             const int32_t* local_col, const int64_t* edge_ptr, const int64_t* level_ptr,
                                             const float* const* params, float* z, void* arena, size_t arena_bytes,
                                             void* stream) {
  TSG_REQUIRE(shape_ok(sh), "sag_encoder_embed_compact: bad shape");
  TSG_REQUIRE(label && edge_ptr && level_ptr && params && z && arena && (sh->num_edges == 0 || (local_row && local_col)),
              "sag_encoder_embed_compact: null pointer");
  TSG_REQUIRE(tsg_embed_bwd_weight_workspace_bytes(sh->in_feat, sh->hidden) > 0,
              "sag_encoder_embed_compact: %lld labels x %lld hidden does not fit the label-table kernels; expand with tsg_pack_batch",
              (long long)sh->in_feat, (long long)sh->hidden);
  const SagInput in{nullptr, nullptr, nullptr, label, local_row, local_col, edge_ptr};
  return sag_fwd(sh, in, level_ptr, params, z, arena, arena_bytes, stream, true);
}

static int sag_bwd(const tsg_sag_shape* sh, const SagInput& in, const int64_t* level_ptr, const float* const* params,
                   const float* dz, float* const* grads, void* arena, size_t arena_bytes, void* stream) {
  SagArena a;
  layout(sh, arena, &a);
  if (arena_bytes < a.total) { set_error("sag_encoder_bwd: arena too small (%zu < %zu)", arena_bytes, a.total); return TSG_EWORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t G = sh->num_graphs, H = sh->hidden;
  // level l > 0's boundary in one pass (tsg_sag_boundary_bwd): conv_l's input and weight gradients and level l-1's
  // readout gradient, in the widths and alignments where the dense K3 kernels it reproduces would run
  static const bool no_dense = getenv("TSG_LIN_NODENSE") != nullptr;
  auto boundary = [&](int l) {
    if (l == 0) return false;
    const uintptr_t al = (uintptr_t)a.dxw | (uintptr_t)a.dxg | (uintptr_t)a.lv[l - 1].xg | (uintptr_t)a.lv[l - 1].argmax |
                         (uintptr_t)dz;
    return H % 4 == 0 && H >= 8 && H <= 64 && (al & 15) == 0 && !no_dense && !sag_unfused_env();
  };
  for (int l = 2; l >= 0; --l) {
    LevelBuf& b = a.lv[l];
    const int64_t n = sh->n[l], k = sh->n[l + 1], fin = l == 0 ? sh->in_feat : H;
    const float *W = params[4 * l], *ws = params[4 * l + 2];
    float *dW = grads[4 * l], *dbias = grads[4 * l + 1], *dws = grads[4 * l + 2], *dbs = grads[4 * l + 3];
    const float* xin = l == 0 ? in.x : a.lv[l - 1].xg;
    const int64_t* ptr_n = level_ptr + (size_t)(l + 1) * (G + 1);
    // d(x_{l+1}) = readout backward (+ the next level's input gradient)
    //   (the next level's linear backward already wrote its dX into a.dxg: accumulate in place; its boundary pass
    //   already added this readout term)
    if (l == 2 || !boundary(l + 1))
      TSG_TRY(tsg_readout_bwd(dz, 2 * H, b.argmax, ptr_n, G, k, H,
                              TSG_READOUT_MAX | TSG_READOUT_MEAN | (l < 2 ? TSG_READOUT_ACCUM : 0), a.dxg, stream));
    // fused level backward (k_sag_conv_bwd_v4): dh is never materialised and h is read once for mask, dbias and dws
    const bool fused = H % 4 == 0 && H <= 512 && (((uintptr_t)ws) & 15) == 0 && !sag_unfused_env();
    // score layer: score = A_hat (h ws) + bs; dscore from the gate, its sum = dbs
    if (fused) {
      TSG_TRY(tsg_gate_score_bwd(a.dxg, b.h, b.score, b.perm, k, n, H, a.dscore, dbs, a.scratch, a.scratch_bytes, stream));
    } else {
      TSG_TRY(tsg_gate_gather_bwd(a.dxg, b.h, b.score, b.inv, a.dh, a.dscore, n, H, stream));
      TSG_TRY(tsg_relu_bwd_colsum(a.dscore, nullptr, nullptr, dbs, n, 1, a.scratch, a.scratch_bytes, stream));
    }
    TSG_TRY(tsg_spmm(b.t_rowptr, b.t_colidx, b.t_val, a.dscore, nullptr, a.dsw, n, 1, 0, stream));
    // conv layer: h = ReLU(A_hat (x W) + b); its incoming gradient is dh + dsw ws^T, added on the fly
    if (fused) {
      TSG_TRY(tsg_sag_conv_bwd_fused(a.dxg, b.inv, b.score, b.h, a.dsw, ws, a.dhm, dbias, dws, n, H, a.scratch,
                                     a.scratch_bytes, stream));
    } else {
      TSG_TRY(tsg_linear_bwd_weight(b.h, a.dsw, dws, nullptr, n, H, 1, a.scratch, a.scratch_bytes, stream));
      TSG_TRY(tsg_relu_bwd_colsum_rank1(a.dh, b.h, a.dsw, ws, a.dhm, dbias, n, H, a.scratch, a.scratch_bytes, stream));
    }
    TSG_TRY(tsg_spmm(b.t_rowptr, b.t_colidx, b.t_val, a.dhm, nullptr, a.dxw, n, H, 0, stream));
    if (boundary(l)) {                 // d(x_l) + level l-1's readout gradient, and dW_l; k_{l-1} = n rows
      TSG_TRY(tsg_sag_boundary_bwd(a.dxw, xin, W, dz, 2 * H, a.lv[l - 1].argmax, level_ptr + (size_t)l * (G + 1), G, n, H,
                                   a.dxg, dW, a.scratch, a.scratch_bytes, stream));
    } else {
      if (l > 0) TSG_TRY(tsg_linear_fwd(a.dxw, W, nullptr, a.dxg, n, H, fin, 1, 0, stream));   // d(x_l), k_{l-1} = n rows
      if (l == 0 && in.label) TSG_TRY(tsg_embed_bwd_weight(in.label, a.dxw, dW, n, fin, H, a.scratch, a.scratch_bytes, stream));
      else TSG_TRY(tsg_linear_bwd_weight(xin, a.dxw, dW, nullptr, n, fin, H, a.scratch, a.scratch_bytes, stream));
    }
  }
  return check_launch("sag_encoder_bwd");
}

extern "C" int tsg_sag_encoder_bwd(const tsg_sag_shape* sh, const float* x, const int64_t* level_ptr,
                                   const float* const* params, const float* dz, float* const* grads,
                                   void* arena, size_t arena_bytes, void* stream) {
  TSG_REQUIRE(shape_ok(sh), "sag_encoder_bwd: bad shape");
  TSG_REQUIRE(x && level_ptr && params && dz && grads && arena, "sag_encoder_bwd: null pointer");
  const SagInput in{x, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  return sag_bwd(sh, in, level_ptr, params, dz, grads, arena, arena_bytes, stream);
}

extern "C" int tsg_sag_encoder_bwd_compact(const tsg_sag_shape* sh, const int32_t* label, const int64_t* level_ptr,
                                           const float* const* params, const float* dz, float* const* grads,
                                           void* arena, size_t arena_bytes, void* stream) {
  TSG_REQUIRE(shape_ok(sh), "sag_encoder_bwd_compact: bad shape");
  TSG_REQUIRE(label && level_ptr && params && dz && grads && arena, "sag_encoder_bwd_compact: null pointer");
  const SagInput in{nullptr, nullptr, nullptr, label, nullptr, nullptr, nullptr};
  return sag_bwd(sh, in, level_ptr, params, dz, grads, arena, arena_bytes, stream);
}
