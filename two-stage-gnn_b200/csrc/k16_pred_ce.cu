// K16 -- the prediction head and cross-entropy of the dense encoders' supervised settings (include/tsg.h).
//
// The dense step of Code/sage+gat+diffpool/train.py is encoder -> readout r [G, D0] -> a short chain of nn.Linear
// layers (ReLU where build_pred_layers puts one) -> F.cross_entropy, and the 2stg+ stage 2 of
// train_triplet_pre_train.py:249-256 the same with a softmax before the loss.  The encoder already runs on our kernels;
// this file is the rest of the step:
//
//   k_pred_fwd   one warp per row: every layer's units (one fmaf chain each, input index ascending from 0.f, + bias,
//                the chain tsg_linear_fwd's row kernels run), the optional softmax, CE = logsumexp(q) - q_y with max
//                subtraction; the activations go to the workspace (training) or the argmax / hit to it (evaluation)
//   k_sum_fixed  the mean (or the sum) of the per-row losses, and the correct count, in a fixed order (common.cuh)
//   k_pred_bwd   one warp per row: delta = (softmax(q) - onehot(y)) / G * dloss, back through the optional softmax
//                (p * (dq - <p, dq>)) and the layers' ReLU masks to dr; every layer's delta goes to the workspace
//   K3           dW_l = delta_l^T a_(l-1) (tsg_linear_bwd_weight), db_l = colsum(delta_l) (tsg_relu_bwd_colsum)
//
// Weights are read through the read-only cache: the heads are small (at most 8 layers of at most 256 x 256) and a
// step's head work is a few tens of microseconds against milliseconds of encoder.  No floating-point atomics.
#include "common.cuh"

namespace tsg {

constexpr int PRED_THREADS = 256;
constexpr int PRED_WARPS = PRED_THREADS / 32;
constexpr int PRED_W = TSG_PRED_MAX_WIDTH;

// the descriptor as the kernels read it (by value): widths, flags, parameters, and where each layer's [G, out_l]
// block of activations / deltas starts in the workspace
struct PredDesc {
  int L, D0, C, relu_mask, softmax_first;
  int out[TSG_PRED_MAX_LAYERS];
  int64_t off[TSG_PRED_MAX_LAYERS];
  const float* W[TSG_PRED_MAX_LAYERS];
  const float* b[TSG_PRED_MAX_LAYERS];
};

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// out[j] = softmax(in)[j] over n entries (shared memory, one warp); in and out may alias
__device__ __forceinline__ void row_softmax(const float* in, float* out, int n, int lane) {
  float mx = -INFINITY;
  for (int j = lane; j < n; j += 32) mx = fmaxf(mx, in[j]);
  mx = warp_max(mx);
  float se = 0.f;
  for (int j = lane; j < n; j += 32) se += expf(in[j] - mx);
  se = warp_sum(se);
  __syncwarp();
  for (int j = lane; j < n; j += 32) out[j] = expf(in[j] - mx) / se;
  __syncwarp();
}

// the head's forward for row g on one warp: cur holds r's row; returns the buffer holding the C logits.
// acts (nullable): layer l's outputs are stored at acts + off[l] + g * out[l].
__device__ __forceinline__ float* head_rows_fwd(const PredDesc& d, int g, int lane, float* cur, float* nxt, float* acts) {
  int in = d.D0;
  for (int l = 0; l < d.L; ++l) {
    const int out = d.out[l];
    const float* __restrict__ W = d.W[l];
    const float* __restrict__ b = d.b[l];
    const bool relu = (d.relu_mask >> l) & 1;
    for (int j = lane; j < out; j += 32) {
      const float* wr = W + (size_t)j * in;
      float acc = 0.f;
      for (int k = 0; k < in; ++k) acc = fmaf(cur[k], __ldg(wr + k), acc);
      acc += b ? __ldg(b + j) : 0.f;
      if (relu) acc = fmaxf(acc, 0.f);
      nxt[j] = acc;
      if (acts) acts[d.off[l] + (int64_t)g * out + j] = acc;
    }
    __syncwarp();
    float* t = cur; cur = nxt; nxt = t;
    in = out;
  }
  return cur;
}

// mode bits of k_pred_fwd
constexpr int PF_SAVE = 1;        // training: store every layer's activations
constexpr int PF_CLASSIFY = 2;    // evaluation: pred (and hit) per row

// per row: logits, the row loss ce[g] (with labels), pred[g] / hit[g] (PF_CLASSIFY)
__global__ void __launch_bounds__(PRED_THREADS)
k_pred_fwd(PredDesc d, const float* __restrict__ r, const int64_t* __restrict__ y, int G, int mode,
           float* __restrict__ acts, float* __restrict__ logits_out, float* __restrict__ ce, int64_t* __restrict__ pred,
           int* __restrict__ hit, int* status) {
  pdl_wait();
  pdl_launch_dependents();
  __shared__ float sm[PRED_WARPS][3][PRED_W];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int bad = 0;
  for (int g = blockIdx.x * PRED_WARPS + w; g < G; g += gridDim.x * PRED_WARPS) {
    float* cur = sm[w][0];
    for (int k = lane; k < d.D0; k += 32) cur[k] = r[(size_t)g * d.D0 + k];
    __syncwarp();
    const float* z = head_rows_fwd(d, g, lane, cur, sm[w][1], (mode & PF_SAVE) ? acts : nullptr);
    const int C = d.C;
    if (logits_out)
      for (int j = lane; j < C; j += 32) logits_out[(size_t)g * C + j] = z[j];
    if (mode & PF_CLASSIFY) {                      // first-index argmax of the logits
      float bv = -INFINITY;
      int bj = C;
      for (int j = lane; j < C; j += 32)
        if (z[j] > bv || bj == C) { bv = z[j]; bj = j; }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
        if (oj < C && (bj == C || ov > bv || (ov == bv && oj < bj))) { bv = ov; bj = oj; }
      }
      if (lane == 0) {
        pred[g] = bj;
        if (y) hit[g] = (int64_t)bj == y[g];
      }
    }
    if (y) {
      const int yc = clamp_label(y[g], C, bad);
      const float* q = z;
      if (d.softmax_first) {
        float* p = sm[w][2];
        row_softmax(z, p, C, lane);
        q = p;
      }
      float mx = -INFINITY;
      for (int j = lane; j < C; j += 32) mx = fmaxf(mx, q[j]);
      mx = warp_max(mx);
      float se = 0.f;
      for (int j = lane; j < C; j += 32) se += expf(q[j] - mx);
      se = warp_sum(se);
      if (lane == 0) ce[g] = (mx + logf(se)) - q[yc];
    }
    __syncwarp();
  }
  if (bad && status) atomicOr(status, bad);
}

// per row: the deltas of every layer (to the workspace) and dr
__global__ void __launch_bounds__(PRED_THREADS)
k_pred_bwd(PredDesc d, const float* __restrict__ r, const int64_t* __restrict__ y, int G,
           const float* __restrict__ acts, const float* __restrict__ dloss, float* __restrict__ deltas,
           float* __restrict__ dr) {
  pdl_wait();
  pdl_launch_dependents();
  __shared__ float sm[PRED_WARPS][3][PRED_W];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const float dl = dloss ? *dloss : 1.f;
  const int C = d.C;
  int bad = 0;
  for (int g = blockIdx.x * PRED_WARPS + w; g < G; g += gridDim.x * PRED_WARPS) {
    float* z = sm[w][0];                           // logits, then softmax(q)
    float* p = sm[w][1];                           // softmax_first: p = softmax(z)
    float* dq = sm[w][2];
    const float* zsrc = d.L ? acts + d.off[d.L - 1] + (int64_t)g * C : r + (size_t)g * d.D0;
    for (int j = lane; j < C; j += 32) z[j] = zsrc[j];
    __syncwarp();
    const int yc = clamp_label(y[g], C, bad);
    if (d.softmax_first) row_softmax(z, p, C, lane);
    row_softmax(d.softmax_first ? p : z, z, C, lane);                   // z <- softmax(q)
    for (int j = lane; j < C; j += 32) dq[j] = (z[j] - (j == yc ? 1.f : 0.f)) / (float)G * dl;
    __syncwarp();
    float* dcur = dq;                              // d(loss) / d(logits)
    if (d.softmax_first) {                         // through the softmax: p * (dp - <p, dp>)
      float t = 0.f;
      for (int j = lane; j < C; j += 32) t += p[j] * dq[j];
      t = warp_sum(t);
      for (int j = lane; j < C; j += 32) z[j] = p[j] * (dq[j] - t);
      __syncwarp();
      dcur = z;
    }
    // layer l: delta_l = dcur * relu'(a_l) -> workspace; d(a_(l-1)) = delta_l . W_l, one fmaf chain per input column
    for (int l = d.L - 1; l >= 0; --l) {
      const int out = d.out[l], in = l ? d.out[l - 1] : d.D0;
      const bool relu = (d.relu_mask >> l) & 1;
      const float* a = acts + d.off[l] + (int64_t)g * out;
      float* dst = deltas + d.off[l] + (int64_t)g * out;
      for (int j = lane; j < out; j += 32) {
        const float v = relu && !(a[j] > 0.f) ? 0.f : dcur[j];
        dcur[j] = v;
        dst[j] = v;
      }
      __syncwarp();
      float* dn = dcur == sm[w][2] ? sm[w][1] : sm[w][2];
      const float* __restrict__ W = d.W[l];
      for (int k = lane; k < in; k += 32) {
        float t = 0.f;
        for (int j = 0; j < out; ++j) t = fmaf(dcur[j], __ldg(W + (size_t)j * in + k), t);
        dn[k] = t;
      }
      __syncwarp();
      dcur = dn;
    }
    if (dr)
      for (int k = lane; k < d.D0; k += 32) dr[(size_t)g * d.D0 + k] = dcur[k];
    __syncwarp();
  }
  (void)bad;                                       // the forward reported it
}

}  // namespace tsg

using namespace tsg;

#define TSG_TRY(call)                 \
  do {                                \
    int _rc = (call);                 \
    if (_rc != TSG_OK) return _rc;    \
  } while (0)

static bool pred_head_ok(const tsg_pred_head* h) {
  if (!h || h->num_layers < 0 || h->num_layers > TSG_PRED_MAX_LAYERS) return false;
  if (h->in_dim < 1 || h->in_dim > TSG_PRED_MAX_WIDTH) return false;
  for (int64_t l = 0; l < h->num_layers; ++l)
    if (h->out_dim[l] < 1 || h->out_dim[l] > TSG_PRED_MAX_WIDTH) return false;
  return true;
}

static bool pred_weights_ok(const tsg_pred_head* h) {
  for (int64_t l = 0; l < h->num_layers; ++l)
    if (!h->weight[l]) return false;
  return true;
}

static bool rows_ok(int64_t G) { return G >= 1 && G < (int64_t)0x7fffffff; }

// activations (= deltas) per row: the sum of the layers' widths
static int64_t pred_width_sum(const tsg_pred_head* h) {
  int64_t s = 0;
  for (int64_t l = 0; l < h->num_layers; ++l) s += h->out_dim[l];
  return s;
}

static PredDesc pred_desc(const tsg_pred_head* h, int64_t G) {
  PredDesc d{};
  d.L = (int)h->num_layers; d.D0 = (int)h->in_dim;
  d.C = d.L ? (int)h->out_dim[d.L - 1] : d.D0;
  d.relu_mask = (int)h->relu_mask; d.softmax_first = h->softmax_first != 0;
  int64_t off = 0;
  for (int l = 0; l < d.L; ++l) {
    d.out[l] = (int)h->out_dim[l]; d.off[l] = off; off += G * h->out_dim[l];
    d.W[l] = h->weight[l]; d.b[l] = h->bias[l];
  }
  return d;
}

struct PredCeWs {
  float *acts, *deltas, *ce;
  void *lin_ws, *cs_ws;
  size_t lin_bytes, cs_bytes, total;
};

static void pred_ce_layout(const tsg_pred_head* h, int64_t G, void* base, PredCeWs* w) {
  *w = PredCeWs{};
  char* b = (char*)base;
  size_t off = 0;
  auto take = [&](size_t bytes) -> void* { void* p = b ? (void*)(b + off) : nullptr; off += align_up(bytes, 256); return p; };
  const int64_t S = pred_width_sum(h);
  w->acts = (float*)take((size_t)(G * S) * 4);
  w->deltas = (float*)take((size_t)(G * S) * 4);
  w->ce = (float*)take((size_t)G * 4);
  for (int64_t l = 0; l < h->num_layers; ++l) {
    const int64_t out = h->out_dim[l], in = l ? h->out_dim[l - 1] : h->in_dim;
    const size_t lb = tsg_linear_bwd_weight_workspace_bytes(out, in), cb = tsg_colsum_workspace_bytes(G, out);
    if (lb > w->lin_bytes) w->lin_bytes = lb;
    if (cb > w->cs_bytes) w->cs_bytes = cb;
  }
  w->lin_ws = take(w->lin_bytes); w->cs_ws = take(w->cs_bytes);
  w->total = off;
}

static int pred_grid(int64_t G) { return grid_for(G, PRED_WARPS, 8); }

extern "C" size_t tsg_pred_ce_workspace_bytes(const tsg_pred_head* h, int64_t G) {
  if (!pred_head_ok(h) || !rows_ok(G)) return 0;
  PredCeWs w;
  pred_ce_layout(h, G, nullptr, &w);
  return w.total;
}

extern "C" int tsg_pred_ce_fwd(const tsg_pred_head* h, const float* r, const int64_t* y, int64_t G, float* loss,
                               float* logits_out, int32_t* status, void* workspace, size_t workspace_bytes, void* stream) {
  TSG_REQUIRE(pred_head_ok(h), "pred_ce_fwd: bad head (0 to %d layers, every width in [1, %d])", TSG_PRED_MAX_LAYERS,
              TSG_PRED_MAX_WIDTH);
  TSG_REQUIRE(rows_ok(G), "pred_ce_fwd: bad row count %lld", (long long)G);
  TSG_REQUIRE(pred_weights_ok(h) && r && y && loss && workspace, "pred_ce_fwd: null pointer");
  PredCeWs w;
  pred_ce_layout(h, G, workspace, &w);
  if (workspace_bytes < w.total) { set_error("pred_ce_fwd: workspace too small (%zu < %zu)", workspace_bytes, w.total); return TSG_EWORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  TSG_LAUNCH_PDL("pred_ce_fwd", k_pred_fwd, pred_grid(G), PRED_THREADS, 0, st, pred_desc(h, G), r, y, (int)G, PF_SAVE,
                 w.acts, logits_out, w.ce, (int64_t*)nullptr, (int*)nullptr, (int*)status);
  TSG_LAUNCH_PDL("pred_ce_fwd(loss)", k_sum_fixed, 1, SUM_THREADS, 0, st, (const float*)w.ce, (const int*)nullptr, (int)G,
                 (float)G, loss, (int64_t*)nullptr);
  return TSG_OK;
}

extern "C" int tsg_pred_ce_bwd(const tsg_pred_head* h, const float* r, const int64_t* y, int64_t G, const float* dloss,
                               float* dr, float* const* dweight, float* const* dbias, void* workspace,
                               size_t workspace_bytes, void* stream) {
  TSG_REQUIRE(pred_head_ok(h), "pred_ce_bwd: bad head (0 to %d layers, every width in [1, %d])", TSG_PRED_MAX_LAYERS,
              TSG_PRED_MAX_WIDTH);
  TSG_REQUIRE(rows_ok(G), "pred_ce_bwd: bad row count %lld", (long long)G);
  TSG_REQUIRE(pred_weights_ok(h) && r && y && workspace, "pred_ce_bwd: null pointer");
  TSG_REQUIRE(h->num_layers == 0 || (dweight && dbias), "pred_ce_bwd: null gradient array");
  for (int64_t l = 0; l < h->num_layers; ++l)
    TSG_REQUIRE(dweight[l] && (dbias[l] == nullptr || h->bias[l]), "pred_ce_bwd: layer %lld: null dweight, or dbias without a bias",
                (long long)l);
  PredCeWs w;
  pred_ce_layout(h, G, workspace, &w);
  if (workspace_bytes < w.total) { set_error("pred_ce_bwd: workspace too small (%zu < %zu)", workspace_bytes, w.total); return TSG_EWORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  const PredDesc d = pred_desc(h, G);
  TSG_LAUNCH_PDL("pred_ce_bwd", k_pred_bwd, pred_grid(G), PRED_THREADS, 0, st, d, r, y, (int)G, (const float*)w.acts, dloss,
                 w.deltas, dr);
  // nn.Linear's [out, in] gradient delta^T . input is K3's X^T . dY with X = the delta, dY = the layer's input
  for (int l = 0; l < d.L; ++l) {
    const int64_t out = d.out[l], in = l ? d.out[l - 1] : d.D0;
    const float* input = l ? w.acts + d.off[l - 1] : r;
    TSG_TRY(tsg_linear_bwd_weight(w.deltas + d.off[l], input, dweight[l], nullptr, G, out, in, w.lin_ws, w.lin_bytes, stream));
    if (dbias[l]) TSG_TRY(tsg_relu_bwd_colsum(w.deltas + d.off[l], nullptr, nullptr, dbias[l], G, out, w.cs_ws, w.cs_bytes, stream));
  }
  return check_launch("pred_ce_bwd");
}

struct PredClassifyWs { float* ce; int* hit; size_t total; };

static void pred_classify_layout(int64_t G, void* base, PredClassifyWs* w) {
  char* b = (char*)base;
  size_t off = 0;
  auto take = [&](size_t bytes) -> void* { void* p = b ? (void*)(b + off) : nullptr; off += align_up(bytes, 256); return p; };
  w->ce = (float*)take((size_t)G * 4);
  w->hit = (int*)take((size_t)G * 4);
  w->total = off;
}

extern "C" size_t tsg_pred_classify_workspace_bytes(const tsg_pred_head* h, int64_t G) {
  if (!pred_head_ok(h) || !rows_ok(G)) return 0;
  PredClassifyWs w;
  pred_classify_layout(G, nullptr, &w);
  return w.total;
}

extern "C" int tsg_pred_classify(const tsg_pred_head* h, const float* r, const int64_t* y, int64_t G, int64_t* pred,
                                 float* logits_out, int64_t* correct, float* ce_sum, int32_t* status, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  TSG_REQUIRE(pred_head_ok(h), "pred_classify: bad head (0 to %d layers, every width in [1, %d])", TSG_PRED_MAX_LAYERS,
              TSG_PRED_MAX_WIDTH);
  TSG_REQUIRE(rows_ok(G), "pred_classify: bad row count %lld", (long long)G);
  TSG_REQUIRE(pred_weights_ok(h) && r && pred && workspace, "pred_classify: null pointer");
  TSG_REQUIRE(y || (!correct && !ce_sum), "pred_classify: correct / ce_sum need the labels y");
  PredClassifyWs w;
  pred_classify_layout(G, workspace, &w);
  if (workspace_bytes < w.total) { set_error("pred_classify: workspace too small (%zu < %zu)", workspace_bytes, w.total); return TSG_EWORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  TSG_LAUNCH_PDL("pred_classify", k_pred_fwd, pred_grid(G), PRED_THREADS, 0, st, pred_desc(h, G), r, y, (int)G, PF_CLASSIFY,
                 (float*)nullptr, logits_out, w.ce, pred, w.hit, (int*)status);
  if (correct || ce_sum)
    TSG_LAUNCH_PDL("pred_classify(totals)", k_sum_fixed, 1, SUM_THREADS, 0, st, (const float*)w.ce, (const int*)w.hit, (int)G,
                   1.0f, ce_sum, correct);
  return TSG_OK;
}
