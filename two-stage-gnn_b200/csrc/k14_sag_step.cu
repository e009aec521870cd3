// K14 -- the whole 2stg SAGPool training step behind ONE C-ABI call.
//
// Round 1 enqueued the encoder from C++ (K10) but the head MLP, the triplet loss and their backward went through
// Python: three autograd Functions for the Linear layers, aten ReLU / dropout / log_softmax, the triplet Function --
// 1.46 ms of host time per 1.69 ms step, the limit of 8-GPU scaling (eight processes share the box's cores and every
// rank waits for the slowest at the all-reduce).  Here the step is
//
//   encoder forward (K10)  ->  head forward (k_head_fwd)  ->  triplet loss (K9)  ->  triplet backward (K9)
//   ->  head backward (k_head_bwd, fixed-order parameter gradients)  ->  encoder backward (K10)
//
// enqueued by tsg_sag_triplet_step_compact without returning to the interpreter; Python keeps the sampler, one
// NCCL all-reduce over the flat gradient buffer and the optimiser.
//
// Head = Code/sag/network.py:48-52: lin1 (2H -> H) / ReLU / dropout(p) / lin2 (H -> H/2) / ReLU / lin3 (H/2 -> C) /
// log_softmax.  One warp per graph, weights in shared memory (rows padded to an odd pitch), sequential dot products.
// Dropout: a caller-provided keep-multiplier matrix (parity tests inject the oracle's) or a counter-based hash of
// (seed, graph, column) -- the reference draws from torch's unseeded-per-step generator, so no mask sequence can be
// "the reference's"; SURVEY A.2 (RNG).
//
// The same head serves the supervised setting of Code/sag/train.py: tsg_sag_nll_step_compact (NLL loss in place of
// K9) and tsg_sag_classify_compact (evaluation: forward-only encoder, head with dropout off, argmax / NLL totals).
#include "common.cuh"

namespace tsg {

constexpr int HEAD_THREADS = 256;
constexpr int HEAD_WARPS = HEAD_THREADS / 32;

struct HeadDims { int G, H, H2, C; };

__device__ __forceinline__ unsigned head_hash(unsigned long long seed, unsigned idx) {
  unsigned long long x = seed + 0x9E3779B97F4A7C15ull * (unsigned long long)(idx + 1u);
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return (unsigned)((x ^ (x >> 31)) >> 32);
}

// shared-memory image of the head parameters: W1 [H][2H+1], b1 [H], W2 [H2][H+1], b2 [H2], W3 [C][H2+1], b3 [C]
__host__ __device__ inline int head_param_floats(int H, int H2, int C) {
  return H * (2 * H + 1) + H + H2 * (H + 1) + H2 + C * (H2 + 1) + C;
}

__device__ void head_load_params(const float* const* hp, float* sm, HeadDims d) {
  const int p1 = 2 * d.H + 1, p2 = d.H + 1, p3 = d.H2 + 1;
  float* W1 = sm; float* b1 = W1 + d.H * p1; float* W2 = b1 + d.H; float* b2 = W2 + d.H2 * p2;
  float* W3 = b2 + d.H2; float* b3 = W3 + d.C * p3;
  for (int i = threadIdx.x; i < d.H * 2 * d.H; i += blockDim.x) W1[(i / (2 * d.H)) * p1 + i % (2 * d.H)] = hp[0][i];
  for (int i = threadIdx.x; i < d.H; i += blockDim.x) b1[i] = hp[1][i];
  for (int i = threadIdx.x; i < d.H2 * d.H; i += blockDim.x) W2[(i / d.H) * p2 + i % d.H] = hp[2][i];
  for (int i = threadIdx.x; i < d.H2; i += blockDim.x) b2[i] = hp[3][i];
  for (int i = threadIdx.x; i < d.C * d.H2; i += blockDim.x) W3[(i / d.H2) * p3 + i % d.H2] = hp[4][i];
  for (int i = threadIdx.x; i < d.C; i += blockDim.x) b3[i] = hp[5][i];
}

struct HeadPtrs { const float* hp[6]; };

// z [G, 2H] -> a1 [G, H] (after ReLU and dropout), m [G, H] (dropout keep multiplier), a2 [G, H2], emb [G, C]
__global__ void __launch_bounds__(HEAD_THREADS)
k_head_fwd(HeadPtrs P, const float* __restrict__ z, HeadDims d, float dropout_p, unsigned long long seed,
           const float* __restrict__ mask_in, float* __restrict__ a1, float* __restrict__ m, float* __restrict__ a2,
           float* __restrict__ emb) {
  pdl_wait();
  pdl_launch_dependents();
  extern __shared__ __align__(16) float hsm[];
  float* prm = hsm;
  float* stage = hsm + head_param_floats(d.H, d.H2, d.C);          // per warp: 2H + H + H2 + C floats
  head_load_params(P.hp, prm, d);
  __syncthreads();
  const int p1 = 2 * d.H + 1, p2 = d.H + 1, p3 = d.H2 + 1;
  const float* W1 = prm; const float* b1 = W1 + d.H * p1; const float* W2 = b1 + d.H; const float* b2 = W2 + d.H2 * p2;
  const float* W3 = b2 + d.H2; const float* b3 = W3 + d.C * p3;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float* sz = stage + (size_t)w * (2 * d.H + d.H + d.H2 + d.C);
  float* s1 = sz + 2 * d.H; float* s2 = s1 + d.H; float* s3 = s2 + d.H2;
  const float scale = dropout_p > 0.f ? 1.0f / (1.0f - dropout_p) : 1.0f;
  for (int g = blockIdx.x * HEAD_WARPS + w; g < d.G; g += gridDim.x * HEAD_WARPS) {
    for (int i = lane; i < 2 * d.H; i += 32) sz[i] = z[(size_t)g * 2 * d.H + i];
    __syncwarp();
    for (int j = lane; j < d.H; j += 32) {                          // lin1 + ReLU + dropout      network.py:48-49
      float acc = 0.f;
      for (int k = 0; k < 2 * d.H; ++k) acc = fmaf(sz[k], W1[j * p1 + k], acc);
      acc = fmaxf(acc + b1[j], 0.f);
      float keep;
      if (mask_in) keep = mask_in[(size_t)g * d.H + j];
      else if (dropout_p > 0.f) keep = (head_hash(seed, (unsigned)(g * d.H + j)) >> 8) * (1.0f / 16777216.0f) >= dropout_p ? scale : 0.f;
      else keep = 1.f;
      acc *= keep;
      s1[j] = acc;
      a1[(size_t)g * d.H + j] = acc; m[(size_t)g * d.H + j] = keep;
    }
    __syncwarp();
    for (int j = lane; j < d.H2; j += 32) {                         // lin2 + ReLU                 network.py:50
      float acc = 0.f;
      for (int k = 0; k < d.H; ++k) acc = fmaf(s1[k], W2[j * p2 + k], acc);
      acc = fmaxf(acc + b2[j], 0.f);
      s2[j] = acc; a2[(size_t)g * d.H2 + j] = acc;
    }
    __syncwarp();
    float mx = -3.4e38f;
    for (int j = lane; j < d.C; j += 32) {                          // lin3                        network.py:51
      float acc = 0.f;
      for (int k = 0; k < d.H2; ++k) acc = fmaf(s2[k], W3[j * p3 + k], acc);
      acc += b3[j];
      s3[j] = acc; mx = fmaxf(mx, acc);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float se = 0.f;
    for (int j = lane; j < d.C; j += 32) se += expf(s3[j] - mx);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
    const float lse = mx + logf(se);
    for (int j = lane; j < d.C; j += 32) emb[(size_t)g * d.C + j] = s3[j] - lse;      // log_softmax
    __syncwarp();
  }
}

// demb [G, C] -> dz [G, 2H]; parameter gradients as ONE partial row per CTA (fixed graph ranges, fixed order inside)
// layout of a partial row / of the packed head gradient: [dW1 H*2H | db1 H | dW2 H2*H | db2 H2 | dW3 C*H2 | db3 C]
__host__ __device__ inline int head_grad_floats(int H, int H2, int C) { return H * 2 * H + H + H2 * H + H2 + C * H2 + C; }

// One graph's deltas on one warp: do = log_softmax backward of demb, da2 = (do W3) * relu', da1 = (da2 W2) * keep * relu',
// dz = da1 W1 (written to global).  s1 / s2 hold the graph's a1 / a2; dO / d2 / d1 receive the deltas (shared memory).
__device__ __forceinline__ void head_delta(const float* W1, const float* W2, const float* W3, HeadDims d, int g, int lane,
                                           const float* s1, const float* s2, const float* __restrict__ m,
                                           const float* __restrict__ emb, const float* __restrict__ demb, float* dO,
                                           float* d2, float* d1, float* __restrict__ dz) {
  const int p1 = 2 * d.H + 1, p2 = d.H + 1, p3 = d.H2 + 1;
  // log_softmax backward: do = demb - softmax * sum(demb)
  float sd = 0.f;
  for (int j = lane; j < d.C; j += 32) sd += demb[(size_t)g * d.C + j];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sd += __shfl_xor_sync(0xffffffffu, sd, o);
  for (int j = lane; j < d.C; j += 32) dO[j] = demb[(size_t)g * d.C + j] - expf(emb[(size_t)g * d.C + j]) * sd;
  __syncwarp();
  for (int k = lane; k < d.H2; k += 32) {                           // da2 = (do W3) * relu'
    float t = 0.f;
    for (int j = 0; j < d.C; ++j) t = fmaf(dO[j], W3[j * p3 + k], t);
    d2[k] = s2[k] > 0.f ? t : 0.f;
  }
  __syncwarp();
  for (int k = lane; k < d.H; k += 32) {                            // da1 = (da2 W2) * keep * relu'
    float t = 0.f;
    for (int j = 0; j < d.H2; ++j) t = fmaf(d2[j], W2[j * p2 + k], t);
    // a1 is stored AFTER dropout: a1 > 0 <=> pre-dropout activation > 0 and kept
    d1[k] = s1[k] > 0.f ? t * m[(size_t)g * d.H + k] : 0.f;
  }
  __syncwarp();
  for (int k = lane; k < 2 * d.H; k += 32) {                        // dz = da1 W1
    float t = 0.f;
    for (int j = 0; j < d.H; ++j) t = fmaf(d1[j], W1[j * p1 + k], t);
    dz[(size_t)g * 2 * d.H + k] = t;
  }
}

__global__ void __launch_bounds__(HEAD_THREADS)
k_head_bwd(HeadPtrs P, const float* __restrict__ z, HeadDims d, const float* __restrict__ a1, const float* __restrict__ m,
           const float* __restrict__ a2, const float* __restrict__ emb, const float* __restrict__ demb,
           float* __restrict__ dz, float* __restrict__ part) {
  pdl_wait();
  pdl_launch_dependents();
  extern __shared__ __align__(16) float hsm[];
  float* prm = hsm;
  const int per = 2 * d.H + d.H + d.H + d.H2 + d.H2 + d.C;         // staged per graph: z, a1, da1, a2, da2, do
  float* stage = hsm + head_param_floats(d.H, d.H2, d.C);          // HEAD_WARPS graphs
  float* acc = stage + (size_t)HEAD_WARPS * per;                   // this CTA's gradient row
  head_load_params(P.hp, prm, d);
  const int NG = head_grad_floats(d.H, d.H2, d.C);
  for (int i = threadIdx.x; i < NG; i += HEAD_THREADS) acc[i] = 0.f;
  __syncthreads();
  const int p1 = 2 * d.H + 1, p2 = d.H + 1;
  const float* W1 = prm; const float* W2 = W1 + d.H * p1 + d.H; const float* W3 = W2 + d.H2 * p2 + d.H2;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float* sz = stage + (size_t)w * per;
  float* s1 = sz + 2 * d.H; float* d1 = s1 + d.H; float* s2 = d1 + d.H; float* d2 = s2 + d.H2; float* dO = d2 + d.H2;
  const int gpc = (d.G + gridDim.x - 1) / gridDim.x;               // contiguous graph range of this CTA
  const int g_begin = blockIdx.x * gpc, g_end = min(d.G, g_begin + gpc);
  for (int g0 = g_begin; g0 < g_end; g0 += HEAD_WARPS) {
    const int g = g0 + w;
    const bool on = g < g_end;
    if (on) {
      for (int i = lane; i < 2 * d.H; i += 32) sz[i] = z[(size_t)g * 2 * d.H + i];
      for (int i = lane; i < d.H; i += 32) s1[i] = a1[(size_t)g * d.H + i];
      for (int i = lane; i < d.H2; i += 32) s2[i] = a2[(size_t)g * d.H2 + i];
      head_delta(W1, W2, W3, d, g, lane, s1, s2, m, emb, demb, dO, d2, d1, dz);
    }
    __syncthreads();
    // every thread owns a fixed set of gradient entries and adds this batch of graphs in graph order
    const int nb = min(HEAD_WARPS, g_end - g0);
    for (int i = threadIdx.x; i < NG; i += HEAD_THREADS) {
      float t = acc[i];
      int o = i;
      if (o < d.H * 2 * d.H) {                                       // dW1[j][k] += da1_pre[j] * z[k]; a1 holds post-dropout a1
        const int j = o / (2 * d.H), k = o % (2 * d.H);
        for (int b = 0; b < nb; ++b) { const float* s = stage + (size_t)b * per; t = fmaf(s[3 * d.H + j], s[k], t); }
      } else if ((o -= d.H * 2 * d.H) < d.H) {
        for (int b = 0; b < nb; ++b) t += (stage + (size_t)b * per)[3 * d.H + o];
      } else if ((o -= d.H) < d.H2 * d.H) {                          // dW2[j][k] += da2[j] * a1[k]
        const int j = o / d.H, k = o % d.H;
        for (int b = 0; b < nb; ++b) { const float* s = stage + (size_t)b * per; t = fmaf(s[4 * d.H + d.H2 + j], s[2 * d.H + k], t); }
      } else if ((o -= d.H2 * d.H) < d.H2) {
        for (int b = 0; b < nb; ++b) t += (stage + (size_t)b * per)[4 * d.H + d.H2 + o];
      } else if ((o -= d.H2) < d.C * d.H2) {                         // dW3[j][k] += do[j] * a2[k]
        const int j = o / d.H2, k = o % d.H2;
        for (int b = 0; b < nb; ++b) { const float* s = stage + (size_t)b * per; t = fmaf(s[4 * d.H + 2 * d.H2 + j], s[4 * d.H + k], t); }
      } else {
        o -= d.C * d.H2;
        for (int b = 0; b < nb; ++b) t += (stage + (size_t)b * per)[4 * d.H + 2 * d.H2 + o];
      }
      acc[i] = t;
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < NG; i += HEAD_THREADS) part[(size_t)blockIdx.x * NG + i] = acc[i];
}

// the packed head gradient row -> the six parameter gradient tensors
__global__ void __launch_bounds__(256)
k_head_unpack(const float* __restrict__ packed, float* g0, float* g1, float* g2, float* g3, float* g4, float* g5,
              int n0, int n1, int n2, int n3, int n4, int n5) {
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  int o = i;
  if (o < n0) { g0[o] = packed[i]; return; }
  if ((o -= n0) < n1) { g1[o] = packed[i]; return; }
  if ((o -= n1) < n2) { g2[o] = packed[i]; return; }
  if ((o -= n2) < n3) { g3[o] = packed[i]; return; }
  if ((o -= n3) < n4) { g4[o] = packed[i]; return; }
  if ((o -= n4) < n5) { g5[o] = packed[i]; return; }
}

// Wide heads (k_head_bwd's parameters + staging + one gradient row exceed shared memory; from H ~ 96 on): the same
// per-graph deltas, written out as do [G, C], da2 [G, H2], da1 [G, H] (and dz), so that the parameter gradients are
// K3's fixed-order reductions over graphs (tsg_linear_bwd_weight / tsg_relu_bwd_colsum) instead of a per-CTA row.
__global__ void __launch_bounds__(HEAD_THREADS)
k_head_delta(HeadPtrs P, HeadDims d, const float* __restrict__ a1, const float* __restrict__ m,
             const float* __restrict__ a2, const float* __restrict__ emb, const float* __restrict__ demb,
             float* __restrict__ dz, float* __restrict__ dO_out, float* __restrict__ da2_out, float* __restrict__ da1_out) {
  pdl_wait();
  pdl_launch_dependents();
  extern __shared__ __align__(16) float hsm[];
  const int per = 2 * d.H + 2 * d.H2 + d.C;                       // staged per warp: a1, da1, a2, da2, do
  float* stage = hsm + head_param_floats(d.H, d.H2, d.C);
  head_load_params(P.hp, hsm, d);
  __syncthreads();
  const int p1 = 2 * d.H + 1, p2 = d.H + 1;
  const float* W1 = hsm; const float* W2 = W1 + d.H * p1 + d.H; const float* W3 = W2 + d.H2 * p2 + d.H2;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float* s1 = stage + (size_t)w * per; float* d1 = s1 + d.H; float* s2 = d1 + d.H; float* d2 = s2 + d.H2; float* dO = d2 + d.H2;
  for (int g = blockIdx.x * HEAD_WARPS + w; g < d.G; g += gridDim.x * HEAD_WARPS) {
    for (int i = lane; i < d.H; i += 32) s1[i] = a1[(size_t)g * d.H + i];
    for (int i = lane; i < d.H2; i += 32) s2[i] = a2[(size_t)g * d.H2 + i];
    head_delta(W1, W2, W3, d, g, lane, s1, s2, m, emb, demb, dO, d2, d1, dz);
    for (int j = lane; j < d.C; j += 32) dO_out[(size_t)g * d.C + j] = dO[j];
    for (int k = lane; k < d.H2; k += 32) da2_out[(size_t)g * d.H2 + k] = d2[k];
    for (int k = lane; k < d.H; k += 32) da1_out[(size_t)g * d.H + k] = d1[k];
    __syncwarp();
  }
}

constexpr int TSG_LABEL_RANGE = TSG_SAG_LABEL_RANGE;     // status bit: a graph label outside [0, C) (clamped for the read)

__device__ __forceinline__ int64_t clamp_label(int64_t y, int C) { return y < 0 ? 0 : (y >= C ? C - 1 : y); }

// F.nll_loss(emb, y) (mean) backward as autograd builds it: demb = -(1/G) onehot(y); nll[g] = -emb[g, y_g]
__global__ void k_nll_demb(const float* __restrict__ emb, const int64_t* __restrict__ y, int G, int C,
                           float* __restrict__ demb, float* __restrict__ nll, int* status) {
  pdl_wait();
  pdl_launch_dependents();
  const float grad = -(1.0f / (float)G);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < (int64_t)G * C; i += (int64_t)gridDim.x * blockDim.x) {
    const int g = (int)(i / C), j = (int)(i % C);
    const int64_t yc = clamp_label(y[g], C);
    if (j == 0 && yc != y[g]) atomicOr(status, TSG_LABEL_RANGE);
    demb[i] = j == yc ? grad : 0.f;
    if (j == yc) nll[g] = -emb[i];
  }
}

// evaluation rows: pred[g] = argmax_j emb[g, j] (first index on ties, as out.max(dim=1)[1]); with labels
// nll[g] = -emb[g, y_g] and hit[g] = (pred == y_g)
__global__ void k_classify_rows(const float* __restrict__ emb, const int64_t* __restrict__ y, int G, int C,
                                int64_t* __restrict__ pred, float* __restrict__ nll, int* __restrict__ hit, int* status) {
  for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < G; g += gridDim.x * blockDim.x) {
    const float* r = emb + (size_t)g * C;
    int best = 0;
    float bv = r[0];
    for (int j = 1; j < C; ++j)
      if (r[j] > bv) { bv = r[j]; best = j; }
    pred[g] = best;
    if (y) {
      const int64_t yc = clamp_label(y[g], C);
      if (yc != y[g]) atomicOr(status, TSG_LABEL_RANGE);
      nll[g] = -r[yc];
      hit[g] = (int64_t)best == y[g];
    }
  }
}

static int head_ctas(int G) {
  // one batch of HEAD_WARPS graphs per CTA up to two CTAs per SM (ncu, first cut: 110 CTAs of 4 batches = 12 % warps
  // active, 55 us for 3,504 graphs -- the kernel is latency bound, so it wants every SM busy)
  int c = (G + HEAD_WARPS - 1) / HEAD_WARPS;
  if (c > 2 * TSG_NUM_SMS) c = 2 * TSG_NUM_SMS;
  return c < 1 ? 1 : c;
}

}  // namespace tsg

using namespace tsg;

#define TSG_TRY(call)                 \
  do {                                \
    int _rc = (call);                 \
    if (_rc != TSG_OK) return _rc;    \
  } while (0)

constexpr size_t HEAD_SMEM = 200 * 1024;
static size_t head_fwd_smem(int H, int H2, int C) { return ((size_t)head_param_floats(H, H2, C) + (size_t)HEAD_WARPS * (3 * H + H2 + C)) * 4; }
static size_t head_bwd_smem(int H, int H2, int C) {
  return ((size_t)head_param_floats(H, H2, C) + (size_t)HEAD_WARPS * (4 * H + 2 * H2 + C) + head_grad_floats(H, H2, C)) * 4;
}
static size_t head_delta_smem(int H, int H2, int C) { return ((size_t)head_param_floats(H, H2, C) + (size_t)HEAD_WARPS * (2 * H + 2 * H2 + C)) * 4; }

// k_head_bwd does not fit: the head backward runs as k_head_delta + K3's reductions.  Every shape k_head_bwd takes keeps it.
static bool head_wide(int H, int H2, int C) { return head_bwd_smem(H, H2, C) > HEAD_SMEM; }

// the head of any loss: even hidden width, a forward that fits shared memory, and a backward that fits one of the two ways
// (the wide way also within tsg_linear_bwd_weight's in_feat <= 256 for every layer's output width)
static bool head_shape_ok(const tsg_sag_shape* sh, const tsg_sag_head* hd) {
  if (!sh || !hd || hd->num_classes <= 0 || sh->hidden < 2 || sh->hidden % 2) return false;
  if (!(hd->dropout_p >= 0.f && hd->dropout_p < 1.f)) return false;
  const int H = (int)sh->hidden, H2 = H / 2, C = (int)hd->num_classes;
  if (head_fwd_smem(H, H2, C) > HEAD_SMEM) return false;
  return !head_wide(H, H2, C) || (head_delta_smem(H, H2, C) <= HEAD_SMEM && H <= 256 && C <= 256);
}

static bool head_ok(const tsg_sag_shape* sh, const tsg_sag_head* hd) { return head_shape_ok(sh, hd) && hd->num_triplets > 0; }

enum StepLoss { LOSS_TRIPLET, LOSS_NLL };

struct StepWs {
  float *z, *a1, *m, *a2, *emb, *demb, *dz, *dp, *dn, *part, *packed, *one;
  void* trip_ws; size_t trip_bytes;
  float *dO, *da2, *da1;                         // wide head: per-graph deltas
  void *lin_ws, *cs_ws; size_t lin_bytes, cs_bytes;
  float* nll;                                    // NLL: -emb[g, y_g]
  size_t total;
};

static void step_layout(const tsg_sag_shape* sh, const tsg_sag_head* hd, StepLoss loss, void* base, StepWs* w) {
  *w = StepWs{};
  char* b = (char*)base;
  size_t off = 0;
  auto take = [&](size_t bytes) -> void* { void* p = b ? (void*)(b + off) : nullptr; off += align_up(bytes, 256); return p; };
  const int64_t G = sh->num_graphs, H = sh->hidden, H2 = H / 2, C = hd->num_classes, T = hd->num_triplets;
  w->z = (float*)take(G * 2 * H * 4); w->a1 = (float*)take(G * H * 4); w->m = (float*)take(G * H * 4);
  w->a2 = (float*)take(G * H2 * 4); w->emb = (float*)take(G * C * 4); w->demb = (float*)take(G * C * 4);
  w->dz = (float*)take(G * 2 * H * 4);
  if (loss == LOSS_TRIPLET) { w->dp = (float*)take(T * 4); w->dn = (float*)take(T * 4); }
  if (!head_wide((int)H, (int)H2, (int)C)) {
    const size_t NG = head_grad_floats((int)H, (int)H2, (int)C);
    w->part = (float*)take((size_t)head_ctas((int)G) * NG * 4); w->packed = (float*)take(NG * 4);
  } else {
    w->dO = (float*)take(G * C * 4); w->da2 = (float*)take(G * H2 * 4); w->da1 = (float*)take(G * H * 4);
    const int64_t lin[3][2] = {{H, 2 * H}, {H2, H}, {C, H2}};
    for (const auto& k : lin) {
      const size_t lb = tsg_linear_bwd_weight_workspace_bytes(k[0], k[1]), cb = tsg_colsum_workspace_bytes(G, k[0]);
      if (lb > w->lin_bytes) w->lin_bytes = lb;
      if (cb > w->cs_bytes) w->cs_bytes = cb;
    }
    w->lin_ws = take(w->lin_bytes); w->cs_ws = take(w->cs_bytes);
  }
  w->one = (float*)take(256);
  if (loss == LOSS_TRIPLET) {
    w->trip_bytes = tsg_triplet_workspace_bytes(T, G, C);
    w->trip_ws = take(w->trip_bytes);
  } else {
    w->nll = (float*)take(G * 4);
  }
  w->total = off;
}

extern "C" size_t tsg_sag_triplet_step_workspace_bytes(const tsg_sag_shape* sh, const tsg_sag_head* hd) {
  if (!head_ok(sh, hd)) return 0;
  StepWs w;
  step_layout(sh, hd, LOSS_TRIPLET, nullptr, &w);
  return w.total;
}

static void head_attr_once() {
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(k_head_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, HEAD_SMEM);
    cudaFuncSetAttribute(k_head_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, HEAD_SMEM);
    cudaFuncSetAttribute(k_head_delta, cudaFuncAttributeMaxDynamicSharedMemorySize, HEAD_SMEM);
    attr = true;
  }
}

static HeadPtrs head_ptrs(const float* const* params) {
  HeadPtrs P;
  for (int i = 0; i < 6; ++i) P.hp[i] = params[12 + i];
  return P;
}

// head forward: z [G, 2H] -> a1, m, a2 and emb [G, C]
static int head_fwd(const tsg_sag_shape* sh, const tsg_sag_head* hd, const float* const* params, float dropout_p,
                    const float* dropout_mask, const float* z, float* a1, float* m, float* a2, float* emb, cudaStream_t st) {
  const int H = (int)sh->hidden, H2 = H / 2, C = (int)hd->num_classes, G = (int)sh->num_graphs;
  head_attr_once();
  return launch_pdl("sag_step(head fwd)", k_head_fwd, grid_for(G, HEAD_WARPS, 2), HEAD_THREADS, head_fwd_smem(H, H2, C), st,
                    head_ptrs(params), z, HeadDims{G, H, H2, C}, dropout_p, (unsigned long long)hd->seed, dropout_mask, a1, m, a2, emb);
}

// encoder forward (K10) + head forward -> emb [G, C]
static int step_fwd(const tsg_sag_shape* sh, const tsg_sag_head* hd, const int32_t* label, const int32_t* local_row,
                    const int32_t* local_col, const int64_t* edge_ptr, const int64_t* level_ptr, const float* const* params,
                    const float* dropout_mask, float* emb, const StepWs& w, void* arena, size_t arena_bytes, void* stream) {
  TSG_TRY(tsg_sag_encoder_fwd_compact(sh, label, local_row, local_col, edge_ptr, level_ptr, params, w.z, arena, arena_bytes, stream));
  return head_fwd(sh, hd, params, hd->dropout_p, dropout_mask, w.z, w.a1, w.m, w.a2, emb, (cudaStream_t)stream);
}

// head backward (dz + fixed-order parameter gradients) + encoder backward (K10), from d(loss)/d(emb)
static int step_bwd(const tsg_sag_shape* sh, const tsg_sag_head* hd, const int32_t* label, const int64_t* level_ptr,
                    const float* const* params, const float* emb, const float* demb, float* const* grads, const StepWs& w,
                    void* arena, size_t arena_bytes, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int H = (int)sh->hidden, H2 = H / 2, C = (int)hd->num_classes, G = (int)sh->num_graphs;
  HeadDims d{G, H, H2, C};
  const HeadPtrs P = head_ptrs(params);
  head_attr_once();
  if (head_wide(H, H2, C)) {
    TSG_LAUNCH_PDL("sag_step(head delta)", k_head_delta, grid_for(G, HEAD_WARPS, 1), HEAD_THREADS, head_delta_smem(H, H2, C), st,
                   P, d, (const float*)w.a1, (const float*)w.m, (const float*)w.a2, emb, demb, w.dz, w.dO, w.da2, w.da1);
    // nn.Linear's [out, in] gradient delta^T . input is K3's X^T . dY with X = the delta, dY = the layer's input
    const float* delta[3] = {w.da1, w.da2, w.dO};
    const float* input[3] = {w.z, w.a1, w.a2};
    const int out[3] = {H, H2, C}, in[3] = {2 * H, H, H2};
    for (int l = 0; l < 3; ++l) {
      TSG_TRY(tsg_linear_bwd_weight(delta[l], input[l], grads[12 + 2 * l], nullptr, G, out[l], in[l], w.lin_ws, w.lin_bytes, stream));
      TSG_TRY(tsg_relu_bwd_colsum(delta[l], nullptr, nullptr, grads[13 + 2 * l], G, out[l], w.cs_ws, w.cs_bytes, stream));
    }
  } else {
    const int ctas = head_ctas(G);
    const int NG = head_grad_floats(H, H2, C);
    TSG_LAUNCH_PDL("sag_step(head bwd)", k_head_bwd, ctas, HEAD_THREADS, head_bwd_smem(H, H2, C), st, P, (const float*)w.z, d,
                   (const float*)w.a1, (const float*)w.m, (const float*)w.a2, emb, demb, w.dz, w.part);
    TSG_TRY(launch_partial_sum_final(w.part, w.packed, NG, nullptr, ctas, NG, st));
    TSG_LAUNCH_PDL("sag_step(head grads)", k_head_unpack, (NG + 255) / 256, 256, 0, st, (const float*)w.packed, grads[12], grads[13],
                   grads[14], grads[15], grads[16], grads[17], H * 2 * H, H, H2 * H, H2, C * H2, C);
  }
  return tsg_sag_encoder_bwd_compact(sh, label, level_ptr, params, w.dz, grads, arena, arena_bytes, stream);
}

extern "C" int tsg_sag_triplet_step_compact(const tsg_sag_shape* sh, const tsg_sag_head* hd, const int32_t* label,
                                            const int32_t* local_row, const int32_t* local_col, const int64_t* edge_ptr,
                                            const int64_t* level_ptr, const float* const* params, const int64_t* triplets,
                                            const float* dropout_mask, float* const* grads, float* loss, float* emb_out,
                                            void* arena, size_t arena_bytes, void* workspace, size_t workspace_bytes,
                                            void* stream) {
  TSG_REQUIRE(head_ok(sh, hd), "sag_triplet_step: bad head / shape (hidden must be even, head must fit shared memory)");
  TSG_REQUIRE(params && grads && triplets && loss && workspace, "sag_triplet_step: null pointer");
  StepWs w;
  step_layout(sh, hd, LOSS_TRIPLET, workspace, &w);
  if (workspace_bytes < w.total) { set_error("sag_triplet_step: workspace too small (%zu < %zu)", workspace_bytes, w.total); return TSG_EWORKSPACE; }
  const int C = (int)hd->num_classes, G = (int)sh->num_graphs;
  const int64_t T = hd->num_triplets;
  float* emb = emb_out ? emb_out : w.emb;
  TSG_TRY(step_fwd(sh, hd, label, local_row, local_col, edge_ptr, level_ptr, params, dropout_mask, emb, w, arena, arena_bytes, stream));
  // triplet loss forward + backward (K9), d(loss) = 1
  TSG_TRY(triplet_fwd(emb, triplets, T, G, C, hd->margin, hd->eps, w.dp, w.dn, loss, w.one, w.trip_ws, w.trip_bytes, stream));
  TSG_TRY(tsg_triplet_bwd(emb, triplets, T, G, C, hd->margin, hd->eps, w.dp, w.dn, w.one, w.demb, w.trip_ws, w.trip_bytes, stream));
  return step_bwd(sh, hd, label, level_ptr, params, emb, w.demb, grads, w, arena, arena_bytes, stream);
}

/* The two halves of the step for losses evaluated OUTSIDE the call (the all-gather formulation: embeddings of every rank
 * are gathered, the global triplet loss is evaluated on the gathered matrix, this rank's slice of its gradient comes
 * back).  Same arena / workspace in both calls; num_triplets of `head` only sizes the workspace (>= 1). */
extern "C" int tsg_sag_step_fwd_compact(const tsg_sag_shape* sh, const tsg_sag_head* hd, const int32_t* label,
                                        const int32_t* local_row, const int32_t* local_col, const int64_t* edge_ptr,
                                        const int64_t* level_ptr, const float* const* params, const float* dropout_mask,
                                        float* emb, void* arena, size_t arena_bytes, void* workspace, size_t workspace_bytes,
                                        void* stream) {
  TSG_REQUIRE(head_ok(sh, hd), "sag_step_fwd: bad head / shape");
  TSG_REQUIRE(params && emb && workspace, "sag_step_fwd: null pointer");
  StepWs w;
  step_layout(sh, hd, LOSS_TRIPLET, workspace, &w);
  if (workspace_bytes < w.total) { set_error("sag_step_fwd: workspace too small"); return TSG_EWORKSPACE; }
  return step_fwd(sh, hd, label, local_row, local_col, edge_ptr, level_ptr, params, dropout_mask, emb, w, arena, arena_bytes, stream);
}

extern "C" int tsg_sag_step_bwd_compact(const tsg_sag_shape* sh, const tsg_sag_head* hd, const int32_t* label,
                                        const int64_t* level_ptr, const float* const* params, const float* emb,
                                        const float* demb, float* const* grads, void* arena, size_t arena_bytes,
                                        void* workspace, size_t workspace_bytes, void* stream) {
  TSG_REQUIRE(head_ok(sh, hd), "sag_step_bwd: bad head / shape");
  TSG_REQUIRE(params && emb && demb && grads && workspace, "sag_step_bwd: null pointer");
  StepWs w;
  step_layout(sh, hd, LOSS_TRIPLET, workspace, &w);
  if (workspace_bytes < w.total) { set_error("sag_step_bwd: workspace too small"); return TSG_EWORKSPACE; }
  return step_bwd(sh, hd, label, level_ptr, params, emb, demb, grads, w, arena, arena_bytes, stream);
}

// where the label check ORs TSG_LABEL_RANGE: the caller's persistent word, else the arena's (zeroed by every forward)
static int* step_status(const tsg_sag_shape* sh, void* arena) {
  if (sh->status) return sh->status;
  size_t off = 0, bytes = 0;
  tsg_sag_arena_locate(sh, 0, TSG_SAG_STATUS, &off, &bytes);
  return (int*)((char*)arena + off);
}

/* Supervised step (the "original" setting, Code/sag/train.py:194): forward, F.nll_loss(emb, y) and its backward.
 * demb = -(1/G) onehot(y) is what autograd hands tsg_sag_step_bwd_compact, so the gradients are those of the halves
 * with ATen's nll_loss in between, bit for bit; the loss is the same mean summed in a fixed order. */
extern "C" size_t tsg_sag_nll_step_workspace_bytes(const tsg_sag_shape* sh, const tsg_sag_head* hd) {
  if (!head_shape_ok(sh, hd)) return 0;
  StepWs w;
  step_layout(sh, hd, LOSS_NLL, nullptr, &w);
  return w.total;
}

extern "C" int tsg_sag_nll_step_compact(const tsg_sag_shape* sh, const tsg_sag_head* hd, const int32_t* label,
                                        const int32_t* local_row, const int32_t* local_col, const int64_t* edge_ptr,
                                        const int64_t* level_ptr, const float* const* params, const int64_t* y,
                                        const float* dropout_mask, float* const* grads, float* loss, float* emb_out,
                                        void* arena, size_t arena_bytes, void* workspace, size_t workspace_bytes,
                                        void* stream) {
  TSG_REQUIRE(head_shape_ok(sh, hd), "sag_nll_step: bad head / shape (hidden must be even, head must fit shared memory)");
  TSG_REQUIRE(params && grads && y && loss && arena && workspace, "sag_nll_step: null pointer");
  StepWs w;
  step_layout(sh, hd, LOSS_NLL, workspace, &w);
  if (workspace_bytes < w.total) { set_error("sag_nll_step: workspace too small (%zu < %zu)", workspace_bytes, w.total); return TSG_EWORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  const int C = (int)hd->num_classes, G = (int)sh->num_graphs;
  float* emb = emb_out ? emb_out : w.emb;
  TSG_TRY(step_fwd(sh, hd, label, local_row, local_col, edge_ptr, level_ptr, params, dropout_mask, emb, w, arena, arena_bytes, stream));
  TSG_LAUNCH_PDL("sag_nll_step(demb)", k_nll_demb, grid_for((int64_t)G * C, 256, 8), 256, 0, st, (const float*)emb, y, G, C, w.demb,
                 w.nll, step_status(sh, arena));
  TSG_LAUNCH_PDL("sag_nll_step(loss)", k_sum_fixed, 1, SUM_THREADS, 0, st, (const float*)w.nll, (const int*)nullptr, G, (float)G, loss,
                 (int64_t*)nullptr);
  return step_bwd(sh, hd, label, level_ptr, params, emb, w.demb, grads, w, arena, arena_bytes, stream);
}

/* Evaluation (Code/sag/train.py:19-29 `test()`): forward-only encoder (K13 where the shape allows, else K10), the head
 * with dropout off, pred = argmax of the log-probabilities, and with labels the per-graph NLL and hit, summed in a fixed
 * order into *nll_sum and *correct. */
struct ClassifyWs { float *z, *a1, *m, *a2, *emb, *nll; int* hit; size_t total; };

static void classify_layout(const tsg_sag_shape* sh, const tsg_sag_head* hd, void* base, ClassifyWs* w) {
  char* b = (char*)base;
  size_t off = 0;
  auto take = [&](size_t bytes) -> void* { void* p = b ? (void*)(b + off) : nullptr; off += align_up(bytes, 256); return p; };
  const int64_t G = sh->num_graphs, H = sh->hidden, H2 = H / 2, C = hd->num_classes;
  w->z = (float*)take(G * 2 * H * 4); w->a1 = (float*)take(G * H * 4); w->m = (float*)take(G * H * 4);
  w->a2 = (float*)take(G * H2 * 4); w->emb = (float*)take(G * C * 4); w->nll = (float*)take(G * 4);
  w->hit = (int*)take(G * 4);
  w->total = off;
}

extern "C" size_t tsg_sag_classify_workspace_bytes(const tsg_sag_shape* sh, const tsg_sag_head* hd) {
  if (!head_shape_ok(sh, hd)) return 0;
  ClassifyWs w;
  classify_layout(sh, hd, nullptr, &w);
  return w.total;
}

extern "C" int tsg_sag_classify_compact(const tsg_sag_shape* sh, const tsg_sag_head* hd, const int32_t* label,
                                        const int32_t* local_row, const int32_t* local_col, const int64_t* edge_ptr,
                                        const int64_t* level_ptr, const float* const* params, const int64_t* y,
                                        int64_t* pred, float* logp_out, int64_t* correct, float* nll_sum, void* arena,
                                        size_t arena_bytes, void* workspace, size_t workspace_bytes, void* stream) {
  TSG_REQUIRE(head_shape_ok(sh, hd), "sag_classify: bad head / shape (hidden must be even, head must fit shared memory)");
  TSG_REQUIRE(params && pred && arena && workspace, "sag_classify: null pointer");
  TSG_REQUIRE(y || (!correct && !nll_sum), "sag_classify: correct / nll_sum need the labels y");
  ClassifyWs w;
  classify_layout(sh, hd, workspace, &w);
  if (workspace_bytes < w.total) { set_error("sag_classify: workspace too small (%zu < %zu)", workspace_bytes, w.total); return TSG_EWORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  const int C = (int)hd->num_classes, G = (int)sh->num_graphs;
  float* emb = logp_out ? logp_out : w.emb;
  TSG_TRY(tsg_sag_encoder_embed_compact(sh, label, local_row, local_col, edge_ptr, level_ptr, params, w.z, arena, arena_bytes, stream));
  TSG_TRY(head_fwd(sh, hd, params, 0.f, nullptr, w.z, w.a1, w.m, w.a2, emb, st));
  k_classify_rows<<<grid_for(G, 256), 256, 0, st>>>(emb, y, G, C, pred, w.nll, w.hit, step_status(sh, arena));
  if (correct || nll_sum) k_sum_fixed<<<1, SUM_THREADS, 0, st>>>(w.nll, w.hit, G, 1.0f, nll_sum, correct);
  return check_launch("sag_classify");
}
