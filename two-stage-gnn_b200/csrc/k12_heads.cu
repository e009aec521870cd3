// K12 -- stage-2 evaluation heads on graph embeddings (SURVEY 8f n4).
//
// (a) tsg_knn_classify / tsg_knn_predict: the k-nearest-neighbour classifier of `evaluate`
//     (Code/sage+gat+diffpool/train_triplet.py:80-85: sklearn KNeighborsClassifier(n_neighbors=3).fit(train)
//     .predict(val); Euclidean metric, uniform weights).  Warp per query: every lane scans a strided slice of
//     the train rows keeping its k best (distance, index) pairs in shared memory, the lanes' lists are merged by k
//     warp-wide arg-min rounds, the k winners vote into a per-warp shared-memory histogram of C classes; distance
//     ties -> lower train index, vote ties -> lower class id (the rule of scipy.stats.mode that sklearn's predict
//     applies).  With query labels, the correct count is an integer sum (shared, then one global atomic per CTA).
// (b) tsg_mlp1_train: the stage-2 classifier of `evaluate_mlp` (train_triplet.py:148-165): an MLP
//     in -> 64 -> 32 -> 2 with LeakyReLU(0.01), trained with Adam(lr 1e-3) on ONE embedding per step, in order --
//     inherently sequential, ~30 tiny kernels per sample when driven from Python.  Here ONE CTA keeps the
//     weights and both Adam moments in shared memory and runs all N steps (forward, cross-entropy, backward,
//     Adam) back to back; the weight gradients are outer products formed inside the update.
//     Arithmetic: fp32, torch's Adam formulas (bias-corrected step size, denom = sqrt(v)/sqrt(bc2) + eps).
// (c) tsg_mlp1_predict: that MLP's forward over many rows, warp per row, weights in shared memory.  Every unit is
//     the same fmaf chain (mlp1_unit) the trainer's forward runs, so its logits equal the trainer's bit for bit.
//
// Labels outside [0, C) are read clamped and OR TSG_SAG_LABEL_RANGE into the caller's status word (when given).
#include "common.cuh"
#include <float.h>

namespace tsg {

constexpr int KNN_MAXK = 32;
constexpr int KNN_MAXC = 1024;

// Per-CTA integer tallies, the first KNN_TALLIES words of the dynamic shared memory: [0] correct count, [1] status
// bits.  Flushed once per CTA: one 64-bit integer atomic for the count (no floating-point atomics), one OR.
constexpr int KNN_TALLIES = 2;

__device__ __forceinline__ void flush_tallies(const unsigned int* tally, int64_t* correct, int32_t* status) {
  if (correct && tally[0]) atomicAdd(reinterpret_cast<unsigned long long*>(correct), (unsigned long long)tally[0]);
  if (status && tally[1]) atomicOr(status, (int)tally[1]);
}

__global__ void __launch_bounds__(128)
k_knn_classify(const float* __restrict__ train, const int64_t* __restrict__ labels, const float* __restrict__ query,
               const int64_t* __restrict__ qlabels, int M, int Q, int D, int k, int C, int64_t* __restrict__ pred,
               int64_t* __restrict__ correct, int32_t* __restrict__ status) {
  extern __shared__ float sm[];              // tallies, then per warp: query row [D], k x 32 distances, k x 32 indices, C votes
  unsigned int* tally = reinterpret_cast<unsigned int*>(sm);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  float* qrow = sm + KNN_TALLIES + (size_t)warp * (D + 64 * k + C);
  float* cd = qrow + D;                                  // cd[j * 32 + lane]: lane's j-th best distance
  int* ci = reinterpret_cast<int*>(cd + 32 * k);         // ci[j * 32 + lane]: its train index
  int* votes = ci + 32 * k;                              // [C]
  if (threadIdx.x == 0) { tally[0] = 0; tally[1] = 0; }
  __syncthreads();
  int bad = 0;
  unsigned int hits = 0;
  for (int q = blockIdx.x * wpb + warp; q < Q; q += gridDim.x * wpb) {
    for (int d = lane; d < D; d += 32) qrow[d] = query[(int64_t)q * D + d];
    for (int c = lane; c < C; c += 32) votes[c] = 0;
    for (int j = 0; j < k; ++j) { cd[j * 32 + lane] = FLT_MAX; ci[j * 32 + lane] = 0x7fffffff; }
    __syncwarp();
    for (int r = lane; r < M; r += 32) {
      const float* t = train + (int64_t)r * D;
      float s = 0.f;
      for (int d = 0; d < D; ++d) { const float df = t[d] - qrow[d]; s = fmaf(df, df, s); }
      // insert (s, r) into the sorted list of the k best (ties -> lower index; r ascends, so strict <)
      if (s < cd[(k - 1) * 32 + lane]) {
        int j = k - 1;
        while (j > 0 && s < cd[(j - 1) * 32 + lane]) { cd[j * 32 + lane] = cd[(j - 1) * 32 + lane]; ci[j * 32 + lane] = ci[(j - 1) * 32 + lane]; --j; }
        cd[j * 32 + lane] = s; ci[j * 32 + lane] = r;
      }
    }
    // k rounds of a warp-wide arg-min over the lanes' list heads by (distance, index); row r lives in lane r % 32
    int head = 0;
    for (int round = 0; round < k; ++round) {
      float md = FLT_MAX; int mi = 0x7fffffff;
      if (head < k) { md = cd[head * 32 + lane]; mi = ci[head * 32 + lane]; }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float od = __shfl_xor_sync(0xffffffffu, md, o);
        const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
        if (od < md || (od == md && oi < mi)) { md = od; mi = oi; }
      }
      if (mi == 0x7fffffff) break;                       // fewer than k train rows
      if ((mi & 31) == lane) ++head;
      if (lane == 0) ++votes[clamp_label(labels[mi], C, bad)];
    }
    __syncwarp();
    // first class with the most votes
    int bv = -1, bc = 0x7fffffff;
    for (int c = lane; c < C; c += 32) if (votes[c] > bv) { bv = votes[c]; bc = c; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const int ov = __shfl_xor_sync(0xffffffffu, bv, o), oc = __shfl_xor_sync(0xffffffffu, bc, o);
      if (ov > bv || (ov == bv && oc < bc)) { bv = ov; bc = oc; }
    }
    if (lane == 0) {
      pred[q] = bc;
      if (qlabels) hits += (clamp_label(qlabels[q], C, bad) == bc);
    }
    __syncwarp();
  }
  if (hits) atomicAdd(&tally[0], hits);
  if (bad) atomicOr(&tally[1], (unsigned int)bad);
  __syncthreads();
  if (threadIdx.x == 0) flush_tallies(tally, correct, status);
}

// ------------------------------------------------------------------------------------------ sequential MLP trainer
__device__ __forceinline__ float leaky(float x, float slope) { return x > 0.f ? x : slope * x; }

// One unit of the MLP's forward: bias + sum_d w[d] * x[d] as ONE fmaf chain over d ascending.  The trainer and the
// predictor both call this, so their logits agree bit for bit for the same parameters.
__device__ __forceinline__ float mlp1_unit(const float* w, float bias, const float* x, int n) {
  float a = bias;
  for (int d = 0; d < n; ++d) a = fmaf(w[d], x[d], a);
  return a;
}

struct AdamCfg { float lr, b1, b2, eps; };

__device__ __forceinline__ void adam_update(float& p, float& m, float& v, float g, const AdamCfg& a, float bc1, float sqrt_bc2) {
  m = m + (1.f - a.b1) * (g - m);                       // exp_avg.lerp_(grad, 1 - beta1)
  v = a.b2 * v + (1.f - a.b2) * g * g;                  // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
  const float denom = sqrtf(v) / sqrt_bc2 + a.eps;
  p = p - (a.lr / bc1) * (m / denom);
}

__global__ void __launch_bounds__(256)
k_mlp1_train(const float* __restrict__ emb, const int64_t* __restrict__ labels, int N, int D, int H1, int H2, int C,
             float* __restrict__ params, float* __restrict__ am, float* __restrict__ av, long long step0,
             AdamCfg cfg, float slope, float* __restrict__ losses) {
  extern __shared__ float sm[];
  const int P = H1 * D + H1 + H2 * H1 + H2 + C * H2 + C;
  float* w = sm; float* m = w + P; float* v = m + P;
  float* x = v + P; float* z1 = x + D; float* h1 = z1 + H1; float* dz1 = h1 + H1;
  float* z2 = dz1 + H1; float* h2 = z2 + H2; float* dz2 = h2 + H2; float* dl = dz2 + H2;   // dl[C]
  const int oW1 = 0, ob1 = oW1 + H1 * D, oW2 = ob1 + H1, ob2 = oW2 + H2 * H1, oW3 = ob2 + H2, ob3 = oW3 + C * H2;
  for (int i = threadIdx.x; i < P; i += blockDim.x) { w[i] = params[i]; m[i] = am[i]; v[i] = av[i]; }
  __syncthreads();
  for (int s = 0; s < N; ++s) {
    const long long t = step0 + s + 1;
    // torch evaluates the bias corrections in double on the host (1 - beta ** step) and rounds once
    const float bc1 = (float)(1.0 - pow((double)cfg.b1, (double)t));
    const float sqrt_bc2 = (float)sqrt(1.0 - pow((double)cfg.b2, (double)t));
    for (int d = threadIdx.x; d < D; d += blockDim.x) x[d] = emb[(int64_t)s * D + d];
    __syncthreads();
    if (threadIdx.x < H1) {
      const float a = mlp1_unit(w + oW1 + threadIdx.x * D, w[ob1 + threadIdx.x], x, D);
      z1[threadIdx.x] = a; h1[threadIdx.x] = leaky(a, slope);
    }
    __syncthreads();
    if (threadIdx.x < H2) {
      const float a = mlp1_unit(w + oW2 + threadIdx.x * H1, w[ob2 + threadIdx.x], h1, H1);
      z2[threadIdx.x] = a; h2[threadIdx.x] = leaky(a, slope);
    }
    __syncthreads();
    if (threadIdx.x == 0) {                              // logits, softmax, cross-entropy (C is tiny)
      float mx = -FLT_MAX;
      for (int c = 0; c < C; ++c) {
        const float a = mlp1_unit(w + oW3 + c * H2, w[ob3 + c], h2, H2);
        dl[c] = a; mx = fmaxf(mx, a);
      }
      float se = 0.f;
      for (int c = 0; c < C; ++c) se += expf(dl[c] - mx);
      const int y = (int)labels[s];
      if (losses) losses[s] = logf(se) + mx - dl[y];
      for (int c = 0; c < C; ++c) dl[c] = expf(dl[c] - mx) / se - (c == y ? 1.f : 0.f);
    }
    __syncthreads();
    if (threadIdx.x < H2) {                              // dz2 = (W3^T dl) * leaky'(z2)
      float a = 0.f;
      for (int c = 0; c < C; ++c) a = fmaf(w[oW3 + c * H2 + threadIdx.x], dl[c], a);
      dz2[threadIdx.x] = a * (z2[threadIdx.x] > 0.f ? 1.f : slope);
    }
    __syncthreads();
    if (threadIdx.x < H1) {                              // dz1 = (W2^T dz2) * leaky'(z1)
      float a = 0.f;
      for (int o = 0; o < H2; ++o) a = fmaf(w[oW2 + o * H1 + threadIdx.x], dz2[o], a);
      dz1[threadIdx.x] = a * (z1[threadIdx.x] > 0.f ? 1.f : slope);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < P; i += blockDim.x) {  // gradients are outer products: formed in the update
      float g;
      if (i < ob1) { const int o = i / D, d = i - o * D; g = dz1[o] * x[d]; }
      else if (i < oW2) g = dz1[i - ob1];
      else if (i < ob2) { const int j = i - oW2, o = j / H1, d = j - o * H1; g = dz2[o] * h1[d]; }
      else if (i < oW3) g = dz2[i - ob2];
      else if (i < ob3) { const int j = i - oW3, o = j / H2, d = j - o * H2; g = dl[o] * h2[d]; }
      else g = dl[i - ob3];
      adam_update(w[i], m[i], v[i], g, cfg, bc1, sqrt_bc2);
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < P; i += blockDim.x) { params[i] = w[i]; am[i] = m[i]; av[i] = v[i]; }
}


// ------------------------------------------------------------------------------------------ MLP predictor
// Each layer's weight rows sit in shared memory at the odd stride n | 1 (n = the layer's input width): lane o reads row
// o, so the 32 lanes of a warp hit 32 different banks whatever the widths.  Biases follow each layer's rows.
__host__ __device__ inline int mlp1_padded_floats(int D, int H1, int H2, int C) {
  return H1 * (D | 1) + H1 + H2 * (H1 | 1) + H2 + C * (H2 | 1) + C;
}

__global__ void __launch_bounds__(256)
k_mlp1_predict(const float* __restrict__ emb, const int64_t* __restrict__ labels, int Q, int D, int H1, int H2, int C,
               const float* __restrict__ params, float slope, int64_t* __restrict__ pred, float* __restrict__ logits,
               int64_t* __restrict__ correct, int32_t* __restrict__ status) {
  extern __shared__ float sm[];              // tallies, padded params, then per warp: x [D], h1 [H1], h2 [H2]
  unsigned int* tally = reinterpret_cast<unsigned int*>(sm);
  const int sD = D | 1, sH1 = H1 | 1, sH2 = H2 | 1;
  const int oW1 = 0, ob1 = oW1 + H1 * sD, oW2 = ob1 + H1, ob2 = oW2 + H2 * sH1, oW3 = ob2 + H2, ob3 = oW3 + C * sH2;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  float* w = sm + KNN_TALLIES;
  float* x = w + mlp1_padded_floats(D, H1, H2, C) + (size_t)warp * (D + H1 + H2);
  float* h1 = x + D; float* h2 = h1 + H1;
  {                                          // flat [W1, b1, W2, b2, W3, b3] -> padded rows
    const int segs[6] = {H1 * D, H1, H2 * H1, H2, C * H2, C}, width[6] = {D, 1, H1, 1, H2, 1};
    const int stride[6] = {sD, 1, sH1, 1, sH2, 1}, dst[6] = {oW1, ob1, oW2, ob2, oW3, ob3};
    int src = 0;
    for (int sg = 0; sg < 6; ++sg) {
      for (int i = threadIdx.x; i < segs[sg]; i += blockDim.x)
        w[dst[sg] + (i / width[sg]) * stride[sg] + i % width[sg]] = params[src + i];
      src += segs[sg];
    }
  }
  if (threadIdx.x == 0) { tally[0] = 0; tally[1] = 0; }
  __syncthreads();
  int bad = 0;
  unsigned int hits = 0;
  for (int q = blockIdx.x * wpb + warp; q < Q; q += gridDim.x * wpb) {
    for (int d = lane; d < D; d += 32) x[d] = emb[(int64_t)q * D + d];
    __syncwarp();
    for (int o = lane; o < H1; o += 32) h1[o] = leaky(mlp1_unit(w + oW1 + o * sD, w[ob1 + o], x, D), slope);
    __syncwarp();
    for (int o = lane; o < H2; o += 32) h2[o] = leaky(mlp1_unit(w + oW2 + o * sH1, w[ob2 + o], h1, H1), slope);
    __syncwarp();
    float bv = -FLT_MAX; int bc = 0x7fffffff;
    for (int c = lane; c < C; c += 32) {
      const float a = mlp1_unit(w + oW3 + c * sH2, w[ob3 + c], h2, H2);
      if (logits) logits[(int64_t)q * C + c] = a;
      if (bc == 0x7fffffff || a > bv) { bv = a; bc = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {                   // argmax, first index on ties
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oc = __shfl_xor_sync(0xffffffffu, bc, o);
      if (oc != 0x7fffffff && (bc == 0x7fffffff || ov > bv || (ov == bv && oc < bc))) { bv = ov; bc = oc; }
    }
    if (lane == 0) {
      pred[q] = bc;
      if (labels) hits += (clamp_label(labels[q], C, bad) == bc);
    }
    __syncwarp();
  }
  if (hits) atomicAdd(&tally[0], hits);
  if (bad) atomicOr(&tally[1], (unsigned int)bad);
  __syncthreads();
  if (threadIdx.x == 0) flush_tallies(tally, correct, status);
}

}  // namespace tsg

using namespace tsg;

// *correct = 0 (an empty query set counts 0); reports only this memset's own error
static int zero_count(int64_t* correct, void* stream, const char* what) {
  if (!correct) return TSG_OK;
  const cudaError_t e = cudaMemsetAsync(correct, 0, sizeof(int64_t), (cudaStream_t)stream);
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return TSG_ELAUNCH;
  }
  return TSG_OK;
}

extern "C" int tsg_knn_classify(const float* train, const int64_t* train_labels, const float* query,
                                const int64_t* query_labels, int64_t num_train, int64_t num_query, int64_t dim, int k,
                                int num_classes, int64_t* pred, int64_t* correct, int32_t* status, void* stream) {
  TSG_REQUIRE(num_train > 0 && num_query >= 0 && dim > 0, "knn_classify: bad shape");
  TSG_REQUIRE(k >= 1 && k <= KNN_MAXK, "knn_classify: k must be in [1, %d]", KNN_MAXK);
  TSG_REQUIRE(num_classes >= 1 && num_classes <= KNN_MAXC, "knn_classify: num_classes must be in [1, %d]", KNN_MAXC);
  TSG_REQUIRE(num_train < (int64_t)0x7fffffff && num_query < (int64_t)0x7fffffff, "knn_classify: too large");
  TSG_REQUIRE(!correct || query_labels || num_query == 0, "knn_classify: a correct count needs query labels");
  const int rc = zero_count(correct, stream, "knn_classify");
  if (rc != TSG_OK || num_query == 0) return rc;
  TSG_REQUIRE(train && train_labels && query && pred, "knn_classify: null pointer");
  const int wpb = 4;
  const size_t smem = (KNN_TALLIES + (size_t)wpb * ((size_t)dim + 64 * (size_t)k + (size_t)num_classes)) * sizeof(float);
  TSG_REQUIRE(smem <= 200 * 1024, "knn_classify: embedding width %lld too large", (long long)dim);
  if (smem > 48 * 1024) cudaFuncSetAttribute(k_knn_classify, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k_knn_classify<<<grid_for(num_query, wpb), wpb * 32, smem, (cudaStream_t)stream>>>(
      train, train_labels, query, query_labels, (int)num_train, (int)num_query, (int)dim, k, num_classes, pred, correct, status);
  return check_launch("knn_classify");
}

extern "C" int tsg_knn_predict(const float* train, const int64_t* train_labels, const float* query,
                               int64_t num_train, int64_t num_query, int64_t dim, int k, int num_classes,
                               int64_t* pred, void* stream) {
  return tsg_knn_classify(train, train_labels, query, nullptr, num_train, num_query, dim, k, num_classes, pred, nullptr,
                          nullptr, stream);
}

extern "C" int tsg_mlp1_train(const float* emb, const int64_t* labels, int64_t num_samples, int64_t dim,
                              int64_t hidden1, int64_t hidden2, int64_t num_classes,
                              float* params, float* adam_m, float* adam_v, int64_t step0,
                              float lr, float beta1, float beta2, float eps, float slope,
                              float* losses, void* stream) {
  TSG_REQUIRE(num_samples >= 0 && dim > 0 && hidden1 > 0 && hidden2 > 0 && num_classes > 0, "mlp1_train: bad shape");
  TSG_REQUIRE(hidden1 <= 256 && hidden2 <= 256 && num_classes <= 32, "mlp1_train: layer too wide for one CTA");
  if (num_samples == 0) return TSG_OK;
  TSG_REQUIRE(emb && labels && params && adam_m && adam_v, "mlp1_train: null pointer");
  const size_t P = (size_t)(hidden1 * dim + hidden1 + hidden2 * hidden1 + hidden2 + num_classes * hidden2 + num_classes);
  const size_t smem = (3 * P + (size_t)dim + 3 * hidden1 + 3 * hidden2 + num_classes + 8) * sizeof(float);
  TSG_REQUIRE(smem <= 220 * 1024, "mlp1_train: %zu parameters do not fit shared memory", P);
  if (smem > 48 * 1024) cudaFuncSetAttribute(k_mlp1_train, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  AdamCfg cfg{lr, beta1, beta2, eps};
  k_mlp1_train<<<1, 256, smem, (cudaStream_t)stream>>>(emb, labels, (int)num_samples, (int)dim, (int)hidden1, (int)hidden2,
                                                      (int)num_classes, params, adam_m, adam_v, (long long)step0, cfg, slope, losses);
  return check_launch("mlp1_train");
}

extern "C" int tsg_mlp1_predict(const float* emb, const int64_t* labels, int64_t num_rows, int64_t dim, int64_t hidden1,
                                int64_t hidden2, int64_t num_classes, const float* params, float slope, int64_t* pred,
                                float* logits, int64_t* correct, int32_t* status, void* stream) {
  TSG_REQUIRE(num_rows >= 0 && dim > 0 && hidden1 > 0 && hidden2 > 0 && num_classes > 0, "mlp1_predict: bad shape");
  TSG_REQUIRE(num_rows < (int64_t)0x7fffffff, "mlp1_predict: too many rows");
  TSG_REQUIRE(!correct || labels || num_rows == 0, "mlp1_predict: a correct count needs labels");
  const int rc = zero_count(correct, stream, "mlp1_predict");
  if (rc != TSG_OK || num_rows == 0) return rc;
  TSG_REQUIRE(emb && params && pred, "mlp1_predict: null pointer");
  const int wpb = 8;
  const size_t P = (size_t)(hidden1 * dim + hidden1 + hidden2 * hidden1 + hidden2 + num_classes * hidden2 + num_classes);
  TSG_REQUIRE(P <= 220 * 1024 / sizeof(float), "mlp1_predict: %zu parameters do not fit shared memory", P);
  const size_t smem = (KNN_TALLIES + (size_t)mlp1_padded_floats((int)dim, (int)hidden1, (int)hidden2, (int)num_classes) +
                       (size_t)wpb * (size_t)(dim + hidden1 + hidden2)) * sizeof(float);
  TSG_REQUIRE(smem <= 220 * 1024, "mlp1_predict: %zu parameters do not fit shared memory", P);
  if (smem > 48 * 1024) cudaFuncSetAttribute(k_mlp1_predict, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k_mlp1_predict<<<grid_for(num_rows, wpb, 1), wpb * 32, smem, (cudaStream_t)stream>>>(
      emb, labels, (int)num_rows, (int)dim, (int)hidden1, (int)hidden2, (int)num_classes, params, slope, pred, logits,
      correct, status);
  return check_launch("mlp1_predict");
}
