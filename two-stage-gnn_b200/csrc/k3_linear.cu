// K3 -- tall-skinny row-local dense kernels: Y = X.W (+b) with the dense-directory epilogue
// (row L2-normalise -> ReLU -> node-wise BatchNorm), its backward, and dW = X^T.dY / db.
//
// Replaces, for N ~ 10^6 packed node rows and K, M <= 128..256 feature columns:
//   * `x @ weight` of PyG GCNConv (Code/sag/network.py:34 via GCNConv.forward) and its autograd
//     (dX = dH.W^T, dW = X^T.dH), which torch hands to cuBLAS SIMT sgemm kernels that cost more
//     than every aggregation kernel together (profiles/r01_launch_summary.md);
//   * `torch.matmul(y, self.weight) + self.bias` -> `F.normalize(y, p=2, dim=2)` of the dense
//     GraphConv (Code/sage+gat+diffpool/encoders.py:36-40; Code/eigengcn/encoders.py:34-39),
//     `self.act` (ReLU) and `apply_bn` (encoders.py:134-138: a FRESH BatchNorm1d(num_nodes) per
//     call => per-node statistics over the feature axis, biased variance, eps 1e-5, no affine, no
//     running state; with the scripts' batch size of one graph it is a per-node LayerNorm).
//
// These products are HBM-bound (AI = K.M/(2(K+M)) flop/B ~ 12 at 89x32): the design goal is to read X
// once, keep W in shared memory, and skip exact zeros (one-hot node-label features have ONE
// non-zero in 89 columns: the dot product stays bit-identical because the skipped terms are +0).
// Plain FP32 FFMA; no tensor cores (TF32 would break the 1e-5 parity bar; DiffPool's contractions
// use the 3xTF32 split on tcgen05 in k7).
#include "common.cuh"
#include <stdlib.h>

namespace tsg {

constexpr int LIN_THREADS = 256;
constexpr int LIN_RPT = 2;                 // rows per thread
constexpr float NORM_EPS = 1e-12f;         // F.normalize eps
constexpr float BN_EPS = 1e-5f;            // BatchNorm1d eps


__device__ __forceinline__ void cp_async4(float* smem_dst, const float* gsrc) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N_> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N_) : "memory"); }

__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(s), "l"(gsrc) : "memory");
}

// shared-memory row pitch: odd K needs no padding (odd stride = conflict free) and lets a tile be copied
// as ONE contiguous 16-byte stream; K % 4 == 0 pads by 4 floats so every row stays 16-byte aligned.
__host__ __device__ __forceinline__ int lin_pitch(int K) { return (K & 1) ? K : ((K & 3) == 0 ? K + 4 : K + 1); }

// asynchronously stage rows [r0, r0+R) of X[N,K] (row stride ldx) into Xs[R][pitch] (rows past N are zero filled)
__device__ __forceinline__ void stage_rows_async(float* Xs, const float* __restrict__ X, int r0, int R,
                                                 int N, int K, int pitch, int ldx) {
  const int rows = min(R, N - r0);
  const bool base16 = ((((size_t)(X + (size_t)r0 * ldx)) & 15) == 0);
  if (pitch == K && ldx == K && base16) {        // contiguous tile: 16-byte stream + scalar tail
    const float* src = X + (size_t)r0 * K;
    const int total = rows * K, total4 = total & ~3;
    for (int i = threadIdx.x * 4; i < total4; i += LIN_THREADS * 4) cp_async16(Xs + i, src + i);
    for (int i = total4 + threadIdx.x; i < total; i += LIN_THREADS) cp_async4(Xs + i, src + i);
    for (int i = total + threadIdx.x; i < R * K; i += LIN_THREADS) Xs[i] = 0.f;
  } else if ((K & 3) == 0 && (ldx & 3) == 0 && base16) {     // 16-byte aligned rows, padded pitch
    const int K4 = K >> 2;
    for (int i = threadIdx.x; i < R * K4; i += LIN_THREADS) {
      const int r = i / K4, k = (i - r * K4) * 4;
      float* dst = Xs + r * pitch + k;
      if (r < rows) cp_async16(dst, X + (size_t)(r0 + r) * ldx + k);
      else { dst[0] = 0.f; dst[1] = 0.f; dst[2] = 0.f; dst[3] = 0.f; }
    }
  } else {
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int r = w; r < R; r += LIN_THREADS / 32) {
      float* dst = Xs + r * pitch;
      if (r < rows) {
        const float* src = X + (size_t)(r0 + r) * ldx;
        for (int k = lane; k < K; k += 32) cp_async4(dst + k, src + k);
      } else {
        for (int k = lane; k < K; k += 32) dst[k] = 0.f;
      }
    }
  }
  cp_async_commit();
}

template <int CG>
__device__ __forceinline__ float group_sum(float v, unsigned mask) {
#pragma unroll
  for (int d = CG / 2; d > 0; d >>= 1) v += __shfl_xor_sync(mask, v, d);
  return v;
}

template <int CG>
__device__ __forceinline__ float group_max(float v, unsigned mask) {
#pragma unroll
  for (int d = CG / 2; d > 0; d >>= 1) v = fmaxf(v, __shfl_xor_sync(mask, v, d));
  return v;
}

// epilogue on one row held as 4 columns per lane across CG lanes. `ok[c]` masks padded columns.
template <int CG>
__device__ __forceinline__ void row_epilogue(float (&u)[4], const bool (&ok)[4], int M, int flags,
                                             unsigned gmask) {
  if (flags & TSG_LIN_NORMALIZE) {
    float ss = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) if (ok[c]) ss += u[c] * u[c];
    ss = group_sum<CG>(ss, gmask);
    float nrm = fmaxf(sqrtf(ss), NORM_EPS);
#pragma unroll
    for (int c = 0; c < 4; ++c) u[c] = u[c] / nrm;
  }
  if (flags & TSG_LIN_RELU) {
#pragma unroll
    for (int c = 0; c < 4; ++c) u[c] = fmaxf(u[c], 0.f);
  }
  if (flags & TSG_LIN_NODEBN) {
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) if (ok[c]) s += u[c];
    float mean = group_sum<CG>(s, gmask) / (float)M;
    float q = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) if (ok[c]) { float d = u[c] - mean; q += d * d; }
    float var = group_sum<CG>(q, gmask) / (float)M;
    float rstd = 1.0f / sqrtf(var + BN_EPS);
#pragma unroll
    for (int c = 0; c < 4; ++c) u[c] = (u[c] - mean) * rstd;
  }
  if (flags & TSG_LIN_SOFTMAX) {                 // DiffPool's assignment: softmax over the row (encoders.py:369)
    float mx = -3.4e38f;
#pragma unroll
    for (int c = 0; c < 4; ++c) if (ok[c]) mx = fmaxf(mx, u[c]);
    mx = group_max<CG>(mx, gmask);
    float se = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) { u[c] = ok[c] ? expf(u[c] - mx) : 0.f; se += u[c]; }
    se = group_sum<CG>(se, gmask);
#pragma unroll
    for (int c = 0; c < 4; ++c) u[c] = u[c] / se;
  }
}

// Y[N,M] = epilogue(X[N,K] . Wop + bias), Wop = W[K,M] or W[M,K]^T.  Persistent CTAs: W staged in
// shared memory once, then a grid-stride loop over tiles of R = (256/CG)*2 rows.
// A K too long for W's slab runs as consecutive launches over blocks of K (X row stride ldx): LIN_KACC_IN starts every
// accumulator from Y, LIN_KPARTIAL stores it without bias and epilogue -- one k-ascending FMA chain per output, as in a
// single pass.
constexpr int LIN_KACC_IN = 1, LIN_KPARTIAL = 2;
template <int CG>
__global__ void __launch_bounds__(LIN_THREADS)
k_linear_fwd(const float* __restrict__ X, const float* __restrict__ W, const float* __restrict__ bias,
             float* __restrict__ Y, int N, int K, int M, int ldw, int ldy, int w_transposed, int flags, int ldx,
             int kmode) {
  pdl_wait();
  pdl_launch_dependents();
  extern __shared__ __align__(16) float smem[];
  constexpr int RS = LIN_THREADS / CG;
  constexpr int R = RS * LIN_RPT;
  const int Mp = CG * 4;
  const int pitch = lin_pitch(K);
  float* Ws = smem;                              // [K][Mp]
  float* Xs = smem + (size_t)K * Mp;             // [R][pitch]
  const int cg = threadIdx.x % CG, rs = threadIdx.x / CG;
  const unsigned gmask = CG == 32 ? 0xffffffffu : (((1u << CG) - 1u) << (((threadIdx.x & 31) / CG) * CG));

  for (int i = threadIdx.x; i < K * Mp; i += LIN_THREADS) {
    int k = i / Mp, m = i - k * Mp;
    float w = 0.f;
    if (m < M) w = w_transposed ? W[(size_t)m * ldw + k] : W[(size_t)k * ldw + m];
    Ws[i] = w;
  }
  bool ok[4]; float b4[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    ok[c] = cg * 4 + c < M;
    b4[c] = (bias != nullptr && ok[c]) ? bias[cg * 4 + c] : 0.f;
  }
  const int num_tiles = (N + R - 1) / R;
  int buf = 0;
  if ((int)blockIdx.x < num_tiles) stage_rows_async(Xs, X, blockIdx.x * R, R, N, K, pitch, ldx);
  for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
    const int r0 = tile * R;
    const int rows = min(R, N - r0);
    const int next = tile + gridDim.x;
    float* Xcur = Xs + (size_t)buf * R * pitch;
    if (next < num_tiles) {                      // prefetch the next tile into the other buffer
      stage_rows_async(Xs + (size_t)(buf ^ 1) * R * pitch, X, next * R, R, N, K, pitch, ldx);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();                             // this tile's rows (and Ws on the first pass) visible
    float acc[LIN_RPT][4];
#pragma unroll
    for (int j = 0; j < LIN_RPT; ++j)
#pragma unroll
      for (int c = 0; c < 4; ++c)
        acc[j][c] = (kmode & LIN_KACC_IN) && rs + j * RS < rows && ok[c] ? Y[(size_t)(r0 + rs + j * RS) * ldy + cg * 4 + c] : 0.f;
    const float* x0 = Xcur + (rs)*pitch;
    const float* x1 = Xcur + (rs + RS) * pitch;
    for (int k = 0; k < K; ++k) {
      float a0 = x0[k], a1 = x1[k];
      if (!__any_sync(0xffffffffu, (a0 != 0.f) | (a1 != 0.f))) continue;   // exact zeros contribute +0
      float4 w = *reinterpret_cast<const float4*>(Ws + k * Mp + cg * 4);
      acc[0][0] = fmaf(a0, w.x, acc[0][0]); acc[0][1] = fmaf(a0, w.y, acc[0][1]);
      acc[0][2] = fmaf(a0, w.z, acc[0][2]); acc[0][3] = fmaf(a0, w.w, acc[0][3]);
      acc[1][0] = fmaf(a1, w.x, acc[1][0]); acc[1][1] = fmaf(a1, w.y, acc[1][1]);
      acc[1][2] = fmaf(a1, w.z, acc[1][2]); acc[1][3] = fmaf(a1, w.w, acc[1][3]);
    }
#pragma unroll
    for (int j = 0; j < LIN_RPT; ++j) {
      const int r = rs + j * RS;
      if (!(kmode & LIN_KPARTIAL)) {
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[j][c] += b4[c];
        if (flags) row_epilogue<CG>(acc[j], ok, M, flags, gmask);
      }
      if (r < rows) {
        float* dst = Y + (size_t)(r0 + r) * ldy + cg * 4;
        if ((M & 3) == 0 && (ldy & 3) == 0) {
          if (ok[0]) *reinterpret_cast<float4*>(dst) = make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]);
        } else {
#pragma unroll
          for (int c = 0; c < 4; ++c) if (ok[c]) dst[c] = acc[j][c];
        }
      }
    }
    __syncthreads();                             // everyone is done with Xcur before it is refilled
    buf ^= 1;
  }
}

// Dense-input variant (K % 4 == 0): no per-k zero test (the warp vote + scalar LDS per k made the K = 32 products
// of the pooled levels and of the backward issue bound: 62 us for 124 MB), x read as float4, 4 rows x 4 columns
// of register blocking per thread.  Same k-ascending FMA sequence per output as k_linear_fwd, so the two kernels
// agree bit for bit (a skipped zero term is fma(0, w, acc) = acc).
constexpr int LIND_RPT = 4;
template <int CG>
__global__ void __launch_bounds__(LIN_THREADS)
k_linear_fwd_dense(const float* __restrict__ X, const float* __restrict__ W, const float* __restrict__ bias,
                   float* __restrict__ Y, int N, int K, int M, int ldw, int ldy, int w_transposed, int flags) {
  pdl_wait();
  pdl_launch_dependents();
  extern __shared__ __align__(16) float smem[];
  constexpr int RS = LIN_THREADS / CG;
  constexpr int R = RS * LIND_RPT;
  const int Mp = CG * 4;
  const int pitch = K + 4;
  float* Ws = smem;                              // [K][Mp]
  float* Xs = smem + (size_t)K * Mp;             // 2 x [R][pitch]
  const int cg = threadIdx.x % CG, rs = threadIdx.x / CG;
  const unsigned gmask = CG == 32 ? 0xffffffffu : (((1u << CG) - 1u) << (((threadIdx.x & 31) / CG) * CG));
  for (int i = threadIdx.x; i < K * Mp; i += LIN_THREADS) {
    int k = i / Mp, m = i - k * Mp;
    float w = 0.f;
    if (m < M) w = w_transposed ? W[(size_t)m * ldw + k] : W[(size_t)k * ldw + m];
    Ws[i] = w;
  }
  bool ok[4]; float b4[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    ok[c] = cg * 4 + c < M;
    b4[c] = (bias != nullptr && ok[c]) ? bias[cg * 4 + c] : 0.f;
  }
  const int num_tiles = (N + R - 1) / R;
  int buf = 0;
  if ((int)blockIdx.x < num_tiles) stage_rows_async(Xs, X, blockIdx.x * R, R, N, K, pitch, K);
  for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
    const int r0 = tile * R;
    const int rows = min(R, N - r0);
    const int next = tile + gridDim.x;
    const float* Xcur = Xs + (size_t)buf * R * pitch;
    if (next < num_tiles) {
      stage_rows_async(Xs + (size_t)(buf ^ 1) * R * pitch, X, next * R, R, N, K, pitch, K);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    float acc[LIND_RPT][4];
#pragma unroll
    for (int j = 0; j < LIND_RPT; ++j)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[j][c] = 0.f;
    for (int k = 0; k < K; k += 4) {
      float4 w[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) w[q] = *reinterpret_cast<const float4*>(Ws + (k + q) * Mp + cg * 4);
#pragma unroll
      for (int j = 0; j < LIND_RPT; ++j) {
        const float4 a = *reinterpret_cast<const float4*>(Xcur + (rs + j * RS) * pitch + k);
        acc[j][0] = fmaf(a.x, w[0].x, acc[j][0]); acc[j][1] = fmaf(a.x, w[0].y, acc[j][1]);
        acc[j][2] = fmaf(a.x, w[0].z, acc[j][2]); acc[j][3] = fmaf(a.x, w[0].w, acc[j][3]);
        acc[j][0] = fmaf(a.y, w[1].x, acc[j][0]); acc[j][1] = fmaf(a.y, w[1].y, acc[j][1]);
        acc[j][2] = fmaf(a.y, w[1].z, acc[j][2]); acc[j][3] = fmaf(a.y, w[1].w, acc[j][3]);
        acc[j][0] = fmaf(a.z, w[2].x, acc[j][0]); acc[j][1] = fmaf(a.z, w[2].y, acc[j][1]);
        acc[j][2] = fmaf(a.z, w[2].z, acc[j][2]); acc[j][3] = fmaf(a.z, w[2].w, acc[j][3]);
        acc[j][0] = fmaf(a.w, w[3].x, acc[j][0]); acc[j][1] = fmaf(a.w, w[3].y, acc[j][1]);
        acc[j][2] = fmaf(a.w, w[3].z, acc[j][2]); acc[j][3] = fmaf(a.w, w[3].w, acc[j][3]);
      }
    }
#pragma unroll
    for (int j = 0; j < LIND_RPT; ++j) {
      const int r = rs + j * RS;
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[j][c] += b4[c];
      if (flags) row_epilogue<CG>(acc[j], ok, M, flags, gmask);
      if (r < rows) {
        float* dst = Y + (size_t)(r0 + r) * ldy + cg * 4;
        if ((M & 3) == 0 && (ldy & 3) == 0) {
          if (ok[0]) *reinterpret_cast<float4*>(dst) = make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]);
        } else {
#pragma unroll
          for (int c = 0; c < 4; ++c) if (ok[c]) dst[c] = acc[j][c];
        }
      }
    }
    __syncthreads();
    buf ^= 1;
  }
}

// Backward of the dense-directory epilogue: dU from dO, recomputing u = agg.W + b (agg is read for
// dW anyway; recomputing saves writing + re-reading u, v and the statistics).  A.4 of SURVEY:
//   BN:  dR = rstd * (dO - mean(dO) - o * mean(dO*o));  ReLU: dV = dR * (v > 0)
//   normalise: dU = (dV - v * (v.dV)) / max(||u||, eps)   (||u|| < eps: dU = dV / eps)
template <int CG>
__global__ void __launch_bounds__(LIN_THREADS)
k_dense_epilogue_bwd(const float* __restrict__ X, const float* __restrict__ W, const float* __restrict__ bias,
                     const float* __restrict__ dO, float* __restrict__ dU, int N, int K, int M, int flags) {
  extern __shared__ __align__(16) float smem[];
  constexpr int RS = LIN_THREADS / CG;
  constexpr int R = RS * LIN_RPT;
  const int Mp = CG * 4;
  const int pitch = lin_pitch(K);
  float* Ws = smem;
  float* Xs = smem + (size_t)K * Mp;
  const int cg = threadIdx.x % CG, rs = threadIdx.x / CG;
  const unsigned gmask = CG == 32 ? 0xffffffffu : (((1u << CG) - 1u) << (((threadIdx.x & 31) / CG) * CG));
  for (int i = threadIdx.x; i < K * Mp; i += LIN_THREADS) {
    int k = i / Mp, m = i - k * Mp;
    Ws[i] = m < M ? W[(size_t)k * M + m] : 0.f;
  }
  bool ok[4]; float b4[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    ok[c] = cg * 4 + c < M;
    b4[c] = (bias != nullptr && ok[c]) ? bias[cg * 4 + c] : 0.f;
  }
  const int num_tiles = (N + R - 1) / R;
  int buf = 0;
  if ((int)blockIdx.x < num_tiles) stage_rows_async(Xs, X, blockIdx.x * R, R, N, K, pitch, K);
  for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
    const int r0 = tile * R;
    const int rows = min(R, N - r0);
    const int next = tile + gridDim.x;
    float* Xcur = Xs + (size_t)buf * R * pitch;
    if (next < num_tiles) {                      // prefetch the next tile into the other buffer
      stage_rows_async(Xs + (size_t)(buf ^ 1) * R * pitch, X, next * R, R, N, K, pitch, K);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();                             // this tile's rows (and Ws on the first pass) visible
    float u[LIN_RPT][4];
#pragma unroll
    for (int j = 0; j < LIN_RPT; ++j)
#pragma unroll
      for (int c = 0; c < 4; ++c) u[j][c] = 0.f;
    const float* x0 = Xcur + (rs)*pitch;
    const float* x1 = Xcur + (rs + RS) * pitch;
    for (int k = 0; k < K; ++k) {
      float a0 = x0[k], a1 = x1[k];
      if (!__any_sync(0xffffffffu, (a0 != 0.f) | (a1 != 0.f))) continue;
      float4 w = *reinterpret_cast<const float4*>(Ws + k * Mp + cg * 4);
      u[0][0] = fmaf(a0, w.x, u[0][0]); u[0][1] = fmaf(a0, w.y, u[0][1]);
      u[0][2] = fmaf(a0, w.z, u[0][2]); u[0][3] = fmaf(a0, w.w, u[0][3]);
      u[1][0] = fmaf(a1, w.x, u[1][0]); u[1][1] = fmaf(a1, w.y, u[1][1]);
      u[1][2] = fmaf(a1, w.z, u[1][2]); u[1][3] = fmaf(a1, w.w, u[1][3]);
    }
#pragma unroll
    for (int j = 0; j < LIN_RPT; ++j) {
      const int r = rs + j * RS;
      const bool live = r < rows;
      float g[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        u[j][c] += b4[c];
        g[c] = (live && ok[c]) ? dO[(size_t)(r0 + r) * M + cg * 4 + c] : 0.f;
      }
      if (flags & TSG_LIN_SOFTMAX) {             // dL = S * (dS - rowsum(S * dS)), S recomputed from the logits
        float mx = -3.4e38f;
#pragma unroll
        for (int c = 0; c < 4; ++c) if (ok[c]) mx = fmaxf(mx, u[j][c]);
        mx = group_max<CG>(mx, gmask);
        float se = 0.f, sm4[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) { sm4[c] = ok[c] ? expf(u[j][c] - mx) : 0.f; se += sm4[c]; }
        se = group_sum<CG>(se, gmask);
        float dot = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) { sm4[c] = sm4[c] / se; dot += sm4[c] * g[c]; }
        dot = group_sum<CG>(dot, gmask);
        if (live) {
#pragma unroll
          for (int c = 0; c < 4; ++c) if (ok[c]) dU[(size_t)(r0 + r) * M + cg * 4 + c] = sm4[c] * (g[c] - dot);
        }
        continue;
      }
      // forward recompute
      float nrm = 1.f, v[4], rl[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) v[c] = u[j][c];
      if (flags & TSG_LIN_NORMALIZE) {
        float ss = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) if (ok[c]) ss += v[c] * v[c];
        ss = group_sum<CG>(ss, gmask);
        nrm = fmaxf(sqrtf(ss), NORM_EPS);
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = v[c] / nrm;
      }
#pragma unroll
      for (int c = 0; c < 4; ++c) rl[c] = (flags & TSG_LIN_RELU) ? fmaxf(v[c], 0.f) : v[c];
      if (flags & TSG_LIN_NODEBN) {
        float s = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) if (ok[c]) s += rl[c];
        float mean = group_sum<CG>(s, gmask) / (float)M;
        float q = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) if (ok[c]) { float d = rl[c] - mean; q += d * d; }
        float var = group_sum<CG>(q, gmask) / (float)M;
        float rstd = 1.0f / sqrtf(var + BN_EPS);
        float sg = 0.f, sgo = 0.f, o[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          o[c] = (rl[c] - mean) * rstd;
          if (ok[c]) { sg += g[c]; sgo += g[c] * o[c]; }
        }
        float mg = group_sum<CG>(sg, gmask) / (float)M;
        float mgo = group_sum<CG>(sgo, gmask) / (float)M;
#pragma unroll
        for (int c = 0; c < 4; ++c) g[c] = rstd * (g[c] - mg - o[c] * mgo);
      }
      if (flags & TSG_LIN_RELU) {
#pragma unroll
        for (int c = 0; c < 4; ++c) if (!(v[c] > 0.f)) g[c] = 0.f;
      }
      if (flags & TSG_LIN_NORMALIZE) {
        float dot = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) if (ok[c]) dot += v[c] * g[c];
        dot = group_sum<CG>(dot, gmask);
        // torch: y = x / clamp_min(||x||, eps).  Above the clamp d||x||/dx = x/||x|| = v;
        // at / below the clamp the denominator is the constant eps.
        const bool clamped = !(nrm > NORM_EPS);
#pragma unroll
        for (int c = 0; c < 4; ++c) g[c] = clamped ? g[c] / nrm : (g[c] - v[c] * dot) / nrm;
      }
      if (live) {
#pragma unroll
        for (int c = 0; c < 4; ++c) if (ok[c]) dU[(size_t)(r0 + r) * M + cg * 4 + c] = g[c];
      }
    }
    __syncthreads();
    buf ^= 1;
  }
}

// ------------------------------------------------------------------------------------------
// dW[K,M] = X^T . dY  -- deterministic two-stage reduction that streams X and dY exactly once.
// A warp owns rows r = w, w + W, ... of its CTA's contiguous row range.  Per row the lanes read
// X[r, 32c + lane] (coalesced) for every 32-column chunk c of K and dY[r, m0 + lane] (coalesced);
// all loads of U rows are issued before any is used (memory-level parallelism).  Non-zeros are
// found with a ballot and applied one by one to the warp's PRIVATE accumulator tile acc[k][lane] in
// shared memory (bank = lane: conflict free) -- with one-hot features that is one update per row.
// Order: rows ascending inside a warp, warps combined in index order, CTAs (fixed grid) in index
// order: bit-reproducible.  M is covered in passes of 32 columns.
// db (when requested) is the deterministic column sum of dY (tsg_relu_bwd_colsum's kernels).
// ------------------------------------------------------------------------------------------
constexpr int LBW_GRID = TSG_NUM_SMS * 2;

template <int NK, int U>
__global__ void __launch_bounds__(256)
k_linear_bwd_weight(const float* __restrict__ X, const float* __restrict__ dY, float* __restrict__ part,
                    int N, int K, int M, int m0, int ldx) {
  pdl_wait();
  pdl_launch_dependents();
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  float* acc = smem + (size_t)w * K * 32;                   // [K][32] private to this warp
  for (int i = lane; i < K * 32; i += 32) acc[i] = 0.f;
  __syncwarp();
  const int rows_per_cta = (N + gridDim.x - 1) / gridDim.x;
  const int r_begin = blockIdx.x * rows_per_cta;
  const int r_end = min(N, r_begin + rows_per_cta);
  const bool mok = m0 + lane < M;
  // dense rows (many non-zeros) accumulate in REGISTERS (one accumulator per k for this lane's
  // column) to avoid a serial shared-memory read-modify-write chain; only for K <= 64.
  constexpr bool REG = NK <= 2;
  float racc[REG ? NK * 32 : 1];
#pragma unroll
  for (int i = 0; i < (REG ? NK * 32 : 1); ++i) racc[i] = 0.f;
  for (int rb = r_begin + w; rb < r_end; rb += nw * U) {
    float xv[U][NK], dy[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int r = rb + u * nw;
      const bool rok = r < r_end;
      dy[u] = (rok && mok) ? __ldg(dY + (size_t)r * M + m0 + lane) : 0.f;
#pragma unroll
      for (int c = 0; c < NK; ++c) {
        const int k = c * 32 + lane;
        xv[u][c] = (rok && k < K) ? __ldg(X + (size_t)r * ldx + k) : 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
#pragma unroll
      for (int c = 0; c < NK; ++c) {
        unsigned mask = __ballot_sync(0xffffffffu, xv[u][c] != 0.f);
        if (REG && __popc(mask) > 6) {
#pragma unroll
          for (int b = 0; b < 32; ++b) {
            const float x = __shfl_sync(0xffffffffu, xv[u][c], b);
            racc[(REG ? c : 0) * 32 + b] = fmaf(x, dy[u], racc[(REG ? c : 0) * 32 + b]);
          }
          mask = 0;
        }
        while (mask) {
          const int b = __ffs(mask) - 1;
          mask &= mask - 1;
          const float x = __shfl_sync(0xffffffffu, xv[u][c], b);
          float* a = acc + (c * 32 + b) * 32 + lane;
          *a = fmaf(x, dy[u], *a);
        }
      }
    }
  }
  if (REG) {
    __syncwarp();
#pragma unroll
    for (int i = 0; i < NK * 32; ++i)
      if (i < K) acc[i * 32 + lane] += racc[i];
  }
  __syncthreads();
  // combine the warps in index order, write this CTA's partial for columns [m0, m0+32)
  float* mypart = part + (size_t)blockIdx.x * K * M;
  for (int i = threadIdx.x; i < K * 32; i += blockDim.x) {
    float s = smem[i];
    for (int ww = 1; ww < nw; ++ww) s += smem[(size_t)ww * K * 32 + i];
    const int k = i >> 5, m = m0 + (i & 31);
    if (m < M) mypart[(size_t)k * M + m] = s;
  }
}

// Dense-operand variant of dW = X^T dY for K % 4 == 0, M % 4 == 0, (K/4)(M/4) <= 256 (the 32x32 products of the
// pooled levels: the warp-per-row kernel above spends 32 shuffles + 32 FMAs per row per lane there, 81 us for
// 124 MB).  Row tiles of X and dY are staged in shared memory with 16-byte cp.async (double buffered); a thread
// owns a 4x4 block of dW and one of G = 256 / blocks row groups: two LDS.128 feed 16 FMAs.  Fixed partition
// (CTA row range, row group, k-ascending rows) => deterministic; groups then CTAs are combined in index order.
constexpr int LBWD_ROWS = 128;
__global__ void __launch_bounds__(256)
k_linear_bwd_weight_dense(const float* __restrict__ X, const float* __restrict__ dY, float* __restrict__ part,
                          int N, int K, int M) {
  pdl_wait();
  pdl_launch_dependents();
  extern __shared__ __align__(16) float smem[];
  const int KB = K >> 2, MB = M >> 2, NB = KB * MB;
  const int groups = 256 / NB;                       // >= 1
  const int blk = threadIdx.x % NB, grp = threadIdx.x / NB;
  const int kb = blk / MB, mb = blk - kb * MB;
  const bool active = grp < groups;
  float* Xs = smem;                                  // 2 x [ROWS][K]
  float* Ys = smem + 2 * LBWD_ROWS * K;              // 2 x [ROWS][M]
  const int rows_per_cta = (N + gridDim.x - 1) / gridDim.x;
  const int r_begin = blockIdx.x * rows_per_cta;
  const int r_end = min(N, r_begin + rows_per_cta);
  auto stage = [&](int buf, int r0) {
    const int rows = max(0, min(LBWD_ROWS, r_end - r0));
    const float* xs = X + (size_t)r0 * K; const float* ys = dY + (size_t)r0 * M;
    float* xd = Xs + buf * LBWD_ROWS * K; float* yd = Ys + buf * LBWD_ROWS * M;
    for (int i = threadIdx.x * 4; i < rows * K; i += 256 * 4) cp_async16(xd + i, xs + i);
    for (int i = threadIdx.x * 4; i < rows * M; i += 256 * 4) cp_async16(yd + i, ys + i);
    cp_async_commit();
  };
  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
  int buf = 0;
  if (r_begin < r_end) stage(0, r_begin);
  for (int r0 = r_begin; r0 < r_end; r0 += LBWD_ROWS) {
    const int rows = min(LBWD_ROWS, r_end - r0);
    if (r0 + LBWD_ROWS < r_end) { stage(buf ^ 1, r0 + LBWD_ROWS); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
    __syncthreads();
    if (active) {
      const float* xb = Xs + buf * LBWD_ROWS * K + kb * 4;
      const float* yb = Ys + buf * LBWD_ROWS * M + mb * 4;
      for (int r = grp; r < rows; r += groups) {
        const float4 a = *reinterpret_cast<const float4*>(xb + r * K);
        const float4 b = *reinterpret_cast<const float4*>(yb + r * M);
        acc[0][0] = fmaf(a.x, b.x, acc[0][0]); acc[0][1] = fmaf(a.x, b.y, acc[0][1]); acc[0][2] = fmaf(a.x, b.z, acc[0][2]); acc[0][3] = fmaf(a.x, b.w, acc[0][3]);
        acc[1][0] = fmaf(a.y, b.x, acc[1][0]); acc[1][1] = fmaf(a.y, b.y, acc[1][1]); acc[1][2] = fmaf(a.y, b.z, acc[1][2]); acc[1][3] = fmaf(a.y, b.w, acc[1][3]);
        acc[2][0] = fmaf(a.z, b.x, acc[2][0]); acc[2][1] = fmaf(a.z, b.y, acc[2][1]); acc[2][2] = fmaf(a.z, b.z, acc[2][2]); acc[2][3] = fmaf(a.z, b.w, acc[2][3]);
        acc[3][0] = fmaf(a.w, b.x, acc[3][0]); acc[3][1] = fmaf(a.w, b.y, acc[3][1]); acc[3][2] = fmaf(a.w, b.z, acc[3][2]); acc[3][3] = fmaf(a.w, b.w, acc[3][3]);
      }
    }
    __syncthreads();
    buf ^= 1;
  }
  // combine the row groups in index order through shared memory (reuse the staging buffers)
  float* red = smem;                                  // [groups][K*M]
  if (active) {
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) red[(size_t)grp * K * M + (kb * 4 + a) * M + mb * 4 + b] = acc[a][b];
  }
  __syncthreads();
  float* mypart = part + (size_t)blockIdx.x * K * M;
  for (int i = threadIdx.x; i < K * M; i += 256) {
    float t = red[i];
    for (int g2 = 1; g2 < groups; ++g2) t += red[(size_t)g2 * K * M + i];
    mypart[i] = t;
  }
}

// ------------------------------------------------------------------------------------------
// SAGPool level boundary of the encoder backward (K10 sag_bwd, levels 2 and 1): from dxw = A_hat^T dhm [N, H],
//   dxg = readout_bwd_{l-1}(dz) + dxw . W^T     (k_linear_fwd_dense, then k_readout_bwd MAX|MEAN|ACCUM)
//   part = per-CTA partials of x^T . dxw        (k_linear_bwd_weight_dense)
// in one pass: each LBWD_ROWS tile of dxw and x is staged once, dxg is written once.  Warps 0-7 accumulate dW over
// k_linear_bwd_weight_dense's exact partition (LBW_GRID CTAs, rows_per_cta, tiles from r_begin, row i of a tile to
// group i mod groups); warps 8-15 compute dX for the same tile with k_linear_fwd_dense's per-output chain (acc = 0,
// fmaf over k ascending, then + 0.f) and add the readout term as k_readout_bwd does: (gs + (am == r ? gm : 0)) + dX.
// Rows are staged at pitch H + 4 so the dX warps' float4 reads of four different rows hit different banks.
// ------------------------------------------------------------------------------------------
constexpr int SBB_THREADS = 512;

// largest g in [-1, G] with gptr[g] <= r (gptr[-1] taken as -inf): the graph of row r when 0 <= g < G
__device__ __forceinline__ int graph_search(const int64_t* __restrict__ gptr, int G, int64_t r) {
  int lo = -1, hi = G;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(gptr + mid) <= r) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// shared memory of k_sag_boundary_bwd<H>: W, two double-buffered row tiles, the tile's graph table, the dW accumulators
__host__ __device__ constexpr size_t sbb_smem_bytes(int H) {
  return ((size_t)H * H + 4 * LBWD_ROWS * (H + 4)) * sizeof(float) + 2 * LBWD_ROWS * sizeof(int) + 4 * 256 * sizeof(float4);
}

// two CTAs per SM up to H = 32; from H = 36 the 64 registers that allows spill, and from H = 44 two CTAs' shared
// memory does not fit an SM anyway
template <int H>
__global__ void __launch_bounds__(SBB_THREADS, H <= 32 ? 2 : 1)
k_sag_boundary_bwd(const float* __restrict__ dxw, const float* __restrict__ X, const float* __restrict__ W,
                   const float* __restrict__ dz, int64_t dz_stride, const int* __restrict__ argmax,
                   const int64_t* __restrict__ gptr, int G, int N, float* __restrict__ dxg, float* __restrict__ part) {
  pdl_wait();
  pdl_launch_dependents();
  constexpr int P = H + 4, CG = H / 4, NB = CG * CG, GROUPS = 256 / NB;
  extern __shared__ __align__(16) float smem[];
  float* Ws = smem;                                   // [H][H], Ws[k][m] = W[m][k]
  float* Xs = Ws + H * H;                             // 2 x [ROWS][P]
  float* Ys = Xs + 2 * LBWD_ROWS * P;                 // 2 x [ROWS][P] (dxw)
  int* rg = reinterpret_cast<int*>(Ys + 2 * LBWD_ROWS * P);    // [ROWS] graph of the tile's row (-1: none)
  float* rn = reinterpret_cast<float*>(rg + LBWD_ROWS);        // [ROWS] (float)max(n_g, 1)
  float4* accs = reinterpret_cast<float4*>(rn + LBWD_ROWS);    // [4][256] dW accumulators
  const int tid = threadIdx.x;
  const int rows_per_cta = (N + gridDim.x - 1) / gridDim.x;
  const int r_begin = blockIdx.x * rows_per_cta;
  const int r_end = min(N, r_begin + rows_per_cta);
  auto stage = [&](int buf, int r0) {
    const int rows = max(0, min(LBWD_ROWS, r_end - r0));
    float* xd = Xs + buf * LBWD_ROWS * P; float* yd = Ys + buf * LBWD_ROWS * P;
    for (int i = tid; i < rows * CG; i += SBB_THREADS) {
      const int r = i / CG, c = (i - r * CG) * 4;
      cp_async16(xd + r * P + c, X + (size_t)(r0 + r) * H + c);
      cp_async16(yd + r * P + c, dxw + (size_t)(r0 + r) * H + c);
    }
    cp_async_commit();
  };
  int buf = 0;
  if (r_begin < r_end) stage(0, r_begin);
  for (int i = tid; i < H * H; i += SBB_THREADS) {
    const int k = i / H, m = i - k * H;
    Ws[i] = W[(size_t)m * H + k];
  }
  // threads 256 + t look up the graph of row t of every tile, walking forward from the previous tile's row
  const int lt = tid - 256;
  const bool looker = lt >= 0 && lt < LBWD_ROWS;
  int gw = (looker && r_begin + lt < r_end) ? graph_search(gptr, G, r_begin + lt) : -1;
  // dW: thread tid < 256 owns the 4x4 block (kb, mb) of row group grp; its accumulators stay in shared memory
  // between tiles, so they are not live in registers while the same warps' code path for dX runs
  const int blk = tid % NB, grp = tid / NB;
  const int kb = blk / CG, mb = blk - kb * CG;
  const bool dw_thread = tid < 256 && grp < GROUPS;
  if (dw_thread)
#pragma unroll
    for (int a = 0; a < 4; ++a) accs[a * 256 + tid] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int r0 = r_begin; r0 < r_end; r0 += LBWD_ROWS) {
    const int rows = min(LBWD_ROWS, r_end - r0);
    if (looker) {
      int g = -1; float nf = 1.f;
      if (lt < rows) {
        const int64_t r = r0 + lt;
        while (gw < G && __ldg(gptr + gw + 1) <= r) ++gw;
        if (gw >= 0 && gw < G) {
          const int n = (int)(__ldg(gptr + gw + 1) - __ldg(gptr + gw));
          g = gw; nf = (float)(n > 0 ? n : 1);
        }
      }
      rg[lt] = g; rn[lt] = nf;
    }
    if (r0 + LBWD_ROWS < r_end) { stage(buf ^ 1, r0 + LBWD_ROWS); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
    __syncthreads();
    const float* xt = Xs + buf * LBWD_ROWS * P;
    const float* yt = Ys + buf * LBWD_ROWS * P;
    if (tid < 256) {
      if (dw_thread) {
        float acc[4][4];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          const float4 v = accs[a * 256 + tid];
          acc[a][0] = v.x; acc[a][1] = v.y; acc[a][2] = v.z; acc[a][3] = v.w;
        }
        const float* xb = xt + kb * 4;
        const float* yb = yt + mb * 4;
        for (int r = grp; r < rows; r += GROUPS) {
          const float4 a = *reinterpret_cast<const float4*>(xb + r * P);
          const float4 b = *reinterpret_cast<const float4*>(yb + r * P);
          acc[0][0] = fmaf(a.x, b.x, acc[0][0]); acc[0][1] = fmaf(a.x, b.y, acc[0][1]); acc[0][2] = fmaf(a.x, b.z, acc[0][2]); acc[0][3] = fmaf(a.x, b.w, acc[0][3]);
          acc[1][0] = fmaf(a.y, b.x, acc[1][0]); acc[1][1] = fmaf(a.y, b.y, acc[1][1]); acc[1][2] = fmaf(a.y, b.z, acc[1][2]); acc[1][3] = fmaf(a.y, b.w, acc[1][3]);
          acc[2][0] = fmaf(a.z, b.x, acc[2][0]); acc[2][1] = fmaf(a.z, b.y, acc[2][1]); acc[2][2] = fmaf(a.z, b.z, acc[2][2]); acc[2][3] = fmaf(a.z, b.w, acc[2][3]);
          acc[3][0] = fmaf(a.w, b.x, acc[3][0]); acc[3][1] = fmaf(a.w, b.y, acc[3][1]); acc[3][2] = fmaf(a.w, b.z, acc[3][2]); acc[3][3] = fmaf(a.w, b.w, acc[3][3]);
        }
#pragma unroll
        for (int a = 0; a < 4; ++a) accs[a * 256 + tid] = make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
      }
    } else {
      // unit u: columns 4 cg .. 4 cg + 3 of rows q, q + 32, q + 64, q + 96
      for (int u = tid - 256; u < 32 * CG; u += SBB_THREADS - 256) {
        const int cg = u % CG, q = u / CG;
        float d[4][4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int c = 0; c < 4; ++c) d[j][c] = 0.f;
#pragma unroll 1
        for (int k = 0; k < H; k += 4) {
          float4 w[4];
#pragma unroll
          for (int s = 0; s < 4; ++s) w[s] = *reinterpret_cast<const float4*>(Ws + (k + s) * H + cg * 4);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 a = *reinterpret_cast<const float4*>(yt + (q + 32 * j) * P + k);
            d[j][0] = fmaf(a.x, w[0].x, d[j][0]); d[j][1] = fmaf(a.x, w[0].y, d[j][1]);
            d[j][2] = fmaf(a.x, w[0].z, d[j][2]); d[j][3] = fmaf(a.x, w[0].w, d[j][3]);
            d[j][0] = fmaf(a.y, w[1].x, d[j][0]); d[j][1] = fmaf(a.y, w[1].y, d[j][1]);
            d[j][2] = fmaf(a.y, w[1].z, d[j][2]); d[j][3] = fmaf(a.y, w[1].w, d[j][3]);
            d[j][0] = fmaf(a.z, w[2].x, d[j][0]); d[j][1] = fmaf(a.z, w[2].y, d[j][1]);
            d[j][2] = fmaf(a.z, w[2].z, d[j][2]); d[j][3] = fmaf(a.z, w[2].w, d[j][3]);
            d[j][0] = fmaf(a.w, w[3].x, d[j][0]); d[j][1] = fmaf(a.w, w[3].y, d[j][1]);
            d[j][2] = fmaf(a.w, w[3].z, d[j][2]); d[j][3] = fmaf(a.w, w[3].w, d[j][3]);
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int r = q + 32 * j;
          if (r >= rows) continue;
          float o[4];
#pragma unroll
          for (int c = 0; c < 4; ++c) o[c] = d[j][c] + 0.f;     // the bias-less add of k_linear_fwd_dense (-0 -> +0)
          const int g = rg[r];
          if (g >= 0) {
            const float* dzg = dz + (int64_t)g * dz_stride + cg * 4;
            const float4 gm = __ldg(reinterpret_cast<const float4*>(dzg));
            const float4 gd = __ldg(reinterpret_cast<const float4*>(dzg + H));
            const int4 am = __ldg(reinterpret_cast<const int4*>(argmax + (int64_t)g * H + cg * 4));
            const float nf = rn[r];
            const int row = r0 + r;
            o[0] = (gd.x / nf + (am.x == row ? gm.x : 0.f)) + o[0];
            o[1] = (gd.y / nf + (am.y == row ? gm.y : 0.f)) + o[1];
            o[2] = (gd.z / nf + (am.z == row ? gm.z : 0.f)) + o[2];
            o[3] = (gd.w / nf + (am.w == row ? gm.w : 0.f)) + o[3];
          }
          *reinterpret_cast<float4*>(dxg + (size_t)(r0 + r) * H + cg * 4) = make_float4(o[0], o[1], o[2], o[3]);
        }
      }
    }
    __syncthreads();
    buf ^= 1;
  }
  // combine the row groups in index order through shared memory (reuse the staging buffers)
  float* red = Xs;                                    // [GROUPS][H * H]
  if (dw_thread) {
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const float4 v = accs[a * 256 + tid];
      const float vals[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int b = 0; b < 4; ++b) red[grp * H * H + (kb * 4 + a) * H + mb * 4 + b] = vals[b];
    }
  }
  __syncthreads();
  float* mypart = part + (size_t)blockIdx.x * H * H;
  for (int i = tid; i < H * H; i += SBB_THREADS) {
    float t = red[i];
    for (int g2 = 1; g2 < GROUPS; ++g2) t += red[g2 * H * H + i];
    mypart[i] = t;
  }
}

// ------------------------------------------------------------------------------------------
// Narrow outputs (M <= 4: SAGPool's score layer is F -> 1): GEMV-shaped, pure streaming of X.
//   fwd : LPR = K/4 lanes read one row as float4s, M dot products, width-LPR shuffle reduction.
//   dW  : the same lanes keep acc[4][M] for their 4 feature rows over the CTA's row range; row groups
//         are combined through shared memory in index order, CTAs by the fixed-grid second stage.
// ------------------------------------------------------------------------------------------
template <int LPR>
__global__ void __launch_bounds__(256)
k_linear_fwd_small(const float* __restrict__ X, const float* __restrict__ W, const float* __restrict__ bias,
                   float* __restrict__ Y, int N, int K, int M, int w_transposed) {
  pdl_wait();
  pdl_launch_dependents();
  __shared__ float Ws[4][512];                   // [m][k], K <= 512
  for (int i = threadIdx.x; i < M * K; i += 256) {
    int m = i / K, k = i - m * K;
    Ws[m][k] = w_transposed ? W[(size_t)m * K + k] : W[(size_t)k * M + m];
  }
  __syncthreads();
  const int l = threadIdx.x % LPR;
  const int K4 = K >> 2;
  const int groups = 256 / LPR;
  const int iters = (N + gridDim.x * groups - 1) / (gridDim.x * groups);      // warp-uniform trip count
  for (int it = 0; it < iters; ++it) {
    const int r = (it * gridDim.x + blockIdx.x) * groups + threadIdx.x / LPR;
    const bool rok = r < N;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    if (rok) {
      const float4* xr = reinterpret_cast<const float4*>(X + (size_t)r * K);
      for (int k4 = l; k4 < K4; k4 += LPR) {
        const float4 x = __ldg(xr + k4);
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          if (m < M) {
            const float* w = &Ws[m][k4 * 4];
            acc[m] = fmaf(x.x, w[0], acc[m]); acc[m] = fmaf(x.y, w[1], acc[m]);
            acc[m] = fmaf(x.z, w[2], acc[m]); acc[m] = fmaf(x.w, w[3], acc[m]);
          }
        }
      }
    }
#pragma unroll
    for (int m = 0; m < 4; ++m)
#pragma unroll
      for (int d = LPR / 2; d > 0; d >>= 1) acc[m] += __shfl_xor_sync(0xffffffffu, acc[m], d, LPR);
    if (rok && l == 0)
      for (int m = 0; m < M; ++m) Y[(size_t)r * M + m] = acc[m] + (bias ? bias[m] : 0.f);
  }
}

template <int LPR>
__global__ void __launch_bounds__(256)
k_linear_bwd_weight_small(const float* __restrict__ X, const float* __restrict__ dY, float* __restrict__ part,
                          int N, int K, int M, float* __restrict__ dW, unsigned* ticket) {
  pdl_wait();
  pdl_launch_dependents();
  extern __shared__ __align__(16) float smem[];            // [groups][K*M] for the in-CTA combine
  const int l = threadIdx.x % LPR, grp = threadIdx.x / LPR;
  const int groups = 256 / LPR;
  const int K4 = K >> 2;
  const int rows_per_cta = (N + gridDim.x - 1) / gridDim.x;
  const int r_begin = blockIdx.x * rows_per_cta, r_end = min(N, r_begin + rows_per_cta);
  // a lane owns k4 = l (and l + LPR, ... when K4 > LPR is not supported: K <= 4*LPR)
  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int m = 0; m < 4; ++m) acc[a][m] = 0.f;
  const bool lok = l < K4;
  for (int rb = r_begin + grp; rb < r_end; rb += groups * 4) {
    float4 xv[4]; float dv[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int r = rb + u * groups;
      const bool rok = r < r_end;
      xv[u] = (rok && lok) ? __ldg(reinterpret_cast<const float4*>(X + (size_t)r * K) + l) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int m = 0; m < 4; ++m) dv[u][m] = (rok && m < M) ? __ldg(dY + (size_t)r * M + m) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        acc[0][m] = fmaf(xv[u].x, dv[u][m], acc[0][m]); acc[1][m] = fmaf(xv[u].y, dv[u][m], acc[1][m]);
        acc[2][m] = fmaf(xv[u].z, dv[u][m], acc[2][m]); acc[3][m] = fmaf(xv[u].w, dv[u][m], acc[3][m]);
      }
  }
  if (lok)
    for (int a = 0; a < 4; ++a)
      for (int m = 0; m < M; ++m) smem[(size_t)grp * K * M + (size_t)(l * 4 + a) * M + m] = acc[a][m];
  __syncthreads();
  float* mypart = part + (size_t)blockIdx.x * K * M;
  for (int i = threadIdx.x; i < K * M; i += 256) {
    float sacc = smem[i];
    for (int g = 1; g < groups; ++g) sacc += smem[(size_t)g * K * M + i];
    mypart[i] = sacc;
  }
  if (ticket) partial_sum_tail(part, dW, K * M, nullptr, gridDim.x, K * M, ticket);
}

// lanes per row: enough for M columns (4 per lane) and few enough rows per tile that the X tile
// (R = 256/cg*2 rows x K floats) stays below ~64 KB of shared memory
static int pick_cg(int64_t M, int64_t K) {
  int c = 1;
  while (c * 4 < M && c < 32) c <<= 1;
  while (c < 32 && (size_t)(LIN_THREADS / c) * LIN_RPT * (size_t)lin_pitch((int)K) * 4 > 64 * 1024) c <<= 1;
  return c;
}

constexpr int LIN_KBLOCK = 256;       // K block of k_linear_fwd where W's whole slab does not fit

static size_t lin_smem_bytes(int cg, int64_t K) {
  int R = (LIN_THREADS / cg) * LIN_RPT;
  return ((size_t)K * cg * 4 + 2 * (size_t)R * lin_pitch((int)K)) * sizeof(float);      // W + two X tiles
}

}  // namespace tsg

using namespace tsg;

template <typename Kern>
static int set_smem(Kern kern, size_t bytes, const char* what) {
  if (bytes > 227 * 1024) { set_error("%s: needs %zu B of shared memory (> 227 KB): K*M too large", what, bytes); return TSG_EINVAL; }
  if (bytes > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) { set_error("%s: cudaFuncSetAttribute: %s", what, cudaGetErrorString(e)); return TSG_ELAUNCH; }
  }
  return TSG_OK;
}

extern "C" int tsg_linear_fwd(const float* X, const float* W, const float* bias, float* Y,
                              int64_t N, int64_t K, int64_t M, int w_transposed, int flags, void* stream) {
  TSG_REQUIRE(N >= 0 && K > 0 && M > 0, "linear_fwd: bad shape");
  TSG_REQUIRE(M <= 128 || flags == 0, "linear_fwd: the fused epilogue needs out_feat <= 128 (got %lld)", (long long)M);
  TSG_REQUIRE(N < (int64_t)0x7fffffff / (K > M ? K : M), "linear_fwd: N*K overflows int32 tiles");
  if (N == 0) return TSG_OK;
  TSG_REQUIRE(X && W && Y, "linear_fwd: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (M <= 4 && flags == 0 && (K & 3) == 0 && K <= 128 && (((uintptr_t)X) & 15) == 0) {   // GEMV-shaped
    int lpr = 1; while (lpr * 4 < K) lpr <<= 1;
    int grid = grid_for(N, 256 / lpr, 16);
#define TSG_GOS(L) TSG_LAUNCH_PDL("linear_fwd(small)", k_linear_fwd_small<L>, grid, 256, 0, st, X, W, bias, Y, (int)N, (int)K, (int)M, w_transposed)
    switch (lpr) {
      case 1: TSG_GOS(1); break; case 2: TSG_GOS(2); break; case 4: TSG_GOS(4); break;
      case 8: TSG_GOS(8); break; case 16: TSG_GOS(16); break; default: TSG_GOS(32); break;
    }
#undef TSG_GOS
    return check_launch("linear_fwd(small)");
  }
  // output columns are produced in chunks of <= 128 (one float4 per lane, 32 lanes per row)
  for (int64_t m0 = 0; m0 < M; m0 += 128) {
    int64_t mc = M - m0 < 128 ? M - m0 : 128;
    int cg = pick_cg(mc, K);
    const float* Wc = w_transposed ? W + m0 * K : W + m0;
    int ldw = w_transposed ? (int)K : (int)M;
    const float* bc = bias ? bias + m0 : nullptr;
    float* Yc = Y + m0;
    int rc;
    static const bool no_dense = getenv("TSG_LIN_NODENSE") != nullptr;
    const size_t smem_d = ((size_t)K * cg * 4 + 2 * (size_t)(LIN_THREADS / cg) * LIND_RPT * (K + 4)) * sizeof(float);
    if (!no_dense && (K & 3) == 0 && (((uintptr_t)X) & 15) == 0 && smem_d <= 160 * 1024) {
      int Rd = (LIN_THREADS / cg) * LIND_RPT;
      int tiles_d = (int)((N + Rd - 1) / Rd);
      int grid_d = tiles_d < TSG_NUM_SMS * 4 ? tiles_d : TSG_NUM_SMS * 4;
#define TSG_GOD(C)                                                                                  \
      rc = set_smem(k_linear_fwd_dense<C>, smem_d, "linear_fwd(dense)"); if (rc) return rc;           \
      TSG_LAUNCH_PDL("linear_fwd(dense)", k_linear_fwd_dense<C>, grid_d, LIN_THREADS, smem_d, st, X, Wc, bc, Yc, (int)N, (int)K, (int)mc, ldw, \
                     (int)M, w_transposed, flags)
      switch (cg) {
        case 1: TSG_GOD(1); break; case 2: TSG_GOD(2); break; case 4: TSG_GOD(4); break;
        case 8: TSG_GOD(8); break; case 16: TSG_GOD(16); break; default: TSG_GOD(32); break;
      }
#undef TSG_GOD
      continue;
    }
    // W's slab [K][4 cg] and two X tiles in shared memory; a K beyond that (the input gradient of a classifier layer
    // with ~1,000 classes) runs in blocks of LIN_KBLOCK -- shapes that fit keep their single launch
    const int64_t kb = lin_smem_bytes(cg, K) <= 227 * 1024 ? K : LIN_KBLOCK;
    for (int64_t k0 = 0; k0 < K; k0 += kb) {
      const int64_t kc = K - k0 < kb ? K - k0 : kb;
      const int cgb = kb == K ? cg : pick_cg(mc, kc);
      const int kmode = (k0 > 0 ? LIN_KACC_IN : 0) | (k0 + kc < K ? LIN_KPARTIAL : 0);
      const float* Wb = w_transposed ? Wc + k0 : Wc + k0 * ldw;
      size_t smem = lin_smem_bytes(cgb, kc);
      int R = (LIN_THREADS / cgb) * LIN_RPT;
      int tiles = (int)((N + R - 1) / R);
      int grid = tiles < TSG_NUM_SMS * 4 ? tiles : TSG_NUM_SMS * 4;
#define TSG_GO(C)                                                                                  \
      rc = set_smem(k_linear_fwd<C>, smem, "linear_fwd"); if (rc) return rc;                        \
      TSG_LAUNCH_PDL("linear_fwd", k_linear_fwd<C>, grid, LIN_THREADS, smem, st, X + k0, Wb, bc, Yc, (int)N, (int)kc, (int)mc, \
                     ldw, (int)M, w_transposed, flags, (int)K, kmode)
      switch (cgb) {
        case 1: TSG_GO(1); break; case 2: TSG_GO(2); break; case 4: TSG_GO(4); break;
        case 8: TSG_GO(8); break; case 16: TSG_GO(16); break; default: TSG_GO(32); break;
      }
#undef TSG_GO
    }
  }
  return check_launch("linear_fwd");
}

extern "C" int tsg_dense_epilogue_bwd(const float* X, const float* W, const float* bias, const float* dO,
                                      float* dU, int64_t N, int64_t K, int64_t M, int flags, void* stream) {
  TSG_REQUIRE(N >= 0 && K > 0 && M > 0 && M <= 128, "dense_epilogue_bwd: bad shape");
  if (N == 0) return TSG_OK;
  TSG_REQUIRE(X && W && dO && dU, "dense_epilogue_bwd: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  int cg = pick_cg(M, K);
  size_t smem = lin_smem_bytes(cg, K);
  int R = (LIN_THREADS / cg) * LIN_RPT;
  int tiles = (int)((N + R - 1) / R);
  int grid = tiles < TSG_NUM_SMS * 4 ? tiles : TSG_NUM_SMS * 4;
  int rc;
#define TSG_GO(C)                                                                                  \
  rc = set_smem(k_dense_epilogue_bwd<C>, smem, "dense_epilogue_bwd"); if (rc) return rc;            \
  k_dense_epilogue_bwd<C><<<grid, LIN_THREADS, smem, st>>>(X, W, bias, dO, dU, (int)N, (int)K, (int)M, flags)
  switch (cg) {
    case 1: TSG_GO(1); break; case 2: TSG_GO(2); break; case 4: TSG_GO(4); break;
    case 8: TSG_GO(8); break; case 16: TSG_GO(16); break; default: TSG_GO(32); break;
  }
#undef TSG_GO
  return check_launch("dense_epilogue_bwd");
}

extern "C" size_t tsg_colsum_workspace_bytes(int64_t N, int64_t F);
extern "C" int tsg_relu_bwd_colsum(const float* dY, const float* Y, float* dYm, float* dbias, int64_t N,
                                   int64_t F, void* workspace, size_t workspace_bytes, void* stream);

extern "C" size_t tsg_linear_bwd_weight_workspace_bytes(int64_t K, int64_t M) {
  return ws_bytes((size_t)LBW_GRID * (size_t)K * (size_t)M, 4) + tsg_colsum_workspace_bytes(1 << 30, M) + 512;
}

extern "C" int tsg_linear_bwd_weight(const float* X, const float* dY, float* dW, float* db,
                                     int64_t N, int64_t K, int64_t M,
                                     void* workspace, size_t workspace_bytes, void* stream) {
  TSG_REQUIRE(N >= 0 && K > 0 && M > 0, "linear_bwd_weight: bad shape");
  TSG_REQUIRE(X && dY && (dW || db), "linear_bwd_weight: null pointer");
  TSG_REQUIRE(N < (int64_t)0x7fffffff, "linear_bwd_weight: too many rows");
  if (workspace_bytes < tsg_linear_bwd_weight_workspace_bytes(K, M)) { set_error("linear_bwd_weight: workspace too small"); return TSG_EWORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  float* part = ws.take<float>((size_t)LBW_GRID * K * M);
  size_t cs_bytes = tsg_colsum_workspace_bytes(1 << 30, M);
  char* cs_ws = ws.take<char>(cs_bytes);
  if (db) {
    int rc = tsg_relu_bwd_colsum(dY, nullptr, nullptr, db, N, M, cs_ws, cs_bytes, stream);
    if (rc) return rc;
  }
  if (!dW) return TSG_OK;
  if (M <= 4 && (K & 3) == 0 && K <= 128 && (((uintptr_t)X) & 15) == 0) {                 // GEMV-shaped
    int lpr = 1; while (lpr * 4 < K) lpr <<= 1;
    int groups = 256 / lpr;
    size_t smem_s = (size_t)groups * K * M * sizeof(float);
    if (smem_s <= 200 * 1024) {
      int grid = LBW_GRID;
      unsigned* ticket = fused_tail_ok(grid, K * M) ? ticket_next() : nullptr;
#define TSG_GOS(L)                                                                                          \
      { int rc = set_smem(k_linear_bwd_weight_small<L>, smem_s, "linear_bwd_weight(small)"); if (rc) return rc; \
        TSG_LAUNCH_PDL("linear_bwd_weight(small)", k_linear_bwd_weight_small<L>, grid, 256, smem_s, st, X, dY, part, (int)N, (int)K, (int)M, dW, ticket); }
      switch (lpr) {
        case 1: TSG_GOS(1) break; case 2: TSG_GOS(2) break; case 4: TSG_GOS(4) break;
        case 8: TSG_GOS(8) break; case 16: TSG_GOS(16) break; default: TSG_GOS(32) break;
      }
#undef TSG_GOS
      if (!ticket) { int rc = launch_partial_sum_final(part, dW, (int)(K * M), nullptr, grid, (int)(K * M), st); if (rc) return rc; }
      return check_launch("linear_bwd_weight(small)");
    }
  }
  static const bool no_dense = getenv("TSG_LIN_NODENSE") != nullptr;
  if (!no_dense && (K & 3) == 0 && (M & 3) == 0 && (K / 4) * (M / 4) <= 256 && M > 4 &&
      ((((uintptr_t)X) | ((uintptr_t)dY)) & 15) == 0) {
    size_t smem_d = (size_t)2 * LBWD_ROWS * (K + M) * sizeof(float);
    const size_t red = (size_t)(256 / ((K / 4) * (M / 4))) * K * M * sizeof(float);
    if (red > smem_d) smem_d = red;
    if (smem_d <= 200 * 1024) {
      int rc = set_smem(k_linear_bwd_weight_dense, smem_d, "linear_bwd_weight(dense)"); if (rc) return rc;
      TSG_LAUNCH_PDL("linear_bwd_weight(dense)", k_linear_bwd_weight_dense, LBW_GRID, 256, smem_d, st, X, dY, part, (int)N, (int)K, (int)M);
      rc = launch_partial_sum_final(part, dW, (int)(K * M), nullptr, LBW_GRID, (int)(K * M), st); if (rc) return rc;
      return check_launch("linear_bwd_weight(dense)");
    }
  }
  // blocks of <= 256 input columns (one block up to 256; more for the 2 * nhid inputs of the head's lin1 from nhid 130),
  // each the kernel's [kc][32] accumulators -- dW rows [k0, k0 + kc) are contiguous, and every entry keeps its order
  const int grid = LBW_GRID;                 // fixed => the summation order never depends on the device
  for (int64_t k0 = 0; k0 < K; k0 += 256) {
    const int64_t kc = K - k0 < 256 ? K - k0 : 256;
    int nk = (int)((kc + 31) / 32);
    int nwarps = 8;
    while (nwarps > 1 && (size_t)nwarps * kc * 32 * 4 > 200 * 1024) --nwarps;
    size_t smem = (size_t)nwarps * kc * 32 * sizeof(float);
    for (int m0 = 0; m0 < M; m0 += 32) {
#define TSG_GO(NK_, U_)                                                                                    \
      { int rc = set_smem(k_linear_bwd_weight<NK_, U_>, smem, "linear_bwd_weight"); if (rc) return rc;       \
        TSG_LAUNCH_PDL("linear_bwd_weight", k_linear_bwd_weight<NK_, U_>, grid, nwarps * 32, smem, st, X + k0, dY, part, (int)N, (int)kc, \
                       (int)M, m0, (int)K); }
      switch (nk) {
        case 1: TSG_GO(1, 8); break; case 2: TSG_GO(2, 8); break; case 3: TSG_GO(3, 4); break;
        case 4: TSG_GO(4, 4); break; case 5: TSG_GO(5, 2); break; case 6: TSG_GO(6, 2); break;
        case 7: TSG_GO(7, 2); break; default: TSG_GO(8, 2); break;
      }
#undef TSG_GO
    }
    int rc = launch_partial_sum_final(part, dW + k0 * M, (int)(kc * M), nullptr, grid, (int)(kc * M), st);
    if (rc) return rc;
  }
  return check_launch("linear_bwd_weight");
}

extern "C" int tsg_sag_boundary_bwd(const float* dxw, const float* x, const float* W, const float* dz, int64_t dz_stride,
                                    const int32_t* argmax, const int64_t* graph_ptr, int64_t G, int64_t N, int64_t H,
                                    float* dxg, float* dW, void* workspace, size_t workspace_bytes, void* stream) {
  TSG_REQUIRE(H % 4 == 0 && H >= 8 && H <= 64, "sag_boundary_bwd: hidden %lld is not a multiple of 4 in [8, 64]", (long long)H);
  TSG_REQUIRE(N >= 0 && G >= 0 && N < (int64_t)0x7fffffff && G < (int64_t)0x7fffffff, "sag_boundary_bwd: bad shape");
  TSG_REQUIRE(dz_stride >= 2 * H && dz_stride % 4 == 0, "sag_boundary_bwd: dz stride %lld must be >= 2 * hidden and a multiple of 4",
              (long long)dz_stride);
  TSG_REQUIRE(W && dW && graph_ptr && (N == 0 || (dxw && x && dxg)) && (G == 0 || (dz && argmax)), "sag_boundary_bwd: null pointer");
  TSG_REQUIRE(((((uintptr_t)dxw) | ((uintptr_t)x) | ((uintptr_t)dxg) | ((uintptr_t)dz) | ((uintptr_t)argmax)) & 15) == 0,
              "sag_boundary_bwd: dxw, x, dxg, dz and argmax must be 16-byte aligned");
  if (workspace_bytes < ws_bytes((size_t)LBW_GRID * H * H, 4)) { set_error("sag_boundary_bwd: workspace too small"); return TSG_EWORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  float* part = (float*)workspace;
  const size_t smem = sbb_smem_bytes((int)H);
  int rc;
#define TSG_GO(H_)                                                                                                        \
  case H_:                                                                                                                \
    rc = set_smem(k_sag_boundary_bwd<H_>, smem, "sag_boundary_bwd"); if (rc) return rc;                                  \
    TSG_LAUNCH_PDL("sag_boundary_bwd", k_sag_boundary_bwd<H_>, LBW_GRID, SBB_THREADS, smem, st, dxw, x, W, dz, dz_stride, \
                   argmax, graph_ptr, (int)G, (int)N, dxg, part);                                                         \
    break;
  switch (H) {
    TSG_GO(8) TSG_GO(12) TSG_GO(16) TSG_GO(20) TSG_GO(24) TSG_GO(28) TSG_GO(32) TSG_GO(36)
    TSG_GO(40) TSG_GO(44) TSG_GO(48) TSG_GO(52) TSG_GO(56) TSG_GO(60) TSG_GO(64)
  }
#undef TSG_GO
  rc = launch_partial_sum_final(part, dW, (int)(H * H), nullptr, LBW_GRID, (int)(H * H), st); if (rc) return rc;
  return check_launch("sag_boundary_bwd");
}


// Row-softmax backward from the SAVED output: dL = S * (dS - rowsum(S * dS)).  Warp per row.  (The epilogue backward
// above could recompute S from the logits, but that re-does the 164 x 100 product of DiffPool's assignment layer:
// +1 ms per step measured; the forward already wrote S.)
namespace tsg {
__global__ void __launch_bounds__(256)
k_softmax_bwd(const float* __restrict__ S, const float* __restrict__ dS, float* __restrict__ dL, int64_t N, int M) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = warp; r < N; r += nwarps) {
    const float* s = S + r * M; const float* g = dS + r * M;
    float dot = 0.f;
    for (int c = lane; c < M; c += 32) dot = fmaf(s[c], g[c], dot);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
    for (int c = lane; c < M; c += 32) dL[r * M + c] = s[c] * (g[c] - dot);
  }
}
}  // namespace tsg

extern "C" int tsg_softmax_bwd(const float* S, const float* dS, float* dL, int64_t N, int64_t M, void* stream) {
  TSG_REQUIRE(N >= 0 && M > 0 && M < (int64_t)0x7fffffff, "softmax_bwd: bad shape");
  if (N == 0) return TSG_OK;
  TSG_REQUIRE(S && dS && dL, "softmax_bwd: null pointer");
  tsg::k_softmax_bwd<<<tsg::grid_for(N, 8), 256, 0, (cudaStream_t)stream>>>(S, dS, dL, N, (int)M);
  return tsg::check_launch("softmax_bwd");
}
