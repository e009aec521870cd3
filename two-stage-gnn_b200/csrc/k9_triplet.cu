// K9 -- stage-1 triplet distances, margin-ranking loss and the pairwise-distance matrix.
//
// Replaces F.pairwise_distance(embed_a, embed_p, 2) / (embed_a, embed_n, 2)
// (Code/sag/tripletnet.py:21-22; Code/sage+gat+diffpool/tripletnet.py:42-43;
// Code/eigengcn/tripletnet.py:152-153) and torch.nn.MarginRankingLoss(margin=alpha) with
// target = -1 (Code/sag/train_triplet.py:196,208-211):
//     d(a,b) = || e_a - e_b + eps ||_2           (eps is added to the DIFFERENCE)
//     loss   = mean_t max(0, (d_ap - d_an) + margin)
// Backward is deterministic: an inverted index (embedding row -> triplet slots, slot order)
// is built on the device with K1's counting sort, then one warp per embedding row sums its
// contributions sequentially.  No atomics anywhere.
#include "common.cuh"

namespace tsg {

__global__ void __launch_bounds__(256)
k_triplet_fwd(const float* __restrict__ emb, const int64_t* __restrict__ trip, int64_t T, int D,
              float margin, float eps, float* __restrict__ dpos, float* __restrict__ dneg,
              float* __restrict__ hinge) {
  pdl_wait();
  pdl_launch_dependents();
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t t = warp; t < T; t += nwarps) {
    const float* a = emb + trip[t * 3 + 0] * D;
    const float* p = emb + trip[t * 3 + 1] * D;
    const float* n = emb + trip[t * 3 + 2] * D;
    float sp = 0.f, sn = 0.f;
    for (int d = lane; d < D; d += 32) {
      float av = a[d];
      float up = av - p[d] + eps, un = av - n[d] + eps;
      sp += up * up; sn += un * un;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      sp += __shfl_xor_sync(0xffffffffu, sp, o);
      sn += __shfl_xor_sync(0xffffffffu, sn, o);
    }
    if (lane == 0) {
      float dp = sqrtf(sp), dn = sqrtf(sn);
      dpos[t] = dp; dneg[t] = dn;
      float u = (dp - dn) + margin;
      hinge[t] = u > 0.f ? u : 0.f;
    }
  }
}

// deterministic mean of T values with one block; *seed (if given) receives 1.0, the d(loss) the step's backward starts from
__global__ void __launch_bounds__(1024)
k_mean_1block(const float* __restrict__ v, int64_t T, float* __restrict__ out, float* __restrict__ seed) {
  pdl_wait();
  pdl_launch_dependents();
  __shared__ float sm[1024];
  float s = 0.f;
  for (int64_t i = threadIdx.x; i < T; i += 1024) s += v[i];
  sm[threadIdx.x] = s;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if (threadIdx.x < o) sm[threadIdx.x] += sm[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    *out = T > 0 ? sm[0] / (float)T : 0.f;
    if (seed) *seed = 1.0f;
  }
}

__global__ void k_iota64(int64_t* p, int64_t n) {
  pdl_wait();
  pdl_launch_dependents();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) p[i] = i;
}

__global__ void __launch_bounds__(256)
k_triplet_bwd(const float* __restrict__ emb, const int64_t* __restrict__ trip, int64_t T, int64_t M,
              int D, float margin, float eps, const float* __restrict__ dpos,
              const float* __restrict__ dneg, const float* __restrict__ dloss,
              const int* __restrict__ rowptr, const int* __restrict__ slots, float* __restrict__ demb) {
  pdl_wait();
  pdl_launch_dependents();
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const float gscale = dloss[0] / (float)T;
  for (int64_t m = warp; m < M; m += nwarps) {
    const int s0 = rowptr[m], s1 = rowptr[m + 1];
    for (int d = lane; d < D; d += 32) {
      float acc = 0.f;
      for (int q = s0; q < s1; ++q) {
        const int slot = slots[q];
        const int64_t t = slot / 3; const int role = slot - (int)t * 3;
        const float dp = dpos[t], dn = dneg[t];
        if (!((dp - dn) + margin >= 0.f)) continue;          // clamp_min backward: x >= 0
        const float av = emb[trip[t * 3 + 0] * D + d];
        float c = 0.f;
        if (role != 2) {       // anchor or positive: d_ap term
          float up = av - emb[trip[t * 3 + 1] * D + d] + eps;
          float gp = dp > 0.f ? up / dp : 0.f;
          c += role == 0 ? gp : -gp;
        }
        if (role != 1) {       // anchor or negative: -d_an term
          float un = av - emb[trip[t * 3 + 2] * D + d] + eps;
          float gn = dn > 0.f ? un / dn : 0.f;
          c += role == 0 ? -gn : gn;
        }
        acc += gscale * c;
      }
      demb[m * D + d] = acc;
    }
  }
}

__global__ void __launch_bounds__(256)
k_pairdist(const float* __restrict__ emb, int64_t M, int D, float eps, float* __restrict__ dist) {
  const int64_t total = M * M;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int64_t i = idx / M, j = idx - i * M;
    const float* a = emb + i * D; const float* b = emb + j * D;
    float s = 0.f;
    for (int d = 0; d < D; ++d) { float u = a[d] - b[d] + eps; s += u * u; }
    dist[idx] = sqrtf(s);
  }
}

}  // namespace tsg

using namespace tsg;

extern "C" size_t tsg_triplet_workspace_bytes(int64_t T, int64_t M, int64_t D) {
  (void)D;
  size_t b = ws_bytes((size_t)T + 1, 4);                 // hinge
  b += ws_bytes((size_t)3 * T + 1, 8);                   // slot iota
  b += ws_bytes((size_t)M + 2, 4);                       // rowptr
  b += 2 * ws_bytes((size_t)3 * T + 1, 4);               // slots, val
  b += tsg_csr_build_workspace_bytes(3 * T, M);
  return b + 1024;
}

int tsg::triplet_fwd(const float* emb, const int64_t* trip, int64_t T, int64_t M, int64_t D, float margin, float eps,
                     float* dpos, float* dneg, float* loss, float* dloss_seed, void* workspace, size_t workspace_bytes,
                     void* stream) {
  TSG_REQUIRE(T >= 0 && M >= 0 && D > 0, "triplet_fwd: bad shape");
  TSG_REQUIRE(loss && (T == 0 || (emb && trip && dpos && dneg)), "triplet_fwd: null pointer");
  if (workspace_bytes < tsg_triplet_workspace_bytes(T, M, D)) { set_error("triplet_fwd: workspace too small"); return TSG_EWORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  float* hinge = ws.take<float>(T + 1);
  if (T > 0) TSG_LAUNCH_PDL("triplet_fwd", k_triplet_fwd, grid_for(T, 8), 256, 0, st, emb, trip, T, (int)D, margin, eps, dpos, dneg, hinge);
  return launch_pdl("triplet_fwd(mean)", k_mean_1block, 1, 1024, 0, st, (const float*)hinge, T, loss, dloss_seed);
}

extern "C" int tsg_triplet_fwd(const float* emb, const int64_t* trip, int64_t T, int64_t M, int64_t D,
                               float margin, float eps, float* dpos, float* dneg, float* loss,
                               void* workspace, size_t workspace_bytes, void* stream) {
  return triplet_fwd(emb, trip, T, M, D, margin, eps, dpos, dneg, loss, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int tsg_triplet_bwd(const float* emb, const int64_t* trip, int64_t T, int64_t M, int64_t D,
                               float margin, float eps, const float* dpos, const float* dneg,
                               const float* dloss, float* demb,
                               void* workspace, size_t workspace_bytes, void* stream) {
  TSG_REQUIRE(T >= 0 && M >= 0 && D > 0, "triplet_bwd: bad shape");
  if (M == 0) return TSG_OK;
  TSG_REQUIRE(emb && demb && dloss && (T == 0 || (trip && dpos && dneg)), "triplet_bwd: null pointer");
  if (workspace_bytes < tsg_triplet_workspace_bytes(T, M, D)) { set_error("triplet_bwd: workspace too small"); return TSG_EWORKSPACE; }
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  ws.take<float>(T + 1);
  int64_t* iota = ws.take<int64_t>(3 * T + 1);
  int* rowptr = ws.take<int>(M + 2);
  int* slots = ws.take<int>(3 * T + 1);
  float* val = ws.take<float>(3 * T + 1);
  size_t csr_ws_bytes = tsg_csr_build_workspace_bytes(3 * T, M);
  char* csr_ws = ws.take<char>(csr_ws_bytes);
  if (!ws.ok()) { set_error("triplet_bwd: workspace carve failed"); return TSG_EWORKSPACE; }
  if (T > 0) TSG_LAUNCH_PDL("triplet_bwd(iota)", k_iota64, grid_for(3 * T, 256), 256, 0, st, iota, 3 * T);
  // inverted index: "edge" slot -> embedding row, grouped by embedding row in slot order
  int rc = tsg_csr_build(iota, trip, nullptr, 3 * T, nullptr, M, TSG_CSR_RAW, rowptr, slots, val, nullptr,
                         nullptr, nullptr, nullptr, nullptr, csr_ws, csr_ws_bytes, stream);
  if (rc) return rc;
  return launch_pdl("triplet_bwd", k_triplet_bwd, grid_for(M, 8), 256, 0, st, emb, trip, T, M, (int)D, margin, eps, dpos, dneg, dloss,
                    (const int*)rowptr, (const int*)slots, demb);
}

extern "C" int tsg_pairdist_matrix(const float* emb, int64_t M, int64_t D, float eps, float* dist, void* stream) {
  TSG_REQUIRE(M >= 0 && D > 0, "pairdist_matrix: bad shape");
  if (M == 0) return TSG_OK;
  TSG_REQUIRE(emb && dist, "pairdist_matrix: null pointer");
  k_pairdist<<<grid_for(M * M, 256), 256, 0, (cudaStream_t)stream>>>(emb, M, (int)D, eps, dist);
  return check_launch("pairdist_matrix");
}
