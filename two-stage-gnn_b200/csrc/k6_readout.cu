// K6 -- per-graph readouts (segment max with arg-max, mean, sum), forward and backward.
//
// Replaces torch.cat([global_max_pool(x,batch), global_mean_pool(x,batch)],1) of
// Code/sag/network.py:36,40,44 (torch-scatter atomics + a batch.max().item() sync upstream) and
// the torch.max(x, dim=1) readouts of Code/sage+gat+diffpool/encoders.py:183,190,197,353,383.
//
// One warp per graph.  A row is covered by LPR lanes x VEC floats (128-bit loads when F%4==0);
// the 32/LPR lane groups stride over the graph's rows so a warp keeps 32/LPR independent
// row loads in flight; groups are combined with xor-shuffles in a fixed order (deterministic).
// Max ties resolve to the FIRST (lowest) row, the torch-scatter CPU rule; the backward routes
// the max gradient to that row only.  Streaming, HBM-bound: x is read once, dx written once.
#include "common.cuh"
#include <float.h>

namespace tsg {

constexpr int RO_THREADS = 128;   // 4 graphs per block
constexpr int RO_U = 8;            // k_readout_fwd: rows per lane group in flight
constexpr int RO_BWD_THREADS = 256;

template <int VEC, int LPR>
__global__ void __launch_bounds__(RO_THREADS)
k_readout_fwd(const float* __restrict__ x, const int64_t* __restrict__ gptr, int G, int F, int mode,
              float* __restrict__ out, int64_t out_stride, int* __restrict__ argmax) {
  pdl_wait();
  pdl_launch_dependents();
  constexpr int RPW = 32 / LPR;
  const int lane = threadIdx.x & 31;
  const int sub = lane / LPR, l = lane % LPR;
  const int FV = F / VEC;
  const int warps_per_block = RO_THREADS / 32;
  for (int g = blockIdx.x * warps_per_block + (threadIdx.x >> 5); g < G;
       g += gridDim.x * warps_per_block) {
    const int64_t lo = gptr[g], hi = gptr[g + 1];
    const int n = (int)(hi - lo);
    for (int fb = 0; fb < FV; fb += LPR) {           // warp-uniform trip count
      const int f = fb + l;
      const bool fok = f < FV;
      float mx[VEC], sm[VEC]; int am[VEC];
#pragma unroll
      for (int v = 0; v < VEC; ++v) { mx[v] = -FLT_MAX; sm[v] = 0.f; am[v] = -1; }
      if (fok) {
        int i = sub;
        if (VEC == 4) {
          // RO_U rows per sub-group in flight (the loads do not depend on the sums): a graph's walk is RO_U times
          // shorter -- the launch lasts as long as its largest graph.  Same order of additions as the plain loop below.
          for (; i + (RO_U - 1) * RPW < n; i += RO_U * RPW) {
            float4 t[RO_U];
#pragma unroll
            for (int u = 0; u < RO_U; ++u) t[u] = __ldg(reinterpret_cast<const float4*>(x) + (lo + i + u * RPW) * FV + f);
#pragma unroll
            for (int u = 0; u < RO_U; ++u) {
              const float vals[4] = {t[u].x, t[u].y, t[u].z, t[u].w};
#pragma unroll
              for (int v = 0; v < VEC; ++v) {
                sm[v] += vals[v % 4];
                if (vals[v % 4] > mx[v] || am[v] < 0) { mx[v] = vals[v % 4]; am[v] = i + u * RPW; }
              }
            }
          }
        }
        for (; i < n; i += RPW) {
          float vals[VEC];
          if (VEC == 4) {
            float4 t = __ldg(reinterpret_cast<const float4*>(x) + (lo + i) * FV + f);
            vals[0] = t.x; vals[1 % VEC] = t.y; vals[2 % VEC] = t.z; vals[3 % VEC] = t.w;
          } else {
            vals[0] = __ldg(x + (lo + i) * FV + f);
          }
#pragma unroll
          for (int v = 0; v < VEC; ++v) {
            sm[v] += vals[v];
            if (vals[v] > mx[v] || am[v] < 0) { mx[v] = vals[v]; am[v] = i; }
          }
        }
      }
      // combine the RPW sub-groups (all 32 lanes participate)
#pragma unroll
      for (int d = LPR; d < 32; d <<= 1) {
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          float omx = __shfl_xor_sync(0xffffffffu, mx[v], d);
          int oam = __shfl_xor_sync(0xffffffffu, am[v], d);
          float osm = __shfl_xor_sync(0xffffffffu, sm[v], d);
          // sum: fixed pairing => deterministic; both partners compute the same value
          sm[v] = (sub & (d / LPR)) ? osm + sm[v] : sm[v] + osm;
          bool take = oam >= 0 && (am[v] < 0 || omx > mx[v] || (omx == mx[v] && oam < am[v]));
          if (take) { mx[v] = omx; am[v] = oam; }
        }
      }
      if (fok && sub == 0) {
        int col = 0;
        if (mode & TSG_READOUT_MAX) {
#pragma unroll
          for (int v = 0; v < VEC; ++v) {
            out[(int64_t)g * out_stride + f * VEC + v] = am[v] >= 0 ? mx[v] : 0.f;
            if (argmax) argmax[(int64_t)g * F + f * VEC + v] = am[v] >= 0 ? (int)(lo + am[v]) : -1;
          }
          col = F;
        }
        if (mode & (TSG_READOUT_MEAN | TSG_READOUT_SUM)) {
          float inv = (mode & TSG_READOUT_MEAN) ? 1.f / (float)(n > 0 ? n : 1) : 1.f;
#pragma unroll
          for (int v = 0; v < VEC; ++v) {
            float r = (mode & TSG_READOUT_MEAN) ? sm[v] / (float)(n > 0 ? n : 1) : sm[v];
            (void)inv;
            out[(int64_t)g * out_stride + col + f * VEC + v] = r;
          }
        }
      }
    }
  }
}

// SAGPool gate + readout in one pass (K10 executor, F % 4 == 0): row i of graph g is
//     xo[lo + i] = x[perm[lo + i]] * tanh(score[perm[lo + i]])                 layers.py:21
// written once and reduced on the fly into [gmp || gap] (network.py:36,40,44) -- the gated rows are not read back.
// Same reduction order as k_readout_fwd<4, LPR> (sub-group s takes rows s, s + RPW, ... in order, then the fixed
// butterfly) and the same products as k_gate_gather_fwd<4>: out, argmax and xo are bit-identical to the two-kernel
// sequence.  GRO_U row batches per sub-group are loaded before any is reduced (perm -> score / x is a dependent chain).
constexpr int GRO_U = 4;

template <int LPR>
__global__ void __launch_bounds__(RO_THREADS)
k_gate_readout_fwd(const float4* __restrict__ x, const float* __restrict__ score, const int64_t* __restrict__ perm,
                   const int64_t* __restrict__ gptr, int G, int F4, float4* __restrict__ xo,
                   float* __restrict__ out, int64_t out_stride, int* __restrict__ argmax) {
  pdl_wait();
  pdl_launch_dependents();
  constexpr int RPW = 32 / LPR;
  const int lane = threadIdx.x & 31;
  const int sub = lane / LPR, l = lane % LPR;
  const int F = F4 * 4;
  const int warps_per_block = RO_THREADS / 32;
  for (int g = blockIdx.x * warps_per_block + (threadIdx.x >> 5); g < G; g += gridDim.x * warps_per_block) {
    const int64_t lo = gptr[g], hi = gptr[g + 1];
    const int n = (int)(hi - lo);
    for (int fb = 0; fb < F4; fb += LPR) {           // warp-uniform trip count
      const int f = fb + l;
      const bool fok = f < F4;
      float mx[4], sm[4]; int am[4];
#pragma unroll
      for (int v = 0; v < 4; ++v) { mx[v] = -FLT_MAX; sm[v] = 0.f; am[v] = -1; }
      if (fok) {
        for (int ib = sub; ib < n; ib += RPW * GRO_U) {
          int64_t j[GRO_U]; float t[GRO_U]; float4 xv[GRO_U];
#pragma unroll
          for (int u = 0; u < GRO_U; ++u) {
            const int i = ib + u * RPW;
            j[u] = i < n ? __ldg(perm + lo + i) : -1;
          }
#pragma unroll
          for (int u = 0; u < GRO_U; ++u) {
            t[u] = 0.f; xv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (j[u] >= 0) { t[u] = __ldg(score + j[u]); xv[u] = __ldg(x + j[u] * F4 + f); }
          }
#pragma unroll
          for (int u = 0; u < GRO_U; ++u) {
            if (j[u] < 0) continue;
            const int i = ib + u * RPW;
            const float th = tanhf(t[u]);
            float4 w = xv[u];
            w.x *= th; w.y *= th; w.z *= th; w.w *= th;
            xo[(lo + i) * F4 + f] = w;
            const float vals[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int v = 0; v < 4; ++v) {
              sm[v] += vals[v];
              if (vals[v] > mx[v] || am[v] < 0) { mx[v] = vals[v]; am[v] = i; }
            }
          }
        }
      }
#pragma unroll
      for (int d = LPR; d < 32; d <<= 1) {
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          float omx = __shfl_xor_sync(0xffffffffu, mx[v], d);
          int oam = __shfl_xor_sync(0xffffffffu, am[v], d);
          float osm = __shfl_xor_sync(0xffffffffu, sm[v], d);
          sm[v] = (sub & (d / LPR)) ? osm + sm[v] : sm[v] + osm;
          bool take = oam >= 0 && (am[v] < 0 || omx > mx[v] || (omx == mx[v] && oam < am[v]));
          if (take) { mx[v] = omx; am[v] = oam; }
        }
      }
      if (fok && sub == 0) {
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          out[(int64_t)g * out_stride + f * 4 + v] = am[v] >= 0 ? mx[v] : 0.f;
          argmax[(int64_t)g * F + f * 4 + v] = am[v] >= 0 ? (int)(lo + am[v]) : -1;
          out[(int64_t)g * out_stride + F + f * 4 + v] = sm[v] / (float)(n > 0 ? n : 1);
        }
      }
    }
  }
}

// Gate + the next conv's x W in one flat pass over the pooled rows (round 2):
//     xo[i] = x[perm[i]] * tanh(score[perm[i]])        layers.py:21
//     xw[i] = xo[i] @ W_next                           network.py:38,42 -> GCNConv: x W before the propagation
// No graph structure: a warp takes RPW * GL_WU consecutive rows, gates them into xo and into a private shared-memory tile,
// and multiplies the tile by W_next with k_linear_fwd_dense's k-ascending FMA chain per output, so xo is bit-identical
// to k_gate_gather_fwd and xw to tsg_linear_fwd on xo -- without reading the pooled rows back from HBM, and with one
// launch less per level.  The readout then runs on xo (k_readout_fwd).
//   Tried first and measured slower (profiles/r02f_gate_readout.md): doing the readout in the same kernel, a CTA per
//   graph with the ordered sum taken from shared-memory tiles -- the readout's fixed summation order needs a per-graph
//   owner, and per-graph owners mean either few graphs in flight (CTA per graph) or long dependent walks (warp per
//   graph); a flat pass has neither.
constexpr int GL_THREADS = 256;
constexpr int GL_WU = 4;              // rows per lane group

// 4 outputs of `ROWS` rows: acc[u][c] = sum_k a_u[k] * W[k][4l + c], k ascending, one FMA per term (k_linear_fwd_dense)
template <int F, int ROWS>
__device__ __forceinline__ void gl_rows_times_w(const float* __restrict__ Ws, const float* const (&arow)[ROWS], int l,
                                                float (&acc)[ROWS][4]) {
#pragma unroll
  for (int u = 0; u < ROWS; ++u)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[u][c] = 0.f;
#pragma unroll 2
  for (int k = 0; k < F; k += 4) {
    float4 wq[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) wq[q] = *reinterpret_cast<const float4*>(Ws + (k + q) * F + 4 * l);
#pragma unroll
    for (int u = 0; u < ROWS; ++u) {
      const float4 a = *reinterpret_cast<const float4*>(arow[u] + k);
      acc[u][0] = fmaf(a.x, wq[0].x, acc[u][0]); acc[u][1] = fmaf(a.x, wq[0].y, acc[u][1]);
      acc[u][2] = fmaf(a.x, wq[0].z, acc[u][2]); acc[u][3] = fmaf(a.x, wq[0].w, acc[u][3]);
      acc[u][0] = fmaf(a.y, wq[1].x, acc[u][0]); acc[u][1] = fmaf(a.y, wq[1].y, acc[u][1]);
      acc[u][2] = fmaf(a.y, wq[1].z, acc[u][2]); acc[u][3] = fmaf(a.y, wq[1].w, acc[u][3]);
      acc[u][0] = fmaf(a.z, wq[2].x, acc[u][0]); acc[u][1] = fmaf(a.z, wq[2].y, acc[u][1]);
      acc[u][2] = fmaf(a.z, wq[2].z, acc[u][2]); acc[u][3] = fmaf(a.z, wq[2].w, acc[u][3]);
      acc[u][0] = fmaf(a.w, wq[3].x, acc[u][0]); acc[u][1] = fmaf(a.w, wq[3].y, acc[u][1]);
      acc[u][2] = fmaf(a.w, wq[3].z, acc[u][2]); acc[u][3] = fmaf(a.w, wq[3].w, acc[u][3]);
    }
  }
}

template <int LPR>
__global__ void __launch_bounds__(GL_THREADS)
k_gate_linear(const float4* __restrict__ x, const float* __restrict__ score, const int64_t* __restrict__ perm, int64_t K,
              float4* __restrict__ xo, const float* __restrict__ Wn, float4* __restrict__ xw) {
  pdl_wait();
  pdl_launch_dependents();
  constexpr int F4 = LPR, F = 4 * LPR;
  constexpr int RPW = 32 / LPR;
  constexpr int WROWS = RPW * GL_WU;                  // rows per warp: 16 (F = 32), 8 (F = 64)
  constexpr int PITCH = F + 4;                        // float4-aligned, rows of the warp's lane groups on distinct banks
  extern __shared__ __align__(16) float gl_smem[];
  float* Ws = gl_smem;                                // [F][F]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane / LPR, l = lane % LPR;
  float* Tw = gl_smem + F * F + warp * WROWS * PITCH;
  const int64_t base = ((int64_t)blockIdx.x * (GL_THREADS / 32) + warp) * WROWS;
  int64_t j[GL_WU];
#pragma unroll
  for (int u = 0; u < GL_WU; ++u) {                   // the dependent chain perm -> score / x starts before the W fill
    const int64_t i = base + sub + u * RPW;
    j[u] = i < K ? __ldg(perm + i) : -1;
  }
  for (int i = threadIdx.x; i < F * F / 4; i += GL_THREADS)
    reinterpret_cast<float4*>(Ws)[i] = __ldg(reinterpret_cast<const float4*>(Wn) + i);
  float tv[GL_WU]; float4 xv[GL_WU];
#pragma unroll
  for (int u = 0; u < GL_WU; ++u) {
    tv[u] = 0.f; xv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (j[u] >= 0) { tv[u] = __ldg(score + j[u]); xv[u] = __ldg(x + j[u] * F4 + l); }
  }
#pragma unroll
  for (int u = 0; u < GL_WU; ++u) {
    if (j[u] < 0) continue;
    const float th = tanhf(tv[u]);
    float4 w = xv[u];
    w.x *= th; w.y *= th; w.z *= th; w.w *= th;
    xo[(base + sub + u * RPW) * F4 + l] = w;
    *reinterpret_cast<float4*>(Tw + (sub + u * RPW) * PITCH + 4 * l) = w;
  }
  __syncthreads();                                    // Ws (whole CTA) and Tw (this warp)
  // all GL_WU rows of the lane group against one pass over W: ncu on the two-rows-at-a-time version showed the kernel
  // waiting on shared memory (short_scoreboard 5.7, mio_throttle 4.6 per issue), and W's float4 loads are what halves
  if (base < K) {                                     // warp-uniform
    const float* arow[GL_WU];
#pragma unroll
    for (int u = 0; u < GL_WU; ++u) arow[u] = Tw + (sub + u * RPW) * PITCH;
    float acc[GL_WU][4];
    gl_rows_times_w<F, GL_WU>(Ws, arow, l, acc);
#pragma unroll
    for (int u = 0; u < GL_WU; ++u) {
      const int64_t i = base + sub + u * RPW;
      if (i < K)     // "+ 0.f" = the bias-less add of k_linear_fwd_dense (turns -0 into +0 as it does)
        xw[i * F4 + l] = make_float4(acc[u][0] + 0.f, acc[u][1] + 0.f, acc[u][2] + 0.f, acc[u][3] + 0.f);
    }
  }
}

template <int VEC, int LPR>
__global__ void __launch_bounds__(RO_BWD_THREADS)
k_readout_bwd(const float* __restrict__ dout, int64_t dstride, const int* __restrict__ argmax,
              const int64_t* __restrict__ gptr, int G, int F, int mode, float* __restrict__ dx) {
  pdl_wait();
  pdl_launch_dependents();
  constexpr int RPW = 32 / LPR;
  const int lane = threadIdx.x & 31;
  const int sub = lane / LPR, l = lane % LPR;
  const int FV = F / VEC;
  // CTA per graph (a warp per graph left 3,504 warps streaming 62 MB: 65 us): the 8 warps of a CTA interleave
  // the graph's rows, every thread keeps the graph's gradient row for its feature column(s) in registers
  const int warps_per_block = RO_BWD_THREADS / 32;
  const int wsub = (threadIdx.x >> 5) * RPW + sub;
  for (int g = blockIdx.x; g < G; g += gridDim.x) {
    const int64_t lo = gptr[g], hi = gptr[g + 1];
    const int n = (int)(hi - lo);
    for (int f = l; f < FV; f += LPR) {
      float gm[VEC], gs[VEC]; int am[VEC];
      int col = 0;
#pragma unroll
      for (int v = 0; v < VEC; ++v) { gm[v] = 0.f; gs[v] = 0.f; am[v] = -1; }
      if (mode & TSG_READOUT_MAX) {
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          gm[v] = dout[(int64_t)g * dstride + f * VEC + v];
          am[v] = argmax[(int64_t)g * F + f * VEC + v];
        }
        col = F;
      }
      if (mode & (TSG_READOUT_MEAN | TSG_READOUT_SUM)) {
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          float d = dout[(int64_t)g * dstride + col + f * VEC + v];
          gs[v] = (mode & TSG_READOUT_MEAN) ? d / (float)(n > 0 ? n : 1) : d;
        }
      }
      for (int i = wsub; i < n; i += RPW * warps_per_block) {
        float r[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) r[v] = gs[v] + ((am[v] == (int)(lo + i)) ? gm[v] : 0.f);
        if (VEC == 4) {
          float4* p = reinterpret_cast<float4*>(dx) + (lo + i) * FV + f;
          float4 o = make_float4(r[0], r[1 % VEC], r[2 % VEC], r[3 % VEC]);
          if (mode & TSG_READOUT_ACCUM) { const float4 e = *p; o.x += e.x; o.y += e.y; o.z += e.z; o.w += e.w; }
          *p = o;
        } else {
          float* p = dx + (lo + i) * FV + f;
          *p = (mode & TSG_READOUT_ACCUM) ? *p + r[0] : r[0];
        }
      }
    }
  }
}

}  // namespace tsg

using namespace tsg;

template <int VEC>
static int launch_fwd(int lpr, int grid, cudaStream_t st, const float* x, const int64_t* gptr, int G,
                      int F, int mode, float* out, int64_t os, int* am) {
#define TSG_GO(L) TSG_LAUNCH_PDL("readout_fwd", k_readout_fwd<VEC, L>, grid, RO_THREADS, 0, st, x, gptr, G, F, mode, out, os, am)
  switch (lpr) {
    case 1: TSG_GO(1); break; case 2: TSG_GO(2); break; case 4: TSG_GO(4); break;
    case 8: TSG_GO(8); break; case 16: TSG_GO(16); break; default: TSG_GO(32); break;
  }
#undef TSG_GO
  return check_launch("readout_fwd");
}

template <int VEC>
static int launch_bwd(int lpr, int grid, cudaStream_t st, const float* dout, int64_t ds, const int* am,
                      const int64_t* gptr, int G, int F, int mode, float* dx) {
#define TSG_GO(L) TSG_LAUNCH_PDL("readout_bwd", k_readout_bwd<VEC, L>, grid, RO_BWD_THREADS, 0, st, dout, ds, am, gptr, G, F, mode, dx)
  switch (lpr) {
    case 1: TSG_GO(1); break; case 2: TSG_GO(2); break; case 4: TSG_GO(4); break;
    case 8: TSG_GO(8); break; case 16: TSG_GO(16); break; default: TSG_GO(32); break;
  }
#undef TSG_GO
  return check_launch("readout_bwd");
}

static int pick_lpr(int64_t fv) { int l = 1; while (l < fv && l < 32) l <<= 1; return l; }

extern "C" int tsg_readout_fwd(const float* x, const int64_t* gptr, int64_t G, int64_t F, int mode,
                               float* out, int64_t out_stride, int32_t* argmax, void* stream) {
  TSG_REQUIRE(G >= 0 && F > 0 && G < (int64_t)0x7fffffff, "readout_fwd: bad shape");
  TSG_REQUIRE((mode & (TSG_READOUT_MAX | TSG_READOUT_MEAN | TSG_READOUT_SUM)) != 0, "readout_fwd: empty mode");
  TSG_REQUIRE(!((mode & TSG_READOUT_MEAN) && (mode & TSG_READOUT_SUM)), "readout_fwd: mean and sum are exclusive");
  if (G == 0) return TSG_OK;
  TSG_REQUIRE(gptr && out, "readout_fwd: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  int grid = grid_for(G, RO_THREADS / 32);
  bool vec = F % 4 == 0 && (((uintptr_t)x) & 15) == 0;
  if (vec) return launch_fwd<4>(pick_lpr(F / 4), grid, st, x, gptr, (int)G, (int)F, mode, out, out_stride, argmax);
  return launch_fwd<1>(pick_lpr(F), grid, st, x, gptr, (int)G, (int)F, mode, out, out_stride, argmax);
}

extern "C" int tsg_readout_bwd(const float* dout, int64_t dout_stride, const int32_t* argmax,
                               const int64_t* gptr, int64_t G, int64_t N, int64_t F, int mode,
                               float* dx, void* stream) {
  TSG_REQUIRE(G >= 0 && F > 0 && N >= 0 && G < (int64_t)0x7fffffff, "readout_bwd: bad shape");
  if (G == 0 || N == 0) return TSG_OK;
  TSG_REQUIRE(dout && gptr && dx, "readout_bwd: null pointer");
  TSG_REQUIRE(!(mode & TSG_READOUT_MAX) || argmax, "readout_bwd: max mode needs argmax");
  cudaStream_t st = (cudaStream_t)stream;
  int grid = grid_for(G, 1);
  bool vec = F % 4 == 0 && (((uintptr_t)dx) & 15) == 0;
  if (vec) return launch_bwd<4>(pick_lpr(F / 4), grid, st, dout, dout_stride, argmax, gptr, (int)G, (int)F, mode, dx);
  return launch_bwd<1>(pick_lpr(F), grid, st, dout, dout_stride, argmax, gptr, (int)G, (int)F, mode, dx);
}

/* gate (x[perm] * tanh(score[perm])) + [max || mean] readout in one pass; see k_gate_readout_fwd.  feat % 4 == 0. */
extern "C" int tsg_gate_readout_fwd(const float* x, const float* score, const int64_t* perm, const int64_t* gptr,
                                    int64_t G, int64_t F, float* xo, float* out, int64_t out_stride, int32_t* argmax,
                                    void* stream) {
  TSG_REQUIRE(G >= 0 && F > 0 && F % 4 == 0 && G < (int64_t)0x7fffffff, "gate_readout_fwd: bad shape");
  if (G == 0) return TSG_OK;
  TSG_REQUIRE(x && score && perm && gptr && xo && out && argmax, "gate_readout_fwd: null pointer");
  TSG_REQUIRE(((((uintptr_t)x) | ((uintptr_t)xo)) & 15) == 0, "gate_readout_fwd: operands must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = grid_for(G, RO_THREADS / 32);
  const int F4 = (int)(F / 4);
#define TSG_GR(L) TSG_LAUNCH_PDL("gate_readout_fwd", k_gate_readout_fwd<L>, grid, RO_THREADS, 0, st, (const float4*)x, score, perm, gptr, (int)G, F4, (float4*)xo, out, out_stride, argmax)
  switch (pick_lpr(F4)) {
    case 1: TSG_GR(1); break; case 2: TSG_GR(2); break; case 4: TSG_GR(4); break;
    case 8: TSG_GR(8); break; case 16: TSG_GR(16); break; default: TSG_GR(32); break;
  }
#undef TSG_GR
  return check_launch("gate_readout_fwd");
}

/* Gate + readout + (when w_next is given) xw_next = xo @ w_next, the next GCNConv's x W (network.py:38,42).
 * feat = 32 / 64 with w_next: k_gate_linear (gate and product in one flat pass) + k_readout_fwd on xo; without w_next or for
 * other widths: tsg_gate_readout_fwd (+ tsg_linear_fwd).  Either way bit-identical to gate_gather, readout, linear_fwd. */
extern "C" int tsg_gate_readout_linear_fwd(const float* x, const float* score, const int64_t* perm, const int64_t* gptr,
                                           int64_t G, int64_t num_rows_out, int64_t F, float* xo, float* out,
                                           int64_t out_stride, int32_t* argmax, const float* w_next, float* xw_next,
                                           void* stream) {
  TSG_REQUIRE(G >= 0 && num_rows_out >= 0 && F > 0 && F % 4 == 0 && G < (int64_t)0x7fffffff, "gate_readout_linear_fwd: bad shape");
  TSG_REQUIRE((w_next == nullptr) == (xw_next == nullptr), "gate_readout_linear_fwd: w_next and xw_next go together");
  if (G == 0) return TSG_OK;
  static const bool v1 = getenv("TSG_GATE_V1") != nullptr;
  const bool aligned = ((((uintptr_t)x) | ((uintptr_t)xo) | ((uintptr_t)xw_next) | ((uintptr_t)w_next)) & 15) == 0;
  if (v1 || !w_next || !(F == 32 || F == 64) || !aligned) {
    int rc = tsg_gate_readout_fwd(x, score, perm, gptr, G, F, xo, out, out_stride, argmax, stream);
    if (rc == TSG_OK && w_next && num_rows_out > 0) rc = tsg_linear_fwd(xo, w_next, nullptr, xw_next, num_rows_out, F, F, 0, 0, stream);
    return rc;
  }
  TSG_REQUIRE(x && score && perm && gptr && xo && out && argmax, "gate_readout_linear_fwd: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (num_rows_out > 0) {
    const int wrows = (32 / (int)(F / 4)) * GL_WU;
    const int64_t rows_per_cta = (int64_t)(GL_THREADS / 32) * wrows;
    const int64_t grid = (num_rows_out + rows_per_cta - 1) / rows_per_cta;
    TSG_REQUIRE(grid < (int64_t)0x7fffffff, "gate_readout_linear_fwd: too many rows");
    const size_t smem = ((size_t)F * F + (size_t)(GL_THREADS / 32) * wrows * (F + 4)) * sizeof(float);
    if (F == 32) TSG_LAUNCH_PDL("gate_readout_linear_fwd", k_gate_linear<8>, (int)grid, GL_THREADS, smem, st, (const float4*)x, score, perm,
                                num_rows_out, (float4*)xo, w_next, (float4*)xw_next);
    else TSG_LAUNCH_PDL("gate_readout_linear_fwd", k_gate_linear<16>, (int)grid, GL_THREADS, smem, st, (const float4*)x, score, perm,
                        num_rows_out, (float4*)xo, w_next, (float4*)xw_next);
  }
  return tsg_readout_fwd(xo, gptr, G, F, TSG_READOUT_MAX | TSG_READOUT_MEAN, out, out_stride, argmax, stream);
}
