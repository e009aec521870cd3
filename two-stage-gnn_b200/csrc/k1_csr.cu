// K1 -- CSR construction + GCN normalisation (integer work: bit-exact, deterministic).
//
// Replaces PyG 1.6.3 `gcn_norm` (add_remaining_self_loops -> scatter_add degree -> deg^-1/2 A
// deg^-1/2) reached from Code/sag/network.py:34,38,42 and Code/sag/layers.py:18 of the reference,
// and produces the CSR (both orientations) that K2 aggregates over.
//
// Algorithm (stable counting sort without a device-wide sort):
//   1. count   : per edge, atomicAdd on per-row counters of both orientations (integer atomics:
//                the COUNT is order independent);
//   2. scan    : exclusive scan of (count [+1 self loop]) -> rowptr;
//   3. fill    : per edge, claim a slot in its row with atomicAdd (arbitrary order), store edge id;
//   4. place   : per edge, rank = number of edge ids in its row smaller than its own (rows are
//                tiny: ~5 entries on DD, ~18 on JAN.Y.) -> final slot = rowptr + rank.  Edge ids are
//                unique, so the result equals a stable sort whatever order step 3 produced;
//   5. degree  : per row, sequential sum of the in-edge weights in CSR order (+ loop weight), the
//                order index_add_ uses, then dis = 1/sqrt(deg) with IEEE div/sqrt (inf -> 0);
//   6. values  : val = (dis[src] * w) * dis[dst], rounded after each product like the reference.
// HBM-bound integer/byte work: coalesced 8-byte loads of row/col, 4-byte scattered writes.
#include "common.cuh"

namespace tsg {

struct CsrArgs {
  const int64_t* row; const int64_t* col; const float* w;
  int64_t E_cap; const int64_t* E_dev; int N; int gcn;
};

__global__ void k_csr_count(CsrArgs a, int* cnt_dst, int* cnt_src, int* loop_eid) {
  pdl_wait();
  pdl_launch_dependents();
  int64_t E = dev_count(a.E_cap, a.E_dev);
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E;
       e += (int64_t)gridDim.x * blockDim.x) {
    int r = (int)a.row[e], c = (int)a.col[e];
    if (a.gcn && r == c) {
      if (a.w != nullptr) atomicMax(&loop_eid[r], (int)e);   // last listed loop's weight wins
      continue;
    }
    atomicAdd(&cnt_dst[c], 1);
    if (cnt_src != nullptr) atomicAdd(&cnt_src[r], 1);
  }
}

struct CountPlus {
  const int* cnt; int add;
  __device__ int operator()(int64_t i) const { return cnt[i] + add; }
};

__global__ void k_csr_fill(CsrArgs a, const int* rowptr, int* fill_dst, int* tmp_dst,
                           const int* t_rowptr, int* fill_src, int* tmp_src) {
  pdl_wait();
  pdl_launch_dependents();
  int64_t E = dev_count(a.E_cap, a.E_dev);
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E;
       e += (int64_t)gridDim.x * blockDim.x) {
    int r = (int)a.row[e], c = (int)a.col[e];
    if (a.gcn && r == c) continue;
    tmp_dst[rowptr[c] + atomicAdd(&fill_dst[c], 1)] = (int)e;
    if (t_rowptr != nullptr) tmp_src[t_rowptr[r] + atomicAdd(&fill_src[r], 1)] = (int)e;
  }
}

__device__ __forceinline__ int rank_in_row(const int* __restrict__ tmp, int start, int len, int e) {
  int rank = 0;
  for (int q = 0; q < len; ++q) rank += (tmp[start + q] < e);
  return rank;
}

__global__ void k_csr_place(CsrArgs a, const int* rowptr, const int* cnt_dst, const int* tmp_dst,
                            int* colidx, int* eid,
                            const int* t_rowptr, const int* cnt_src, const int* tmp_src,
                            int* t_colidx, int* t_eid) {
  pdl_wait();
  pdl_launch_dependents();
  int64_t E = dev_count(a.E_cap, a.E_dev);
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (int64_t e = tid; e < E; e += stride) {
    int r = (int)a.row[e], c = (int)a.col[e];
    if (a.gcn && r == c) continue;
    {
      int s = rowptr[c];
      int p = s + rank_in_row(tmp_dst, s, cnt_dst[c], (int)e);
      colidx[p] = r;
      if (eid) eid[p] = (int)e;
    }
    if (t_rowptr != nullptr) {
      int s = t_rowptr[r];
      int p = s + rank_in_row(tmp_src, s, cnt_src[r], (int)e);
      t_colidx[p] = c;
      if (t_eid) t_eid[p] = (int)e;
    }
  }
  if (a.gcn) {   // appended self loops: last slot of every row, id = E_cap + node
    for (int64_t i = tid; i < a.N; i += stride) {
      int p = rowptr[i + 1] - 1;
      colidx[p] = (int)i;
      if (eid) eid[p] = (int)(a.E_cap + i);
      if (t_rowptr != nullptr) {
        int q = t_rowptr[i + 1] - 1;
        t_colidx[q] = (int)i;
        if (t_eid) t_eid[q] = (int)(a.E_cap + i);
      }
    }
  }
}

// dis[c] = 1/sqrt(sum of weights into c) ; sequential in CSR (= COO) order.
__global__ void k_csr_degree(CsrArgs a, const int* rowptr, const int* eid_or_tmp, const int* loop_eid,
                             float* dis) {
  pdl_wait();
  pdl_launch_dependents();
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < a.N;
       c += (int64_t)gridDim.x * blockDim.x) {
    int s = rowptr[c], t = rowptr[c + 1] - 1;    // last slot is the loop
    float deg;
    if (a.w == nullptr) {
      deg = (float)(t - s) + 1.0f;
    } else {
      deg = 0.f;
      for (int p = s; p < t; ++p) deg = __fadd_rn(deg, a.w[eid_or_tmp[p]]);
      int le = loop_eid[c];
      deg = __fadd_rn(deg, le >= 0 ? a.w[le] : 1.0f);
    }
    float d = __fdiv_rn(1.0f, __fsqrt_rn(deg));
    dis[c] = isinf(d) ? 0.f : d;
  }
}

// one thread per CSR slot of one orientation; `rows` says which endpoint indexes the row.
__global__ void k_csr_values(CsrArgs a, const int* rowptr, const int* colidx, const int* eid,
                             const int* loop_eid, const float* dis, float* val, int dst_major) {
  pdl_wait();
  pdl_launch_dependents();
  // thread per row, walking its slots: rows are short and this keeps row id for free.
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < a.N;
       r += (int64_t)gridDim.x * blockDim.x) {
    int s = rowptr[r], t = rowptr[r + 1];
    float dr = a.gcn ? dis[r] : 1.f;
    for (int p = s; p < t; ++p) {
      int o = colidx[p];
      float w = 1.0f;
      if (a.w != nullptr) {
        int e = eid[p];
        if (e < a.E_cap) w = a.w[e];
        else { int le = loop_eid[r]; w = le >= 0 ? a.w[le] : 1.0f; }
      }
      if (a.gcn) {
        // norm = (dis[src] * w) * dis[dst]
        float dsrc = dst_major ? dis[o] : dr;
        float ddst = dst_major ? dr : dis[o];
        val[p] = __fmul_rn(__fmul_rn(dsrc, w), ddst);
      } else {
        val[p] = w;
      }
    }
  }
}

}  // namespace tsg

using namespace tsg;

extern "C" size_t tsg_csr_build_workspace_bytes(int64_t E, int64_t N) {
  size_t b = 0;
  b += 5 * ws_bytes((size_t)N + 1, 4);      // cnt_dst, cnt_src, fill_dst, fill_src, loop_eid
  b += ws_bytes((size_t)N + 1, 4);          // dis
  b += 2 * ws_bytes((size_t)E + (size_t)N + 1, 4);   // tmp_dst, tmp_src (indexed by rowptr slots)
  b += 2 * ws_bytes((size_t)E + (size_t)N + 1, 4);   // eid scratch when caller passes NULL eid
  b += ws_bytes(scan_ws_ints(N), 4);
  return b + 1024;
}

extern "C" int tsg_csr_build(const int64_t* row, const int64_t* col, const float* edge_weight,
                             int64_t E, const int64_t* E_dev, int64_t N, int mode,
                             int32_t* rowptr, int32_t* colidx, float* val, int32_t* eid,
                             int32_t* t_rowptr, int32_t* t_colidx, float* t_val, int32_t* t_eid,
                             void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TSG_REQUIRE(N >= 0 && E >= 0, "csr_build: negative size");
  TSG_REQUIRE(N + E < (int64_t)0x7fffffff, "csr_build: sum n + sum E must stay below 2^31");
  TSG_REQUIRE(mode == TSG_CSR_GCN || mode == TSG_CSR_RAW, "csr_build: bad mode %d", mode);
  TSG_REQUIRE(rowptr && (E + N == 0 || (colidx && val)), "csr_build: null output");
  TSG_REQUIRE(E == 0 || (row && col), "csr_build: null edge list");
  bool both = t_rowptr != nullptr;
  TSG_REQUIRE(!both || E + N == 0 || (t_colidx && t_val), "csr_build: null transposed output");
  if (workspace_bytes < tsg_csr_build_workspace_bytes(E, N)) {
    set_error("csr_build: workspace %zu < %zu", workspace_bytes, tsg_csr_build_workspace_bytes(E, N));
    return TSG_EWORKSPACE;
  }
  Workspace ws(workspace, workspace_bytes);
  int* cnt_dst = ws.take<int>(N + 1);
  int* cnt_src = ws.take<int>(N + 1);
  int* fill_dst = ws.take<int>(N + 1);
  int* fill_src = ws.take<int>(N + 1);
  int* loop_eid = ws.take<int>(N + 1);
  float* dis = ws.take<float>(N + 1);
  int* tmp_dst = ws.take<int>(E + N + 1);
  int* tmp_src = ws.take<int>(E + N + 1);
  int* eid_s = ws.take<int>(E + N + 1);
  int* t_eid_s = ws.take<int>(E + N + 1);
  int* scan_ws = ws.take<int>(scan_ws_ints(N));
  if (!ws.ok()) { set_error("csr_build: workspace carve failed"); return TSG_EWORKSPACE; }
  int gcn = mode == TSG_CSR_GCN;
  if (edge_weight != nullptr) {          // weights are read back through eid
    if (!eid) eid = eid_s;
    if (both && !t_eid) t_eid = t_eid_s;
  }
  CsrArgs a{row, col, edge_weight, E, E_dev, (int)N, gcn};

  // cnt_dst .. fill_src are contiguous (4 * aligned(N+1)) -> one memset; loop_eid = -1
  size_t one = ws_bytes((size_t)N + 1, 4);
  cudaMemsetAsync(cnt_dst, 0, 4 * one, st);
  cudaMemsetAsync(loop_eid, 0xFF, one, st);
  if (N == 0) { cudaMemsetAsync(rowptr, 0, 4, st); if (both) cudaMemsetAsync(t_rowptr, 0, 4, st); return check_launch("csr_build(empty)"); }

  const int T = 256;
  int ge = grid_for(E, T), gn = grid_for(N, T);
  if (E > 0) TSG_LAUNCH_PDL("csr_build(count)", k_csr_count, ge, T, 0, st, a, cnt_dst, both ? cnt_src : nullptr, loop_eid);
  int rc = exclusive_scan(CountPlus{cnt_dst, gcn}, N, rowptr, scan_ws, st);
  if (rc) return rc;
  if (both) { rc = exclusive_scan(CountPlus{cnt_src, gcn}, N, t_rowptr, scan_ws, st); if (rc) return rc; }
  const int* no_rows = nullptr;
  if (E > 0) TSG_LAUNCH_PDL("csr_build(fill)", k_csr_fill, ge, T, 0, st, a, (const int*)rowptr, fill_dst, tmp_dst, both ? t_rowptr : no_rows,
                            fill_src, tmp_src);
  TSG_LAUNCH_PDL("csr_build(place)", k_csr_place, grid_for(E > N ? E : N, T), T, 0, st, a, (const int*)rowptr, (const int*)cnt_dst,
                 (const int*)tmp_dst, colidx, eid, both ? t_rowptr : no_rows, (const int*)cnt_src, (const int*)tmp_src, t_colidx, t_eid);
  if (gcn) TSG_LAUNCH_PDL("csr_build(degree)", k_csr_degree, gn, T, 0, st, a, (const int*)rowptr, (const int*)eid, (const int*)loop_eid, dis);
  TSG_LAUNCH_PDL("csr_build(values)", k_csr_values, gn, T, 0, st, a, (const int*)rowptr, (const int*)colidx, (const int*)eid,
                 (const int*)loop_eid, (const float*)dis, val, 1);
  if (both) TSG_LAUNCH_PDL("csr_build(values)", k_csr_values, gn, T, 0, st, a, (const int*)t_rowptr, (const int*)t_colidx,
                           (const int*)t_eid, (const int*)loop_eid, (const float*)dis, t_val, 0);
  return TSG_OK;
}
