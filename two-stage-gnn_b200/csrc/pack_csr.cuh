// pack_csr.cuh -- the per-graph pieces of a RAW CSR built from a COALESCED, SYMMETRIC graph-local list (sorted by
// (row, col), loop free, (r, c) listed <=> (c, r) listed), shared by K0d (adjacency) and K0e (adjacency and the
// coarsened EigenPooling adjacency).  Row r's entries are the run of lrow == r, so row starts fall out of the run
// boundaries: no counting pass, no scan, no atomics.
#pragma once
#include "common.cuh"
#include "sag_fused.cuh"

namespace tsg {

// One CTA's threads (tid, stride nthreads) verify a graph's list lrow / lcol [0, e) with ids local to [0, n) and record
// its row starts: rs[r] = first position of row r for r in [0, n], rs[n] = e; rows without entries point at the next
// run.  Returns this thread's violations (TSG_FUSED_BAD_EDGE: id out of range or self loop; TSG_FUSED_UNSORTED: not
// strictly increasing in (row, col)); rs is only meaningful when no thread of the CTA found one.
__device__ __forceinline__ int coalesced_row_starts(const int32_t* __restrict__ lrow, const int32_t* __restrict__ lcol,
                                                    int n, int e, int* __restrict__ rs, int tid, int nthreads) {
  int bad = 0;
  for (int p = tid; p <= e; p += nthreads) {
    const int r = p < e ? lrow[p] : n;
    const int r0 = p > 0 ? lrow[p - 1] : -1;
    if (p < e) {
      const int q = lcol[p];
      if ((unsigned)r >= (unsigned)n || (unsigned)q >= (unsigned)n || r == q) { bad |= TSG_FUSED_BAD_EDGE; continue; }
      if (p > 0 && !(r0 < r || (r0 == r && lcol[p - 1] < q))) { bad |= TSG_FUSED_UNSORTED; continue; }
    }
    if (r0 != -1 && (unsigned)r0 >= (unsigned)n) continue;
    for (int rr = r0 + 1; rr <= r; ++rr) rs[rr] = p;          // rows r0+1 .. r start here (empty rows included)
  }
  return bad;
}

// Position of row q's entry r in the list (binary search in q's run, rs from coalesced_row_starts), or -1 when the list
// does not hold it -- i.e. the entry (r, q) has no mirror.
__device__ __forceinline__ int coalesced_find(const int32_t* __restrict__ lcol, const int* __restrict__ rs, int q, int r) {
  int lo = rs[q], hi = rs[q + 1];
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const int v = lcol[mid];
    if (v == r) return mid;
    if (v < r) lo = mid + 1; else hi = mid;
  }
  return -1;
}

}  // namespace tsg
