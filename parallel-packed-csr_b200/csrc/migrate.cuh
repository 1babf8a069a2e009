// migrate.cuh -- a shard laid out afresh from a device-resident CSR (ppcsr_load_csr, ppcsr_group_repartition).
//
// The items of a shard in key order are, per vertex v, its sentinel followed by its out-edges: with rowptr of the
// CSR, the sentinel of v has rank rowptr[v] + v and its i-th edge rank rowptr[v] + v + 1 + i, j = E + n items in all.
// k_layout_from_csr places them exactly as a root-window rebuild does (rebalance*.cuh, DESIGN §3b): output leaf o of m
// receives the ranks [(o*j) >> lg m, ((o+1)*j) >> lg m), left-packed, the rest of the leaf null.  It is a pure gather:
// nothing of the previous layout is read, so the target can be a fresh array of any size.
#pragma once
#include "common.cuh"

namespace mig {

constexpr int MT = 256;  // 8 warps, one output leaf each

// out[i] = in[i] - base + add for i in [0, count]: a slice of an exported rowptr rebased into the spliced CSR
__global__ void __launch_bounds__(MT) k_rebase_rowptr(const uint64_t *__restrict__ in, uint64_t count, uint64_t base,
                                                      uint64_t add, uint64_t *__restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i <= count) out[i] = in[i] - base + add;
}

// num_neighbors == row length (ppcsr_load_csr without an nn array)
__global__ void __launch_bounds__(MT) k_row_lengths(const uint64_t *__restrict__ rowptr, uint32_t n,
                                                    uint32_t *__restrict__ nn) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v < n) nn[v] = (uint32_t)(rowptr[v + 1] - rowptr[v]);
}

// Validation of a CSR that comes from outside (ppcsr_load_csr): *bad != 0 if rowptr[0] != 0, rowptr decreases,
// rowptr[n] != E, a row is not strictly ascending, a col is the sentinel marker or a value is 0.  One thread per
// vertex (rowptr) and one per edge; an edge finds its row by binary search, which stays inside [0, n] even when rowptr
// is not monotone (the rowptr check flags that case anyway).
__global__ void __launch_bounds__(MT) k_validate_csr(const uint64_t *__restrict__ rowptr, const uint32_t *__restrict__ col,
                                                     const uint32_t *__restrict__ val, uint32_t n, uint64_t E,
                                                     unsigned int *__restrict__ bad) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned int b = 0;
  if (i <= n) {
    if (i == 0 && rowptr[0] != 0) b |= 1u;
    if (i == n && rowptr[n] != E) b |= 1u;
    if (i < n && rowptr[i + 1] < rowptr[i]) b |= 1u;
  }
  if (i < E) {
    const uint32_t c = col[i];
    if (c == PPCSR_SENT) b |= 2u;
    if (val && val[i] == 0) b |= 4u;
    if (i + 1 < E) {
      uint32_t lo = 0, hi = n;  // row of edge i: the last v with rowptr[v] <= i
      while (lo < hi) {
        const uint32_t mid = lo + (hi - lo + 1) / 2;
        if (rowptr[mid] <= i) lo = mid;
        else hi = mid - 1;
      }
      const uint64_t row_end = lo < n ? rowptr[lo + 1] : E;
      if (i + 1 < row_end && col[i + 1] <= c) b |= 8u;
    }
  }
  if (b) atomicOr(bad, b);
}

// One warp per output leaf o of m = 1 << lg_m leaves of 1 << ls <= 32 slots (make_geometry keeps logN <= 32 up to 2^31
// slots).  Lane 0 finds v0, the vertex of the leaf's first rank, by binary search over the item prefix
// P(v) = rowptr[v] + v; lane t loads P(v0 + 1 + t), and the vertex of the rank in lane f is v0 + the number of those
// not above it (a leaf holds fewer than 32 items, so fewer than 32 sentinels start inside it).  Every lane writes one
// slot of dest / val: the leaf's lines are written whole, nulls included.
__global__ void __launch_bounds__(MT) k_layout_from_csr(const uint64_t *__restrict__ rowptr,
                                                        const uint32_t *__restrict__ col,
                                                        const uint32_t *__restrict__ w, uint32_t w_uniform, uint32_t n,
                                                        uint64_t j, uint32_t lg_m, uint32_t ls,
                                                        uint32_t *__restrict__ dest, uint32_t *__restrict__ val,
                                                        uint32_t *__restrict__ beg, uint32_t *__restrict__ leaf_cnt,
                                                        uint32_t *__restrict__ tree_leaf) {
  const uint32_t o = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31u;
  if (o >= (1u << lg_m)) return;  // whole warps leave together
  const uint64_t r0 = ((uint64_t)o * j) >> lg_m, r1 = ((uint64_t)(o + 1) * j) >> lg_m;
  const uint32_t cnt = (uint32_t)(r1 - r0);
  // v0 = the last v with P(v) <= r0, by a 32-ary search of the whole warp: P(lo) <= r0 < P(hi) (P(n) = infinity),
  // every round probes 32 points of (lo, hi) and keeps the gap after the last one not above r0: 4 rounds of loads at
  // 2^20 vertices where a binary search would issue 20 dependent ones
  uint32_t lo = 0, hi = n;
  while (cnt && hi - lo > 1) {
    const uint32_t span = hi - lo;
    const uint32_t probe = span <= 32 ? lo + lane : lo + (uint32_t)(((uint64_t)span * lane) >> 5);
    const bool le = probe < hi && rowptr[probe] + probe <= r0;
    const uint32_t last = 31 - __clz(__ballot_sync(0xFFFFFFFFu, le));  // lane 0 probes lo: never empty
    const uint32_t next = __shfl_sync(0xFFFFFFFFu, probe, (last + 1) & 31u);
    lo = __shfl_sync(0xFFFFFFFFu, probe, last);
    if (span <= 32) break;
    hi = last == 31 ? hi : next;
  }
  const uint32_t v0 = lo;
  const uint64_t p_lane = (cnt && (uint64_t)v0 + 1 + lane < n) ? rowptr[v0 + 1 + lane] + v0 + 1 + lane : ~0ull;
  const uint64_t p_v0 = __shfl_sync(0xFFFFFFFFu, cnt && lane == 0 ? rowptr[v0] + v0 : 0ull, 0);
  uint32_t mine = 0;
  for (uint32_t f = 0; f < cnt; f++) {
    const uint32_t c = __popc(__ballot_sync(0xFFFFFFFFu, p_lane <= r0 + f));
    if (lane == f) mine = c;
  }
  const uint64_t p_prev = __shfl_sync(0xFFFFFFFFu, p_lane, (mine ? mine - 1 : 0) & 31u);
  const size_t slot = ((size_t)o << ls) + lane;
  if (lane < cnt) {
    const uint32_t v = v0 + mine;
    const uint64_t k = r0 + lane, pv = mine ? p_prev : p_v0;
    if (k == pv) {
      dest[slot] = PPCSR_SENT;
      val[slot] = v + 1u;
      beg[v] = (uint32_t)slot;
    } else {
      const uint64_t e = k - v - 1;
      dest[slot] = col[e];
      val[slot] = w ? w[e] : w_uniform;
    }
  } else if (lane < (1u << ls)) {
    dest[slot] = 0;
    val[slot] = 0;
  }
  if (lane == 0) {
    leaf_cnt[o] = cnt;
    tree_leaf[o] = cnt;
  }
}

}  // namespace mig
