// isolate.cuh -- vertex isolation (ppcsr_isolate_vertices, ppcsr_group_isolate_vertices): every edge out of or into a
// vertex set removed in one streaming pass over the packed array.
//
// The set arrives as a bitmap of the n_bits global vertex ids (k_isolate_bitmap).  k_isolate_filter then walks the
// array the way the PageRank leaf walk does (queries.cuh, k_pagerank_push_leaves): a warp streams a run of consecutive
// 32-slot groups, finds the vertex of its first slot with one binary search over beg[], and a ballot + shuffle hands
// every live slot the nearest sentinel below it, i.e. its source.  A live edge (src, dst) whose src (made global with
// the shard's first vertex) or dst (if dst < n_bits) is in the set is removed exactly as k_locate removes one
// (batch.cuh): val[slot] = 0 as a tombstone, del_cnt[leaf] counts it, num_neighbors[src] drops by one, n_deleted and
// the touched-leaf tally n_touched_est grow.  The back half of a batch (finish_batch: window selection, the
// tombstone-compacting rebalance, resize, tree, beg[]) then runs unchanged with an empty insert list.
#pragma once
#include "common.cuh"

namespace iso {

constexpr int IT = 256;
constexpr int FL_BATCH = 4;  // groups whose loads are issued together

__device__ __forceinline__ bool bit_of(const uint32_t *__restrict__ bits, uint32_t v) {
  return (bits[v >> 5] >> (v & 31u)) & 1u;
}

// bits[v >> 5] |= 1 << (v & 31) for every listed id (all < n_bits, checked on the host); an id whose bit this launch
// set first counts toward n_unique, so duplicates are counted once
__global__ void __launch_bounds__(IT) k_isolate_bitmap(const uint32_t *__restrict__ ids, uint64_t count,
                                                       uint32_t *__restrict__ bits, BatchScalars *sc) {
  uint32_t fresh = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t v = ids[i], b = 1u << (v & 31u);
    if (!(atomicOr(&bits[v >> 5], b) & b)) fresh++;
  }
  fresh = __reduce_add_sync(0xFFFFFFFFu, fresh);
  if (lane_id() == 0 && fresh) atomicAdd(&sc->n_unique, (unsigned long long)fresh);
}

// The filter pass.  A leaf has at most 32 slots (logN = 1 << ls with ls <= 5 below 2^32 slots), so every leaf lies
// inside one 32-slot group and one warp owns it whole: its delete count is a plain store into the cleared del_cnt[],
// and the leaves that lost items are tallied once each, as k_locate tallies a leaf on its first delete.
// num_neighbors takes one atomic per source run of a group.
__global__ void __launch_bounds__(IT) k_isolate_filter(const uint32_t *__restrict__ dest, uint32_t *__restrict__ val,
                                                       const uint32_t *__restrict__ leaf_cnt,
                                                       const uint32_t *__restrict__ beg, uint32_t *__restrict__ nn,
                                                       uint32_t *__restrict__ del_cnt, uint32_t ls, uint32_t n,
                                                       uint64_t n_slots, const uint32_t *__restrict__ bits,
                                                       uint32_t n_bits, uint32_t vertex_offset, BatchScalars *sc) {
  const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
  const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = lane_id();
  const uint32_t groups = (uint32_t)(n_slots >> 5);
  const uint32_t per = (groups + warps - 1) / warps;
  const uint32_t g0 = min(w * per, groups), g1 = min(g0 + per, groups);
  if (g0 >= g1 || n == 0) return;
  // vertex owning the first slot of my run (the last v with beg[v] <= slot) and whether it is in the set
  uint32_t carry;
  {
    const uint32_t s0 = g0 << 5;
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1) {
      const uint32_t mid = lo + ((hi - lo) >> 1);
      if (beg[mid] <= s0) lo = mid;
      else hi = mid;
    }
    carry = lo;
  }
  bool carry_in = bit_of(bits, vertex_offset + carry);
  const uint32_t lsm = (1u << ls) - 1u;
  const unsigned lt = lanemask_lt(), le = lt | (1u << lane);
  const uint32_t leaves_per_group = 32u >> ls;
  // the slots of leaf `lane` of a group (lanes < leaves_per_group)
  const unsigned leaf_mask = (unsigned)(((1ull << (1u << ls)) - 1ull) << ((lane << ls) & 31u));
  uint32_t removed = 0, touched = 0;  // lane 0: edges removed; lane l: groups in which leaf l of the group lost items
  for (uint32_t g = g0; g < g1; g += FL_BATCH) {
    uint32_t d[FL_BATCH];
    bool live[FL_BATCH];
#pragma unroll
    for (int u = 0; u < FL_BATCH; u++) {
      const uint32_t slot = ((g + u) << 5) + lane;
      live[u] = g + u < g1 && (slot & lsm) < leaf_cnt[slot >> ls];
      d[u] = live[u] ? dest[slot] : 0u;
    }
#pragma unroll
    for (int u = 0; u < FL_BATCH; u++) {
      if (g + u >= g1) break;  // warp-uniform
      const uint32_t slot = ((g + u) << 5) + lane;
      const bool sent = live[u] && d[u] == PPCSR_SENT;
      const uint32_t sv = sent ? val[slot] - 1u : 0u;
      const bool s_in = sent && bit_of(bits, vertex_offset + sv);
      const unsigned m = __ballot_sync(0xFFFFFFFFu, sent);
      const unsigned m_in = __ballot_sync(0xFFFFFFFFu, s_in);
      const unsigned below = m & le;
      const int at = below ? 31 - __clz(below) : 0;
      uint32_t src = __shfl_sync(0xFFFFFFFFu, sv, at);
      bool src_in = (m_in >> at) & 1u;
      if (!below) {
        src = carry;
        src_in = carry_in;
      }
      const bool rm = live[u] && !sent && (src_in || (d[u] < n_bits && bit_of(bits, d[u])));
      if (rm) val[slot] = 0;  // tombstone; compacted away by the rebalance of this leaf
      const unsigned rmask = __ballot_sync(0xFFFFFFFFu, rm);
      if (rmask) {  // warp-uniform
        const unsigned peers = __match_any_sync(0xFFFFFFFFu, rm ? src : PPCSR_SENT);
        if (rm && (peers & lt) == 0) atomicSub(&nn[src], (uint32_t)__popc(peers));
        if (lane < leaves_per_group) {
          const uint32_t c = (uint32_t)__popc(rmask & leaf_mask);
          if (c) {
            del_cnt[(((g + u) << 5) >> ls) + lane] = c;
            touched++;
          }
        }
        if (lane == 0) removed += (uint32_t)__popc(rmask);
      }
      if (m) {
        const int last = 31 - __clz(m);
        carry = __shfl_sync(0xFFFFFFFFu, sv, last);
        carry_in = (m_in >> last) & 1u;
      }
    }
  }
  touched = __reduce_add_sync(0xFFFFFFFFu, touched);
  if (lane == 0) {
    if (removed) atomicAdd(&sc->n_deleted, (unsigned long long)removed);
    if (touched) atomicAdd(&sc->n_touched_est, (unsigned long long)touched);
  }
}

}  // namespace iso
