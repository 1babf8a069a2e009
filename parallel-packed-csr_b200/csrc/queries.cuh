// queries.cuh -- read side: point queries, neighbour scans, CSR export, the PageRank push step,
// level-synchronous BFS and the PMA invariant checker.
// Replaces reference PCSR::edge_exists / get_neighbourhood / read_neighbourhood (src/pcsr/PCSR.cpp:860-912),
// pagerank.h:16-29 and bfs.h:15-36.
#pragma once
#include "batch.cuh"
#include "common.cuh"
#include "primitives.cuh"

namespace qry {

constexpr int QT = 256;

__global__ void __launch_bounds__(QT) k_edges_exist(const uint32_t *__restrict__ src, const uint32_t *__restrict__ dst,
                                                    size_t count, uint32_t n, const uint32_t *__restrict__ dest,
                                                    const uint32_t *__restrict__ val,
                                                    const uint32_t *__restrict__ leaf_cnt,
                                                    const uint32_t *__restrict__ beg, uint32_t ls,
                                                    uint8_t *__restrict__ exists, uint32_t *__restrict__ out_val) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const uint32_t s = src[i], d = dst[i];
  uint8_t hit = 0;
  uint32_t v = 0;
  if (s < n && d != PPCSR_SENT) {
    uint32_t slot;
    if (batch::find_edge(dest, leaf_cnt, beg[s], beg[s + 1], ls, d, &slot)) {
      hit = 1;
      v = val[slot];
    }
  }
  exists[i] = hit;
  if (out_val) out_val[i] = v;
}

// global live rank of a slot: rank_off[leaf] + offset (valid for live slots and for slot == N)
__device__ __forceinline__ uint32_t slot_rank(const uint32_t *__restrict__ rank_off, uint32_t ls, uint32_t slot) {
  return rank_off[slot >> ls] + (slot & ((1u << ls) - 1u));
}

// rowptr[v] = live non-sentinel items before v's sentinel = rank(beg[v]) - v
__global__ void __launch_bounds__(QT) k_rowptr(const uint32_t *__restrict__ beg, const uint32_t *__restrict__ rank_off,
                                               uint32_t ls, uint32_t n, uint64_t *__restrict__ rowptr) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v > n) return;
  rowptr[v] = (uint64_t)slot_rank(rank_off, ls, beg[v]) - v;
}

// all live non-sentinel slots in array order = the concatenated adjacency lists
struct InIsEdge {
  const uint32_t *dest, *leaf_cnt;
  uint32_t ls;
  __device__ uint32_t operator()(size_t slot) const {
    const uint32_t f = (uint32_t)slot & ((1u << ls) - 1u);
    return (f < leaf_cnt[slot >> ls] && dest[slot] != PPCSR_SENT) ? 1u : 0u;
  }
};
struct OutEdge {
  const uint32_t *dest, *val;
  uint32_t *col, *w;
  __device__ void operator()(size_t slot, uint32_t ex, uint32_t own) const {
    if (own) {
      col[ex] = dest[slot];
      if (w) w[ex] = val[slot];
    }
  }
};

// neighbours of one vertex, ascending (get_neighbourhood): live slots of (beg[v], beg[v+1])
__global__ void __launch_bounds__(QT) k_neighbours(const uint32_t *__restrict__ dest,
                                                   const uint32_t *__restrict__ leaf_cnt,
                                                   const uint32_t *__restrict__ rank_off, uint32_t ls, uint32_t b,
                                                   uint32_t e, uint32_t *__restrict__ out, uint64_t cap) {
  const uint32_t r0 = slot_rank(rank_off, ls, b) + 1;
  for (uint32_t slot = b + 1 + blockIdx.x * blockDim.x + threadIdx.x; slot < e; slot += gridDim.x * blockDim.x) {
    const uint32_t f = slot & ((1u << ls) - 1u);
    if (f < leaf_cnt[slot >> ls]) {
      const uint32_t k = rank_off[slot >> ls] + f - r0;
      if (k < cap) out[k] = dest[slot];
    }
  }
}

// read_neighbourhood: touch every slot of the range (PCSR.cpp:892-899), return a checksum so the loads stay
__global__ void __launch_bounds__(QT) k_touch(const uint32_t *__restrict__ dest, uint32_t b, uint32_t e,
                                              unsigned long long *sum) {
  unsigned long long acc = 0;
  for (uint32_t slot = b + 1 + blockIdx.x * blockDim.x + threadIdx.x; slot < e; slot += gridDim.x * blockDim.x)
    acc += dest[slot];
  for (int d = 16; d; d >>= 1) acc += __shfl_down_sync(0xFFFFFFFFu, acc, d);
  if (lane_id() == 0 && acc) atomicAdd(sum, acc);
}

// ---- PageRank push step, leaf walk: a warp streams a run of consecutive 32-slot groups ----------------------
// out[dst] += in[v] / num_neighbors[v] for every edge (v,dst)  (reference pagerank.h:19-26; the divisor is the
// call-count num_neighbors, not the degree).  A vertex without live edges contributes nothing, whatever its divisor.
// A warp per vertex would pay a dependent chain (beg[v], beg[v+1], in[v], nn[v]) per vertex and leave most lanes idle
// on an R-MAT graph (half of the vertices own at most a couple of edges).  The packed array itself
// carries everything a full scan needs, in order: a sentinel (dest == SENT, val == v + 1) opens vertex v's run, every
// live slot after it is one of v's edges.  So: one coalesced 128-byte read of dest[] per group, the sentinels of the
// group fetch their vertex's contribution, a ballot + shuffle hands every edge the contribution of the nearest
// sentinel below it (or the one carried in from the previous group), and the warp finds the vertex of its first
// slot with ONE binary search over beg[].  The contribution is computed in W, the accumulation is fp64.
constexpr int PRL_BATCH = 4;  // groups whose loads are issued together
template <typename W>
__global__ void __launch_bounds__(QT) k_pagerank_push_leaves(const uint32_t *__restrict__ dest,
                                                             const uint32_t *__restrict__ val,
                                                             const uint32_t *__restrict__ leaf_cnt,
                                                             const uint32_t *__restrict__ beg,
                                                             const uint32_t *__restrict__ nn, uint32_t ls, uint32_t n,
                                                             uint64_t n_slots, const W *__restrict__ in,
                                                             double *__restrict__ acc, uint64_t out_len) {
  const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
  const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = lane_id();
  const uint32_t groups = (uint32_t)(n_slots >> 5);
  const uint32_t per = (groups + warps - 1) / warps;
  const uint32_t g0 = min(w * per, groups), g1 = min(g0 + per, groups);
  if (g0 >= g1 || n == 0) return;
  // vertex owning the first slot of my run: the last v with beg[v] <= slot (beg[0] == 0)
  W carry;
  {
    const uint32_t s0 = g0 << 5;
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1) {
      const uint32_t mid = lo + ((hi - lo) >> 1);
      if (beg[mid] <= s0) lo = mid;
      else hi = mid;
    }
    carry = in[lo] / (W)nn[lo];
  }
  const uint32_t lsm = (1u << ls) - 1u;
  const unsigned le = lanemask_lt() | (1u << lane);
  for (uint32_t g = g0; g < g1; g += PRL_BATCH) {
    uint32_t d[PRL_BATCH];
    bool live[PRL_BATCH];
#pragma unroll
    for (int u = 0; u < PRL_BATCH; u++) {
      const uint32_t slot = ((g + u) << 5) + lane;
      live[u] = g + u < g1 && (slot & lsm) < leaf_cnt[slot >> ls];
      d[u] = live[u] ? dest[slot] : 0u;
    }
#pragma unroll
    for (int u = 0; u < PRL_BATCH; u++) {
      if (g + u >= g1) break;  // warp-uniform
      const bool sent = live[u] && d[u] == PPCSR_SENT;
      W c = (W)0;
      if (sent) {
        const uint32_t v = val[((g + u) << 5) + lane] - 1u;
        c = in[v] / (W)nn[v];
      }
      const unsigned m = __ballot_sync(0xFFFFFFFFu, sent);
      const unsigned below = m & le;
      W mine = __shfl_sync(0xFFFFFFFFu, c, below ? 31 - __clz(below) : 0);
      if (!below) mine = carry;
      if (live[u] && !sent && d[u] < out_len) atomicAdd(&acc[d[u]], (double)mine);
      if (m) carry = __shfl_sync(0xFFFFFFFFu, c, 31 - __clz(m));
    }
  }
}

// iterated PageRank: r[v] = base + damping * acc[v]; acc is cleared for the next push step
__global__ void k_pagerank_finish(double *__restrict__ r, double *__restrict__ acc, uint64_t n, double base,
                                  double damping) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    r[i] = base + damping * acc[i];
    acc[i] = 0.0;
  }
}
__global__ void k_fill_f64(double *__restrict__ p, double v, uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
template <typename W>
__global__ void k_cast_out(const double *__restrict__ acc, W *__restrict__ out, uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (W)acc[i];
}
template <typename W>
__global__ void k_cast_in(const W *__restrict__ in, double *__restrict__ out, uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (double)in[i];
}

// ---- BFS (level synchronous, frontier queues; reference src/utility/bfs.h:15-36) -------------------------------
// One warp per vertex of the current frontier scans its slot range; a neighbour reached for the first time
// (compare-and-swap on its distance) joins the next frontier, the warp takes its places in the queue with one atomic.
// Work per level is O(frontier edges), not O(n).
__global__ void __launch_bounds__(QT) k_bfs_frontier(const uint32_t *__restrict__ dest,
                                                     const uint32_t *__restrict__ leaf_cnt,
                                                     const uint32_t *__restrict__ beg, uint32_t ls, uint32_t n,
                                                     uint32_t *__restrict__ dist, uint32_t level,
                                                     const uint32_t *__restrict__ frontier, uint32_t n_frontier,
                                                     uint32_t *__restrict__ next, uint32_t *n_next) {
  const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
  const uint32_t lane = lane_id();
  const unsigned lt = lanemask_lt();
  for (uint32_t f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; f < n_frontier; f += warps) {
    const uint32_t v = frontier[f];
    const uint32_t b = beg[v], e = beg[v + 1];
    for (uint32_t base = b + 1; base < e; base += 32) {
      const uint32_t slot = base + lane;
      bool fresh = false;
      uint32_t d = 0;
      if (slot < e && (slot & ((1u << ls) - 1u)) < leaf_cnt[slot >> ls]) {
        d = dest[slot];
        fresh = d < n && atomicCAS(&dist[d], 0xFFFFFFFFu, level + 1u) == 0xFFFFFFFFu;
      }
      const unsigned m = __ballot_sync(0xFFFFFFFFu, fresh);
      if (m) {
        uint32_t at = 0;
        const unsigned leader = (unsigned)__ffs(m) - 1u;
        if (lane == leader) at = atomicAdd(n_next, (uint32_t)__popc(m));
        at = __shfl_sync(0xFFFFFFFFu, at, leader);
        if (fresh) next[at + __popc(m & lt)] = d;
      }
    }
  }
}
__global__ void k_fill_u32(uint32_t *p, uint32_t v, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// ---- checksum of the logical graph (parity anchor at sizes where an adjacency dump is impractical) -----------
// edges, sum of mix64(global_src << 32 | dst) over all edges, sum of num_neighbors[v] * mix64(global v) -- the same
// order-independent sums oracle/ref_driver.cpp --checksum takes over the reference's get_neighbourhood().  Same leaf
// walk as the PageRank push: the sentinels carry the source vertex.
__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
  x ^= x >> 30;
  x *= 0xBF58476D1CE4E5B9ull;
  x ^= x >> 27;
  x *= 0x94D049BB133111EBull;
  x ^= x >> 31;
  return x;
}
__global__ void __launch_bounds__(QT) k_checksum_leaves(const uint32_t *__restrict__ dest,
                                                        const uint32_t *__restrict__ val,
                                                        const uint32_t *__restrict__ leaf_cnt,
                                                        const uint32_t *__restrict__ beg, uint32_t ls, uint32_t n,
                                                        uint64_t n_slots, unsigned long long vertex_offset,
                                                        unsigned long long *__restrict__ out) {
  const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
  const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = lane_id();
  const uint32_t groups = (uint32_t)(n_slots >> 5);
  const uint32_t per = (groups + warps - 1) / warps;
  const uint32_t g0 = min(w * per, groups), g1 = min(g0 + per, groups);
  if (g0 >= g1 || n == 0) return;
  uint32_t carry;  // vertex owning the first slot of my run: the last v with beg[v] <= slot
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
  const uint32_t lsm = (1u << ls) - 1u;
  const unsigned le = lanemask_lt() | (1u << lane);
  unsigned long long cnt = 0, hash = 0;
  for (uint32_t g = g0; g < g1; g++) {
    const uint32_t slot = (g << 5) + lane;
    const bool live = (slot & lsm) < leaf_cnt[slot >> ls];
    const uint32_t d = live ? dest[slot] : 0u;
    const bool sent = live && d == PPCSR_SENT;
    const uint32_t sv = sent ? val[slot] - 1u : 0u;
    const unsigned m = __ballot_sync(0xFFFFFFFFu, sent);
    const unsigned below = m & le;
    uint32_t mine = __shfl_sync(0xFFFFFFFFu, sv, below ? 31 - __clz(below) : 0);
    if (!below) mine = carry;
    if (live && !sent) {
      cnt++;
      hash += mix64(((vertex_offset + mine) << 32) | d);
    }
    if (m) carry = __shfl_sync(0xFFFFFFFFu, sv, 31 - __clz(m));
  }
  for (int o = 16; o; o >>= 1) {
    cnt += __shfl_down_sync(0xFFFFFFFFu, cnt, o);
    hash += __shfl_down_sync(0xFFFFFFFFu, hash, o);
  }
  if (lane == 0) {
    atomicAdd(&out[0], cnt);
    atomicAdd(&out[1], hash);
  }
}
__global__ void __launch_bounds__(QT) k_checksum_nn(const uint32_t *__restrict__ nn, uint32_t n,
                                                    unsigned long long vertex_offset,
                                                    unsigned long long *__restrict__ out) {
  unsigned long long acc = 0;
  for (uint32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < n; v += gridDim.x * blockDim.x)
    acc += (unsigned long long)nn[v] * mix64(vertex_offset + v);
  for (int o = 16; o; o >>= 1) acc += __shfl_down_sync(0xFFFFFFFFu, acc, o);
  if (lane_id() == 0 && acc) atomicAdd(&out[2], acc);
}

// ---- invariants (SURVEY §8a I1-I6) -------------------------------------------------------------------
struct InvCounters {
  unsigned long long bad_sentinel, bad_order, bad_leaf_layout, bad_upper, bad_lower, bad_tree, live_items, sentinels,
      full_leaves;
};

// one thread per leaf: left-packed layout, null tail, ascending order inside the leaf and across to the
// next non-empty leaf (a sentinel restarts the order: the next vertex begins)
__global__ void __launch_bounds__(QT) k_check_leaves(const uint32_t *__restrict__ dest,
                                                     const uint32_t *__restrict__ val,
                                                     const uint32_t *__restrict__ leaf_cnt,
                                                     const uint32_t *__restrict__ tree, uint32_t n_leaves, uint32_t ls,
                                                     InvCounters *c) {
  const uint32_t l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= n_leaves) return;
  const uint32_t logN = 1u << ls, cnt = leaf_cnt[l];
  const size_t base = (size_t)l << ls;
  unsigned bad_layout = 0, bad_order = 0, sent = 0;
  if (cnt > logN) bad_layout++;
  if (tree[n_leaves + l] != cnt) atomicAdd(&c->bad_tree, 1ull);
  if (cnt == logN) atomicAdd(&c->full_leaves, 1ull);
  uint32_t prev = 0;
  bool have_prev = false;
  for (uint32_t f = 0; f < logN; f++) {
    const uint32_t d = dest[base + f], v = val[base + f];
    if (f < cnt) {
      if (v == 0) bad_layout++;
      if (d == PPCSR_SENT) {
        sent++;
        have_prev = false;
      } else {
        if (have_prev && d <= prev) bad_order++;
        prev = d;
        have_prev = true;
      }
    } else if (v != 0 || d != 0) {
      bad_layout++;
    }
  }
  if (cnt > 0 && have_prev) {  // compare with the first item of the next non-empty leaf
    uint32_t l2 = l + 1;
    while (l2 < n_leaves && leaf_cnt[l2] == 0) l2++;
    if (l2 < n_leaves) {
      const uint32_t d2 = dest[(size_t)l2 << ls];
      if (d2 != PPCSR_SENT && d2 <= prev) bad_order++;
    }
  }
  if (bad_layout) atomicAdd(&c->bad_leaf_layout, (unsigned long long)bad_layout);
  if (bad_order) atomicAdd(&c->bad_order, (unsigned long long)bad_order);
  {  // every leaf adds to the same two words: sum over the warp first
    const unsigned peers = __activemask();
    const uint32_t w_sent = __reduce_add_sync(peers, sent), w_cnt = __reduce_add_sync(peers, cnt);
    if ((peers & ((1u << (threadIdx.x & 31u)) - 1u)) == 0u) {
      if (w_sent) atomicAdd(&c->sentinels, (unsigned long long)w_sent);
      if (w_cnt) atomicAdd(&c->live_items, (unsigned long long)w_cnt);
    }
  }
}

__global__ void __launch_bounds__(QT) k_check_vertices(const uint32_t *__restrict__ dest,
                                                       const uint32_t *__restrict__ val,
                                                       const uint32_t *__restrict__ leaf_cnt,
                                                       const uint32_t *__restrict__ beg, uint32_t n, uint64_t N,
                                                       uint32_t ls, InvCounters *c) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v > n) return;
  if (v == n) {
    if (beg[n] != (uint32_t)N) atomicAdd(&c->bad_sentinel, 1ull);
    return;
  }
  const uint32_t b = beg[v];
  bool bad = b >= N || b >= beg[v + 1];
  if (!bad) {
    bad = dest[b] != PPCSR_SENT || val[b] != v + 1u || (b & ((1u << ls) - 1u)) >= leaf_cnt[b >> ls];
  }
  if (bad) atomicAdd(&c->bad_sentinel, 1ull);
}

__global__ void __launch_bounds__(QT) k_check_tree(const uint32_t *__restrict__ tree, uint32_t n_leaves,
                                                   InvCounters *c) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x + 1;
  if (i >= n_leaves) return;  // internal nodes 1 .. n_leaves-1
  if (tree[i] != tree[2 * i] + tree[2 * i + 1]) atomicAdd(&c->bad_tree, 1ull);
}

// density bounds on every path touched by the last batch (ins_cnt/del_cnt still hold its per-leaf counts, unless
// the batch rebuilt the whole array)
__global__ void __launch_bounds__(QT) k_check_bounds(const uint32_t *__restrict__ tree,
                                                     const uint32_t *__restrict__ ins_cnt,
                                                     const uint32_t *__restrict__ del_cnt, uint32_t all_touched,
                                                     uint32_t n_leaves, uint32_t logN, int H, int check_lower,
                                                     InvCounters *c) {
  const uint32_t l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= n_leaves) return;
  // all_touched bit 2: the last batch rewrote the whole array -- every leaf counts as touched by its inserts (bit 0)
  // and deletes (bit 1), and the per-leaf arrays are not meaningful
  const bool ins = (all_touched & 4u) ? (all_touched & 1u) != 0 : ins_cnt[l] != 0;
  const bool del = (all_touched & 4u) ? (all_touched & 2u) != 0 : del_cnt[l] != 0;
  if (!ins && !del) return;
  uint32_t node = n_leaves + l;
  uint64_t len = logN;
  unsigned up = 0, lo = 0;
  for (int depth = H; depth >= 0; depth--) {
    const uint32_t cnt = tree[node];
    if (ins && !window_ok_upper(cnt, len, logN, depth, H)) up++;
    if (del && check_lower && !window_ok_lower(cnt, len, depth, H)) lo++;
    node >>= 1;
    len <<= 1;
  }
  if (up) atomicAdd(&c->bad_upper, (unsigned long long)up);
  if (lo) atomicAdd(&c->bad_lower, (unsigned long long)lo);
}

}  // namespace qry
