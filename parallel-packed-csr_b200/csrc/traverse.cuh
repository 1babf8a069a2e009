// traverse.cuh -- traversals across the shards of a group (ppcsr_group_bfs / ppcsr_group_pagerank, group.inl).
//
// BFS: level synchronous like qry::k_bfs_frontier, routed like batch::k_bin_scatter_peers -- atomics stay on the GPU
// that issues them, only plain stores cross GPUs.  Per level:
//   1. expand (sender s, its stream): warp per frontier vertex over its slot range; every live dst < n_global that s
//      has not forwarded before (test-and-set in s's bitmap `seen` of the GLOBAL vertices) takes a place in s's
//      cursor for its owner (one atomicAdd per warp and owner) and is stored, as a local id of the owner, into region
//      s of the owner's inbox.  k_group_bfs_publish then deposits the cursors in the owners' count arrays.
//   2. merge (owner p, its stream, after every sender's event): the entries of every region between the count seen
//      at the previous level and the count just published claim their distance (atomicCAS from UINT32_MAX); the
//      winners form p's next frontier.  k_group_bfs_level_end hands its size to the host.
// The inbox is an append-only log for the whole BFS.  Capacity bound: sender s forwards each global vertex at most
// once per BFS (its `seen` bit), and only vertices owned by p go to p, so region s of owner p never receives more
// than n_p entries.  Regions of n_p entries therefore cannot overflow, nothing is reset between levels, and no
// atomic ever targets another GPU's memory.
//
// PageRank: every shard pushes into its own full-length fp64 accumulator (global dst ids, qry::k_pagerank_push*),
// then every owner sums its slice of all accumulators in the fixed shard order (k_group_pagerank_reduce): the
// reduce-scatter is the only traffic between GPUs.
#pragma once
#include "batch.cuh"
#include "common.cuh"

namespace trv {

constexpr int TT = 256;
constexpr uint32_t MAX_PARTS = batch::BIN_MAX_PARTS;

// Where the BFS entries of every owner go (device pointers, peer-mapped where the owner is another GPU).
struct InboxTable {
  uint32_t *inbox[MAX_PARTS];  // owner p: n_shards regions of region[p] entries
  uint32_t *cnt[MAX_PARTS];    // owner p: n_shards counts, entry s written by sender s
  uint32_t start[MAX_PARTS];   // first global vertex of every owner (vertex ids are 32-bit)
  uint32_t region[MAX_PARTS];  // entries per region of owner p = its vertex count
};

// owner of v: the last shard whose first vertex is <= v (reference PPPCSR::get_partiton: the first boundary greater
// than v, otherwise the last shard).  Branch-free over the table padded with UINT32_MAX.
__device__ __forceinline__ uint32_t owner_of(const uint32_t *s_start, uint32_t parts, uint32_t v) {
  uint32_t d = 0;
#pragma unroll
  for (uint32_t step = MAX_PARTS / 2; step >= 1; step >>= 1)
    if (d + step < parts && s_start[d + step] <= v) d += step;
  return d;
}

__global__ void __launch_bounds__(TT) k_group_bfs_expand(const uint32_t *__restrict__ dest,
                                                         const uint32_t *__restrict__ leaf_cnt,
                                                         const uint32_t *__restrict__ beg, uint32_t ls,
                                                         uint32_t n_global, uint32_t parts, uint32_t me,
                                                         const uint32_t *__restrict__ frontier, uint32_t n_frontier,
                                                         uint32_t *seen, uint32_t *__restrict__ cursor,
                                                         InboxTable T) {
  __shared__ uint32_t s_start[MAX_PARTS];
  if (threadIdx.x < MAX_PARTS) s_start[threadIdx.x] = threadIdx.x < parts ? T.start[threadIdx.x] : 0xFFFFFFFFu;
  __syncthreads();
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
        if (d < n_global) {  // dst is not range checked on insert
          const uint32_t bit = 1u << (d & 31u);
          fresh = (seen[d >> 5] & bit) == 0u && (atomicOr(&seen[d >> 5], bit) & bit) == 0u;
        }
      }
      if (!__ballot_sync(0xFFFFFFFFu, fresh)) continue;
      const uint32_t own = fresh ? owner_of(s_start, parts, d) : 0xFFFFFFFFu;
      const unsigned peers = __match_any_sync(0xFFFFFFFFu, own);
      const uint32_t leader = (uint32_t)__ffs(peers) - 1u;
      uint32_t at = 0;
      if (fresh && lane == leader) at = atomicAdd(&cursor[own], (uint32_t)__popc(peers));
      at = __shfl_sync(0xFFFFFFFFu, at, leader);
      if (fresh) T.inbox[own][(size_t)me * T.region[own] + at + __popc(peers & lt)] = d - s_start[own];
    }
  }
}

// after the expand: this sender's cursor for every owner, deposited at the owner
__global__ void k_group_bfs_publish(uint32_t parts, uint32_t me, const uint32_t *__restrict__ cursor, InboxTable T) {
  if (threadIdx.x < parts) T.cnt[threadIdx.x][me] = cursor[threadIdx.x];
}

// owner side: every entry of region s in [seen_cnt[s], cnt[s]) is a local vertex reached at level + 1 unless it
// already has a distance
__global__ void __launch_bounds__(TT) k_group_bfs_merge(const uint32_t *__restrict__ inbox, uint32_t region,
                                                        const uint32_t *__restrict__ cnt,
                                                        const uint32_t *__restrict__ seen_cnt, uint32_t parts,
                                                        uint32_t *__restrict__ dist, uint32_t level,
                                                        uint32_t *__restrict__ next, uint32_t *n_next) {
  const uint32_t lane = lane_id();
  const unsigned lt = lanemask_lt();
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t s = 0; s < parts; s++) {
    const uint32_t lo = seen_cnt[s], hi = cnt[s];
    const uint32_t *reg = inbox + (size_t)s * region;
    // warp-uniform trip count: the whole warp reaches the ballot
    for (uint32_t i0 = lo + (blockIdx.x * blockDim.x + threadIdx.x - lane); i0 < hi; i0 += stride) {
      const uint32_t i = i0 + lane;
      bool fresh = false;
      uint32_t v = 0;
      if (i < hi) {
        v = reg[i];
        fresh = atomicCAS(&dist[v], 0xFFFFFFFFu, level + 1u) == 0xFFFFFFFFu;
      }
      const unsigned m = __ballot_sync(0xFFFFFFFFu, fresh);
      if (m) {
        uint32_t at = 0;
        const unsigned leader = (unsigned)__ffs(m) - 1u;
        if (lane == leader) at = atomicAdd(n_next, (uint32_t)__popc(m));
        at = __shfl_sync(0xFFFFFFFFu, at, leader);
        if (fresh) next[at + __popc(m & lt)] = v;
      }
    }
  }
}

// one block: the counts just merged become the start of the next level's ranges, the next frontier's size goes to
// pinned host memory (mapped: the kernel stores it there directly) and the counter restarts at 0
__global__ void k_group_bfs_level_end(uint32_t parts, const uint32_t *__restrict__ cnt, uint32_t *__restrict__ seen_cnt,
                                      uint32_t *n_next, uint32_t *h_front) {
  if (threadIdx.x < parts) seen_cnt[threadIdx.x] = cnt[threadIdx.x];
  if (threadIdx.x == 0) {
    *h_front = *n_next;
    *n_next = 0;
  }
}

struct AccTable {
  double *acc[MAX_PARTS];  // every shard's full-length accumulator (peer-mapped)
};

// owner side of one PageRank iteration: r[v] = base + damping * sum_q acc_q[first + v], summed over q = 0..parts-1 in
// this fixed order (coalesced peer loads), then every entry read is cleared for the next push
__global__ void __launch_bounds__(TT) k_group_pagerank_reduce(AccTable A, uint32_t parts, uint64_t first, uint32_t n,
                                                              double *__restrict__ r, double base, double damping) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  const uint64_t i = first + v;
  double sum = A.acc[0][i];
  for (uint32_t q = 1; q < parts; q++) sum += A.acc[q][i];  // loads only: all of them in flight
  for (uint32_t q = 0; q < parts; q++) A.acc[q][i] = 0.0;
  r[v] = base + damping * sum;
}

}  // namespace trv
