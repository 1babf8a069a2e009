// batch.cuh -- front half of the batch pipeline:
//   build 64-bit keys (src<<32 | dst) with the reference's guards  -> radix sort -> last-op-wins
//   -> num_neighbors call counts -> segmented search of every unique update inside its vertex range
//   -> per-leaf insert/delete counts and the compacted, key-ordered insert list.
// Replaces, per update, reference PCSR::add_edge_parallel / remove_edge up to and including
// PCSR::binary_search (src/pcsr/PCSR.cpp:1374-1424, 709-747, 427-502).
#pragma once
#include "common.cuh"
#include "primitives.cuh"
#include "sort.cuh"

namespace batch {

enum : uint8_t { CLS_INSERT = 0, CLS_OVERWRITE = 1, CLS_DELETE = 2, CLS_MISS = 3 };

constexpr int BT = 256;
constexpr int BIN_MAX_PARTS = 64;  // shards a batch can be routed to

// Per-update values ride along as the payload of the sort -- unless they are all the same: a mixed stream of adds (one
// value, e.g. the thread pools' 1) and removes needs ONE bit per update, and bit 63 of the key word is free as long as
// vertex ids stay below 2^31 (the sort's digits cover only the live (src,dst) field, so the bit travels with the key
// without taking part in the order).  The builders set it for removes and report the largest and the smallest
// non-zero value; the host then sorts keys only when they coincide (8 instead of 12 bytes per update and pass).
constexpr uint64_t KEY_OP_BIT = 1ull << 63;
__device__ __forceinline__ uint64_t emit_key(bool ok, uint64_t key, uint32_t v, uint32_t n, uint32_t op_bit) {
  if (!ok) return (uint64_t)n << 32;  // rejected: sorts behind every valid key
  return (op_bit && v == 0u) ? (key | KEY_OP_BIT) : key;
}

// ---- raw key sources: the sort's first pass (prim::k_os_pass / k_os_hist / k_sort_small) builds the key word of
// update i straight from the caller's arrays, guards included, so the unsorted batch is never written as a key array.
// Same arithmetic as the builders below (which then only take the scalars and the histograms).
__device__ __forceinline__ bool update_ok(uint32_t s, uint32_t d, uint32_t v, uint32_t n) {
  return s < n && !(v != 0 && d == PPCSR_SENT);
}
struct RawArrays {
  const uint32_t *src, *dst, *val;  // val nullable: every update carries default_val
  uint32_t default_val, n, op_bit;
  __device__ __forceinline__ uint64_t key(size_t i) const {
    const uint32_t s = src[i], d = dst[i], v = val ? val[i] : default_val;
    return emit_key(update_ok(s, d, v, n), ((uint64_t)s << 32) | d, v, n, op_bit);
  }
  __device__ __forceinline__ uint32_t payload(size_t i) const {
    const uint32_t v = val[i];
    return update_ok(src[i], dst[i], v, n) ? v : 0u;
  }
};
struct RawPacked {
  const uint64_t *packed;
  const uint32_t *val;
  uint32_t default_val, n, op_bit, swap_halves;
  __device__ __forceinline__ uint64_t word(size_t i) const {
    const uint64_t k = packed[i];
    return swap_halves ? (k << 32) | (k >> 32) : k;
  }
  __device__ __forceinline__ uint64_t key(size_t i) const {
    const uint64_t k = word(i);
    const uint32_t v = val ? val[i] : default_val;
    return emit_key(update_ok((uint32_t)(k >> 32), (uint32_t)k, v, n), k, v, n, op_bit);
  }
  __device__ __forceinline__ uint32_t payload(size_t i) const {
    const uint64_t k = word(i);
    const uint32_t v = val[i];
    return update_ok((uint32_t)(k >> 32), (uint32_t)k, v, n) ? v : 0u;
  }
};
// records deposited by the peers: n_seg regions of `cap` records, region r holding prefix[r + 1] - prefix[r] of them
// (prefix: a DEVICE array written by k_build_keys_segments)
struct RawSegments {
  const uint64_t *packed;
  const uint32_t *val;
  const unsigned long long *prefix;
  unsigned long long cap;
  uint32_t n_seg, default_val, n, op_bit;
  __device__ __forceinline__ size_t at(size_t i) const {
    uint32_t lo = 0, hi = n_seg;  // last region with prefix <= i
    while (hi - lo > 1) {
      const uint32_t mid = (lo + hi) >> 1;
      if (prefix[mid] <= i) lo = mid;
      else hi = mid;
    }
    return (size_t)lo * cap + (i - (size_t)prefix[lo]);
  }
  __device__ __forceinline__ uint64_t key(size_t i) const {
    const size_t a = at(i);
    const uint64_t k = packed[a];
    const uint32_t v = val ? val[a] : default_val;
    return emit_key(update_ok((uint32_t)(k >> 32), (uint32_t)k, v, n), k, v, n, op_bit);
  }
  __device__ __forceinline__ uint32_t payload(size_t i) const {
    const size_t a = at(i);
    const uint64_t k = packed[a];
    const uint32_t v = val[a];
    return update_ok((uint32_t)(k >> 32), (uint32_t)k, v, n) ? v : 0u;
  }
};

// The key builders can also take the sort's digit histograms (all passes, prim::k_os_hist's job) while the keys pass
// through their registers: the host SPECULATES the sort layout from the widest dst seen so far and the vertex count,
// and falls back to prim::k_os_hist when the batch turns out wider (capi.cu).  Saves one read of the batch.
struct HistArgs {
  prim::SortPasses P;
  uint32_t *ghist;  // nullptr: no histogram
};
__device__ __forceinline__ void hist_init(uint32_t *s_h, const HistArgs &H) {
  if (H.ghist)
    for (int i = threadIdx.x; i < H.P.n_pass * prim::OS_RADIX; i += blockDim.x) s_h[i] = 0;
}
__device__ __forceinline__ void hist_add(uint32_t *s_h, const HistArgs &H, uint64_t key) {
  if (!H.ghist) return;
  const uint64_t ck = prim::sort_compact(key, H.P.lo_bits);
#pragma unroll
  for (int p = 0; p < prim::OS_MAX_PASSES; p++)
    if (p < H.P.n_pass) atomicAdd(&s_h[p * prim::OS_RADIX + ((uint32_t)(ck >> H.P.shift[p]) & H.P.mask[p])], 1u);
}
__device__ __forceinline__ void hist_flush(const uint32_t *s_h, const HistArgs &H) {  // after a block barrier
  if (H.ghist)
    for (int i = threadIdx.x; i < H.P.n_pass * prim::OS_RADIX; i += blockDim.x)
      if (s_h[i]) atomicAdd(&H.ghist[i], s_h[i]);
}

// ---- keys -------------------------------------------------------------------------------------
// Guards: add with value != 0 needs src < n (reference PCSR.cpp:1375) and dst != SENT; remove needs
// src < n (the reference would read out of bounds, PCSR.cpp:717).  Rejected updates get the key
// (n << 32), which sorts after every valid key, and are counted.
__global__ void __launch_bounds__(BT) k_build_keys(const uint32_t *__restrict__ src, const uint32_t *__restrict__ dst,
                                                   const uint32_t *__restrict__ val, uint32_t default_val,
                                                   size_t count, uint32_t n, uint32_t op_bit, uint64_t *__restrict__ keys,
                                                   uint32_t *__restrict__ pay, BatchScalars *sc, HistArgs H) {
  __shared__ uint32_t s_or, s_bad, s_vmax, s_vinv;
  __shared__ uint32_t s_h[prim::OS_MAX_PASSES * prim::OS_RADIX];
  hist_init(s_h, H);
  if (threadIdx.x == 0) {
    s_or = 0;
    s_bad = 0;
    s_vmax = 0;
    s_vinv = 0;
  }
  __syncthreads();
  uint32_t my_or = 0, my_bad = 0, my_vmax = 0, my_vinv = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
    const uint32_t s = src[i], d = dst[i];
    const uint32_t v = val ? val[i] : default_val;
    const bool ok = s < n && !(v != 0 && d == PPCSR_SENT);
    const uint64_t kq = emit_key(ok, ((uint64_t)s << 32) | d, v, n, op_bit);
    if (keys) keys[i] = kq;  // nullptr: the sort reads the raw arrays itself (RawArrays)
    hist_add(s_h, H, kq);
    if (pay && keys) pay[i] = ok ? v : 0u;
    if (ok) my_or |= d;
    else my_bad++;
    if (pay && ok && v) my_vmax = max(my_vmax, v), my_vinv = max(my_vinv, ~v);
  }
  my_or = __reduce_or_sync(0xFFFFFFFFu, my_or);
  my_bad = __reduce_add_sync(0xFFFFFFFFu, my_bad);
  my_vmax = __reduce_max_sync(0xFFFFFFFFu, my_vmax);
  my_vinv = __reduce_max_sync(0xFFFFFFFFu, my_vinv);
  if (lane_id() == 0) {
    if (my_or) atomicOr(&s_or, my_or);
    if (my_bad) atomicAdd(&s_bad, my_bad);
    if (my_vmax) atomicMax(&s_vmax, my_vmax);
    if (my_vinv) atomicMax(&s_vinv, my_vinv);
  }
  __syncthreads();
  hist_flush(s_h, H);
  if (threadIdx.x == 0) {
    if (s_or) atomicOr(&sc->dst_or, s_or);
    if (s_bad) atomicAdd(&sc->n_ignored, (unsigned long long)s_bad);
    if (s_vmax) atomicMax(&sc->val_max, s_vmax);
    if (s_vinv) atomicMax(&sc->val_inv_min, s_vinv);
  }
}

// same guards for records that arrive already packed as (src << 32 | dst) (the all-to-all payload)
__global__ void __launch_bounds__(BT) k_build_keys_packed(const uint64_t *__restrict__ packed,
                                                          const uint32_t *__restrict__ val, uint32_t default_val,
                                                          size_t count, uint32_t n, uint32_t op_bit, uint64_t *__restrict__ keys,
                                                          uint32_t *__restrict__ pay, BatchScalars *sc,
                                                          uint32_t swap_halves, HistArgs H) {
  // swap_halves: the records are interleaved little-endian (src, dst) pairs read as one word (dst << 32 | src)
  __shared__ uint32_t s_or, s_bad, s_vmax, s_vinv;
  __shared__ uint32_t s_h[prim::OS_MAX_PASSES * prim::OS_RADIX];
  hist_init(s_h, H);
  if (threadIdx.x == 0) {
    s_or = 0;
    s_bad = 0;
    s_vmax = 0;
    s_vinv = 0;
  }
  __syncthreads();
  uint32_t my_or = 0, my_bad = 0, my_vmax = 0, my_vinv = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
    uint64_t k = packed[i];
    if (swap_halves) k = (k << 32) | (k >> 32);
    const uint32_t s = (uint32_t)(k >> 32), d = (uint32_t)k;
    const uint32_t v = val ? val[i] : default_val;
    const bool ok = s < n && !(v != 0 && d == PPCSR_SENT);
    const uint64_t kq = emit_key(ok, k, v, n, op_bit);
    if (keys) keys[i] = kq;  // nullptr: the sort reads the raw records itself (RawPacked / RawSegments)
    hist_add(s_h, H, kq);
    if (pay && keys) pay[i] = ok ? v : 0u;
    if (ok) my_or |= d;
    else my_bad++;
    if (pay && ok && v) my_vmax = max(my_vmax, v), my_vinv = max(my_vinv, ~v);
  }
  my_or = __reduce_or_sync(0xFFFFFFFFu, my_or);
  my_bad = __reduce_add_sync(0xFFFFFFFFu, my_bad);
  my_vmax = __reduce_max_sync(0xFFFFFFFFu, my_vmax);
  my_vinv = __reduce_max_sync(0xFFFFFFFFu, my_vinv);
  if (lane_id() == 0) {
    if (my_or) atomicOr(&s_or, my_or);
    if (my_bad) atomicAdd(&s_bad, my_bad);
    if (my_vmax) atomicMax(&s_vmax, my_vmax);
    if (my_vinv) atomicMax(&s_vinv, my_vinv);
  }
  __syncthreads();
  hist_flush(s_h, H);
  if (threadIdx.x == 0) {
    if (s_or) atomicOr(&sc->dst_or, s_or);
    if (s_bad) atomicAdd(&sc->n_ignored, (unsigned long long)s_bad);
    if (s_vmax) atomicMax(&sc->val_max, s_vmax);
    if (s_vinv) atomicMax(&sc->val_inv_min, s_vinv);
  }
}

// Records that arrived through peer memory: `n_seg` regions of `cap` records each, region r holding prefix[r+1] -
// prefix[r] valid records (one region per sending rank, see k_bin_scatter_peers).  Same guards as above.
struct SegmentTable {
  uint32_t n_seg;
  uint64_t cap;
  const uint64_t *counts;  // DEVICE array: valid records of every region (deposited by the senders)
  unsigned long long *prefix_out;  // DEVICE array of n_seg + 1 entries (nullable): exclusive prefix of the counts
  uint64_t bound;  // keys the key array holds: a larger deposited total is reported (seg_total), not written
};
__global__ void __launch_bounds__(BT) k_build_keys_segments(const uint64_t *__restrict__ packed,
                                                            const uint32_t *__restrict__ val, uint32_t default_val,
                                                            SegmentTable T, uint32_t n, uint32_t op_bit, uint64_t *__restrict__ keys,
                                                            uint32_t *__restrict__ pay, BatchScalars *sc, HistArgs H) {
  __shared__ uint32_t s_or, s_bad, s_vmax, s_vinv;
  __shared__ uint32_t s_h[prim::OS_MAX_PASSES * prim::OS_RADIX];
  hist_init(s_h, H);
  __shared__ uint64_t s_prefix[BIN_MAX_PARTS + 1];  // exclusive prefix of the regions' counts
  if (threadIdx.x == 0) {
    s_or = 0;
    s_bad = 0;
    s_vmax = 0;
    s_vinv = 0;
    uint64_t run = 0;
    for (uint32_t r = 0; r < T.n_seg; r++) {
      s_prefix[r] = run;
      run += min(T.counts[r], T.cap);
    }
    s_prefix[T.n_seg] = run;
    if (blockIdx.x == 0) {
      sc->seg_total = run;  // the host learns the batch size with the sort width
      if (T.prefix_out)
        for (uint32_t r = 0; r <= T.n_seg; r++) T.prefix_out[r] = s_prefix[r];  // for RawSegments
    }
  }
  __syncthreads();
  uint32_t my_or = 0, my_bad = 0, my_vmax = 0, my_vinv = 0;
  const size_t count = min((size_t)s_prefix[T.n_seg], (size_t)T.bound);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t lo = 0, hi = T.n_seg;  // last region with prefix <= i
    while (hi - lo > 1) {
      const uint32_t mid = (lo + hi) >> 1;
      if (s_prefix[mid] <= i) lo = mid;
      else hi = mid;
    }
    const size_t at = (size_t)lo * T.cap + (i - (size_t)s_prefix[lo]);
    const uint64_t k = packed[at];
    const uint32_t s = (uint32_t)(k >> 32), d = (uint32_t)k;
    const uint32_t v = val ? val[at] : default_val;
    const bool ok = s < n && !(v != 0 && d == PPCSR_SENT);
    const uint64_t kq = emit_key(ok, k, v, n, op_bit);
    if (keys) keys[i] = kq;  // nullptr: the sort reads the raw records itself (RawPacked / RawSegments)
    hist_add(s_h, H, kq);
    if (pay && keys) pay[i] = ok ? v : 0u;
    if (ok) my_or |= d;
    else my_bad++;
    if (pay && ok && v) my_vmax = max(my_vmax, v), my_vinv = max(my_vinv, ~v);
  }
  my_or = __reduce_or_sync(0xFFFFFFFFu, my_or);
  my_bad = __reduce_add_sync(0xFFFFFFFFu, my_bad);
  my_vmax = __reduce_max_sync(0xFFFFFFFFu, my_vmax);
  my_vinv = __reduce_max_sync(0xFFFFFFFFu, my_vinv);
  if (lane_id() == 0) {
    if (my_or) atomicOr(&s_or, my_or);
    if (my_bad) atomicAdd(&s_bad, my_bad);
    if (my_vmax) atomicMax(&s_vmax, my_vmax);
    if (my_vinv) atomicMax(&s_vinv, my_vinv);
  }
  __syncthreads();
  hist_flush(s_h, H);
  if (threadIdx.x == 0) {
    if (s_or) atomicOr(&sc->dst_or, s_or);
    if (s_bad) atomicAdd(&sc->n_ignored, (unsigned long long)s_bad);
    if (s_vmax) atomicMax(&sc->val_max, s_vmax);
    if (s_vinv) atomicMax(&sc->val_inv_min, s_vinv);
  }
}

// ---- segmented search ----------------------------------------------------------------------------
// Finds (src,dst) inside vertex src's slot range (beg[src], beg[src+1]).  Two levels: a binary search
// over the LEAVES of the range on their first item (empty leaves are skipped to the right), then a
// lower_bound inside the chosen leaf's live prefix.  Returns true and the slot of the edge if it exists;
// otherwise false and the slot of its PREDECESSOR (the largest item with a smaller key -- at worst the
// vertex's own sentinel).  A new edge joins the leaf of its predecessor.
// Same contract as reference PCSR::binary_search (PCSR.cpp:427-502): position of the smallest element
// >= key, with the gap probing replaced by per-leaf live counts.
__device__ __forceinline__ bool find_edge(const uint32_t *__restrict__ dest, const uint32_t *__restrict__ leaf_cnt,
                                          uint32_t b, uint32_t e, uint32_t ls, uint32_t d, uint32_t *slot) {
  const uint32_t Lb = b >> ls, Le = (e - 1) >> ls;
  uint32_t lo = Lb, hi = Le + 1;
  while (hi - lo > 1) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    uint32_t m2 = mid;
    while (m2 < hi && leaf_cnt[m2] == 0) m2++;
    if (m2 == hi) {
      hi = mid;
      continue;
    }
    if (dest[(size_t)m2 << ls] <= d) lo = m2;
    else hi = mid;
  }
  const uint32_t base = lo << ls;
  const uint32_t cnt = leaf_cnt[lo];
  uint32_t f_lo = (lo == Lb) ? (b - base) + 1 : 0;
  uint32_t f_hi = cnt;
  if (lo == (e >> ls) && (e - base) < f_hi) f_hi = e - base;
  uint32_t x = f_lo, y = f_hi;  // lower_bound of d in dest[base + [f_lo, f_hi))
  while (x < y) {
    const uint32_t mid = (x + y) >> 1;
    if (dest[base + mid] < d) x = mid + 1;
    else y = mid;
  }
  if (x < f_hi && dest[base + x] == d) {
    *slot = base + x;
    return true;
  }
  *slot = base + x - 1;
  return false;
}

// find_edge over an explicit slot window and through (possibly staged) views of dest[] / leaf_cnt[]:
//   D[slot - doff] is dest[slot], C[leaf - coff] is leaf_cnt[leaf]; the search covers the slots [b, e) of ONE vertex,
//   `skip_first` says that slot b is the vertex's sentinel (false when the window was clipped from below: then b is
//   leaf aligned and its leaf holds an item <= d, see k_locate).  Same result as find_edge on the whole range.
__device__ __forceinline__ bool find_in(const uint32_t *D, uint32_t doff, const uint32_t *C, uint32_t coff, uint32_t b,
                                        uint32_t e, bool skip_first, uint32_t ls, uint32_t d, uint32_t *slot) {
  const uint32_t Lb = b >> ls, Le = (e - 1) >> ls;
  uint32_t lo = Lb, hi = Le + 1;
  while (hi - lo > 1) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    uint32_t m2 = mid;
    while (m2 < hi && C[m2 - coff] == 0) m2++;
    if (m2 == hi) {
      hi = mid;
      continue;
    }
    if (D[(m2 << ls) - doff] <= d) lo = m2;
    else hi = mid;
  }
  const uint32_t base = lo << ls;
  const uint32_t cnt = C[lo - coff];
  const uint32_t f_lo = (lo == Lb) ? (b - base) + (skip_first ? 1u : 0u) : 0u;
  uint32_t f_hi = cnt;
  if (lo == (e >> ls) && (e - base) < f_hi) f_hi = e - base;
  const uint32_t *L = D + (base - doff);
  uint32_t x = f_lo, y = f_hi;  // lower_bound of d in the leaf's live prefix
  while (x < y) {
    const uint32_t mid = (x + y) >> 1;
    if (L[mid] < d) x = mid + 1;
    else y = mid;
  }
  if (x < f_hi && L[x] == d) {
    *slot = base + x;
    return true;
  }
  *slot = base + x - 1;
  return false;
}

// find_edge with the leaf-level half on a staged table (first item and live count of the leaves from leaf l0 on) and
// the in-leaf half in global memory.  Same result as find_edge.
__device__ __forceinline__ bool find_tab(const uint32_t *first, const uint8_t *cnt8, uint32_t l0,
                                         const uint32_t *__restrict__ dest, uint32_t b, uint32_t e, uint32_t ls,
                                         uint32_t d, uint32_t *slot) {
  const uint32_t Lb = b >> ls, Le = (e - 1) >> ls;
  uint32_t lo = Lb, hi = Le + 1;
  while (hi - lo > 1) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    uint32_t m2 = mid;
    while (m2 < hi && cnt8[m2 - l0] == 0) m2++;
    if (m2 == hi) {
      hi = mid;
      continue;
    }
    if (first[m2 - l0] <= d) lo = m2;
    else hi = mid;
  }
  const uint32_t base = lo << ls;
  const uint32_t f_lo = (lo == Lb) ? (b - base) + 1u : 0u;
  uint32_t f_hi = cnt8[lo - l0];
  if (lo == (e >> ls) && (e - base) < f_hi) f_hi = e - base;
  const uint32_t *L = dest + base;
  uint32_t x = f_lo, y = f_hi;  // lower_bound of d in the leaf's live prefix
  while (x < y) {
    const uint32_t mid = (x + y) >> 1;
    if (L[mid] < d) x = mid + 1;
    else y = mid;
  }
  if (x < f_hi && L[x] == d) {
    *slot = base + x;
    return true;
  }
  *slot = base + x - 1;
  return false;
}

// ---- locate: one CTA per TILE of 512 consecutive sorted updates ------------------------------------------------
// Fuses, over the sorted batch:
//   * num_neighbors += (#add calls) - (#remove calls) per source, duplicates included (reference PCSR.cpp:1392,747);
//     sorted by src => one warp-aggregated atomic per run;
//   * last-op-wins: only the last element of a run of equal keys acts on the structure (the batch result equals the
//     sequential reference on the same stream); `not found` by the sequential rule (reference PCSR.cpp:750-754): a
//     remove misses iff the previous op on the same key in this batch was a remove, or it is the key's first op and
//     the edge is absent;
//   * the segmented search of every winner (find_in), overwrite / tombstone in place, per-leaf insert / delete counts;
//   * the tile's inserts (dst, value, predecessor slot), compacted in key order into the TILE'S OWN region of a scratch
//     list, and the tile's insert count: a scan over the tile counts and k_gather_inserts then make the global
//     key-ordered insert list.  (Measured: resolving the global offset inside this kernel by a decoupled look-back
//     costs far more than the extra copy -- tile times vary widely (hub tiles search global memory), and with a
//     look-back every tile waits for the slowest tile before it while holding its SM slot: 3.6 -> 5.2..6.9 ms on the
//     100 M-update batch.)
// Both sequences are sorted, so the tile's updates land in ONE contiguous slot window of the packed array: from the
// first key's source vertex to the end of the last key's -- or, when a hub vertex makes that too long, between the
// end of the last key's.  A window of <= LCAP slots is STAGED in shared memory with coalesced 16-byte loads and every
// search of the tile runs there (measured on the per-element kernel: 17 cycles of long-scoreboard stall per issued
// instruction, ~5 dependent DRAM/L2 round trips per update); longer windows (hub vertices) are searched in global
// memory like before.
constexpr int LT = 256;         // threads of a locate CTA
constexpr int LI = 2;           // sorted updates per thread
constexpr int LTILE = LT * LI;  // updates per tile
// Window capacity, measured on B200 (locate stage, ms: 100 M skewed updates into 2^29 slots / 10 M uniform into 2^25 /
// 10 M deletes): 8192 slots (47 KB of shared memory, 4 CTAs per SM) 4.68 / 0.357 / 0.410; 4096 (7 CTAs) 3.45 / 0.265 /
// 0.295; 2048 (8 CTAs = all 64 warps) 3.27 / 0.251 / 0.286; the per-element kernel with a separate three-pass
// compaction it replaces: 3.63 / 0.276 / 0.308.  Resident warps matter more than the share of tiles that is staged.
#ifndef PPCSR_LOC_CAP
#define PPCSR_LOC_CAP 2048
#endif
constexpr int LCAP = PPCSR_LOC_CAP;    // slots of dest[] a tile can stage
constexpr int LCAP_LEAVES = LCAP / 8;  // leaves are >= 8 slots

// A window too long to stage whole is staged as a TABLE -- the first item and the live count of each of its leaves
// (one 32-byte sector per leaf instead of the whole line): the leaf-level half of every search then runs in shared
// memory and only the in-leaf half (one 128-byte line per update, shared by neighbouring keys) goes to global memory.
// At C4's update density (one update per ~5 slots) a tile of 512 sorted updates spans ~2.7 K slots: too long to stage,
// ~90 table entries.
#ifndef PPCSR_LOC_TAB
#define PPCSR_LOC_TAB 1
#endif
#ifndef PPCSR_LOC_FAST1  // find_fast for whole-staged windows too
#define PPCSR_LOC_FAST1 0
#endif
constexpr int LTAB = PPCSR_LOC_TAB ? 1536 : 0;  // leaves a tile can stage as a table (in the place of dest[])
struct LocTable {
  uint32_t first[LTAB + 1];
  uint8_t cnt8[LTAB + 1];
};
static_assert(sizeof(LocTable) <= sizeof(uint32_t) * LCAP, "the table lies in the staging area of dest[]");

struct LocSmem {
  union {
    uint32_t dest[LCAP];       // staged window of dest[]
    LocTable tab;              // or: first item + live count of each leaf of a longer window
  };
  uint32_t cnt[LCAP_LEAVES];   // leaf counts of the window
  uint64_t key[LTILE + 2];     // the tile's keys; [0] and [LTILE + 1] are the neighbours' (or ~0: none)
  uint32_t o_dst[LTILE], o_val[LTILE], o_pred[LTILE];  // the tile's inserts, compacted in key order
  uint32_t warp[33];
  uint32_t stat[8];
  uint32_t win[4];             // window [a, b), mode (0 nothing to search, 1 staged, 2 global, 3 leaf table), valid keys
};
static_assert(sizeof(LocSmem) <= 48 * 1024, "k_locate is launched without a shared-memory opt-in");

// The search of a staged tile without empty leaves, with UNIFORM trip counts: a warp's lanes search vertex ranges of
// different lengths, so the data-dependent loops of find_in / find_tab run for the longest range in the warp at ~12
// instructions per step, diverged (ncu: 47 % of k_locate's instructions, which is issue-bound).  Here the leaf level
// takes `steps` = ceil(log2(leaves of the window)) branch-free halvings and the in-leaf lower_bound five (a leaf has
// <= 32 slots).  TAB: the window is staged as a leaf table (the in-leaf half reads global memory), else whole.
// Same result as find_in / find_tab when no leaf of the window is empty.
template <bool TAB>
__device__ __forceinline__ bool find_fast(const LocSmem &S, const uint32_t *__restrict__ dest, uint32_t wa,
                                          uint32_t steps, uint32_t b, uint32_t e, uint32_t ls, uint32_t d,
                                          uint32_t *slot) {
  const uint32_t l0 = wa >> ls, fs = TAB ? 0u : ls;
  const uint32_t Lb = b >> ls, Le = (e - 1) >> ls;
  uint32_t lo = Lb - l0, n = Le - Lb + 1u;  // candidates: the window's leaves [lo, lo + n)
  // as many halvings as the longest range among the lanes searching right now needs (most vertices span one or two
  // leaves; the window's own ceil(log2(leaves)) bounds it)
  steps = min(steps, 32u - (uint32_t)__clz(__reduce_max_sync(__activemask(), n)));
  for (uint32_t st = 0; st < steps; st++) {
    const uint32_t half = n >> 1;
    // unconditional probe (branch-free): half == 0 re-reads [lo] and adds nothing.  S.tab.first aliases S.dest
    lo += S.dest[(lo + half) << fs] <= d ? half : 0u;
    n -= half;
  }
  const uint32_t leaf = lo + l0, base = leaf << ls;
  const uint32_t cnt = TAB ? (uint32_t)S.tab.cnt8[lo] : S.cnt[lo];
  const uint32_t f_lo = (leaf == Lb) ? (b - base) + 1u : 0u;
  uint32_t f_hi = cnt;
  if (leaf == (e >> ls) && (e - base) < f_hi) f_hi = e - base;
  const uint32_t *L = TAB ? dest + base : S.dest + (base - wa);
  uint32_t x = f_lo, m = f_hi > f_lo ? f_hi - f_lo : 0u;  // lower_bound of d in [f_lo, f_hi): the answer lies in [x, x + m]
#pragma unroll
  for (int st = 0; st < 5; st++) {
    const uint32_t half = m >> 1;
    x += L[x + half - (half != 0u ? 1u : 0u)] < d ? half : 0u;  // branch-free; half == 0 probes [x] (<= one slot past the leaf) and adds nothing
    m -= half;
  }
  if (m != 0u && L[x] < d) x++;
  if (x < f_hi && L[x] == d) {
    *slot = base + x;
    return true;
  }
  *slot = base + x - 1;
  return false;
}

// SPARSE: the small-batch variant (appends the touched leaves); a template so that the general instantiation keeps its
// 32 registers -- 8 CTAs = all 64 warps of an SM (at 40 registers: 6 CTAs, locate stage 3.27 -> 4.02 ms on C4).
// INSONLY: the batch has neither per-update values nor an op bit and its one value is non-zero -- every update is an
// insert: the remove / `not found` bookkeeping (runs of equal keys walked back to their first op, delete counts, three
// of the seven ballots) is compiled out.  k_locate is issue-bound (ncu: 77 % issue-active) and that part was a quarter
// of its instructions on an insert batch.
// DELONLY: the mirror image -- no values, no op bit, value 0: every update is a remove (no insert counts, no insert
// list; a remove misses iff the edge is absent or the previous update of the batch removed the same key).
template <bool SPARSE, bool INSONLY = false, bool DELONLY = false>
__global__ void __launch_bounds__(LT, 8) k_locate(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ pay,
                                               uint32_t default_val, size_t count, uint64_t invalid_key,
                                               const uint32_t *__restrict__ dest, uint32_t *__restrict__ val,
                                               const uint32_t *__restrict__ leaf_cnt, const uint32_t *__restrict__ beg,
                                               uint32_t ls, uint32_t n_slots, uint32_t *__restrict__ nn,
                                               uint32_t *__restrict__ tile_dst, uint32_t *__restrict__ tile_val,
                                               uint32_t *__restrict__ tile_pred, uint32_t *__restrict__ tile_cnt,
                                               uint32_t *__restrict__ ins_cnt, uint32_t *__restrict__ del_cnt,
                                               uint32_t op_bit, BatchScalars *sc, uint32_t *touched,
                                               uint32_t *touch_stamp, uint32_t touch_epoch, uint32_t dst_mask) {
  // Small-batch path (SPARSE, sparse.cuh): the batch was sorted on a SPECULATED dst width (no host round
  // trip after the key builder); a dst beyond it means the order is wrong -- leave before anything is modified, the
  // host runs the batch again the general way.  The first update to reach a leaf appends it to the touched list.
  if (SPARSE && (sc->dst_or & ~dst_mask)) {
    if (blockIdx.x == 0 && threadIdx.x == 0) sc->sparse_abort = 1u;
    return;
  }
  extern __shared__ __align__(16) unsigned char loc_smem_raw[];
  LocSmem &S = *reinterpret_cast<LocSmem *>(loc_smem_raw);
  const uint32_t tid = threadIdx.x;
  const unsigned lt = lanemask_lt();
  const size_t base = (size_t)blockIdx.x * LTILE;
  const uint32_t tile_n = (uint32_t)min((size_t)LTILE, count - base);
  // op_bit: bit 63 of a key word marks a remove (KEY_OP_BIT) and is not part of the key
  const uint64_t km = op_bit ? ~KEY_OP_BIT : ~0ull;
  for (uint32_t x = tid; x < (uint32_t)LTILE + 2u; x += LT) {
    const size_t g = base + x;  // element g - 1
    S.key[x] = (g >= 1 && g - 1 < count) ? keys[g - 1] : ~0ull;
  }
  if (tid < 8) S.stat[tid] = 0;
  __syncthreads();
  // ---- the tile's slot window
  if (tid == 0) {
    uint32_t lo = 0, hi = tile_n;  // rejected updates carry invalid_key and sort last: count the valid ones
    if (tile_n && (S.key[tile_n] & km) < invalid_key) lo = tile_n;  // (none in this tile: no search)
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      if ((S.key[1 + mid] & km) < invalid_key) lo = mid + 1;
      else hi = mid;
    }
    const uint32_t nv = lo;
    uint32_t a = 0, b = 0, mode = 0;
    if (nv) {
      const uint32_t s0 = (uint32_t)((S.key[1] & km) >> 32), s1 = (uint32_t)((S.key[nv] & km) >> 32);
      const uint32_t leaf = 1u << ls;
      a = (beg[s0] >> ls) << ls;
      b = (uint32_t)min((unsigned long long)n_slots, (((unsigned long long)beg[s1 + 1] + leaf - 1u) >> ls) << ls);
      mode = (b - a <= (uint32_t)LCAP) ? 1u : (((b - a) >> ls) <= (uint32_t)LTAB) ? 3u : 2u;
    }
    S.win[0] = a;
    S.win[1] = b;
    S.win[2] = mode;
    S.win[3] = nv;
  }
  // the vertex ranges of my updates do not depend on the window: their loads fly while thread 0 finds it
  uint32_t vb[LI], ve[LI];
#pragma unroll
  for (int r = 0; r < LI; r++) {
    vb[r] = ve[r] = 0u;
    const uint32_t e = r * LT + tid;
    const uint64_t k = S.key[e + 1] & km;
    if (e < tile_n && k < invalid_key) {
      vb[r] = beg[(uint32_t)(k >> 32)];
      ve[r] = beg[(uint32_t)(k >> 32) + 1u];
    }
  }
  __syncthreads();
  // (Measured and dropped: clipping a hub tile's window to the leaves between the positions of its first and last key
  // -- two global searches by two threads, then the tile is staged after all -- made the stage SLOWER, C4 3.18 -> 3.88
  // ms: the 512 parallel searches of such a tile share their upper probes through L1 and cost less than the serial
  // pair plus a barrier.)
  const uint32_t wa = S.win[0], wb = S.win[1], mode = S.win[2];
  bool fast = false;           // a staged window without empty leaves: uniform-trip-count searches (find_fast)
  uint32_t steps = 0;
  if (mode == 1u || mode == 3u) {
    const uint32_t nl = (wb - wa) >> ls, l0 = wa >> ls;
    steps = 32u - (uint32_t)__clz(nl);
    int empty = 0;
    if (mode == 1u) {  // stage the window: coalesced 16-byte loads (wa is leaf aligned, leaves are >= 32 bytes)
      for (uint32_t x = tid * 4u; x < wb - wa; x += LT * 4u)
        *reinterpret_cast<uint4 *>(&S.dest[x]) = *reinterpret_cast<const uint4 *>(&dest[wa + x]);
      for (uint32_t x = tid; x < nl; x += LT) {
        const uint32_t c = leaf_cnt[l0 + x];
        S.cnt[x] = c;
        empty |= c == 0u;
      }
    } else {  // the window's leaf table
      for (uint32_t x = tid; x < nl; x += LT) {
        const uint32_t c = leaf_cnt[l0 + x];
        S.tab.first[x] = dest[(size_t)(l0 + x) << ls];
        S.tab.cnt8[x] = (uint8_t)c;
        empty |= c == 0u;
      }
    }
    fast = !__syncthreads_or(empty);
  }
  const uint32_t *D = mode == 1u ? S.dest : dest, *C = mode == 1u ? S.cnt : leaf_cnt;
  const uint32_t doff = mode == 1u ? wa : 0u, coff = mode == 1u ? wa >> ls : 0u;

  uint32_t is_ins[LI], o_d[LI], o_v[LI], o_p[LI];
#pragma unroll
  for (int r = 0; r < LI; r++) {
    const uint32_t e = r * LT + tid;
    const size_t i = base + e;
    uint32_t cls = 0xFFu, leaf = 0xFFFFFFFFu, s = 0xFFFFFFFFu;
    int delta = 0;
    bool miss_dup = false, miss_first = false, winner = false;
    is_ins[r] = 0u;
    o_d[r] = o_v[r] = o_p[r] = 0u;
    if (e < tile_n) {
      auto value_at = [&](size_t x) -> uint32_t {
        return pay ? pay[x] : (op_bit && (keys[x] & KEY_OP_BIT)) ? 0u : default_val;
      };
      const uint64_t kw = S.key[e + 1];
      const uint64_t k = kw & km;
      if (k < invalid_key) {
        s = (uint32_t)(k >> 32);
        const uint32_t v = INSONLY ? default_val : DELONLY ? 0u : pay ? pay[i] : (op_bit && (kw & KEY_OP_BIT)) ? 0u : default_val;
        delta = INSONLY ? 1 : DELONLY ? -1 : v != 0 ? 1 : -1;
        const bool same_prev = !INSONLY && (S.key[e] & km) == k && i > 0;
        winner = (S.key[e + 2] & km) != k || i + 1 == count;
        // a remove right after a remove of the same key: the sequential reference reports `not found`
        if (DELONLY) miss_dup = same_prev;
        else if (!INSONLY && v == 0 && same_prev && value_at(i - 1) == 0) miss_dup = true;
        if (winner) {
          bool first_del = !INSONLY && v == 0;  // is the FIRST op of this key's run a remove?
          if (same_prev && !DELONLY) {
            size_t h = i - 1;
            while (h > 0 && (keys[h - 1] & km) == k) h--;
            first_del = value_at(h) == 0;
          }
          const uint32_t d = (uint32_t)k;
          uint32_t slot;
          bool hit;
#if PPCSR_LOC_FAST1
          if (fast) {
            hit = mode == 3u ? find_fast<true>(S, dest, wa, steps, vb[r], ve[r], ls, d, &slot)
                             : find_fast<false>(S, dest, wa, steps, vb[r], ve[r], ls, d, &slot);
          } else {
#else
          if (fast && mode == 3u) {  // (whole-staged windows: measured 4 % slower than find_in's short loops, C2)
            hit = find_fast<true>(S, dest, wa, steps, vb[r], ve[r], ls, d, &slot);
          } else {
#endif
            hit = mode == 3u ? find_tab(S.tab.first, S.tab.cnt8, wa >> ls, dest, vb[r], ve[r], ls, d, &slot)
                             : find_in(D, doff, C, coff, vb[r], ve[r], true, ls, d, &slot);
          }
          if (INSONLY || (!DELONLY && v != 0)) {
            cls = hit ? CLS_OVERWRITE : CLS_INSERT;
            if (hit) val[slot] = v;  // duplicate insert overwrites the value (reference PCSR.cpp:529-532)
          } else {
            cls = hit ? CLS_DELETE : CLS_MISS;
            if (hit) val[slot] = 0;  // tombstone; compacted away by the rebalance of this leaf (PCSR.cpp:605-606)
          }
          if (first_del && !hit) miss_first = true;  // counted on the winner: the run's head op found nothing
          leaf = slot >> ls;
          if (cls == CLS_INSERT) {
            is_ins[r] = 1u;
            o_d[r] = d;
            o_v[r] = v;
            o_p[r] = slot;
          }
        }
      }
    }
    // call counts: one atomic per run of equal sources inside the warp
    {
      const unsigned peers = __match_any_sync(0xFFFFFFFFu, s);
      if (INSONLY || DELONLY) {  // every valid update is one add (remove) call
        if (s != 0xFFFFFFFFu && (peers & lt) == 0)
          atomicAdd(&nn[s], INSONLY ? (uint32_t)__popc(peers) : 0u - (uint32_t)__popc(peers));
      } else {
        const unsigned adds = __ballot_sync(0xFFFFFFFFu, delta > 0);
        const unsigned dels = __ballot_sync(0xFFFFFFFFu, delta < 0);
        if (s != 0xFFFFFFFFu && (peers & lt) == 0) {
          const int sum = __popc(peers & adds) - __popc(peers & dels);
          if (sum) atomicAdd(&nn[s], (uint32_t)sum);
        }
      }
    }
    // per-leaf counts: the batch is key-sorted, so equal leaves are adjacent -> one atomic per warp run.  The first
    // update to reach a leaf also counts it as touched (a leaf hit by inserts AND deletes counts twice: the total
    // only steers the whole-array-versus-windows policy).
    bool first_touch = false;
    if (!DELONLY) {
      const uint32_t key = (cls == CLS_INSERT) ? leaf : 0xFFFFFFFFu;
      const unsigned peers = __match_any_sync(0xFFFFFFFFu, key);
      if (key != 0xFFFFFFFFu && (peers & lt) == 0)
        first_touch = atomicAdd(&ins_cnt[leaf], (uint32_t)__popc(peers)) == 0u;
    }
    if (!INSONLY) {
      const uint32_t key = (cls == CLS_DELETE) ? leaf : 0xFFFFFFFFu;
      const unsigned peers = __match_any_sync(0xFFFFFFFFu, key);
      if (key != 0xFFFFFFFFu && (peers & lt) == 0)
        first_touch |= atomicAdd(&del_cnt[leaf], (uint32_t)__popc(peers)) == 0u;
    }
    {
      const unsigned m0 = DELONLY ? 0u : __ballot_sync(0xFFFFFFFFu, cls == CLS_INSERT);
      const unsigned m1 = DELONLY ? 0u : __ballot_sync(0xFFFFFFFFu, cls == CLS_OVERWRITE);
      const unsigned m2 = INSONLY ? 0u : __ballot_sync(0xFFFFFFFFu, cls == CLS_DELETE);
      const unsigned m3 = INSONLY ? 0u : __ballot_sync(0xFFFFFFFFu, miss_dup);
      const unsigned m5 = INSONLY ? 0u : __ballot_sync(0xFFFFFFFFu, miss_first);
      const unsigned m4 = __ballot_sync(0xFFFFFFFFu, winner);
      const unsigned m6 = __ballot_sync(0xFFFFFFFFu, first_touch);
      if (SPARSE) {  // one entry per leaf and batch, whatever touched it first; the warp takes its places in one go
        const bool fresh = first_touch && atomicExch(&touch_stamp[leaf], touch_epoch) != touch_epoch;
        const unsigned fm = __ballot_sync(0xFFFFFFFFu, fresh);
        unsigned long long at = 0;
        if (fm && lane_id() == (unsigned)(__ffs(fm) - 1)) at = atomicAdd(&sc->n_touched, (unsigned long long)__popc(fm));
        at = __shfl_sync(0xFFFFFFFFu, at, fm ? __ffs(fm) - 1 : 0);
        if (fresh) touched[at + __popc(fm & lt)] = leaf;
      }
      if (lane_id() == 0) {
        if (m6) atomicAdd(&S.stat[5], (uint32_t)__popc(m6));
        if (m0) atomicAdd(&S.stat[0], (uint32_t)__popc(m0));
        if (m1) atomicAdd(&S.stat[1], (uint32_t)__popc(m1));
        if (m2) atomicAdd(&S.stat[2], (uint32_t)__popc(m2));
        if (m3 | m5) atomicAdd(&S.stat[3], (uint32_t)(__popc(m3) + __popc(m5)));
        if (m4) atomicAdd(&S.stat[4], (uint32_t)__popc(m4));
      }
    }
  }
  // ---- the tile's inserts, compacted in element order (element = r * LT + tid): ONE block scan over both rounds'
  // flags, 16 bits each
  static_assert(LI == 2 && LT <= 32768, "the two rounds' counts share one scan word");
  uint32_t total;
  {
    uint32_t both;
    const uint32_t ex = prim::block_excl_scan(is_ins[0] | (is_ins[1] << 16), &both, S.warp);  // ends with a block barrier
    const uint32_t total0 = both & 0xFFFFu;
    total = total0 + (both >> 16);
    const uint32_t at[LI] = {ex & 0xFFFFu, total0 + (ex >> 16)};
#pragma unroll
    for (int r = 0; r < LI; r++) {
      if (is_ins[r]) {
        S.o_dst[at[r]] = o_d[r];
        S.o_val[at[r]] = o_v[r];
        S.o_pred[at[r]] = o_p[r];
      }
    }
  }
  if (tid == 0) {
    tile_cnt[blockIdx.x] = total;
    if (S.stat[0]) atomicAdd(&sc->n_inserted, (unsigned long long)S.stat[0]);
    if (S.stat[1]) atomicAdd(&sc->n_overwritten, (unsigned long long)S.stat[1]);
    if (S.stat[2]) atomicAdd(&sc->n_deleted, (unsigned long long)S.stat[2]);
    if (S.stat[3]) atomicAdd(&sc->n_not_found, (unsigned long long)S.stat[3]);
    if (S.stat[4]) atomicAdd(&sc->n_unique, (unsigned long long)S.stat[4]);
    if (S.stat[5]) atomicAdd(&sc->n_touched_est, (unsigned long long)S.stat[5]);
  }
  __syncthreads();
  for (uint32_t x = tid; x < total; x += LT) {  // coalesced, into the tile's own region
    tile_dst[base + x] = S.o_dst[x];
    if (tile_val) tile_val[base + x] = S.o_val[x];  // nullptr: every insert carries the batch's one value
    tile_pred[base + x] = S.o_pred[x];
  }
}

// the tiles' insert runs, moved to their place in the global key-ordered insert list (tile_off = exclusive scan of the
// tile counts)
constexpr int GATHER_TILES = 8;
__global__ void __launch_bounds__(LT) k_gather_inserts(const uint32_t *__restrict__ tile_dst,
                                                       const uint32_t *__restrict__ tile_val,
                                                       const uint32_t *__restrict__ tile_pred,
                                                       const uint32_t *__restrict__ tile_off,
                                                       uint32_t *__restrict__ ins_dst, uint32_t *__restrict__ ins_val,
                                                       uint32_t *__restrict__ ins_pred, const BatchScalars *sc,
                                                       uint32_t n_tiles) {
  if (sc->sparse_abort) return;  // small-batch path: k_locate left without doing anything
  // GATHER_TILES tiles per CTA (a tile's run is ~500 elements: one tile per CTA left the kernel bound by CTA turnover)
  const uint32_t t0 = blockIdx.x * GATHER_TILES, t1 = min(t0 + (uint32_t)GATHER_TILES, n_tiles);
  for (uint32_t t = t0; t < t1; t++) {
    const uint32_t off = tile_off[t], cnt = tile_off[t + 1] - off;
    const size_t base = (size_t)t * LTILE;
    for (uint32_t x = threadIdx.x; x < cnt; x += LT) {
      ins_dst[off + x] = tile_dst[base + x];
      if (tile_val) ins_val[off + x] = tile_val[base + x];
      ins_pred[off + x] = tile_pred[base + x];
    }
  }
}

// ---- owner binning for the multi-GPU all-to-all (reference PPPCSR::get_partiton, PPPCSR.cpp:58-66) ----
__device__ __forceinline__ uint32_t owner_of(const uint64_t *starts, uint32_t parts, uint64_t v) {
  uint32_t lo = 0, hi = parts;  // last p with starts[p] <= v
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (starts[mid] <= v) lo = mid;
    else hi = mid;
  }
  return lo;
}


__global__ void __launch_bounds__(BT) k_bin_count(const uint32_t *__restrict__ src, size_t count,
                                                  const uint64_t *__restrict__ starts, uint32_t parts,
                                                  uint32_t *__restrict__ block_hist, uint32_t nblocks) {
  __shared__ uint32_t s_h[BIN_MAX_PARTS];
  __shared__ uint64_t s_st[BIN_MAX_PARTS];
  if (threadIdx.x < parts) {
    s_h[threadIdx.x] = 0;
    s_st[threadIdx.x] = starts[threadIdx.x];
  }
  __syncthreads();
  const size_t base = (size_t)blockIdx.x * prim::SORT_TILE;
  uint32_t sv[prim::SORT_ROUNDS];
#pragma unroll
  for (int r = 0; r < prim::SORT_ROUNDS; r++) {  // every load of the tile in flight before the first use
    const size_t i = base + (size_t)r * BT + threadIdx.x;
    sv[r] = i < count ? src[i] : 0u;
  }
#pragma unroll
  for (int r = 0; r < prim::SORT_ROUNDS; r++) {
    const size_t i = base + (size_t)r * BT + threadIdx.x;
    if (i < count) atomicAdd(&s_h[owner_of(s_st, parts, sv[r])], 1u);
  }
  __syncthreads();
  if (threadIdx.x < parts) block_hist[(size_t)threadIdx.x * nblocks + blockIdx.x] = s_h[threadIdx.x];
}

// stable scatter: same warp-synchronous ranking as the radix sort, digit = owner
__global__ void __launch_bounds__(BT) k_bin_scatter(const uint32_t *__restrict__ src, const uint32_t *__restrict__ dst,
                                                    const uint32_t *__restrict__ val, size_t count,
                                                    const uint64_t *__restrict__ starts, uint32_t parts,
                                                    const uint32_t *__restrict__ offs, uint32_t nblocks,
                                                    uint32_t *__restrict__ out_src, uint32_t *__restrict__ out_dst,
                                                    uint32_t *__restrict__ out_val, uint64_t *__restrict__ out_packed) {
  __shared__ uint32_t s_cnt[prim::SORT_WARPS][BIN_MAX_PARTS];
  __shared__ uint64_t s_st[BIN_MAX_PARTS];
  for (int d = threadIdx.x; d < prim::SORT_WARPS * BIN_MAX_PARTS; d += BT) (&s_cnt[0][0])[d] = 0;
  if (threadIdx.x < parts) s_st[threadIdx.x] = starts[threadIdx.x];
  __syncthreads();
  const unsigned w = threadIdx.x >> 5, l = lane_id(), lt = lanemask_lt();
  const size_t wbase = (size_t)blockIdx.x * prim::SORT_TILE + (size_t)w * (32 * prim::SORT_ROUNDS);
  uint32_t own[prim::SORT_ROUNDS], rank[prim::SORT_ROUNDS];
#pragma unroll
  for (int r = 0; r < prim::SORT_ROUNDS; r++) {
    const size_t i = wbase + (size_t)r * 32 + l;
    const bool valid = i < count;
    const uint32_t d = valid ? owner_of(s_st, parts, src[i]) : 0x1FFu;
    own[r] = d;
    const unsigned peers = __match_any_sync(0xFFFFFFFFu, d);
    uint32_t base = 0;
    if (valid) base = s_cnt[w][d];
    __syncwarp();
    if (valid && (peers & lt) == 0) s_cnt[w][d] = base + __popc(peers);
    __syncwarp();
    rank[r] = base + __popc(peers & lt);
  }
  __syncthreads();
  if (threadIdx.x < parts) {
    uint32_t run = offs[(size_t)threadIdx.x * nblocks + blockIdx.x];
    for (int ww = 0; ww < prim::SORT_WARPS; ww++) {
      uint32_t t = s_cnt[ww][threadIdx.x];
      s_cnt[ww][threadIdx.x] = run;
      run += t;
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < prim::SORT_ROUNDS; r++) {
    const size_t i = wbase + (size_t)r * 32 + l;
    if (i < count) {
      const uint32_t d = own[r];
      const uint32_t pos = s_cnt[w][d] + rank[r];
      const uint32_t local = src[i] - (uint32_t)s_st[d];  // shard-local id (reference PPPCSR.cpp:46-52)
      if (out_packed) {
        out_packed[pos] = ((uint64_t)local << 32) | dst[i];
      } else {
        out_src[pos] = local;
        out_dst[pos] = dst[i];
      }
      if (out_val) out_val[pos] = val ? val[i] : 1u;
    }
  }
}

// Routing fused with the exchange: the stable owner binning of k_bin_scatter, but every record goes STRAIGHT INTO THE
// OWNING GPU'S RECEIVE BUFFER over NVLink (peer pointers of a symmetric allocation) -- no send buffer, no count
// exchange before the data moves, no NCCL all-to-all.  Rank `me` owns region `me` (cap records) of every peer's
// buffer; the tile is first reordered by destination in shared memory so that the peer stores are coalesced runs
// (a tile of 4096 records gives runs of ~512 records = 4 KB per destination on 8 GPUs), and block 0 deposits the
// per-destination counts in the peers' count arrays.  A cross-GPU barrier after this kernel publishes everything.
//   dynamic shared memory: u64 rec[SORT_TILE] | u32 val[SORT_TILE] (when values travel) | u8 owner[SORT_TILE]
struct PeerTable {
  uint64_t *rec[BIN_MAX_PARTS];  // receive buffer of every rank (records)
  uint32_t *val[BIN_MAX_PARTS];  // receive buffer of every rank (values), used when d_val != nullptr
  uint64_t *cnt[BIN_MAX_PARTS];  // count array of every rank: cnt[dest][sender]
};
inline size_t bin_peers_smem(bool has_val) {
  return (size_t)prim::SORT_TILE * 8 + (has_val ? (size_t)prim::SORT_TILE * 4 : 0) + (size_t)prim::SORT_TILE;
}
// ORDERED == false: the tiles take their places in the destinations' regions by one atomicAdd per tile and destination
// on `cursor` (no count pass, no scan in front of this kernel); the records of a region then stand in tile-arrival
// order, which is indistinguishable from submission order when every update of the batch is the same operation (no
// per-update values: only then the caller may use it).  k_publish_peer_counts deposits the counts afterwards.
template <bool HAS_VAL, bool ORDERED = true>
__global__ void __launch_bounds__(BT, 4) k_bin_scatter_peers(const uint32_t *__restrict__ src,
                                                             const uint32_t *__restrict__ dst,
                                                             const uint32_t *__restrict__ val, size_t count,
                                                             const uint64_t *__restrict__ starts, uint32_t parts,
                                                             const uint32_t *__restrict__ offs, uint32_t nblocks,
                                                             uint32_t me, uint64_t cap, PeerTable P,
                                                             uint32_t *__restrict__ cursor = nullptr) {
  extern __shared__ __align__(16) unsigned char s_dyn[];
  uint64_t *s_rec = reinterpret_cast<uint64_t *>(s_dyn);
  uint32_t *s_v = reinterpret_cast<uint32_t *>(s_dyn + (size_t)prim::SORT_TILE * 8);
  uint8_t *s_own = s_dyn + (size_t)prim::SORT_TILE * 8 + (HAS_VAL ? (size_t)prim::SORT_TILE * 4 : 0);
  __shared__ uint32_t s_cnt[prim::SORT_WARPS][BIN_MAX_PARTS];
  __shared__ uint32_t s_tbase[BIN_MAX_PARTS + 1];  // tile-local start of every destination's run
  __shared__ uint32_t s_gbase[BIN_MAX_PARTS];      // region-relative position of the tile's run
  __shared__ uint32_t s_st[BIN_MAX_PARTS];         // first vertex of every shard (vertex ids are 32-bit)
  for (int d = threadIdx.x; d < prim::SORT_WARPS * BIN_MAX_PARTS; d += BT) (&s_cnt[0][0])[d] = 0;
  if (threadIdx.x < BIN_MAX_PARTS) s_st[threadIdx.x] = threadIdx.x < parts ? (uint32_t)starts[threadIdx.x] : 0xFFFFFFFFu;
  __syncthreads();
  const unsigned w = threadIdx.x >> 5, l = lane_id(), lt = lanemask_lt();
  const size_t wbase = (size_t)blockIdx.x * prim::SORT_TILE + (size_t)w * (32 * prim::SORT_ROUNDS);
  // all of the warp's sources first (16 independent loads in flight), then owner + stable rank of every record,
  // kept as one packed word per record: owner << 16 | rank inside the warp's run for that owner
  uint32_t sv[prim::SORT_ROUNDS];
#pragma unroll
  for (int r = 0; r < prim::SORT_ROUNDS; r++) {
    const size_t i = wbase + (size_t)r * 32 + l;
    sv[r] = i < count ? src[i] : 0xFFFFFFFFu;
  }
  uint32_t pk[prim::SORT_ROUNDS];
#pragma unroll
  for (int r = 0; r < prim::SORT_ROUNDS; r++) {
    const bool valid = wbase + (size_t)r * 32 + l < count;
    uint32_t d = 0x1FFu;
    if (valid) {  // last shard whose first vertex is <= src: branch-free over the (padded) table
      d = 0;
#pragma unroll
      for (uint32_t step = BIN_MAX_PARTS / 2; step >= 1; step >>= 1)
        if (d + step < parts && s_st[d + step] <= sv[r]) d += step;
    }
    const unsigned peers = __match_any_sync(0xFFFFFFFFu, d);
    uint32_t base = 0;
    if (valid) base = s_cnt[w][d];
    __syncwarp();
    if (valid && (peers & lt) == 0) s_cnt[w][d] = base + __popc(peers);
    __syncwarp();
    pk[r] = (d << 16) | (base + __popc(peers & lt));
  }
  __syncthreads();
  if (threadIdx.x < 32) {  // tile-local layout: destination-major, warp-minor (stable); one warp scans the totals
    uint32_t tot[BIN_MAX_PARTS / 32];
#pragma unroll
    for (int k = 0; k < BIN_MAX_PARTS / 32; k++) {
      const uint32_t p = k * 32 + l;
      tot[k] = 0;
      if (p < parts)
        for (int ww = 0; ww < prim::SORT_WARPS; ww++) tot[k] += s_cnt[ww][p];
    }
    uint32_t carry = 0;
#pragma unroll
    for (int k = 0; k < BIN_MAX_PARTS / 32; k++) {
      uint32_t inc = tot[k];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, inc, o);
        if (l >= (unsigned)o) inc += y;
      }
      const uint32_t p = k * 32 + l;
      uint32_t run = carry + inc - tot[k];
      if (p < parts) {
        s_tbase[p] = run;
        for (int ww = 0; ww < prim::SORT_WARPS; ww++) {
          const uint32_t t = s_cnt[ww][p];
          s_cnt[ww][p] = run;
          run += t;
        }
      }
      carry += __shfl_sync(0xFFFFFFFFu, inc, 31);
    }
    if (l == 0) s_tbase[parts] = carry;
  }
  if (ORDERED && threadIdx.x >= 32 && threadIdx.x - 32 < parts) {
    const uint32_t p = threadIdx.x - 32;
    const size_t row = (size_t)p * nblocks;
    s_gbase[p] = offs[row + blockIdx.x] - offs[row];
    if (blockIdx.x == 0) {  // this rank's count for destination p, deposited at the destination
      const uint32_t next = p + 1 < parts ? offs[row + nblocks] : (uint32_t)count;
      P.cnt[p][me] = next - offs[row];
    }
  }
  __syncthreads();
  if (!ORDERED && threadIdx.x < parts) {  // (ordered against the write-out by the barrier behind the reorder loop)
    const uint32_t p = threadIdx.x;
    s_gbase[p] = atomicAdd(&cursor[p], s_tbase[p + 1] - s_tbase[p]);
  }
#pragma unroll
  for (int r = 0; r < prim::SORT_ROUNDS; r++) {
    const size_t i = wbase + (size_t)r * 32 + l;
    if (i < count) {
      const uint32_t d = pk[r] >> 16;
      const uint32_t at = s_cnt[w][d] + (pk[r] & 0xFFFFu);
      s_rec[at] = ((uint64_t)(sv[r] - s_st[d]) << 32) | dst[i];  // shard-local id (PPPCSR.cpp:46-52)
      if (HAS_VAL) s_v[at] = val[i];
      s_own[at] = (uint8_t)d;
    }
  }
  __syncthreads();
  const uint32_t tile_n = s_tbase[parts];
  for (uint32_t x = threadIdx.x; x < tile_n; x += BT) {
    const uint32_t d = s_own[x];
    const size_t at = (size_t)me * cap + s_gbase[d] + (x - s_tbase[d]);
    P.rec[d][at] = s_rec[x];
    if (HAS_VAL) P.val[d][at] = s_v[x];
  }
}
// after an unordered scatter: this rank's count for every destination, deposited at the destination
__global__ void k_publish_peer_counts(uint32_t parts, uint32_t me, const uint32_t *__restrict__ cursor, PeerTable P) {
  if (threadIdx.x < parts) P.cnt[threadIdx.x][me] = cursor[threadIdx.x];
}
// an empty local batch still has to tell every peer "nothing from me"
__global__ void k_zero_peer_counts(uint32_t parts, uint32_t me, PeerTable P) {
  if (threadIdx.x < parts) P.cnt[threadIdx.x][me] = 0;
}

}  // namespace batch
