// rebalance.cuh -- what the rebalance kernels share, and the small-window kernel.
// A rebalance merges the kept items of a window with the batch's inserts, drops the tombstones, and spreads the result
// evenly over the window's leaves, fixing the vertex sentinels' back pointers in the same pass.
// Replaces reference PCSR::redistribute + fix_sentinel + slide_right/slide_left + double_list/half_list
// (src/pcsr/PCSR.cpp:222-249, 168-183, 326-390, 251-320).
//
// Rank arithmetic.  For a window of m source leaves the merged sequence is the concatenation over source leaves i of
// merge(kept(i), inserts(i)); its ranks are
//     rank(kept item at offset f of leaf i) = R[i] + #kept before f + #inserts of i whose predecessor < f
//     rank(q-th insert of leaf i)           = R[i] + q + #kept items of i at offsets <= offset(pred)
// with R = exclusive scan of the post-batch leaf counts.  Output leaf o of m_out (a power of two: windows are
// nodes of the implicit tree) receives the ranks [(o*j) >> lg(m_out), ((o+1)*j) >> lg(m_out)) left-packed,
// the rest of the leaf is nulled.
//
// Here: the arguments of the chunked kernel (k_rebalance_m, rebalance_m.cuh) and the searches, bulk-copy (TMA) and
// mbarrier helpers it uses; k_rebalance_small, which takes the windows of <= SMALL_MAX_LEAVES leaves one warp each; and
// the kernels that lay out a fresh array.
#pragma once
#include "common.cuh"
#include "primitives.cuh"

namespace reb {

constexpr int RT = 256;
constexpr int RWARPS = RT / 32;
#ifndef PPCSR_CHUNK_SLOTS
#define PPCSR_CHUNK_SLOTS 2048
#endif
#ifndef PPCSR_SEG_SLOTS
#define PPCSR_SEG_SLOTS 2048
#endif
constexpr int CHUNK_SLOTS = PPCSR_CHUNK_SLOTS;     // output slots per chunk
constexpr int SEG_LEAVES_SLOTS = PPCSR_SEG_SLOTS;  // source slots examined per segment (64 leaves of 32 slots): 2 quads per thread
// leaves per segment: 64 of 32 slots; arrays with smaller leaves are tiny, their segments are capped at 128 leaves
constexpr int SEG_MAX_LEAVES = SEG_LEAVES_SLOTS / 32 > 128 ? SEG_LEAVES_SLOTS / 32 : 128;

// k_rebalance_m reads neither leaf_cnt, windows, n_windows nor ins_sentinels.  They stay for now: without them the other
// parameters move, and ptxas allocates the kernel's registers differently.
struct Args {
  const uint32_t *src_dest, *src_val;  // source slots
  const uint32_t *leaf_cnt;            // source physical leaf counts (tombstones included)
  const uint32_t *rank_off;            // R[], n_leaves_src + 1
  const uint32_t *ins_off;             // first insert of each source leaf, n_leaves_src + 1
  const uint32_t *ins_dst, *ins_val, *ins_pred;
  uint32_t *out_dest_single, *out_val_single;  // target of single-CTA windows (in place)
  uint32_t *out_dest_multi, *out_val_multi;    // target of multi-CTA windows (out of place)
  uint32_t *tree_leaf_out;                     // post-rebalance leaf counts (leaf level of the tree)
  uint32_t *leaf_cnt_out;                      // nullable: the same counts, straight into the new leaf_cnt[]
  uint32_t *beg;
  const WindowDesc *windows;
  uint32_t n_windows;
  uint32_t ls_src, ls_dst;
  uint32_t m_dst_override;  // != 0: resize, the single window maps onto this many output leaves from leaf 0
  uint32_t ins_sentinels;   // != 0: the insert list itself holds sentinels (add_nodes)
  uint32_t ins_uniform;     // ins_val == nullptr: the value every insert of the batch carries
};

__device__ __forceinline__ uint32_t upper_bound_u32(const uint32_t *a, uint32_t n, uint32_t key) {
  uint32_t lo = 0, hi = n;  // first index with a[idx] > key
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (a[mid] <= key) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}
__device__ __forceinline__ uint32_t lower_bound_u32(const uint32_t *a, uint32_t n, uint32_t key) {
  uint32_t lo = 0, hi = n;  // first index with a[idx] >= key
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (a[mid] < key) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

// first rank of output leaf o when j items are spread over 2^lg leaves (rank_begin() with the division as a shift)
__device__ __forceinline__ uint32_t leaf_rank0(uint32_t o, uint32_t j, uint32_t lg) {
  return (uint32_t)(((uint64_t)o * j) >> lg);
}

// ---- TMA (bulk async copy) helpers: sm_90+/sm_100a PTX -----------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
// generic-proxy writes to shared memory become visible to the async proxy (the TMA engine)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// shared -> global bulk copy (SASS: UBLKCP); both addresses 16-byte aligned, bytes a non-zero multiple of 16
__device__ __forceinline__ void bulk_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
               "r"(bytes)
               : "memory");
}
// pull a byte range into L2 ahead of its consumer (no destination, no completion to wait for)
__device__ __forceinline__ void bulk_prefetch_l2(const void *src_gmem, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src_gmem), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// inclusive scan of x over runs of `lpl` consecutive lanes (lpl = 2, 4 or 8: the lanes holding one source leaf)
__device__ __forceinline__ uint32_t leaf_incl_scan(uint32_t x, unsigned lane, uint32_t lpl) {
  const uint32_t in_leaf = lane & (lpl - 1u);
#pragma unroll
  for (uint32_t d = 1; d < 8; d <<= 1) {
    const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, d);
    if (in_leaf >= d) x += y;
  }
  return x;
}

// ---- mbarrier + bulk copy global -> shared (the TMA engine; sm_90+/sm_100a PTX) ------------------------------
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "LAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\t"
      "bra LAB_WAIT;\n\t"
      "DONE:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// both addresses 16-byte aligned, bytes a non-zero multiple of 16 (SASS: UBLKCP.S.G)
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ---------------------------------------------------------------------------------------------------------
// Small windows (<= SMALL_MAX_LEAVES leaves, the overwhelmingly common case of a steady-state batch: a touched
// leaf that stays within its bounds is its own window): ONE WARP per window, no block barriers, in place.
// The rank arithmetic above, window by window; the window's items are staged in the warp's 2 KB slice of shared memory.
// ---------------------------------------------------------------------------------------------------------
constexpr int SMALL_MAX_LEAVES = 8;
constexpr int SMALL_MAX_SLOTS = SMALL_MAX_LEAVES * 32;

struct SmallArgs {
  uint32_t *dest, *val;          // rebalanced in place
  const uint32_t *leaf_cnt, *rank_off, *ins_off;
  const uint32_t *ins_dst, *ins_val, *ins_pred;  // ins_val == nullptr: every insert carries ins_uniform
  uint32_t ins_uniform;
  uint32_t *tree_leaf_out, *beg;
  const WindowDesc *windows;
  uint32_t n_windows;            // one warp per window of the list; chunked (large) windows are skipped
  uint32_t ls;
};

__global__ void __launch_bounds__(RT) k_rebalance_small(SmallArgs A) {
  __shared__ uint32_t s_dest[RWARPS][SMALL_MAX_SLOTS];
  __shared__ uint32_t s_val[RWARPS][SMALL_MAX_SLOTS];
  __shared__ uint32_t s_last[RWARPS][SMALL_MAX_LEAVES][32];
  __shared__ uint32_t s_mask[RWARPS][SMALL_MAX_LEAVES], s_rank[RWARPS][SMALL_MAX_LEAVES],
      s_ioff[RWARPS][SMALL_MAX_LEAVES + 1];
  const unsigned warp = threadIdx.x >> 5, lane = lane_id(), lt = lanemask_lt();
  const uint32_t wid = blockIdx.x * RWARPS + warp;
  if (wid >= A.n_windows) return;  // whole warp exits together
  const WindowDesc w = A.windows[wid];
  if (w.n_chunks != 0) return;     // a large window: k_rebalance_m owns it
  const uint32_t m = w.m, j = w.items, logN = 1u << A.ls;
  const uint32_t R0 = A.rank_off[w.leaf0];
  uint32_t *sd = s_dest[warp], *sv = s_val[warp];

  // per-leaf metadata: lane k < m owns leaf k
  uint32_t my_cnt = 0;
  if (lane <= m) {
    const uint32_t i = w.leaf0 + lane;
    s_ioff[warp][lane] = A.ins_off[i];
    if (lane < m) {
      my_cnt = A.leaf_cnt[i];
      s_rank[warp][lane] = A.rank_off[i] - R0;
    }
  }
  for (uint32_t x = lane; x < m * 32; x += 32) (&s_last[warp][0][0])[x] = 0;
  uint32_t d[SMALL_MAX_LEAVES], v[SMALL_MAX_LEAVES];
#pragma unroll
  for (int k = 0; k < SMALL_MAX_LEAVES; k++) {
    d[k] = 0;
    v[k] = 0;
    const uint32_t cnt_k = __shfl_sync(0xFFFFFFFFu, my_cnt, k);
    if ((uint32_t)k < m && lane < cnt_k) {
      const size_t slot = ((size_t)(w.leaf0 + k) << A.ls) + lane;
      d[k] = A.dest[slot];
      v[k] = A.val[slot];
    }
  }
#pragma unroll
  for (int k = 0; k < SMALL_MAX_LEAVES; k++) {
    const unsigned mask = __ballot_sync(0xFFFFFFFFu, v[k] != 0u);
    if ((uint32_t)k < m && lane == 0) s_mask[warp][k] = mask;
  }
  __syncwarp();
  // inserts of the window
  const uint32_t q_end = s_ioff[warp][m];
  for (uint32_t q = s_ioff[warp][0] + lane; q < q_end; q += 32) {
    const uint32_t pred = A.ins_pred[q];
    const uint32_t k = (pred >> A.ls) - w.leaf0;
    const uint32_t f = pred & (logN - 1u);
    const uint32_t t = q - s_ioff[warp][k];
    const uint32_t r = s_rank[warp][k] + t + (uint32_t)__popc(s_mask[warp][k] & ((2u << f) - 1u));
    atomicMax(&s_last[warp][k][f], t + 1u);
    sd[r] = A.ins_dst[q];
    sv[r] = A.ins_val ? A.ins_val[q] : A.ins_uniform;
  }
  __syncwarp();
  // kept items
#pragma unroll
  for (int k = 0; k < SMALL_MAX_LEAVES; k++) {
    if ((uint32_t)k < m) {  // warp-uniform
      const unsigned mask = s_mask[warp][k];
      const uint32_t last = s_last[warp][k][lane];
      const unsigned hang = __ballot_sync(0xFFFFFFFFu, last != 0u) & lt;
      uint32_t ib = __shfl_sync(0xFFFFFFFFu, last, hang ? 31 - __clz(hang) : 0);
      if (!hang) ib = 0;
      if ((mask >> lane) & 1u) {
        const uint32_t r = s_rank[warp][k] + (uint32_t)__popc(mask & lt) + ib;
        sd[r] = d[k];
        sv[r] = v[k];
      }
    }
  }
  __syncwarp();
  // write-out (in place: every source slot of the window has been read above)
  const uint32_t out_slots = m << A.ls;
  const size_t slot0 = (size_t)w.leaf0 << A.ls;
  for (uint32_t x = lane * 4; x < out_slots; x += 32 * 4) {
    const uint32_t ol = x >> A.ls, f0 = x & (logN - 1u);
    const uint32_t a_o = (ol * j) / m, b_o = ((ol + 1) * j) / m;  // j <= m*(logN-1): 32-bit is plenty
    const uint32_t live_n = b_o - a_o > f0 ? min(4u, b_o - a_o - f0) : 0u;
    const uint32_t base = a_o + f0;
    uint4 dd = make_uint4(0u, 0u, 0u, 0u), vv = make_uint4(0u, 0u, 0u, 0u);
    if (live_n > 0) { dd.x = sd[base]; vv.x = sv[base]; }
    if (live_n > 1) { dd.y = sd[base + 1]; vv.y = sv[base + 1]; }
    if (live_n > 2) { dd.z = sd[base + 2]; vv.z = sv[base + 2]; }
    if (live_n > 3) { dd.w = sd[base + 3]; vv.w = sv[base + 3]; }
    if (dd.x == PPCSR_SENT) A.beg[vv.x - 1u] = (uint32_t)(slot0 + x);
    if (dd.y == PPCSR_SENT) A.beg[vv.y - 1u] = (uint32_t)(slot0 + x + 1);
    if (dd.z == PPCSR_SENT) A.beg[vv.z - 1u] = (uint32_t)(slot0 + x + 2);
    if (dd.w == PPCSR_SENT) A.beg[vv.w - 1u] = (uint32_t)(slot0 + x + 3);
    *reinterpret_cast<uint4 *>(A.dest + slot0 + x) = dd;
    *reinterpret_cast<uint4 *>(A.val + slot0 + x) = vv;
    if (f0 == 0) A.tree_leaf_out[w.leaf0 + ol] = b_o - a_o;
  }
}

// copy the chunks of multi-CTA windows back from the out-of-place target into the live array

// initial layout: src_n sentinels spread evenly (reference PCSR::PCSR, PCSR.cpp:796-837, in leaf-packed form)
__global__ void k_init_sentinels(uint32_t *__restrict__ dest, uint32_t *__restrict__ val, uint32_t *__restrict__ beg,
                                 uint32_t first_vertex, uint32_t count, uint32_t n_total, uint32_t m, uint32_t ls) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  // rank k of n_total items spread over m leaves: leaf = last o with floor(o*n/m) <= k
  const uint64_t o = (((uint64_t)k + 1) * m - 1) / n_total;
  const uint32_t f = k - (uint32_t)rank_begin(o, n_total, m);
  const size_t slot = ((size_t)o << ls) + f;
  dest[slot] = PPCSR_SENT;
  val[slot] = first_vertex + k + 1u;
  beg[first_vertex + k] = (uint32_t)slot;
}
__global__ void k_init_leaf_counts(uint32_t *__restrict__ leaf_cnt, uint32_t *__restrict__ tree, uint32_t n_total,
                                   uint32_t m) {
  const uint32_t o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= m) return;
  const uint32_t c = (uint32_t)(rank_begin((uint64_t)o + 1, n_total, m) - rank_begin(o, n_total, m));
  leaf_cnt[o] = c;
  tree[m + o] = c;
}
__global__ void k_set_u32(uint32_t *p, uint32_t v) { *p = v; }
__global__ void k_copy_u32(uint32_t *__restrict__ dst, const uint32_t *__restrict__ src, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i];
}

}  // namespace reb
