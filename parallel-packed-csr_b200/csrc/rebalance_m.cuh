// rebalance_m.cuh -- reb::k_rebalance_m: the rebalance of the windows that span more than SMALL_MAX_LEAVES leaves, and
// of the whole array.  The rank arithmetic of rebalance.cuh, dealt by OUTPUT RANK: the windows are cut into chunks of
// <= CHUNK_SLOTS output slots (k_plan_chunks_m), and a warp takes 32 CONSECUTIVE RANKS of the merged sequence per step
// ("unit"), so every lane has an item.  (Dealing SOURCE slots instead leaves half the lanes idle at the 50-65 % density
// of a PMA and costs every kept item a segmented scan, a marker look-up and a running maximum: ~760 instructions per
// chunk and warp whatever the chunk holds, issue-bound at 0.76 slots per cycle on the 2^29-slot rebuild, ncu.)
//
//   Two bit masks over the chunk's ranks say what a rank is:
//     B   bit t set <=> rank t is one of the batch's inserts      (one shared-memory atomicOr per insert)
//     HB  bit t set <=> a source leaf's merged run begins at t    (one atomicOr per non-empty source leaf)
//   and popcounts turn them into addresses:  q = (#B bits below t) + first insert index  is the insert a rank holds
//   or -- for a kept item -- the number of inserts before it; (#HB bits up to t) names its source leaf x, and
//       source slot = (t - q) + D[x],   D[x] = (x << ls) + a - R[x] + ins_off[x]
//   because the leaves are LEFT-PACKED: the kept items of a leaf are the first ones of its line.  (Tombstones of
//   this batch break that; batches with deletes run the TOMB instantiation, whose pre-pass maps kept index -> slot
//   per leaf.)  An item is read straight from the staged source line or the staged insert list and stored into its
//   final slot of the staging buffer through the rank -> slot table; ONE bulk store (TMA) per array writes the chunk.
//   ~36 branch-free instructions per unit of 32 items; the per-leaf and per-insert work is one atomicOr each.
//
// Pipeline: persistent CTAs (grid = SMs x M_CTAS) of eight consumer warps and one producer warp; a ROUND = one segment
// of <= 64 source leaves of one chunk; the bulk loads (cp.async.bulk -> mbarrier) of round r+1 -- source lines, R /
// insert-offset slices, the chunk's first 512 (1024 when the batch carries one value: no value list) inserts -- are
// issued by the producer at the top of round r into the other half of a double buffer, a full round ahead.
// Two block barriers per round (three for a chunk with tombstones AND inserts); the producer only arrives at the
// second one.  Measured (B200): the 2^29-slot rebuild of C4 in 1.67 ms = 78 % of the HBM copy peak, DRAM-bound; the
// scale-20 rebuilds are bound by the shared-memory data pipe (68 % busy: left-packed rows put every leaf's items on the
// low banks) at 60-67 %.
#pragma once
#include <type_traits>

#include "rebalance.cuh"

namespace reb {

struct ChunkPlanM {  // one 64-byte entry per chunk (k_plan_chunks_m)
  uint32_t leaf0;      // first leaf of the chunk's window
  uint32_t multi;      // != 0: the window spans several chunks (written out of place)
  uint32_t o_lo;       // first output leaf of the chunk, relative to the window
  uint32_t n_out;      // output leaves of the chunk
  uint32_t i_lo;       // first source leaf (relative to the window) feeding the chunk
  uint32_t nl;         // source leaves feeding the chunk (0: the chunk receives no items)
  uint32_t q_lo, q_hi; // inserts of those leaves that can rank inside the chunk
  uint32_t R0;         // rank_off[leaf0]
  uint32_t a;          // first window rank of the chunk
  uint32_t span;       // items the chunk receives
  uint32_t out_slot0;  // first output slot
  uint32_t items;      // live items of the window after the batch
  uint32_t lg;         // log2(output leaves of the window)
  uint32_t dst_leaf;   // first output leaf (absolute)
  uint32_t pad;
};
static_assert(sizeof(ChunkPlanM) == 64, "four 16-byte loads");

__global__ void __launch_bounds__(RT) k_plan_chunks_m(const WindowDesc *__restrict__ windows, uint32_t n_windows,
                                                      const uint32_t *__restrict__ rank_off,
                                                      const uint32_t *__restrict__ ins_off, uint32_t ls_src,
                                                      uint32_t ls_dst, uint32_t m_dst_override, uint32_t n_chunks,
                                                      uint32_t CL, ChunkPlanM *__restrict__ plan) {
  const uint32_t chunk = blockIdx.x * blockDim.x + threadIdx.x;
  if (chunk >= n_chunks) return;
  uint32_t lo = 0, hi = n_windows;  // last window with chunk0 <= chunk
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (windows[mid].chunk0 <= chunk) lo = mid;
    else hi = mid;
  }
  const WindowDesc w = windows[lo];
  const uint32_t m_dst = m_dst_override ? m_dst_override : w.m;
  const uint32_t lg = 31u - (uint32_t)__clz(m_dst);
  const uint32_t o_lo = (chunk - w.chunk0) * CL;
  const uint32_t o_hi = min(o_lo + CL, m_dst);
  const uint32_t a = leaf_rank0(o_lo, w.items, lg);
  const uint32_t b = leaf_rank0(o_hi, w.items, lg);
  const uint32_t *R = rank_off + w.leaf0;
  const uint32_t *IO = ins_off + w.leaf0;
  const uint32_t R0 = R[0];
  ChunkPlanM p;
  p.leaf0 = w.leaf0;
  p.multi = w.n_chunks > 1 ? 1u : 0u;
  p.o_lo = o_lo;
  p.n_out = o_hi - o_lo;
  p.R0 = R0;
  p.a = a;
  p.span = b - a;
  const uint32_t dst_leaf0 = m_dst_override ? 0u : w.leaf0;
  p.dst_leaf = dst_leaf0 + o_lo;
  p.out_slot0 = (dst_leaf0 + o_lo) << ls_dst;
  p.items = w.items;
  p.lg = lg;
  p.pad = 0;
  if (b > a) {
    const uint32_t i_lo = upper_bound_u32(R, w.m, R0 + a) - 1;      // source leaf holding rank a
    const uint32_t i_hi = upper_bound_u32(R, w.m, R0 + b - 1) - 1;  // source leaf holding rank b-1
    const uint32_t below = a - (R[i_lo] - R0);                      // ranks of the first leaf below the chunk
    const uint32_t leaf = 1u << ls_src;
    // an insert ranks at R[leaf] + (its index in the leaf's run) + (kept items up to its predecessor, <= one leaf):
    // those of the first leaf before IO + (below - leaf) rank below a, those of the last from IO + (b - R) on at or
    // above b -- a hub run spanning thousands of chunks is clipped to <= span + leaf inserts per chunk without a search
    p.i_lo = i_lo;
    p.nl = i_hi - i_lo + 1u;
    p.q_lo = min(IO[i_lo] + (below > leaf ? below - leaf : 0u), IO[i_lo + 1]);
    p.q_hi = max(p.q_lo, min(IO[i_hi] + (b - (R[i_hi] - R0)), IO[i_hi + 1]));
  } else {
    p.i_lo = 0;
    p.nl = 0;
    p.q_lo = p.q_hi = 0;
  }
  plan[chunk] = p;
}

#ifndef PPCSR_M_CTAS
#define PPCSR_M_CTAS 3
#endif
#ifndef PPCSR_M_PINS
#define PPCSR_M_PINS 512
#endif
constexpr int MT = 256;                        // consumer threads of a k_rebalance_m CTA (warps 0..7)
constexpr int MTT = MT + 32;                   // + the producer warp
constexpr int MCHUNK = CHUNK_SLOTS;            // output slots per chunk
constexpr int MSEG = SEG_LEAVES_SLOTS;         // source slots per round
constexpr int MSEG_MAX_LEAVES = SEG_MAX_LEAVES;
constexpr int MTBL = MSEG_MAX_LEAVES + 1;
// staged inserts per chunk: what fits beside the other buffers at three CTAs per SM.  UNIV (every insert of the batch
// carries the same value: no value array is read at all) leaves room for more of them
template <bool TOMB, bool UNIV>
struct MCfg {
  static constexpr int PINS = UNIV ? (TOMB ? 768 : 1024) : PPCSR_M_PINS;
};
constexpr int MWORDS = MCHUNK / 32;            // mask words
static_assert(MT == 256, "k_rebalance_m deals its phases to eight warps");
static_assert(MCHUNK <= 65536, "rank -> slot table entries are 16-bit");

#ifdef PPCSR_M_TRACE
// development: clock stamps of the first rounds of four CTAs (lane 0 of every warp), dumped by capi.cu after the launch
__device__ uint32_t g_m_trace[4][64][9][8];
#define MTRACE(ev)                                                                     \
  do {                                                                                 \
    if (blockIdx.x < 4 && r < 64 && lane == 0) g_m_trace[blockIdx.x][r][warp][ev] = (uint32_t)clock64(); \
  } while (0)
#else
#define MTRACE(ev) \
  do {             \
  } while (0)
#endif

template <bool TOMB, bool UNIV>
struct MSmem {
  static constexpr int MPINS = MCfg<TOMB, UNIV>::PINS;
  uint32_t out_d[MCHUNK];  // the chunk's output slots in their final layout (first member: at the base, see k_rebalance_m)
  uint32_t out_v[MCHUNK];
  // one word-indexed region W: the source lines and staged inserts.  st_v - st_d == st_iv - st_id (== VOFF words), so
  // an item's value sits VOFF words behind its dest whichever it is (UNIV: no st_iv; the insert lanes read a word of
  // st_ip there and drop it)
  uint32_t st_d[2][MSEG];        // [round parity]
  uint32_t st_id[2][MPINS + 8];  // [chunk parity]
  uint32_t st_v[2][MSEG];
  uint32_t st_iv[UNIV ? 1 : 2][UNIV ? 4 : MPINS + 8];
  uint32_t st_ip[2][MPINS + 8];
  alignas(16) uint32_t st_R[2][MTBL + 7];     // R slice of the round's leaves; entry x sits at [x + (first leaf & 3)]
  alignas(16) uint32_t st_ioff[2][MTBL + 7];  // insert offsets of the same leaves
  alignas(16) uint32_t B[2][MWORDS];          // [round parity] insert ranks
  alignas(16) uint32_t HB[2][MWORDS];         // leaf heads
  uint32_t D[MSEG_MAX_LEAVES];                // per non-empty leaf of the round, in order: source slot - (rank - inserts before)
  uint16_t pos[MCHUNK];                       // chunk-relative rank -> output slot
  uint8_t kmap[TOMB ? MSEG : 16];             // [leaf base + kept index] -> offset of that kept item in its leaf
  uint8_t kupto[TOMB ? MSEG : 16];            // kept items of the leaf up to and including a slot
  alignas(16) uint4 plan[2][4];               // [chunk parity]
  uint32_t n_below[2];                        // [chunk parity] staged inserts of the chunk's first leaf that rank below it
  alignas(8) uint64_t full[2];                // [round parity] the round's bulk loads have landed
};

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bar_consumers() { asm volatile("bar.sync 1, %0;" ::"n"(MT) : "memory"); }
// mid-round barrier: the consumers wait, the producer only arrives (its part -- staging buffers free -- is done)
__device__ __forceinline__ void bar_mid_sync() { asm volatile("bar.sync 2, %0;" ::"n"(MTT) : "memory"); }
__device__ __forceinline__ void bar_mid_arrive() { asm volatile("bar.arrive 2, %0;" ::"n"(MTT) : "memory"); }

// Warps 0..7 are CONSUMERS (masks, tables, placement); warp 8 is the PRODUCER: after the round's opening barrier its
// lane 0 stores the finished chunk (bulk store), issues the bulk loads of the NEXT round -- one cp.async.bulk costs the
// issuing thread 70-170 cycles (benchmarks/micro/tma_issue.cu), a dozen of them was the longest path of a round when a
// consumer issued them --, waits until the copy engine has read the staging buffers, re-nulls them where needed and
// arrives on `stready`.  It takes no part in the consumers' mid-round barrier.
template <bool TOMB, bool UNIV>
__global__ void __launch_bounds__(MTT, PPCSR_M_CTAS) k_rebalance_m(Args A, const ChunkPlanM *__restrict__ gplan,
                                                                  uint32_t n_chunks) {
  // The kernel has no static shared memory, so its dynamic shared memory starts at the base of the CTA's window,
  // whatever alignment is declared here.  16, like every dynamic shared-memory declaration of the library: ptxas aligns
  // the dynamic shared memory of ALL kernels of the module to one of these declarations (which one depends on the order
  // the kernels are emitted in), and a larger one here would move it in the sort and routing kernels.
  extern __shared__ __align__(16) uint8_t m_smem_raw[];
  using SM = MSmem<TOMB, UNIV>;
  constexpr int MPINS = SM::MPINS;
  SM &S = *reinterpret_cast<SM *>(m_smem_raw);
  constexpr uint32_t VOFF = (uint32_t)(offsetof(SM, st_v) - offsetof(SM, st_d)) / 4u;
  static_assert(offsetof(SM, st_iv) - offsetof(SM, st_id) == offsetof(SM, st_v) - offsetof(SM, st_d), "VOFF");
  static_assert(sizeof(SM) <= 75 * 1024, "three CTAs per SM");
  const uint32_t uval = A.ins_uniform;
  constexpr uint32_t INS_W = (uint32_t)(offsetof(SM, st_id) - offsetof(SM, st_d)) / 4u;  // word index of st_id[0][0]
  const uint32_t *W = &S.st_d[0][0];

  const unsigned lane = lane_id(), lt = lanemask_lt(), le = lt | (1u << lane);
  const unsigned warp = threadIdx.x >> 5;
  const bool producer = warp == 8;
  const uint32_t ls_src = A.ls_src, ls_dst = A.ls_dst;
  const uint32_t leaf_mask = (1u << ls_src) - 1u;
  const uint32_t seg_leaves = min((uint32_t)MSEG >> ls_src, (uint32_t)MSEG_MAX_LEAVES);
  const uint32_t G = gridDim.x;
  uint32_t c = blockIdx.x;
  if (c >= n_chunks) return;

  // ---- the bulk loads of one round (producer, lane 0): source lines + table slices of the leaves [gl, gl + snl), and,
  // when the round opens a chunk, the chunk's first MPINS inserts
  auto issue_round = [&](uint32_t rpar, uint32_t gl, uint32_t snl, bool first, uint32_t cpar, uint32_t q_lo,
                         uint32_t q_hi) {
    uint64_t *bar = &S.full[rpar];
    if (snl == 0) {
      mbar_expect_tx(bar, 0u);
      return;
    }
    const uint32_t qb = (snl << ls_src) * 4u;
    const uint32_t sh = gl & 3u;
    // 16-byte granules: reads up to 3 entries past the logical end of the arrays (covered by DEV_PAD_ELEMS)
    const uint32_t tb = ((snl + 1u + sh + 3u) & ~3u) * 4u;
    const uint32_t nq = first ? min(q_hi - q_lo, (uint32_t)MPINS) : 0u;
    const uint32_t ish = q_lo & 3u;
    const uint32_t ib = nq ? ((nq + ish + 3u) & ~3u) * 4u : 0u;
    mbar_expect_tx(bar, 2u * qb + 2u * tb + (UNIV ? 2u : 3u) * ib);
    bulk_g2s(S.st_R[rpar], A.rank_off + (gl - sh), tb, bar);
    bulk_g2s(S.st_ioff[rpar], A.ins_off + (gl - sh), tb, bar);
    if (ib) {
      bulk_g2s(S.st_ip[cpar], A.ins_pred + (q_lo - ish), ib, bar);
      bulk_g2s(S.st_id[cpar], A.ins_dst + (q_lo - ish), ib, bar);
      if (!UNIV) bulk_g2s(S.st_iv[cpar], A.ins_val + (q_lo - ish), ib, bar);
    }
    bulk_g2s(S.st_d[rpar], A.src_dest + ((size_t)gl << ls_src), qb, bar);
    bulk_g2s(S.st_v[rpar], A.src_val + ((size_t)gl << ls_src), qb, bar);
    if (ib && q_hi - q_lo > (uint32_t)MPINS) {  // a longer run is read straight from global memory: pull it into L2
      const uint32_t q1 = (q_lo + MPINS) & ~3u;
      const uint32_t pb = min(((q_hi - q1 + 3u) & ~3u) * 4u, 16384u);
      bulk_prefetch_l2(A.ins_pred + q1, pb);
      bulk_prefetch_l2(A.ins_dst + q1, pb);
      if (!UNIV) bulk_prefetch_l2(A.ins_val + q1, pb);
    }
  };

  // ---- prologue: the first chunk's plan entry, clear masks, arm the barriers, loads of round 0
  uint4 n0, n1, n2, n3;  // producer: plan entry of this CTA's NEXT chunk
  n0 = n1 = n2 = n3 = make_uint4(0u, 0u, 0u, 0u);
  {
    const uint4 *g = reinterpret_cast<const uint4 *>(gplan + c);
    const uint4 p0 = __ldg(g), p1 = __ldg(g + 1);
    if (threadIdx.x == 0) {
      S.plan[0][0] = p0;
      S.plan[0][1] = p1;
      S.plan[0][2] = __ldg(g + 2);
      S.plan[0][3] = __ldg(g + 3);
    }
    if (threadIdx.x < 2u * MWORDS) {
      (&S.B[0][0])[threadIdx.x] = 0u;
      (&S.HB[0][0])[threadIdx.x] = 0u;
    }
    if (threadIdx.x == 0) {
      S.n_below[0] = S.n_below[1] = 0u;
      mbar_init(&S.full[0], 1u);
      mbar_init(&S.full[1], 1u);
    }
    __syncthreads();
    if (producer && lane == 0) {
      issue_round(0u, p0.x + p1.x, min(seg_leaves, p1.y), true, 0u, p1.z, p1.w);
      if (c + G < n_chunks) {
        const uint4 *gn = reinterpret_cast<const uint4 *>(gplan + c + G);
        n0 = __ldg(gn);
        n1 = __ldg(gn + 1);
        n2 = __ldg(gn + 2);
        n3 = __ldg(gn + 3);
      }
    }
  }

  uint32_t k = 0, seg = 0, r = 0;  // chunks done by this CTA, first leaf of the segment within the chunk, round
  bool store_pending = false;
  // the chunk in progress (registers, set by its first round)
  uint32_t nl = 0, q_lo = 0, q_hi = 0, a = 0, span = 0, R0 = 0, gl0 = 0, out_slot0 = 0, n_out = 0, multi = 0;
  uint32_t *const beg_m1 = A.beg - 1;  // a sentinel's value is its vertex + 1
  const uint32_t lbit = 1u << lane;

  for (;;) {
    if (store_pending && !producer) fence_proxy_async_smem();  // my placements are visible to the bulk-copy engine
    __syncthreads();                                           // B0: everybody has left round r-1
    if (store_pending) {
      if (producer && lane == 0) {  // the finished chunk leaves: one bulk store per array
        const uint32_t bytes = (n_out << ls_dst) * 4u;
        bulk_s2g((multi ? A.out_dest_multi : A.out_dest_single) + out_slot0, S.out_d, bytes);
        bulk_s2g((multi ? A.out_val_multi : A.out_val_single) + out_slot0, S.out_v, bytes);
        bulk_commit();
      }
      store_pending = false;
      if (c >= n_chunks) break;
    }
    MTRACE(0);
    const uint32_t rpar = r & 1u, cpar = k & 1u;
    const bool first_seg = seg == 0;
    if (first_seg) {
      const uint4 p0 = S.plan[cpar][0], p1 = S.plan[cpar][1], p2 = S.plan[cpar][2];
      multi = p0.y;
      n_out = p0.w;
      gl0 = p0.x + p1.x;
      nl = p1.y;
      q_lo = p1.z;
      q_hi = p1.w;
      R0 = p2.x;
      a = p2.y;
      span = p2.z;
      out_slot0 = p2.w;
    }
    const bool last_seg = seg + seg_leaves >= nl;
    // A whole-array rebuild gives every output leaf floor(j / m) or that + 1 items, chunk after chunk: the staging
    // buffers need no re-nulling between chunks -- the only slot of a leaf that can hold a stale item is the one
    // behind its last item (nulled by the leaf's thread, see zpos).  Chunks of <= 64 output leaves only.
    const bool keep_nulls = A.m_dst_override != 0u && k > 0u && n_out <= 64u;

    if (producer) {
      if (lane == 0) {
        // ---- the next round's operands
        if (!last_seg) {
          issue_round(rpar ^ 1u, gl0 + seg + seg_leaves, min(seg_leaves, nl - seg - seg_leaves), false, cpar, 0u, 0u);
        } else if (c + G < n_chunks) {
          S.plan[cpar ^ 1u][0] = n0;
          S.plan[cpar ^ 1u][1] = n1;
          S.plan[cpar ^ 1u][2] = n2;
          S.plan[cpar ^ 1u][3] = n3;
          issue_round(rpar ^ 1u, n0.x + n1.x, min(seg_leaves, n1.y), true, cpar ^ 1u, n1.z, n1.w);
          if (c + 2u * G < n_chunks) {
            const uint4 *gn = reinterpret_cast<const uint4 *>(gplan + c + 2u * G);
            n0 = __ldg(gn);
            n1 = __ldg(gn + 1);
            n2 = __ldg(gn + 2);
            n3 = __ldg(gn + 3);
          }
        }
        if (first_seg) bulk_wait_read0();  // the copy engine has read the previous chunk out of the staging buffers
      }
      if (first_seg && !keep_nulls) {
        __syncwarp();
        const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
        uint4 *z = reinterpret_cast<uint4 *>(S.out_d);  // out_d and out_v are adjacent
#pragma unroll 8
        for (int x = 0; x < 2 * MCHUNK / 4 / 32; x++) z[x * 32 + lane] = zero;
      }
      __syncwarp();
      bar_mid_arrive();  // the staging buffers are free (and nulled)
      MTRACE(1);
    } else {
      mbar_wait(&S.full[rpar], (r >> 1) & 1u);  // this round's operands have landed
      MTRACE(2);

      const uint32_t snl = min(seg_leaves, nl - seg);  // nl == 0: seg == 0, snl == 0
      const uint32_t seg_slot0 = (gl0 + seg) << ls_src;
      const uint32_t seg_slots = snl << ls_src;
      const uint32_t *t_R = S.st_R[rpar] + ((gl0 + seg) & 3u), *t_ioff = S.st_ioff[rpar] + ((gl0 + seg) & 3u);
      const uint32_t ish = q_lo & 3u;
      const uint32_t Ra = R0 + a;  // absolute rank of the chunk's first item
      // the segment's inserts [qa, qb) and its chunk-relative rank range [ta, tb); a chunk of one segment needs no look-up
      uint32_t qa = q_lo, qb = q_hi, ta = 0, tb = span;
      if (!(first_seg && last_seg)) {
        qa = max(q_lo, t_ioff[0]);
        qb = min(q_hi, t_ioff[snl]);
        const uint32_t r_lo = t_R[0], r_hi = t_R[snl];
        ta = r_lo > Ra ? r_lo - Ra : 0u;
        tb = min(span, r_hi > Ra ? r_hi - Ra : 0u);
        if (tb < ta) tb = ta;
      }
      const bool staged_all = q_hi - q_lo <= (uint32_t)MPINS;  // every insert of the chunk sits in the stage

      if (TOMB) {
        // ---- pre-pass: kept flags of the staged lines (tombstones have val 0), per leaf: kept index -> offset (kmap)
        // and, when the chunk has inserts, kept items up to each slot (kupto).  One 16-byte quad per thread and step, a
        // leaf = 2, 4 or 8 lanes.
        const uint32_t lpl = 1u << (ls_src - 2u);
        const uint32_t warp_rel0 = (threadIdx.x & ~31u) * 4u;
        const bool want_kupto = q_hi != q_lo;
#pragma unroll
        for (int u = 0; u < MSEG / 4 / MT; u++) {
          if (u * MT * 4u + warp_rel0 >= seg_slots) continue;  // warp-uniform
          const uint32_t rel = (u * MT + threadIdx.x) * 4u;
          uint4 V = make_uint4(0u, 0u, 0u, 0u);
          if (rel < seg_slots) V = *reinterpret_cast<const uint4 *>(&S.st_v[rpar][rel]);
          const uint32_t k0 = V.x != 0u, k1 = V.y != 0u, k2 = V.z != 0u, k3 = V.w != 0u;
          const uint32_t cc = k0 + k1 + k2 + k3;
          const uint32_t pre = leaf_incl_scan(cc, lane, lpl) - cc;  // kept items of my leaf in lower lanes
          const uint32_t p0 = pre + k0, p1 = p0 + k1, p2 = p1 + k2;
          if (rel < seg_slots) {
            if (want_kupto)
              *reinterpret_cast<uint32_t *>(&S.kupto[rel]) = p0 | (p1 << 8) | (p2 << 16) | ((p2 + k3) << 24);
            uint8_t *km = &S.kmap[rel & ~leaf_mask];
            const uint32_t f0 = rel & leaf_mask;
            if (k0) km[pre] = (uint8_t)f0;
            if (k1) km[p0] = (uint8_t)(f0 + 1u);
            if (k2) km[p1] = (uint8_t)(f0 + 2u);
            if (k3) km[p2] = (uint8_t)(f0 + 3u);
          }
        }
        if (want_kupto) bar_consumers();  // the inserts below read kupto (chunk-uniform)
      }

      // ---- phase 1: a small task for the warps 0..2, then the segment's inserts dealt over the warps 3..7, 0..2
      uint32_t zpos = 0xFFFFFFFFu;  // warps 1, 2: the slot of my output leaf that may hold a stale item (keep_nulls)
      if (warp == 0) {
        // leaf heads + per-leaf address offsets; the other parity's masks are cleared for the next round
        static_assert(MWORDS == 64, "16 lanes x 16 bytes clear one mask");
        if (lane < 16u) reinterpret_cast<uint4 *>(S.B[rpar ^ 1u])[lane] = make_uint4(0u, 0u, 0u, 0u);
        else reinterpret_cast<uint4 *>(S.HB[rpar ^ 1u])[lane - 16u] = make_uint4(0u, 0u, 0u, 0u);
        if (lane == 0) S.n_below[cpar ^ 1u] = 0u;
        uint32_t base = 0;
        for (uint32_t x0 = 0; x0 < snl; x0 += 32u) {
          const uint32_t x = x0 + lane;
          bool ne = false;
          uint32_t p = 0, dv = 0;
          if (x < snl) {
            const uint32_t Rx = t_R[x], Rx1 = t_R[x + 1u];
            // the leaf's merged run [Rx, Rx1) meets the chunk's ranks [Ra, Ra + span)
            ne = Rx1 > Rx && Rx1 > Ra && Rx < Ra + span;
            p = Rx > Ra ? Rx - Ra : 0u;
            dv = (x << ls_src) + Ra - Rx + t_ioff[x];
          }
          const unsigned nm = __ballot_sync(0xFFFFFFFFu, ne);
          if (ne) {
            atomicOr(&S.HB[rpar][p >> 5], 1u << (p & 31u));
            S.D[base + __popc(nm & lt)] = dv;
          }
          base += __popc(nm);
        }
      } else if (warp <= 2) {
        if (first_seg) {  // rank -> slot table and post-rebalance leaf counts of the chunk: one thread per output leaf
          const uint4 p0 = S.plan[cpar][0], p3 = S.plan[cpar][3];
          const uint32_t o_lo = p0.z, items = p3.x, lg = p3.y, dst_leaf = p3.z;
          for (uint32_t kk = threadIdx.x - 32u; kk < n_out; kk += 64u) {
            const uint32_t a_k = leaf_rank0(o_lo + kk, items, lg) - a;
            const uint32_t c_k = leaf_rank0(o_lo + kk + 1u, items, lg) - a - a_k;
            uint16_t *pk = &S.pos[a_k];
            const uint32_t b_k = kk << ls_dst;
#pragma unroll 4
            for (uint32_t i = 0; i < c_k; i++) pk[i] = (uint16_t)(b_k + i);
            A.tree_leaf_out[dst_leaf + kk] = c_k;
            if (A.leaf_cnt_out) A.leaf_cnt_out[dst_leaf + kk] = c_k;
            if (keep_nulls && (c_k >> ls_dst) == 0u) zpos = b_k + c_k;
          }
        }
      }
      {
        // the segment's inserts: rank = R[leaf] + index in the leaf's run + kept items up to the predecessor -> B
        uint32_t below = 0;
        const uint32_t wbase = ((warp + 5u) & 7u) * 32u;   // the warps without a task of their own come first
        const uint32_t *sip = S.st_ip[cpar] + ish - q_lo;  // + q = staged predecessor of insert q
        for (uint32_t q0 = qa + wbase; q0 < qb; q0 += (uint32_t)MT) {  // warp-uniform trip count
          const uint32_t q = q0 + lane;
          uint32_t word = 0xFFFFFFFFu, bit = 0;
          if (q < qb) {
            const uint32_t pred = (staged_all || q - q_lo < (uint32_t)MPINS) ? sip[q] : A.ins_pred[q];
            const uint32_t rel = pred - seg_slot0;
            const uint32_t x = rel >> ls_src;
            const uint32_t kup = TOMB ? (uint32_t)S.kupto[rel] : (rel & leaf_mask) + 1u;
            const uint32_t tt = t_R[x] + (q - t_ioff[x]) + kup - Ra;
            if (tt < span) {
              word = tt >> 5;
              bit = 1u << (tt & 31u);
            } else if ((int32_t)tt < 0) {
              below++;
            }
          }
          // (one atomic per lane: warp-aggregating the lanes that share a word through match.any measured slower than
          // the ~10-way same-word atomics it avoids)
          if (word != 0xFFFFFFFFu) atomicOr(&S.B[rpar][word], bit);
        }
        if (first_seg) {
          below = __reduce_add_sync(0xFFFFFFFFu, below);
          if (lane == 0 && below) atomicAdd(&S.n_below[cpar], below);
        }
      }
      MTRACE(3);
      bar_mid_sync();  // B1: masks and tables are complete, the staging buffers are free (producer)
      MTRACE(4);
      if (zpos != 0xFFFFFFFFu) {  // the slot behind my leaf's last item (see keep_nulls)
        S.out_d[zpos] = 0u;
        S.out_v[zpos] = 0u;
      }

      // ---- phase 2: the segment's ranks [ta, tb), 32 per warp and step ("unit"), each warp a contiguous run of units
      const uint32_t wa = ta >> 5, wb = (tb + 31u) >> 5, nu = wb - wa;
      const uint32_t w0 = wa + ((nu * warp) >> 3), w1 = wa + ((nu * (warp + 1u)) >> 3);
      if (w0 < w1) {
        // inserts / leaf heads before my first unit
        uint32_t cnt = 0;
        if (lane < w0) cnt = __popc(S.B[rpar][lane]) | (__popc(S.HB[rpar][lane]) << 16);
        if (lane + 32u < w0) cnt += __popc(S.B[rpar][lane + 32u]) | (__popc(S.HB[rpar][lane + 32u]) << 16);
        cnt = __reduce_add_sync(0xFFFFFFFFu, cnt);
        uint32_t pbase = (first_seg ? q_lo + S.n_below[cpar] : qa) + (cnt & 0xFFFFu);
        uint32_t fbase = (cnt >> 16) - 1u;
        MTRACE(5);
        const uint32_t sbt = rpar * (uint32_t)MSEG + lane;                        // + 32 w - q + D = word of a kept item
        const uint32_t insb = INS_W + cpar * (uint32_t)(MPINS + 8) + ish - q_lo;  // + q = word of staged insert q
        const uint32_t *Bm = S.B[rpar], *Hm = S.HB[rpar];
        // one unit; CHECK: the unit is cut by the segment's rank range, STAGED: no insert lies beyond the stage
        // NOINS: the chunk has no inserts at all (a batch of deletes)
        auto unit = [&](auto CHECK, auto STAGED, auto NOINS, uint32_t w) {
          const uint32_t bw = decltype(NOINS)::value ? 0u : Bm[w], hb = Hm[w];
          const uint32_t q = pbase + __popc(bw & lt);
          const uint32_t kidx = fbase + __popc(hb & le);
          pbase += __popc(bw);
          fbase += __popc(hb);
          const uint32_t t = (w << 5) + lane;
          if (decltype(CHECK)::value && !(t >= ta && t < tb)) return;
          const uint32_t dk = S.D[kidx];
          uint32_t idx;
          if (TOMB) {
            const uint32_t ki = t - q + dk;  // leaf base + kept index
            idx = rpar * (uint32_t)MSEG + (ki & ~leaf_mask) + S.kmap[ki & (uint32_t)(MSEG - 1)];
          } else {
            idx = sbt + (w << 5) - q + dk;
          }
          const bool isins = (bw & lbit) != 0u;
          if (isins) idx = insb + q;
          uint32_t d, v;
          if (!decltype(STAGED)::value && isins && q - q_lo >= (uint32_t)MPINS) {  // a long run of inserts
            d = A.ins_dst[q];
            v = UNIV ? uval : A.ins_val[q];
          } else {
            d = W[idx];
            v = W[idx + VOFF];
            if (UNIV && isins) v = uval;
          }
          const uint32_t pos = S.pos[t];
          S.out_d[pos] = d;
          S.out_v[pos] = v;
          // fix_sentinel (reference PCSR.cpp:168-183): a sentinel that lands here refreshes its vertex's back pointer
          if (d == PPCSR_SENT) beg_m1[v] = out_slot0 + pos;
        };
        auto run = [&](auto STAGED, auto NOINS) {
          uint32_t w = w0, wl = w1;
          if (w == wa && (ta & 31u)) unit(std::true_type{}, STAGED, NOINS, w++);
          const bool cut_tail = w1 == wb && (tb & 31u) && w < w1;
          if (cut_tail) wl--;
#pragma unroll 4
          for (; w < wl; w++) unit(std::false_type{}, STAGED, NOINS, w);
          if (cut_tail) unit(std::true_type{}, STAGED, NOINS, w);
        };
        if (q_hi == q_lo) run(std::true_type{}, std::true_type{});
        else if (staged_all) run(std::true_type{}, std::false_type{});
        else run(std::false_type{}, std::false_type{});
      }
      MTRACE(6);
    }
    r++;
    if (!last_seg) {
      seg += seg_leaves;
      continue;
    }
    // every source leaf of the chunk has been read and placed: the chunk is stored after the next barrier
    store_pending = true;
    c += G;
    k++;
    seg = 0;
  }
  if (producer && lane == 0) bulk_wait_read0();  // the staging buffers must outlive the last copy
}

// copy the chunks of multi-CTA windows back from the out-of-place target into the live array
__global__ void __launch_bounds__(RT) k_copy_back_m(const ChunkPlanM *__restrict__ plan, uint32_t ls,
                                                    const uint32_t *__restrict__ alt_dest,
                                                    const uint32_t *__restrict__ alt_val, uint32_t *__restrict__ dest,
                                                    uint32_t *__restrict__ val) {
  const ChunkPlanM p = plan[blockIdx.x];
  if (!p.multi) return;
  const size_t base = (size_t)p.out_slot0;
  const uint32_t slots = p.n_out << ls;
  for (uint32_t x = threadIdx.x * 4; x < slots; x += RT * 4) {
    *reinterpret_cast<uint4 *>(dest + base + x) = *reinterpret_cast<const uint4 *>(alt_dest + base + x);
    *reinterpret_cast<uint4 *>(val + base + x) = *reinterpret_cast<const uint4 *>(alt_val + base + x);
  }
}

}  // namespace reb
