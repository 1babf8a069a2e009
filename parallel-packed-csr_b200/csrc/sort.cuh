// sort.cuh -- stable LSD radix sort of the update batch by (src,dst): single-pass-per-digit ("onesweep")
// with decoupled look-back, hand-written for sm_100a (no CUB/Thrust).
//
// Orders the batch the way the reference's per-op lock acquisition would serialise it
// (src/pcsr/PCSR.cpp:1374-1445): by source vertex, then by destination, submission order kept among
// equal keys, so that the LAST element of a run of equal keys is the last op submitted for that edge.
//
// The key (src << 32 | dst) is compacted on the fly to (src << lo_bits | dst): only lo_bits + hi_bits
// bits are live (40 at R-MAT scale 20, 48 at scale 24) and the passes cover exactly that field in
// digits of <= 8 bits (5 passes at scale 20).
//
//   k_os_hist   one read of the keys: the global digit histograms of ALL passes (shared-memory atomics)
//   k_os_scan   exclusive scan of each pass's 256 bins  -> first output position of every digit
//   k_os_pass   per pass, ONE read and ONE write of the batch: a CTA takes the next tile of 4096 keys
//               (ticket counter, so that every earlier tile is already running), ranks its keys
//               warp-synchronously, publishes the tile's digit counts, resolves the counts of all
//               earlier tiles by decoupled look-back (aggregate / inclusive-prefix flags in one word),
//               reorders the tile in shared memory and writes digit runs (16 keys = 128 B on average).
// HBM traffic per pass: 16 B per update (+8 with per-update values) -- the floor for an LSD pass.
#pragma once
#include <algorithm>
#include <mutex>

#include "common.cuh"
#include "primitives.cuh"

namespace prim {

constexpr int OS_THREADS = 256;
constexpr int OS_WARPS = OS_THREADS / 32;
constexpr int OS_ITEMS = 16;
constexpr int OS_TILE = OS_THREADS * OS_ITEMS;  // 4096 keys per CTA
constexpr int OS_RADIX_BITS = 8;
constexpr int OS_RADIX = 1 << OS_RADIX_BITS;
constexpr int OS_MAX_PASSES = 8;
constexpr uint32_t OS_FLAG_AGG = 1u << 30;  // tile-local count published
constexpr uint32_t OS_FLAG_INC = 2u << 30;  // inclusive prefix over all tiles up to this one published
constexpr uint32_t OS_VAL_MASK = (1u << 30) - 1u;
constexpr int OS_LB_DEPTH = 8;               // predecessors examined per look-back step
constexpr size_t OS_LATE_MIN_KEYS = (size_t)1 << 25;  // see k_os_pass<.., EARLY>
constexpr uint64_t OS_MAX_COUNT = OS_VAL_MASK;  // look-back words carry 30-bit counts

struct SortPasses {
  int n_pass;
  int lo_bits;
  int shift[OS_MAX_PASSES];
  uint32_t mask[OS_MAX_PASSES];
};

inline SortPasses make_sort_passes(int lo_bits, int hi_bits) {
  SortPasses P{};
  P.lo_bits = lo_bits;
  const int total = lo_bits + hi_bits;
  P.n_pass = (total + OS_RADIX_BITS - 1) / OS_RADIX_BITS;
  const int width = (total + P.n_pass - 1) / P.n_pass;
  int done = 0;
  for (int p = 0; p < P.n_pass; p++) {
    const int w = (total - done) < width ? (total - done) : width;
    P.shift[p] = done;
    P.mask[p] = (1u << w) - 1u;
    done += w;
  }
  return P;
}

__device__ __forceinline__ uint64_t sort_compact(uint64_t key, int lo_bits) {
  return lo_bits >= 32 ? key : (((key >> 32) << lo_bits) | (uint32_t)key);
}
__device__ __forceinline__ uint32_t sort_digit(uint64_t key, int lo_bits, int shift, uint32_t mask) {
  return (uint32_t)(sort_compact(key, lo_bits) >> shift) & mask;
}

// Where a pass of the sort takes its keys (and payloads) from.  The kernels take it as a template parameter, so their
// instance names (k_os_pass<false,prim::KeyArray,true>, which tests and profiles match) carry it.
struct KeyArray {
  const uint64_t *keys;
  const uint32_t *pay;
  __device__ __forceinline__ uint64_t key(size_t i) const { return keys[i]; }
  __device__ __forceinline__ uint32_t payload(size_t i) const { return pay[i]; }
};

// ---- global histograms of every pass, one read of the keys --------------------------------------------
constexpr int OSH_THREADS = 512;
constexpr int OSH_ITEMS = 8;

template <class Src>
__global__ void __launch_bounds__(OSH_THREADS) k_os_hist(Src src, size_t n, SortPasses P,
                                                         uint32_t *__restrict__ ghist) {
  __shared__ uint32_t s_h[OS_MAX_PASSES * OS_RADIX];
  for (int i = threadIdx.x; i < P.n_pass * OS_RADIX; i += OSH_THREADS) s_h[i] = 0;
  __syncthreads();
  const size_t chunk = (size_t)OSH_THREADS * OSH_ITEMS;
  for (size_t base = (size_t)blockIdx.x * chunk; base < n; base += (size_t)gridDim.x * chunk) {
    uint64_t k[OSH_ITEMS];
#pragma unroll
    for (int r = 0; r < OSH_ITEMS; r++) {
      const size_t i = base + (size_t)r * OSH_THREADS + threadIdx.x;
      k[r] = i < n ? src.key(i) : 0;
    }
#pragma unroll
    for (int r = 0; r < OSH_ITEMS; r++) {
      const size_t i = base + (size_t)r * OSH_THREADS + threadIdx.x;
      if (i < n) {
        const uint64_t ck = sort_compact(k[r], P.lo_bits);
#pragma unroll
        for (int p = 0; p < OS_MAX_PASSES; p++)
          if (p < P.n_pass) atomicAdd(&s_h[p * OS_RADIX + ((uint32_t)(ck >> P.shift[p]) & P.mask[p])], 1u);
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < P.n_pass * OS_RADIX; i += OSH_THREADS)
    if (s_h[i]) atomicAdd(&ghist[i], s_h[i]);
}

// one block per pass: ghist[p][d] -> exclusive prefix (first output position of digit d in pass p); also
// stamps the (INC, 0) rows in front of the pass's look-back table
__global__ void __launch_bounds__(OS_RADIX) k_os_scan(uint32_t *__restrict__ ghist, uint32_t *__restrict__ lookback,
                                                      size_t rows_per_pass) {
  __shared__ uint32_t s_warp[33];
  uint32_t *h = ghist + (size_t)blockIdx.x * OS_RADIX;
  const uint32_t v = h[threadIdx.x];
  uint32_t total;
  const uint32_t ex = block_excl_scan(v, &total, s_warp);
  h[threadIdx.x] = ex;
  uint32_t *pad = lookback + (size_t)blockIdx.x * rows_per_pass * OS_RADIX;
  for (int x = 0; x < OS_LB_DEPTH; x++) pad[x * OS_RADIX + threadIdx.x] = OS_FLAG_INC;
}

__device__ __forceinline__ uint32_t ld_relaxed_gpu(const uint32_t *p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_gpu(uint32_t *p, uint32_t v) {
  asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Where the digit of one pass sits in the (hi = src, lo = dst) halves of a key: digit = ((lo >> a) | (hi << c)
// | (hi >> e)) & mask with PTX shift semantics (a shift count >= 32 yields 0), so that no 64-bit compaction is
// needed per key: a pass inside the dst field uses only `a`, one inside the src field only `e`, the straddling
// pass `a` and `c`.
struct DigitSel {
  uint32_t a, c, e, mask;
};
inline DigitSel make_digit_sel(int lo_bits, int shift, uint32_t mask) {
  DigitSel g;
  g.mask = mask;
  if (lo_bits >= 32) {  // no compaction: plain 64-bit key
    g.a = shift < 32 ? (uint32_t)shift : 32u;
    g.c = shift < 32 ? (uint32_t)(32 - shift) : 32u;
    g.e = shift >= 32 ? (uint32_t)(shift - 32) : 32u;
    if (shift == 0) g.c = 32u;
    return g;
  }
  if (shift >= lo_bits) {
    g.a = 32u;
    g.c = 32u;
    g.e = (uint32_t)(shift - lo_bits);
  } else {
    g.a = (uint32_t)shift;
    g.c = (uint32_t)(lo_bits - shift);  // bits of hi enter above the remaining lo bits (harmless beyond the mask)
    g.e = 32u;
  }
  return g;
}
__device__ __forceinline__ uint32_t shr_clamp(uint32_t x, uint32_t n) {
  uint32_t r;
  asm("shr.b32 %0, %1, %2;" : "=r"(r) : "r"(x), "r"(n));
  return r;
}
__device__ __forceinline__ uint32_t shl_clamp(uint32_t x, uint32_t n) {
  uint32_t r;
  asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(x), "r"(n));
  return r;
}
__device__ __forceinline__ uint32_t sel_digit(uint64_t key, const DigitSel &g) {
  const uint32_t lo = (uint32_t)key, hi = (uint32_t)(key >> 32);
  return (shr_clamp(lo, g.a) | shl_clamp(hi, g.c) | shr_clamp(hi, g.e)) & g.mask;
}

// Lanes holding the same digit.  MATCH.ANY costs one step per DISTINCT value in the warp (~30 for random 8-bit
// digits; measured: it alone made a pass issue-bound), so the peers are intersected from one ballot per digit
// bit: test-bit, VOTE, conditional NOT, AND -- four instructions per bit.
template <int B>
__device__ __forceinline__ unsigned match_bit(uint32_t d) {
  unsigned m;
  asm volatile(
      "{\n"
      " .reg .pred p;\n"
      " .reg .b32 t;\n"
      " and.b32 t, %1, %2;\n"
      " setp.ne.u32 p, t, 0;\n"
      " vote.sync.ballot.b32 %0, p, 0xffffffff;\n"
      " @!p not.b32 %0, %0;\n"
      "}\n"
      : "=r"(m)
      : "r"(d), "n"(1 << B));
  return m;
}
__device__ __forceinline__ unsigned match_digit(uint32_t d) {
  static_assert(OS_RADIX_BITS == 8, "match_digit is unrolled for 8-bit digits");
  // the eight per-bit masks are combined with three-input logic ops (4 instead of 7)
  const unsigned m0 = match_bit<0>(d), m1 = match_bit<1>(d), m2 = match_bit<2>(d), m3 = match_bit<3>(d);
  const unsigned m4 = match_bit<4>(d), m5 = match_bit<5>(d), m6 = match_bit<6>(d), m7 = match_bit<7>(d);
  return (m0 & m1 & m2) & (m3 & m4 & m5) & (m6 & m7);
}

// dynamic shared memory of k_os_pass (bytes): keys[OS_TILE] u64 | pay[OS_TILE] u32 (HAS_PAY) |
// cnt[OS_WARPS][OS_RADIX] u16 | goff[OS_RADIX] u32
inline size_t os_pass_smem(bool has_pay) {
  return (size_t)OS_TILE * 8 + (has_pay ? (size_t)OS_TILE * 4 : 0) + (size_t)OS_WARPS * OS_RADIX * 2 +
         (size_t)OS_RADIX * 4;
}

// EARLY: the tile's digit counts are taken by shared-memory atomics and published before the ranking (see below);
// !EARLY: they fall out of the ranking and are published after it -- measured faster for large batches (100 M keys:
// 0.561 -> 0.545 ms per pass), slower for small ones (12.5 M: +3 %), so the host picks by batch size.
template <bool HAS_PAY, class Src = KeyArray, bool EARLY = true>
__global__ void __launch_bounds__(OS_THREADS, 4) k_os_pass(Src src, size_t n, DigitSel sel,
                                                           const uint32_t *__restrict__ gbase,
                                                           uint32_t *__restrict__ lookback, uint32_t *tile_counter,
                                                           uint64_t *__restrict__ out_keys,
                                                           uint32_t *__restrict__ out_pay) {
  extern __shared__ __align__(16) unsigned char s_dyn[];
  uint64_t *s_keys = reinterpret_cast<uint64_t *>(s_dyn);
  uint32_t *s_pay = reinterpret_cast<uint32_t *>(s_dyn + (size_t)OS_TILE * 8);
  uint16_t *s_cnt = reinterpret_cast<uint16_t *>(s_dyn + (size_t)OS_TILE * 8 + (HAS_PAY ? (size_t)OS_TILE * 4 : 0));
  uint32_t *s_goff = reinterpret_cast<uint32_t *>(s_cnt + OS_WARPS * OS_RADIX);
  __shared__ uint32_t s_warp[33];
  __shared__ uint32_t s_tile;
  if (threadIdx.x == 0) s_tile = atomicAdd(tile_counter, 1u);
  for (uint32_t d = threadIdx.x; d < OS_WARPS * OS_RADIX / 2; d += OS_THREADS) reinterpret_cast<uint32_t *>(s_cnt)[d] = 0;
  s_goff[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t tile = s_tile;
  const unsigned w = threadIdx.x >> 5, l = lane_id(), lt = lanemask_lt();
  uint16_t *my_cnt = s_cnt + (size_t)w * OS_RADIX;
  // warp w owns the contiguous sub-tile [w*512, (w+1)*512): round r covers 32 consecutive keys (stability).
  // Keys past the end of the batch are all-ones: they carry the largest digit of every pass and, being the last
  // elements of the last tile, rank behind every real key, so they need no special case until the write-out.
  const size_t tile0 = (size_t)tile * OS_TILE;
  const size_t wbase = tile0 + (size_t)w * (32 * OS_ITEMS);
  uint64_t k[OS_ITEMS];
  uint32_t rank[OS_ITEMS / 2];  // two 16-bit ranks per register
#pragma unroll
  for (int r = 0; r < OS_ITEMS; r++) {
    const size_t i = wbase + (size_t)r * 32 + l;
    k[r] = (i < n) ? src.key(i) : ~0ull;
  }
  // early counts: the tile's digit histogram by shared-memory atomics, published BEFORE the (long) ranking phase,
  // so that by the time this tile looks back most of its predecessors have already resolved their prefix
  static_assert(OS_THREADS == OS_RADIX, "one thread per digit");
  const uint32_t dg = threadIdx.x;
  uint32_t cnt = 0;
  if (EARLY) {
#pragma unroll
    for (int r = 0; r < OS_ITEMS; r++) atomicAdd(&s_goff[sel_digit(k[r], sel)], 1u);
    __syncthreads();
    // the padding keys of a partial last tile are counted in digit `mask`; nobody looks back through the last tile
    cnt = s_goff[dg];
    st_relaxed_gpu(lookback + (size_t)tile * OS_RADIX + dg, cnt | (tile == 0 ? OS_FLAG_INC : OS_FLAG_AGG));
  }
#pragma unroll
  for (int r = 0; r < OS_ITEMS; r++) {
    const uint32_t d = sel_digit(k[r], sel);
    const unsigned peers = match_digit(d);
    const uint32_t base = my_cnt[d];
    __syncwarp();
    if ((peers & lt) == 0) my_cnt[d] = (uint16_t)(base + __popc(peers));
    __syncwarp();
    const uint32_t rk = base + __popc(peers & lt);
    if (r & 1) rank[r >> 1] |= rk << 16;
    else rank[r >> 1] = rk;
  }
  __syncthreads();
  if (!EARLY) {
#pragma unroll
    for (int ww = 0; ww < OS_WARPS; ww++) cnt += s_cnt[ww * OS_RADIX + dg];
    st_relaxed_gpu(lookback + (size_t)tile * OS_RADIX + dg, cnt | (tile == 0 ? OS_FLAG_INC : OS_FLAG_AGG));
  }
  uint32_t total;
  const uint32_t dbase = block_excl_scan(cnt, &total, s_warp);
  {  // s_cnt[w][d] := first tile-local position of warp w's keys of digit d
    uint32_t run = dbase;
#pragma unroll
    for (int ww = 0; ww < OS_WARPS; ww++) {
      const uint32_t t = s_cnt[ww * OS_RADIX + dg];
      s_cnt[ww * OS_RADIX + dg] = (uint16_t)run;
      run += t;
    }
  }
  __syncthreads();
  // reorder the tile in shared memory: position = (digit base + warp offset) + rank inside the warp
#pragma unroll
  for (int r = 0; r < OS_ITEMS; r++) {
    const uint32_t d = sel_digit(k[r], sel);
    const uint32_t rk = (r & 1) ? (rank[r >> 1] >> 16) : (rank[r >> 1] & 0xFFFFu);
    const uint32_t pos = my_cnt[d] + rk;
    s_keys[pos] = k[r];
    if (HAS_PAY) {
      const size_t i = wbase + (size_t)r * 32 + l;
      s_pay[pos] = i < n ? src.payload(i) : 0u;
    }
  }
  // decoupled look-back: sum the counts of the earlier tiles until one with an inclusive prefix is met.
  // OS_LB_DEPTH predecessors are read at once (independent loads, not one dependent L2 round trip each); the
  // OS_LB_DEPTH rows in front of tile 0 hold (INC, 0), so the walk needs no bounds checks.
  {
    uint32_t excl = 0;
    if (tile > 0) {
      const uint32_t *p = lookback + (size_t)(tile - 1) * OS_RADIX + dg;
      for (;;) {
        uint32_t v[OS_LB_DEPTH];
#pragma unroll
        for (int x = 0; x < OS_LB_DEPTH; x++) v[x] = ld_relaxed_gpu(p - x * OS_RADIX);
        bool done = false;
#pragma unroll
        for (int x = 0; x < OS_LB_DEPTH; x++) {
          while (v[x] < OS_FLAG_AGG) v[x] = ld_relaxed_gpu(p - x * OS_RADIX);
          if (!done) {
            excl += v[x] & OS_VAL_MASK;
            done = v[x] >= OS_FLAG_INC;
          }
        }
        if (done) break;
        p -= OS_LB_DEPTH * OS_RADIX;
      }
      st_relaxed_gpu(lookback + (size_t)tile * OS_RADIX + dg, (excl + cnt) | OS_FLAG_INC);
    }
    s_goff[dg] = gbase[dg] + excl - dbase;
  }
  __syncthreads();
  const uint32_t tile_n = (uint32_t)min((size_t)OS_TILE, n - tile0);
#pragma unroll 4
  for (uint32_t j = threadIdx.x; j < tile_n; j += OS_THREADS) {
    const uint64_t key = s_keys[j];
    const uint32_t pos = s_goff[sel_digit(key, sel)] + j;
    out_keys[pos] = key;
    if (HAS_PAY) out_pay[pos] = s_pay[j];
  }
}

// ---- small batches: ONE CTA, every pass inside the kernel ---------------------------------------------------------
// A batch of a few thousand keys spends its time in launch and dependency latency, not in bandwidth: the multi-kernel
// sort above needs 3 + n_pass dependent launches of ~7 us each (63 us for 1 K keys, measured).  Here the keys stay in
// registers, a pass is rank -> scatter through shared memory -> read back, and the whole sort is one launch.
// Same stable ranking as k_os_pass (warp-contiguous sub-tiles, per-bit ballots).
constexpr int SS_THREADS = 1024;
constexpr int SS_WARPS = SS_THREADS / 32;
constexpr uint32_t SS_MAX = SS_THREADS * 16;  // 16384 keys
inline size_t sort_small_smem(int items, bool has_pay) {
  return (size_t)SS_THREADS * items * (8 + (has_pay ? 4 : 0)) + (size_t)SS_WARPS * OS_RADIX * 2;
}
template <int ITEMS, bool HAS_PAY, class Src>
__global__ void __launch_bounds__(SS_THREADS, 1) k_sort_small(Src src, uint32_t n, SortPasses P,
                                                               uint64_t *__restrict__ out_keys,
                                                               uint32_t *__restrict__ out_pay) {
  extern __shared__ __align__(16) unsigned char s_dyn[];
  constexpr uint32_t TILE = SS_THREADS * ITEMS;
  uint64_t *s_keys = reinterpret_cast<uint64_t *>(s_dyn);
  uint32_t *s_pay = reinterpret_cast<uint32_t *>(s_dyn + (size_t)TILE * 8);
  uint16_t *s_cnt = reinterpret_cast<uint16_t *>(s_dyn + (size_t)TILE * (8 + (HAS_PAY ? 4 : 0)));
  __shared__ uint32_t s_warp[33];
  const unsigned w = threadIdx.x >> 5, l = lane_id(), lt = lanemask_lt();
  uint16_t *my_cnt = s_cnt + (size_t)w * OS_RADIX;
  const uint32_t wbase = w * (32 * ITEMS);
  uint64_t k[ITEMS];
  uint32_t v[ITEMS];
#pragma unroll
  for (int r = 0; r < ITEMS; r++) {
    const uint32_t i = wbase + r * 32 + l;
    k[r] = i < n ? src.key(i) : ~0ull;  // padding carries the largest digit of every pass and sits behind every real key
    v[r] = (HAS_PAY && i < n) ? src.payload(i) : 0u;
  }
  for (int p = 0; p < P.n_pass; p++) {
    const int shift = P.shift[p];
    const uint32_t mask = P.mask[p];
    for (uint32_t d = threadIdx.x; d < SS_WARPS * OS_RADIX / 2; d += SS_THREADS) reinterpret_cast<uint32_t *>(s_cnt)[d] = 0;
    __syncthreads();
    uint32_t rank[ITEMS];
#pragma unroll
    for (int r = 0; r < ITEMS; r++) {
      const uint32_t d = sort_digit(k[r], P.lo_bits, shift, mask);
      const unsigned peers = match_digit(d);
      const uint32_t base = my_cnt[d];
      __syncwarp();
      if ((peers & lt) == 0) my_cnt[d] = (uint16_t)(base + __popc(peers));
      __syncwarp();
      rank[r] = base + __popc(peers & lt);
    }
    __syncthreads();
    uint32_t tot = 0;  // thread t < 256: keys of digit t in the tile
    if (threadIdx.x < OS_RADIX)
      for (int ww = 0; ww < SS_WARPS; ww++) tot += s_cnt[ww * OS_RADIX + threadIdx.x];
    uint32_t all;
    uint32_t run = block_excl_scan(tot, &all, s_warp);
    if (threadIdx.x < OS_RADIX) {  // s_cnt[w][d] := first position of warp w's keys of digit d
      for (int ww = 0; ww < SS_WARPS; ww++) {
        const uint32_t t = s_cnt[ww * OS_RADIX + threadIdx.x];
        s_cnt[ww * OS_RADIX + threadIdx.x] = (uint16_t)run;
        run += t;
      }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < ITEMS; r++) {
      const uint32_t pos = my_cnt[sort_digit(k[r], P.lo_bits, shift, mask)] + rank[r];
      s_keys[pos] = k[r];
      if (HAS_PAY) s_pay[pos] = v[r];
    }
    __syncthreads();
    if (p + 1 < P.n_pass) {
#pragma unroll
      for (int r = 0; r < ITEMS; r++) {
        const uint32_t i = wbase + r * 32 + l;
        k[r] = s_keys[i];
        if (HAS_PAY) v[r] = s_pay[i];
      }
      __syncthreads();
    }
  }
  for (uint32_t i = threadIdx.x; i < n; i += SS_THREADS) {
    out_keys[i] = s_keys[i];
    if (HAS_PAY) out_pay[i] = s_pay[i];
  }
}

template <int ITEMS, bool HAS_PAY, class Src>
inline int launch_sort_small(ppcsr_shard *s, const Src &src, uint32_t n, const SortPasses &P, uint64_t *kb,
                             uint32_t *pb) {
  static std::once_flag once[64];
  static cudaError_t once_err[64];
  const int dv = s->device & 63;
  std::call_once(once[dv], [&] {
    once_err[dv] = cudaFuncSetAttribute(k_sort_small<ITEMS, HAS_PAY, Src>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)sort_small_smem(ITEMS, HAS_PAY));
  });
  CUDA_TRY(once_err[dv]);
  k_sort_small<ITEMS, HAS_PAY, Src><<<1, SS_THREADS, sort_small_smem(ITEMS, HAS_PAY), s->stream>>>(src, n, P, kb, pb);
  return PPCSR_OK;
}
template <bool HAS_PAY, class Src>
inline int sort_small_dispatch(ppcsr_shard *s, const Src &src, uint32_t n, const SortPasses &P, uint64_t *kb,
                               uint32_t *pb) {
  if (n <= SS_THREADS) return launch_sort_small<1, HAS_PAY, Src>(s, src, n, P, kb, pb);
  if (n <= SS_THREADS * 4) return launch_sort_small<4, HAS_PAY, Src>(s, src, n, P, kb, pb);
  return launch_sort_small<16, HAS_PAY, Src>(s, src, n, P, kb, pb);
}

// scratch (u32 words) the sort needs in s->hist for `n` keys
inline size_t radix_sort_scratch_words(size_t n) {
  const size_t ntiles = (n + OS_TILE - 1) / OS_TILE;
  return (size_t)OS_MAX_PASSES * OS_RADIX + 64 + (size_t)OS_MAX_PASSES * (ntiles + OS_LB_DEPTH) * OS_RADIX;
}

// scratch layout in s->hist: ghist[8][256] | tile counters[64] | lookback[n_pass][OS_LB_DEPTH + ntiles][256]
inline size_t radix_sort_words(size_t n, int n_pass) {
  const size_t ntiles = (n + OS_TILE - 1) / OS_TILE;
  return (size_t)OS_MAX_PASSES * OS_RADIX + 64 + (size_t)n_pass * (ntiles + OS_LB_DEPTH) * OS_RADIX;
}
// Reserves and clears the scratch of a sort of up to n keys in P.n_pass passes.  Called BEFORE the key builder when the
// builder takes the histograms itself (see batch::HistArgs); *ghist = where they go.
inline int radix_sort_prepare(ppcsr_shard *s, size_t n, const SortPasses &P, uint32_t **ghist) {
  const size_t words = radix_sort_words(n, P.n_pass);
  PPCSR_TRY(dev_reserve(s->hist, words, s->stream));
  CUDA_TRY(cudaMemsetAsync(s->hist.p, 0, words * sizeof(uint32_t), s->stream));
  *ghist = s->hist.p;
  return PPCSR_OK;
}

// Sorts n (key,payload) pairs by the key bits [0,lo_bits) and [32, 32+hi_bits).  The keys (and payloads) are the
// arrays ka / pa; ka / kb (pa / pb) are the two buffer pairs the passes alternate between.  The sorted result ends up in
// *rk / *rp, which point at either pair.  pa == nullptr sorts keys only.
// hist_done: the scratch was prepared (radix_sort_prepare, for at least n keys and this layout) and already holds the
// digit histograms of this layout: no clearing, no k_os_hist.
inline int radix_sort_pairs(ppcsr_shard *s, uint64_t *ka, uint32_t *pa, uint64_t *kb, uint32_t *pb, size_t n,
                            int lo_bits, int hi_bits, uint64_t **rk, uint32_t **rp, bool hist_done = false) {
  const bool has_pay = pa != nullptr;
  const KeyArray src{ka, pa};
  *rk = ka;
  *rp = has_pay ? pa : nullptr;
  if (n == 0) return PPCSR_OK;
  if (n > OS_MAX_COUNT) {
    g_ppcsr_error = "batch too large for one sort (>= 2^30 updates); split it";
    return PPCSR_ERR_ARG;
  }
  const SortPasses P = make_sort_passes(lo_bits, hi_bits);
  if (n <= SS_MAX) {  // one CTA, one launch
    s->launches += 1;
    const uint32_t m = (uint32_t)n;
    PPCSR_TRY(has_pay ? (sort_small_dispatch<true, KeyArray>(s, src, m, P, kb, pb))
                      : (sort_small_dispatch<false, KeyArray>(s, src, m, P, kb, pb)));
    CUDA_TRY(cudaGetLastError());
    *rk = kb;
    *rp = has_pay ? pb : nullptr;
    return PPCSR_OK;
  }
  const size_t ntiles = (n + OS_TILE - 1) / OS_TILE;
  const size_t rows = ntiles + OS_LB_DEPTH;
  if (!hist_done) {
    uint32_t *g;
    PPCSR_TRY(radix_sort_prepare(s, n, P, &g));
  }
  uint32_t *ghist = s->hist.p;
  uint32_t *counters = ghist + OS_MAX_PASSES * OS_RADIX;
  uint32_t *lookback = counters + 64;
  {  // > 48 KB of dynamic shared memory needs an explicit opt-in: per device, once, thread-safe
    static std::once_flag once[64];
    static cudaError_t once_err[64];
    const int dv = s->device & 63;
    std::call_once(once[dv], [&] {
      once_err[dv] = cudaFuncSetAttribute(k_os_pass<true, KeyArray>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)os_pass_smem(true));
      if (once_err[dv] == cudaSuccess)
        once_err[dv] = cudaFuncSetAttribute(k_os_pass<false, KeyArray>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)os_pass_smem(false));
      if (once_err[dv] == cudaSuccess)
        once_err[dv] = cudaFuncSetAttribute(k_os_pass<false, KeyArray, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)os_pass_smem(false));
    });
    CUDA_TRY(once_err[dv]);
  }
  s->launches += 1 + P.n_pass;
  if (!hist_done) {
    const unsigned hblocks = (unsigned)std::min<size_t>((n + (size_t)OSH_THREADS * OSH_ITEMS - 1) / ((size_t)OSH_THREADS * OSH_ITEMS), 148 * 4);
    s->launches += 1;
    k_os_hist<KeyArray><<<hblocks, OSH_THREADS, 0, s->stream>>>(src, n, P, ghist);
  }
  k_os_scan<<<P.n_pass, OS_RADIX, 0, s->stream>>>(ghist, lookback, rows);
  const bool late_counts = n >= OS_LATE_MIN_KEYS;  // keys-only passes of a large batch publish their counts after the ranking
  // the passes alternate between the two buffer pairs; pass 0 publishes its counts early whatever the batch size
  uint64_t *src_k = ka, *dst_k = kb;
  uint32_t *src_p = pa, *dst_p = pb;
  for (int p = 0; p < P.n_pass; p++) {
    const DigitSel sel = make_digit_sel(lo_bits, P.shift[p], P.mask[p]);
    uint32_t *gb = ghist + p * OS_RADIX, *lb = lookback + ((size_t)p * rows + OS_LB_DEPTH) * OS_RADIX;
    const KeyArray a{src_k, src_p};
    if (has_pay) k_os_pass<true, KeyArray><<<(unsigned)ntiles, OS_THREADS, os_pass_smem(true), s->stream>>>(a, n, sel, gb, lb, counters + p, dst_k, dst_p);
    else if (late_counts && p > 0) k_os_pass<false, KeyArray, false><<<(unsigned)ntiles, OS_THREADS, os_pass_smem(false), s->stream>>>(a, n, sel, gb, lb, counters + p, dst_k, nullptr);
    else k_os_pass<false, KeyArray><<<(unsigned)ntiles, OS_THREADS, os_pass_smem(false), s->stream>>>(a, n, sel, gb, lb, counters + p, dst_k, nullptr);
    std::swap(src_k, dst_k);
    std::swap(src_p, dst_p);
  }
  CUDA_TRY(cudaGetLastError());
  *rk = src_k;
  *rp = has_pay ? src_p : nullptr;
  return PPCSR_OK;
}

}  // namespace prim
