// common.cuh -- shard state, geometry and small device helpers shared by every stage.
//
// HBM layout of one shard (one PCSR instance, reference src/pcsr/PCSR.h:37-44 + :128):
//   dest[N], val[N]     SoA slots (8 B/slot).  Slot empty <=> val == 0 (reference PCSR.h:57-60).
//                       Sentinel of vertex v: dest = 0xFFFFFFFF, val = v + 1 (reference PCSR.cpp:64,
//                       685-697 keep the vertex id in `value`; +1 here so vertex 0 needs no special case).
//                       `src` is not stored: it is implied by the sentinel order (beg[]).
//   leaf_cnt[N/logN]    live items of each leaf.  Leaves are LEFT-PACKED: the live items of a leaf occupy
//                       its first leaf_cnt slots in key order, the rest is null.  A leaf of 32 slots is
//                       exactly one 128-B line of dest[] and one of val[].
//   tree[2*N/logN]      implicit binary tree of live counts in heap order (tree[1] = root,
//                       tree[n_leaves + l] = leaf l): get_density() of the reference (PCSR.cpp:126-133)
//                       becomes one load.
//   beg[n+1]            slot of v's sentinel = node_t::beginning; node_t::end == beg[v+1]; beg[n] = N
//                       (reference PCSR.h:18-23, fix_sentinel PCSR.cpp:168-183).
//   nn[n]               node_t::num_neighbors with the reference's call-count semantics.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>

#include "../../include/ppcsr_b200.h"

#define PPCSR_SENT 0xFFFFFFFFu
#define PPCSR_MAX_SLOTS (1ull << 31)
#define PPCSR_MIN_SLOTS 32ull

extern thread_local std::string g_ppcsr_error;

#define CUDA_TRY(expr)                                                                          \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) {                                                                    \
      char _b[512];                                                                             \
      snprintf(_b, sizeof(_b), "%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      g_ppcsr_error = _b;                                                                       \
      return PPCSR_ERR_CUDA;                                                                    \
    }                                                                                           \
  } while (0)

#define PPCSR_TRY(expr)          \
  do {                           \
    int _s = (expr);             \
    if (_s != PPCSR_OK) return _s; \
  } while (0)

// ---------------------------------------------------------------------------------------------
// geometry: reference src/pcsr/PCSR.cpp:22-33 (bsr) and :68-73 (resizeEdgeArray)
// ---------------------------------------------------------------------------------------------
__host__ __device__ inline int ppcsr_bsr(uint64_t w) {
  int r = 0;
  while (w >>= 1) r++;
  return r;
}

struct Geometry {
  uint64_t N;
  uint32_t logN;        // leaf size (slots)
  uint32_t leaf_shift;  // log2(logN)
  uint32_t H;           // tree height: leaves at depth H
  uint32_t n_leaves;    // N / logN == 1 << H
};

inline Geometry make_geometry(uint64_t N) {
  Geometry g;
  g.N = N;
  g.leaf_shift = (uint32_t)ppcsr_bsr((uint64_t)ppcsr_bsr(N) * 2 + 1);
  g.logN = 1u << g.leaf_shift;
  g.H = (uint32_t)ppcsr_bsr(N / g.logN);
  g.n_leaves = (uint32_t)(N / g.logN);
  return g;
}

// reference PCSR::PCSR, src/pcsr/PCSR.cpp:777
inline uint64_t initial_slots(uint32_t init_n, uint32_t src_n) {
  uint64_t m = (uint64_t)init_n + (uint64_t)src_n;
  if (m < 1024) m = 1024;
  return 2ull << ppcsr_bsr(m);
}

// density bounds, reference src/pcsr/PCSR.cpp:156-165; same double expressions so that the comparisons
// `density >= upper` (PCSR.cpp:578,1028) and `density < lower` (PCSR.cpp:616,1197) round identically.
// H == 0 (N == logN) would divide by zero in the reference; the root bounds are used instead.
__host__ __device__ inline double bound_upper(int depth, int H) {
  return H > 0 ? 3.0 / 4.0 + ((.25 * depth) / H) : 0.75;
}
__host__ __device__ inline double bound_lower(int depth, int H) {
  return H > 0 ? 1.0 / 4.0 - ((0.125 * depth) / H) : 0.25;
}

// A window of `len` slots (m leaves of `logN` slots) holding `cnt` items is acceptable for an insert iff
// its density is below the reference's upper bound AND spreading it evenly leaves no leaf 100 % full
// (cnt <= m * (logN-1)); the second clause is the batch form of the reference's "leaf completely
// full -> rewrite the parent" rule (PCSR.cpp:555-560) and is strictly tighter (SURVEY §8a I4).
__host__ __device__ inline bool window_ok_upper(uint64_t cnt, uint64_t len, uint32_t logN, int depth, int H) {
  const double dens = (double)cnt / (double)len;
  if (dens >= bound_upper(depth, H)) return false;
  return cnt <= (len / logN) * (uint64_t)(logN - 1);
}
__host__ __device__ inline bool window_ok_lower(uint64_t cnt, uint64_t len, int depth, int H) {
  const double dens = (double)cnt / (double)len;
  return !(dens < bound_lower(depth, H));
}

// ---------------------------------------------------------------------------------------------
// shard state
// ---------------------------------------------------------------------------------------------
template <typename T>
struct DevBuf {
  T *p = nullptr;
  size_t cap = 0;  // elements
};

struct Snapshot {
  bool valid = false;
  Geometry geo{};
  uint32_t n = 0;
  uint64_t items = 0;
  DevBuf<uint32_t> dest, val, leaf_cnt, tree, beg, nn;
};

// Device-side scalars of one batch, read back in two small copies.
struct BatchScalars {
  unsigned long long n_ignored;
  unsigned long long n_unique;
  unsigned long long n_inserted;
  unsigned long long n_overwritten;
  unsigned long long n_deleted;
  unsigned long long n_not_found;
  unsigned long long n_touched;
  unsigned long long n_windows;
  unsigned long long n_chunks;
  unsigned long long window_slots;
  unsigned long long window_sentinels;
  unsigned long long multi_slots;   // slots in windows that need more than one CTA (copy-back path)
  unsigned long long n_small;       // windows handled one per warp
  unsigned int dst_or;              // OR of all dst (sort width)
  unsigned int root_violation;      // bit0: root above upper bound, bit1: root below lower bound
  unsigned int val_max;             // largest per-update value of the batch (0: none non-zero)
  unsigned int val_inv_min;         // ~(smallest non-zero value)
  unsigned long long n_touched_est;  // leaves that received inserts + leaves that lost items (k_locate's tally)
  unsigned long long seg_total;      // batch size when it is only known on the device (records deposited by peers)
  unsigned int sparse_abort;         // small-batch path: a dst is wider than the speculated sort width -- nothing was modified
  unsigned int sparse_done;          // small-batch path: every window was small, the batch is complete
  unsigned int sp_blocks_done;       // small-batch path: CTAs of k_sp_tree that have finished (the last one sums the top)
  unsigned int pad0;
};
static_assert(sizeof(BatchScalars) % 8 == 0, "BatchScalars must stay 8-byte sized");

struct WindowDesc {
  uint32_t node;        // heap index of the tree node
  uint32_t leaf0;       // first leaf (source == destination geometry unless resizing)
  uint32_t m;           // leaves in the window
  uint32_t items;       // live items after the batch
  uint32_t chunk0;      // first chunk id (exclusive scan of chunk counts)
  uint32_t n_chunks;
};

namespace reb {
struct ChunkPlanM;  // one entry per chunk of the chunked rebalance (rebalance_m.cuh)
}

struct ppcsr_shard {
  int device = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  Geometry geo{};
  uint32_t n = 0;        // vertices
  uint64_t items = 0;    // live slots (edges + sentinels), host mirror of tree[1]
  uint32_t epoch = 0;    // batch counter, stamps `mark`
  uint32_t launches = 0; // kernels launched since the current batch started

  DevBuf<uint32_t> dest, val;          // [N]
  DevBuf<uint32_t> dest_alt, val_alt;  // out-of-place target (resize / multi-CTA windows)
  DevBuf<uint32_t> leaf_cnt;           // [n_leaves]
  DevBuf<uint32_t> tree;               // [2*n_leaves]
  DevBuf<uint32_t> beg;                // [n+1]
  DevBuf<uint32_t> nn;                 // [n]

  // per-batch leaf-granular scratch
  DevBuf<uint32_t> ins_cnt, del_cnt;   // [n_leaves]
  DevBuf<uint32_t> rank_off;           // [n_leaves+1] exclusive scan of the post-batch leaf counts
  DevBuf<uint32_t> ins_off;            // [n_leaves+1] exclusive scan of ins_cnt
  DevBuf<uint32_t> mark;               // [2*n_leaves] epoch stamps of chosen windows
  DevBuf<uint32_t> touched;            // [n_leaves] compact list of touched leaves
  DevBuf<uint32_t> touched_win;        // [n_leaves] window node of each touched leaf
  DevBuf<WindowDesc> windows;          // [n_leaves]
  DevBuf<uint32_t> win_chunk_off;      // [n_leaves+1]
  DevBuf<reb::ChunkPlanM> plan;        // [n_chunks]
  bool ins_sentinels = false;          // the pending insert list holds sentinels (ppcsr_add_nodes)
  uint32_t ins_uniform_val = 0;        // != 0: the pending insert list has no value array, every insert carries this
  uint32_t all_touched = 0;            // invariant checker: bit 2 = the last batch rewrote every leaf (bit 0 inserts, bit 1 deletes)
  int whole_policy = 0;                // -1 never / 0 cost model / 1 always: one root window instead of a window list
  // small-batch path (sparse.cuh)
  DevBuf<uint32_t> touch_stamp;        // [n_leaves] epoch of the last batch that touched the leaf
  DevBuf<uint32_t> touched_flags;      // [touched] bit 0 inserts, bit 1 deletes (for the invariant checker)
  uint32_t touch_epoch = 0;
  bool cnt_clean = false;              // ins_cnt / del_cnt are all zero (left so by a sparse batch)
  bool last_sparse = false;            // the last batch took the small-batch path: `touched` lists its leaves
  uint32_t last_touched = 0;
  uint32_t dst_or_seen = 0;            // OR of every dst of every batch so far (speculated sort width of small batches)
  int sparse_policy = 0;               // -1 never, 0 automatic (PPCSR_SPARSE=never|always overrides)
  bool poisoned = false;               // a batch failed after it had begun to modify the shard (capi.cu: reserve_worst_case)

  // per-batch update-granular scratch
  DevBuf<uint64_t> key_a, key_b;       // [batch]
  DevBuf<uint32_t> pay_a, pay_b;       // [batch]
  DevBuf<uint32_t> in_src, in_dst, in_val;  // staging of host batches
  // pipelined host submit (ppcsr_submit_batch / ppcsr_wait): two staging slots filled on a copy stream while the
  // previous batch computes
  struct Pending {
    DevBuf<uint32_t> src, dst, val;
    uint64_t count = 0, ticket = 0;
    uint32_t default_val = 1;
    bool has_val = false, busy = false;
    cudaEvent_t copied = nullptr;
  } pending[2];
  cudaStream_t copy_stream = nullptr;
  uint64_t next_ticket = 1;
  DevBuf<uint64_t> ukey;               // [batch] unique keys (last op wins)
  DevBuf<uint32_t> uval;               // [batch]
  DevBuf<uint32_t> uloc;               // [batch, whole tiles] predecessor slots of the locate tiles' inserts
  DevBuf<uint32_t> tile_cnt;           // [tiles + 1] inserts per locate tile -> exclusive scan
  DevBuf<uint8_t> ucls;                // [batch] class
  DevBuf<uint8_t> ufirst;              // [batch] first op of the key in this batch is a remove
  DevBuf<uint32_t> ins_dst, ins_val, ins_pred;  // [batch] compacted pure inserts, key order
  DevBuf<uint32_t> block_tmp;          // scan/sort block scratch
  DevBuf<unsigned long long> scan_state;   // look-back words of the single-pass scan, epoch-tagged (primitives.cuh)
  DevBuf<unsigned long long> scan_ticket;  // [1] tile ticket counter of the scans (monotonic)
  unsigned long long scan_ticket_base = 0; // first ticket of the next scan
  uint32_t scan_epoch = 0;                 // scans issued since scan_state was last cleared
  DevBuf<uint32_t> hist;               // radix histograms
  DevBuf<double> pr_acc;               // pagerank fp64 accumulator
  DevBuf<uint32_t> misc;               // misc query scratch
  // change capture (ppcsr_set_change_capture): allocated only while it is on
  bool capture = false;
  DevBuf<uint8_t> cap_kind;            // [batch] per sorted update: class of a winner | misses << 2 (batch::k_locate_capture)
  DevBuf<uint32_t> cap_old;            // [batch] per sorted update: value an overwrite or delete replaced
  DevBuf<uint32_t> chg_src, chg_dst, chg_old, chg_new;  // [batch] the last batch's changes, key order
  DevBuf<uint32_t> nf_src, nf_dst;     // [batch] the last batch's removes that missed, key order
  uint64_t n_changes = 0, n_nf = 0;    // their lengths; 0 after anything but a successful batch

  BatchScalars *d_scalars = nullptr;   // device
  BatchScalars *h_scalars = nullptr;   // pinned host
  void *h_pinned = nullptr;            // pinned staging for small D2H/H2D
  size_t h_pinned_bytes = 0;

  cudaEvent_t ev[8] = {};  // 0 start, 1 sorted, 2 located, 3 selected, 4 done, 5/6 around the rebalance kernels
  ppcsr_batch_stats last{};
  Snapshot snap;
};

// Every device array comes from dev_reserve and ends with at least DEV_PAD_ELEMS elements beyond the requested count.
// The bulk (TMA) loads of reb::k_rebalance_m round their length up to 16 bytes and may READ up to 3 elements past the
// logical end of rank_off / ins_off / ins_pred / ins_dst / ins_val (rebalance_m.cuh: issue_round): the pad is what makes
// that legal, whatever size the caller asked for.
constexpr size_t DEV_PAD_ELEMS = 64;
static_assert(DEV_PAD_ELEMS >= 4, "the rebalance kernel's 16-byte bulk loads over-read by up to 3 elements");
template <typename T>
inline int dev_reserve(DevBuf<T> &b, size_t elems, cudaStream_t stream, bool keep = false) {
  if (elems <= b.cap) return PPCSR_OK;
  // slack so slowly growing batches do not realloc every time; b.cap counts the usable elements, the pad lies beyond
  const size_t cap_new = elems + elems / 8;
  const size_t want = cap_new + DEV_PAD_ELEMS;
  static const bool log_alloc = getenv("PPCSR_LOG_ALLOC") != nullptr;  // development aid: who allocates mid-run?
  if (log_alloc) fprintf(stderr, "[ppcsr] dev_reserve: %zu -> %zu elements of %zu bytes\n", b.cap, want, sizeof(T));
  T *np_ = nullptr;
  cudaError_t e = cudaMalloc((void **)&np_, want * sizeof(T));
  if (e != cudaSuccess) {
    char m[256];
    snprintf(m, sizeof(m), "cudaMalloc(%zu bytes) failed: %s", want * sizeof(T), cudaGetErrorString(e));
    g_ppcsr_error = m;
    cudaGetLastError();
    return PPCSR_ERR_CAPACITY;
  }
  if (keep && b.p && b.cap) {
    e = cudaMemcpyAsync(np_, b.p, b.cap * sizeof(T), cudaMemcpyDeviceToDevice, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) {  // do not leak the new block
      cudaFree(np_);
      g_ppcsr_error = std::string("dev_reserve: copy into the grown buffer failed: ") + cudaGetErrorString(e);
      return PPCSR_ERR_CUDA;
    }
  }
  if (b.p) {
    CUDA_TRY(cudaStreamSynchronize(stream));
    CUDA_TRY(cudaFree(b.p));
  }
  b.p = np_;
  b.cap = cap_new;
  return PPCSR_OK;
}

template <typename T>
inline void dev_free(DevBuf<T> &b) {
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
}

static inline unsigned int div_up(uint64_t a, uint64_t b) { return (unsigned int)((a + b - 1) / b); }

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }
__device__ __forceinline__ unsigned lanemask_lt() {
  unsigned m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

// floor(o * j / m) in 64-bit: first rank stored in output leaf o when j items are spread over m leaves.
// This is the batch form of the reference's `index + k*len/j` spreading (PCSR.cpp:237-247): leaf o
// receives ranks [rank_begin(o), rank_begin(o+1)), i.e. floor or ceil of j/m items.
__host__ __device__ __forceinline__ uint64_t rank_begin(uint64_t o, uint64_t j, uint64_t m) { return (o * j) / m; }
