// capi.cu -- C-ABI (include/ppcsr_b200.h) and host orchestration of the batch pipeline.
// Unity build: all kernels are included here and compiled for sm_100a only.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "batch.cuh"
#include "common.cuh"
#include "migrate.cuh"
#include "parse.cuh"
#include "primitives.cuh"
#include "queries.cuh"
#include "rebalance.cuh"
#include "rebalance_m.cuh"
#include "sort.cuh"
#include "sparse.cuh"
#include "traverse.cuh"
#include "windows.cuh"

thread_local std::string g_ppcsr_error;

namespace {

constexpr uint64_t SPARSE_MAX_BATCH = 1ull << 17;  // largest batch the small-batch path (sparse.cuh) takes


int bits_of(uint64_t x) { return x == 0 ? 0 : ppcsr_bsr(x) + 1; }

int set_device(ppcsr_shard *s) {
  CUDA_TRY(cudaSetDevice(s->device));
  return PPCSR_OK;
}

// (re)allocate every leaf-granular array for geometry g; contents undefined afterwards except mark (zeroed)
int reserve_leaf_arrays(ppcsr_shard *s, const Geometry &g) {
  const size_t L = g.n_leaves;
  const uint32_t *old_ins = s->ins_cnt.p, *old_del = s->del_cnt.p;
  PPCSR_TRY(dev_reserve(s->ins_cnt, L, s->stream));
  PPCSR_TRY(dev_reserve(s->del_cnt, L, s->stream));
  if (s->ins_cnt.p != old_ins || s->del_cnt.p != old_del) s->cnt_clean = false;  // fresh counters are not clear
  PPCSR_TRY(dev_reserve(s->rank_off, L + 1, s->stream));
  PPCSR_TRY(dev_reserve(s->ins_off, L + 1, s->stream));
  const size_t old_stamp = s->touch_stamp.cap;
  PPCSR_TRY(dev_reserve(s->touch_stamp, L, s->stream));
  if (s->touch_stamp.cap != old_stamp) {
    CUDA_TRY(cudaMemsetAsync(s->touch_stamp.p, 0, s->touch_stamp.cap * sizeof(uint32_t), s->stream));
    s->touch_epoch = 0;
  }
  const size_t old_mark = s->mark.cap;
  PPCSR_TRY(dev_reserve(s->mark, 2 * L, s->stream));
  if (s->mark.cap != old_mark) {
    CUDA_TRY(cudaMemsetAsync(s->mark.p, 0, s->mark.cap * sizeof(uint32_t), s->stream));
    s->epoch = 0;
  }
  return PPCSR_OK;
}

int reserve_batch_arrays(ppcsr_shard *s, size_t count) {
  // the key buffers double as the locate tiles' scratch list (whole tiles): room for one more tile
  PPCSR_TRY(dev_reserve(s->key_a, count + batch::LTILE, s->stream));
  PPCSR_TRY(dev_reserve(s->key_b, count + batch::LTILE, s->stream));
  PPCSR_TRY(dev_reserve(s->pay_a, count, s->stream));
  PPCSR_TRY(dev_reserve(s->pay_b, count, s->stream));
  PPCSR_TRY(dev_reserve(s->ins_dst, count, s->stream));
  PPCSR_TRY(dev_reserve(s->ins_val, count, s->stream));
  PPCSR_TRY(dev_reserve(s->ins_pred, count, s->stream));
  return PPCSR_OK;
}

int reserve_window_arrays(ppcsr_shard *s, size_t count) {
  const size_t cap = std::min<size_t>(s->geo.n_leaves, count) + 1;
  PPCSR_TRY(dev_reserve(s->touched, cap, s->stream));
  PPCSR_TRY(dev_reserve(s->touched_win, cap, s->stream));
  PPCSR_TRY(dev_reserve(s->windows, cap, s->stream));
  return PPCSR_OK;
}

int read_scalars(ppcsr_shard *s) {
  CUDA_TRY(cudaMemcpyAsync(s->h_scalars, s->d_scalars, sizeof(BatchScalars), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return PPCSR_OK;
}

// Lays out `n` sentinels evenly over geometry s->geo (constructor / empty-graph add_node).
int init_layout(ppcsr_shard *s) {
  const Geometry &g = s->geo;
  CUDA_TRY(cudaMemsetAsync(s->dest.p, 0, g.N * sizeof(uint32_t), s->stream));
  CUDA_TRY(cudaMemsetAsync(s->val.p, 0, g.N * sizeof(uint32_t), s->stream));
  CUDA_TRY(cudaMemsetAsync(s->leaf_cnt.p, 0, (size_t)g.n_leaves * sizeof(uint32_t), s->stream));
  CUDA_TRY(cudaMemsetAsync(s->tree.p, 0, (size_t)2 * g.n_leaves * sizeof(uint32_t), s->stream));
  if (s->n) {
    reb::k_init_sentinels<<<div_up(s->n, 256), 256, 0, s->stream>>>(s->dest.p, s->val.p, s->beg.p, 0, s->n, s->n,
                                                                   g.n_leaves, g.leaf_shift);
    reb::k_init_leaf_counts<<<div_up(g.n_leaves, 256), 256, 0, s->stream>>>(s->leaf_cnt.p, s->tree.p, s->n,
                                                                            g.n_leaves);
    CUDA_TRY(cudaMemsetAsync(s->nn.p, 0, (size_t)s->n * sizeof(uint32_t), s->stream));
  }
  reb::k_set_u32<<<1, 1, 0, s->stream>>>(s->beg.p + s->n, (uint32_t)g.N);
  PPCSR_TRY(win::tree_rebuild(s, s->tree.p, g.H));
  CUDA_TRY(cudaMemsetAsync(s->ins_cnt.p, 0, (size_t)g.n_leaves * sizeof(uint32_t), s->stream));
  CUDA_TRY(cudaMemsetAsync(s->del_cnt.p, 0, (size_t)g.n_leaves * sizeof(uint32_t), s->stream));
  CUDA_TRY(cudaGetLastError());
  s->items = s->n;
  return PPCSR_OK;
}

int alloc_geometry(ppcsr_shard *s, const Geometry &g) {
  PPCSR_TRY(dev_reserve(s->dest, g.N, s->stream));
  PPCSR_TRY(dev_reserve(s->val, g.N, s->stream));
  PPCSR_TRY(dev_reserve(s->leaf_cnt, g.n_leaves, s->stream));
  PPCSR_TRY(dev_reserve(s->tree, (size_t)2 * g.n_leaves, s->stream));
  PPCSR_TRY(reserve_leaf_arrays(s, g));
  return PPCSR_OK;
}

// development knob: PPCSR_REB_PAD_SMEM=<bytes> of unused dynamic shared memory caps the resident CTAs per SM of
// k_rebalance (occupancy experiments); unset in production
// the knobs below are read once; function-local statics with an initialiser are thread-safe (PPPCSR drives its shards
// from several host threads)
uint32_t reb_prefetch_dist() {  // development knob: PPCSR_REB_PREFETCH=<chunks>, default one wave of resident CTAs
  static const long d = [] {
    const char *e = getenv("PPCSR_REB_PREFETCH");
    return e ? atol(e) : 148L * 4;
  }();
  return (uint32_t)d;
}
size_t reb_pad_smem() {
  static const long pad = [] {
    const char *e = getenv("PPCSR_REB_PAD_SMEM");
    const long p = e ? atol(e) : 0;
#if PPCSR_HAVE_V6
    if (p > 0) cudaFuncSetAttribute(reb::k_rebalance, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p);
#endif
    return p;
  }();
  return (size_t)pad;
}

// The default is the rank-dense persistent kernel (k_rebalance_m, rebalance_m.cuh).  PPCSR_REB_KERNEL=9 selects the
// slot-dealt persistent kernel of round 1 (k_rebalance_p), =6 the one-chunk-per-CTA kernel (k_rebalance), for A/B runs.
int reb_kernel() {
  static const int k = [] {
    const char *e = getenv("PPCSR_REB_KERNEL");
    return e ? atoi(e) : 10;
  }();
  return k;
}
bool reb_kernel_m() { return reb_kernel() != 6 && reb_kernel() != 9; }
// plan entries are 32 bytes (ChunkPlan) or 64 (ChunkPlanM): the buffer is kept in units of ChunkPlan
int reserve_plan(ppcsr_shard *s, size_t n_chunks) {
  return dev_reserve(s->plan, reb_kernel_m() ? 2 * n_chunks : n_chunks, s->stream);
}
void launch_plan(ppcsr_shard *s, const WindowDesc *windows, uint32_t n_windows, uint32_t ls_src, uint32_t ls_dst,
                 uint32_t m_dst_override, uint32_t n_chunks, uint32_t CL) {
  if (reb_kernel_m())
    reb::k_plan_chunks_m<<<div_up(n_chunks, reb::RT), reb::RT, 0, s->stream>>>(
        windows, n_windows, s->rank_off.p, s->ins_off.p, ls_src, ls_dst, m_dst_override, n_chunks, CL,
        reinterpret_cast<reb::ChunkPlanM *>(s->plan.p));
  else
    reb::k_plan_chunks<<<div_up(n_chunks, reb::RT), reb::RT, 0, s->stream>>>(
        windows, n_windows, s->rank_off.p, s->ins_off.p, ls_src, ls_dst, m_dst_override, n_chunks, CL, s->plan.p);
}
template <bool TOMB, bool UNIV>
int launch_rebalance_m(ppcsr_shard *s, unsigned n_chunks, const reb::Args &A) {
  static std::once_flag once[64];
  static int sms[64] = {0};
  static cudaError_t once_err[64];
  const int dv = s->device & 63;
  std::call_once(once[dv], [&] {
    once_err[dv] = cudaDeviceGetAttribute(&sms[dv], cudaDevAttrMultiProcessorCount, s->device);
    if (once_err[dv] == cudaSuccess)
      once_err[dv] = cudaFuncSetAttribute(reb::k_rebalance_m<TOMB, UNIV>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)sizeof(reb::MSmem<TOMB, UNIV>));
  });
  CUDA_TRY(once_err[dv]);
  static const long ctas = [] {  // development knob: resident CTAs per SM the grid is sized for
    const char *e = getenv("PPCSR_REB_GRID_CTAS");
    return e ? atol(e) : (long)PPCSR_M_CTAS;
  }();
  const unsigned grid = std::min<unsigned>(n_chunks, (unsigned)(sms[dv] * ctas));
  reb::k_rebalance_m<TOMB, UNIV><<<grid, reb::MTT, sizeof(reb::MSmem<TOMB, UNIV>), s->stream>>>(
      A, reinterpret_cast<const reb::ChunkPlanM *>(s->plan.p), n_chunks);
#ifdef PPCSR_M_TRACE
  if (const char *path = getenv("PPCSR_TRACE_OUT")) {  // development build: clock stamps of the launch just made
    static uint32_t host_trace[4 * 64 * 9 * 8];
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    CUDA_TRY(cudaMemcpyFromSymbol(host_trace, reb::g_m_trace, sizeof(host_trace)));
    if (FILE *f = fopen(path, "wb")) {
      fwrite(host_trace, 1, sizeof(host_trace), f);
      fclose(f);
    }
  }
#endif
  return PPCSR_OK;
}
// tomb: the batch wrote tombstones (it deleted edges); without, the leaves are still left-packed
int launch_rebalance(ppcsr_shard *s, unsigned n_chunks, const reb::Args &A, bool tomb) {
  if (reb_kernel_m()) {
    if (A.ins_val == nullptr)
      return tomb ? launch_rebalance_m<true, true>(s, n_chunks, A) : launch_rebalance_m<false, true>(s, n_chunks, A);
    return tomb ? launch_rebalance_m<true, false>(s, n_chunks, A) : launch_rebalance_m<false, false>(s, n_chunks, A);
  }
  if (reb_kernel() == 6) {
#if PPCSR_HAVE_V6
    reb::k_rebalance<<<n_chunks, reb::KT, reb_pad_smem(), s->stream>>>(A);
    return PPCSR_OK;
#else
    g_ppcsr_error = "this build has no one-chunk-per-CTA kernel";
    return PPCSR_ERR_ARG;
#endif
  }
  // per device, once, and thread-safe: PPPCSR drives its shards from several host threads
  static std::once_flag once[64];
  static int sms[64] = {0};
  static cudaError_t once_err[64];
  const int dv = s->device & 63;
  std::call_once(once[dv], [&] {
    once_err[dv] = cudaDeviceGetAttribute(&sms[dv], cudaDevAttrMultiProcessorCount, s->device);
    if (once_err[dv] == cudaSuccess)
      once_err[dv] = cudaFuncSetAttribute(reb::k_rebalance_p, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)sizeof(reb::PSmem));
  });
  CUDA_TRY(once_err[dv]);
  const int n_sm = sms[dv];
  static const long ctas = [] {  // development knob: resident CTAs per SM the grid is sized for
    const char *e = getenv("PPCSR_REB_GRID_CTAS");
    return e ? atol(e) : (long)PPCSR_REB_CTAS;
  }();
  const unsigned grid = std::min<unsigned>(n_chunks, (unsigned)(n_sm * ctas));
  reb::k_rebalance_p<<<grid, reb::KT, sizeof(reb::PSmem), s->stream>>>(A, n_chunks);
  return PPCSR_OK;
}

// Output leaves per chunk of a whole-array rebuild.  A chunk's source range is its share of the source leaves plus
// one or two straddled at the ends, and the kernel takes it in segments of 64 leaves: at the full 2048 output slots
// a 1:1 rebuild reads ~65 source leaves and a halving ~130, i.e. one leaf more than one resp. two segments hold, and
// pays a whole extra round for it.  Slightly smaller chunks fit the range into one segment fewer (measured: C4, 1:1,
// 60 leaves: 2.48 -> 2.32 ms; C3, halving, 56 leaves: 123 -> 118 us; the margin covers the local variation of the
// source density, larger after random deletes).  A doubling (33-34 source leaves) is best at the full size.
// PPCSR_REB_CL=<leaves> overrides (development).
uint32_t whole_array_chunk_leaves(const Geometry &g, const Geometry &g2) {
  const uint32_t cap = reb::CHUNK_SLOTS >> g2.leaf_shift;
  static const long forced = [] {
    const char *e = getenv("PPCSR_REB_CL");
    return e ? atol(e) : 0L;
  }();
  if (forced > 0) return std::max<uint32_t>(1u, std::min<uint32_t>(cap, (uint32_t)forced));
  const double seg = (double)(reb::SEG_LEAVES_SLOTS >> g.leaf_shift);
  const double src_per_out = (double)g.n_leaves / (double)g2.n_leaves;  // source leaves per output leaf
  const double margin = src_per_out > 1.0 ? 1.12 : 1.03;
  const double segments = std::ceil((cap * src_per_out * margin + 2.0) / seg);  // at the full chunk size
  if (segments > 1.0) {
    const double fewer = std::floor(((segments - 1.0) * seg - 2.0) / (src_per_out * margin));
    if (fewer >= 0.75 * cap) return std::min<uint32_t>(cap, (uint32_t)fewer);
  }
  return cap;
}

uint64_t grown_slots(uint64_t N, uint64_t items) {
  uint64_t n2 = N;
  for (;;) {
    n2 *= 2;
    if (n2 > PPCSR_MAX_SLOTS) return 0;
    Geometry g = make_geometry(n2);
    if (window_ok_upper(items, n2, g.logN, 0, (int)g.H)) return n2;
  }
}
uint64_t shrunk_slots(uint64_t N, uint64_t items) {
  uint64_t n2 = N;
  while (n2 / 2 >= PPCSR_MIN_SLOTS) {
    Geometry g = make_geometry(n2);
    if (window_ok_lower(items, n2, 0, (int)g.H)) break;
    Geometry h = make_geometry(n2 / 2);
    if (!window_ok_upper(items, n2 / 2, h.logN, 0, (int)h.H)) break;
    n2 /= 2;
  }
  return n2;
}

// Failure atomicity.  k_locate mutates the shard (values overwritten, tombstones written, num_neighbors bumped) before
// the back half of the batch knows whether the array has to grow, and growing allocates.  So everything the batch can
// need in the WORST case (every update a new edge) is reserved here, before the first mutation: the out-of-place
// target at the grown size, tree / leaf counts (contents kept), the per-leaf scratch, window list, chunk plan and the
// scan scratch.  An allocation that fails here fails the batch cleanly (PPCSR_ERR_CAPACITY, shard untouched).  The one
// case that cannot be decided up front -- the worst case would pass 2^31 slots although the real batch (duplicates,
// overwrites) may not -- reserves up to the limit; if the real batch then needs more, the handle is POISONED: it
// refuses every further update until ppcsr_restore (or ppcsr_destroy).
int reserve_worst_case(ppcsr_shard *s, uint64_t count) {
  const Geometry g = s->geo;
  const uint64_t items_worst = s->items + count;
  uint64_t need = g.N;
  if (!window_ok_upper(items_worst, g.N, g.logN, 0, (int)g.H)) {
    need = grown_slots(g.N, items_worst);
    if (need == 0) need = PPCSR_MAX_SLOTS;
  }
  const Geometry g2 = make_geometry(need);
  PPCSR_TRY(dev_reserve(s->dest_alt, g2.N, s->stream));
  PPCSR_TRY(dev_reserve(s->val_alt, g2.N, s->stream));
  PPCSR_TRY(dev_reserve(s->tree, (size_t)2 * g2.n_leaves, s->stream, true));
  PPCSR_TRY(dev_reserve(s->leaf_cnt, g2.n_leaves, s->stream, true));
  PPCSR_TRY(reserve_leaf_arrays(s, g2));
  PPCSR_TRY(reserve_window_arrays(s, count));
  const uint32_t min_cl = std::max<uint32_t>(1u, ((uint32_t)reb::CHUNK_SLOTS >> g2.leaf_shift) * 3u / 4u);
  PPCSR_TRY(reserve_plan(s, (size_t)g2.n_leaves / min_cl + 2));
  const size_t scan_tiles = (size_t)div_up(std::max<uint64_t>(std::max<uint64_t>(g2.n_leaves, count), 1), prim::SCAN_TILE) + 2;
  PPCSR_TRY(dev_reserve(s->block_tmp, scan_tiles, s->stream));
  PPCSR_TRY(prim::reserve_scan_state(s, std::max<size_t>(scan_tiles, (size_t)div_up(count, batch::LTILE) + 2)));
  return PPCSR_OK;
}
int poisoned_error() {
  g_ppcsr_error = "the handle was left inconsistent by a batch that failed after it had started to modify the shard; "
                  "ppcsr_restore a snapshot or destroy it";
  return PPCSR_ERR_CAPACITY;
}

// post-batch live count of a leaf, straight from the three per-leaf arrays
struct InNewLeafCount {
  const uint32_t *leaf_cnt, *ins_cnt, *del_cnt;
  __device__ uint32_t operator()(size_t l) const { return leaf_cnt[l] + ins_cnt[l] - del_cnt[l]; }
};

// R[] (exclusive scan of the post-batch leaf counts) and the per-leaf insert offsets feed the rebalance
int scan_rank_and_insert_offsets(ppcsr_shard *s, uint32_t L) {
  PPCSR_TRY(prim::device_scan(s, InNewLeafCount{s->leaf_cnt.p, s->ins_cnt.p, s->del_cnt.p},
                              prim::OutPrefixWithTotal{s->rank_off.p, L}, L, nullptr, nullptr));
  PPCSR_TRY(prim::device_scan(s, prim::InArray{s->ins_cnt.p}, prim::OutPrefixWithTotal{s->ins_off.p, L}, L, nullptr,
                              nullptr));
  return PPCSR_OK;
}

// One root window, possibly into a larger / smaller array: double_list / half_list (reference PCSR.cpp:251-320)
// folded into the same streaming pass.  rank_off / ins_off must be current.
int rebuild_whole_array(ppcsr_shard *s, uint64_t new_N, uint64_t items_new, const BatchScalars &h,
                        ppcsr_batch_stats *st) {
  const Geometry g = s->geo;
  const uint32_t L = g.n_leaves;
  const Geometry g2 = make_geometry(new_N);
  PPCSR_TRY(dev_reserve(s->dest_alt, g2.N, s->stream));
  PPCSR_TRY(dev_reserve(s->val_alt, g2.N, s->stream));
  PPCSR_TRY(dev_reserve(s->tree, (size_t)2 * g2.n_leaves, s->stream));
  const uint32_t CL2 = whole_array_chunk_leaves(g, g2);
  WindowDesc *hw = reinterpret_cast<WindowDesc *>(s->h_pinned);
  hw->node = 1;
  hw->leaf0 = 0;
  hw->m = L;
  hw->items = (uint32_t)items_new;
  hw->chunk0 = 0;
  hw->n_chunks = div_up(g2.n_leaves, CL2);
  PPCSR_TRY(dev_reserve(s->windows, 1, s->stream));
  CUDA_TRY(cudaMemcpyAsync(s->windows.p, hw, sizeof(WindowDesc), cudaMemcpyHostToDevice, s->stream));
  reb::Args A{};
  A.src_dest = s->dest.p;
  A.src_val = s->val.p;
  A.leaf_cnt = s->leaf_cnt.p;
  A.rank_off = s->rank_off.p;
  A.ins_off = s->ins_off.p;
  A.ins_dst = s->ins_dst.p;
  A.ins_val = s->ins_uniform_val ? nullptr : s->ins_val.p;
  A.ins_uniform = s->ins_uniform_val;
  A.ins_pred = s->ins_pred.p;
  A.out_dest_single = A.out_dest_multi = s->dest_alt.p;
  A.out_val_single = A.out_val_multi = s->val_alt.p;
  A.tree_leaf_out = s->tree.p + g2.n_leaves;
  // the persistent kernel reads no leaf counts (kept flags come from val[]), so the new counts can go straight into
  // leaf_cnt[]; sized for the new geometry before the launch (old contents are not needed any more)
  PPCSR_TRY(dev_reserve(s->leaf_cnt, g2.n_leaves, s->stream));
  A.leaf_cnt = s->leaf_cnt.p;
  A.leaf_cnt_out = reb_kernel() == 6 ? nullptr : s->leaf_cnt.p;
  A.beg = s->beg.p;
  A.windows = s->windows.p;
  A.n_windows = 1;
  A.ls_src = g.leaf_shift;
  A.ls_dst = g2.leaf_shift;
  A.m_dst_override = g2.n_leaves;
  A.prefetch_dist = reb_prefetch_dist();
  A.chunk_leaves = CL2;
  A.ins_sentinels = s->ins_sentinels ? 1u : 0u;
  PPCSR_TRY(reserve_plan(s, (size_t)hw->n_chunks));
  A.plan = s->plan.p;
  launch_plan(s, s->windows.p, 1u, g.leaf_shift, g2.leaf_shift, g2.n_leaves, hw->n_chunks, CL2);
  s->launches += 4;
  CUDA_TRY(cudaEventRecord(s->ev[5], s->stream));
  PPCSR_TRY(launch_rebalance(s, hw->n_chunks, A, h.n_deleted != 0));
  CUDA_TRY(cudaEventRecord(s->ev[6], s->stream));
  CUDA_TRY(cudaGetLastError());
  std::swap(s->dest, s->dest_alt);
  std::swap(s->val, s->val_alt);
  s->geo = g2;
  s->cnt_clean = false;
  PPCSR_TRY(reserve_leaf_arrays(s, g2));
  if (!A.leaf_cnt_out)  // the one-chunk-per-CTA kernel leaves the counts in the tree only
    reb::k_copy_u32<<<div_up(g2.n_leaves, 256), 256, 0, s->stream>>>(s->leaf_cnt.p, s->tree.p + g2.n_leaves,
                                                                    g2.n_leaves);
  PPCSR_TRY(win::tree_rebuild(s, s->tree.p, g2.H));
  reb::k_set_u32<<<1, 1, 0, s->stream>>>(s->beg.p + s->n, (uint32_t)g2.N);
  // every leaf was rewritten: for the invariant checker all of them count as touched by this batch (a flag, not two
  // fills of the per-leaf count arrays)
  s->all_touched = 4u | (h.n_inserted ? 1u : 0u) | (h.n_deleted ? 2u : 0u);
  CUDA_TRY(cudaGetLastError());
  st->n_windows = 1;
  st->whole_array = 1;
  st->window_slots = std::max<uint64_t>(g.N, g2.N);
  st->rebalance_bytes = (g.N + g2.N) * 8ull;
  st->slots_after = g2.N;
  return PPCSR_OK;
}

// Back half of a batch: s->ins_cnt / del_cnt hold the per-leaf counts, ins_{dst,val,pred} the key-ordered
// insert list, d_scalars the class counts.  Chooses windows, rebalances, refreshes tree and counts.
int finish_batch_impl(ppcsr_shard *s, size_t list_cap, ppcsr_batch_stats *st);
// any failure past this point leaves tombstones / stale counts behind: the handle is poisoned (see reserve_worst_case)
int finish_batch(ppcsr_shard *s, size_t list_cap, ppcsr_batch_stats *st) {
  const int rc = finish_batch_impl(s, list_cap, st);
  if (rc != PPCSR_OK) s->poisoned = true;
  return rc;
}
int finish_batch_impl(ppcsr_shard *s, size_t list_cap, ppcsr_batch_stats *st) {
  const Geometry g = s->geo;
  const uint32_t L = g.n_leaves;
  BatchScalars *sc = s->d_scalars;
  // The class counts decide on the host whether the ROOT leaves its density bounds (reference PCSR.cpp:578-591,
  // 616-628 reach the root => double_list / half_list): then the whole array is rebuilt and no window list is
  // needed at all.
  // R[] and the insert offsets are needed whichever way the batch goes on: their scans are queued BEFORE the host waits
  // for the class counts, so that the device has work while the round trip takes place
  PPCSR_TRY(scan_rank_and_insert_offsets(s, L));
  PPCSR_TRY(read_scalars(s));
  BatchScalars h = *s->h_scalars;
  const uint64_t items_new = s->items + h.n_inserted - h.n_deleted;
  st->n_ignored = h.n_ignored;
  st->n_unique = h.n_unique;
  st->n_inserted = h.n_inserted;
  st->n_overwritten = h.n_overwritten;
  st->n_deleted = h.n_deleted;
  st->n_not_found = h.n_not_found;
  st->slots_before = g.N;
  st->slots_after = g.N;
  const bool root_up = h.n_inserted > 0 && !window_ok_upper(items_new, g.N, g.logN, 0, (int)g.H);
  const bool root_lo = h.n_deleted > 0 && !window_ok_lower(items_new, g.N, 0, (int)g.H);

  uint64_t new_N = g.N;
  bool whole = false;
  if (root_up) {
    new_N = grown_slots(g.N, items_new);
    if (new_N == 0) {
      g_ppcsr_error = "edge array would exceed 2^31 slots";
      return PPCSR_ERR_CAPACITY;
    }
    whole = true;
    st->resized = 1;
  } else if (root_lo) {
    new_N = shrunk_slots(g.N, items_new);
    whole = true;
    st->resized = new_N != g.N ? 2 : 0;
  }
  // Policy: windows or ONE root window?  Measured on B200 at scale 20 (profiles/README.md, "Batch-size sweep";
  // window selection + rebalance stages together): the window path costs ~150 us of launches and host round trip,
  // ~0.012 us per 1000 leaves (its O(leaves) passes: post-batch counts, tree, touched list, the two offset scans)
  // and ~1.05 us per 1000 touched leaves (path walks, window list, one warp per window): 0.19 / 0.23 / 0.40 ms at
  // 10 K / 72 K / 224 K windows.  Streaming the whole array through k_rebalance_p costs ~105 us (scans, plan, tree
  // of the new array) + 16 bytes per slot at ~3.8 TB/s: 0.25 ms at 2^25 slots.  So at scale 20 the root window wins
  // from ~80 K touched leaves on (8 % of them), at scale 24 from ~1.9 M (11 %); the earlier fixed rule (a quarter
  // of the leaves) left a 1 M-update batch on the window path (0.61 ms instead of 0.47 ms).
  // ppcsr_set_whole_array_policy / PPCSR_WHOLE_ARRAY=never|always override it (the tests run every stream under
  // both paths: on small arrays the model always picks the root window).
  if (!whole && (h.n_inserted || h.n_deleted) && L >= 64) {
    static const int env_forced = [] {
      const char *e = getenv("PPCSR_WHOLE_ARRAY");
      return !e ? 0 : std::string(e) == "never" ? -1 : std::string(e) == "always" ? 1 : 0;
    }();
    const int forced = s->whole_policy ? s->whole_policy : env_forced;  // ppcsr_set_whole_array_policy wins
    const double windows_us = 150.0 + 0.012e-3 * (double)L + 1.05e-3 * (double)h.n_touched_est;
    const double whole_us = 105.0 + (double)g.N * 16.0 / 3.8e6;
    if (forced > 0 || (forced == 0 && windows_us > whole_us)) whole = true;
  }
  if (whole) {
    CUDA_TRY(cudaEventRecord(s->ev[3], s->stream));
    PPCSR_TRY(rebuild_whole_array(s, new_N, items_new, h, st));
    s->items = items_new;
    CUDA_TRY(cudaEventRecord(s->ev[4], s->stream));
    return PPCSR_OK;
  }
  if (h.n_inserted == 0 && h.n_deleted == 0) {  // overwrites / misses only: nothing moves
    for (int e = 3; e <= 6; e++) CUDA_TRY(cudaEventRecord(s->ev[e], s->stream));
    st->n_windows = 0;
    return PPCSR_OK;
  }

  PPCSR_TRY(reserve_window_arrays(s, list_cap));
  const size_t cap = std::min<size_t>(L, list_cap);
  s->launches += 2;  // leaf counts + select
  win::k_leaf_new_counts<<<div_up(L, win::WT), win::WT, 0, s->stream>>>(s->leaf_cnt.p, s->ins_cnt.p, s->del_cnt.p, L,
                                                                      s->tree.p);
  PPCSR_TRY(win::tree_rebuild(s, s->tree.p, g.H));
  PPCSR_TRY(prim::device_scan(s, win::InTouched{s->ins_cnt.p, s->del_cnt.p}, win::OutTouched{s->touched.p}, L, nullptr,
                              &sc->n_touched));
  s->epoch++;
  win::k_select<<<div_up(cap, win::WT), win::WT, 0, s->stream>>>(s->touched.p, &sc->n_touched, s->ins_cnt.p,
                                                                s->del_cnt.p, s->tree.p, L, g.logN, (int)g.H,
                                                                s->mark.p, s->epoch, sc);
  const uint32_t CL = reb::CHUNK_SLOTS >> g.leaf_shift;
  s->launches++;
  win::k_touched_windows<<<div_up(cap, win::WT), win::WT, 0, s->stream>>>(s->touched.p, &sc->n_touched, s->mark.p,
                                                                         s->epoch, L, sc, s->touched_win.p);
  PPCSR_TRY(prim::device_scan(s, prim::bounded_in(win::InWindowHead{s->touched_win.p}, &sc->n_touched),
                              prim::bounded_out(win::OutWindow{s->touched_win.p, s->tree.p, L, CL,
                                                                (uint32_t)reb::SMALL_MAX_LEAVES, g.logN, s->windows.p, sc},
                                                &sc->n_touched),
                              cap, nullptr, &sc->n_windows));
  PPCSR_TRY(prim::device_scan(s, prim::bounded_in(win::InWinChunks{s->windows.p}, &sc->n_windows),
                              prim::bounded_out(win::OutWinChunk0{s->windows.p}, &sc->n_windows), cap, nullptr,
                              &sc->n_chunks));
  CUDA_TRY(cudaEventRecord(s->ev[3], s->stream));
  PPCSR_TRY(read_scalars(s));
  h = *s->h_scalars;

  if (h.root_violation) {  // cannot happen (same predicate as above); kept as a guard
    g_ppcsr_error = "window selection and the host disagree about the root bounds";
    return PPCSR_ERR_ARG;
  }
  // a multi-CTA window is written out of place and copied back (4 moves per slot instead of 2):
  // once the windows cost as much as streaming the whole array, rebuild the whole array instead.
  if (h.n_windows > 0 && 2 * h.window_slots + 2 * h.multi_slots >= 2 * g.N) {
    PPCSR_TRY(rebuild_whole_array(s, g.N, items_new, h, st));
    s->items = items_new;
    CUDA_TRY(cudaEventRecord(s->ev[4], s->stream));
    return PPCSR_OK;
  }

  if (h.n_windows == 0) {
    st->n_windows = 0;
    CUDA_TRY(cudaEventRecord(s->ev[5], s->stream));
    CUDA_TRY(cudaEventRecord(s->ev[6], s->stream));
  } else {
    reb::Args A{};
    A.src_dest = s->dest.p;
    A.src_val = s->val.p;
    A.leaf_cnt = s->leaf_cnt.p;
    A.rank_off = s->rank_off.p;
    A.ins_off = s->ins_off.p;
    A.ins_dst = s->ins_dst.p;
    A.ins_val = s->ins_uniform_val ? nullptr : s->ins_val.p;
    A.ins_uniform = s->ins_uniform_val;
    A.ins_pred = s->ins_pred.p;
    A.out_dest_single = s->dest.p;
    A.out_val_single = s->val.p;
    if (h.multi_slots) {
      PPCSR_TRY(dev_reserve(s->dest_alt, g.N, s->stream));
      PPCSR_TRY(dev_reserve(s->val_alt, g.N, s->stream));
    }
    A.out_dest_multi = s->dest_alt.p;
    A.out_val_multi = s->val_alt.p;
    A.tree_leaf_out = s->tree.p + L;
    A.beg = s->beg.p;
    A.windows = s->windows.p;
    A.n_windows = (uint32_t)h.n_windows;
    A.ls_src = A.ls_dst = g.leaf_shift;
    A.m_dst_override = 0;
    A.prefetch_dist = reb_prefetch_dist();
    A.chunk_leaves = CL;
    A.ins_sentinels = s->ins_sentinels ? 1u : 0u;
    CUDA_TRY(cudaEventRecord(s->ev[5], s->stream));
    if (h.n_small) {
      reb::SmallArgs S{};
      S.dest = s->dest.p;
      S.val = s->val.p;
      S.leaf_cnt = s->leaf_cnt.p;
      S.rank_off = s->rank_off.p;
      S.ins_off = s->ins_off.p;
      S.ins_dst = s->ins_dst.p;
      S.ins_val = s->ins_uniform_val ? nullptr : s->ins_val.p;
      S.ins_uniform = s->ins_uniform_val;
      S.ins_pred = s->ins_pred.p;
      S.tree_leaf_out = s->tree.p + L;
      S.beg = s->beg.p;
      S.windows = s->windows.p;
      S.n_windows = (uint32_t)h.n_windows;
      S.ls = g.leaf_shift;
      s->launches++;
      // one warp per window of the list; warps that meet a chunked (large) window leave at once
      reb::k_rebalance_small<<<div_up(h.n_windows, reb::RWARPS), reb::RT, 0, s->stream>>>(S);
    }
    if (h.n_chunks) {
      PPCSR_TRY(reserve_plan(s, (size_t)h.n_chunks));
      A.plan = s->plan.p;
      launch_plan(s, s->windows.p, (uint32_t)h.n_windows, g.leaf_shift, g.leaf_shift, 0, (uint32_t)h.n_chunks, CL);
      s->launches += 2 + (h.multi_slots ? 1 : 0);
      PPCSR_TRY(launch_rebalance(s, (unsigned)h.n_chunks, A, h.n_deleted != 0));
    }
    CUDA_TRY(cudaEventRecord(s->ev[6], s->stream));
    if (h.multi_slots) {
      if (reb_kernel_m())
        reb::k_copy_back_m<<<(unsigned)h.n_chunks, reb::RT, 0, s->stream>>>(
            reinterpret_cast<const reb::ChunkPlanM *>(s->plan.p), g.leaf_shift, s->dest_alt.p, s->val_alt.p, s->dest.p,
            s->val.p);
      else
        reb::k_copy_back<<<(unsigned)h.n_chunks, reb::RT, 0, s->stream>>>(s->plan.p, g.leaf_shift, s->dest_alt.p,
                                                                          s->val_alt.p, s->dest.p, s->val.p);
    }
    s->launches += 1;
    reb::k_copy_u32<<<div_up(L, 256), 256, 0, s->stream>>>(s->leaf_cnt.p, s->tree.p + L, L);
    PPCSR_TRY(win::tree_rebuild(s, s->tree.p, g.H));
    CUDA_TRY(cudaGetLastError());
    st->n_windows = h.n_windows;
    st->window_slots = h.window_slots;
    st->rebalance_bytes = 2ull * h.window_slots * 8ull;
  }
  s->items = items_new;
  CUDA_TRY(cudaEventRecord(s->ev[4], s->stream));
  return PPCSR_OK;
}

int finalize_stats(ppcsr_shard *s, ppcsr_batch_stats *st, bool stages = true) {
  CUDA_TRY(cudaEventSynchronize(s->ev[4]));
  float t;
  CUDA_TRY(cudaEventElapsedTime(&t, s->ev[0], s->ev[4]));
  st->ms_total = t;
  if (!stages) {  // small-batch path: only the two events around the batch were recorded
    st->kernel_launches = s->launches;
    s->last = *st;
    return PPCSR_OK;
  }
  CUDA_TRY(cudaEventElapsedTime(&t, s->ev[0], s->ev[1]));
  st->ms_sort = t;
  CUDA_TRY(cudaEventElapsedTime(&t, s->ev[1], s->ev[2]));
  st->ms_locate = t;
  CUDA_TRY(cudaEventElapsedTime(&t, s->ev[2], s->ev[3]));
  st->ms_select = t;
  CUDA_TRY(cudaEventElapsedTime(&t, s->ev[3], s->ev[4]));
  st->ms_rebalance = t;
  CUDA_TRY(cudaEventElapsedTime(&t, s->ev[5], s->ev[6]));
  st->ms_rebalance_kernel = t;
  st->kernel_launches = s->launches;
  s->last = *st;
  return PPCSR_OK;
}

int refresh_rank_off(ppcsr_shard *s) {
  const uint32_t L = s->geo.n_leaves;
  return prim::device_scan(s, prim::InArray{s->leaf_cnt.p}, prim::OutPrefixWithTotal{s->rank_off.p, L}, L, nullptr,
                           nullptr);
}

__global__ void k_last_live_slot(const uint32_t *__restrict__ leaf_cnt, uint32_t n_leaves, uint32_t ls,
                                 uint32_t *out) {
  // single thread: last live slot of the array (trailing empty leaves are rare and short)
  uint32_t l = n_leaves;
  while (l > 0 && leaf_cnt[l - 1] == 0) l--;
  *out = l ? (((l - 1) << ls) + leaf_cnt[l - 1] - 1) : 0xFFFFFFFFu;
}
__global__ void k_fill_new_nodes(uint32_t *ins_dst, uint32_t *ins_val, uint32_t *ins_pred, uint32_t first_vertex,
                                 uint32_t count, const uint32_t *last_slot, uint32_t *ins_cnt, uint32_t ls,
                                 BatchScalars *sc) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) {
    ins_dst[i] = PPCSR_SENT;
    ins_val[i] = first_vertex + i + 1u;
    ins_pred[i] = *last_slot;
  }
  if (i == 0) {
    ins_cnt[*last_slot >> ls] = count;
    sc->n_inserted = count;
    sc->n_unique = count;
  }
}

// One PageRank push step over the whole shard.  Default: the leaf walk (k_pagerank_push_leaves, a coalesced stream
// over the packed array); PPCSR_PR_KERNEL=vertex selects the warp-per-vertex kernel (A/B).
template <typename W>
static void launch_pagerank_push(ppcsr_shard *s, const W *d_in, double *d_acc, uint64_t out_len) {
  static const bool per_vertex = getenv("PPCSR_PR_KERNEL") && std::string(getenv("PPCSR_PR_KERNEL")) == "vertex";
  if (per_vertex) {
    const unsigned blocks = std::min<unsigned>(div_up((uint64_t)s->n * 32, qry::QT), 148 * 16);
    qry::k_pagerank_push<W><<<blocks, qry::QT, 0, s->stream>>>(s->dest.p, s->leaf_cnt.p, s->beg.p, s->nn.p,
                                                              s->geo.leaf_shift, s->n, d_in, d_acc, out_len);
  } else {
    const unsigned blocks = std::min<unsigned>(div_up(s->geo.N, (uint64_t)qry::QT * qry::PRL_BATCH), 148 * 16);
    qry::k_pagerank_push_leaves<W><<<blocks, qry::QT, 0, s->stream>>>(s->dest.p, s->val.p, s->leaf_cnt.p, s->beg.p,
                                                                     s->nn.p, s->geo.leaf_shift, s->n, s->geo.N, d_in,
                                                                     d_acc, out_len);
  }
}

template <typename W>
static int pagerank_host(ppcsr_shard *s, const W *in, W *out, uint64_t out_len) {
  if (!s || !in || !out) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  DevBuf<W> d_in, d_out;
  PPCSR_TRY(dev_reserve(d_in, (size_t)s->n + 1, s->stream));
  PPCSR_TRY(dev_reserve(d_out, (size_t)out_len + 1, s->stream));
  PPCSR_TRY(dev_reserve(s->pr_acc, (size_t)out_len + 1, s->stream));
  CUDA_TRY(cudaMemcpyAsync(d_in.p, in, (size_t)s->n * sizeof(W), cudaMemcpyHostToDevice, s->stream));
  CUDA_TRY(cudaMemsetAsync(s->pr_acc.p, 0, (size_t)out_len * sizeof(double), s->stream));
  if (s->n) {
    launch_pagerank_push<W>(s, d_in.p, s->pr_acc.p, out_len);
  }
  if (out_len) qry::k_cast_out<W><<<div_up(out_len, 256), 256, 0, s->stream>>>(s->pr_acc.p, d_out.p, out_len);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(out, d_out.p, (size_t)out_len * sizeof(W), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  dev_free(d_in);
  dev_free(d_out);
  return PPCSR_OK;
}

template <typename T>
static int snap_copy(ppcsr_shard *s, DevBuf<T> &dst, const DevBuf<T> &src, size_t elems) {
  PPCSR_TRY(dev_reserve(dst, elems, s->stream));
  if (elems) CUDA_TRY(cudaMemcpyAsync(dst.p, src.p, elems * sizeof(T), cudaMemcpyDeviceToDevice, s->stream));
  return PPCSR_OK;
}

// ---- a shard's content as a device-resident CSR, and a shard laid out afresh from one (migrate.cuh) ------------
struct DevCsr {
  DevBuf<uint64_t> rowptr;        // [n + 1]
  DevBuf<uint32_t> col, val, nn;  // [E], [E], [n]
};
void csr_free(int device, DevCsr &c) {
  cudaSetDevice(device);
  dev_free(c.rowptr);
  dev_free(c.col);
  dev_free(c.val);
  dev_free(c.nn);
}

// The compacted adjacency of the shard into device buffers (each nullable): rowptr[n + 1], col / val [E], enqueued on
// the shard's stream.  The body of ppcsr_export_csr.
int export_device(ppcsr_shard *s, DevBuf<uint64_t> *rowptr, DevBuf<uint32_t> *col, DevBuf<uint32_t> *val) {
  const uint64_t E = s->items - s->n;
  const Geometry g = s->geo;
  if (rowptr) {
    PPCSR_TRY(refresh_rank_off(s));
    PPCSR_TRY(dev_reserve(*rowptr, (size_t)s->n + 1, s->stream));
    qry::k_rowptr<<<div_up((uint64_t)s->n + 1, qry::QT), qry::QT, 0, s->stream>>>(s->beg.p, s->rank_off.p, g.leaf_shift,
                                                                                s->n, rowptr->p);
    CUDA_TRY(cudaGetLastError());
  }
  if (col && E) {
    PPCSR_TRY(dev_reserve(*col, E, s->stream));
    if (val) PPCSR_TRY(dev_reserve(*val, E, s->stream));
    PPCSR_TRY(prim::device_scan(s, qry::InIsEdge{s->dest.p, s->leaf_cnt.p, g.leaf_shift},
                                qry::OutEdge{s->dest.p, s->val.p, col->p, val ? val->p : nullptr}, g.N, nullptr,
                                nullptr));
  }
  return PPCSR_OK;
}

// Slots of a shard laid out afresh with `items` live slots, starting from its current N: grown while the root would be
// above its upper bound, otherwise shrunk while it is below its lower bound (the rules of a batch that reaches the
// root).  0: more than 2^31 slots.
uint64_t layout_slots(uint64_t N, uint64_t items) {
  const Geometry g = make_geometry(N);
  if (!window_ok_upper(items, N, g.logN, 0, (int)g.H)) return grown_slots(N, items);
  return shrunk_slots(N, items);
}

// Every array a layout of n vertices at N slots writes, allocated before the shard is modified: the out-of-place
// target at N, and tree / leaf counts / beg / nn with their contents kept, so that a failure leaves the shard intact.
int reserve_layout(ppcsr_shard *s, uint64_t N, uint32_t n) {
  const Geometry g2 = make_geometry(N);
  PPCSR_TRY(dev_reserve(s->dest_alt, g2.N, s->stream));
  PPCSR_TRY(dev_reserve(s->val_alt, g2.N, s->stream));
  PPCSR_TRY(dev_reserve(s->tree, (size_t)2 * g2.n_leaves, s->stream, true));
  PPCSR_TRY(dev_reserve(s->leaf_cnt, g2.n_leaves, s->stream, true));
  PPCSR_TRY(dev_reserve(s->beg, (size_t)n + 1, s->stream, true));
  PPCSR_TRY(dev_reserve(s->nn, (size_t)n + 1, s->stream, true));
  PPCSR_TRY(reserve_leaf_arrays(s, g2));
  return PPCSR_OK;
}

// Replaces the shard's content with the device CSR (n vertices, E edges; d_val NULL: every value 1, d_nn NULL:
// num_neighbors = row lengths), laid out at N slots (reserve_layout first).  Enqueued only: layout_stats reads the
// timings.  Leaves the state a whole-array rebuild leaves: per-leaf counters clear, every leaf rewritten.
int commit_layout(ppcsr_shard *s, uint64_t N, uint32_t n, const uint64_t *d_rowptr, const uint32_t *d_col,
                  const uint32_t *d_val, const uint32_t *d_nn, uint64_t E, ppcsr_batch_stats *st) {
  const Geometry g = s->geo, g2 = make_geometry(N);
  *st = ppcsr_batch_stats{};
  st->slots_before = g.N;
  st->slots_after = g2.N;
  st->resized = g2.N > g.N ? 1 : g2.N < g.N ? 2 : 0;
  st->whole_array = 1;
  st->n_windows = 1;
  st->window_slots = g2.N;
  // CSR reads (col + val per edge, rowptr per vertex) + slot writes (dest + val) + beg
  st->rebalance_bytes = 8ull * E + 8ull * n + 8ull * g2.N + 4ull * n;
  s->launches = 0;
  CUDA_TRY(cudaEventRecord(s->ev[0], s->stream));
  if (n) {
    if (d_nn) CUDA_TRY(cudaMemcpyAsync(s->nn.p, d_nn, (size_t)n * 4, cudaMemcpyDeviceToDevice, s->stream));
    else mig::k_row_lengths<<<div_up(n, mig::MT), mig::MT, 0, s->stream>>>(d_rowptr, n, s->nn.p);
  }
  CUDA_TRY(cudaEventRecord(s->ev[5], s->stream));
  s->launches++;
  mig::k_layout_from_csr<<<div_up((uint64_t)g2.n_leaves * 32, mig::MT), mig::MT, 0, s->stream>>>(
      d_rowptr, d_col, d_val, 1u, n, E + n, g2.H, g2.leaf_shift, s->dest_alt.p, s->val_alt.p, s->beg.p, s->leaf_cnt.p,
      s->tree.p + g2.n_leaves);
  CUDA_TRY(cudaEventRecord(s->ev[6], s->stream));
  CUDA_TRY(cudaGetLastError());
  PPCSR_TRY(win::tree_rebuild(s, s->tree.p, g2.H));
  reb::k_set_u32<<<1, 1, 0, s->stream>>>(s->beg.p + n, (uint32_t)g2.N);
  CUDA_TRY(cudaMemsetAsync(s->ins_cnt.p, 0, (size_t)g2.n_leaves * sizeof(uint32_t), s->stream));
  CUDA_TRY(cudaMemsetAsync(s->del_cnt.p, 0, (size_t)g2.n_leaves * sizeof(uint32_t), s->stream));
  CUDA_TRY(cudaGetLastError());
  std::swap(s->dest, s->dest_alt);
  std::swap(s->val, s->val_alt);
  s->geo = g2;
  s->n = n;
  s->items = E + n;
  s->cnt_clean = true;
  s->last_sparse = false;
  s->all_touched = 4u | 1u;
  CUDA_TRY(cudaEventRecord(s->ev[4], s->stream));
  return PPCSR_OK;
}

// waits for a commit_layout and fills in its timings; the stats become the shard's ppcsr_last_stats
int layout_stats(ppcsr_shard *s, ppcsr_batch_stats *st) {
  CUDA_TRY(cudaEventSynchronize(s->ev[4]));
  CUDA_TRY(cudaEventElapsedTime(&st->ms_total, s->ev[0], s->ev[4]));
  CUDA_TRY(cudaEventElapsedTime(&st->ms_rebalance, s->ev[5], s->ev[4]));
  CUDA_TRY(cudaEventElapsedTime(&st->ms_rebalance_kernel, s->ev[5], s->ev[6]));
  st->kernel_launches = s->launches;
  s->last = *st;
  return PPCSR_OK;
}

bool submit_pending(const ppcsr_shard *s) { return s->pending[0].busy || s->pending[1].busy; }

}  // namespace

// ================================================================================================
extern "C" {

const char *ppcsr_last_error(void) { return g_ppcsr_error.c_str(); }

int ppcsr_device_count(void) {
  int c = 0;
  if (cudaGetDeviceCount(&c) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return c;
}

int ppcsr_create(uint32_t init_n, uint32_t src_n, int device, ppcsr_shard **out) {
  if (!out) return PPCSR_ERR_ARG;
  *out = nullptr;
  if (ppcsr_device_count() <= device || device < 0) {
    g_ppcsr_error = "no such CUDA device (this engine has no CPU fallback)";
    return PPCSR_ERR_NO_DEVICE;
  }
  const uint64_t N = initial_slots(init_n, src_n);
  if (N > PPCSR_MAX_SLOTS) {
    g_ppcsr_error = "initial edge array exceeds 2^31 slots";
    return PPCSR_ERR_CAPACITY;
  }
  ppcsr_shard *s = new ppcsr_shard();
  s->device = device;
  const int rc = [&]() -> int {
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking));
    s->stream = s->own_stream;
    for (auto &e : s->ev) CUDA_TRY(cudaEventCreate(&e));
    CUDA_TRY(cudaMalloc((void **)&s->d_scalars, sizeof(BatchScalars)));
    CUDA_TRY(cudaMallocHost((void **)&s->h_scalars, sizeof(BatchScalars)));
    s->h_pinned_bytes = 1 << 16;
    CUDA_TRY(cudaMallocHost(&s->h_pinned, s->h_pinned_bytes));
    s->n = src_n;
    s->geo = make_geometry(N);
    PPCSR_TRY(alloc_geometry(s, s->geo));
    PPCSR_TRY(dev_reserve(s->beg, (size_t)src_n + 1, s->stream));
    PPCSR_TRY(dev_reserve(s->nn, (size_t)src_n + 1, s->stream));
    PPCSR_TRY(init_layout(s));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return PPCSR_OK;
  }();
  if (rc != PPCSR_OK) {  // release whatever was created so far (streams, events, pinned and device buffers)
    const std::string why = g_ppcsr_error;
    ppcsr_destroy(s);
    g_ppcsr_error = why;
    return rc;
  }
  *out = s;
  return PPCSR_OK;
}

void ppcsr_destroy(ppcsr_shard *s) {
  if (!s) return;
  cudaSetDevice(s->device);
  if (s->stream) cudaStreamSynchronize(s->stream);
  dev_free(s->dest); dev_free(s->val); dev_free(s->dest_alt); dev_free(s->val_alt);
  dev_free(s->leaf_cnt); dev_free(s->tree); dev_free(s->beg); dev_free(s->nn);
  dev_free(s->ins_cnt); dev_free(s->del_cnt); dev_free(s->rank_off); dev_free(s->ins_off);
  dev_free(s->mark); dev_free(s->touched); dev_free(s->touched_win); dev_free(s->windows);
  dev_free(s->win_chunk_off); dev_free(s->plan); dev_free(s->key_a); dev_free(s->key_b); dev_free(s->pay_a); dev_free(s->pay_b);
  dev_free(s->in_src); dev_free(s->in_dst); dev_free(s->in_val); dev_free(s->ukey); dev_free(s->uval);
  dev_free(s->uloc); dev_free(s->ucls); dev_free(s->ufirst); dev_free(s->ins_dst); dev_free(s->ins_val); dev_free(s->ins_pred);
  dev_free(s->block_tmp); dev_free(s->hist); dev_free(s->pr_acc); dev_free(s->misc);
  dev_free(s->scan_state); dev_free(s->scan_ticket); dev_free(s->tile_cnt);
  dev_free(s->touch_stamp); dev_free(s->touched_flags); dev_free(s->seg_prefix);
  dev_free(s->snap.dest); dev_free(s->snap.val); dev_free(s->snap.leaf_cnt); dev_free(s->snap.tree);
  dev_free(s->snap.beg); dev_free(s->snap.nn);
  for (auto &P : s->pending) {
    dev_free(P.src); dev_free(P.dst); dev_free(P.val);
    if (P.copied) cudaEventDestroy(P.copied);
  }
  if (s->copy_stream) {
    cudaStreamSynchronize(s->copy_stream);
    cudaStreamDestroy(s->copy_stream);
  }
  if (s->d_scalars) cudaFree(s->d_scalars);
  if (s->h_scalars) cudaFreeHost(s->h_scalars);
  if (s->h_pinned) cudaFreeHost(s->h_pinned);
  for (auto &e : s->ev) if (e) cudaEventDestroy(e);
  if (s->own_stream) cudaStreamDestroy(s->own_stream);
  delete s;
}

int ppcsr_set_stream(ppcsr_shard *s, void *cuda_stream) {
  if (!s) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  s->stream = cuda_stream ? (cudaStream_t)cuda_stream : s->own_stream;
  return PPCSR_OK;
}

int ppcsr_sync(ppcsr_shard *s) {
  if (!s) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return PPCSR_OK;
}

int ppcsr_reserve(ppcsr_shard *s, uint64_t max_slots, uint64_t max_batch) {
  if (!s) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  if (max_slots > PPCSR_MAX_SLOTS) return PPCSR_ERR_CAPACITY;
  if (max_slots > s->geo.N) {
    const Geometry g = make_geometry(max_slots);
    // keep the live contents: dest/val/leaf_cnt/tree must survive a capacity bump
    PPCSR_TRY(dev_reserve(s->dest, g.N, s->stream, true));
    PPCSR_TRY(dev_reserve(s->val, g.N, s->stream, true));
    PPCSR_TRY(dev_reserve(s->dest_alt, g.N, s->stream));
    PPCSR_TRY(dev_reserve(s->val_alt, g.N, s->stream));
    PPCSR_TRY(dev_reserve(s->leaf_cnt, g.n_leaves, s->stream, true));
    PPCSR_TRY(dev_reserve(s->tree, (size_t)2 * g.n_leaves, s->stream, true));
    PPCSR_TRY(dev_reserve(s->ins_cnt, g.n_leaves, s->stream, true));
    PPCSR_TRY(dev_reserve(s->del_cnt, g.n_leaves, s->stream, true));
    PPCSR_TRY(dev_reserve(s->touch_stamp, g.n_leaves, s->stream));
    CUDA_TRY(cudaMemsetAsync(s->touch_stamp.p, 0, s->touch_stamp.cap * sizeof(uint32_t), s->stream));
    s->touch_epoch = 0;
    s->cnt_clean = false;
    PPCSR_TRY(dev_reserve(s->rank_off, (size_t)g.n_leaves + 1, s->stream));
    PPCSR_TRY(dev_reserve(s->ins_off, (size_t)g.n_leaves + 1, s->stream));
    PPCSR_TRY(dev_reserve(s->mark, (size_t)2 * g.n_leaves, s->stream));
    CUDA_TRY(cudaMemsetAsync(s->mark.p, 0, s->mark.cap * sizeof(uint32_t), s->stream));
    s->epoch = 0;
    const size_t wcap = std::min<uint64_t>(g.n_leaves, max_batch ? max_batch : g.n_leaves) + 1;
    PPCSR_TRY(dev_reserve(s->touched, wcap, s->stream));
    PPCSR_TRY(dev_reserve(s->touched_win, wcap, s->stream));
    PPCSR_TRY(dev_reserve(s->windows, wcap, s->stream));
    PPCSR_TRY(dev_reserve(s->block_tmp, (size_t)div_up(g.N, prim::SCAN_TILE) + 2, s->stream));
    PPCSR_TRY(prim::reserve_scan_state(s, (size_t)div_up(g.N, prim::SCAN_TILE) + 2));
  } else {
    PPCSR_TRY(dev_reserve(s->dest_alt, s->geo.N, s->stream));
    PPCSR_TRY(dev_reserve(s->val_alt, s->geo.N, s->stream));
  }
  if (max_batch) {
    PPCSR_TRY(reserve_batch_arrays(s, max_batch));
    PPCSR_TRY(dev_reserve(s->in_src, max_batch, s->stream));
    PPCSR_TRY(dev_reserve(s->in_dst, max_batch, s->stream));
    PPCSR_TRY(dev_reserve(s->in_val, max_batch, s->stream));
    PPCSR_TRY(dev_reserve(s->hist, prim::radix_sort_scratch_words(max_batch), s->stream));
    PPCSR_TRY(dev_reserve(s->block_tmp, (size_t)div_up(max_batch, prim::SCAN_TILE) + 2, s->stream));
    PPCSR_TRY(prim::reserve_scan_state(s, (size_t)div_up(max_batch, prim::SCAN_TILE) + 2));
  }
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return PPCSR_OK;
}

// shared by the (src,dst) and the packed entry points: `packed` != nullptr selects the packed key builder
static int apply_device_common(ppcsr_shard *s, const uint32_t *d_src, const uint32_t *d_dst, const uint64_t *d_packed,
                               const uint32_t *d_val, uint64_t count, uint32_t default_val, ppcsr_batch_stats *stats,
                               const batch::SegmentTable *segments = nullptr, bool pairs = false,
                               bool no_sparse = false) {
  PPCSR_TRY(set_device(s));
  ppcsr_batch_stats st{};
  st.batch_size = count;
  st.slots_before = st.slots_after = s->geo.N;
  if (count == 0) {
    s->last = st;
    if (stats) *stats = st;
    return PPCSR_OK;
  }
  if (count >= (1ull << 31)) {
    g_ppcsr_error = "batch too large (>= 2^31 updates); split it";
    return PPCSR_ERR_ARG;
  }
  if (s->poisoned) return poisoned_error();
  const Geometry g = s->geo;
  PPCSR_TRY(reserve_worst_case(s, count));  // before anything is modified: see reserve_worst_case
  if (segments) {  // only an upper bound of the batch size is known: the keys (and values) are sized for it
    PPCSR_TRY(dev_reserve(s->key_a, count + batch::LTILE, s->stream));
    if (d_val) PPCSR_TRY(dev_reserve(s->pay_a, count, s->stream));
  } else {
    PPCSR_TRY(reserve_batch_arrays(s, count));
  }
  BatchScalars *sc = s->d_scalars;
  CUDA_TRY(cudaMemsetAsync(sc, 0, sizeof(BatchScalars), s->stream));
  s->all_touched = 0;
  CUDA_TRY(cudaEventRecord(s->ev[0], s->stream));
  s->launches = 2;  // build_keys, locate

  // 1. keys + guards.  With no per-update values every payload is default_val: sort keys only.
  const bool has_pay = d_val != nullptr;
  // per-update values: removes are also flagged in bit 63 of the key word (free while vertex ids stay below 2^31),
  // so that a stream whose non-zero values are all equal can be sorted keys-only (see batch::emit_key)
  const uint32_t op_bit = (has_pay && s->n < (1u << 31)) ? 1u : 0u;
  // Speculated sort layout: the widest dst seen so far (at least the vertex ids) and, for the sources, "nothing is
  // rejected".  The key builder takes the digit histograms of that layout along (batch::HistArgs); if the batch turns
  // out wider, or needs fewer passes, prim::k_os_hist runs on the real layout as before.
  const uint32_t dst_spec = s->dst_or_seen | (s->n ? s->n - 1u : 0u);
  const int lo_spec = std::max(1, bits_of(dst_spec));
  const int hi_spec = std::max(1, bits_of(s->n ? s->n - 1 : 0));
  batch::HistArgs H{};
  H.P = prim::make_sort_passes(lo_spec, hi_spec);
  H.ghist = nullptr;
  const bool fused_hist = count > prim::SS_MAX;  // (smaller batches are sorted by one CTA: no global histograms)
  if (fused_hist) PPCSR_TRY(prim::radix_sort_prepare(s, count, H.P, &H.ghist));
  // The builder writes the batch out as an array of key words.  PPCSR_RAW_FIRST_PASS=1 (development knob) skips that:
  // the first pass of the sort then builds the key words from the caller's arrays itself (batch::RawArrays / RawPacked /
  // RawSegments).  Measured on B200: one write and one read of the batch less, but two 4-byte streams and the guards
  // inside the instruction-bound sort pass cost more than they save -- sort stage 3.35 -> 3.69 ms on C4, 0.364 -> 0.403 ms
  // on C2 -- so it is off by default.
  static const bool raw_first_pass = getenv("PPCSR_RAW_FIRST_PASS") != nullptr;
  const bool materialize = !raw_first_pass || (!segments && count <= prim::SS_MAX);
  uint64_t *key_out = materialize ? s->key_a.p : nullptr;
  const uint32_t src_default = default_val;  // (default_val may be replaced below when the values are all equal)
  const unsigned kb = std::min<unsigned>(div_up(count, batch::BT * 8), 148 * (fused_hist ? 8 : 16));
  if (segments) {
    PPCSR_TRY(dev_reserve(s->seg_prefix, (size_t)segments->n_seg + 2, s->stream));
    batch::SegmentTable T = *segments;
    T.prefix_out = s->seg_prefix.p;
    batch::k_build_keys_segments<<<kb, batch::BT, 0, s->stream>>>(d_packed, d_val, default_val, T, s->n, op_bit, key_out,
                                                                 has_pay ? s->pay_a.p : nullptr, sc, H);
  } else if (d_packed) {
    batch::k_build_keys_packed<<<kb, batch::BT, 0, s->stream>>>(d_packed, d_val, default_val, count, s->n, op_bit, key_out,
                                                               has_pay ? s->pay_a.p : nullptr, sc, pairs ? 1u : 0u, H);
  } else {
    batch::k_build_keys<<<kb, batch::BT, 0, s->stream>>>(d_src, d_dst, d_val, default_val, count, s->n, op_bit, key_out,
                                                        has_pay ? s->pay_a.p : nullptr, sc, H);
  }
  CUDA_TRY(cudaGetLastError());
  // Small-batch path (sparse.cuh): no host round trip here -- the sort width is speculated from the dsts seen so far
  // (k_locate checks it on the device) -- and none for the windows; see below.
  static const int env_sparse = [] {
    const char *e = getenv("PPCSR_SPARSE");
    return !e ? 0 : std::string(e) == "never" ? -1 : std::string(e) == "always" ? 1 : 0;
  }();
  const bool sparse = !no_sparse && !segments && env_sparse >= 0 && s->sparse_policy >= 0 && s->whole_policy <= 0 &&
                      g.n_leaves >= 1024 && count <= SPARSE_MAX_BATCH && (count * 4 <= g.n_leaves || env_sparse > 0);
  // every API call counts on a batch of a thousand updates: the small-batch path records the per-stage events only on
  // request (PPCSR_STAGE_TIMING=1); ms_total is always measured
  static const bool env_stage = getenv("PPCSR_STAGE_TIMING") != nullptr;
  const bool stage_ev = !sparse || env_stage;
  int lo_bits, hi_bits;
  bool sort_pay = has_pay, hist_done = false;
  if (sparse) {
    lo_bits = lo_spec;
    hi_bits = std::max(1, bits_of(s->n));  // wide enough for the rejected key (n << 32) too
    hist_done = fused_hist && hi_bits == hi_spec;
  } else {
    PPCSR_TRY(read_scalars(s));
    s->dst_or_seen |= s->h_scalars->dst_or;
    if (segments) {  // the real batch size arrives with the sort width
      if (s->h_scalars->seg_total > count) {
        g_ppcsr_error = "the peers deposited more records than max_total allows";
        return PPCSR_ERR_CAPACITY;
      }
      count = s->h_scalars->seg_total;
      st.batch_size = count;
      if (count == 0) {
        s->last = st;
        if (stats) *stats = st;
        return PPCSR_OK;
      }
      PPCSR_TRY(reserve_batch_arrays(s, count));
    }
    lo_bits = std::max(1, bits_of(s->h_scalars->dst_or));
    // rejected updates carry the key (n << 32): they need bits_of(n) source bits, valid ones bits_of(n-1)
    hi_bits = std::max(1, s->h_scalars->n_ignored ? bits_of(s->n) : bits_of(s->n ? s->n - 1 : 0));
    // the values travel as payload unless they are all the same
    if (op_bit) {
      const uint32_t vmax = s->h_scalars->val_max, vmin = ~s->h_scalars->val_inv_min;
      if (vmax == 0u || vmax == vmin) {  // removes only, or ONE non-zero value: the key's op bit says it all
        sort_pay = false;
        default_val = vmax ? vmax : 1u;
      }
    }
    // the speculated layout holds if the batch is no wider and would not get away with fewer passes
    if (fused_hist && count > prim::SS_MAX && lo_bits <= lo_spec && hi_bits <= hi_spec &&
        prim::make_sort_passes(lo_bits, hi_bits).n_pass == H.P.n_pass) {
      lo_bits = lo_spec;
      hi_bits = hi_spec;
      hist_done = true;
    }
  }
  // 2. stable radix sort by (src,dst)
  uint64_t *keys;
  uint32_t *pay;
  if (materialize) {
    PPCSR_TRY(prim::radix_sort_pairs(s, s->key_a.p, sort_pay ? s->pay_a.p : nullptr, s->key_b.p, s->pay_b.p, count,
                                     lo_bits, hi_bits, &keys, &pay, hist_done));
  } else if (segments) {
    const batch::RawSegments R{d_packed, d_val, s->seg_prefix.p, segments->cap, segments->n_seg, src_default, s->n, op_bit};
    PPCSR_TRY(prim::radix_sort_from(s, R, sort_pay, s->key_a.p, s->pay_a.p, s->key_b.p, s->pay_b.p, count, lo_bits,
                                    hi_bits, &keys, &pay, hist_done));
  } else if (d_packed) {
    const batch::RawPacked R{d_packed, d_val, src_default, s->n, op_bit, pairs ? 1u : 0u};
    PPCSR_TRY(prim::radix_sort_from(s, R, sort_pay, s->key_a.p, s->pay_a.p, s->key_b.p, s->pay_b.p, count, lo_bits,
                                    hi_bits, &keys, &pay, hist_done));
  } else {
    const batch::RawArrays R{d_src, d_dst, d_val, src_default, s->n, op_bit};
    PPCSR_TRY(prim::radix_sort_from(s, R, sort_pay, s->key_a.p, s->pay_a.p, s->key_b.p, s->pay_b.p, count, lo_bits,
                                    hi_bits, &keys, &pay, hist_done));
  }
  if (stage_ev) CUDA_TRY(cudaEventRecord(s->ev[1], s->stream));
  // 3+4. call counts, last-op-wins, locate, per-leaf counts -- one kernel over the sorted batch
  const uint64_t invalid_key = (uint64_t)s->n << 32;
  if (sparse) {  // the per-leaf batch counters are kept clear between small batches: no O(leaves) fill per batch
    PPCSR_TRY(dev_reserve(s->touched_flags, std::min<size_t>(g.n_leaves, count) + 1, s->stream));
    if (!s->cnt_clean) {
      CUDA_TRY(cudaMemsetAsync(s->ins_cnt.p, 0, (size_t)g.n_leaves * sizeof(uint32_t), s->stream));
      CUDA_TRY(cudaMemsetAsync(s->del_cnt.p, 0, (size_t)g.n_leaves * sizeof(uint32_t), s->stream));
      s->cnt_clean = true;
    }
    if (++s->touch_epoch == 0u) {  // the stamps wrapped: no old stamp may look current
      CUDA_TRY(cudaMemsetAsync(s->touch_stamp.p, 0, s->touch_stamp.cap * sizeof(uint32_t), s->stream));
      s->touch_epoch = 1u;
    }
  } else {
    CUDA_TRY(cudaMemsetAsync(s->ins_cnt.p, 0, (size_t)g.n_leaves * sizeof(uint32_t), s->stream));
    CUDA_TRY(cudaMemsetAsync(s->del_cnt.p, 0, (size_t)g.n_leaves * sizeof(uint32_t), s->stream));
    s->cnt_clean = false;
  }
  s->last_sparse = false;
  // one CTA per tile of sorted updates; every tile leaves its inserts, compacted, in its own region of a scratch list
  // (the sort's spare key buffer holds dst and value, uloc the predecessor slots); a scan of the tile counts and a
  // gather make the global key-ordered insert list
  const unsigned lblocks = div_up(count, batch::LTILE);
  const size_t padded = (size_t)lblocks * batch::LTILE;
  uint64_t *spare = keys == s->key_a.p ? s->key_b.p : s->key_a.p;
  uint32_t *tile_dst = reinterpret_cast<uint32_t *>(spare), *tile_val = tile_dst + padded;
  PPCSR_TRY(dev_reserve(s->uloc, padded, s->stream));
  PPCSR_TRY(dev_reserve(s->tile_cnt, (size_t)lblocks + 1, s->stream));
  // a batch of ONE tile needs no scan and no gather: the tile's run is the insert list
  // With no payload every insert of the batch carries default_val: the general path then neither writes nor reads a
  // value list (k_rebalance_m / k_rebalance_small take the one value; the small-batch path and the round-1 kernels
  // keep the list)
  s->ins_uniform_val = (!pay && !sparse && reb_kernel_m()) ? default_val : 0u;
  if (s->ins_uniform_val) tile_val = nullptr;
  uint32_t *t_dst = lblocks == 1 ? s->ins_dst.p : tile_dst;
  uint32_t *t_val = s->ins_uniform_val ? nullptr : lblocks == 1 ? s->ins_val.p : tile_val;
  uint32_t *t_pred = lblocks == 1 ? s->ins_pred.p : s->uloc.p;
  const uint32_t dst_mask = lo_bits >= 32 ? 0xFFFFFFFFu : ((1u << lo_bits) - 1u);
  const bool ins_only = !pay && !op_bit && default_val != 0u;  // every update of the batch is an insert
  const bool del_only = !pay && !op_bit && default_val == 0u;  // ... a remove
  auto locate = [&](auto kernel, uint32_t *touched, uint32_t *stamp, uint32_t epoch) {
    kernel<<<lblocks, batch::LT, sizeof(batch::LocSmem), s->stream>>>(
        keys, pay, default_val, count, invalid_key, s->dest.p, s->val.p, s->leaf_cnt.p, s->beg.p, g.leaf_shift,
        (uint32_t)g.N, s->nn.p, t_dst, t_val, t_pred, s->tile_cnt.p, s->ins_cnt.p, s->del_cnt.p, op_bit, sc, touched,
        stamp, epoch, dst_mask);
  };
  if (sparse) {
    if (ins_only) locate(batch::k_locate<true, true>, s->touched.p, s->touch_stamp.p, s->touch_epoch);
    else locate(batch::k_locate<true, false>, s->touched.p, s->touch_stamp.p, s->touch_epoch);
  } else {
    if (ins_only) locate(batch::k_locate<false, true>, nullptr, nullptr, 0u);
    else if (del_only) locate(batch::k_locate<false, false, true>, nullptr, nullptr, 0u);
    else locate(batch::k_locate<false, false>, nullptr, nullptr, 0u);
  }
  if (lblocks > 1) {
    PPCSR_TRY(prim::device_scan(s, prim::InArray{s->tile_cnt.p}, prim::OutPrefixWithTotal{s->tile_cnt.p, lblocks},
                                lblocks, nullptr, nullptr));
    s->launches++;
    batch::k_gather_inserts<<<div_up(lblocks, batch::GATHER_TILES), batch::LT, 0, s->stream>>>(
        tile_dst, tile_val, s->uloc.p, s->tile_cnt.p, s->ins_dst.p, s->ins_val.p, s->ins_pred.p, sc, lblocks);
  }
  if (stage_ev) CUDA_TRY(cudaEventRecord(s->ev[2], s->stream));
  if (sparse) {
    // 5s. tree, windows and rebalance of the small-batch path, then the ONE host synchronisation of the batch
    const unsigned tb = div_up(std::min<uint64_t>(count, g.n_leaves), sp::ST);
    s->epoch++;
    s->launches += 4;
    sp::k_sp_tree<<<tb, sp::ST, 0, s->stream>>>(s->touched.p, sc, s->ins_cnt.p, s->del_cnt.p, g.n_leaves, s->tree.p,
                                               s->touched_flags.p);
    win::k_select<<<tb, win::WT, 0, s->stream>>>(s->touched.p, &sc->n_touched, s->ins_cnt.p, s->del_cnt.p, s->tree.p,
                                                g.n_leaves, g.logN, (int)g.H, s->mark.p, s->epoch, sc);
    sp::k_sp_windows<<<tb, sp::ST, 0, s->stream>>>(s->touched.p, s->mark.p, s->epoch, s->tree.p, g.n_leaves, g.logN,
                                                  s->windows.p, sc);
    if (stage_ev) {
      CUDA_TRY(cudaEventRecord(s->ev[3], s->stream));
      CUDA_TRY(cudaEventRecord(s->ev[5], s->stream));
    }
    sp::RebArgs R{};
    R.dest = s->dest.p;
    R.val = s->val.p;
    R.leaf_cnt = s->leaf_cnt.p;
    R.tree = s->tree.p;
    R.ins_cnt = s->ins_cnt.p;
    R.del_cnt = s->del_cnt.p;
    R.ins_dst = s->ins_dst.p;
    R.ins_val = s->ins_val.p;
    R.ins_pred = s->ins_pred.p;
    R.beg = s->beg.p;
    R.windows = s->windows.p;
    R.sc = sc;
    R.n_leaves = g.n_leaves;
    R.ls = g.leaf_shift;
    sp::k_sp_rebalance<<<std::max(1u, div_up(std::min<uint64_t>(count, g.n_leaves), reb::RWARPS)), reb::RT, 0,
                         s->stream>>>(R);
    if (stage_ev) CUDA_TRY(cudaEventRecord(s->ev[6], s->stream));
    CUDA_TRY(cudaEventRecord(s->ev[4], s->stream));
    CUDA_TRY(cudaGetLastError());
    PPCSR_TRY(read_scalars(s));
    const BatchScalars h = *s->h_scalars;
    s->dst_or_seen |= h.dst_or;
    if (h.sparse_abort)  // a dst wider than the speculated sort width: nothing was modified, run the batch the general way
      return apply_device_common(s, d_src, d_dst, d_packed, d_val, count, default_val, stats, segments, pairs, true);
    if (h.sparse_done) {
      st.n_ignored = h.n_ignored;
      st.n_unique = h.n_unique;
      st.n_inserted = h.n_inserted;
      st.n_overwritten = h.n_overwritten;
      st.n_deleted = h.n_deleted;
      st.n_not_found = h.n_not_found;
      st.n_windows = h.n_windows;
      st.window_slots = h.window_slots;
      st.rebalance_bytes = 2ull * h.window_slots * 8ull;
      st.sparse_path = 1;
      s->items += h.n_inserted - h.n_deleted;
      s->last_sparse = true;
      s->last_touched = (uint32_t)h.n_touched;
      PPCSR_TRY(finalize_stats(s, &st, stage_ev));
      if (stats) *stats = st;
      return PPCSR_OK;
    }
    // a window larger than one warp handles, or the root out of bounds: the general path takes over from the per-leaf
    // counts and the insert list (its own window list, scans and tree)
    CUDA_TRY(cudaMemsetAsync(&sc->n_touched, 0, offsetof(BatchScalars, dst_or) - offsetof(BatchScalars, n_touched),
                             s->stream));
    CUDA_TRY(cudaMemsetAsync(&sc->root_violation, 0, sizeof(unsigned int), s->stream));
    s->cnt_clean = false;
    if (!stage_ev) {  // the general path's statistics read every stage event
      CUDA_TRY(cudaEventRecord(s->ev[1], s->stream));
      CUDA_TRY(cudaEventRecord(s->ev[2], s->stream));
    }
  }
  // 5. windows + rebalance
  PPCSR_TRY(finish_batch(s, count, &st));
  PPCSR_TRY(finalize_stats(s, &st));
  if (stats) *stats = st;
  return PPCSR_OK;
}

int ppcsr_apply_batch_device(ppcsr_shard *s, const uint32_t *d_src, const uint32_t *d_dst, const uint32_t *d_val,
                             uint64_t count, uint32_t default_val, ppcsr_batch_stats *stats) {
  if (!s || (count && (!d_src || !d_dst))) return PPCSR_ERR_ARG;
  return apply_device_common(s, d_src, d_dst, nullptr, d_val, count, default_val, stats);
}

int ppcsr_apply_batch_packed_device(ppcsr_shard *s, const uint64_t *d_packed, const uint32_t *d_val, uint64_t count,
                                    uint32_t default_val, ppcsr_batch_stats *stats) {
  if (!s || (count && !d_packed)) return PPCSR_ERR_ARG;
  return apply_device_common(s, nullptr, nullptr, d_packed, d_val, count, default_val, stats);
}

int ppcsr_apply_batch_segments_device(ppcsr_shard *s, const uint64_t *d_packed, const uint32_t *d_val,
                                      uint64_t region_cap, const uint64_t *d_counts, uint32_t n_segments,
                                      uint64_t max_total, uint32_t default_val, ppcsr_batch_stats *stats) {
  if (!s || !d_counts || !d_packed || n_segments == 0 || n_segments > batch::BIN_MAX_PARTS) return PPCSR_ERR_ARG;
  batch::SegmentTable T{};
  T.n_seg = n_segments;
  T.cap = region_cap;
  T.counts = d_counts;
  uint64_t bound = max_total ? std::min<uint64_t>(max_total, (uint64_t)n_segments * region_cap)
                             : (uint64_t)n_segments * region_cap;
  bound = std::min<uint64_t>(bound, (1ull << 31) - 1);  // one batch holds < 2^31 updates
  T.bound = bound;  // the keys are sized for `bound`: k_build_keys_segments writes no more than that
  return apply_device_common(s, nullptr, nullptr, d_packed, d_val, bound, default_val, stats, &T);
}

int ppcsr_apply_batch(ppcsr_shard *s, const uint32_t *src, const uint32_t *dst, const uint32_t *val, uint64_t count,
                      uint32_t default_val, ppcsr_batch_stats *stats) {
  if (!s || (count && (!src || !dst))) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  if (count == 0) return ppcsr_apply_batch_device(s, nullptr, nullptr, nullptr, 0, default_val, stats);
  PPCSR_TRY(dev_reserve(s->in_src, count, s->stream));
  PPCSR_TRY(dev_reserve(s->in_dst, count, s->stream));
  CUDA_TRY(cudaMemcpyAsync(s->in_src.p, src, count * sizeof(uint32_t), cudaMemcpyHostToDevice, s->stream));
  CUDA_TRY(cudaMemcpyAsync(s->in_dst.p, dst, count * sizeof(uint32_t), cudaMemcpyHostToDevice, s->stream));
  if (val) {
    PPCSR_TRY(dev_reserve(s->in_val, count, s->stream));
    CUDA_TRY(cudaMemcpyAsync(s->in_val.p, val, count * sizeof(uint32_t), cudaMemcpyHostToDevice, s->stream));
  }
  return ppcsr_apply_batch_device(s, s->in_src.p, s->in_dst.p, val ? s->in_val.p : nullptr, count, default_val, stats);
}

// ---- pipelined host submit: the copy of batch i+1 runs under the compute of batch i -----------------------------
int ppcsr_submit_batch(ppcsr_shard *s, const uint32_t *src, const uint32_t *dst, const uint32_t *val, uint64_t count,
                       uint32_t default_val, uint64_t *ticket) {
  if (!s || !ticket || (count && (!src || !dst))) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  ppcsr_shard::Pending &P = s->pending[s->next_ticket & 1u];
  if (P.busy) {
    g_ppcsr_error = "ppcsr_submit_batch: two batches are already in flight; ppcsr_wait for the older one first";
    return PPCSR_ERR_ARG;
  }
  if (!s->copy_stream) CUDA_TRY(cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking));
  if (!P.copied) CUDA_TRY(cudaEventCreateWithFlags(&P.copied, cudaEventDisableTiming));
  PPCSR_TRY(dev_reserve(P.src, count, s->copy_stream));
  PPCSR_TRY(dev_reserve(P.dst, count, s->copy_stream));
  if (val) PPCSR_TRY(dev_reserve(P.val, count, s->copy_stream));
  if (count) {
    CUDA_TRY(cudaMemcpyAsync(P.src.p, src, count * sizeof(uint32_t), cudaMemcpyHostToDevice, s->copy_stream));
    CUDA_TRY(cudaMemcpyAsync(P.dst.p, dst, count * sizeof(uint32_t), cudaMemcpyHostToDevice, s->copy_stream));
    if (val) CUDA_TRY(cudaMemcpyAsync(P.val.p, val, count * sizeof(uint32_t), cudaMemcpyHostToDevice, s->copy_stream));
  }
  CUDA_TRY(cudaEventRecord(P.copied, s->copy_stream));
  P.count = count;
  P.default_val = default_val;
  P.has_val = val != nullptr;
  P.busy = true;
  P.ticket = s->next_ticket++;
  *ticket = P.ticket;
  return PPCSR_OK;
}

int ppcsr_wait(ppcsr_shard *s, uint64_t ticket, ppcsr_batch_stats *stats) {
  if (!s) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  ppcsr_shard::Pending &P = s->pending[ticket & 1u];
  if (!P.busy || P.ticket != ticket) {
    g_ppcsr_error = "ppcsr_wait: no such batch in flight";
    return PPCSR_ERR_ARG;
  }
  // batches are applied in submission order: the other slot must not hold an older batch
  const ppcsr_shard::Pending &O = s->pending[(ticket & 1u) ^ 1u];
  if (O.busy && O.ticket < ticket) {
    g_ppcsr_error = "ppcsr_wait: an older batch is still pending; wait for it first (batches apply in order)";
    return PPCSR_ERR_ARG;
  }
  CUDA_TRY(cudaStreamWaitEvent(s->stream, P.copied, 0));
  const int rc = apply_device_common(s, P.src.p, P.dst.p, nullptr, P.has_val ? P.val.p : nullptr, P.count,
                                     P.default_val, stats);
  P.busy = false;
  return rc;
}

// ---- binary input path: interleaved (src, dst) pairs, e.g. an mmap'd edge file -----------------------------------
int ppcsr_apply_batch_pairs(ppcsr_shard *s, const uint32_t *pairs, uint64_t count, uint32_t default_val,
                            ppcsr_batch_stats *stats) {
  if (!s || (count && !pairs)) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  if (count == 0) return ppcsr_apply_batch_device(s, nullptr, nullptr, nullptr, 0, default_val, stats);
  // staged as u64 words: little-endian (src, dst) reads as dst << 32 | src, the key builder swaps the halves
  PPCSR_TRY(dev_reserve(s->in_src, 2 * count, s->stream));
  CUDA_TRY(cudaMemcpyAsync(s->in_src.p, pairs, count * 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, s->stream));
  return apply_device_common(s, nullptr, nullptr, reinterpret_cast<const uint64_t *>(s->in_src.p), nullptr, count,
                             default_val, stats, nullptr, true);
}

// ---- text input path: the reference's edge-list reader on the GPU (parse.cuh) -----------------------------------
int ppcsr_parse_edge_list(int device, const char *text, uint64_t bytes, uint32_t default_val, uint32_t **d_src,
                          uint32_t **d_dst, uint32_t **d_val, uint64_t *count, uint64_t *n_parsed, uint32_t *max_id) {
  if (!d_src || !d_dst || !d_val || !count || (bytes && !text)) return PPCSR_ERR_ARG;
  *d_src = *d_dst = *d_val = nullptr;
  *count = 0;
  if (n_parsed) *n_parsed = 0;
  if (max_id) *max_id = 0;
  if (ppcsr_device_count() <= device || device < 0) return PPCSR_ERR_NO_DEVICE;
  if (bytes == 0) return PPCSR_OK;
  CUDA_TRY(cudaSetDevice(device));
  ppcsr_shard tmp;  // scan scratch only
  tmp.device = device;
  tmp.stream = nullptr;
  DevBuf<char> d_text;
  DevBuf<unsigned long long> d_starts, d_misc;
  DevBuf<uint32_t> o_src, o_dst, o_val;
  int rc = [&]() -> int {
    PPCSR_TRY(dev_reserve(d_text, bytes, nullptr));
    CUDA_TRY(cudaMemcpy(d_text.p, text, bytes, cudaMemcpyHostToDevice));
    PPCSR_TRY(dev_reserve(d_misc, 4, nullptr));
    CUDA_TRY(cudaMemset(d_misc.p, 0, 4 * sizeof(unsigned long long)));
    // pass 1: count the newlines (sizes the line table), pass 2: the line starts
    PPCSR_TRY(prim::device_scan(&tmp, parse::InIsNewline{d_text.p}, prim::OutNothing{}, bytes, nullptr, d_misc.p));
    unsigned long long newlines = 0;
    CUDA_TRY(cudaMemcpy(&newlines, d_misc.p, sizeof(newlines), cudaMemcpyDeviceToHost));
    const unsigned long long n_lines = newlines + (text[bytes - 1] == '\n' ? 0ull : 1ull);
    if (n_lines == 0) return PPCSR_OK;
    PPCSR_TRY(dev_reserve(d_starts, newlines + 2, nullptr));
    CUDA_TRY(cudaMemset(d_starts.p, 0, sizeof(unsigned long long)));  // line 0 starts at byte 0
    PPCSR_TRY(prim::device_scan(&tmp, parse::InIsNewline{d_text.p}, parse::OutLineStart{d_starts.p}, bytes, nullptr,
                                nullptr));
    PPCSR_TRY(dev_reserve(o_src, n_lines, nullptr));
    PPCSR_TRY(dev_reserve(o_dst, n_lines, nullptr));
    PPCSR_TRY(dev_reserve(o_val, n_lines, nullptr));
    parse::k_parse_lines<<<div_up(n_lines, parse::PT), parse::PT>>>(
        d_text.p, bytes, d_starts.p, n_lines, default_val, o_src.p, o_dst.p, o_val.p,
        reinterpret_cast<unsigned int *>(d_misc.p + 1), d_misc.p + 2);
    CUDA_TRY(cudaGetLastError());
    unsigned long long h[4];
    CUDA_TRY(cudaMemcpy(h, d_misc.p, sizeof(h), cudaMemcpyDeviceToHost));
    *count = n_lines;
    if (max_id) *max_id = (uint32_t)h[1];
    if (n_parsed) *n_parsed = h[2];
    return PPCSR_OK;
  }();
  dev_free(d_text); dev_free(d_starts); dev_free(d_misc);
  dev_free(tmp.block_tmp); dev_free(tmp.scan_state); dev_free(tmp.scan_ticket);
  if (rc != PPCSR_OK) {
    dev_free(o_src); dev_free(o_dst); dev_free(o_val);
    return rc;
  }
  *d_src = o_src.p;
  *d_dst = o_dst.p;
  *d_val = o_val.p;
  return PPCSR_OK;
}

int ppcsr_free_device(int device, void *p) {
  if (!p) return PPCSR_OK;
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(cudaFree(p));
  return PPCSR_OK;
}

int ppcsr_copy_to_host(int device, void *host, const void *dev, uint64_t bytes) {
  if (bytes && (!host || !dev)) return PPCSR_ERR_ARG;
  CUDA_TRY(cudaSetDevice(device));
  if (bytes) CUDA_TRY(cudaMemcpy(host, dev, bytes, cudaMemcpyDeviceToHost));
  return PPCSR_OK;
}

int ppcsr_add_edge(ppcsr_shard *s, uint32_t src, uint32_t dst, uint32_t value) {
  if (value == 0) return PPCSR_OK;  // reference PCSR.cpp:1375: a zero value is silently ignored
  return ppcsr_apply_batch(s, &src, &dst, &value, 1, 1, nullptr);
}

int ppcsr_remove_edge(ppcsr_shard *s, uint32_t src, uint32_t dst, int *found) {
  ppcsr_batch_stats st{};
  const uint32_t zero = 0;
  PPCSR_TRY(ppcsr_apply_batch(s, &src, &dst, &zero, 1, 0, &st));
  if (found) *found = st.n_deleted ? 1 : 0;
  return PPCSR_OK;
}

int ppcsr_add_nodes(ppcsr_shard *s, uint32_t count) {
  if (!s) return PPCSR_ERR_ARG;
  if (count == 0) return PPCSR_OK;
  PPCSR_TRY(set_device(s));
  if (s->poisoned) return poisoned_error();
  if ((uint64_t)s->n + count >= 0xFFFFFFFEull) return PPCSR_ERR_CAPACITY;
  const uint32_t n_old = s->n, n_new = s->n + count;
  PPCSR_TRY(dev_reserve(s->beg, (size_t)n_new + 1, s->stream, true));
  PPCSR_TRY(dev_reserve(s->nn, (size_t)n_new + 1, s->stream, true));
  CUDA_TRY(cudaMemsetAsync(s->nn.p + n_old, 0, (size_t)count * sizeof(uint32_t), s->stream));
  ppcsr_batch_stats st{};
  st.batch_size = count;
  if (s->items == 0) {  // empty structure: lay the new sentinels out directly
    s->n = n_new;
    const uint64_t need = initial_slots(n_new, n_new);
    if (need > s->geo.N) {
      s->geo = make_geometry(need);
      PPCSR_TRY(alloc_geometry(s, s->geo));
    }
    PPCSR_TRY(init_layout(s));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    s->last = st;
    return PPCSR_OK;
  }
  const Geometry g = s->geo;
  PPCSR_TRY(reserve_batch_arrays(s, count));
  PPCSR_TRY(reserve_worst_case(s, count));
  BatchScalars *sc = s->d_scalars;
  CUDA_TRY(cudaMemsetAsync(sc, 0, sizeof(BatchScalars), s->stream));
  s->all_touched = 0;
  for (int e = 0; e < 3; e++) CUDA_TRY(cudaEventRecord(s->ev[e], s->stream));
  s->launches = 2;
  CUDA_TRY(cudaMemsetAsync(s->ins_cnt.p, 0, (size_t)g.n_leaves * sizeof(uint32_t), s->stream));
  CUDA_TRY(cudaMemsetAsync(s->del_cnt.p, 0, (size_t)g.n_leaves * sizeof(uint32_t), s->stream));
  PPCSR_TRY(dev_reserve(s->misc, 16, s->stream));
  k_last_live_slot<<<1, 1, 0, s->stream>>>(s->leaf_cnt.p, g.n_leaves, g.leaf_shift, s->misc.p);
  k_fill_new_nodes<<<div_up(count, 256), 256, 0, s->stream>>>(s->ins_dst.p, s->ins_val.p, s->ins_pred.p, n_old, count,
                                                             s->misc.p, s->ins_cnt.p, g.leaf_shift, sc);
  CUDA_TRY(cudaGetLastError());
  s->n = n_new;  // beg[n_new] = N is (re)written below; sentinel fix-up fills beg[n_old .. n_new)
  s->cnt_clean = false;
  s->last_sparse = false;
  s->ins_sentinels = true;
  s->ins_uniform_val = 0;  // the new sentinels carry their vertex ids
  const int fb = finish_batch(s, count, &st);
  s->ins_sentinels = false;
  PPCSR_TRY(fb);
  reb::k_set_u32<<<1, 1, 0, s->stream>>>(s->beg.p + s->n, (uint32_t)s->geo.N);
  PPCSR_TRY(finalize_stats(s, &st));
  return PPCSR_OK;
}

int ppcsr_set_whole_array_policy(ppcsr_shard *s, int mode) {
  if (!s || mode < -1 || mode > 1) return PPCSR_ERR_ARG;
  s->whole_policy = mode;
  return PPCSR_OK;
}

int ppcsr_last_stats(ppcsr_shard *s, ppcsr_batch_stats *stats) {
  if (!s || !stats) return PPCSR_ERR_ARG;
  *stats = s->last;
  return PPCSR_OK;
}

// scratch of the binning entry points: one per device, kept for the life of the process so that routing a batch
// never allocates (a cudaMalloc/cudaFree pair costs more than the binning kernels themselves)
struct BinScratch {
  ppcsr_shard shard;  // provides hist / block_tmp for the scan
  uint32_t *d_firsts = nullptr;
  uint32_t *h_firsts = nullptr;  // pinned
};
// One scratch per (device, stream), created under a lock: the scan inside the binning (ticket counter, look-back words,
// histogram buffer) is only correct when every use of one scratch is ordered on ONE stream, so two callers on the same
// device but different streams (or threads) must not share it.  Calls that share a stream are stream-ordered and safe.
static BinScratch *bin_scratch(int device, cudaStream_t stream) {
  static std::mutex mu;
  static std::vector<std::pair<std::pair<int, cudaStream_t>, BinScratch *>> all;
  std::lock_guard<std::mutex> lock(mu);
  for (auto &e : all)
    if (e.first.first == device && e.first.second == stream) return e.second;
  BinScratch *b = new BinScratch();
  b->shard.device = device;
  if (cudaMalloc((void **)&b->d_firsts, (batch::BIN_MAX_PARTS + 1) * sizeof(uint32_t)) != cudaSuccess ||
      cudaMallocHost((void **)&b->h_firsts, (batch::BIN_MAX_PARTS + 1) * sizeof(uint32_t)) != cudaSuccess) {
    cudaGetLastError();
    delete b;
    return nullptr;
  }
  all.push_back({{device, stream}, b});
  return b;
}
__global__ void k_gather_firsts(const uint32_t *__restrict__ offs, uint32_t nblocks, uint32_t parts,
                                uint32_t *__restrict__ firsts) {
  const uint32_t p = threadIdx.x;
  if (p < parts) firsts[p] = offs[(size_t)p * nblocks];
}

static int bin_common(int device, void *cuda_stream, const uint64_t *d_starts, uint32_t n_parts, const uint32_t *d_src,
                      const uint32_t *d_dst, const uint32_t *d_val, uint64_t count, uint32_t *d_out_src,
                      uint32_t *d_out_dst, uint32_t *d_out_val, uint64_t *d_out_packed, uint64_t *h_counts) {
  if (n_parts == 0 || n_parts > batch::BIN_MAX_PARTS || !h_counts) return PPCSR_ERR_ARG;
  for (uint32_t p = 0; p < n_parts; p++) h_counts[p] = 0;
  if (count == 0) return PPCSR_OK;
  CUDA_TRY(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  BinScratch *bs = bin_scratch(device, st);
  if (!bs) {
    g_ppcsr_error = "bin_by_owner: cannot allocate scratch";
    return PPCSR_ERR_CAPACITY;
  }
  ppcsr_shard &tmp = bs->shard;
  tmp.stream = st;
  const unsigned nblocks = div_up(count, prim::SORT_TILE);
  const size_t hn = (size_t)n_parts * nblocks;
  PPCSR_TRY(dev_reserve(tmp.hist, hn + 1, st));
  batch::k_bin_count<<<nblocks, batch::BT, 0, st>>>(d_src, count, d_starts, n_parts, tmp.hist.p, nblocks);
  PPCSR_TRY(prim::device_scan(&tmp, prim::InArray{tmp.hist.p}, prim::OutPrefixWithTotal{tmp.hist.p, hn}, hn, nullptr,
                              nullptr));
  batch::k_bin_scatter<<<nblocks, batch::BT, 0, st>>>(d_src, d_dst, d_val, count, d_starts, n_parts, tmp.hist.p, nblocks,
                                                     d_out_src, d_out_dst, d_out_val, d_out_packed);
  k_gather_firsts<<<1, batch::BIN_MAX_PARTS, 0, st>>>(tmp.hist.p, nblocks, n_parts, bs->d_firsts);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(bs->h_firsts, bs->d_firsts, n_parts * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  for (uint32_t p = 0; p < n_parts; p++) {
    const uint64_t next = p + 1 < n_parts ? bs->h_firsts[p + 1] : count;
    h_counts[p] = next - bs->h_firsts[p];
  }
  return PPCSR_OK;
}

int ppcsr_bin_to_peers(int device, void *cuda_stream, const uint64_t *d_starts, uint32_t n_parts, uint32_t my_rank,
                       const uint32_t *d_src, const uint32_t *d_dst, const uint32_t *d_val, uint64_t count,
                       const uint64_t *h_peer_rec, const uint64_t *h_peer_val, const uint64_t *h_peer_cnt,
                       uint64_t region_cap) {
  if (n_parts == 0 || n_parts > batch::BIN_MAX_PARTS || my_rank >= n_parts || !h_peer_rec || !h_peer_cnt ||
      (d_val && !h_peer_val) || (count && (!d_src || !d_dst)))
    return PPCSR_ERR_ARG;
  if (count > region_cap || count >= (1ull << 32)) {
    g_ppcsr_error = "bin_to_peers: the batch exceeds the capacity of this rank's region in the peers' buffers";
    return PPCSR_ERR_CAPACITY;
  }
  CUDA_TRY(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  batch::PeerTable P{};
  for (uint32_t p = 0; p < n_parts; p++) {
    P.rec[p] = reinterpret_cast<uint64_t *>(h_peer_rec[p]);
    P.val[p] = h_peer_val ? reinterpret_cast<uint32_t *>(h_peer_val[p]) : nullptr;
    P.cnt[p] = reinterpret_cast<uint64_t *>(h_peer_cnt[p]);
  }
  if (count == 0) {
    batch::k_zero_peer_counts<<<1, batch::BIN_MAX_PARTS, 0, st>>>(n_parts, my_rank, P);
    CUDA_TRY(cudaGetLastError());
    return PPCSR_OK;
  }
  BinScratch *bs = bin_scratch(device, st);
  if (!bs) {
    g_ppcsr_error = "bin_to_peers: cannot allocate scratch";
    return PPCSR_ERR_CAPACITY;
  }
  ppcsr_shard &tmp = bs->shard;
  tmp.stream = st;
  const unsigned nblocks = div_up(count, prim::SORT_TILE);
  const size_t hn = (size_t)n_parts * nblocks;
  PPCSR_TRY(dev_reserve(tmp.hist, std::max<size_t>(hn + 1, batch::BIN_MAX_PARTS), st));
  // Without per-update values every update of the batch is the same operation and their order inside a destination's
  // region does not matter: the tiles then claim their places with one atomicAdd per destination (tmp.hist[0 .. parts) is
  // the cursor) and the count pass + scan in front of the scatter go away (PPCSR_ROUTE_ORDERED=1 keeps them).
  static const bool force_ordered = getenv("PPCSR_ROUTE_ORDERED") != nullptr;
  const bool ordered = d_val != nullptr || force_ordered;
  if (ordered) {
    batch::k_bin_count<<<nblocks, batch::BT, 0, st>>>(d_src, count, d_starts, n_parts, tmp.hist.p, nblocks);
    PPCSR_TRY(prim::device_scan(&tmp, prim::InArray{tmp.hist.p}, prim::OutPrefixWithTotal{tmp.hist.p, hn}, hn, nullptr,
                                nullptr));
  } else {
    CUDA_TRY(cudaMemsetAsync(tmp.hist.p, 0, (size_t)n_parts * sizeof(uint32_t), st));
  }
  {  // per device, once, thread-safe
    static std::once_flag once[64];
    static cudaError_t once_err[64];
    const int dv = device & 63;
    std::call_once(once[dv], [&] {
      once_err[dv] = cudaFuncSetAttribute(batch::k_bin_scatter_peers<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)batch::bin_peers_smem(true));
      if (once_err[dv] == cudaSuccess)
        once_err[dv] = cudaFuncSetAttribute(batch::k_bin_scatter_peers<false>,
                                            cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)batch::bin_peers_smem(false));
      if (once_err[dv] == cudaSuccess)
        once_err[dv] = cudaFuncSetAttribute(batch::k_bin_scatter_peers<false, false>,
                                            cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)batch::bin_peers_smem(false));
    });
    CUDA_TRY(once_err[dv]);
  }
  if (d_val) {
    batch::k_bin_scatter_peers<true><<<nblocks, batch::BT, batch::bin_peers_smem(true), st>>>(
        d_src, d_dst, d_val, count, d_starts, n_parts, tmp.hist.p, nblocks, my_rank, region_cap, P);
  } else if (ordered) {
    batch::k_bin_scatter_peers<false><<<nblocks, batch::BT, batch::bin_peers_smem(false), st>>>(
        d_src, d_dst, nullptr, count, d_starts, n_parts, tmp.hist.p, nblocks, my_rank, region_cap, P);
  } else {
    batch::k_bin_scatter_peers<false, false><<<nblocks, batch::BT, batch::bin_peers_smem(false), st>>>(
        d_src, d_dst, nullptr, count, d_starts, n_parts, nullptr, nblocks, my_rank, region_cap, P, tmp.hist.p);
    batch::k_publish_peer_counts<<<1, batch::BIN_MAX_PARTS, 0, st>>>(n_parts, my_rank, tmp.hist.p, P);
  }
  CUDA_TRY(cudaGetLastError());
  return PPCSR_OK;
}

int ppcsr_bin_by_owner(int device, void *cuda_stream, const uint64_t *d_starts, uint32_t n_parts,
                       const uint32_t *d_src, const uint32_t *d_dst, const uint32_t *d_val, uint64_t count,
                       uint32_t *d_out_src, uint32_t *d_out_dst, uint32_t *d_out_val, uint64_t *h_counts) {
  if (count && (!d_out_src || !d_out_dst)) return PPCSR_ERR_ARG;
  return bin_common(device, cuda_stream, d_starts, n_parts, d_src, d_dst, d_val, count, d_out_src, d_out_dst, d_out_val,
                    nullptr, h_counts);
}

int ppcsr_bin_by_owner_packed(int device, void *cuda_stream, const uint64_t *d_starts, uint32_t n_parts,
                              const uint32_t *d_src, const uint32_t *d_dst, const uint32_t *d_val, uint64_t count,
                              uint64_t *d_out_packed, uint32_t *d_out_val, uint64_t *h_counts) {
  if (count && !d_out_packed) return PPCSR_ERR_ARG;
  return bin_common(device, cuda_stream, d_starts, n_parts, d_src, d_dst, d_val, count, nullptr, nullptr, d_out_val,
                    d_out_packed, h_counts);
}

// ---- reads ------------------------------------------------------------------------------------------
int ppcsr_geometry_of(ppcsr_shard *s, ppcsr_geometry *out) {
  if (!s || !out) return PPCSR_ERR_ARG;
  out->N = s->geo.N;
  out->logN = s->geo.logN;
  out->H = s->geo.H;
  out->n = s->n;
  out->items = s->items;
  return PPCSR_OK;
}

int ppcsr_edges_exist(ppcsr_shard *s, const uint32_t *src, const uint32_t *dst, uint64_t count, uint8_t *exists) {
  if (!s || (count && (!src || !dst || !exists))) return PPCSR_ERR_ARG;
  if (count == 0) return PPCSR_OK;
  PPCSR_TRY(set_device(s));
  PPCSR_TRY(dev_reserve(s->in_src, count, s->stream));
  PPCSR_TRY(dev_reserve(s->in_dst, count, s->stream));
  PPCSR_TRY(dev_reserve(s->ucls, count, s->stream));
  CUDA_TRY(cudaMemcpyAsync(s->in_src.p, src, count * 4, cudaMemcpyHostToDevice, s->stream));
  CUDA_TRY(cudaMemcpyAsync(s->in_dst.p, dst, count * 4, cudaMemcpyHostToDevice, s->stream));
  qry::k_edges_exist<<<div_up(count, qry::QT), qry::QT, 0, s->stream>>>(s->in_src.p, s->in_dst.p, count, s->n,
                                                                       s->dest.p, s->val.p, s->leaf_cnt.p, s->beg.p,
                                                                       s->geo.leaf_shift, s->ucls.p, nullptr);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(exists, s->ucls.p, count, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return PPCSR_OK;
}

int ppcsr_edge_exists(ppcsr_shard *s, uint32_t src, uint32_t dst, int *exists, uint32_t *out_value) {
  if (!s || !exists) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  PPCSR_TRY(dev_reserve(s->misc, 16, s->stream));
  uint32_t *hp = reinterpret_cast<uint32_t *>(s->h_pinned);
  hp[0] = src;
  hp[1] = dst;
  CUDA_TRY(cudaMemcpyAsync(s->misc.p, hp, 8, cudaMemcpyHostToDevice, s->stream));
  qry::k_edges_exist<<<1, 32, 0, s->stream>>>(s->misc.p, s->misc.p + 1, 1, s->n, s->dest.p, s->val.p, s->leaf_cnt.p,
                                             s->beg.p, s->geo.leaf_shift, reinterpret_cast<uint8_t *>(s->misc.p + 2),
                                             s->misc.p + 3);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(hp + 2, s->misc.p + 2, 8, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  *exists = (hp[2] & 0xFF) ? 1 : 0;
  if (out_value) *out_value = hp[3];
  return PPCSR_OK;
}

static int vertex_range(ppcsr_shard *s, uint32_t v, uint32_t *b, uint32_t *e) {
  uint32_t *hp = reinterpret_cast<uint32_t *>(s->h_pinned);
  CUDA_TRY(cudaMemcpyAsync(hp, s->beg.p + v, 8, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  *b = hp[0];
  *e = hp[1];
  return PPCSR_OK;
}

int ppcsr_neighbours(ppcsr_shard *s, uint32_t v, uint32_t *out, uint64_t cap, uint64_t *count) {
  if (!s || !count) return PPCSR_ERR_ARG;
  *count = 0;
  if (v >= s->n) return PPCSR_OK;  // reference PCSR.cpp:903: out-of-range vertex -> empty
  PPCSR_TRY(set_device(s));
  PPCSR_TRY(refresh_rank_off(s));
  uint32_t b, e;
  PPCSR_TRY(vertex_range(s, v, &b, &e));
  // degree = rank(e) - rank(b) - 1, ranks from rank_off (two small reads)
  const uint32_t ls = s->geo.leaf_shift, msk = s->geo.logN - 1;
  uint32_t *hp = reinterpret_cast<uint32_t *>(s->h_pinned);
  CUDA_TRY(cudaMemcpyAsync(hp, s->rank_off.p + (b >> ls), 4, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaMemcpyAsync(hp + 1, s->rank_off.p + (e >> ls), 4, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  const uint64_t deg = (uint64_t)(hp[1] + (e & msk)) - (hp[0] + (b & msk)) - 1;
  *count = deg;
  const uint64_t want = std::min<uint64_t>(deg, cap);
  if (want == 0 || !out) return PPCSR_OK;
  PPCSR_TRY(dev_reserve(s->misc, want + 16, s->stream));
  const unsigned blocks = std::min<unsigned>(div_up((uint64_t)e - b, qry::QT), 148 * 8);
  qry::k_neighbours<<<blocks, qry::QT, 0, s->stream>>>(s->dest.p, s->leaf_cnt.p, s->rank_off.p, ls, b, e, s->misc.p,
                                                      want);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(out, s->misc.p, want * 4, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return PPCSR_OK;
}

int ppcsr_read_neighbourhood(ppcsr_shard *s, uint32_t v, uint64_t *checksum) {
  if (!s) return PPCSR_ERR_ARG;
  if (checksum) *checksum = 0;
  if (v >= s->n) return PPCSR_OK;
  PPCSR_TRY(set_device(s));
  uint32_t b, e;
  PPCSR_TRY(vertex_range(s, v, &b, &e));
  PPCSR_TRY(dev_reserve(s->misc, 16, s->stream));
  CUDA_TRY(cudaMemsetAsync(s->misc.p, 0, 8, s->stream));
  const unsigned blocks = std::max(1u, std::min<unsigned>(div_up((uint64_t)e - b, qry::QT), 148 * 8));
  qry::k_touch<<<blocks, qry::QT, 0, s->stream>>>(s->dest.p, b, e, reinterpret_cast<unsigned long long *>(s->misc.p));
  CUDA_TRY(cudaGetLastError());
  uint64_t *hp = reinterpret_cast<uint64_t *>(s->h_pinned);
  CUDA_TRY(cudaMemcpyAsync(hp, s->misc.p, 8, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  if (checksum) *checksum = hp[0];
  return PPCSR_OK;
}

int ppcsr_num_neighbors(ppcsr_shard *s, uint32_t *out) {
  if (!s || (s->n && !out)) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  if (s->n) CUDA_TRY(cudaMemcpyAsync(out, s->nn.p, (size_t)s->n * 4, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return PPCSR_OK;
}

int ppcsr_node_ranges(ppcsr_shard *s, uint32_t *beginning, uint32_t *end) {
  if (!s) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  if (s->n == 0) return PPCSR_OK;
  std::vector<uint32_t> tmp((size_t)s->n + 1);
  CUDA_TRY(cudaMemcpyAsync(tmp.data(), s->beg.p, ((size_t)s->n + 1) * 4, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  for (uint32_t v = 0; v < s->n; v++) {
    if (beginning) beginning[v] = tmp[v];
    // the reference keeps the last vertex's end at N-1 (PCSR.cpp:180-182,811-813)
    if (end) end[v] = (v + 1 == s->n) ? (uint32_t)(s->geo.N - 1) : tmp[v + 1];
  }
  return PPCSR_OK;
}

int ppcsr_export_csr(ppcsr_shard *s, uint64_t *rowptr, uint32_t *col, uint32_t *val, uint64_t *edges) {
  if (!s) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  const uint64_t E = s->items - s->n;
  if (edges) *edges = E;
  DevCsr d;
  const int rc = [&]() -> int {
    PPCSR_TRY(export_device(s, rowptr ? &d.rowptr : nullptr, col ? &d.col : nullptr, col && val ? &d.val : nullptr));
    if (rowptr)
      CUDA_TRY(cudaMemcpyAsync(rowptr, d.rowptr.p, ((size_t)s->n + 1) * 8, cudaMemcpyDeviceToHost, s->stream));
    if (col && E) {
      CUDA_TRY(cudaMemcpyAsync(col, d.col.p, E * 4, cudaMemcpyDeviceToHost, s->stream));
      if (val) CUDA_TRY(cudaMemcpyAsync(val, d.val.p, E * 4, cudaMemcpyDeviceToHost, s->stream));
    }
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return PPCSR_OK;
  }();
  csr_free(s->device, d);
  return rc;
}

int ppcsr_load_csr(ppcsr_shard *s, uint32_t n, const uint64_t *rowptr, const uint32_t *col, const uint32_t *val,
                   const uint32_t *nn) {
  if (!s || !rowptr) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  if (s->poisoned) {
    g_ppcsr_error = "ppcsr_load_csr: the shard is poisoned by a failed batch; ppcsr_restore it first";
    return PPCSR_ERR_ARG;
  }
  if (submit_pending(s)) {
    g_ppcsr_error = "ppcsr_load_csr: a submitted batch is still pending; ppcsr_wait for it first";
    return PPCSR_ERR_ARG;
  }
  if ((uint64_t)n >= 0xFFFFFFFEull || rowptr[0] != 0 || (rowptr[n] && !col)) {
    g_ppcsr_error = "ppcsr_load_csr: rowptr[0] must be 0, n below 2^32 - 2, and col given when there are edges";
    return PPCSR_ERR_ARG;
  }
  const uint64_t E = rowptr[n];
  const uint64_t N2 = E < PPCSR_MAX_SLOTS ? layout_slots(s->geo.N, E + n) : 0;
  if (N2 == 0) {
    g_ppcsr_error = "ppcsr_load_csr: edge array would exceed 2^31 slots";
    return PPCSR_ERR_CAPACITY;
  }
  DevCsr d;
  const int rc = [&]() -> int {
    // the input, then its validation on the device: nothing of the shard is modified before it passes
    PPCSR_TRY(dev_reserve(d.rowptr, (size_t)n + 1, s->stream));
    PPCSR_TRY(dev_reserve(d.col, E, s->stream));
    if (val) PPCSR_TRY(dev_reserve(d.val, E, s->stream));
    if (nn) PPCSR_TRY(dev_reserve(d.nn, n, s->stream));
    PPCSR_TRY(dev_reserve(s->misc, 16, s->stream));
    CUDA_TRY(cudaMemcpyAsync(d.rowptr.p, rowptr, ((size_t)n + 1) * 8, cudaMemcpyHostToDevice, s->stream));
    if (E) CUDA_TRY(cudaMemcpyAsync(d.col.p, col, E * 4, cudaMemcpyHostToDevice, s->stream));
    if (E && val) CUDA_TRY(cudaMemcpyAsync(d.val.p, val, E * 4, cudaMemcpyHostToDevice, s->stream));
    if (n && nn) CUDA_TRY(cudaMemcpyAsync(d.nn.p, nn, (size_t)n * 4, cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaMemsetAsync(s->misc.p, 0, 4, s->stream));
    mig::k_validate_csr<<<div_up(std::max<uint64_t>((uint64_t)n + 1, E), mig::MT), mig::MT, 0, s->stream>>>(
        d.rowptr.p, d.col.p, val ? d.val.p : nullptr, n, E, s->misc.p);
    CUDA_TRY(cudaGetLastError());
    uint32_t *hp = reinterpret_cast<uint32_t *>(s->h_pinned);
    CUDA_TRY(cudaMemcpyAsync(hp, s->misc.p, 4, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    if (hp[0]) {
      g_ppcsr_error = std::string("ppcsr_load_csr: invalid CSR:") + ((hp[0] & 1u) ? " rowptr not 0 .. E non-decreasing;" : "") +
                      ((hp[0] & 2u) ? " col holds 0xFFFFFFFF;" : "") + ((hp[0] & 4u) ? " a value is 0;" : "") +
                      ((hp[0] & 8u) ? " a row is not strictly ascending;" : "");
      return PPCSR_ERR_ARG;
    }
    PPCSR_TRY(reserve_layout(s, N2, n));
    ppcsr_batch_stats st;
    PPCSR_TRY(commit_layout(s, N2, n, d.rowptr.p, d.col.p, val ? d.val.p : nullptr, nn ? d.nn.p : nullptr, E, &st));
    PPCSR_TRY(layout_stats(s, &st));
    return PPCSR_OK;
  }();
  csr_free(s->device, d);
  return rc;
}

int ppcsr_pagerank_push_device(ppcsr_shard *s, const double *d_in, double *d_out, uint64_t out_len) {
  if (!s || !d_in || !d_out) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  if (s->n == 0) return PPCSR_OK;
  launch_pagerank_push<double>(s, d_in, d_out, out_len);
  CUDA_TRY(cudaGetLastError());
  return PPCSR_OK;
}

int ppcsr_pagerank(ppcsr_shard *s, uint32_t iterations, double damping, double *out) {
  if (!s || !out) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  const uint64_t n = s->n;
  if (n == 0) return PPCSR_OK;
  DevBuf<double> d_r;
  PPCSR_TRY(dev_reserve(d_r, (size_t)n + 1, s->stream));
  PPCSR_TRY(dev_reserve(s->pr_acc, (size_t)n + 1, s->stream));
  const unsigned nb = div_up(n, 256);
  qry::k_fill_f64<<<nb, 256, 0, s->stream>>>(d_r.p, 1.0 / (double)n, n);
  CUDA_TRY(cudaMemsetAsync(s->pr_acc.p, 0, (size_t)n * sizeof(double), s->stream));
  for (uint32_t it = 0; it < iterations; it++) {
    launch_pagerank_push<double>(s, d_r.p, s->pr_acc.p, n);
    qry::k_pagerank_finish<<<nb, 256, 0, s->stream>>>(d_r.p, s->pr_acc.p, n, (1.0 - damping) / (double)n, damping);
  }
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(out, d_r.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  dev_free(d_r);
  return PPCSR_OK;
}

int ppcsr_pagerank_step_f64(ppcsr_shard *s, const double *in, double *out, uint64_t out_len) {
  return pagerank_host<double>(s, in, out, out_len);
}
int ppcsr_pagerank_step_f32(ppcsr_shard *s, const float *in, float *out, uint64_t out_len) {
  return pagerank_host<float>(s, in, out, out_len);
}

int ppcsr_bfs(ppcsr_shard *s, uint32_t start, uint32_t *dist) {
  if (!s || (s->n && !dist)) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  if (s->n == 0) return PPCSR_OK;
  DevBuf<uint32_t> d_dist, d_fa, d_fb;
  const int rc = [&]() -> int {
    PPCSR_TRY(dev_reserve(d_dist, (size_t)s->n + 1, s->stream));
    PPCSR_TRY(dev_reserve(d_fa, (size_t)s->n + 1, s->stream));
    PPCSR_TRY(dev_reserve(d_fb, (size_t)s->n + 1, s->stream));
    PPCSR_TRY(dev_reserve(s->misc, 16, s->stream));
    qry::k_fill_u32<<<div_up(s->n, 256), 256, 0, s->stream>>>(d_dist.p, 0xFFFFFFFFu, s->n);
    if (start < s->n) {
      reb::k_set_u32<<<1, 1, 0, s->stream>>>(d_dist.p + start, 0u);
      reb::k_set_u32<<<1, 1, 0, s->stream>>>(d_fa.p, start);
      uint32_t *hp = reinterpret_cast<uint32_t *>(s->h_pinned);
      uint32_t n_front = 1;
      uint32_t *cur = d_fa.p, *nxt = d_fb.p;
      // one launch and one 4-byte read-back (the size of the next frontier) per level
      for (uint32_t level = 0; n_front != 0 && level < s->n; level++) {
        CUDA_TRY(cudaMemsetAsync(s->misc.p, 0, 4, s->stream));
        const unsigned blocks = std::max(1u, std::min<unsigned>(div_up((uint64_t)n_front * 32, qry::QT), 148 * 16));
        qry::k_bfs_frontier<<<blocks, qry::QT, 0, s->stream>>>(s->dest.p, s->leaf_cnt.p, s->beg.p, s->geo.leaf_shift,
                                                              s->n, d_dist.p, level, cur, n_front, nxt, s->misc.p);
        CUDA_TRY(cudaMemcpyAsync(hp, s->misc.p, 4, cudaMemcpyDeviceToHost, s->stream));
        CUDA_TRY(cudaStreamSynchronize(s->stream));
        n_front = hp[0];
        std::swap(cur, nxt);
      }
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(dist, d_dist.p, (size_t)s->n * 4, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return PPCSR_OK;
  }();
  dev_free(d_dist);
  dev_free(d_fa);
  dev_free(d_fb);
  return rc;
}

// ---- checks and snapshots ---------------------------------------------------------------------------
int ppcsr_check_invariants(ppcsr_shard *s, int check_lower, ppcsr_invariant_report *r) {
  if (!s || !r) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  memset(r, 0, sizeof(*r));
  const Geometry g = s->geo;
  const Geometry want = make_geometry(g.N);
  if ((g.N & (g.N - 1)) != 0 || want.logN != g.logN || want.H != g.H || g.n_leaves != (1u << g.H)) r->bad_geometry = 1;
  DevBuf<qry::InvCounters> d_c;
  PPCSR_TRY(dev_reserve(d_c, 1, s->stream));
  CUDA_TRY(cudaMemsetAsync(d_c.p, 0, sizeof(qry::InvCounters), s->stream));
  const uint32_t L = g.n_leaves;
  qry::k_check_leaves<<<div_up(L, qry::QT), qry::QT, 0, s->stream>>>(s->dest.p, s->val.p, s->leaf_cnt.p, s->tree.p, L,
                                                                    g.leaf_shift, d_c.p);
  qry::k_check_vertices<<<div_up((uint64_t)s->n + 1, qry::QT), qry::QT, 0, s->stream>>>(
      s->dest.p, s->val.p, s->leaf_cnt.p, s->beg.p, s->n, g.N, g.leaf_shift, d_c.p);
  if (L > 1) qry::k_check_tree<<<div_up(L, qry::QT), qry::QT, 0, s->stream>>>(s->tree.p, L, d_c.p);
  if (s->last_sparse) {  // the small-batch path cleared the per-leaf counters: it left the list of touched leaves
    if (s->last_touched)
      sp::k_sp_check_bounds<<<div_up(s->last_touched, sp::ST), sp::ST, 0, s->stream>>>(
          s->tree.p, s->touched.p, s->touched_flags.p, s->last_touched, L, g.logN, (int)g.H, check_lower,
          &d_c.p->bad_upper, &d_c.p->bad_lower);
  } else {
    qry::k_check_bounds<<<div_up(L, qry::QT), qry::QT, 0, s->stream>>>(s->tree.p, s->ins_cnt.p, s->del_cnt.p,
                                                                      s->all_touched, L, g.logN, (int)g.H, check_lower,
                                                                      d_c.p);
  }
  CUDA_TRY(cudaGetLastError());
  qry::InvCounters *hc = reinterpret_cast<qry::InvCounters *>(s->h_pinned);
  CUDA_TRY(cudaMemcpyAsync(hc, d_c.p, sizeof(qry::InvCounters), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  r->bad_sentinel = hc->bad_sentinel + (hc->sentinels != s->n ? 1 : 0);
  r->bad_order = hc->bad_order;
  r->bad_leaf_layout = hc->bad_leaf_layout;
  r->bad_upper = hc->bad_upper;
  r->bad_lower = hc->bad_lower;
  r->bad_tree = hc->bad_tree + (hc->live_items != s->items ? 1 : 0);
  r->live_items = hc->live_items;
  r->edges = hc->live_items - hc->sentinels;
  r->full_leaves = hc->full_leaves;
  dev_free(d_c);
  return PPCSR_OK;
}

int ppcsr_checksum(ppcsr_shard *s, uint64_t vertex_offset, uint64_t out[3]) {
  if (!s || !out) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  out[0] = out[1] = out[2] = 0;
  if (s->n == 0) return PPCSR_OK;
  DevBuf<unsigned long long> d_o;
  PPCSR_TRY(dev_reserve(d_o, 4, s->stream));
  CUDA_TRY(cudaMemsetAsync(d_o.p, 0, 4 * sizeof(unsigned long long), s->stream));
  const unsigned blocks = std::min<unsigned>(div_up(s->geo.N, (uint64_t)qry::QT * 4), 148 * 16);
  qry::k_checksum_leaves<<<blocks, qry::QT, 0, s->stream>>>(s->dest.p, s->val.p, s->leaf_cnt.p, s->beg.p,
                                                           s->geo.leaf_shift, s->n, s->geo.N, vertex_offset, d_o.p);
  qry::k_checksum_nn<<<std::min<unsigned>(div_up(s->n, qry::QT), 148 * 8), qry::QT, 0, s->stream>>>(
      s->nn.p, s->n, vertex_offset, d_o.p);
  CUDA_TRY(cudaGetLastError());
  unsigned long long *hp = reinterpret_cast<unsigned long long *>(s->h_pinned);
  CUDA_TRY(cudaMemcpyAsync(hp, d_o.p, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  for (int k = 0; k < 3; k++) out[k] = hp[k];
  dev_free(d_o);
  return PPCSR_OK;
}

int ppcsr_snapshot(ppcsr_shard *s) {
  if (!s) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  Snapshot &k = s->snap;
  k.geo = s->geo;
  k.n = s->n;
  k.items = s->items;
  PPCSR_TRY(snap_copy(s, k.dest, s->dest, s->geo.N));
  PPCSR_TRY(snap_copy(s, k.val, s->val, s->geo.N));
  PPCSR_TRY(snap_copy(s, k.leaf_cnt, s->leaf_cnt, s->geo.n_leaves));
  PPCSR_TRY(snap_copy(s, k.tree, s->tree, (size_t)2 * s->geo.n_leaves));
  PPCSR_TRY(snap_copy(s, k.beg, s->beg, (size_t)s->n + 1));
  PPCSR_TRY(snap_copy(s, k.nn, s->nn, s->n));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  k.valid = true;
  return PPCSR_OK;
}

int ppcsr_restore(ppcsr_shard *s) {
  if (!s || !s->snap.valid) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  Snapshot &k = s->snap;
  s->geo = k.geo;
  s->n = k.n;
  s->items = k.items;
  PPCSR_TRY(alloc_geometry(s, k.geo));
  PPCSR_TRY(dev_reserve(s->beg, (size_t)k.n + 1, s->stream));
  PPCSR_TRY(dev_reserve(s->nn, (size_t)k.n + 1, s->stream));
  PPCSR_TRY(snap_copy(s, s->dest, k.dest, k.geo.N));
  PPCSR_TRY(snap_copy(s, s->val, k.val, k.geo.N));
  PPCSR_TRY(snap_copy(s, s->leaf_cnt, k.leaf_cnt, k.geo.n_leaves));
  PPCSR_TRY(snap_copy(s, s->tree, k.tree, (size_t)2 * k.geo.n_leaves));
  PPCSR_TRY(snap_copy(s, s->beg, k.beg, (size_t)k.n + 1));
  PPCSR_TRY(snap_copy(s, s->nn, k.nn, k.n));
  CUDA_TRY(cudaMemsetAsync(s->ins_cnt.p, 0, (size_t)k.geo.n_leaves * 4, s->stream));
  CUDA_TRY(cudaMemsetAsync(s->del_cnt.p, 0, (size_t)k.geo.n_leaves * 4, s->stream));
  // the restored layout was touched by no batch: the checker must not apply the last batch's flags to it
  s->all_touched = 0;
  s->last_sparse = false;
  s->cnt_clean = false;
  s->last = ppcsr_batch_stats{};
  s->poisoned = false;
  return PPCSR_OK;
}

int ppcsr_debug_dump(ppcsr_shard *s, uint32_t *dest, uint32_t *val, uint32_t *leaf_cnt) {
  if (!s) return PPCSR_ERR_ARG;
  PPCSR_TRY(set_device(s));
  if (dest) CUDA_TRY(cudaMemcpyAsync(dest, s->dest.p, s->geo.N * 4, cudaMemcpyDeviceToHost, s->stream));
  if (val) CUDA_TRY(cudaMemcpyAsync(val, s->val.p, s->geo.N * 4, cudaMemcpyDeviceToHost, s->stream));
  if (leaf_cnt)
    CUDA_TRY(cudaMemcpyAsync(leaf_cnt, s->leaf_cnt.p, (size_t)s->geo.n_leaves * 4, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return PPCSR_OK;
}

int ppcsr_debug_sort_pairs(int device, uint64_t *keys, uint32_t *payload, uint64_t count, int lo_bits, int hi_bits) {
  if (ppcsr_device_count() <= device) return PPCSR_ERR_NO_DEVICE;
  if (count && !keys) return PPCSR_ERR_ARG;
  if (lo_bits < 1 || lo_bits > 32 || hi_bits < 1 || hi_bits > 32) return PPCSR_ERR_ARG;
  if (count == 0) return PPCSR_OK;
  CUDA_TRY(cudaSetDevice(device));
  ppcsr_shard tmp;
  tmp.device = device;
  tmp.stream = nullptr;
  int rc = reserve_batch_arrays(&tmp, count);
  if (rc != PPCSR_OK) return rc;
  CUDA_TRY(cudaMemcpy(tmp.key_a.p, keys, count * 8, cudaMemcpyHostToDevice));
  if (payload) CUDA_TRY(cudaMemcpy(tmp.pay_a.p, payload, count * 4, cudaMemcpyHostToDevice));
  uint64_t *rk;
  uint32_t *rp;
  rc = prim::radix_sort_pairs(&tmp, tmp.key_a.p, payload ? tmp.pay_a.p : nullptr, tmp.key_b.p, tmp.pay_b.p, count,
                              lo_bits, hi_bits, &rk, &rp);
  if (rc == PPCSR_OK) {
    CUDA_TRY(cudaMemcpy(keys, rk, count * 8, cudaMemcpyDeviceToHost));
    if (payload) CUDA_TRY(cudaMemcpy(payload, rp, count * 4, cudaMemcpyDeviceToHost));
  }
  dev_free(tmp.key_a); dev_free(tmp.key_b); dev_free(tmp.pay_a); dev_free(tmp.pay_b);
  dev_free(tmp.ukey); dev_free(tmp.uval); dev_free(tmp.uloc); dev_free(tmp.ucls); dev_free(tmp.ufirst);
  dev_free(tmp.ins_dst); dev_free(tmp.ins_val); dev_free(tmp.ins_pred);
  dev_free(tmp.hist); dev_free(tmp.block_tmp); dev_free(tmp.scan_state); dev_free(tmp.scan_ticket);
  return rc;
}

int ppcsr_debug_exclusive_scan(int device, const uint32_t *in, uint32_t *out, uint64_t count) {
  if (ppcsr_device_count() <= device) return PPCSR_ERR_NO_DEVICE;
  CUDA_TRY(cudaSetDevice(device));
  ppcsr_shard tmp;
  tmp.device = device;
  tmp.stream = nullptr;
  DevBuf<uint32_t> a, b;
  PPCSR_TRY(dev_reserve(a, count + 1, nullptr));
  PPCSR_TRY(dev_reserve(b, count + 1, nullptr));
  CUDA_TRY(cudaMemset(b.p, 0, (count + 1) * 4));
  if (count) CUDA_TRY(cudaMemcpy(a.p, in, count * 4, cudaMemcpyHostToDevice));
  int rc = prim::device_scan(&tmp, prim::InArray{a.p}, prim::OutPrefixWithTotal{b.p, (size_t)count}, count, nullptr,
                             nullptr);
  if (rc == PPCSR_OK) CUDA_TRY(cudaMemcpy(out, b.p, (count + 1) * 4, cudaMemcpyDeviceToHost));
  dev_free(a); dev_free(b); dev_free(tmp.block_tmp); dev_free(tmp.scan_state); dev_free(tmp.scan_ticket);
  return rc;
}

#include "group.inl"

}  // extern "C"
