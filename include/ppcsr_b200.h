/*
 * ppcsr_b200.h -- C-ABI of the B200-native Parallel Packed CSR edge-update engine.
 *
 * This is the drop-in boundary for the hot path named by BASELINE.json:north_star.  The reference
 * (domargan/parallel-packed-csr) has no FFI layer: its boundary is the C++ class surface
 *   PCSR            reference src/pcsr/PCSR.h:64-124
 *   PPPCSR          reference src/pppcsr/PPPCSR.h:11-60
 *   ThreadPool      reference src/thread_pool/thread_pool.h:17-40
 *   ThreadPoolPPPCSR reference src/thread_pool_pppcsr/thread_pool_pppcsr.h:17-47
 * and `parallel-packed-csr_b200/host/` re-implements exactly those classes on top of the entry points
 * below (see INTEGRATION.md for the binding a maintainer of the reference would add).
 *
 * One handle = one shard = one PCSR instance living in the HBM of one GPU.  All functions return 0 on
 * success and a negative ppcsr_status on failure; ppcsr_last_error() gives the message.  Plain
 * pointers and sizes only.  A handle is NOT thread-safe: one in-flight batch per shard (the reference's
 * submit_* calls are single-threaded as well, reference src/main.cpp:68-82).
 *
 * Conventions shared by the batch entry points
 *   - an update is (src, dst, val): val != 0 inserts/overwrites the edge with that value
 *     (reference PCSR::add_edge, src/pcsr/PCSR.cpp:706,1374-1445); val == 0 removes it
 *     (reference PCSR::remove_edge, src/pcsr/PCSR.cpp:709-773).  `val == NULL` means "all `default_val`".
 *   - a batch is applied in array order with last-op-wins per (src,dst), i.e. the result of the
 *     reference run with -threads=1 on the same stream.
 *   - inserts with src >= n are ignored (reference PCSR.cpp:1375); dst is not range checked except
 *     that dst == 0xFFFFFFFF is rejected (it is the sentinel marker, reference PCSR.h:32, PCSR.cpp:64).
 *   - num_neighbors follows the reference's call-count semantics: +1 per accepted add call, -1 per
 *     remove call, duplicates and misses included (reference PCSR.cpp:1392,747).
 *
 * Failure atomicity of a batch: everything a batch can need in the worst case (every update a new edge: the grown
 * array, trees, scratch) is allocated BEFORE the shard is modified, so PPCSR_ERR_CAPACITY from an apply_* / submit /
 * wait / add_nodes call normally means "nothing was applied, the handle is intact".  The exception is the 2^31-slot
 * limit, which can only be decided after duplicates have been resolved: a batch that hits it after it has begun leaves
 * the handle POISONED -- every further update returns PPCSR_ERR_CAPACITY until ppcsr_restore() brings back a snapshot
 * (or the handle is destroyed).  PPCSR_ERR_CUDA is always fatal for the handle.
 */
#ifndef PPCSR_B200_H
#define PPCSR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ppcsr_shard ppcsr_shard; /* opaque; owns all device memory of one shard */

typedef enum {
  PPCSR_OK = 0,
  PPCSR_ERR_CUDA = -1,     /* a CUDA runtime call failed (fatal for the handle) */
  PPCSR_ERR_ARG = -2,      /* bad argument */
  PPCSR_ERR_CAPACITY = -3, /* slot count would exceed 2^31 or allocation failed (see "Failure atomicity" below) */
  PPCSR_ERR_NO_DEVICE = -4 /* no CUDA device: there is NO CPU fallback */
} ppcsr_status;

/* Geometry exactly as reference PCSR::resizeEdgeArray computes it (src/pcsr/PCSR.cpp:68-73). */
typedef struct {
  uint64_t N;       /* slots, power of two                       (edge_list_t::N)    */
  uint32_t logN;    /* leaf size = 1 << bsr(2*bsr(N)+1)          (edge_list_t::logN) */
  uint32_t H;       /* tree height = bsr(N/logN)                 (edge_list_t::H)    */
  uint64_t n;       /* vertices                                  (PCSR::get_n)       */
  uint64_t items;   /* live slots = edges + one sentinel per vertex                  */
} ppcsr_geometry;

/* What one batch did.  Byte counts are ALGORITHMIC bytes (SURVEY.md §8d) at this build's slot size
 * of 8 B (SoA: u32 dest + u32 value; the reference's 12-B edge_t also stores src, which is implied by
 * the sentinel order here). */
typedef struct {
  uint64_t batch_size;     /* updates submitted                                              */
  uint64_t n_ignored;      /* inserts with src >= n or dst == 0xFFFFFFFF, removes with src >= n */
  uint64_t n_unique;       /* distinct (src,dst) keys after last-op-wins                     */
  uint64_t n_inserted;     /* new edges                                                      */
  uint64_t n_overwritten;  /* inserts that hit an existing edge (value replaced)             */
  uint64_t n_deleted;      /* removes that found their edge                                  */
  uint64_t n_not_found;    /* removes of absent edges (the reference prints "not found s d") */
  uint64_t n_windows;      /* disjoint rebalance windows chosen (1 if the whole array was rebuilt) */
  uint64_t window_slots;   /* sum of window lengths in slots (resize: N_before + N_after)/2 .. see DESIGN.md */
  uint64_t rebalance_bytes;/* algorithmic bytes of the rebalance: sum 2*len*8 (+8 per moved sentinel) */
  uint64_t slots_before;   /* N before the batch                                             */
  uint64_t slots_after;    /* N after the batch (doubling / halving folded into the same pass) */
  uint32_t resized;        /* 1 grew, 2 shrank, 0 unchanged                                  */
  uint32_t whole_array;    /* 1 if the batch was applied as one root window                  */
  float ms_total;          /* device time of the whole pipeline (CUDA events on the shard stream) */
  float ms_sort;           /* key build + radix sort + last-op-wins                          */
  float ms_locate;         /* segmented search + per-leaf counts                             */
  float ms_select;         /* count tree + bottom-up window selection                        */
  float ms_rebalance;      /* scan + scatter rebalance (+ copy back for multi-CTA windows)   */
  float ms_rebalance_kernel; /* the k_rebalance launch alone (roofline numerator: rebalance_bytes / this) */
  uint32_t kernel_launches;  /* kernels launched for this batch                                */
  uint32_t sparse_path;      /* 1 if the batch took the small-batch path (O(touched leaves) work, one host sync) */
} ppcsr_batch_stats;

typedef struct {
  uint64_t bad_geometry;     /* I1 */
  uint64_t bad_sentinel;     /* I2: beg[v] does not hold v's sentinel / ranges not contiguous */
  uint64_t bad_order;        /* I3: neighbours not strictly ascending                     */
  uint64_t bad_leaf_layout;  /* leaf not left-packed / count mismatch / tail not null     */
  uint64_t bad_upper;        /* I4: tree nodes at or above their upper density bound      */
  uint64_t bad_lower;        /* I5: tree nodes below their lower bound (only meaningful after deletes) */
  uint64_t bad_tree;         /* count tree inconsistent with the leaves                   */
  uint64_t live_items;       /* I6: must equal edges + n                                  */
  uint64_t edges;
  uint64_t full_leaves;      /* leaves left 100% full (must be 0)                         */
} ppcsr_invariant_report;

const char *ppcsr_last_error(void);
int ppcsr_device_count(void);

/* ---- lifetime: reference PCSR::PCSR(init_n, src_n, lock_search, domain), src/pcsr/PCSR.cpp:775-838 ---- */
/* Creates a shard with src_n vertices on CUDA device `device`; initial N = 2 << bsr(max(init_n+src_n,1024)). */
int ppcsr_create(uint32_t init_n, uint32_t src_n, int device, ppcsr_shard **out);
void ppcsr_destroy(ppcsr_shard *h); /* reference PCSR::~PCSR, src/pcsr/PCSR.cpp:840-851 */
/* Use an external CUDA stream (cudaStream_t) for all work of this shard; NULL = the shard's own stream. */
int ppcsr_set_stream(ppcsr_shard *h, void *cuda_stream);
int ppcsr_sync(ppcsr_shard *h);
/* Pre-allocate buffers so that batches up to `max_batch` updates and arrays up to `max_slots` slots need
 * no allocation inside a timed region. */
int ppcsr_reserve(ppcsr_shard *h, uint64_t max_slots, uint64_t max_batch);

/* ---- the hot path: batched add_edge / remove_edge ---- */
/* Host buffers (pageable or pinned).  Replaces the ThreadPool start()/stop() region
 * (reference src/thread_pool/thread_pool.cpp:78-113) for the queued tasks. */
int ppcsr_apply_batch(ppcsr_shard *h, const uint32_t *src, const uint32_t *dst, const uint32_t *val,
                      uint64_t count, uint32_t default_val, ppcsr_batch_stats *stats);
/* Same, buffers already resident in this shard's device memory (not modified). */
int ppcsr_apply_batch_device(ppcsr_shard *h, const uint32_t *d_src, const uint32_t *d_dst, const uint32_t *d_val,
                             uint64_t count, uint32_t default_val, ppcsr_batch_stats *stats);
/* Pipelined form of ppcsr_apply_batch for a stream of batches (replaces a sequence of ThreadPool start()/stop()
 * regions, reference src/thread_pool/thread_pool.cpp:78-113): ppcsr_submit_batch starts the host->device copy of the
 * batch into one of TWO staging slots on a copy stream and returns at once with a ticket; ppcsr_wait(ticket) applies
 * that batch (after its copy) and returns its stats.  With
 *     submit(b0); for i: { submit(b[i+1]); wait(b[i]); }
 * the copy of batch i+1 runs under the compute of batch i.  At most two batches in flight; batches are applied in
 * submission order (wait for the older ticket first).  The host buffers must stay valid until the matching
 * ppcsr_wait returns; they should be page-locked (cudaHostAlloc / cudaHostRegister) -- a pageable buffer makes the
 * submit itself block for the duration of the copy. */
int ppcsr_submit_batch(ppcsr_shard *h, const uint32_t *src, const uint32_t *dst, const uint32_t *val, uint64_t count,
                       uint32_t default_val, uint64_t *ticket);
int ppcsr_wait(ppcsr_shard *h, uint64_t ticket, ppcsr_batch_stats *stats);
/* ---- input path (reference src/main.cpp:29-62, read_input) ---- */
/* Binary edge file: `count` interleaved little-endian (src, dst) u32 pairs (host memory, e.g. an mmap'd file), every
 * update with value `default_val` (0 = remove).  Same result as ppcsr_apply_batch on the de-interleaved arrays. */
int ppcsr_apply_batch_pairs(ppcsr_shard *h, const uint32_t *pairs, uint64_t count, uint32_t default_val,
                            ppcsr_batch_stats *stats);
/* Text edge list parsed ON THE GPU with the reference reader's rules: one edge per line `src<1 char>dst[<1 char>op]`,
 * op '1' = add (value 1), '0' = remove (value 0), absent = default_val.  `text` is host memory (the raw file bytes).
 * Outputs DEVICE arrays of *count entries (one per line; free them with ppcsr_free_device) that feed
 * ppcsr_apply_batch_device directly; lines without a parsable pair come out as (0xFFFFFFFF, 0xFFFFFFFF), which every
 * batch entry point ignores.  *n_parsed = lines that parsed, *max_id = largest vertex id seen (reference
 * main.cpp:44,145,155: n = max id + 1 over both files). */
int ppcsr_parse_edge_list(int device, const char *text, uint64_t bytes, uint32_t default_val, uint32_t **d_src,
                          uint32_t **d_dst, uint32_t **d_val, uint64_t *count, uint64_t *n_parsed, uint32_t *max_id);
int ppcsr_free_device(int device, void *p);
int ppcsr_copy_to_host(int device, void *host, const void *dev, uint64_t bytes);

/* Single operations = batches of one (reference PCSR::add_edge / remove_edge). Correctness path, slow. */
int ppcsr_add_edge(ppcsr_shard *h, uint32_t src, uint32_t dst, uint32_t value);
int ppcsr_remove_edge(ppcsr_shard *h, uint32_t src, uint32_t dst, int *found);
/* How a batch that leaves the root within its bounds is rebalanced: 0 (default) = cost model -- a list of disjoint
 * windows, or ONE root window (the whole array streamed once) when that is cheaper; -1 = always the window list;
 * 1 = always the root window.  Does not change results, only the physical layout (tests run both paths). */
int ppcsr_set_whole_array_policy(ppcsr_shard *h, int mode);
/* reference PCSR::add_node (src/pcsr/PCSR.cpp:681-703): appends `count` vertices after the last one. */
int ppcsr_add_nodes(ppcsr_shard *h, uint32_t count);
/* Every edge out of or into the listed vertices removed (host ids < n); the vertices stay, without edges.  The result
 * is that of ONE remove batch holding exactly the live edges (u, w) with u or w in the set (reference
 * PCSR::remove_edge per edge, src/pcsr/PCSR.cpp:709-773): num_neighbors[u] drops by one per removed edge out of u (an
 * isolated vertex keeps its old value minus its degree), edges to ids >= n are removed only with their source, n and
 * the sentinels do not change.  For a shard holding the whole graph (as ppcsr_bfs): ids are that shard's vertex ids.
 * Found on the device in one pass over the packed array (no edge reaches the host), then window selection and
 * rebalance as after a batch.  Duplicate ids are allowed; count == 0 is a no-op with zeroed stats.  An id >= n returns
 * PPCSR_ERR_ARG and a poisoned handle PPCSR_ERR_CAPACITY, both with nothing changed; everything the call needs (n / 8 B
 * of bitmap and the id list, freed at the end, plus what a batch of removes needs) is allocated before the shard is
 * modified, so PPCSR_ERR_CAPACITY also means "nothing removed".  A failure in the rebalance poisons the handle, as a
 * batch does.  Stats (nullable; ppcsr_last_stats returns the same) as for a batch: batch_size = ids passed, n_unique =
 * distinct ids, n_deleted = edges removed, the window / resize / rebalance fields as usual; ms_sort times the copy of
 * the ids and the bitmap build, ms_locate the filter pass over the array.  A snapshot stays valid: ppcsr_restore
 * brings back the graph before the isolation. */
int ppcsr_isolate_vertices(ppcsr_shard *h, const uint32_t *ids, uint64_t count, ppcsr_batch_stats *stats);
int ppcsr_last_stats(ppcsr_shard *h, ppcsr_batch_stats *stats);

/* ---- change capture: what each batch changed, left on the device ----
 * Off by default, per shard; while it is off a batch runs exactly as without this feature (same kernels, no extra
 * allocation, launch or host synchronisation).  While it is on, every batch -- ppcsr_apply_batch[_device|_pairs|
 * _packed_device|_segments_device], ppcsr_wait, ppcsr_group_apply / ppcsr_group_wait on each shard, ppcsr_add_edge /
 * ppcsr_remove_edge (batches of one) -- leaves two lists in the shard's device memory, valid until the next call that
 * modifies the shard:
 *   changes    one entry per key whose state the batch changed, ascending (src, dst); src is shard-local.  old_val = 0:
 *              absent before the batch (inserted); new_val = 0: absent after it (deleted); both non-zero: overwritten,
 *              also with the same value.  A key absent before and after (e.g. insert then remove of a new edge) is not
 *              listed.  n_changes = n_inserted + n_overwritten + n_deleted of the batch's stats, per kind as well.
 *   not found  one (src, dst) per remove CALL that missed under the sequential rule of n_not_found (a remove of an
 *              absent edge, or right after a remove of the same key), ascending, a key repeated once per miss:
 *              n_not_found entries, as a multiset the `not found s d` lines the reference prints at -threads=1
 *              (reference PCSR.cpp:751).
 * Ignored updates (src >= n, dst == 0xFFFFFFFF) appear in neither list.  Both lists are empty after a failed call
 * (any status), an empty batch, and every modifying call that is not a batch: ppcsr_isolate_vertices /
 * ppcsr_group_isolate_vertices, ppcsr_load_csr, ppcsr_add_nodes, ppcsr_restore, ppcsr_group_repartition.
 * Applying (src, dst, val = old_val) of the changes as one batch restores the edges and values before the batch (not
 * num_neighbors, which keeps its call-count meaning).
 * Memory while on: about 29 B per update of the largest batch (a kind byte and an old value per update, 16 B per
 * change entry and 8 B per not-found entry, each list bounded by the batch), reserved with the batch's other worst-case
 * buffers before the shard is modified, so PPCSR_ERR_CAPACITY still means "nothing applied".  Turning capture off
 * frees it. */
int ppcsr_set_change_capture(ppcsr_shard *h, int on);
typedef struct {
  const uint32_t *src, *dst, *old_val, *new_val; /* DEVICE pointers on `device`, n_changes entries each (NULL if 0) */
  uint64_t n_changes;
  const uint32_t *nf_src, *nf_dst;               /* DEVICE pointers, n_not_found entries each (NULL if 0)           */
  uint64_t n_not_found;
  int device;
} ppcsr_changes;
/* The lists of the last batch (PPCSR_ERR_ARG while capture is off).  The pointers belong to the shard: read them with
 * ppcsr_copy_to_host or on the device, and copy them before passing them back into the same shard -- the next batch
 * may reallocate or overwrite them. */
int ppcsr_last_changes(ppcsr_shard *h, ppcsr_changes *out);

/* ---- multi-GPU routing helper (reference PPPCSR::get_partiton, src/pppcsr/PPPCSR.cpp:58-66) ---- */
/* Bins `count` device-resident updates by owning shard: shard p owns sources [starts[p], starts[p+1]).
 * Writes the updates grouped by owner (stable) with src made shard-local (src - starts[owner],
 * reference PPPCSR.cpp:46-52) and the per-owner counts.  All pointers are device pointers on `device`
 * except h_counts (host, n_parts entries).  d_val / d_out_val may be NULL. */
int ppcsr_bin_by_owner(int device, void *cuda_stream, const uint64_t *d_starts, uint32_t n_parts,
                       const uint32_t *d_src, const uint32_t *d_dst, const uint32_t *d_val, uint64_t count,
                       uint32_t *d_out_src, uint32_t *d_out_dst, uint32_t *d_out_val, uint64_t *h_counts);

/* Same binning, but emits the packed 64-bit records (local_src << 32 | dst) that travel through the all-to-all
 * and that ppcsr_apply_batch_packed_device consumes directly. */
int ppcsr_bin_by_owner_packed(int device, void *cuda_stream, const uint64_t *d_starts, uint32_t n_parts,
                              const uint32_t *d_src, const uint32_t *d_dst, const uint32_t *d_val, uint64_t count,
                              uint64_t *d_out_packed, uint32_t *d_out_val, uint64_t *h_counts);
/* Routing fused with the exchange (NVLink / NVSwitch peer memory): bins the batch by owner like
 * ppcsr_bin_by_owner_packed, but every packed record is stored straight into the OWNING GPU's receive buffer.
 * h_peer_rec / h_peer_val / h_peer_cnt are HOST arrays of n_parts device pointers (one per rank, peer-mapped, e.g.
 * the buffer_ptrs of a symmetric allocation): rank r's receive buffer holds n_parts regions of `region_cap` records,
 * region s written by sender s; its count array holds n_parts u64 counts, entry s written by sender s.  No host
 * synchronisation; the caller runs a cross-GPU barrier on the same stream before the owners read their buffers.
 * Replaces the hand-over of reference ThreadPoolPPPCSR::submit_* (src/thread_pool_pppcsr/thread_pool_pppcsr.cpp:96-118). */
int ppcsr_bin_to_peers(int device, void *cuda_stream, const uint64_t *d_starts, uint32_t n_parts, uint32_t my_rank,
                       const uint32_t *d_src, const uint32_t *d_dst, const uint32_t *d_val, uint64_t count,
                       const uint64_t *h_peer_rec, const uint64_t *h_peer_val, const uint64_t *h_peer_cnt,
                       uint64_t region_cap);
/* Applies what the peers deposited: `n_segments` regions of `region_cap` packed records at d_packed (values at d_val,
 * nullable), region r holding d_counts[r] valid records.  d_counts is a DEVICE array (the senders wrote it): the
 * batch size reaches the host together with the sort width, so the exchange adds no host synchronisation.
 * max_total (0 = n_segments * region_cap) bounds the total for the allocation of the key array. */
int ppcsr_apply_batch_segments_device(ppcsr_shard *h, const uint64_t *d_packed, const uint32_t *d_val,
                                      uint64_t region_cap, const uint64_t *d_counts, uint32_t n_segments,
                                      uint64_t max_total, uint32_t default_val, ppcsr_batch_stats *stats);
/* Applies a device-resident batch of packed records (src << 32 | dst), e.g. what the all-to-all delivered. */
int ppcsr_apply_batch_packed_device(ppcsr_shard *h, const uint64_t *d_packed, const uint32_t *d_val, uint64_t count,
                                    uint32_t default_val, ppcsr_batch_stats *stats);

/* ---- several shards on several GPUs driven by ONE process: reference PPPCSR + ThreadPoolPPPCSR
 *      (src/pppcsr/PPPCSR.cpp:13-66, src/thread_pool_pppcsr/thread_pool_pppcsr.cpp:96-118) ---- */
typedef struct ppcsr_group ppcsr_group;
/* shards[r] (already created, on any devices that can address each other) owns the global vertices
 * [starts[r], starts[r+1]); region_cap = the largest batch / n_shards the group will route (records per sender and
 * receiver); with_values != 0 if batches carry per-update values. */
int ppcsr_group_create(ppcsr_shard **shards, uint32_t n_shards, const uint64_t *starts, uint64_t region_cap,
                       int with_values, ppcsr_group **out);
void ppcsr_group_destroy(ppcsr_group *g); /* the shards stay alive */
uint32_t ppcsr_group_owner(const ppcsr_group *g, uint64_t vertex); /* reference PPPCSR::get_partiton */
/* One batch of GLOBAL updates in host memory: slice r of the batch is copied to GPU r (all PCIe links at once), binned
 * there by owner and stored straight into the owners' receive buffers over NVLink peer memory (ppcsr_bin_to_peers),
 * then every shard applies what it received.  stats (nullable) gets one entry per shard. */
int ppcsr_group_apply(ppcsr_group *g, const uint32_t *src, const uint32_t *dst, const uint32_t *val, uint64_t count,
                      uint32_t default_val, ppcsr_batch_stats *stats);
/* Pipelined form of ppcsr_group_apply for a stream of batches (replaces a sequence of ThreadPoolPPPCSR start()/stop()
 * regions): ppcsr_group_submit starts the host->device copy of every slice (cut as ppcsr_group_apply cuts it) and
 * enqueues its binning and peer stores on the sending shard's copy stream, then returns at once with a ticket -- no
 * host synchronisation; ppcsr_group_wait(ticket) makes every shard apply what it received
 * (ppcsr_apply_batch_segments_device, one host thread per shard) and returns the per-shard stats (n_shards entries,
 * nullable).  With
 *     submit(b0); for i: { submit(b[i+1]); wait(b[i]); }
 * the copy and routing of batch i+1 run on the devices while the shards apply batch i, and the graph, num_neighbors
 * and per-shard counters are exactly those of ppcsr_group_apply(b0); ppcsr_group_apply(b1); ...  Global ids, values,
 * default_val and the with_values rule are those of ppcsr_group_apply.  At most two batches in flight, applied in
 * submission order: a third submit, a wait for the newer ticket first or for an unknown ticket return PPCSR_ERR_ARG.
 * The host buffers must stay valid until the matching wait returns; they should be page-locked.  A slice above
 * region_cap or a failed allocation returns PPCSR_ERR_CAPACITY with nothing in flight: everything the routing needs
 * is allocated in submit.  A failing wait reports the first failing shard, as ppcsr_group_apply does; the other batch
 * in flight stays valid and is applied by its own wait.  While a batch is in flight, ppcsr_group_apply,
 * ppcsr_group_bfs, ppcsr_group_pagerank, ppcsr_group_repartition and ppcsr_group_isolate_vertices return PPCSR_ERR_ARG
 * and change nothing, and the
 * group's shards must not be modified through shard-level calls; ppcsr_group_destroy synchronises and frees the
 * batches in flight without applying them.  Ordering: a streamed batch is ordered after the group's last apply,
 * traversal or repartition and before the next, also when the shards run on external streams (ppcsr_set_stream).
 * Device memory, allocated on the first submit and kept until ppcsr_group_destroy: per receiver a second receive set,
 * n_shards * region_cap * (8 [+ 4 with values]) B plus n_shards * 8 B of counts; per sender two staging slots of its
 * slice, 2 * slice * (8 [+ 4 with values]) B.  A group that only uses ppcsr_group_apply allocates none of it. */
int ppcsr_group_submit(ppcsr_group *g, const uint32_t *src, const uint32_t *dst, const uint32_t *val, uint64_t count,
                       uint32_t default_val, uint64_t *ticket);
int ppcsr_group_wait(ppcsr_group *g, uint64_t ticket, ppcsr_batch_stats *stats);
/* Traversals across all shards of the group, on the devices.  n = starts[n_shards-1] + (vertices of the last shard
 * now): the last shard may have grown through ppcsr_add_nodes (PPPCSR::add_node appends there); if any other shard no
 * longer holds exactly its range, both calls return PPCSR_ERR_ARG.  All work of shard r runs on shard r's stream, the
 * shards wait for each other through events: a traversal is ordered after the group's last ppcsr_group_apply and
 * before the next one.  A traversal modifies no shard.
 * Device memory the group keeps for traversals (allocated on first use, reallocated when n changes, freed by
 * ppcsr_group_destroy), per shard r with n_r vertices:
 *   BFS       n_shards * n_r * 4 B of inbox + n / 8 B of bitmap + 3 * n_r * 4 B of distances and frontier queues
 *   PageRank  n * 8 B of accumulator + n_r * 8 B of ranks
 * reference src/utility/bfs.h:15-36 over all shards of the group: dist[n] (host), UINT32_MAX = unreached,
 * start >= n leaves every vertex unreached.  Same result as ppcsr_bfs on one shard holding the graph. */
int ppcsr_group_bfs(ppcsr_group *g, uint32_t start, uint32_t *dist);
/* ppcsr_pagerank's recurrence over all shards of the group (n = n_global, divisor num_neighbors, no dangling
 * redistribution), out[n] on the host; iterations == 0 gives 1/n everywhere.  No host round trip between iterations. */
int ppcsr_group_pagerank(ppcsr_group *g, uint32_t iterations, double damping, double *out);

/* What one ppcsr_group_repartition did. */
typedef struct {
  uint64_t vertices_moved;  /* vertices whose owner changed                                 */
  uint64_t edges_moved;     /* their out-edges                                              */
  uint64_t bytes_copied;    /* bytes copied from one shard's buffers to another's (peer or
                               same device): col + val + num_neighbors + rowptr of the moved
                               vertices                                                     */
  uint32_t shards_rebuilt;  /* shards whose vertex range changed                            */
  float ms_total;           /* host clock around the call, ending after a device synchronise */
} ppcsr_repartition_stats;
/* Moves vertex ranges between the shards of the group: afterwards shard r owns the global vertices
 * [new_starts[r], new_starts[r+1]).  Every vertex whose owner changes goes to its new shard with all its out-edges
 * (dst >= n included), their values and its num_neighbors; the logical graph is unchanged.  The data moves device to
 * device (peer memory across GPUs), never through the host.  new_starts has n_shards + 1 entries: new_starts[0] = 0,
 * new_starts[n_shards] = n (the first vertex of the last shard + its current vertex count: the vertices the last shard
 * gained through ppcsr_add_nodes can be spread out this way), each entry strictly larger than the one before.  Every
 * shard whose range changes is rebuilt whole from a CSR of its new range (a root-window layout, DESIGN.md §5b): its
 * ppcsr_last_stats then describes that rebuild (whole_array = 1, rebalance_bytes / ms_rebalance_kernel = the layout
 * pass) and its snapshot is invalidated.  Shards whose range stays the same are not touched; identical boundaries
 * rebuild nothing.  PPCSR_ERR_ARG, with nothing changed: bad boundaries, a shard other than the last that no longer
 * holds exactly its range, a poisoned shard, a submitted batch not yet waited for.  Every allocation happens before any
 * shard is modified, so PPCSR_ERR_CAPACITY (a shard would pass 2^31 slots, or device memory ran out) also means
 * "nothing moved".  PPCSR_ERR_CUDA (fatal, as everywhere) during the build phase leaves the rebuilt shards POISONED:
 * they then hold neither their old nor their new ranges.  Transient device memory per rebuilt shard of E edges, n vertices and N slots after the call: the
 * export of its old range and the CSR of its new one, about 2 * (8 E + 12 n) bytes, plus the out-of-place slot
 * arrays at N (8 N bytes, kept by the shard as it keeps them after a resize).  The traversal buffers of the group
 * are freed (their sizes depend on the ranges).  Ordered after the group's last apply or traversal, before the next;
 * stats nullable. */
int ppcsr_group_repartition(ppcsr_group *g, const uint64_t *new_starts, ppcsr_repartition_stats *stats);
/* ppcsr_isolate_vertices over all shards of the group: GLOBAL ids < n (n counted as the traversals count it; a shard
 * other than the last that no longer holds exactly its range gives PPCSR_ERR_ARG).  Every shard filters its own array
 * with a bitmap of the n global ids on its device (n / 8 B each, freed at the end; only the id list is copied to each
 * device, no edge crosses shards): the out-edges of a vertex are removed at its owner, its in-edges wherever they are.
 * Checks and allocations for every shard come first, so PPCSR_ERR_ARG (bad id, a submitted batch in flight) and
 * PPCSR_ERR_CAPACITY (a poisoned shard, no memory) leave the whole group unchanged.  Each shard then runs on its own
 * host thread, ordered after the group's last apply, traversal or repartition, and before the next routed batch, also
 * on external streams.  A failing shard is reported as ppcsr_group_apply reports one.  stats (nullable): one entry per
 * shard, its n_deleted the edges removed from that shard. */
int ppcsr_group_isolate_vertices(ppcsr_group *g, const uint32_t *ids, uint64_t count, ppcsr_batch_stats *stats);

/* ---- reads ---- */
int ppcsr_geometry_of(ppcsr_shard *h, ppcsr_geometry *out);
/* reference PCSR::edge_exists (src/pcsr/PCSR.cpp:860-869); `out_value` (nullable) gets the stored value. */
int ppcsr_edge_exists(ppcsr_shard *h, uint32_t src, uint32_t dst, int *exists, uint32_t *out_value);
/* Batched point queries, host buffers: exists[i] = 1/0. */
int ppcsr_edges_exist(ppcsr_shard *h, const uint32_t *src, const uint32_t *dst, uint64_t count, uint8_t *exists);
/* reference PCSR::get_neighbourhood (src/pcsr/PCSR.cpp:901-912): ascending dests of v into out[0..cap);
 * *count gets the degree even if it exceeds cap. */
int ppcsr_neighbours(ppcsr_shard *h, uint32_t v, uint32_t *out, uint64_t cap, uint64_t *count);
/* reference PCSR::read_neighbourhood (src/pcsr/PCSR.cpp:892-899): touch-only scan; returns a checksum. */
int ppcsr_read_neighbourhood(ppcsr_shard *h, uint32_t v, uint64_t *checksum);
/* getNode(v).num_neighbors for all v (host buffer of n entries). */
int ppcsr_num_neighbors(ppcsr_shard *h, uint32_t *out);
/* getNode(v).{beginning,end} for all v: beg has n entries, end has n entries (last end = N-1). */
int ppcsr_node_ranges(ppcsr_shard *h, uint32_t *beginning, uint32_t *end);
/* Compacted adjacency (the logical graph): rowptr[n+1], then col/val with *edges entries.  Call with
 * col == NULL to size.  Doubles as the snapshot/export of SURVEY.md §5. */
int ppcsr_export_csr(ppcsr_shard *h, uint64_t *rowptr, uint32_t *col, uint32_t *val, uint64_t *edges);
/* The inverse: replaces the shard's whole content with the CSR of n vertices (host buffers): rowptr[n+1], col / val
 * [rowptr[n]] (val NULL: every value 1), nn[n] the num_neighbors (NULL: the row lengths).  The shard is laid out
 * afresh, as a root-window rebuild would leave it, at the slot count the density bounds give from its current N.  The
 * input is validated on the device -- rowptr[0] = 0 and non-decreasing, col strictly ascending within a row and never
 * 0xFFFFFFFF, no value 0 -- and PPCSR_ERR_ARG leaves the shard untouched (as it does for a poisoned shard or a
 * submitted batch not yet waited for).  Needs no sort: an exported graph loads in one streaming pass.
 * ppcsr_last_stats describes the layout pass. */
int ppcsr_load_csr(ppcsr_shard *h, uint32_t n, const uint64_t *rowptr, const uint32_t *col, const uint32_t *val,
                   const uint32_t *nn);
/* One PageRank push step, reference src/utility/pagerank.h:16-29: out[dst] += in[v] / num_neighbors[v].
 * `out_len` entries of out are zeroed then accumulated (dst >= out_len is skipped; the reference would
 * write out of bounds).  Accumulation is fp64 on device.  Host buffers. */
int ppcsr_pagerank_step_f64(ppcsr_shard *h, const double *in, double *out, uint64_t out_len);
int ppcsr_pagerank_step_f32(ppcsr_shard *h, const float *in, float *out, uint64_t out_len);
/* Device-buffer variant used by the multi-GPU path: accumulates (no zeroing) into d_out[out_len] fp64;
 * `d_in` is indexed by shard-local vertex. */
int ppcsr_pagerank_push_device(ppcsr_shard *h, const double *d_in, double *d_out, uint64_t out_len);
/* Iterated PageRank with damping on one shard holding the whole graph (SURVEY.md §8f rank 2): `iterations` push steps
 * of the reference's kernel (src/utility/pagerank.h:16-29, divisor num_neighbors) kept on the device,
 *     r_0 = 1/n,   r_{t+1}[v] = (1 - damping)/n + damping * sum_{(u,v)} r_t[u] / num_neighbors[u],
 * out[n] on the host.  No host round trip between the steps. */
int ppcsr_pagerank(ppcsr_shard *h, uint32_t iterations, double damping, double *out);
/* reference src/utility/bfs.h:15-36 on one shard holding the whole graph: dist[n], UINT32_MAX = unreached. */
int ppcsr_bfs(ppcsr_shard *h, uint32_t start, uint32_t *dist);

/* ---- checks and snapshots ---- */
/* PMA invariants I1-I6 (SURVEY.md §8a).  `check_lower` != 0 also counts lower-bound violations. */
int ppcsr_check_invariants(ppcsr_shard *h, int check_lower, ppcsr_invariant_report *report);
/* Order-independent checksum of the logical graph: out[0] = edges, out[1] = sum (mod 2^64) of
 * mix64((vertex_offset + src) << 32 | dst) over all edges, out[2] = sum of num_neighbors[v] * mix64(vertex_offset + v)
 * (mix64 = the splitmix64 finaliser).  Sums of several shards add up to the checksum of the whole graph when
 * vertex_offset is the shard's first global vertex (reference PPPCSR.cpp:46-52).  The parity anchor at sizes where
 * per-vertex get_neighbourhood dumps (reference PCSR.cpp:901-912) are impractical. */
int ppcsr_checksum(ppcsr_shard *h, uint64_t vertex_offset, uint64_t out[3]);
/* Device-side copy of the whole shard state (arrays + geometry); restore makes the shard identical
 * to the snapshot again.  One snapshot per shard. */
int ppcsr_snapshot(ppcsr_shard *h);
int ppcsr_restore(ppcsr_shard *h);
/* Raw physical state for debugging/tests: dest[N], val[N], leaf_cnt[N/logN] (host buffers, nullable). */
int ppcsr_debug_dump(ppcsr_shard *h, uint32_t *dest, uint32_t *val, uint32_t *leaf_cnt);

/* ---- primitives exposed for unit tests (host buffers, in place) ---- */
/* Stable LSD radix sort of (key, payload) pairs by key bits [0,lo_bits) and [32,32+hi_bits), 1 <= lo_bits, hi_bits
 * <= 32.  payload == NULL sorts the keys alone (the keys-only passes the batch pipeline runs when the values need no
 * sorting). */
int ppcsr_debug_sort_pairs(int device, uint64_t *keys, uint32_t *payload, uint64_t count, int lo_bits, int hi_bits);
/* out[i] = sum of in[0..i), out[count] = total (out has count+1 entries). */
int ppcsr_debug_exclusive_scan(int device, const uint32_t *in, uint32_t *out, uint64_t count);

#ifdef __cplusplus
}
#endif
#endif /* PPCSR_B200_H */
