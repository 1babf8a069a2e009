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
int ppcsr_last_stats(ppcsr_shard *h, ppcsr_batch_stats *stats);

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
