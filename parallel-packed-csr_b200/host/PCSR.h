// PCSR -- host shell with the reference's class surface (reference src/pcsr/PCSR.h:64-124) over one
// GPU-resident shard (include/ppcsr_b200.h).  Every method forwards to the C-ABI; a single add_edge /
// remove_edge is a batch of one (correctness path), the scheduler classes submit whole batches.
#pragma once
#include <cstdint>
#include <memory>
#include <utility>
#include <vector>

#include "fastLock.h"
#include "hybridLock.h"
#include "ppcsr_b200.h"

// reference src/pcsr/PCSR.h:18-23
typedef struct _node {
  uint32_t beginning;      // slot of the vertex's sentinel
  uint32_t end;            // exclusive: slot of the next vertex's sentinel (N-1 for the last vertex)
  uint32_t num_neighbors;  // add calls minus remove calls with this source (reference semantics)
} node_t;

// reference src/pcsr/PCSR.h:30-35 (kept for the migration stubs' signatures)
typedef struct _edge {
  uint32_t src;
  uint32_t dest;
  uint32_t value;
} edge_t;

// reference src/pcsr/PCSR.h:37-44.  `items` lives in HBM and is not host-addressable: it stays null.
typedef struct edge_list {
  uint64_t N;
  int H;
  int logN;
  std::shared_ptr<FastLock> global_lock;
  HybridLock **node_locks;
  edge_t *items;
} edge_list_t;

class PCSR {
 public:
  edge_list_t edges;

  PCSR(uint32_t init_n, uint32_t src_n, bool lock_search, int domain = 0);
  PCSR(PCSR &&other) noexcept;
  PCSR(const PCSR &) = delete;
  PCSR &operator=(const PCSR &) = delete;
  ~PCSR();

  bool edge_exists(uint32_t src, uint32_t dest);
  void add_node();
  void add_edge(uint32_t src, uint32_t dest, uint32_t value);
  void remove_edge(uint32_t src, uint32_t dest);
  void read_neighbourhood(int src);
  std::vector<int> get_neighbourhood(int src) const;
  uint64_t get_n() const;

  // partition-migration hooks: empty in the reference as well (src/pcsr/PCSR.cpp:1447-1468)
  void insert_nodes_and_edges_front(std::vector<node_t> nodes, std::vector<edge_t> new_edges);
  void insert_nodes_and_edges_back(std::vector<node_t> nodes, std::vector<edge_t> new_edges);
  std::pair<std::vector<node_t>, std::vector<edge_t>> remove_nodes_and_edges_front(int num_nodes);
  std::pair<std::vector<node_t>, std::vector<edge_t>> remove_nodes_and_edges_back(int num_nodes);

  node_t &getNode(int id);
  const node_t &getNode(int id) const;

  // ---- batched surface used by the schedulers (no reference counterpart: the reference applies one
  //      op per call from its worker threads, src/thread_pool/thread_pool.cpp:43-49) ----
  // value[i] != 0 inserts, 0 removes; returns the device milliseconds of the batch
  float apply_batch(const std::vector<uint32_t> &src, const std::vector<uint32_t> &dst,
                    const std::vector<uint32_t> &value, ppcsr_batch_stats *stats = nullptr);
  float apply_batch(const uint32_t *src, const uint32_t *dst, const uint32_t *value /*nullable: all 1*/, size_t count,
                    ppcsr_batch_stats *stats = nullptr);
  // interleaved (src, dst) pairs, e.g. an mmap'd binary edge file; every update carries default_val (0 = remove)
  float apply_batch_pairs(const uint32_t *pairs, size_t count, uint32_t default_val, ppcsr_batch_stats *stats = nullptr);
  void batch_applied();  // refresh the host mirror after a batch reached the shard through the C-ABI directly
  // one pagerank push step (reference src/utility/pagerank.h:16-29) accumulated into out[0..out.size())
  void pagerank_push(const std::vector<double> &in, std::vector<double> &out) const;
  std::vector<uint32_t> bfs_levels(uint32_t start) const;
  // iterated PageRank with damping on the device (ppcsr_pagerank): r_0 = 1/n,
  // r_{t+1}[v] = (1 - damping)/n + damping * sum_{(u,v)} r_t[u] / num_neighbors[u]
  std::vector<double> pagerank(uint32_t iterations, double damping) const;
  bool check_invariants(bool check_lower, ppcsr_invariant_report *report = nullptr) const;
  ppcsr_shard *handle() const { return shard_; }
  int device() const { return device_; }
  bool print_not_found = true;  // the reference prints "not found s d" per miss (PCSR.cpp:751)

  // What each batch changed (C-ABI ppcsr_set_change_capture / ppcsr_last_changes), copied to the host: one entry per
  // changed key (old_val 0 = inserted, new_val 0 = deleted) and one (nf_src, nf_dst) per remove that missed, both in
  // ascending (src, dst) order.  Sources are shard-local plus `vertex_offset`.
  struct Changes {
    std::vector<uint32_t> src, dst, old_val, new_val, nf_src, nf_dst;
  };
  void set_change_capture(bool on);
  Changes last_changes(uint64_t vertex_offset = 0) const;

 private:
  void refresh_geometry();
  void refresh_nodes() const;
  void fail(const char *what) const;

  ppcsr_shard *shard_ = nullptr;
  int device_ = 0;
  bool lock_bsearch_ = false;
  std::vector<std::unique_ptr<HybridLock>> lock_store_;
  std::vector<HybridLock *> lock_ptrs_;
  mutable std::vector<node_t> nodes_;
  mutable bool nodes_dirty_ = true;
};
