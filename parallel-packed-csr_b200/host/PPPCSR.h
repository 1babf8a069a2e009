// PPPCSR -- vertex-range partitioned graph with the reference's class surface
// (reference src/pppcsr/PPPCSR.h:11-60): numDomain * partitionsPerDomain independent PCSR shards over
// contiguous source ranges; `src` is made partition-local, `dest` stays global.  A "domain" is a GPU here
// (the reference's NUMA domain): partition p lives on GPU (p / partitionsPerDomain) % #GPUs when
// use_numa is set, else on GPU 0.
#pragma once
#include <cstddef>
#include <vector>

#include "PCSR.h"

class PPPCSR {
 public:
  edge_list_t edges;  // present in the reference too, never initialised there (PPPCSR.h:14)

  PPPCSR(uint32_t init_n, uint32_t src_n, bool lock_search, int numDomain, int partitionsPerDomain, bool use_numa);
  // same, with explicit first vertices of the partitions (ascending, boundaries[0] == 0): the reference's
  // `distribution` vector admits any monotone boundaries (PPPCSR.h:57); edge-balanced ones keep a skewed graph from
  // putting 44 % of its edges on the first of eight GPUs
  PPPCSR(uint32_t init_n, bool lock_search, int partitionsPerDomain, bool use_numa,
         const std::vector<size_t> &boundaries);
  ~PPPCSR();
  PPPCSR(const PPPCSR &) = delete;
  PPPCSR &operator=(const PPPCSR &) = delete;

  bool edge_exists(uint32_t src, uint32_t dest);
  void add_node();
  void add_edge(uint32_t src, uint32_t dest, uint32_t value);
  void remove_edge(uint32_t src, uint32_t dest);
  void read_neighbourhood(int src);
  std::size_t get_partiton(size_t vertex_id) const;  // [sic] the reference's spelling
  std::vector<int> get_neighbourhood(int src) const;
  uint64_t get_n();
  node_t &getNode(int id);
  const node_t &getNode(int id) const;
  void registerThread(int par) { partitions[par].edges.global_lock->registerThread(); }
  void unregisterThread(int par) { partitions[par].edges.global_lock->unregisterThread(); }

  // ---- batched surface for ThreadPoolPPPCSR ----
  std::size_t partition_count() const { return partitions.size(); }
  PCSR &partition(std::size_t p) { return partitions[p]; }
  std::size_t partition_start(std::size_t p) const { return distribution[p]; }
  void pagerank_push(const std::vector<double> &in, std::vector<double> &out) const;
  // One batch of GLOBAL updates (value 0 = remove, value == nullptr = all adds): the batch is cut into one slice per
  // partition, every GPU bins its slice by owner ON THE DEVICE and stores the records straight into the owner's receive
  // buffer over NVLink peer memory, every partition applies what it received (C-ABI ppcsr_group_apply).  Replaces the
  // per-op hand-over of reference ThreadPoolPPPCSR::submit_* (thread_pool_pppcsr.cpp:96-118).  stats: one per partition.
  void apply_batch(const uint32_t *src, const uint32_t *dst, const uint32_t *value, size_t count,
                   std::vector<ppcsr_batch_stats> *stats = nullptr);
  // The same batch as a stream (C-ABI ppcsr_group_submit / ppcsr_group_wait): submit_batch starts the copy and the
  // routing and returns a ticket, wait_batch applies that batch on every partition.  With
  //     submit(b0); for i: { submit(b[i+1]); wait(b[i]); }
  // batch i+1 is routed while the partitions apply batch i, with the result of apply_batch(b0); apply_batch(b1); ...
  // At most two batches in flight, waited for in submission order; the arrays must stay valid until the wait.
  uint64_t submit_batch(const uint32_t *src, const uint32_t *dst, const uint32_t *value, size_t count);
  void wait_batch(uint64_t ticket, std::vector<ppcsr_batch_stats> *stats = nullptr);
  // Creates the device-side group over the partitions, or recreates it when `cap` records per (sender, receiver)
  // region or per-update values exceed what it was created for (never while a submitted batch is in flight).  A
  // traversal before any batch needs it too.
  void ensure_group(std::size_t cap, bool values);
  // Traversals over all partitions on the devices (ppcsr_group_bfs / ppcsr_group_pagerank): hop counts from `start`
  // (UINT32_MAX = unreached), and `iterations` damped PageRank iterations with the recurrence of PCSR::pagerank.
  std::vector<uint32_t> bfs_levels(uint32_t start);
  std::vector<double> pagerank(uint32_t iterations, double damping);
  // Moves vertex ranges between the partitions on the devices (ppcsr_group_repartition): partition p then starts at
  // boundaries[p] (boundaries[0] == 0, strictly ascending, one entry per partition; the last partition ends at
  // get_n()).  The logical graph is unchanged.
  ppcsr_repartition_stats repartition(const std::vector<size_t> &boundaries);

 private:
  void build(uint32_t init_n, bool lock_search, bool use_numa);
  std::vector<PCSR> partitions;
  std::vector<size_t> distribution;  // first vertex of every partition
  int partitionsPerDomain;
  ppcsr_group *group_ = nullptr;     // device-side router over the partitions, (re)created for the largest batch seen
  size_t group_cap_ = 0;
  bool group_values_ = false;
  int in_flight_ = 0;                // batches submitted and not yet waited for
};
