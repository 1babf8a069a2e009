// ThreadPoolPPPCSR -- the reference's partition-aware scheduler surface
// (reference src/thread_pool_pppcsr/thread_pool_pppcsr.h:17-47).  submit_* route every op to the shard
// that owns `src` (the reference routes it to a thread of the owning NUMA domain,
// thread_pool_pppcsr.cpp:96-101); start() launches one batch per shard, each on its own GPU stream, so
// shards on different GPUs run concurrently; stop() joins them and prints the elapsed time.
#pragma once
#include <atomic>
#include <chrono>
#include <cstdint>
#include <vector>

#include "PPPCSR.h"
#include "task.h"

class ThreadPoolPPPCSR {
 public:
  PPPCSR *pcsr;

  explicit ThreadPoolPPPCSR(const int NUM_OF_THREADS, bool lock_search, uint32_t init_num_nodes,
                            int partitions_per_domain, bool use_numa);
  // same, with explicit partition boundaries (first vertex of every partition; see PPPCSR.h)
  explicit ThreadPoolPPPCSR(const int NUM_OF_THREADS, bool lock_search, uint32_t init_num_nodes,
                            int partitions_per_domain, bool use_numa, const std::vector<size_t> &boundaries);
  ~ThreadPoolPPPCSR();

  void submit_add(int thread_id, int src, int dest);
  void submit_delete(int thread_id, int src, int dest);
  void submit_read(int thread_id, int src);
  // a whole array of updates at once (value 0 = delete, value == nullptr = all adds): what the loaders hand over
  void submit_bulk(const uint32_t *src, const uint32_t *dst, const uint32_t *value, size_t count);
  void start(int threads);
  void stop();
  // start() applies the staged updates as `k` consecutive batches of ceil(count / k), streamed two ahead through
  // PPPCSR::submit_batch / wait_batch (k = 1: one batch); last_stats() then sums the counters over the batches
  void set_batches(int k) { batches_ = k; }
  // on: the batches capture what they change, and stop() prints one "not found <src> <dst>" line (global ids) per
  // remove that missed, as the reference does (PCSR.cpp:751), in place of the "not found <N> edges" count
  void set_not_found_lines(bool on);

  // thread -> domain table of the reference (thread_pool_pppcsr.cpp:32-47), kept for the CPU-side reads
  const std::vector<int> &thread_to_domain() const { return threadToDomain; }
  const std::vector<int> &first_thread_of_domain() const { return firstThreadDomain; }
  const std::vector<int> &threads_of_domain() const { return numThreadsDomain; }
  const std::vector<ppcsr_batch_stats> &last_stats() const { return stats_; }

 private:
  void stage(int src, int dest, uint32_t value);
  void init_tables(int NUM_OF_THREADS);

  std::vector<uint32_t> src_, dst_, val_;  // ONE staging batch of global ids, submission order; routed on the device
  std::vector<int> reads_;
  std::chrono::steady_clock::time_point t0_, t1_;
  std::atomic_bool finished_;
  uint64_t not_found_ = 0;
  std::vector<ppcsr_batch_stats> stats_;
  int batches_ = 1;
  bool nf_lines_ = false;
  std::vector<uint32_t> nf_src_, nf_dst_;  // the misses of the phase, batch by batch (set_not_found_lines)
  void collect_not_found();

  const int available_nodes;  // GPUs used as "domains"
  int partitions_per_domain = 1;
  std::vector<int> threadToDomain;
  std::vector<int> firstThreadDomain;
  std::vector<int> numThreadsDomain;
};
