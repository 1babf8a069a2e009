// ThreadPool -- the reference's scheduler surface (reference src/thread_pool/thread_pool.h:17-40) over one
// GPU shard.  submit_* only stage the operation (the reference also fills its queues before start(),
// src/main.cpp:68-82); start() stamps the clock and launches the staged batch on the device, stop()
// synchronises and prints "Elapsed wall clock time: <ms>" exactly like the reference
// (src/thread_pool/thread_pool.cpp:108-111) -- the line its benchmark scripts scrape.
#pragma once
#include <atomic>
#include <chrono>
#include <cstdint>
#include <vector>

#include "PCSR.h"
#include "task.h"

class ThreadPool {
 public:
  PCSR *pcsr;

  explicit ThreadPool(const int NUM_OF_THREADS, bool lock_search, uint32_t init_num_nodes, int partitions_per_domain);
  ~ThreadPool();

  void submit_add(int thread_id, int src, int dest);
  void submit_delete(int thread_id, int src, int dest);
  void submit_read(int thread_id, int src);
  // a whole array of updates at once (value 0 = delete, value == nullptr = all adds): what the loaders hand over
  void submit_bulk(const uint32_t *src, const uint32_t *dst, const uint32_t *value, size_t count);
  void start(int threads);
  void stop();
  // start() applies the staged updates as `k` consecutive batches of ceil(count / k), streamed two ahead through
  // ppcsr_submit_batch / ppcsr_wait (k = 1: one batch); last_stats() then sums the counters over the batches
  void set_batches(int k) { batches_ = k; }
  // on: the batches capture what they change, and stop() prints one "not found <src> <dst>" line (global ids) per
  // remove that missed, as the reference does (PCSR.cpp:751), in place of the "not found <N> edges" count
  void set_not_found_lines(bool on);

  const ppcsr_batch_stats &last_stats() const { return stats_; }

 private:
  std::vector<uint32_t> src_, dst_, val_;  // staged updates, submission order (value 0 = delete)
  std::vector<int> reads_;
  std::chrono::steady_clock::time_point t0_, t1_;
  std::atomic_bool finished_;
  ppcsr_batch_stats stats_{};
  int threads_;
  int batches_ = 1;
  bool nf_lines_ = false;
  std::vector<uint32_t> nf_src_, nf_dst_;  // the misses of the phase, batch by batch (set_not_found_lines)
  void collect_not_found();
};
