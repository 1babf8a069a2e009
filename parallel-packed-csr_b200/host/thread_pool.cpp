// ThreadPool over one GPU shard: see thread_pool.h.
#include "thread_pool.h"

#include <cstdlib>
#include <iostream>

#include "stream.h"

ThreadPool::ThreadPool(const int NUM_OF_THREADS, bool lock_search, uint32_t init_num_nodes, int partitions_per_domain)
    : finished_(false), threads_(NUM_OF_THREADS) {
  (void)partitions_per_domain;
  pcsr = new PCSR(init_num_nodes, init_num_nodes, lock_search, -1);
  pcsr->print_not_found = false;  // batch mode reports the miss count once instead of one line per miss
}

ThreadPool::~ThreadPool() { delete pcsr; }

void ThreadPool::set_not_found_lines(bool on) {
  nf_lines_ = on;
  pcsr->set_change_capture(on);
}

void ThreadPool::collect_not_found() {
  if (!nf_lines_) return;
  const PCSR::Changes c = pcsr->last_changes();
  nf_src_.insert(nf_src_.end(), c.nf_src.begin(), c.nf_src.end());
  nf_dst_.insert(nf_dst_.end(), c.nf_dst.begin(), c.nf_dst.end());
}

// thread_id is irrelevant on the device (ThreadPoolPPPCSR ignores it in the reference too,
// src/thread_pool_pppcsr/thread_pool_pppcsr.cpp:97); submission order is kept: last op wins per edge.
void ThreadPool::submit_add(int thread_id, int src, int dest) {
  (void)thread_id;
  src_.push_back((uint32_t)src);
  dst_.push_back((uint32_t)dest);
  val_.push_back(1u);  // the pools always insert value 1 (reference thread_pool.cpp:44)
}

void ThreadPool::submit_delete(int thread_id, int src, int dest) {
  (void)thread_id;
  src_.push_back((uint32_t)src);
  dst_.push_back((uint32_t)dest);
  val_.push_back(0u);
}

void ThreadPool::submit_read(int thread_id, int src) {
  (void)thread_id;
  reads_.push_back(src);
}

void ThreadPool::submit_bulk(const uint32_t *src, const uint32_t *dst, const uint32_t *value, size_t count) {
  src_.insert(src_.end(), src, src + count);
  dst_.insert(dst_.end(), dst, dst + count);
  if (value) val_.insert(val_.end(), value, value + count);
  else val_.insert(val_.end(), count, 1u);
}

void ThreadPool::start(int threads) {
  (void)threads;
  t0_ = std::chrono::steady_clock::now();
  finished_ = false;
  nf_src_.clear();
  nf_dst_.clear();
  std::cout << "Thread 0 has " << src_.size() + reads_.size() << " tasks" << std::endl;
  pcsr->edges.global_lock->registerThread();
  if (batches_ > 1 && !src_.empty()) {
    stats_ = ppcsr_batch_stats{};
    ppcsr_shard *h = pcsr->handle();
    stream_batches(
        src_.size(), (size_t)batches_,
        [&](size_t lo, size_t len) {
          uint64_t ticket = 0;
          if (ppcsr_submit_batch(h, src_.data() + lo, dst_.data() + lo, val_.data() + lo, len, 1, &ticket) != PPCSR_OK) {
            std::cout << "ppcsr_submit_batch failed: " << ppcsr_last_error() << ". Abort\n";
            std::exit(EXIT_FAILURE);
          }
          return ticket;
        },
        [&](uint64_t ticket) {
          ppcsr_batch_stats st{};
          if (ppcsr_wait(h, ticket, &st) != PPCSR_OK) {
            std::cout << "ppcsr_wait failed: " << ppcsr_last_error() << ". Abort\n";
            std::exit(EXIT_FAILURE);
          }
          add_batch_stats(stats_, st);
          collect_not_found();
        });
    pcsr->batch_applied();
  } else if (!src_.empty()) {
    pcsr->apply_batch(src_, dst_, val_, &stats_);
    collect_not_found();
  }
  for (int v : reads_) pcsr->read_neighbourhood(v);
  pcsr->edges.global_lock->unregisterThread();
}

void ThreadPool::stop() {
  finished_ = true;
  if (ppcsr_sync(pcsr->handle()) != PPCSR_OK) {
    std::cout << "device synchronisation failed: " << ppcsr_last_error() << ". Abort\n";
    std::exit(EXIT_FAILURE);
  }
  std::cout << "Done" << std::endl;
  t1_ = std::chrono::steady_clock::now();
  if (nf_lines_) {
    for (size_t i = 0; i < nf_src_.size(); i++) std::cout << "not found " << nf_src_[i] << " " << nf_dst_[i] << "\n";
    std::cout << std::flush;
  } else if (stats_.n_not_found) {
    std::cout << "not found " << stats_.n_not_found << " edges" << std::endl;
  }
  std::cout << "Elapsed wall clock time: "
            << std::chrono::duration_cast<std::chrono::milliseconds>(t1_ - t0_).count() << std::endl;
  src_.clear();
  dst_.clear();
  val_.clear();
  reads_.clear();
}
