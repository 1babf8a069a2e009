// ThreadPoolPPPCSR over per-GPU shards: see thread_pool_pppcsr.h.
#include "thread_pool_pppcsr.h"

#include <algorithm>
#include <cstdlib>
#include <iostream>
#include <thread>

#include "stream.h"

static int usable_gpus(int threads) {
  int gpus = ppcsr_device_count();
  if (const char *e = std::getenv("PPCSR_GPUS")) gpus = std::min(gpus, std::max(1, std::atoi(e)));
  // the reference uses min(#NUMA nodes, #threads) domains (thread_pool_pppcsr.cpp:24)
  return std::max(1, std::min(gpus, threads));
}

ThreadPoolPPPCSR::ThreadPoolPPPCSR(const int NUM_OF_THREADS, bool lock_search, uint32_t init_num_nodes,
                                   int partitions_per_domain, bool use_numa)
    : finished_(false),
      available_nodes(usable_gpus(NUM_OF_THREADS)),
      partitions_per_domain(partitions_per_domain),
      threadToDomain(NUM_OF_THREADS),
      firstThreadDomain(available_nodes, 0),
      numThreadsDomain(available_nodes, 0) {
  pcsr = new PPPCSR(init_num_nodes, init_num_nodes, lock_search, available_nodes, partitions_per_domain, use_numa);
  init_tables(NUM_OF_THREADS);
}

ThreadPoolPPPCSR::ThreadPoolPPPCSR(const int NUM_OF_THREADS, bool lock_search, uint32_t init_num_nodes,
                                   int partitions_per_domain, bool use_numa, const std::vector<size_t> &boundaries)
    : finished_(false),
      available_nodes(usable_gpus(NUM_OF_THREADS)),
      partitions_per_domain(partitions_per_domain),
      threadToDomain(NUM_OF_THREADS),
      firstThreadDomain(available_nodes, 0),
      numThreadsDomain(available_nodes, 0) {
  pcsr = new PPPCSR(init_num_nodes, lock_search, partitions_per_domain, use_numa, boundaries);
  init_tables(NUM_OF_THREADS);
}

void ThreadPoolPPPCSR::init_tables(int NUM_OF_THREADS) {
  for (std::size_t p = 0; p < pcsr->partition_count(); p++) pcsr->partition(p).print_not_found = false;
  // threads are dealt to domains in contiguous blocks, the first (threads % domains) domains get one more
  const int base = NUM_OF_THREADS / available_nodes, extra = NUM_OF_THREADS % available_nodes;
  int t = 0;
  for (int d = 0; d < available_nodes && t < NUM_OF_THREADS; d++) {
    const int take = base + (d < extra ? 1 : 0);
    firstThreadDomain[d] = t;
    numThreadsDomain[d] = take;
    for (int k = 0; k < take; k++) threadToDomain[t++] = d;
  }
}

ThreadPoolPPPCSR::~ThreadPoolPPPCSR() { delete pcsr; }

void ThreadPoolPPPCSR::set_not_found_lines(bool on) {
  nf_lines_ = on;
  pcsr->set_change_capture(on);
}

void ThreadPoolPPPCSR::collect_not_found() {
  if (!nf_lines_) return;
  const PCSR::Changes c = pcsr->last_changes();
  nf_src_.insert(nf_src_.end(), c.nf_src.begin(), c.nf_src.end());
  nf_dst_.insert(nf_dst_.end(), c.nf_dst.begin(), c.nf_dst.end());
}

// Global ids, submission order: the owner of every op is found ON THE DEVICE when the batch starts (the reference
// looks it up here, per op: thread_pool_pppcsr.cpp:98).
void ThreadPoolPPPCSR::stage(int src, int dest, uint32_t value) {
  src_.push_back((uint32_t)src);
  dst_.push_back((uint32_t)dest);
  val_.push_back(value);
}

void ThreadPoolPPPCSR::submit_add(int thread_id, int src, int dest) {
  (void)thread_id;
  stage(src, dest, 1u);
}
void ThreadPoolPPPCSR::submit_delete(int thread_id, int src, int dest) {
  (void)thread_id;
  stage(src, dest, 0u);
}
void ThreadPoolPPPCSR::submit_read(int thread_id, int src) {
  (void)thread_id;
  reads_.push_back(src);
}
void ThreadPoolPPPCSR::submit_bulk(const uint32_t *src, const uint32_t *dst, const uint32_t *value, size_t count) {
  src_.insert(src_.end(), src, src + count);
  dst_.insert(dst_.end(), dst, dst + count);
  if (value) val_.insert(val_.end(), value, value + count);
  else val_.insert(val_.end(), count, 1u);
}

void ThreadPoolPPPCSR::start(int threads) {
  (void)threads;
  t0_ = std::chrono::steady_clock::now();
  finished_ = false;
  not_found_ = 0;
  nf_src_.clear();
  nf_dst_.clear();
  std::cout << "Thread 0 has " << src_.size() << " tasks for " << pcsr->partition_count()
            << " partitions, routed on the device" << std::endl;
  for (std::size_t p = 0; p < pcsr->partition_count(); p++) pcsr->registerThread((int)p);
  if (batches_ > 1 && !src_.empty()) {
    stats_.assign(pcsr->partition_count(), ppcsr_batch_stats{});
    std::vector<ppcsr_batch_stats> st;
    stream_batches(
        src_.size(), (size_t)batches_,
        [&](size_t lo, size_t len) { return pcsr->submit_batch(src_.data() + lo, dst_.data() + lo, val_.data() + lo, len); },
        [&](uint64_t ticket) {
          pcsr->wait_batch(ticket, &st);
          for (std::size_t p = 0; p < st.size(); p++) add_batch_stats(stats_[p], st[p]);
          collect_not_found();
        });
  } else if (!src_.empty()) {
    pcsr->apply_batch(src_.data(), dst_.data(), val_.data(), src_.size(), &stats_);
    collect_not_found();
  }
  for (std::size_t p = 0; p < pcsr->partition_count(); p++) pcsr->unregisterThread((int)p);
  for (auto &st : stats_) not_found_ += st.n_not_found;
  for (int v : reads_) pcsr->read_neighbourhood(v);
}

void ThreadPoolPPPCSR::stop() {
  finished_ = true;
  for (std::size_t p = 0; p < pcsr->partition_count(); p++) {
    if (ppcsr_sync(pcsr->partition(p).handle()) != PPCSR_OK) {
      std::cout << "device synchronisation failed: " << ppcsr_last_error() << ". Abort\n";
      std::exit(EXIT_FAILURE);
    }
    std::cout << "Done" << std::endl;
  }
  t1_ = std::chrono::steady_clock::now();
  if (nf_lines_) {
    for (size_t i = 0; i < nf_src_.size(); i++) std::cout << "not found " << nf_src_[i] << " " << nf_dst_[i] << "\n";
    std::cout << std::flush;
  } else if (not_found_) {
    std::cout << "not found " << not_found_ << " edges" << std::endl;
  }
  std::cout << "Elapsed wall clock time: "
            << std::chrono::duration_cast<std::chrono::milliseconds>(t1_ - t0_).count() << std::endl;
  src_.clear();
  dst_.clear();
  val_.clear();
  reads_.clear();
}
