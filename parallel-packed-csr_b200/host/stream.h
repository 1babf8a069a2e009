// Streaming one phase of updates as several batches (the CLI's -batches=<k>), shared by ThreadPool and
// ThreadPoolPPPCSR.
#pragma once
#include <algorithm>
#include <cstddef>
#include <cstdint>
#include <deque>

#include "ppcsr_b200.h"

// Cuts [0, count) into k consecutive batches of ceil(count / k) updates and keeps two of them in flight:
//     submit(b0); for i: { submit(b[i+1]); wait(b[i]); }
// submit(first, len) returns the ticket of the batch [first, first + len), wait(ticket) applies it.
template <typename Submit, typename Wait>
void stream_batches(size_t count, size_t k, Submit submit, Wait wait) {
  const size_t step = (count + k - 1) / k;
  std::deque<uint64_t> in_flight;
  for (size_t lo = 0; lo < count; lo += step) {
    in_flight.push_back(submit(lo, std::min(step, count - lo)));
    if (in_flight.size() == 2) {
      wait(in_flight.front());
      in_flight.pop_front();
    }
  }
  for (; !in_flight.empty(); in_flight.pop_front()) wait(in_flight.front());
}

// The stats of a stream: counters, bytes and times add up, the geometry is that before the first and after the last
// batch.  `sum` starts zeroed.
inline void add_batch_stats(ppcsr_batch_stats &sum, const ppcsr_batch_stats &b) {
  const bool first = sum.batch_size == 0 && sum.slots_after == 0;
  sum.batch_size += b.batch_size;
  sum.n_ignored += b.n_ignored;
  sum.n_unique += b.n_unique;
  sum.n_inserted += b.n_inserted;
  sum.n_overwritten += b.n_overwritten;
  sum.n_deleted += b.n_deleted;
  sum.n_not_found += b.n_not_found;
  sum.n_windows += b.n_windows;
  sum.window_slots += b.window_slots;
  sum.rebalance_bytes += b.rebalance_bytes;
  if (first) sum.slots_before = b.slots_before;
  sum.slots_after = b.slots_after;
  sum.resized |= b.resized;
  sum.whole_array |= b.whole_array;
  sum.ms_total += b.ms_total;
  sum.ms_sort += b.ms_sort;
  sum.ms_locate += b.ms_locate;
  sum.ms_select += b.ms_select;
  sum.ms_rebalance += b.ms_rebalance;
  sum.ms_rebalance_kernel += b.ms_rebalance_kernel;
  sum.kernel_launches += b.kernel_launches;
  sum.sparse_path |= b.sparse_path;
}
