// PPPCSR host shell: see PPPCSR.h.
#include "PPPCSR.h"

#include <algorithm>
#include <cstdlib>
#include <iostream>

PPPCSR::PPPCSR(uint32_t init_n, uint32_t src_n, bool lock_search, int numDomain, int partitionsPerDomain,
               bool use_numa)
    : partitionsPerDomain(partitionsPerDomain) {
  (void)src_n;
  const std::size_t parts = (std::size_t)numDomain * (std::size_t)partitionsPerDomain;
  // equal vertex counts, the last partition takes the remainder (reference PPPCSR.cpp:20,27-29)
  const std::size_t share = init_n / parts;
  for (std::size_t p = 0; p < parts; p++) distribution.push_back(p * share);
  build(init_n, lock_search, use_numa);
}

PPPCSR::PPPCSR(uint32_t init_n, bool lock_search, int partitionsPerDomain, bool use_numa,
               const std::vector<size_t> &boundaries)
    : distribution(boundaries), partitionsPerDomain(partitionsPerDomain) {
  build(init_n, lock_search, use_numa);
}

void PPPCSR::build(uint32_t init_n, bool lock_search, bool use_numa) {
  const std::size_t parts = distribution.size();
  partitions.reserve(parts);
  for (std::size_t p = 0; p < parts; p++) {
    const std::size_t size = (p + 1 == parts ? (std::size_t)init_n : distribution[p + 1]) - distribution[p];
    const int gpu = use_numa ? (int)(p / partitionsPerDomain) : 0;
    partitions.emplace_back((uint32_t)size, (uint32_t)size, lock_search, gpu);
  }
  std::cout << "Number of partitions: " << partitions.size() << std::endl;
}

PPPCSR::~PPPCSR() {
  if (group_) ppcsr_group_destroy(group_);
}

void PPPCSR::ensure_group(std::size_t cap, bool values) {
  const std::size_t parts = partitions.size();
  if (group_ && cap <= group_cap_ && (!values || group_values_)) return;
  if (in_flight_) {  // destroying the group would drop the batches in flight
    std::cout << "PPPCSR: a batch needs a larger group while submitted batches are in flight. Abort\n";
    std::exit(EXIT_FAILURE);
  }
  if (group_) ppcsr_group_destroy(group_);  // (re)size the receive buffers
  group_ = nullptr;
  std::vector<ppcsr_shard *> handles;
  std::vector<uint64_t> starts;
  uint64_t n = 0;
  for (std::size_t p = 0; p < parts; p++) {
    handles.push_back(partitions[p].handle());
    starts.push_back(distribution[p]);
    n = distribution[p] + partitions[p].get_n();
  }
  starts.push_back(n);
  group_cap_ = std::max<std::size_t>(cap + cap / 8, 1024);
  group_values_ = group_values_ || values;
  if (ppcsr_group_create(handles.data(), (uint32_t)parts, starts.data(), group_cap_, group_values_ ? 1 : 0,
                         &group_) != PPCSR_OK) {
    std::cout << "ppcsr_group_create failed: " << ppcsr_last_error() << ". Abort\n";
    std::exit(EXIT_FAILURE);
  }
}

void PPPCSR::apply_batch(const uint32_t *src, const uint32_t *dst, const uint32_t *value, size_t count,
                         std::vector<ppcsr_batch_stats> *stats) {
  const std::size_t parts = partitions.size();
  ensure_group((count + parts - 1) / parts, value != nullptr);
  std::vector<ppcsr_batch_stats> st(parts);
  if (ppcsr_group_apply(group_, src, dst, value, count, 1, st.data()) != PPCSR_OK) {
    std::cout << "ppcsr_group_apply failed: " << ppcsr_last_error() << ". Abort\n";
    std::exit(EXIT_FAILURE);
  }
  for (auto &part : partitions) part.batch_applied();
  if (stats) *stats = st;
}

uint64_t PPPCSR::submit_batch(const uint32_t *src, const uint32_t *dst, const uint32_t *value, size_t count) {
  const std::size_t parts = partitions.size();
  ensure_group((count + parts - 1) / parts, value != nullptr);
  uint64_t ticket = 0;
  if (ppcsr_group_submit(group_, src, dst, value, count, 1, &ticket) != PPCSR_OK) {
    std::cout << "ppcsr_group_submit failed: " << ppcsr_last_error() << ". Abort\n";
    std::exit(EXIT_FAILURE);
  }
  in_flight_++;
  return ticket;
}

void PPPCSR::wait_batch(uint64_t ticket, std::vector<ppcsr_batch_stats> *stats) {
  std::vector<ppcsr_batch_stats> st(partitions.size());
  if (ppcsr_group_wait(group_, ticket, st.data()) != PPCSR_OK) {
    std::cout << "ppcsr_group_wait failed: " << ppcsr_last_error() << ". Abort\n";
    std::exit(EXIT_FAILURE);
  }
  in_flight_--;
  for (auto &part : partitions) part.batch_applied();
  if (stats) *stats = st;
}

std::size_t PPPCSR::get_partiton(size_t vertex_id) const {
  // first partition whose successor starts beyond the vertex; ids past the end go to the last one
  // (reference PPPCSR.cpp:58-66)
  for (std::size_t p = 1; p < distribution.size(); p++) {
    if (distribution[p] > vertex_id) return p - 1;
  }
  return distribution.size() - 1;
}

bool PPPCSR::edge_exists(uint32_t src, uint32_t dest) {
  const auto p = get_partiton(src);
  return partitions[p].edge_exists(src - (uint32_t)distribution[p], dest);
}

std::vector<int> PPPCSR::get_neighbourhood(int src) const {
  const auto p = get_partiton(src);
  return partitions[p].get_neighbourhood(src - (int)distribution[p]);
}

void PPPCSR::add_node() { partitions.back().add_node(); }

void PPPCSR::add_edge(uint32_t src, uint32_t dest, uint32_t value) {
  const auto p = get_partiton(src);
  partitions[p].add_edge(src - (uint32_t)distribution[p], dest, value);
}

void PPPCSR::remove_edge(uint32_t src, uint32_t dest) {
  const auto p = get_partiton(src);
  partitions[p].remove_edge(src - (uint32_t)distribution[p], dest);
}

void PPPCSR::read_neighbourhood(int src) {
  const auto p = get_partiton(src);
  partitions[p].read_neighbourhood(src - (int)distribution[p]);
}

uint64_t PPPCSR::get_n() {
  uint64_t n = 0;
  for (auto &part : partitions) n += part.get_n();
  return n;
}

node_t &PPPCSR::getNode(int id) {
  const auto p = get_partiton(id);
  return partitions[p].getNode(id - (int)distribution[p]);
}

const node_t &PPPCSR::getNode(int id) const {
  const auto p = get_partiton(id);
  return partitions[p].getNode(id - (int)distribution[p]);
}

void PPPCSR::pagerank_push(const std::vector<double> &in, std::vector<double> &out) const {
  for (std::size_t p = 0; p < partitions.size(); p++) {
    const std::size_t lo = distribution[p];
    const std::size_t n_local = partitions[p].get_n();
    std::vector<double> slice(in.begin() + lo, in.begin() + lo + n_local);
    partitions[p].pagerank_push(slice, out);
  }
}

std::vector<uint32_t> PPPCSR::bfs_levels(uint32_t start) {
  ensure_group(0, false);
  std::vector<uint32_t> d(get_n());
  if (ppcsr_group_bfs(group_, start, d.data()) != PPCSR_OK) {
    std::cout << "ppcsr_group_bfs failed: " << ppcsr_last_error() << ". Abort\n";
    std::exit(EXIT_FAILURE);
  }
  return d;
}

std::vector<double> PPPCSR::pagerank(uint32_t iterations, double damping) {
  ensure_group(0, false);
  std::vector<double> r(get_n());
  if (ppcsr_group_pagerank(group_, iterations, damping, r.data()) != PPCSR_OK) {
    std::cout << "ppcsr_group_pagerank failed: " << ppcsr_last_error() << ". Abort\n";
    std::exit(EXIT_FAILURE);
  }
  return r;
}

ppcsr_repartition_stats PPPCSR::repartition(const std::vector<size_t> &boundaries) {
  ensure_group(0, false);
  std::vector<uint64_t> starts(boundaries.begin(), boundaries.end());
  starts.push_back(get_n());
  ppcsr_repartition_stats st{};
  if (starts.size() != partitions.size() + 1 || ppcsr_group_repartition(group_, starts.data(), &st) != PPCSR_OK) {
    std::cout << "ppcsr_group_repartition failed: " << ppcsr_last_error() << ". Abort\n";
    std::exit(EXIT_FAILURE);
  }
  distribution = boundaries;
  for (auto &part : partitions) part.batch_applied();
  return st;
}
