// PCSR host shell: see PCSR.h.  Error convention of the reference: no return codes, fatal problems print
// and exit(EXIT_FAILURE) (reference src/pcsr/PCSR.cpp:48-54).
#include "PCSR.h"

#include <cstdio>
#include <cstdlib>
#include <iostream>

void PCSR::fail(const char *what) const {
  std::cout << what << " failed: " << ppcsr_last_error() << ". Abort\n";
  std::exit(EXIT_FAILURE);
}

PCSR::PCSR(uint32_t init_n, uint32_t src_n, bool lock_search, int domain) : lock_bsearch_(lock_search) {
  // `domain` was the NUMA node of the partition (reference PCSR.cpp:781-786); here it selects the GPU.
  const int devices = ppcsr_device_count();
  if (devices <= 0) {
    std::cout << "No CUDA device available (the B200 engine has no CPU path). Abort\n";
    std::exit(EXIT_FAILURE);
  }
  device_ = domain > 0 ? domain % devices : 0;
  if (ppcsr_create(init_n, src_n, device_, &shard_) != PPCSR_OK) fail("ppcsr_create");
  edges.global_lock = std::make_shared<FastLock>();
  edges.items = nullptr;
  edges.node_locks = nullptr;
  edges.N = 0;
  refresh_geometry();
}

PCSR::PCSR(PCSR &&o) noexcept
    : edges(o.edges), print_not_found(o.print_not_found), shard_(o.shard_), device_(o.device_),
      lock_bsearch_(o.lock_bsearch_), lock_store_(std::move(o.lock_store_)), lock_ptrs_(std::move(o.lock_ptrs_)),
      nodes_(std::move(o.nodes_)), nodes_dirty_(o.nodes_dirty_) {
  o.shard_ = nullptr;
  edges.node_locks = lock_ptrs_.data();
}

PCSR::~PCSR() {
  if (shard_) ppcsr_destroy(shard_);
}

// Mirrors what reference resizeEdgeArray publishes (PCSR.cpp:68-73), including its log line on a resize.
void PCSR::refresh_geometry() {
  ppcsr_geometry g;
  if (ppcsr_geometry_of(shard_, &g) != PPCSR_OK) fail("ppcsr_geometry_of");
  if (g.N != edges.N) {
    edges.N = g.N;
    edges.logN = (int)g.logN;
    edges.H = (int)g.H;
    std::cout << "Edges: " << edges.N << " logN: " << edges.logN << " #count: " << edges.N / edges.logN << std::endl;
    // node_locks[i] of every leaf is ONE always-free stub (no per-leaf locking in a batch design): a per-leaf object
    // would cost 16 M allocations at scale 24 and an O(leaves) version bump per batch
    const size_t leaves = edges.N / edges.logN;
    if (lock_store_.empty()) lock_store_.emplace_back(new HybridLock());
    lock_ptrs_.assign(leaves, lock_store_[0].get());
    edges.node_locks = lock_ptrs_.data();
  }
}

void PCSR::refresh_nodes() const {
  if (!nodes_dirty_) return;
  const uint64_t n = get_n();
  std::vector<uint32_t> b(n), e(n), k(n);
  if (n) {
    if (ppcsr_node_ranges(shard_, b.data(), e.data()) != PPCSR_OK) fail("ppcsr_node_ranges");
    if (ppcsr_num_neighbors(shard_, k.data()) != PPCSR_OK) fail("ppcsr_num_neighbors");
  }
  nodes_.resize(n);
  for (uint64_t v = 0; v < n; v++) nodes_[v] = node_t{b[v], e[v], k[v]};
  nodes_dirty_ = false;
}

uint64_t PCSR::get_n() const {
  ppcsr_geometry g;
  if (ppcsr_geometry_of(shard_, &g) != PPCSR_OK) fail("ppcsr_geometry_of");
  return g.n;
}

node_t &PCSR::getNode(int id) {
  refresh_nodes();
  return nodes_[id];
}
const node_t &PCSR::getNode(int id) const {
  refresh_nodes();
  return nodes_[id];
}

bool PCSR::edge_exists(uint32_t src, uint32_t dest) {
  std::lock_guard<std::mutex> g(edges.global_lock->mutex());
  int e = 0;
  if (ppcsr_edge_exists(shard_, src, dest, &e, nullptr) != PPCSR_OK) fail("ppcsr_edge_exists");
  return e != 0;
}

void PCSR::add_node() {
  std::lock_guard<std::mutex> g(edges.global_lock->mutex());
  if (ppcsr_add_nodes(shard_, 1) != PPCSR_OK) fail("ppcsr_add_nodes");
  nodes_dirty_ = true;
  refresh_geometry();
}

void PCSR::add_edge(uint32_t src, uint32_t dest, uint32_t value) {
  std::lock_guard<std::mutex> g(edges.global_lock->mutex());
  if (ppcsr_add_edge(shard_, src, dest, value) != PPCSR_OK) fail("ppcsr_add_edge");
  nodes_dirty_ = true;
  refresh_geometry();
}

void PCSR::remove_edge(uint32_t src, uint32_t dest) {
  std::lock_guard<std::mutex> g(edges.global_lock->mutex());
  int found = 0;
  if (ppcsr_remove_edge(shard_, src, dest, &found) != PPCSR_OK) fail("ppcsr_remove_edge");
  if (!found && print_not_found) std::cout << "not found " << src << " " << dest << std::endl;
  nodes_dirty_ = true;
  refresh_geometry();
}

void PCSR::read_neighbourhood(int src) {
  if (src < 0) return;
  std::lock_guard<std::mutex> g(edges.global_lock->mutex());
  if (ppcsr_read_neighbourhood(shard_, (uint32_t)src, nullptr) != PPCSR_OK) fail("ppcsr_read_neighbourhood");
}

std::vector<int> PCSR::get_neighbourhood(int src) const {
  std::vector<int> out;
  if (src < 0) return out;
  std::lock_guard<std::mutex> g(edges.global_lock->mutex());
  uint64_t deg = 0;
  if (ppcsr_neighbours(shard_, (uint32_t)src, nullptr, 0, &deg) != PPCSR_OK) fail("ppcsr_neighbours");
  if (deg == 0) return out;
  std::vector<uint32_t> tmp(deg);
  if (ppcsr_neighbours(shard_, (uint32_t)src, tmp.data(), deg, &deg) != PPCSR_OK) fail("ppcsr_neighbours");
  out.assign(tmp.begin(), tmp.end());
  return out;
}

float PCSR::apply_batch(const std::vector<uint32_t> &src, const std::vector<uint32_t> &dst,
                        const std::vector<uint32_t> &value, ppcsr_batch_stats *stats) {
  return apply_batch(src.data(), dst.data(), value.empty() ? nullptr : value.data(), src.size(), stats);
}

float PCSR::apply_batch(const uint32_t *src, const uint32_t *dst, const uint32_t *value, size_t count,
                        ppcsr_batch_stats *stats) {
  std::lock_guard<std::mutex> g(edges.global_lock->mutex());
  ppcsr_batch_stats st{};
  if (ppcsr_apply_batch(shard_, src, dst, value, count, 1, &st) != PPCSR_OK) fail("ppcsr_apply_batch");
  batch_applied();
  if (stats) *stats = st;
  return st.ms_total;
}

float PCSR::apply_batch_pairs(const uint32_t *pairs, size_t count, uint32_t default_val, ppcsr_batch_stats *stats) {
  std::lock_guard<std::mutex> g(edges.global_lock->mutex());
  ppcsr_batch_stats st{};
  if (ppcsr_apply_batch_pairs(shard_, pairs, count, default_val, &st) != PPCSR_OK) fail("ppcsr_apply_batch_pairs");
  batch_applied();
  if (stats) *stats = st;
  return st.ms_total;
}

// after a batch went through the C-ABI behind this object's back (PPPCSR's group route) or through apply_batch
void PCSR::batch_applied() {
  nodes_dirty_ = true;
  refresh_geometry();
  ++(*lock_store_[0]);  // the version counter counts the batches that rewrote the structure
}

void PCSR::pagerank_push(const std::vector<double> &in, std::vector<double> &out) const {
  std::lock_guard<std::mutex> g(edges.global_lock->mutex());
  std::vector<double> part(out.size(), 0.0);
  if (ppcsr_pagerank_step_f64(shard_, in.data(), part.data(), part.size()) != PPCSR_OK) fail("ppcsr_pagerank_step");
  for (size_t i = 0; i < out.size(); i++) out[i] += part[i];
}

std::vector<uint32_t> PCSR::bfs_levels(uint32_t start) const {
  std::lock_guard<std::mutex> g(edges.global_lock->mutex());
  std::vector<uint32_t> d(get_n());
  if (ppcsr_bfs(shard_, start, d.data()) != PPCSR_OK) fail("ppcsr_bfs");
  return d;
}

std::vector<double> PCSR::pagerank(uint32_t iterations, double damping) const {
  std::lock_guard<std::mutex> g(edges.global_lock->mutex());
  std::vector<double> r(get_n());
  if (!r.empty() && ppcsr_pagerank(shard_, iterations, damping, r.data()) != PPCSR_OK) fail("ppcsr_pagerank");
  return r;
}

bool PCSR::check_invariants(bool check_lower, ppcsr_invariant_report *report) const {
  std::lock_guard<std::mutex> g(edges.global_lock->mutex());
  ppcsr_invariant_report r{};
  if (ppcsr_check_invariants(shard_, check_lower ? 1 : 0, &r) != PPCSR_OK) fail("ppcsr_check_invariants");
  if (report) *report = r;
  return !(r.bad_geometry || r.bad_sentinel || r.bad_order || r.bad_leaf_layout || r.bad_upper || r.bad_tree ||
           r.full_leaves || (check_lower && r.bad_lower));
}

void PCSR::insert_nodes_and_edges_front(std::vector<node_t> nodes, std::vector<edge_t> new_edges) {
  (void)nodes;
  (void)new_edges;
}
void PCSR::insert_nodes_and_edges_back(std::vector<node_t> nodes, std::vector<edge_t> new_edges) {
  (void)nodes;
  (void)new_edges;
}
std::pair<std::vector<node_t>, std::vector<edge_t>> PCSR::remove_nodes_and_edges_front(int num_nodes) {
  (void)num_nodes;
  return {};
}
std::pair<std::vector<node_t>, std::vector<edge_t>> PCSR::remove_nodes_and_edges_back(int num_nodes) {
  (void)num_nodes;
  return {};
}
