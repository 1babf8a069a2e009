// parallel-packed-csr (B200 build) -- command line driver with the reference's flags and stdout contract
// (reference src/main.cpp:111-189):
//   -threads= -size= -lock_free -insert -delete -pppcsrnuma -pppcsr -ppcsr -partitions_per_domain=
//   -core_graph= -update_file=
// Flags are matched by prefix in the same order as the reference, so the same ordering rules hold:
// -insert/-delete and -size= must come before -update_file=.  Input: one edge per line,
// `src<sep>dst[<sep>{1|0}]`, 1 = add, 0 = delete, absent = the default op (reference main.cpp:29-62).
// The core graph is loaded through the same insert path, then the first `size` updates are applied; each
// phase prints "Elapsed wall clock time: <ms>" -- benchmark scripts keep the second line
// (reference src/benchmarking/benchmark-strong-scaling.sh:116).
// Input path (SURVEY 8f rank 1): the text reader of the reference runs ON THE GPU (C-ABI ppcsr_parse_edge_list: same
// per-line rules, one thread per line), -host_parse selects the line-by-line host reader instead; a file named *.bin
// holds raw little-endian u32 (src, dst) pairs, *.bin3 (src, dst, op) triples (op 1 = add, 0 = delete) and is mmap'd.
// Extra: -gpus=<k> limits the GPUs used as partitions' domains; -check verifies the PMA invariants; -balanced cuts the
// partitions at edge-balanced vertex boundaries computed from the core graph instead of the reference's equal vertex
// counts (reference PPPCSR.cpp:20,27-29); -repartition (partitioned modes) recuts the partitions after the updates at
// boundaries balanced on the current out-degrees, moving the vertices and their edges between the devices, and prints
// "Repartition: moved <V> vertices <E> edges, <S> partitions rebuilt, <ms> ms" -- -check, -checksum and the traversals
// then run on the new layout; -checksum prints an order-independent checksum of the logical graph
// ("Graph checksum: edges <E> edge_hash <016x>").
// -batches=<k> cuts the update phase (the first `size` updates) into k consecutive batches of ceil(size / k) and streams
// them two ahead (-ppcsr: ppcsr_submit_batch / ppcsr_wait; partitioned modes: PPPCSR::submit_batch / wait_batch), so the
// copy (and, partitioned, the routing) of the next batch runs while the current one is applied; the second "Elapsed
// wall clock time" line covers the whole stream, "not found" sums over its batches.  Default 1: one batch.
// -not_found_lines turns change capture on for the update phase and prints one "not found <src> <dst>" line (global
// ids) per remove that missed, as the reference prints them (reference PCSR.cpp:751), in place of the
// "not found <N> edges" count: the same multiset of lines as the reference at -threads=1, batch by batch in ascending
// (src, dst) order rather than in call order.
// Traversals after the updates, on the devices (-ppcsr: one shard; partitioned modes: across all partitions):
//   -bfs=<start>         prints "BFS from <start>: reached <k> levels <L> hash <016x>": k reached vertices, L = 1 + the
//                        largest hop count (0 if nothing is reached), hash = sum mod 2^64 of
//                        mix64(v << 32 | dist[v]) over the reached v (mix64 = the splitmix64 finaliser)
//   -pagerank=<it>       prints "PageRank <it> iterations: sum <%.17g> max <%.17g>" of <it> iterations with damping 0.85
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <memory>
#include <string>
#include <tuple>
#include <vector>

#include "bfs.h"
#include "thread_pool.h"
#include "thread_pool_pppcsr.h"

enum class Operation { READ, ADD, DELETE };
using EdgeOp = std::tuple<Operation, int, int>;

static bool starts_with(const std::string &s, const char *prefix) { return s.rfind(prefix, 0) == 0; }

// Parses an edge list; returns the ops and the largest vertex id seen.
static std::pair<std::vector<EdgeOp>, int> read_input(const std::string &filename, Operation default_op) {
  std::ifstream f(filename);
  if (!f.good()) {
    std::cerr << "Invalid file" << std::endl;
    std::exit(EXIT_FAILURE);
  }
  std::vector<EdgeOp> ops;
  int max_id = 0;
  std::string line;
  while (std::getline(f, line)) {
    if (line.empty()) continue;
    const char *p = line.c_str();
    char *end = nullptr;
    const long s = std::strtol(p, &end, 10);
    if (end == p) continue;
    const char *q = (*end != '\0') ? end + 1 : end;  // exactly one separator character
    char *end2 = nullptr;
    const long d = std::strtol(q, &end2, 10);
    Operation op = default_op;
    if (end2 != q && *end2 != '\0' && *(end2 + 1) != '\0') {
      const char c = *(end2 + 1);
      if (c == '1') op = Operation::ADD;
      else if (c == '0') op = Operation::DELETE;
      else std::cerr << "Invalid operation";
    }
    max_id = std::max(max_id, (int)std::max(s, d));
    ops.emplace_back(op, (int)s, (int)d);
  }
  return {std::move(ops), max_id};
}

// A loaded edge list as three arrays (value 1 = add, 0 = delete): what the loaders hand to submit_bulk.
struct EdgeArrays {
  std::vector<uint32_t> src, dst, val;
  int max_id = 0;
  size_t size() const { return src.size(); }
};

static EdgeArrays from_ops(const std::vector<EdgeOp> &ops, int max_id) {
  EdgeArrays e;
  e.max_id = max_id;
  e.src.reserve(ops.size());
  e.dst.reserve(ops.size());
  e.val.reserve(ops.size());
  for (const auto &o : ops) {
    if (std::get<0>(o) == Operation::READ) continue;
    e.src.push_back((uint32_t)std::get<1>(o));
    e.dst.push_back((uint32_t)std::get<2>(o));
    e.val.push_back(std::get<0>(o) == Operation::ADD ? 1u : 0u);
  }
  return e;
}

static bool ends_with(const std::string &s, const char *suffix) {
  const size_t n = std::strlen(suffix);
  return s.size() >= n && s.compare(s.size() - n, n, suffix) == 0;
}

// mmap the whole file read-only; exits like the reference on a bad file (main.cpp:33-36)
static const char *map_file(const std::string &filename, size_t *bytes) {
  const int fd = open(filename.c_str(), O_RDONLY);
  struct stat st;
  if (fd < 0 || fstat(fd, &st) != 0) {
    std::cerr << "Invalid file" << std::endl;
    std::exit(EXIT_FAILURE);
  }
  *bytes = (size_t)st.st_size;
  const char *p = "";
  if (*bytes) {
    p = (const char *)mmap(nullptr, *bytes, PROT_READ, MAP_PRIVATE, fd, 0);
    if (p == MAP_FAILED) {
      std::cerr << "Invalid file" << std::endl;
      std::exit(EXIT_FAILURE);
    }
  }
  close(fd);
  return p;
}

// *.bin / *.bin3 are binary; anything else is the reference's text format, parsed on the GPU unless -host_parse
static EdgeArrays load_edges(const std::string &filename, Operation default_op, bool host_parse) {
  const uint32_t default_val = default_op == Operation::ADD ? 1u : 0u;
  if (ends_with(filename, ".bin") || ends_with(filename, ".bin3")) {
    const bool triples = ends_with(filename, ".bin3");
    size_t bytes = 0;
    const uint32_t *w = (const uint32_t *)map_file(filename, &bytes);
    const size_t stride = triples ? 3 : 2, count = bytes / (4 * stride);
    EdgeArrays e;
    e.src.resize(count);
    e.dst.resize(count);
    e.val.resize(count);
    uint32_t top = 0;
    for (size_t i = 0; i < count; i++) {
      e.src[i] = w[i * stride];
      e.dst[i] = w[i * stride + 1];
      e.val[i] = triples ? (w[i * stride + 2] ? 1u : 0u) : default_val;
      top = std::max(top, std::max(e.src[i], e.dst[i]));
    }
    e.max_id = (int)std::min<uint32_t>(top, 0x7FFFFFFFu);
    if (bytes) munmap((void *)w, bytes);
    return e;
  }
  if (host_parse) {
    auto r = read_input(filename, default_op);
    return from_ops(r.first, r.second);
  }
  size_t bytes = 0;
  const char *text = map_file(filename, &bytes);
  uint32_t *ds = nullptr, *dd = nullptr, *dv = nullptr, top = 0;
  uint64_t lines = 0, parsed = 0;
  if (ppcsr_parse_edge_list(0, text, bytes, default_val, &ds, &dd, &dv, &lines, &parsed, &top) != PPCSR_OK) {
    std::cout << "ppcsr_parse_edge_list failed: " << ppcsr_last_error() << ". Abort\n";
    std::exit(EXIT_FAILURE);
  }
  EdgeArrays e;
  e.src.resize(lines);
  e.dst.resize(lines);
  e.val.resize(lines);
  if (lines) {
    ppcsr_copy_to_host(0, e.src.data(), ds, lines * 4);
    ppcsr_copy_to_host(0, e.dst.data(), dd, lines * 4);
    ppcsr_copy_to_host(0, e.val.data(), dv, lines * 4);
  }
  ppcsr_free_device(0, ds);
  ppcsr_free_device(0, dd);
  ppcsr_free_device(0, dv);
  e.max_id = (int)std::min<uint32_t>(top, 0x7FFFFFFFu);
  if (bytes) munmap((void *)text, bytes);
  return e;
}

template <typename Pool>
static void run_phase(const EdgeArrays &e, Pool *pool, int threads, size_t count) {
  pool->submit_bulk(e.src.data(), e.dst.data(), e.val.data(), std::min(count, e.size()));
  pool->start(threads);
  pool->stop();
}

template <typename Pool>
static void execute(int threads, int size, int batches, bool not_found_lines, const EdgeArrays &core,
                    const EdgeArrays &updates, std::unique_ptr<Pool> &pool) {
  run_phase(core, pool.get(), threads, core.size());
  pool->set_batches(batches);
  if (not_found_lines) pool->set_not_found_lines(true);
  run_phase(updates, pool.get(), threads, (size_t)size);
}

// first vertex of every partition such that the partitions hold about the same number of edges: deg[v] = out-degree
// of vertex v, n vertices
static std::vector<size_t> balanced_boundaries(const std::vector<uint64_t> &deg, size_t n, size_t parts) {
  std::vector<size_t> starts(parts, 0);
  uint64_t total = 0;
  for (size_t v = 0; v < n; v++) total += deg[v];
  uint64_t run = 0;
  size_t p = 1;
  for (size_t v = 0; v < n && p < parts; v++) {
    run += deg[v];
    while (p < parts && run * parts >= total * p) {
      starts[p] = std::min(std::max(v + 1, starts[p - 1] + 1), n - (parts - p));
      p++;
    }
  }
  for (; p < parts; p++) starts[p] = std::min(starts[p - 1] + 1, n - (parts - p));
  return starts;
}

// the core graph's out-degrees (sources >= n are not counted)
static std::vector<uint64_t> core_degrees(const EdgeArrays &core, size_t n) {
  std::vector<uint64_t> deg(n + 1, 0);
  for (uint32_t s : core.src)
    if (s < n) deg[s]++;
  return deg;
}

// the current out-degrees of every vertex of a partitioned graph, from each partition's exported rowptr
static std::vector<uint64_t> current_degrees(PPPCSR &g) {
  std::vector<uint64_t> deg;
  for (std::size_t p = 0; p < g.partition_count(); p++) {
    std::vector<uint64_t> rowptr(g.partition(p).get_n() + 1);
    if (ppcsr_export_csr(g.partition(p).handle(), rowptr.data(), nullptr, nullptr, nullptr) != PPCSR_OK) {
      std::cout << "ppcsr_export_csr failed: " << ppcsr_last_error() << ". Abort\n";
      std::exit(EXIT_FAILURE);
    }
    for (size_t v = 0; v + 1 < rowptr.size(); v++) deg.push_back(rowptr[v + 1] - rowptr[v]);
  }
  return deg;
}

enum class Version { PPCSR, PPPCSR, PPPCSRNUMA };

static uint64_t mix64(uint64_t x) {
  x ^= x >> 30;
  x *= 0xBF58476D1CE4E5B9ull;
  x ^= x >> 27;
  x *= 0x94D049BB133111EBull;
  x ^= x >> 31;
  return x;
}

// the -bfs= and -pagerank= lines (see the header comment)
template <typename G>
static void run_traversals(G &graph, long bfs_start, long pr_iterations) {
  char buf[160];
  if (bfs_start >= 0) {
    const uint32_t s = (uint32_t)bfs_start;
    const std::vector<uint32_t> dist = bfs(graph, s);
    uint64_t reached = 0, hash = 0, levels = 0;
    for (size_t v = 0; v < dist.size(); v++) {
      if (dist[v] == UINT32_MAX) continue;
      reached++;
      hash += mix64(((uint64_t)v << 32) | dist[v]);
      levels = std::max<uint64_t>(levels, (uint64_t)dist[v] + 1);
    }
    snprintf(buf, sizeof(buf), "BFS from %u: reached %llu levels %llu hash %016llx", s, (unsigned long long)reached,
             (unsigned long long)levels, (unsigned long long)hash);
    std::cout << buf << std::endl;
  }
  if (pr_iterations >= 0) {
    const std::vector<double> r = graph.pagerank((uint32_t)pr_iterations, 0.85);
    double sum = 0, mx = 0;
    for (double x : r) {
      sum += x;
      mx = std::max(mx, x);
    }
    snprintf(buf, sizeof(buf), "PageRank %ld iterations: sum %.17g max %.17g", pr_iterations, sum, mx);
    std::cout << buf << std::endl;
  }
}

int main(int argc, char *argv[]) {
  int threads = 8, size = 1000000, num_nodes = 0, partitions_per_domain = 1, batches = 1;
  bool lock_search = true, insert = true, check = false, host_parse = false, balanced = false, checksum = false,
       repartition = false, not_found_lines = false;
  long bfs_start = -1, pr_iterations = -1;  // -bfs= / -pagerank= (negative: not requested)
  Version v = Version::PPPCSRNUMA;
  EdgeArrays core_graph, updates;
  for (int i = 1; i < argc; i++) {
    const std::string s(argv[i]);
    if (starts_with(s, "-threads=")) {
      threads = std::stoi(s.substr(9));
    } else if (starts_with(s, "-size=")) {
      size = std::stoi(s.substr(6));
    } else if (starts_with(s, "-lock_free")) {
      lock_search = false;
    } else if (starts_with(s, "-insert")) {
      insert = true;
    } else if (starts_with(s, "-delete")) {
      insert = false;
    } else if (starts_with(s, "-pppcsrnuma")) {
      v = Version::PPPCSRNUMA;
    } else if (starts_with(s, "-pppcsr")) {
      v = Version::PPPCSR;
    } else if (starts_with(s, "-ppcsr")) {
      v = Version::PPCSR;
    } else if (starts_with(s, "-partitions_per_domain=")) {
      partitions_per_domain = std::stoi(s.substr(23));
    } else if (starts_with(s, "-gpus=")) {
      setenv("PPCSR_GPUS", s.substr(6).c_str(), 1);
    } else if (starts_with(s, "-batches=")) {
      char *end = nullptr;
      const long k = std::strtol(s.c_str() + 9, &end, 10);
      if (end == s.c_str() + 9 || *end != '\0' || k < 1 || k > 0x7FFFFFFF) {
        std::cout << "Invalid -batches value (a number >= 1 expected): " << s.substr(9) << std::endl;
        return EXIT_FAILURE;
      }
      batches = (int)k;
    } else if (starts_with(s, "-bfs=")) {
      bfs_start = std::stol(s.substr(5));
    } else if (starts_with(s, "-pagerank=")) {
      pr_iterations = std::stol(s.substr(10));
    } else if (starts_with(s, "-checksum")) {
      checksum = true;
    } else if (starts_with(s, "-check")) {
      check = true;
    } else if (starts_with(s, "-host_parse")) {
      host_parse = true;
    } else if (starts_with(s, "-not_found_lines")) {
      not_found_lines = true;
    } else if (starts_with(s, "-repartition")) {
      repartition = true;
    } else if (starts_with(s, "-balanced")) {
      balanced = true;
    } else if (starts_with(s, "-core_graph=")) {
      core_graph = load_edges(s.substr(12), Operation::ADD, host_parse);
      num_nodes = std::max(num_nodes, core_graph.max_id);
    } else if (starts_with(s, "-update_file=")) {
      const std::string name = s.substr(13);
      std::cout << name << std::endl;
      updates = load_edges(name, insert ? Operation::ADD : Operation::DELETE, host_parse);
      num_nodes = std::max(num_nodes, updates.max_id);
      size = (int)std::min((size_t)size, updates.size());
    }
  }
  if (core_graph.size() == 0) {
    std::cout << "Core graph file not specified" << std::endl;
    return EXIT_FAILURE;
  }
  if (updates.size() == 0) {
    std::cout << "Updates file not specified" << std::endl;
    return EXIT_FAILURE;
  }
  std::cout << "Core graph size: " << core_graph.size() << std::endl;
  bool ok = true;
  uint64_t sum[3] = {0, 0, 0};  // -checksum: edges, edge hash, num_neighbors hash of the logical graph
  if (v == Version::PPCSR) {
    auto pool = std::make_unique<ThreadPool>(threads, lock_search, num_nodes + 1, partitions_per_domain);
    execute(threads, size, batches, not_found_lines, core_graph, updates, pool);
    const ppcsr_batch_stats &st = pool->last_stats();
    std::cout << "{\"updates\": " << st.batch_size << ", \"device_ms\": " << st.ms_total
              << ", \"rebalance_bytes_per_update\": " << (st.batch_size ? (double)st.rebalance_bytes / st.batch_size : 0)
              << ", \"windows\": " << st.n_windows << ", \"slots\": " << st.slots_after << "}" << std::endl;
    if (check) ok = pool->pcsr->check_invariants(!insert);
    if (checksum) ppcsr_checksum(pool->pcsr->handle(), 0, sum);
    run_traversals(*pool->pcsr, bfs_start, pr_iterations);
  } else {
    std::unique_ptr<ThreadPoolPPPCSR> pool;
    if (balanced) {  // same number of partitions as the reference would make, cut where the core's edges balance
      int gpus = ppcsr_device_count();
      if (const char *e = std::getenv("PPCSR_GPUS")) gpus = std::min(gpus, std::max(1, std::atoi(e)));
      const size_t parts = (size_t)std::max(1, std::min(gpus, threads)) * (size_t)partitions_per_domain;
      pool = std::make_unique<ThreadPoolPPPCSR>(threads, lock_search, num_nodes + 1, partitions_per_domain,
                                                v == Version::PPPCSRNUMA,
                                                balanced_boundaries(core_degrees(core_graph, (size_t)num_nodes + 1),
                                                                    (size_t)num_nodes + 1, parts));
    } else {
      pool = std::make_unique<ThreadPoolPPPCSR>(threads, lock_search, num_nodes + 1, partitions_per_domain,
                                                v == Version::PPPCSRNUMA);
    }
    execute(threads, size, batches, not_found_lines, core_graph, updates, pool);
    const auto &sts = pool->last_stats();
    uint64_t upd = 0, bytes = 0, windows = 0;
    float device_ms = 0;
    for (const auto &st : sts) {
      upd += st.batch_size;
      bytes += st.rebalance_bytes;
      windows += st.n_windows;
      device_ms = std::max(device_ms, st.ms_total);
    }
    std::cout << "{\"updates\": " << upd << ", \"device_ms\": " << device_ms << ", \"rebalance_bytes_per_update\": "
              << (upd ? (double)bytes / upd : 0) << ", \"windows\": " << windows << ", \"partitions\": " << sts.size()
              << "}" << std::endl;
    if (repartition) {
      PPPCSR &g = *pool->pcsr;
      const std::vector<uint64_t> deg = current_degrees(g);
      const ppcsr_repartition_stats rs = g.repartition(balanced_boundaries(deg, deg.size(), g.partition_count()));
      char buf[160];
      snprintf(buf, sizeof(buf), "Repartition: moved %llu vertices %llu edges, %u partitions rebuilt, %.3f ms",
               (unsigned long long)rs.vertices_moved, (unsigned long long)rs.edges_moved, rs.shards_rebuilt,
               rs.ms_total);
      std::cout << buf << std::endl;
    }
    if (check) {
      for (std::size_t p = 0; p < pool->pcsr->partition_count(); p++)
        ok = pool->pcsr->partition(p).check_invariants(!insert) && ok;
    }
    if (checksum) {
      for (std::size_t p = 0; p < pool->pcsr->partition_count(); p++) {
        uint64_t part[3];
        ppcsr_checksum(pool->pcsr->partition(p).handle(), pool->pcsr->partition_start(p), part);
        for (int k = 0; k < 3; k++) sum[k] += part[k];
      }
    }
    run_traversals(*pool->pcsr, bfs_start, pr_iterations);
  }
  if (check) std::cout << "PMA invariants: " << (ok ? "ok" : "VIOLATED") << std::endl;
  if (checksum) {
    char buf[96];
    snprintf(buf, sizeof(buf), "Graph checksum: edges %llu edge_hash %016llx", (unsigned long long)sum[0],
             (unsigned long long)sum[1]);
    std::cout << buf << std::endl;
  }
  return ok ? 0 : 2;
}
