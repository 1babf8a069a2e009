// Breadth-first search with the reference's signature (reference src/utility/bfs.h:15-36): hop counts
// from start_node, UINT32_MAX for unreached vertices.  Both graph types run level-synchronous GPU kernels:
// a PCSR on its one shard (ppcsr_bfs), a PPPCSR across all of its partitions (ppcsr_group_bfs).
#pragma once
#include <cstdint>
#include <vector>

#include "PCSR.h"
#include "PPPCSR.h"

template <typename T>
std::vector<uint32_t> bfs(T &graph, uint32_t start_node);

template <>
inline std::vector<uint32_t> bfs<PCSR>(PCSR &graph, uint32_t start_node) {
  return graph.bfs_levels(start_node);
}

template <>
inline std::vector<uint32_t> bfs<PPPCSR>(PPPCSR &graph, uint32_t start_node) {
  return graph.bfs_levels(start_node);
}
