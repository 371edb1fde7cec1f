// components.cuh -- connected components of the resident operator (cs_b200_components).
//
// The same labelling as Graphs.connected_components / graph.connected_components: an edge is a
// stored off-diagonal entry with a non-zero value, components are numbered in order of their
// smallest node.  Union-find in the style of ECL-CC (Jaiganesh & Burtscher, HPDC 2018):
//   k_cc_init      parent[v] = min(v, smallest neighbour)            one thread per node
//   k_cc_hook      for every stored edge (v, u): find both roots (path halving), hook the LARGER root
//                  under the smaller one with atomicCAS, retry from the value the CAS saw
//   k_cc_flatten   parent[v] = root(v); flag[v] = (root(v) == v)
//   exclusive scan flag -> ordinal of every root (ras::exclusive_scan)
//   k_cc_label     label[v] = ordinal[parent[v]]
// Every write keeps parent[x] <= x, so the root of a finished tree is its minimum node and the
// ordinals come out in the order of the smallest node -- the result is unique, so it does not depend
// on the order in which the threads hooked.  The number of passes over the CSR does not depend on
// the graph's diameter (plain min-label propagation needs one sweep per hop).
#pragma once
#include <cstdint>

namespace ccl {

// root of v with path halving; parent[] is read and written concurrently by other threads, so every
// access goes through a volatile pointer (a racing write only ever replaces a parent by an ancestor)
__device__ __forceinline__ int find_root(volatile int* parent, int v) {
  int cur = parent[v];
  if (cur == v) return v;
  int prev = v, next;
  while (cur > (next = parent[cur])) {
    parent[prev] = next;
    prev = cur;
    cur = next;
  }
  return cur;
}

template <typename T>
__global__ void k_cc_init(int n, const int* __restrict__ rowptr, const int* __restrict__ colidx,
                          const T* __restrict__ vals, int* __restrict__ parent) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < n; v += gridDim.x * blockDim.x) {
    int m = v;
    for (int j = rowptr[v]; j < rowptr[v + 1]; ++j) {
      const int u = colidx[j];
      if (u < m && vals[j] != T(0)) m = u;
    }
    parent[v] = m;
  }
}

template <typename T>
__global__ void k_cc_hook(int n, const int* __restrict__ rowptr, const int* __restrict__ colidx,
                          const T* __restrict__ vals, int* parent) {
  volatile int* p = parent;
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < n; v += gridDim.x * blockDim.x) {
    const int beg = rowptr[v], end = rowptr[v + 1];
    for (int j = beg; j < end; ++j) {
      const int u = colidx[j];
      if (u == v || vals[j] == T(0)) continue;
      int a = find_root(p, v), b = find_root(p, u);
      while (a != b) {
        if (a < b) { const int t = a; a = b; b = t; }      // a: the larger root, hooked under b
        const int seen = atomicCAS(parent + a, a, b);
        if (seen == a) break;
        a = seen;                                          // a was hooked meanwhile: climb from its parent
        a = find_root(p, a);
      }
    }
  }
}

// after k_cc_hook every root is final; other threads shorten the paths this one walks, which only
// replaces a parent by an ancestor
__global__ void k_cc_flatten(int n, int* parent, int* __restrict__ flag) {
  volatile int* p = parent;
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < n; v += gridDim.x * blockDim.x) {
    int r = p[v];
    while (p[r] != r) r = p[r];
    p[v] = r;
    flag[v] = r == v ? 1 : 0;
  }
}

__global__ void k_cc_label(int n, const int* __restrict__ parent, const int* __restrict__ ordinal,
                           int* __restrict__ label) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < n; v += gridDim.x * blockDim.x)
    label[v] = ordinal[parent[v]];
}

}  // namespace ccl
