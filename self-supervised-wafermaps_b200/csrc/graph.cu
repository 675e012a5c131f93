// graph.cu — connected components of a sparse graph whose edges arrive in batches of CSR rows
// (near_duplicate_groups: the radius self-join, unioned batch by batch so that the edge list is
// never held whole).
//
// Union-find on one int32 parent array, parent[x] <= x for every x at all times: a union hooks the
// LARGER of two roots under the smaller with atomicCAS, and path halving only replaces a parent by
// its own parent.  A root therefore only ever gains a smaller parent, and once every edge is
// unioned the root of a component is its smallest member, whatever order the threads ran in: the
// labels are deterministic.
#include "common.cuh"
#include "kernels.h"

namespace b200knn {
namespace {

__device__ __forceinline__ int32_t load_parent(const int32_t* parent, int32_t x) {
  return *reinterpret_cast<const volatile int32_t*>(parent + x);
}

// root of x, with path halving (x's parent becomes its grandparent; a failed CAS means another
// thread already lowered it, which is as good)
__device__ __forceinline__ int32_t find_root(int32_t* parent, int32_t x) {
  while (true) {
    const int32_t p = load_parent(parent, x);
    if (p == x) return x;
    const int32_t g = load_parent(parent, p);
    if (g == p) return p;
    atomicCAS(parent + x, p, g);
    x = g;
  }
}

__device__ __forceinline__ void unite(int32_t* parent, int32_t a, int32_t b) {
  while (true) {
    a = find_root(parent, a);
    b = find_root(parent, b);
    if (a == b) return;
    if (a > b) {
      const int32_t t = a;
      a = b;
      b = t;
    }
    if (atomicCAS(parent + b, b, a) == b) return;  // else b gained a parent meanwhile: retry from it
  }
}

// One warp per CSR row: edges (row_offset + r, indices[j]) for j in [offsets[r], offsets[r + 1]),
// offsets relative to offsets[0].  An endpoint outside [0, n) is skipped and sets *err_flag = 2.
__global__ void __launch_bounds__(256)
    union_edges_kernel(int32_t* __restrict__ parent, int64_t n, const int64_t* __restrict__ offsets,
                       const int64_t* __restrict__ indices, int64_t n_rows, int64_t row_offset,
                       int32_t* __restrict__ err_flag) {
  const int lane = threadIdx.x & 31;
  const int64_t r = int64_t(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  const int64_t a = row_offset + r;
  const int64_t o0 = offsets[0];
  bool bad = false;
  for (int64_t j = offsets[r] - o0 + lane; j < offsets[r + 1] - o0; j += 32) {
    const int64_t b = indices[j];
    if (a < 0 || a >= n || b < 0 || b >= n) {
      bad = true;
      continue;
    }
    unite(parent, int32_t(a), int32_t(b));
  }
  if (bad) atomicExch(err_flag, 2);
}

// labels[x] = root of x (after every union: the smallest index of x's component)
__global__ void __launch_bounds__(256)
    components_kernel(const int32_t* __restrict__ parent, int64_t n, int64_t* __restrict__ labels) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int32_t x = int32_t(i);
  for (int32_t p = parent[x]; p != x; p = parent[x]) x = p;
  labels[i] = x;
}

}  // namespace

cudaError_t launch_union_edges(int32_t* parent, int64_t n, const int64_t* offsets, const int64_t* indices,
                               int64_t n_rows, int64_t row_offset, int32_t* err_flag, cudaStream_t stream) {
  if (n_rows == 0) return cudaSuccess;
  constexpr int kWarps = 8;
  union_edges_kernel<<<unsigned((n_rows + kWarps - 1) / kWarps), kWarps * 32, 0, stream>>>(
      parent, n, offsets, indices, n_rows, row_offset, err_flag);
  return cudaGetLastError();
}

cudaError_t launch_components(const int32_t* parent, int64_t n, int64_t* labels, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  components_kernel<<<unsigned((n + 255) / 256), 256, 0, stream>>>(parent, n, labels);
  return cudaGetLastError();
}

}  // namespace b200knn
