// cluster.cu — single-linkage ANI clustering of one sketch set (hg_cluster_*, DESIGN.md §4.9): a lock-free union-find
// over the linked pairs the dist kernels emit, in the style of ECL-CC (Jaiganesh & Burtscher) and Jayanti & Tarjan.
//
//   hook         unites (i, j) of every record of an edge list; the count is read on the device, from the dist
//                call's own counter, so the kernel can be enqueued behind a dist window without a host round trip;
//   hook_labels  unites (x, other[x]) for every x of another forest: the merge of forests built on different GPUs;
//   flatten      rep[x] = the root of x, and the number of roots;
//   check        caller-supplied edges and forests, before any find runs on them.
//
// The forest is parent[0, n) with the invariant parent[x] <= x; a root is a node with parent[x] == x.
//   - hook links a root under a root of smaller index, by atomicCAS on the larger root's own slot, expecting the root
//     itself: only a root is ever relinked.  When the CAS fails the slot holds that node's new parent, and the hook
//     retries from the root of that value.
//   - find shortens the path with plain stores (path splitting): each store points a non-root at one of its
//     ancestors, and ancestors have smaller indices.  No store writes a root's slot or makes a node its own parent.
// So the invariant holds under every interleaving, every path strictly descends (find terminates), and every root is
// the minimum of its tree.  Trees only merge, and only along edges, and every edge ends with both its ends in one tree;
// so once every edge is united there is one tree per connected component, rooted at the component's smallest index -
// whatever the order in which the edges were united and whichever thread won a CAS.
#include <algorithm>

#include "hg_common.cuh"

namespace {

constexpr int CL_THREADS = 256;

// the root of x; loads are volatile: other threads relink and shorten paths while this one walks
__device__ __forceinline__ uint32_t uf_find(uint32_t *parent, uint32_t x) {
  volatile uint32_t *p = parent;
  uint32_t cur = p[x];
  if (cur == x) return x;
  uint32_t prev = x, next;
  while (cur > (next = p[cur])) {  // cur is not a root: prev skips to its grandparent
    p[prev] = next;
    prev = cur;
    cur = next;
  }
  return cur;
}

__device__ __forceinline__ void uf_unite(uint32_t *parent, uint32_t a, uint32_t b) {
  uint32_t ra = uf_find(parent, a), rb = uf_find(parent, b);
  while (ra != rb) {
    const uint32_t lo = min(ra, rb), hi = max(ra, rb);
    const uint32_t old = atomicCAS(parent + hi, hi, lo);
    if (old == hi) return;
    // hi was linked under `old` meanwhile: its tree's root is now at or above old
    if (ra == hi) ra = uf_find(parent, old);
    else rb = uf_find(parent, old);
  }
}

__global__ void cluster_iota_kernel(uint32_t *__restrict__ parent, uint32_t n) {
  for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x)
    parent[x] = (uint32_t)x;
}

// edges: min(*count, cap) records (count NULL: cap); stats (may be NULL): [0] += that number, [1] = max([1], it)
__global__ void __launch_bounds__(CL_THREADS) cluster_hook_kernel(uint32_t *parent, const hg_hit *edges,
                                                                  const unsigned long long *count, uint64_t cap,
                                                                  unsigned long long *stats) {
  const uint64_t ne = count ? min((uint64_t)*count, cap) : cap;
  if (stats && blockIdx.x == 0 && threadIdx.x == 0) {
    stats[0] += ne;
    stats[1] = max((uint64_t)stats[1], ne);
  }
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < ne; t += (uint64_t)gridDim.x * blockDim.x)
    uf_unite(parent, edges[t].i, edges[t].j);
}

__global__ void __launch_bounds__(CL_THREADS) cluster_hook_labels_kernel(uint32_t *parent, const uint32_t *__restrict__ other,
                                                                         uint32_t n) {
  for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x)
    uf_unite(parent, (uint32_t)x, other[x]);
}

// Runs after every hook has finished, so the roots no longer change.  Each thread walks without shortening and writes
// only its own slot, with the root: a concurrent walk through that slot reads the old ancestor or the root, and
// no other store can land on it after this one.
__global__ void __launch_bounds__(CL_THREADS) cluster_flatten_kernel(uint32_t *parent, uint32_t n, uint32_t *n_roots) {
  volatile uint32_t *p = parent;
  for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < n; base += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t x = base + threadIdx.x;
    bool root = false;
    if (x < n) {
      uint32_t r = p[x], next;
      root = r == (uint32_t)x;
      while (r > (next = p[r])) r = next;
      p[x] = r;
    }
    const int c = __syncthreads_count(root);
    if (threadIdx.x == 0 && c) atomicAdd(n_roots, (uint32_t)c);
  }
}

// status |= 1: some edge index >= n; |= 2: some parent[x] > x (a forest that could hold a cycle)
__global__ void __launch_bounds__(CL_THREADS) cluster_check_kernel(const uint32_t *__restrict__ parent, uint32_t n,
                                                                   const hg_hit *__restrict__ edges, uint64_t n_edges,
                                                                   uint32_t *status) {
  const uint64_t from = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, step = (uint64_t)gridDim.x * blockDim.x;
  uint32_t bad = 0;
  for (uint64_t t = from; t < n_edges; t += step)
    if (edges[t].i >= n || edges[t].j >= n) bad |= 1u;
  for (uint64_t x = from; x < n; x += step)
    if (parent[x] > x) bad |= 2u;
  if (bad) atomicOr(status, bad);
}

uint32_t cl_grid(const hg_ctx *ctx, uint64_t items) {
  return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((items + CL_THREADS - 1) / CL_THREADS, (uint64_t)ctx->sm_count * 8));
}

}  // namespace

int hg_launch_cluster_iota(hg_ctx *ctx, uint32_t *d_parent, uint32_t n) {
  if (n == 0) return HG_OK;
  cluster_iota_kernel<<<cl_grid(ctx, n), CL_THREADS, 0, ctx->stream>>>(d_parent, n);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

int hg_launch_cluster_hook(hg_ctx *ctx, uint32_t *d_parent, const hg_hit *d_edges, const unsigned long long *d_count, uint64_t cap,
                           unsigned long long *d_stats) {
  if (cap == 0) return HG_OK;
  cluster_hook_kernel<<<cl_grid(ctx, cap), CL_THREADS, 0, ctx->stream>>>(d_parent, d_edges, d_count, cap, d_stats);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

int hg_launch_cluster_hook_labels(hg_ctx *ctx, uint32_t *d_parent, const uint32_t *d_other, uint32_t n) {
  if (n == 0) return HG_OK;
  cluster_hook_labels_kernel<<<cl_grid(ctx, n), CL_THREADS, 0, ctx->stream>>>(d_parent, d_other, n);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

int hg_launch_cluster_flatten(hg_ctx *ctx, uint32_t *d_parent, uint32_t n, uint32_t *d_n_roots) {
  if (n == 0) return HG_OK;
  cluster_flatten_kernel<<<cl_grid(ctx, n), CL_THREADS, 0, ctx->stream>>>(d_parent, n, d_n_roots);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

int hg_launch_cluster_check(hg_ctx *ctx, const uint32_t *d_parent, uint32_t n, const hg_hit *d_edges, uint64_t n_edges,
                            uint32_t *d_status) {
  if (n == 0 && n_edges == 0) return HG_OK;
  cluster_check_kernel<<<cl_grid(ctx, std::max<uint64_t>(n, n_edges)), CL_THREADS, 0, ctx->stream>>>(d_parent, n, d_edges, n_edges,
                                                                                                     d_status);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}
