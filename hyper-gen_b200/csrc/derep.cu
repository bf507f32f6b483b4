// derep.cu — greedy ANI dereplication of one sketch set (hg_derep_*, DESIGN.md §4.10): the kernels around the dist
// windows and the top-1 search that api.cu's driver runs.
//
// Everything works in the permuted index space: row t of the working matrix is sketch order[t].
//   gather    rows idx[t] of a matrix (and their norms) into a contiguous matrix: the permutation, and the rep matrix;
//   mark      behind each dist window of column chunk [a, a + w): an edge (i, j) with i < a covers j when i is a
//             representative (is_rep of earlier chunks is final by then); an edge with i >= a sets bit i - a of row
//             j - a of the chunk's adjacency bitmap;
//   greedy    behind the last window of a chunk, one CTA: t is a representative iff it is not covered and no earlier
//             representative of the chunk is adjacent to it.  It writes is_rep for the chunk, appends the chunk's
//             representatives to the rep list in ascending t, and clears the bitmap and the flags for the next chunk;
//   finalize  after the search of every row against the rep matrix: rep[order[t]] = order[representative of t].
#include <algorithm>

#include "hg_common.cuh"

namespace {

constexpr int DR_THREADS = 256;
constexpr uint32_t DR_WORDS = HG_DEREP_CHUNK / 32;  // bitmap words per row
constexpr size_t DR_SMEM = (size_t)HG_DEREP_CHUNK * DR_WORDS * 4;  // the greedy step's staged bitmap rows (128 KB)
static_assert(DR_WORDS == 32, "the greedy scan keeps one word of the chunk's representative mask per lane");

// row t of dst = row idx[t] of src; 16-byte copies, hv_d % 256 == 0
__global__ void __launch_bounds__(DR_THREADS) derep_gather_kernel(const int16_t *__restrict__ src, const int32_t *__restrict__ src_norm,
                                                                  const uint32_t *__restrict__ idx, uint32_t m, uint32_t hv_d,
                                                                  int16_t *__restrict__ dst, int32_t *__restrict__ dst_norm) {
  const uint32_t vec = hv_d / 8;  // uint4 per row
  for (uint32_t t = blockIdx.x; t < m; t += gridDim.x) {
    const uint32_t s = idx[t];
    const uint4 *from = reinterpret_cast<const uint4 *>(src + (size_t)s * hv_d);
    uint4 *to = reinterpret_cast<uint4 *>(dst + (size_t)t * hv_d);
    for (uint32_t v = threadIdx.x; v < vec; v += blockDim.x) to[v] = from[v];
    if (threadIdx.x == 0) dst_norm[t] = src_norm[s];
  }
}

// edges: min(*count, cap) records of one window of column chunk [a, a + w); linked (may be NULL) += that number
__global__ void __launch_bounds__(DR_THREADS) derep_mark_kernel(const hg_hit *__restrict__ edges, const unsigned long long *count,
                                                                uint64_t cap, uint32_t a, uint32_t w, const uint8_t *__restrict__ is_rep,
                                                                uint8_t *covered, uint32_t *adj, unsigned long long *linked) {
  const uint64_t ne = min((uint64_t)*count, cap);
  if (linked && blockIdx.x == 0 && threadIdx.x == 0) *linked += ne;
  for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < ne; e += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t i = edges[e].i, jj = edges[e].j - a;  // the window's pairs have j in the chunk and i < j
    if (jj >= w) continue;
    if (i < a) {
      if (is_rep[i]) covered[jj] = 1;
    } else {
      const uint32_t ii = i - a;
      atomicOr(adj + (size_t)jj * DR_WORDS + (ii >> 5), 1u << (ii & 31));
    }
  }
}

// One CTA of HG_DEREP_CHUNK threads for the chunk [a, a + w).  The uncovered nodes are listed in order (covered flags
// 32 at a time by ballot); warp 0 walks that list with the chunk's representative mask spread over its lanes (lane l
// holds bits 32 l .. 32 l + 31): node t is a representative iff its bitmap row shares no bit with the mask.  The rows
// of the listed nodes are staged in shared memory first, so a step costs a shared load and one vote, not a memory
// round trip.
__global__ void __launch_bounds__(HG_DEREP_CHUNK) derep_greedy_kernel(uint32_t a, uint32_t w, uint8_t *covered, uint32_t *adj,
                                                                      uint8_t *is_rep, uint32_t *rep_list, uint32_t *n_reps) {
  extern __shared__ uint32_t rows[];  // DR_SMEM bytes: up to HG_DEREP_CHUNK rows of DR_WORDS words
  __shared__ uint16_t list[HG_DEREP_CHUNK];
  __shared__ uint32_t warp_base[DR_WORDS + 1], mask[DR_WORDS];
  const uint32_t t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const uint32_t lt = (1u << lane) - 1u;
  const bool unc = t < w && !covered[t];
  const uint32_t bal = __ballot_sync(0xffffffffu, unc);
  if (lane == 0) warp_base[warp] = __popc(bal);
  __syncthreads();
  if (warp == 0) {  // exclusive prefix over the warps' counts
    const uint32_t c = warp_base[lane];
    uint32_t s = c;
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t o = __shfl_up_sync(0xffffffffu, s, d);
      if (lane >= (uint32_t)d) s += o;
    }
    warp_base[lane] = s - c;
    if (lane == 31) warp_base[DR_WORDS] = s;
  }
  __syncthreads();
  if (unc) list[warp_base[warp] + __popc(bal & lt)] = (uint16_t)t;
  __syncthreads();
  // the bitmap rows of the uncovered nodes, in list order, staged in shared memory by the whole CTA (coalesced, every
  // load in flight at once); the walk then reads one 128-byte row per node from there
  const uint32_t total = warp_base[DR_WORDS];
  for (uint32_t v = t; v < total * DR_WORDS; v += blockDim.x) rows[v] = adj[(size_t)list[v / DR_WORDS] * DR_WORDS + v % DR_WORDS];
  __syncthreads();
  if (warp == 0) {
    uint32_t m = 0;
#pragma unroll 8
    for (uint32_t u = 0; u < total; u++) {
      const uint32_t node = list[u];
      if (!__any_sync(0xffffffffu, rows[u * DR_WORDS + lane] & m) && lane == (node >> 5)) m |= 1u << (node & 31);
    }
    mask[lane] = m;
  }
  __syncthreads();
  // the chunk's representatives: warp k's nodes are the bits of mask[k]; their slots in the list follow the prefix of
  // the earlier words' counts
  const uint32_t word = mask[warp];
  const bool rep = (word >> lane) & 1u;
  if (t < w) {
    is_rep[a + t] = rep;
    covered[t] = 0;
  }
  if (warp == 0) {
    const uint32_t c = __popc(mask[lane]);
    uint32_t s = c;
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t o = __shfl_up_sync(0xffffffffu, s, d);
      if (lane >= (uint32_t)d) s += o;
    }
    warp_base[lane] = s - c;
    if (lane == 31) warp_base[DR_WORDS] = s;
  }
  __syncthreads();
  const uint32_t first = *n_reps;
  if (rep) rep_list[first + warp_base[warp] + __popc(word & lt)] = a + t;
  // every row of the chunk is cleared for the next one (rows >= w are never set)
  uint4 *z = reinterpret_cast<uint4 *>(adj);
  for (uint32_t v = t; v < w * (DR_WORDS / 4); v += blockDim.x) z[v] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  if (t == 0) *n_reps = first + warp_base[DR_WORDS];
}

// rep_of[t]: t for a representative, else rep_list[out[t].i] (the first of the best representatives, by the search's
// tie rule); rep[order[t]] = order[rep_of[t]] (order NULL: the identity).  *status |= 1: a non-representative found
// no representative at the threshold.
__global__ void __launch_bounds__(DR_THREADS) derep_finalize_kernel(const uint8_t *__restrict__ is_rep, const uint32_t *__restrict__ rep_list,
                                                                    const hg_hit *__restrict__ out, const uint32_t *__restrict__ n_found,
                                                                    const uint32_t *__restrict__ order, uint32_t n, uint32_t *rep,
                                                                    uint32_t *status) {
  for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) {
    uint32_t r = t;
    if (!is_rep[t]) {
      if (n_found[t]) r = rep_list[out[t].i];
      else atomicOr(status, 1u);
    }
    rep[order ? order[t] : t] = order ? order[r] : r;
  }
}

uint32_t dr_grid(const hg_ctx *ctx, uint64_t items) {
  return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((items + DR_THREADS - 1) / DR_THREADS, (uint64_t)ctx->sm_count * 8));
}

}  // namespace

int hg_launch_derep_gather(hg_ctx *ctx, const int16_t *d_src, const int32_t *d_src_norm, const uint32_t *d_idx, uint32_t m,
                           uint32_t hv_d, int16_t *d_dst, int32_t *d_dst_norm) {
  if (m == 0) return HG_OK;
  derep_gather_kernel<<<std::min<uint32_t>(m, (uint32_t)ctx->sm_count * 16), DR_THREADS, 0, ctx->stream>>>(d_src, d_src_norm, d_idx, m,
                                                                                                            hv_d, d_dst, d_dst_norm);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

int hg_launch_derep_mark(hg_ctx *ctx, const hg_hit *d_edges, const unsigned long long *d_count, uint64_t cap, uint32_t a, uint32_t w,
                         const uint8_t *d_is_rep, uint8_t *d_covered, uint32_t *d_adj, unsigned long long *d_linked) {
  if (cap == 0) return HG_OK;
  derep_mark_kernel<<<dr_grid(ctx, cap), DR_THREADS, 0, ctx->stream>>>(d_edges, d_count, cap, a, w, d_is_rep, d_covered, d_adj, d_linked);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

int hg_launch_derep_greedy(hg_ctx *ctx, uint32_t a, uint32_t w, uint8_t *d_covered, uint32_t *d_adj, uint8_t *d_is_rep,
                           uint32_t *d_rep_list, uint32_t *d_n_reps) {
  if (w == 0 || w > HG_DEREP_CHUNK) { hg_set_error("hg_launch_derep_greedy: chunk width %u outside 1..%u", w, HG_DEREP_CHUNK); return HG_E_INVALID; }
  HG_CUDA(cudaFuncSetAttribute(derep_greedy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DR_SMEM));
  derep_greedy_kernel<<<1, HG_DEREP_CHUNK, DR_SMEM, ctx->stream>>>(a, w, d_covered, d_adj, d_is_rep, d_rep_list, d_n_reps);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

int hg_launch_derep_finalize(hg_ctx *ctx, const uint8_t *d_is_rep, const uint32_t *d_rep_list, const hg_hit *d_out,
                             const uint32_t *d_n_found, const uint32_t *d_order, uint32_t n, uint32_t *d_rep, uint32_t *d_status) {
  if (n == 0) return HG_OK;
  derep_finalize_kernel<<<dr_grid(ctx, n), DR_THREADS, 0, ctx->stream>>>(d_is_rep, d_rep_list, d_out, d_n_found, d_order, n, d_rep,
                                                                         d_status);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}
