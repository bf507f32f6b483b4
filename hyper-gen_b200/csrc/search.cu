// search.cu — the kernels of the top-k sketch search (hg_search_dev / hg_search_packed) around its dist passes:
//
//   gather   a strided sample of the ref rows, on which the floor pass runs;
//   select   the unordered candidate list of a pass -> per query the top_k best by the key (ANI desc, ref index i asc):
//            count per query, scan, scatter into per-query segments of 64-bit keys, then one block per query.
//            A segment of up to SEL_SORT keys is sorted whole in shared memory; a longer one (ties, or a query whose
//            floor is 0) first finds its top_k-th largest key by a radix select over the 64-bit key (8 passes of 8
//            bits), keeps the top_k keys at or above it and sorts those.  The pair enumeration emits every (i, j)
//            at most once, so the keys of a segment are distinct and the selected set is exact;
//   floors   the top_k-th key of every query after the floor pass -> the per-query threshold (hg_floor) of the main pass;
//   merge    the results of searches over contiguous ref blocks -> the result over all of them (hg_search_merge_dev).
//
// The key of a candidate is (ANI bits << 32) | ~i: ANI is a non-negative f32, so its bits order like the value, and the
// complemented index puts the smaller i first among equal ANIs.  No real key is 0 (that would need i = 2^32 - 1).
#include <algorithm>

#include "dist_common.cuh"

namespace {

constexpr int SEL_THREADS = 512;
constexpr int SEL_SORT = 2048;  // >= the largest top_k (1024): what the radix select keeps always fits

__device__ __forceinline__ unsigned long long sel_key(const uint4 &h) {  // hg_hit = {i, j, dot, ani}
  return ((unsigned long long)h.w << 32) | (unsigned long long)(~h.x);
}

// sample row t = ref row floor(t * n_ref / s): spread over the whole ref set, ascending in t
__global__ void gather_rows_kernel(const int16_t *__restrict__ ref, const int32_t *__restrict__ ref_norm, uint32_t n_ref, uint32_t hv_d,
                                   uint32_t s, int16_t *__restrict__ out, int32_t *__restrict__ out_norm) {
  const uint32_t t = blockIdx.x;
  const uint64_t src = (uint64_t)t * n_ref / s;
  const uint4 *a = reinterpret_cast<const uint4 *>(ref + src * hv_d);
  uint4 *b = reinterpret_cast<uint4 *>(out + (uint64_t)t * hv_d);
  for (uint32_t e = threadIdx.x; e < hv_d / 8; e += blockDim.x) b[e] = a[e];
  if (threadIdx.x == 0) out_norm[t] = ref_norm[src];
}

__global__ void seg_count_kernel(const uint4 *__restrict__ cand, uint64_t n, uint32_t *__restrict__ cnt) {
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (uint64_t)gridDim.x * blockDim.x)
    atomicAdd(cnt + cand[t].y, 1u);
}

// off[q] = sum of cnt[0..q) for q = 0..n (one block; every thread owns a contiguous run)
__global__ void __launch_bounds__(1024) seg_scan_kernel(const uint32_t *__restrict__ cnt, uint32_t n, unsigned long long *__restrict__ off) {
  __shared__ unsigned long long s_warp[32];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t items = (n + 1023) / 1024;
  const uint32_t b = threadIdx.x * items, e = min(b + items, n);
  unsigned long long sum = 0;
  for (uint32_t q = b; q < e; ++q) sum += cnt[q];
  unsigned long long x = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= (uint32_t)o) x += y;
  }
  if (lane == 31) s_warp[warp] = x;
  __syncthreads();
  if (warp == 0) {
    const unsigned long long w = s_warp[lane];
    unsigned long long ws = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long y = __shfl_up_sync(0xffffffffu, ws, o);
      if (lane >= (uint32_t)o) ws += y;
    }
    s_warp[lane] = ws - w;
  }
  __syncthreads();
  unsigned long long run = s_warp[warp] + x - sum;
  for (uint32_t q = b; q < e; ++q) {
    off[q] = run;
    run += cnt[q];
  }
  if (threadIdx.x == 1023) off[n] = run;
}

// candidate t -> its query's segment (order inside a segment is arbitrary); cursor starts at 0
__global__ void seg_scatter_kernel(const uint4 *__restrict__ cand, uint64_t n, const unsigned long long *__restrict__ off,
                                   uint32_t *__restrict__ cursor, unsigned long long *__restrict__ keys, int32_t *__restrict__ dots) {
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (uint64_t)gridDim.x * blockDim.x) {
    const uint4 h = cand[t];
    const unsigned long long pos = off[h.y] + atomicAdd(cursor + h.y, 1u);
    keys[pos] = sel_key(h);
    dots[pos] = (int32_t)h.z;
  }
}

// One block per query: its top_k best in key order.  out / n_found / milli (each may be NULL) as hg_search_dev writes
// them; floor_key (may be NULL): the top_k-th key, or 0 if fewer than top_k candidates.
__global__ void __launch_bounds__(SEL_THREADS)
seg_select_kernel(const unsigned long long *__restrict__ off, const unsigned long long *__restrict__ keys, const int32_t *__restrict__ dots,
                  uint32_t top_k, hg_hit *__restrict__ out, uint32_t *__restrict__ n_found, uint32_t *__restrict__ milli,
                  unsigned long long *__restrict__ floor_key) {
  __shared__ unsigned long long s_key[SEL_SORT];
  __shared__ uint32_t s_pos[SEL_SORT];
  __shared__ uint32_t s_hist[256];
  __shared__ unsigned long long s_pref;
  __shared__ uint32_t s_want, s_n;
  const uint32_t j = blockIdx.x, tid = threadIdx.x;
  const unsigned long long b = off[j];
  const uint64_t L = off[j + 1] - b;
  const unsigned long long *K = keys + b;
  const uint32_t nf = L < top_k ? (uint32_t)L : top_k;
  uint32_t m;  // keys to sort
  if (L <= SEL_SORT) {
    for (uint32_t e = tid; e < L; e += SEL_THREADS) { s_key[e] = K[e]; s_pos[e] = e; }
    m = (uint32_t)L;
  } else {
    // radix select of the top_k-th largest key, most significant byte first
    unsigned long long prefix = 0, mask = 0;
    uint32_t want = top_k;
    for (int shift = 56; shift >= 0; shift -= 8) {
      if (tid < 256) s_hist[tid] = 0;
      __syncthreads();
      for (uint64_t e = tid; e < L; e += SEL_THREADS) {
        const unsigned long long k = K[e];
        if ((k & mask) == prefix) atomicAdd(s_hist + ((k >> shift) & 255u), 1u);
      }
      __syncthreads();
      if (tid == 0) {
        uint32_t above = 0;
        for (int d = 255; d >= 0; --d) {
          if (above + s_hist[d] >= want) {
            s_pref = prefix | ((unsigned long long)d << shift);
            s_want = want - above;
            break;
          }
          above += s_hist[d];
        }
      }
      __syncthreads();
      prefix = s_pref;
      want = s_want;
      mask |= 255ull << shift;
    }
    // prefix is the top_k-th largest key: exactly top_k keys are >= it
    if (tid == 0) s_n = 0;
    __syncthreads();
    for (uint64_t e = tid; e < L; e += SEL_THREADS) {
      const unsigned long long k = K[e];
      if (k >= prefix) {
        const uint32_t p = atomicAdd(&s_n, 1u);
        s_key[p] = k;
        s_pos[p] = (uint32_t)e;
      }
    }
    m = top_k;
  }
  uint32_t P = 1;
  while (P < m) P <<= 1;
  for (uint32_t e = m + tid; e < P; e += SEL_THREADS) s_key[e] = 0ull;  // pads sort last
  __syncthreads();
  // bitonic sort, descending
  for (uint32_t k = 2; k <= P; k <<= 1)
    for (uint32_t h = k >> 1; h > 0; h >>= 1) {
      for (uint32_t e = tid; e < P; e += SEL_THREADS) {
        const uint32_t o = e ^ h;
        if (o > e) {
          const unsigned long long a = s_key[e], c = s_key[o];
          if (((e & k) == 0) ? a < c : a > c) {
            s_key[e] = c; s_key[o] = a;
            const uint32_t t = s_pos[e]; s_pos[e] = s_pos[o]; s_pos[o] = t;
          }
        }
      }
      __syncthreads();
    }
  if (out)
    for (uint32_t r = tid; r < top_k; r += SEL_THREADS) {
      hg_hit hit = {0u, 0u, 0, 0.0f};
      uint32_t mi = 0;
      if (r < nf) {
        const unsigned long long k = s_key[r];
        hit.i = ~(uint32_t)k;
        hit.j = j;
        hit.dot = dots[b + s_pos[r]];
        hit.ani = __uint_as_float((uint32_t)(k >> 32));
        mi = (uint32_t)__double2ll_rn((double)hit.ani * 1000.0);  // as ani_milli_kernel (sort.cu)
      }
      out[(uint64_t)j * top_k + r] = hit;
      if (milli) milli[(uint64_t)j * top_k + r] = mi;
    }
  if (tid == 0) {
    if (n_found) n_found[j] = nf;
    if (floor_key) floor_key[j] = L >= top_k ? s_key[top_k - 1] : 0ull;
  }
}

// the floor pass's top_k-th key of every query -> the main pass's per-query thresholds; cfrac_row as hg_floors asks.
// The key's index is a sample row t: ref row floor(t * n_ref / s), as gather_rows_kernel took it.
__global__ void __launch_bounds__(1024) floor_prep_kernel(const unsigned long long *__restrict__ floor_key, uint32_t n_qry, float ani_min,
                                                          uint32_t ksize, uint32_t n_ref, uint32_t s, hg_floor *__restrict__ q,
                                                          float *__restrict__ cfrac_row) {
  __shared__ float s_min[32];
  float mn = INFINITY;
  for (uint32_t j = threadIdx.x; j < n_qry; j += 1024) {
    const unsigned long long k = floor_key[j];
    hg_floor f;
    f.ani = k ? __uint_as_float((uint32_t)(k >> 32)) : ani_min;
    f.imax = k ? (uint32_t)((uint64_t)(~(uint32_t)k) * n_ref / s) : 0xFFFFFFFFu;
    f.jmin = hg::dist_jmin(f.ani, ksize);
    f.cfrac = f.jmin > 0.0f ? (float)((double)f.jmin / (1.0 + (double)f.jmin)) : 0.0f;
    q[j] = f;
    if (f.cfrac > 0.0f) mn = fminf(mn, f.cfrac);
  }
  for (int o = 16; o > 0; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
  if ((threadIdx.x & 31) == 0) s_min[threadIdx.x >> 5] = mn;
  __syncthreads();
  if (threadIdx.x < 32) {
    mn = s_min[threadIdx.x];
    for (int o = 16; o > 0; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    if (threadIdx.x == 0) *cfrac_row = mn < INFINITY ? mn : 0.0f;
  }
}

// Merge of n_lists per-block results (each as hg_search_dev writes it, block m's ref indices offset by i0[m]) into one,
// by rank: live element p of list m for query j has the output rank p + #(keys >= its key in the lists before m) +
// #(keys > its key in the lists after m), each count a binary search in a list that is already in key order.  Keys are
// distinct within a list, so the ranks are a permutation of 0 .. sum(n_found) - 1 - the asymmetric >= / > keeps them
// one even when the same key is in two lists.  The thread of list 0 at position p also zeroes output slot p if it is
// unused.  status: bit 0 = some i + i0 does not fit 32 bits, bit 1 = some n_found above top_k (counted as top_k).
struct MergeOffsets { uint32_t i0[HG_SEARCH_MERGE_MAX_LISTS]; };

__device__ __forceinline__ unsigned long long merge_key(const uint4 &h, uint32_t i0) {
  return ((unsigned long long)h.w << 32) | (unsigned long long)(~(h.x + i0));
}

__device__ __forceinline__ uint32_t merge_found(const uint32_t *in_found, uint32_t m, uint32_t n_qry, uint32_t j, uint32_t top_k,
                                                uint32_t *status) {
  const uint32_t nf = in_found[(uint64_t)m * n_qry + j];
  if (nf > top_k) { atomicOr(status, 2u); return top_k; }
  return nf;
}

__global__ void search_merge_kernel(const uint4 *__restrict__ in, const uint32_t *__restrict__ in_found, MergeOffsets off,
                                    uint32_t n_lists, uint32_t n_qry, uint32_t top_k, hg_hit *__restrict__ out,
                                    uint32_t *__restrict__ n_found, uint32_t *__restrict__ milli, uint32_t *__restrict__ status) {
  const uint64_t total = (uint64_t)n_lists * n_qry * top_k;
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t p = (uint32_t)(t % top_k);
    const uint64_t r = t / top_k;
    const uint32_t j = (uint32_t)(r % n_qry), m = (uint32_t)(r / n_qry);
    const uint64_t o = (uint64_t)j * top_k;
    if (m == 0) {
      uint64_t sum = 0;
      for (uint32_t l = 0; l < n_lists; ++l) sum += merge_found(in_found, l, n_qry, j, top_k, status);
      const uint32_t nf = sum < top_k ? (uint32_t)sum : top_k;
      if (p == 0) n_found[j] = nf;
      if (p >= nf) {
        out[o + p] = hg_hit{0u, 0u, 0, 0.0f};
        if (milli) milli[o + p] = 0;
      }
    }
    if (p >= merge_found(in_found, m, n_qry, j, top_k, status)) continue;
    const uint4 h = in[((uint64_t)m * n_qry + j) * top_k + p];
    if ((uint64_t)h.x + off.i0[m] > 0xFFFFFFFFull) { atomicOr(status, 1u); continue; }
    const unsigned long long key = merge_key(h, off.i0[m]);
    uint32_t rank = p;
    for (uint32_t l = 0; l < n_lists && rank < top_k; ++l) {
      if (l == m) continue;
      const uint4 *L = in + ((uint64_t)l * n_qry + j) * top_k;
      uint32_t lo = 0, hi = merge_found(in_found, l, n_qry, j, top_k, status);  // first position that does not count
      while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        const unsigned long long k = merge_key(L[mid], off.i0[l]);
        if (l < m ? k >= key : k > key) lo = mid + 1;
        else hi = mid;
      }
      rank += lo;
    }
    if (rank >= top_k) continue;
    hg_hit hit;
    hit.i = h.x + off.i0[m];
    hit.j = h.y;
    hit.dot = (int32_t)h.z;
    hit.ani = __uint_as_float(h.w);
    out[o + rank] = hit;
    if (milli) milli[o + rank] = (uint32_t)__double2ll_rn((double)hit.ani * 1000.0);  // as seg_select_kernel
  }
}

}  // namespace

int hg_launch_search_merge(hg_ctx *ctx, uint32_t n_lists, const hg_hit *d_in, const uint32_t *d_in_found, const uint32_t *i0,
                           uint32_t n_qry, uint32_t top_k, hg_hit *d_out, uint32_t *d_n_found, uint32_t *d_milli, uint32_t *d_status) {
  if (n_qry == 0) return HG_OK;
  MergeOffsets off = {};
  for (uint32_t m = 0; m < n_lists; ++m) off.i0[m] = i0[m];
  const uint64_t total = (uint64_t)n_lists * n_qry * top_k;
  const uint32_t grid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((total + 255) / 256, (uint64_t)ctx->sm_count * 16));
  search_merge_kernel<<<grid, 256, 0, ctx->stream>>>((const uint4 *)d_in, d_in_found, off, n_lists, n_qry, top_k, d_out, d_n_found,
                                                     d_milli, d_status);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

int hg_launch_search_gather(hg_ctx *ctx, const int16_t *d_ref, const int32_t *d_ref_norm, uint32_t n_ref, uint32_t hv_d, uint32_t s,
                            int16_t *d_out, int32_t *d_out_norm) {
  if (s == 0) return HG_OK;
  gather_rows_kernel<<<s, 256, 0, ctx->stream>>>(d_ref, d_ref_norm, n_ref, hv_d, s, d_out, d_out_norm);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

int hg_launch_search_select(hg_ctx *ctx, const hg_hit *d_cand, uint64_t n_cand, uint32_t n_qry, uint32_t top_k, hg_hit *d_out,
                            uint32_t *d_n_found, uint32_t *d_milli, unsigned long long *d_floor_key) {
  if (n_qry == 0) return HG_OK;
  int rc;
  void *d_seg, *d_cnt;
  if ((rc = hg_scratch(ctx, HG_S_SORT_TMP, n_cand * 12 + 256, &d_seg))) return rc;
  if ((rc = hg_scratch(ctx, HG_S_SORT_CNT, (size_t)n_qry * 12 + 264, &d_cnt))) return rc;
  unsigned long long *keys = (unsigned long long *)d_seg, *off = (unsigned long long *)d_cnt;
  int32_t *dots = (int32_t *)(keys + n_cand);
  uint32_t *cnt = (uint32_t *)(off + n_qry + 1);
  const uint32_t grid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((n_cand + 255) / 256, (uint64_t)ctx->sm_count * 8));
  HG_CUDA(cudaMemsetAsync(cnt, 0, (size_t)n_qry * 4, ctx->stream));
  seg_count_kernel<<<grid, 256, 0, ctx->stream>>>((const uint4 *)d_cand, n_cand, cnt);
  seg_scan_kernel<<<1, 1024, 0, ctx->stream>>>(cnt, n_qry, off);
  HG_CUDA(cudaMemsetAsync(cnt, 0, (size_t)n_qry * 4, ctx->stream));
  seg_scatter_kernel<<<grid, 256, 0, ctx->stream>>>((const uint4 *)d_cand, n_cand, off, cnt, keys, dots);
  seg_select_kernel<<<n_qry, SEL_THREADS, 0, ctx->stream>>>(off, keys, dots, top_k, d_out, d_n_found, d_milli, d_floor_key);
  ctx->launches += 4;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

int hg_launch_search_floors(hg_ctx *ctx, const unsigned long long *d_floor_key, uint32_t n_qry, float ani_min, uint32_t ksize,
                            uint32_t n_ref, uint32_t s, hg_floor *d_floors, float *d_cfrac_row) {
  floor_prep_kernel<<<1, 1024, 0, ctx->stream>>>(d_floor_key, n_qry, ani_min, ksize, n_ref, s, d_floors, d_cfrac_row);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}
