// encode.cu — stage 1b: hash set -> sketch hypervector -> norm -> quantise -> bit-pack,
// one CTA per genome, everything between the hash table and the packed bytes on-chip.
//
// Replaces, per genome, hd::encode_hash_hd_avx2 (reference src/hd.rs:15-92),
// dist::compute_hv_l2_norm (src/dist.rs:132-137) and hd::compress_hd_sketch
// (src/hd.rs:116-157); hg_unpack replaces hd::decompress_hd_sketch (src/hd.rs:184-212).
//
//   hv[64*i + p] = -n + 2 * sum_h bit_{pi(p)}( wyrng_word(h, i) ),  pi(p) = (p%4)*16 + p/4
//
// Design: the reference walks one RNG per hash sequentially; WyRng's state advances by a
// constant, so word i of hash h is a closed form and every (hash, chunk) pair is independent.
// A warp takes 32 chunks (one per lane) and a strided subset of the hashes; each lane sums
// its 64-bit words bit-sliced (Harley-Seal carry-save adders: ~1 LOP3 per 8 counter updates
// instead of 64 adds per word), then spills the vertical counters into int32 counters in
// shared memory.  min/max/sum-of-squares are block reductions, and the BitPacker8x stream is
// assembled from shared memory and written with one coalesced store per row.
#include "hg_common.cuh"

namespace {

constexpr int EN_THREADS = 512;
constexpr int EN_WARPS = EN_THREADS / 32;
constexpr int EN_BATCH = 4096;  // table slots / hashes staged per pass
constexpr int EN_UP = 10;       // planes for 8s, 16s, ... : per-lane counts up to 8191

__device__ __forceinline__ void csa(uint64_t &hi, uint64_t &lo, uint64_t a, uint64_t b, uint64_t c) {
  const uint64_t u = a ^ b;
  hi = (a & b) | (u & c);
  lo = u ^ c;
}

__device__ __forceinline__ int warp_min(int v) {
  for (int o = 16; o; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int warp_max(int v) {
  for (int o = 16; o; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ uint32_t warp_sum(uint32_t v) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// dynamic smem: [ int32 cnt[64][C+1] | int16 hv[D] | u64 hash[EN_BATCH] ]  (C = D/64; the +1 pad
// keeps both the per-chunk atomics and the per-dimension read-out bank-conflict free)
__global__ void __launch_bounds__(EN_THREADS, 2)
encode_kernel(const hg_genome_desc *__restrict__ desc, const uint64_t *__restrict__ tables,
              const uint32_t *__restrict__ counts, uint32_t hv_d, int16_t *__restrict__ out_hv,
              uint8_t *__restrict__ out_packed, uint8_t *__restrict__ out_bits,
              int32_t *__restrict__ out_norm2, uint32_t *__restrict__ out_n, uint32_t *__restrict__ status) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int32_t *s_cnt = reinterpret_cast<int32_t *>(smem_raw);
  const uint32_t C = hv_d / 64;  // hd.rs:34 num_chunk
  const uint32_t CP = C + 1;     // padded row length of s_cnt
  int16_t *s_hv = reinterpret_cast<int16_t *>(s_cnt + 64 * CP + 2);  // keeps s_hash 8-byte aligned
  uint64_t *s_hash = reinterpret_cast<uint64_t *>(smem_raw + (size_t)hv_d * 6 + 264);
  __shared__ uint32_t s_m;
  __shared__ int s_red[3][EN_WARPS];

  const uint32_t g = blockIdx.x;
  const hg_genome_desc gd = desc[g];
  const uint64_t *table = tables + gd.table_begin;
  const uint32_t slots = gd.table_slots;
  const uint32_t n = counts ? counts[g] : slots;  // dense list mode: every slot is a hash  // distinct sampled hashes (sketch.rs: kmer_hash_set.len())
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  for (uint32_t d = tid; d < 64 * CP; d += EN_THREADS) s_cnt[d] = 0;
  __syncthreads();  // an empty set never enters the batch loop: the read-out below sees other threads' cells

  // work split: chunk-blocks of 32 chunks x strided hash subsets
  const uint32_t nCB = (C + 31) / 32;
  const uint32_t S = nCB <= EN_WARPS ? EN_WARPS / nCB : 1;

  for (uint32_t base = 0; base < slots; base += EN_BATCH) {
    if (tid == 0) s_m = 0;
    __syncthreads();
    // ---- stage the non-empty slots of this slice, compacted ----
    const uint32_t lim = min(base + EN_BATCH, (slots + 31u) & ~31u);  // warp-uniform trip count
    for (uint32_t s = base + tid; s < lim; s += EN_THREADS) {
      const uint64_t h = s < slots ? table[s] : HG_EMPTY_SLOT;
      const bool have = s < slots && (!counts || h != HG_EMPTY_SLOT);  // dense list mode: u64::MAX is a hash too
      const uint32_t bal = __ballot_sync(0xffffffffu, have);
      uint32_t pos = 0;
      if (lane == 0 && bal) pos = atomicAdd(&s_m, (uint32_t)__popc(bal));
      pos = __shfl_sync(0xffffffffu, pos, 0);
      if (have) s_hash[pos + __popc(bal & ((1u << lane) - 1u))] = h;
    }
    __syncthreads();
    const uint32_t m = s_m;

    // ---- bit-sliced accumulation ----
    for (uint32_t item = warp; item < nCB * S; item += EN_WARPS) {
      const uint32_t cb = item % nCB, sub = item / nCB;
      const uint32_t chunk = cb * 32 + lane;
      if (chunk < C) {
        uint64_t ones = 0, twos = 0, fours = 0;
        uint64_t up[EN_UP];
#pragma unroll
        for (int q = 0; q < EN_UP; ++q) up[q] = 0;
        for (uint32_t idx = sub; idx < m; idx += 8 * S) {
          uint64_t w[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const uint32_t ii = idx + e * S;
            w[e] = ii < m ? hg::wyrng_word(s_hash[ii], chunk) : 0ull;  // zero words add nothing
          }
          uint64_t twoA, twoB, fourA, fourB, eight;
          csa(twoA, ones, ones, w[0], w[1]);
          csa(twoB, ones, ones, w[2], w[3]);
          csa(fourA, twos, twos, twoA, twoB);
          csa(twoA, ones, ones, w[4], w[5]);
          csa(twoB, ones, ones, w[6], w[7]);
          csa(fourB, twos, twos, twoA, twoB);
          csa(eight, fours, fours, fourA, fourB);
          // ripple the carry into the upper planes
          uint64_t carry = eight;
#pragma unroll
          for (int q = 0; q < EN_UP; ++q) {
            const uint64_t tq = up[q] & carry;
            up[q] ^= carry;
            carry = tq;
          }
        }
        // ---- spill the vertical counters: bit q of chunk `chunk` is dimension
        //      64*chunk + 4*(q%16) + q/16 (inverse of pi, hd.rs:61-87) ----
#pragma unroll
        for (int q = 0; q < 64; ++q) {
          uint32_t c = (uint32_t)((ones >> q) & 1) + 2u * (uint32_t)((twos >> q) & 1) +
                       4u * (uint32_t)((fours >> q) & 1);
#pragma unroll
          for (int u = 0; u < EN_UP; ++u) c += (uint32_t)((up[u] >> q) & 1) << (3 + u);
          const uint32_t p = 4u * (q & 15) + (q >> 4);
          if (c) atomicAdd(&s_cnt[p * CP + chunk], (int32_t)c);  // [p][chunk]: conflict-free across lanes
        }
      }
    }
    __syncthreads();
  }

  // ---- hv = 2*count - n in wrapping i16 (hd.rs:29,84-87), min / max / sum of squares ----
  int mn = 32767, mx = -32768;
  uint32_t sq = 0;
  for (uint32_t d = tid; d < hv_d; d += EN_THREADS) {
    const uint32_t cnt = (uint32_t)s_cnt[(d & 63) * CP + (d >> 6)];
    const int16_t hv = (int16_t)(uint16_t)(2u * cnt - n);
    s_hv[d] = hv;
    mn = min(mn, (int)hv);
    mx = max(mx, (int)hv);
    sq += (uint32_t)((int)hv * (int)hv);  // wrapping i32 (dist.rs:133-136)
  }
  mn = warp_min(mn); mx = warp_max(mx); sq = warp_sum(sq);
  if (lane == 0) { s_red[0][warp] = mn; s_red[1][warp] = mx; s_red[2][warp] = (int)sq; }
  __syncthreads();
  if (warp == 0) {
    const bool in = lane < EN_WARPS;
    mn = warp_min(in ? s_red[0][lane] : 32767);
    mx = warp_max(in ? s_red[1][lane] : -32768);
    sq = warp_sum(in ? (uint32_t)s_red[2][lane] : 0u);
    if (lane == 0) { s_red[0][0] = mn; s_red[1][0] = mx; s_red[2][0] = (int)sq; }
  }
  __syncthreads();
  mn = s_red[0][0]; mx = s_red[1][0]; sq = (uint32_t)s_red[2][0];

  // smallest b in 6..16 with -2^(b-1) <= min and max <= 2^(b-1)-1 (hd.rs:123-136)
  uint32_t b = 6;
  while (b < 16 && !(-(1 << (b - 1)) <= mn && mx <= (1 << (b - 1)) - 1)) ++b;
  if (b == 16 && tid == 0) atomicOr(status + 1, 1u);  // reference arithmetic breaks here (hd.rs:140)

  if (tid == 0) {
    out_bits[g] = (uint8_t)b;
    out_norm2[g] = (int32_t)sq;
    if (out_n) out_n[g] = n;
  }
  if (out_hv) {
    uint32_t *dst = reinterpret_cast<uint32_t *>(out_hv + (size_t)g * hv_d);
    const uint32_t *src = reinterpret_cast<const uint32_t *>(s_hv);
    for (uint32_t d = tid; d < hv_d / 2; d += EN_THREADS) dst[d] = src[d];
  }

  // ---- BitPacker8x layout (hd.rs:143-153): block of 256 values, lane l = idx%8, row
  //      r = idx/8; word j of lane l's b*32-bit stream lands at u32 index 8*j + l ----
  if (out_packed) {
    uint32_t *row = reinterpret_cast<uint32_t *>(out_packed + (size_t)g * 2 * hv_d);
    const uint32_t words = hv_d * b / 32, row_words = hv_d / 2;
    const uint32_t umask = b >= 16 ? 0xFFFFu : ((1u << b) - 1u);
    const int offset = 1 << (b - 1);
    for (uint32_t ow = tid; ow < row_words; ow += EN_THREADS) {
      uint32_t word = 0;
      if (ow < words) {
        const uint32_t blk = ow / (8 * b), rem = ow % (8 * b), j = rem / 8, l = rem % 8;
        const int16_t *v = s_hv + blk * 256 + l;
        const uint32_t bit0 = 32 * j;
        for (uint32_t r = bit0 / b; r < 32 && b * r < bit0 + 32; ++r) {
          const uint32_t u = (uint32_t)((int)v[8 * r] + offset) & umask;
          const int shv = (int)(b * r) - (int)bit0;
          word |= shv >= 0 ? (u << shv) : (u >> (-shv));
        }
      }
      row[ow] = word;  // bytes past b*hv_d/8 are zero-filled
    }
  }
}

// decompress_hd_sketch (hd.rs:184-212).  BitPacker8x keeps value 8r + l of a 256-value block at bit b*r of lane
// stream l, and word j of stream l at word 8j + l of the block: the 8 values of one "row" r sit at the same bit
// offset of 8 adjacent words.  One thread per row: two (or, when the field straddles a word, four) 16-byte loads,
// 8 funnel shifts, one 16-byte store of 8 int16.
__global__ void __launch_bounds__(256)
unpack_kernel(const uint8_t *__restrict__ packed, uint64_t row_stride, const uint8_t *__restrict__ bits, uint32_t n,
              uint32_t hv_d, int16_t *__restrict__ hv) {
  const uint32_t g = blockIdx.y;
  const uint32_t b = bits[g];
  const uint32_t *row = reinterpret_cast<const uint32_t *>(packed + (size_t)g * row_stride);
  const uint32_t umask = b >= 16 ? 0xFFFFu : ((1u << b) - 1u);
  const uint32_t offset = 1u << (b - 1);
  for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < hv_d / 8; t += gridDim.x * blockDim.x) {
    const uint32_t blk = t >> 5, r = t & 31;
    const uint32_t bit = b * r, j = bit >> 5, sh = bit & 31;
    const uint4 *wb = reinterpret_cast<const uint4 *>(row + blk * 8 * b + 8 * j);  // row_stride % 4 == 0, rows 16-byte aligned when it is % 16
    uint32_t lo[8], hi[8];
    if ((((uintptr_t)wb) & 15) == 0) {
      const uint4 a0 = wb[0], a1 = wb[1];
      lo[0] = a0.x; lo[1] = a0.y; lo[2] = a0.z; lo[3] = a0.w; lo[4] = a1.x; lo[5] = a1.y; lo[6] = a1.z; lo[7] = a1.w;
    } else {
      const uint32_t *w = reinterpret_cast<const uint32_t *>(wb);
#pragma unroll
      for (int l = 0; l < 8; ++l) lo[l] = w[l];
    }
#pragma unroll
    for (int l = 0; l < 8; ++l) hi[l] = 0;
    if (sh + b > 32) {  // the field continues in the next word of every lane stream (then j + 1 < b)
      if ((((uintptr_t)wb) & 15) == 0) {
        const uint4 a0 = wb[2], a1 = wb[3];
        hi[0] = a0.x; hi[1] = a0.y; hi[2] = a0.z; hi[3] = a0.w; hi[4] = a1.x; hi[5] = a1.y; hi[6] = a1.z; hi[7] = a1.w;
      } else {
        const uint32_t *w = reinterpret_cast<const uint32_t *>(wb) + 8;
#pragma unroll
        for (int l = 0; l < 8; ++l) hi[l] = w[l];
      }
    }
    uint32_t o[4];
#pragma unroll
    for (int l = 0; l < 8; l += 2) {
      const uint32_t u0 = (__funnelshift_r(lo[l], hi[l], sh) & umask) - offset;
      const uint32_t u1 = (__funnelshift_r(lo[l + 1], hi[l + 1], sh) & umask) - offset;
      o[l >> 1] = (u0 & 0xFFFFu) | (u1 << 16);
    }
    int16_t *dst = hv + (size_t)g * hv_d + 8 * (size_t)t;
    if ((((uintptr_t)dst) & 15) == 0) {
      *reinterpret_cast<uint4 *>(dst) = make_uint4(o[0], o[1], o[2], o[3]);
    } else {  // caller-provided matrix at an odd address
#pragma unroll
      for (int l = 0; l < 8; ++l) dst[l] = (int16_t)(uint16_t)(o[l >> 1] >> (16 * (l & 1)));
    }
  }
}

// In-place ascending bitonic sort of every genome's table (EMPTY = u64::MAX sorts last), so
// the first count[g] slots become the sorted, de-duplicated hash set (stage hook only).
__global__ void __launch_bounds__(1024) sort_tables_kernel(const hg_genome_desc *__restrict__ desc,
                                                           uint64_t *__restrict__ tables) {
  const hg_genome_desc gd = desc[blockIdx.x];
  volatile uint64_t *t = tables + gd.table_begin;
  const uint32_t n = gd.table_mask + 1;
  for (uint32_t k = 2; k <= n; k <<= 1) {
    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
      for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        const uint32_t ixj = i ^ j;
        if (ixj > i) {
          const uint64_t a = t[i], c = t[ixj];
          const bool asc = (i & k) == 0;
          if ((a > c) == asc) { t[i] = c; t[ixj] = a; }
        }
      }
      __syncthreads();
    }
  }
}

__global__ void absmax_kernel(const int16_t *__restrict__ hv, uint64_t n, int32_t *out) {
  int m = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const int v = hv[i];
    m = max(m, v < 0 ? -v : v);
  }
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

}  // namespace

int hg_launch_encode(hg_ctx *ctx, const hg_genome_desc *d_desc, uint32_t n_genomes, const uint64_t *d_tables,
                     const uint32_t *d_counts, uint32_t hv_d, int16_t *d_hv, uint8_t *d_packed,
                     uint8_t *d_quant_bits, int32_t *d_norm2, uint32_t *d_n_hashes) {
  if (n_genomes == 0) return HG_OK;
  const size_t smem = (size_t)hv_d * 6 + 264 + (size_t)EN_BATCH * 8;
  if (smem > 220 * 1024) {  // 6 B per dimension + the hash batch: hv_d <= 32000 (a multiple of 256)
    hg_set_error("hv_d %u too large for the on-chip encoder (max 32000; dist accepts up to 32768)", hv_d);
    return HG_E_UNSUPPORTED;
  }
  HG_CUDA(cudaFuncSetAttribute(encode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
  encode_kernel<<<n_genomes, EN_THREADS, smem, ctx->stream>>>(d_desc, d_tables, d_counts, hv_d, d_hv, d_packed,
                                                              d_quant_bits, d_norm2, d_n_hashes, ctx->d_status);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

int hg_launch_unpack(hg_ctx *ctx, const uint8_t *d_packed, uint64_t row_stride, const uint8_t *d_quant_bits,
                     uint32_t n, uint32_t hv_d, int16_t *d_hv) {
  if (n == 0) return HG_OK;
  dim3 grid((hv_d / 8 + 255) / 256 < 8 ? (hv_d / 8 + 255) / 256 : 8, n);
  // gridDim.y is limited to 65535
  for (uint32_t g0 = 0; g0 < n; g0 += 65535) {
    const uint32_t cnt = n - g0 < 65535 ? n - g0 : 65535;
    grid.y = cnt;
    unpack_kernel<<<grid, 256, 0, ctx->stream>>>(d_packed + (size_t)g0 * row_stride, row_stride,
                                                 d_quant_bits + g0, cnt, hv_d, d_hv + (size_t)g0 * hv_d);
    ctx->launches++;
  }
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

int hg_launch_sort_tables(hg_ctx *ctx, const hg_genome_desc *d_desc, uint32_t n_genomes, uint64_t *d_tables,
                          uint32_t /*max_slots*/) {
  if (n_genomes == 0) return HG_OK;
  sort_tables_kernel<<<n_genomes, 1024, 0, ctx->stream>>>(d_desc, d_tables);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

int hg_launch_absmax(hg_ctx *ctx, const int16_t *d_hv, uint64_t n_elems, int32_t *d_out) {
  HG_CUDA(cudaMemsetAsync(d_out, 0, sizeof(int32_t), ctx->stream));
  if (n_elems == 0) return HG_OK;
  uint64_t blocks = (n_elems + 256 * 16 - 1) / (256 * 16);
  if (blocks > 148 * 8) blocks = 148 * 8;
  absmax_kernel<<<(unsigned)blocks, 256, 0, ctx->stream>>>(d_hv, n_elems, d_out);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}
