// fasta.cu — FASTA file bytes -> merged sequence, on the GPU.
//
// Replaces fastx_reader::read_merge_seq (reference src/fastx_reader.rs:6-29), the reader of the
// reference's GPU path: every line that starts with '>' contributes one 'N' (so k-mers never span
// records), every other line contributes its bytes minus one trailing '\n' and, before it, one
// trailing '\r'.  A '\r' elsewhere is kept (it then breaks k-mers, exactly as in the reference).
//
// This is a stream compaction with one bit of carried state ("inside a header line").  A run of
// bytes is summarised by (bytes emitted if it starts outside a header, bytes emitted if it starts
// inside one, contains a line start, state handed on); such summaries compose associatively, so one
// scan of one packed word per thread resolves counts and state together.  Three kernels:
//   fasta_scan_kernel    one CTA per 4 KB block of one file: the block's summary (16 bytes per thread
//                        classified with SWAR byte compares, the header state filled bit-parallel);
//   fasta_chain_kernel   one warp per file: chains the block summaries (carry-in state and output
//                        offset of every block, merged length of the file);
//   fasta_emit_kernel    same decomposition: exclusive scan -> each thread's output offset and state,
//                        bytes compacted in shared memory, 16-byte coalesced stores.
// The merged sequence of file f is written at the file's own offset in an output buffer of the
// same size as the input (it can only be shorter), so no cross-file prefix is needed.
#include "hg_common.cuh"

namespace {

constexpr int FA_THREADS = 256;
constexpr int FA_BPT = 16;                       // bytes per thread
constexpr int FA_BLOCK = FA_THREADS * FA_BPT;    // 4096 bytes per CTA

// Per 4 KB block: how many bytes it emits if the carried state at its first byte is "outside a header"
// (c0) or "inside a header line" (c1), whether it contains a line start, and - if so - whether the last
// one opens a header line (the state it hands on).
struct BlockSum {
  uint32_t c0, c1, has_ls, last_hdr;
};

// The same four values for any run of bytes, packed in one word so that a scan moves one register:
// bits 0-13 c0, 14-27 c1 (<= 4096 each), 28 has_ls, 29 last_hdr.  Runs compose left to right.
__device__ __forceinline__ uint32_t seg_make(uint32_t c0, uint32_t c1, uint32_t has, uint32_t hdr) {
  return c0 | (c1 << 14) | (has << 28) | (hdr << 29);
}
__device__ __forceinline__ uint32_t seg_c0(uint32_t x) { return x & 0x3FFFu; }
__device__ __forceinline__ uint32_t seg_c1(uint32_t x) { return (x >> 14) & 0x3FFFu; }
__device__ __forceinline__ uint32_t seg_has(uint32_t x) { return (x >> 28) & 1u; }
__device__ __forceinline__ uint32_t seg_hdr(uint32_t x) { return (x >> 29) & 1u; }
__device__ __forceinline__ uint32_t seg_compose(uint32_t a, uint32_t b) {  // a, then b
  // With a line start in a, b starts in the state a hands on whatever a started in: both counts of a grow by
  // the same count of b.  Without one, b inherits a's incoming state: the counts add field by field.
  const uint32_t cb = b & 0x0FFFFFFFu;
  const uint32_t pick = (a >> 29) & 1u ? (cb >> 14) : (cb & 0x3FFFu);
  const uint32_t add = (a >> 28) & 1u ? pick * 0x4001u : cb;
  const uint32_t flags = (b >> 28) & 1u ? (b & 0x30000000u) : (a & 0x30000000u);
  return ((a & 0x0FFFFFFFu) + add) | flags;
}

// what one thread learns about its 16 bytes (bit i = byte i)
struct Lane {
  uint32_t w[4];       // the bytes
  uint32_t emit_in;    // emitted if NOT inside a header (includes the 'N' of a header start)
  uint32_t hdr_start;  // a '>' at a line start (always emits 'N')
  uint32_t ls;         // starts a line
};

// 4 flags (bit i: byte i of w equals the byte replicated in c4)
__device__ __forceinline__ uint32_t eq4(uint32_t w, uint32_t c4) {
  const uint32_t v = w ^ c4;
  const uint32_t nz = (((v & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | v) & 0x80808080u;  // exact: bit 7 set where the byte differs
  return ((((nz ^ 0x80808080u) >> 7) * 0x00204081u) >> 21) & 0xFu;
}
__device__ __forceinline__ uint32_t eq16(const uint32_t (&w)[4], uint32_t c4) {
  return eq4(w[0], c4) | (eq4(w[1], c4) << 4) | (eq4(w[2], c4) << 8) | (eq4(w[3], c4) << 12);
}
__device__ __forceinline__ bool any_eq16(const uint32_t (&w)[4], uint32_t c4) {  // cheap presence test
  uint32_t z = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const uint32_t v = w[j] ^ c4;
    z |= (v - 0x01010101u) & ~v;
  }
  return (z & 0x80808080u) != 0;
}

// The byte before and the byte after a thread's 16 come from the neighbouring lanes (one extra byte load at
// the warp edges).  Loading is separate from classifying (a CTA may walk several blocks, FA_NB).
struct Raw {
  uint32_t w[4];
  uint32_t edge;  // lane 0: the byte before the warp's bytes; lane 31: the byte after them
};
// Files sit back to back in the buffer, so a file starts at any byte phase: the 16 bytes are cut out of
// two aligned 16-byte loads with funnel shifts (the phase is the same for every thread of a file, so
// the word-shift switch is warp-uniform).  Reads up to 15 bytes before f + p0 (never before the buffer:
// it starts 16-byte aligned) and up to 31 past it (the buffer has that slack).
__device__ __forceinline__ Raw load_raw(const uint8_t *__restrict__ f, uint64_t len, uint64_t p0) {
  Raw r;
  r.w[0] = r.w[1] = r.w[2] = r.w[3] = 0x0A0A0A0Au;  // bytes past the end read as '\n'
  r.edge = (uint32_t)'\n';                          // '\n' before the first byte of the file and after the last
  if (p0 < len) {
    const uintptr_t addr = (uintptr_t)(f + p0);
    const uint32_t mis = (uint32_t)(addr & 15);
    const uint4 *a = reinterpret_cast<const uint4 *>(addr - mis);
    const uint32_t n_valid = len - p0 < FA_BPT ? (uint32_t)(len - p0) : FA_BPT;
    const uint4 v0 = __ldg(a);
    uint4 v1 = make_uint4(0x0A0A0A0Au, 0x0A0A0A0Au, 0x0A0A0A0Au, 0x0A0A0A0Au);
    if (mis + n_valid > 16) v1 = __ldg(a + 1);
    const uint32_t bs = (mis & 3u) * 8u;
    uint32_t y[5];
    switch (mis >> 2) {
      case 0: y[0] = v0.x; y[1] = v0.y; y[2] = v0.z; y[3] = v0.w; y[4] = v1.x; break;
      case 1: y[0] = v0.y; y[1] = v0.z; y[2] = v0.w; y[3] = v1.x; y[4] = v1.y; break;
      case 2: y[0] = v0.z; y[1] = v0.w; y[2] = v1.x; y[3] = v1.y; y[4] = v1.z; break;
      default: y[0] = v0.w; y[1] = v1.x; y[2] = v1.y; y[3] = v1.z; y[4] = v1.w; break;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) r.w[j] = __funnelshift_r(y[j], y[j + 1], bs);
    if (n_valid < FA_BPT) {  // the file's last thread: what follows belongs to the next file
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int keep = (int)n_valid - 4 * j;  // bytes of word j inside the file
        if (keep <= 0) r.w[j] = 0x0A0A0A0Au;
        else if (keep < 4) r.w[j] = (r.w[j] & ((1u << (8 * keep)) - 1u)) | (0x0A0A0A0Au & ~((1u << (8 * keep)) - 1u));
      }
    }
  }
  const int lane = threadIdx.x & 31;
  if (lane == 0 && p0 != 0 && p0 <= len) r.edge = (uint32_t)f[p0 - 1];
  if (lane == 31 && p0 + FA_BPT < len) r.edge = (uint32_t)f[p0 + FA_BPT];
  return r;
}

__device__ __forceinline__ Lane classify(const Raw &r, uint64_t len, uint64_t p0) {
  Lane L;
#pragma unroll
  for (int j = 0; j < 4; ++j) L.w[j] = r.w[j];
  const int lane = threadIdx.x & 31;
  uint32_t prev = __shfl_up_sync(0xffffffffu, L.w[3] >> 24, 1);
  uint32_t next = __shfl_down_sync(0xffffffffu, L.w[0] & 0xFFu, 1);
  if (lane == 0) prev = r.edge;
  if (lane == 31) next = r.edge;
  const uint32_t valid = p0 + FA_BPT <= len ? 0xFFFFu : (p0 < len ? ((1u << (uint32_t)(len - p0)) - 1u) : 0u);
  const uint32_t nl = eq16(L.w, 0x0A0A0A0Au);
  L.ls = ((nl << 1) | (prev == '\n' ? 1u : 0u)) & valid;
  L.hdr_start = (L.ls && any_eq16(L.w, 0x3E3E3E3Eu)) ? (L.ls & eq16(L.w, 0x3E3E3E3Eu)) : 0u;
  uint32_t keep = valid & ~nl;
  if (any_eq16(L.w, 0x0D0D0D0Du)) {  // a '\r' right before a '\n' goes with it (fastx_reader.rs:13-17)
    const uint32_t nl_next = (nl >> 1) | (next == '\n' ? 0x8000u : 0u);
    keep &= ~(eq16(L.w, 0x0D0D0D0Du) & nl_next);
  }
  L.emit_in = keep | L.hdr_start;
  return L;
}

// For the thread's 16 bytes, given whether it starts inside a header: the emit mask and the state
// after its last byte.  A header line runs from its '>' to the next line start; the "inside a header"
// bit of every byte is the hdr_start bit of the last line start at or before it (a segmented fill,
// four doubling steps), or the incoming state before the first line start.
__device__ __forceinline__ uint32_t emit_mask(const Lane &L, bool in_hdr, bool &out_hdr) {
  uint32_t h = L.hdr_start, p = ~L.ls & 0xFFFFu;
  h |= p & (h << 1); p &= p << 1;
  h |= p & (h << 2); p &= p << 2;
  h |= p & (h << 4); p &= p << 4;
  h |= p & (h << 8);
  if (in_hdr) h |= L.ls ? ((L.ls & (0u - L.ls)) - 1u) : 0xFFFFu;  // the bytes before the first line start
  out_hdr = (h >> 15) & 1u;
  return (L.hdr_start | (~h & L.emit_in)) & 0xFFFFu;
}

// the thread's bytes as a run: counts under both incoming states, line start seen, state handed on
__device__ __forceinline__ uint32_t lane_seg(const Lane &L, uint32_t &m0) {
  bool oh;
  m0 = emit_mask(L, false, oh);
  const uint32_t pre = L.ls ? ((L.ls & (0u - L.ls)) - 1u) : 0xFFFFu;
  return seg_make(__popc(m0), __popc(m0 & ~pre), L.ls != 0, oh ? 1u : 0u);
}

// inclusive scan of the runs over the CTA; returns this thread's EXCLUSIVE prefix, `total` = the whole block
__device__ __forceinline__ uint32_t block_seg_scan(uint32_t mine, uint32_t &total) {
  __shared__ uint32_t s_w[FA_THREADS / 32 + 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t x = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t pv = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x = seg_compose(pv, x);
  }
  if (lane == 31) s_w[warp + 1] = x;
  __syncthreads();
  if (warp == 0) {  // exclusive scan of the 8 warp totals: s_w[w] = everything before warp w, s_w[8] = the block
    uint32_t y = (lane >= 1 && lane <= FA_THREADS / 32) ? s_w[lane] : 0u;
#pragma unroll
    for (int o = 1; o < FA_THREADS / 32; o <<= 1) {
      const uint32_t pv = __shfl_up_sync(0xffffffffu, y, o);
      if (lane >= o) y = seg_compose(pv, y);
    }
    if (lane <= FA_THREADS / 32) s_w[lane] = y;
  }
  __syncthreads();
  uint32_t ex = __shfl_up_sync(0xffffffffu, x, 1);
  if (lane == 0) ex = 0;  // the identity run
  total = s_w[FA_THREADS / 32];
  const uint32_t out = seg_compose(s_w[warp], ex);
  __syncthreads();  // s_w may be rewritten by the next call
  return out;
}

// A CTA walks FA_NB consecutive 4 KB blocks of one file with the next block's loads in flight.
constexpr int FA_NB = 1;  // measured: more blocks per CTA do not help, the kernels are instruction-bound, not latency-bound

__global__ void __launch_bounds__(FA_THREADS)
fasta_scan_kernel(const uint8_t *__restrict__ raw, const uint64_t *__restrict__ file_off, const uint64_t *__restrict__ blk_off,
                  BlockSum *__restrict__ sums) {
  const uint32_t f = blockIdx.y;
  const uint64_t len = file_off[f + 1] - file_off[f];
  const uint64_t nb = (len + FA_BLOCK - 1) / FA_BLOCK;
  uint64_t blk = (uint64_t)blockIdx.x * FA_NB;
  if (blk >= nb) return;
  const uint64_t blk_end = blk + FA_NB < nb ? blk + FA_NB : nb;
  const uint8_t *fp = raw + file_off[f];
  Raw cur = load_raw(fp, len, blk * FA_BLOCK + (uint64_t)threadIdx.x * FA_BPT);
  for (; blk < blk_end; ++blk) {
    const uint64_t p0 = blk * FA_BLOCK + (uint64_t)threadIdx.x * FA_BPT;
    Raw nxt = cur;
    if (blk + 1 < blk_end) nxt = load_raw(fp, len, p0 + FA_BLOCK);
    const Lane L = classify(cur, len, p0);
    uint32_t m0, total;
    (void)block_seg_scan(lane_seg(L, m0), total);
    if (threadIdx.x == 0) {
      BlockSum s;
      s.c0 = seg_c0(total);
      s.c1 = seg_c1(total);
      s.has_ls = seg_has(total);
      s.last_hdr = seg_hdr(total);
      sums[blk_off[f] + blk] = s;
    }
    cur = nxt;
  }
}

// one warp per file: the block summaries compose like the runs inside a block, so 32 of them are chained
// with a five-step warp scan (carry-in state and output offset of every block, merged length of the file)
__global__ void fasta_chain_kernel(const uint64_t *__restrict__ file_off, const uint64_t *__restrict__ blk_off,
                                   uint32_t n_files, const BlockSum *__restrict__ sums, uint8_t *__restrict__ carry,
                                   uint64_t *__restrict__ out_off, uint64_t *__restrict__ merged_len) {
  const uint32_t f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (f >= n_files) return;
  const uint64_t nb = blk_off[f + 1] - blk_off[f];
  uint32_t state = 0;  // a file starts at a line start, so the initial state is never inherited
  uint64_t off = 0;
  for (uint64_t base = 0; base < nb; base += 32) {
    const uint64_t b = base + lane;
    BlockSum s = {0, 0, 0, 0};  // the identity run
    if (b < nb) s = sums[blk_off[f] + b];
    // inclusive scan over the 32 summaries: (c0, c1, has, hdr) of blocks base .. base + lane
    uint32_t c0 = s.c0, c1 = s.c1, has = s.has_ls, hdr = s.last_hdr;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t p0 = __shfl_up_sync(0xffffffffu, c0, o), p1 = __shfl_up_sync(0xffffffffu, c1, o);
      const uint32_t ph = __shfl_up_sync(0xffffffffu, has, o), pd = __shfl_up_sync(0xffffffffu, hdr, o);
      if (lane >= (uint32_t)o) {  // (p) then (mine)
        const uint32_t after0 = ph ? pd : 0u, after1 = ph ? pd : 1u;
        const uint32_t n0 = p0 + (after0 ? c1 : c0), n1 = p1 + (after1 ? c1 : c0);
        c0 = n0; c1 = n1;
        hdr = has ? hdr : pd;
        has |= ph;
      }
    }
    // exclusive values of my block = inclusive values of the previous lane, applied to the carried (state, off)
    uint32_t e0 = __shfl_up_sync(0xffffffffu, c0, 1), e1 = __shfl_up_sync(0xffffffffu, c1, 1);
    uint32_t eh = __shfl_up_sync(0xffffffffu, has, 1), ed = __shfl_up_sync(0xffffffffu, hdr, 1);
    if (lane == 0) { e0 = 0; e1 = 0; eh = 0; ed = 0; }
    if (b < nb) {
      carry[blk_off[f] + b] = (uint8_t)(eh ? ed : state);
      out_off[blk_off[f] + b] = off + (state ? e1 : e0);
    }
    const uint32_t t0 = __shfl_sync(0xffffffffu, c0, 31), t1 = __shfl_sync(0xffffffffu, c1, 31);
    const uint32_t th = __shfl_sync(0xffffffffu, has, 31), td = __shfl_sync(0xffffffffu, hdr, 31);
    off += state ? t1 : t0;
    if (th) state = td;
  }
  if (lane == 0) merged_len[f] = off;
}

// Same decomposition as the scan.  The block's output bytes are compacted in shared memory, at the
// 16-byte phase of their destination, and leave with 16-byte stores (byte stores only at the two
// ragged ends, which neighbouring blocks own the rest of).
__global__ void __launch_bounds__(FA_THREADS)
fasta_emit_kernel(const uint8_t *__restrict__ raw, const uint64_t *__restrict__ file_off, const uint64_t *__restrict__ blk_off,
                  const uint8_t *__restrict__ carry, const uint64_t *__restrict__ out_off, uint8_t *__restrict__ merged) {
  __shared__ __align__(16) uint8_t s_out[FA_BLOCK + 32];
  const uint32_t f = blockIdx.y;
  const uint64_t len = file_off[f + 1] - file_off[f];
  const uint64_t nb = (len + FA_BLOCK - 1) / FA_BLOCK;
  uint64_t blk = (uint64_t)blockIdx.x * FA_NB;
  if (blk >= nb) return;
  const uint64_t blk_end = blk + FA_NB < nb ? blk + FA_NB : nb;
  const uint8_t *fp = raw + file_off[f];
  Raw cur = load_raw(fp, len, blk * FA_BLOCK + (uint64_t)threadIdx.x * FA_BPT);
  uint32_t cur_carry = carry[blk_off[f] + blk];
  uint64_t cur_off = out_off[blk_off[f] + blk];
  for (; blk < blk_end; ++blk) {
    const uint64_t p0 = blk * FA_BLOCK + (uint64_t)threadIdx.x * FA_BPT;
    Raw nxt = cur;
    uint32_t nxt_carry = 0;
    uint64_t nxt_off = 0;
    if (blk + 1 < blk_end) {
      nxt = load_raw(fp, len, p0 + FA_BLOCK);
      nxt_carry = carry[blk_off[f] + blk + 1];
      nxt_off = out_off[blk_off[f] + blk + 1];
    }
    const Lane L = classify(cur, len, p0);
    const bool carry_in = cur_carry != 0;
    uint32_t m0, total;
    const uint32_t ex = block_seg_scan(lane_seg(L, m0), total);
    bool oh;
    const uint32_t m = emit_mask(L, seg_has(ex) ? (seg_hdr(ex) != 0) : carry_in, oh);
    uint8_t *dst = merged + file_off[f] + cur_off;
    const uint32_t al = (uint32_t)((uintptr_t)dst & 15);  // staged at the destination's phase
    uint32_t k = al + (carry_in ? seg_c1(ex) : seg_c0(ex));
    if (m == 0xFFFFu && L.hdr_start == 0 && (k & 3u) == 0) {  // every byte kept, word-aligned target
#pragma unroll
      for (int j = 0; j < 4; ++j) *reinterpret_cast<uint32_t *>(s_out + k + 4 * j) = L.w[j];
    } else {
#pragma unroll
      for (int i = 0; i < FA_BPT; ++i)
        if ((m >> i) & 1u) s_out[k++] = ((L.hdr_start >> i) & 1u) ? (uint8_t)'N' : (uint8_t)(L.w[i >> 2] >> (8 * (i & 3)));
    }
    __syncthreads();
    const uint32_t n_out = carry_in ? seg_c1(total) : seg_c0(total);
    const uint32_t end = al + n_out;  // staged bytes are s_out[al, end)
    uint8_t *dst0 = dst - al;         // 16-byte aligned
    for (uint32_t c = threadIdx.x; 16 * c < end; c += FA_THREADS) {
      const uint32_t lo = 16 * c, hi = lo + 16;
      if (lo >= al && hi <= end) {
        *reinterpret_cast<uint4 *>(dst0 + lo) = *reinterpret_cast<const uint4 *>(s_out + lo);
      } else {
        for (uint32_t q = (lo > al ? lo : al); q < (hi < end ? hi : end); ++q) dst0[q] = s_out[q];
      }
    }
    __syncthreads();  // s_out is refilled by the next block
    cur = nxt;
    cur_carry = nxt_carry;
    cur_off = nxt_off;
  }
}

// ---- record index (hg_sketch_fasta_records): runs after the merge, on the same raw bytes ----
// Every header start emitted exactly one 'N', so a record is located by its header's raw index and the merged offset
// of that 'N'.  Table layout of a merge: file f owns slots [first[blk_off[f]] + f, first[blk_off[f + 1]] + f + 1): one
// leading slot, then its headers in file order; the host drops a leading slot whose sequence is empty.

// sum over the CTA (every thread passes its value; the result is valid in thread 0)
__device__ __forceinline__ uint32_t block_sum(uint32_t v) {
  __shared__ uint32_t s_c[FA_THREADS / 32];
  v = __reduce_add_sync(0xffffffffu, v);
  if ((threadIdx.x & 31) == 0) s_c[threadIdx.x >> 5] = v;
  __syncthreads();
  uint32_t t = 0;
  if (threadIdx.x == 0)
#pragma unroll
    for (int w = 0; w < FA_THREADS / 32; ++w) t += s_c[w];
  return t;
}

// header starts per 4 KB block (the header test needs no carried state: a '>' at a line start always opens one)
__global__ void __launch_bounds__(FA_THREADS)
fasta_rec_count_kernel(const uint8_t *__restrict__ raw, const uint64_t *__restrict__ file_off, const uint64_t *__restrict__ blk_off,
                       uint32_t *__restrict__ cnt) {
  const uint32_t f = blockIdx.y;
  const uint64_t len = file_off[f + 1] - file_off[f];
  const uint64_t nb = (len + FA_BLOCK - 1) / FA_BLOCK, blk = blockIdx.x;
  if (blk >= nb) return;
  const uint64_t p0 = blk * FA_BLOCK + (uint64_t)threadIdx.x * FA_BPT;
  const Lane L = classify(load_raw(raw + file_off[f], len, p0), len, p0);
  const uint32_t t = block_sum(__popc(L.hdr_start));
  if (threadIdx.x == 0) cnt[blk_off[f] + blk] = t;
}

// one CTA: first[b] = header starts in blocks before b (all files of the merge), first[nblk] = all of them
__global__ void __launch_bounds__(1024) fasta_rec_prefix_kernel(const uint32_t *__restrict__ cnt, uint64_t nblk,
                                                                uint64_t *__restrict__ first) {
  __shared__ uint64_t s_w[32];
  __shared__ uint64_t s_carry;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (uint64_t base = 0; base < nblk; base += 1024) {
    const uint64_t i = base + threadIdx.x;
    const uint64_t v = i < nblk ? cnt[i] : 0;
    uint64_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint64_t y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) s_w[warp] = x;
    __syncthreads();
    if (warp == 0) {
      uint64_t y = s_w[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint64_t z = __shfl_up_sync(0xffffffffu, y, o);
        if (lane >= o) y += z;
      }
      s_w[lane] = y;
    }
    __syncthreads();
    const uint64_t incl = s_carry + (warp ? s_w[warp - 1] : 0) + x;
    if (i < nblk) first[i] = incl - v;
    __syncthreads();  // s_carry and s_w are read by every thread before they change
    if (threadIdx.x == 1023) s_carry = incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) first[nblk] = s_carry;
}

// the leading slot of every file: its sequence starts at merged offset 0 (rec_n = -1 stands for a virtual 'N' before it)
__global__ void fasta_rec_lead_kernel(const uint64_t *__restrict__ file_off, const uint64_t *__restrict__ blk_off, uint32_t n_files,
                                      const uint64_t *__restrict__ first, hg_fasta_record *__restrict__ rec,
                                      uint64_t *__restrict__ rec_n) {
  const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n_files) return;
  const uint64_t s = first[blk_off[f]] + f;
  hg_fasta_record r;
  r.name_off = file_off[f];
  r.name_len = 0;
  r.seq_len = 0;
  r.file = f;
  r.has_header = 0;
  rec[s] = r;
  rec_n[s] = ~0ull;
}

// Per block with a header start: the merged offset of every header's 'N' (the emit kernel's offsets) and its slot.
// Files f0 .. f0 + gridDim.y - 1 (file_off / blk_off index all files of the merge).
__global__ void __launch_bounds__(FA_THREADS)
fasta_rec_emit_kernel(const uint8_t *__restrict__ raw, const uint64_t *__restrict__ file_off, const uint64_t *__restrict__ blk_off,
                      uint32_t f0, const uint8_t *__restrict__ carry, const uint64_t *__restrict__ out_off,
                      const uint32_t *__restrict__ cnt, const uint64_t *__restrict__ first, hg_fasta_record *__restrict__ rec,
                      uint64_t *__restrict__ rec_n) {
  __shared__ uint32_t s_h[FA_THREADS / 32];
  const uint32_t f = f0 + blockIdx.y;
  const uint64_t len = file_off[f + 1] - file_off[f];
  const uint64_t nb = (len + FA_BLOCK - 1) / FA_BLOCK, blk = blockIdx.x;
  if (blk >= nb) return;
  const uint64_t gb = blk_off[f] + blk;
  if (cnt[gb] == 0) return;  // most blocks of a genome hold no header
  const uint64_t p0 = blk * FA_BLOCK + (uint64_t)threadIdx.x * FA_BPT;
  const Lane L = classify(load_raw(raw + file_off[f], len, p0), len, p0);
  const bool carry_in = carry[gb] != 0;
  uint32_t m0, total;
  const uint32_t ex = block_seg_scan(lane_seg(L, m0), total);
  bool oh;
  const uint32_t m = emit_mask(L, seg_has(ex) ? (seg_hdr(ex) != 0) : carry_in, oh);
  const uint64_t pos = out_off[gb] + (carry_in ? seg_c1(ex) : seg_c0(ex));
  // the thread's headers are preceded by those of lower threads: exclusive scan of the per-thread counts
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t h = __popc(L.hdr_start);
  uint32_t x = h;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) s_h[warp] = x;
  __syncthreads();
  uint32_t before = x - h;
  for (int w = 0; w < warp; ++w) before += s_h[w];
  uint64_t s = first[gb] + f + 1 + before;
  for (uint32_t bits = L.hdr_start; bits; bits &= bits - 1, ++s) {
    const int i = __ffs(bits) - 1;
    hg_fasta_record r;
    r.name_off = file_off[f] + p0 + i + 1;
    r.name_len = 0;
    r.seq_len = 0;
    r.file = f;
    r.has_header = 1;
    rec[s] = r;
    rec_n[s] = pos + __popc(m & ((1u << i) - 1u));
  }
}

// One thread per slot: seq_len from the next slot's 'N' (or the file's merged length), and the header's name span by a
// forward search for the end of its line (headers are short; a long one costs its own thread only).
__global__ void fasta_rec_finish_kernel(const uint8_t *__restrict__ raw, const uint64_t *__restrict__ file_off,
                                        const uint64_t *__restrict__ merged_len, uint64_t n_slots, hg_fasta_record *__restrict__ rec,
                                        const uint64_t *__restrict__ rec_n) {
  const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_slots) return;
  const uint32_t f = rec[s].file;
  const uint64_t next = s + 1 < n_slots && rec[s + 1].file == f ? rec_n[s + 1] : merged_len[f];
  rec[s].seq_len = next - rec_n[s] - 1;
  if (rec[s].has_header) {
    const uint64_t a = rec[s].name_off, end = file_off[f + 1];
    uint64_t q = a;
    while (q < end && raw[q] != '\n') ++q;
    rec[s].name_len = q - a - (q < end && q > a && raw[q - 1] == '\r' ? 1 : 0);
  }
}

}  // namespace

uint32_t hg_fasta_block_bytes() { return FA_BLOCK; }

// d_file_off / d_blk_off: device copies of the per-file byte offsets and block prefix (n_files + 1 each)
int hg_launch_fasta_merge(hg_ctx *ctx, const uint8_t *d_raw, const uint64_t *d_file_off, const uint64_t *d_blk_off,
                          uint32_t n_files, uint32_t max_blocks, void *d_sums, uint8_t *d_carry, uint64_t *d_out_off,
                          uint8_t *d_merged, uint64_t *d_merged_len) {
  if (n_files == 0) return HG_OK;
  for (uint32_t f0 = 0; f0 < n_files; f0 += 65535) {
    const uint32_t nf = n_files - f0 < 65535 ? n_files - f0 : 65535;
    if (max_blocks)
      fasta_scan_kernel<<<dim3((max_blocks + FA_NB - 1) / FA_NB, nf), FA_THREADS, 0, ctx->stream>>>(d_raw, d_file_off + f0, d_blk_off + f0,
                                                                             (BlockSum *)d_sums);
    ctx->launches++;
  }
  fasta_chain_kernel<<<(n_files * 32 + 127) / 128, 128, 0, ctx->stream>>>(d_file_off, d_blk_off, n_files,
                                                                          (const BlockSum *)d_sums, d_carry, d_out_off,
                                                                          d_merged_len);
  ctx->launches++;
  for (uint32_t f0 = 0; f0 < n_files; f0 += 65535) {
    const uint32_t nf = n_files - f0 < 65535 ? n_files - f0 : 65535;
    if (max_blocks)
      fasta_emit_kernel<<<dim3((max_blocks + FA_NB - 1) / FA_NB, nf), FA_THREADS, 0, ctx->stream>>>(d_raw, d_file_off + f0, d_blk_off + f0,
                                                                             d_carry, d_out_off, d_merged);
    ctx->launches++;
  }
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

// Record index, pass 1 (after hg_launch_fasta_merge, same arguments): d_cnt (n_blocks) and d_first (n_blocks + 1, the
// last entry the header count of the merge).  The host reads d_first[n_blocks] back: the table has that + n_files slots.
int hg_launch_fasta_rec_count(hg_ctx *ctx, const uint8_t *d_raw, const uint64_t *d_file_off, const uint64_t *d_blk_off,
                              uint32_t n_files, uint32_t max_blocks, uint64_t n_blocks, uint32_t *d_cnt, uint64_t *d_first) {
  for (uint32_t f0 = 0; f0 < n_files && max_blocks; f0 += 65535) {
    const uint32_t nf = n_files - f0 < 65535 ? n_files - f0 : 65535;
    fasta_rec_count_kernel<<<dim3(max_blocks, nf), FA_THREADS, 0, ctx->stream>>>(d_raw, d_file_off + f0, d_blk_off + f0, d_cnt);
    ctx->launches++;
  }
  fasta_rec_prefix_kernel<<<1, 1024, 0, ctx->stream>>>(d_cnt, n_blocks, d_first);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

// Pass 2: the n_slots-entry table (rec; rec_n the 'N' offsets) from pass 1 and the merge's carry / out_off / lengths.
// name_off is an index into d_raw; file is the index in this merge.
int hg_launch_fasta_rec_table(hg_ctx *ctx, const uint8_t *d_raw, const uint64_t *d_file_off, const uint64_t *d_blk_off,
                              uint32_t n_files, uint32_t max_blocks, const uint8_t *d_carry, const uint64_t *d_out_off,
                              const uint64_t *d_merged_len, const uint32_t *d_cnt, const uint64_t *d_first, uint64_t n_slots,
                              hg_fasta_record *d_rec, uint64_t *d_rec_n) {
  if (n_files == 0) return HG_OK;
  fasta_rec_lead_kernel<<<(n_files + 255) / 256, 256, 0, ctx->stream>>>(d_file_off, d_blk_off, n_files, d_first, d_rec, d_rec_n);
  ctx->launches++;
  for (uint32_t f0 = 0; f0 < n_files && max_blocks; f0 += 65535) {
    const uint32_t nf = n_files - f0 < 65535 ? n_files - f0 : 65535;
    fasta_rec_emit_kernel<<<dim3(max_blocks, nf), FA_THREADS, 0, ctx->stream>>>(d_raw, d_file_off, d_blk_off, f0, d_carry, d_out_off,
                                                                               d_cnt, d_first, d_rec, d_rec_n);
    ctx->launches++;
  }
  fasta_rec_finish_kernel<<<(unsigned)((n_slots + 255) / 256), 256, 0, ctx->stream>>>(d_raw, d_file_off, d_merged_len, n_slots,
                                                                                      d_rec, d_rec_n);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}
