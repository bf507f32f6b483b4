// kmer_hash.cu — stage 1a: canonical k-mer extraction, t1ha2 hashing, FracMinHash filter and
// set insertion for a batch of genomes, in one pass over the sequence bytes.
//
// Replaces cuda_kmer_t1ha2 (reference src/cuda_kernel.cu:250-321) and its host-side result
// scan (src/sketch_cuda.rs:156-163).  WHICH reference semantics: those of the reference's GPU path
// - read_merge_seq bytes (src/fastx_reader.rs:6-29), only ACGT / acgt are bases, every other byte
// breaks the k-mer run (cuda_kernel.cu:272-296) - with two deliberate deviations: no sample is
// dropped when a 512-k-mer stretch yields more than 8 (cuda_kernel.cu:316) and h == 0 is kept
// (sketch_cuda.rs:159).  On ACGT/N input that is also the CPU path's HashSet (src/sketch.rs:71-98);
// it is NOT needletail's normalize(), which maps U/u to T and iterates per record (recalled, not
// vendored) - tests/test_gpu_sketch.py documents the difference on IUPAC / U bytes.
// Survivors are compacted through a per-warp shared-memory queue and inserted with atomicCAS into a
// per-genome hash table (set semantics), not by the warp-ballot / prefix-sum list the north star
// sketches: a list would still need a dedup pass, the table is the dedup.
// Design (not the reference's one-thread-per-512-k-mers walk):
//   * one CTA per tile of 8192 k-mer start positions of ONE genome; the tile's bytes
//     (+ k-1 halo) are read once with aligned, coalesced 16-byte loads, converted SWAR-style
//     to nibble codes + a validity bit per base, and staged in 5 KB of shared memory;
//   * each thread then owns 32 consecutive start positions: the forward and reverse-
//     complement k-mers roll in registers one NIBBLE per base (first base in the low nibble),
//     canonical = lexicographic min via ONE multi-word unsigned compare of the two states (same
//     choice as the reference's byte compare, cuda_kernel.cu:84-89,306-311), and the chosen k-mer becomes
//     its upper-case ASCII bytes with two PRMT table lookups per 8 bases (the hash is defined
//     over the ASCII k-mer, sketch.rs:90); t1ha2_atonce in registers, its first round (K >= 8) from
//     two product tables in shared memory indexed by the first 8 bases; threshold compare;
//   * the rare survivors (1/scaled) are inserted into the genome's open-addressing table in
//     HBM with atomicCAS, which both removes duplicates (the reference keeps a set) and has
//     no per-thread capacity cliff (the reference drops hits beyond 8 per thread,
//     cuda_kernel.cu:316-317).
#include "hg_common.cuh"

namespace {

#ifndef HG_KH_THREADS
#define HG_KH_THREADS 128
#endif
constexpr int KH_THREADS = HG_KH_THREADS;
constexpr int KH_WARPS = KH_THREADS / 32;
constexpr int KH_PPT = 32;                       // k-mer start positions per thread
constexpr int KH_TILE = 32 * KH_PPT;             // start positions per WARP tile
constexpr int KH_CHUNKS = (KH_TILE + 64) / 16;   // 16-base chunks staged per tile (halo + align)
constexpr int KH_QCAP = 64;                      // per-warp queue of survivors, flushed once per tile
#ifndef HG_KH_GROUP
#define HG_KH_GROUP 4
#endif
#ifndef HG_KH_UNROLL
#define HG_KH_UNROLL 1
#endif
constexpr int KH_UNROLL = HG_KH_UNROLL;          // groups of 8 positions unrolled in the per-lane loop
constexpr int KH_GROUP = HG_KH_GROUP;            // positions hashed back to back before survivors are looked at (measured: 4 beats 8 by 1.2 %, fewer hashes kept live)
#ifndef HG_KH_MIN_CTAS
#define HG_KH_MIN_CTAS 8
#endif
constexpr int KH_MIN_CTAS = HG_KH_MIN_CTAS;                   // 32 resident warps per SM at <= 64 registers (measured: occupancy beyond this does not help)

__device__ __forceinline__ uint4 ld_stream16(const void *p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

// raw PRMT: selector nibbles are always < 8 here, so the masking __byte_perm adds is not needed
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}

// Nibble code of a base (one nibble per base everywhere below):  A=1  C=2  G=3  T=4, 0 = "no
// base".  Chosen so that (i) the codes order as the letters do, (ii) complement is 5 - code (no
// borrow between nibbles), and (iii) every code is a PRMT selector (< 8) into an 8-byte ASCII
// table with 0 -> 0x00, so the unused nibbles of the last word expand to the zero bytes t1ha2's
// tail read wants.
//
// (i) + (ii) make the canonical choice a plain multi-word unsigned compare of the two rolling
// states, although those hold the FIRST base in the LOW nibble: comparing a k-mer with its own
// reverse complement from the front tests base[i] against comp(base[K-1-i]); comparing the packed
// values from the top tests base[K-1-i] against comp(base[i]); and a < 5 - b <=> b < 5 - a.  Both
// walks meet the same sequence of decisions, so F < R numerically <=> forward < revcomp
// lexicographically (the reference's strcmp_l, cuda_kernel.cu:84-89,306-311).  No bit reversal.
//
// 4 ASCII bytes -> 16 bits of nibble codes (base 0 in the low nibble) + 4 validity bits
// (only A,C,G,T in either case are bases — cuda_kernel.cu:277-296).
__device__ __forceinline__ void encode4(uint32_t w, uint32_t &nib16, uint32_t &valid4) {
  const uint32_t u = w & 0xDFDFDFDFu;                               // fold case
  const uint32_t code = ((u >> 1) ^ (u >> 2)) & 0x03030303u;        // per byte: A0 C1 G2 T3
  const uint32_t sel = (code | (code >> 12)) & 0xFFFFu;             // nibbles: b0 b2 b1 b3
  const uint32_t nib = prmt(0x04030201u, 0u, sel);           // bytes n0 n2 n1 n3
  nib16 = (nib | (nib >> 12)) & 0xFFFFu;                            // n0 n1 n2 n3
  // re-expand the codes to upper-case ASCII and compare: anything else is not a base
  const uint32_t expect = prmt(0x54474341u, 0u, sel);        // 'A','C','G','T'
  const uint32_t have = prmt(u, 0u, 0x3120u);                // same byte order
  const uint32_t d = expect ^ have;
  const uint32_t nz = (((d & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | d) & 0x80808080u;
  const uint32_t ok = (nz ^ 0x80808080u) >> 7;                      // flags at bits 0,8,16,24
  valid4 = ((ok * 0x01040208u) >> 24) & 0xFu;                       // back to base order
}

// 8 ASCII bytes (w0 = bases 0..3, w1 = bases 4..7) -> 8 nibble codes, base i in nibble i; `bad` collects a non-zero
// byte for every byte that is not a base.  The bytes are first gathered into even / odd bases (two PRMTs on the raw
// words), so that the per-byte 2-bit codes of the two halves interleave into nibbles with one shift-or; the same
// nibbles then select the byte each code stands for (one PRMT per four bases) and the comparison with what was read
// is the validity test.  17 instructions per 8 bases; a byte that is not a base gets SOME code 1..4 - its validity
// bit, not its code, keeps it out of every k-mer.
__device__ __forceinline__ uint32_t encode8(uint32_t w0, uint32_t w1, uint32_t &bad, uint32_t k_fold, uint32_t k_lut) {
  // k_fold = 0xDFDFDFDF, k_lut = 0x15060200 (held in registers by the caller)
  const uint32_t y0 = (w0 & k_fold) ^ 0x41414141u, y1 = (w1 & k_fold) ^ 0x41414141u;  // A 00, C 02, G 06, T 15, either case
  const uint32_t e = prmt(y0, y1, 0x6420u), o = prmt(y0, y1, 0x7531u);
  const uint32_t ce = ((e >> 1) ^ (e >> 2)) & 0x03030303u, co = ((o >> 1) ^ (o >> 2)) & 0x03030303u;  // A0 C1 G2 T3
  const uint32_t sel = ce | (co << 4);
  const uint32_t x0 = prmt(k_lut, 0u, sel), x1 = prmt(k_lut, 0u, sel >> 16);
  bad |= (x0 ^ y0) | (x1 ^ y1);
  return sel + 0x11111111u;
}

__device__ __forceinline__ uint32_t funnel_r(uint32_t lo, uint32_t hi, uint32_t s) {
  return __funnelshift_r(lo, hi, s);
}

// reverse the bit order inside every nibble (undoes what BREV does to the codes)
__device__ __forceinline__ uint32_t rev_in_nibble(uint32_t x) {
  return ((x & 0x11111111u) << 3) | ((x & 0x22222222u) << 1) | ((x >> 1) & 0x22222222u) | ((x >> 3) & 0x11111111u);
}

// Insert h into the genome's table (linear probing).  Duplicates collapse: F3 set semantics.
__device__ __noinline__ void table_insert(uint64_t *__restrict__ table, uint32_t mask, uint64_t h,
                                          uint32_t *count, uint32_t *status) {
  uint32_t slot = (uint32_t)h & mask;
  for (uint32_t probe = 0; probe <= mask; ++probe) {
    const unsigned long long prev =
        atomicCAS((unsigned long long *)(table + slot), (unsigned long long)HG_EMPTY_SLOT,
                  (unsigned long long)h);
    if (prev == HG_EMPTY_SLOT) {
      atomicAdd(count, 1u);
      return;
    }
    if (prev == h) return;
    slot = (slot + 1) & mask;
  }
  atomicOr(status, 1u);  // table full: reported by hg_sketch_status, never silently dropped
}

// ---- t1ha2's first round from product tables (K >= 8) ----
// Word 0 of a k-mer with K >= 8 is the ASCII of its first 8 bases: 4^8 values.  Round 1 is
// mixup64(X, Y, w0, P) (roles and prime: hg::t1ha2_round1), i.e. t = Y + w0 mod 2^64, X ^= lo64(t P),
// Y += hi64(t P).  With w0 = w_lo + 2^32 w_hi (w_lo = bases 0-3, w_hi = bases 4-7) and c = [Y + w0 >= 2^64]:
//   t P = (Y + w_lo) P + w_hi P 2^32 - c P 2^64   (mod 2^128)
// so the round is two lookups and a 128-bit add:
//   L[i] = (Y + w_lo(i)) P mod 2^128, with X_lo xored into word 0 and Y added to the high 64 bits;
//   H[j] = w_hi(j) P (96 bits: words 1-3 of the sum; word 0 of the sum is word 0 of L).
// i, j are the base-4 numbers of bases 0-3 and 4-7 (base 0 least significant, A < C < G < T).  w0 grows
// with j * 256 + i, so c is a threshold test on that index; it can only be 1 when Y is the seed and the
// seed is above 2^64 - w0(TTTTTTTT), which the host decides per launch (the WRAP instantiations).
constexpr int KH_TAB_ENTRIES = 512;                        // L[256] | H[256], 16 bytes each
constexpr size_t KH_TAB_BYTES = KH_TAB_ENTRIES * sizeof(uint4);
constexpr int KH_TAB_COPIES = 2;  // in shared memory (measured: 20.85 ms per 1000 genomes vs 20.94 with one copy)

// ASCII of the 4 bases of a base-4 number e (base 0 in the low 2 bits and the low byte)
__host__ __device__ inline uint32_t ascii4(uint32_t e) {
  uint32_t w = 0;
  for (int k = 0; k < 4; ++k) w |= ((0x54474341u >> (8 * ((e >> (2 * k)) & 3u))) & 0xFFu) << (8 * k);
  return w;
}

template <int K, bool CANON, bool WRAP>
__global__ void __launch_bounds__(KH_THREADS, KH_MIN_CTAS)
kmer_hash_kernel(const uint8_t *__restrict__ seq, const hg_genome_desc *__restrict__ desc,
                 uint32_t n_genomes, uint32_t n_tiles, uint64_t threshold, uint64_t seed,
                 uint64_t *__restrict__ tables, uint32_t *__restrict__ counts,
                 uint32_t *__restrict__ status, uint32_t lut_lo, uint32_t lut_hi,
                 const uint32_t *__restrict__ cta_genome, const uint64_t *__restrict__ actual_len, uint2 consts,
                 const uint4 *__restrict__ round1_tab, uint32_t wrap_at) {
  constexpr int NW = (K + 7) / 8;          // nibble words == t1ha2 input words (8 bases each)
  constexpr int LASTN = K - 8 * (NW - 1);  // bases in the last word, 1..8
  constexpr uint32_t LASTMASK = LASTN == 8 ? 0xFFFFFFFFu : ((1u << (4 * LASTN)) - 1u);
  constexpr bool TAB = K >= 8;             // round 1 from the product tables
  using R1 = hg::t1ha2_round1<K>;
  // The round-1 tables, copied into shared memory once per CTA: the kernel's only CTA-wide barrier, ahead of every
  // return.  Two copies, entry e of copy r at 2 e + r, and the lane's parity picks the copy: the 8 lanes of an LDS.128
  // phase then hit each half of the bank groups with 4 random indices instead of all of them with 8 (fewer conflicts).
  __shared__ uint4 s_tab[TAB ? KH_TAB_COPIES * KH_TAB_ENTRIES : 1];
  if (TAB) {
#pragma unroll
    for (int e = threadIdx.x; e < KH_TAB_ENTRIES; e += KH_THREADS) {
      const uint4 v = round1_tab[e];
      s_tab[2 * e] = v;
      s_tab[2 * e + 1] = v;
    }
    __syncthreads();
  }
  // apart from that every warp owns a private staging area and runs on its own
  __shared__ __align__(8) uint32_t s_nib_all[KH_WARPS][KH_CHUNKS * 2 + 8];    // 8 bases per word
  __shared__ uint32_t s_valid_all[KH_WARPS][KH_CHUNKS / 2 + 4];  // 16 bits per chunk
  // survivors are queued here and inserted together at the end of the tile, so the round trip
  // of the global atomicCAS is paid once per tile (all lanes in flight) instead of once per hit
  __shared__ uint64_t s_queue_all[KH_WARPS][KH_QCAP];
  __shared__ uint32_t s_qn_all[KH_WARPS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t *s_nib = s_nib_all[warp];
  uint32_t *s_valid = s_valid_all[warp];
  uint16_t *s_valid16 = reinterpret_cast<uint16_t *>(s_valid);
  uint64_t *s_queue = s_queue_all[warp];
  uint32_t *s_qn = &s_qn_all[warp];
  if (lane == 0) *s_qn = 0;

  // One tile per warp, 8 consecutive tiles per CTA.  cta_genome[] (written by tile_map_kernel)
  // names the genome of the CTA's first tile; the warp walks the sorted first_tile column
  // forward from there (desc[n_genomes] is a sentinel holding the tile count).
  const uint32_t tile = blockIdx.x * KH_WARPS + warp;
  if (tile >= n_tiles) return;
  uint32_t g = cta_genome[blockIdx.x];
  while (desc[g + 1].first_tile <= tile) ++g;  // warp-uniform, usually zero steps
  {
  hg_genome_desc gd = desc[g];
  // raw-FASTA path: the tiles were planned from an upper bound, the merge kernel wrote the real length
  if (actual_len) gd.seq_len = min(gd.seq_len, actual_len[g]);
  if ((uint64_t)(tile - gd.first_tile) * KH_TILE + K > gd.seq_len) return;  // no complete k-mer starts in this tile
  const uint64_t tile_base = (uint64_t)(tile - gd.first_tile) * KH_TILE;  // first start position
  uint64_t need_end = tile_base + KH_TILE + (K - 1);                      // bases [tile_base, need_end)
  if (need_end > gd.seq_len) need_end = gd.seq_len;

  // ---- phase A: bytes -> nibble codes + validity, staged in this warp's shared memory ----
  const uintptr_t p_lo = (uintptr_t)(seq + gd.seq_begin + tile_base);
  const uintptr_t p_al = p_lo & ~(uintptr_t)15;
  const uint32_t sh = (uint32_t)(p_lo - p_al);                     // 0..15 bases of alignment slack
  const uint32_t hi_off = sh + (uint32_t)(need_end - tile_base);   // bytes [sh, hi_off) of the aligned window are this tile's
  // constants that must live in registers (as immediates they cost an extra instruction per use)
  const uint32_t k_fold = consts.x, k_lut = consts.y;  // 0xDFDFDFDF, 0x15060200 (kernel arguments, see launch_kc)
#pragma unroll
  for (int it = 0; it < (KH_CHUNKS + 4 + 31) / 32; ++it) {
    const uint32_t c = lane + 32u * it, off = 16u * c;
    if (c >= KH_CHUNKS + 4) break;
    uint2 n = make_uint2(0u, 0u);
    uint32_t valid = 0;
    if (c < KH_CHUNKS && off < hi_off) {
      const uint4 v = ld_stream16(reinterpret_cast<const void *>(p_al + off));
      uint32_t bad = 0;
      n.x = encode8(v.x, v.y, bad, k_fold, k_lut);
      n.y = encode8(v.z, v.w, bad, k_fold, k_lut);
      valid = 0xFFFFu;
      if (bad) {  // a byte that is not a base (N runs, IUPAC codes, the bytes past a genome's end): exact validity bits
        uint32_t n16, v4;
        encode4(v.x, n16, v4); valid = v4;
        encode4(v.y, n16, v4); valid |= v4 << 4;
        encode4(v.z, n16, v4); valid |= v4 << 8;
        encode4(v.w, n16, v4); valid |= v4 << 12;
      }
      // bytes of this chunk outside [sh, hi_off) belong to someone else (or nobody)
      const uint32_t first = c == 0 ? sh : 0u, last = min(hi_off - off, 16u);
      valid &= ((1u << last) - 1u) & (0xFFFFFFFFu << first);
    }
    *reinterpret_cast<uint2 *>(s_nib + 2 * c) = n;
    s_valid16[c] = (uint16_t)valid;
  }
  __syncwarp();

  // ---- phase B: 32 start positions per thread ----
  const int t = lane;
  const uint32_t nb0 = sh + 32u * t;  // this thread's first base, as a nibble index into s_nib
  auto window8 = [&](uint32_t nib_off) -> uint32_t {  // 8 consecutive bases starting at nib_off
    const uint32_t idx = nib_off >> 3;
    return funnel_r(s_nib[idx], s_nib[idx + 1], (nib_off & 7u) * 4u);
  };
  uint64_t v;
  {
    const uint32_t b0 = s_valid[t], b1 = s_valid[t + 1], b2 = s_valid[t + 2];
    v = (uint64_t)funnel_r(b0, b1, sh) | ((uint64_t)funnel_r(b1, b2, sh) << 32);
  }
  // kv bit j: all K bases of the k-mer starting at thread-local position j are valid
  uint64_t kv = ~0ull;
  {
    uint64_t r = v;
    int done = 0;
#pragma unroll
    for (int len = 1; len <= 32; len <<= 1) {
      if (K & len) { kv &= (r >> done); done += len; }
      r &= r >> len;
    }
  }
  const uint32_t kv32 = (uint32_t)kv;
  if (kv32 != 0) {

  // Rolling state, one nibble per base, FIRST base of the k-mer in the LOW nibble of word 0
  // (the byte order t1ha2 reads).  F = forward strand, R = reverse complement.  Before each
  // step F holds the previous k-mer; the step drops its first base and appends the new one.
  uint32_t F[NW], R[NW];
  {
    // X = the first K-1 bases of the window, nibble i = base i
    uint32_t X[NW];
#pragma unroll
    for (int m = 0; m < NW; ++m) {
      constexpr int P = K - 1;
      const int have = P - 8 * m;  // bases of X that live in word m
      X[m] = have <= 0 ? 0u : (window8(nb0 + 8 * m) & (have >= 8 ? 0xFFFFFFFFu : ((1u << (4 * (have & 7))) - 1u)));
    }
    // F = X << 4 (so that the first step's shift-right puts base i at nibble i)
#pragma unroll
    for (int m = NW - 1; m >= 0; --m) F[m] = (X[m] << 4) | (m > 0 ? (X[m - 1] >> 28) : 0u);
    // R: nibble i = complement(base[K-2-i]), i < K-1.  Complement = 5 - code on real bases.
    if (CANON) {
      constexpr int P = K - 1;
      uint32_t Y[NW];
#pragma unroll
      for (int m = 0; m < NW; ++m) {
        const int have = P - 8 * m;
        const uint32_t cm = have <= 0 ? 0u : (have >= 8 ? 0x55555555u : (0x55555555u & ((1u << (4 * (have & 7))) - 1u)));
        Y[m] = cm - X[m];
      }
      // reverse the nibble order of the whole NW-word value, then shift the P used nibbles down
      uint32_t V[NW + 1];
#pragma unroll
      for (int m = 0; m < NW; ++m) V[m] = rev_in_nibble(__brev(Y[NW - 1 - m]));
      V[NW] = 0;
      constexpr int SHB = 4 * (8 * NW - P);  // bits to shift right
      constexpr int SW = SHB / 32, SB = SHB % 32;
#pragma unroll
      for (int m = 0; m < NW; ++m) {
        const uint32_t lo = (m + SW) <= NW ? V[(m + SW) <= NW ? (m + SW) : NW] : 0u;
        const uint32_t hi = (m + SW + 1) <= NW ? V[(m + SW + 1) <= NW ? (m + SW + 1) : NW] : 0u;
        R[m] = SB ? funnel_r(lo, hi, SB) : lo;
      }
    } else {
#pragma unroll
      for (int m = 0; m < NW; ++m) R[m] = 0;
    }
  }

  uint64_t *table = tables + gd.table_begin;
  uint32_t *count = counts + g;
  const uint32_t thr_hi = (uint32_t)(threshold >> 32);

#pragma unroll KH_UNROLL
  for (int o = 0; o < KH_PPT / 8; ++o) {
    const uint32_t in32 = window8(nb0 + (K - 1) + 8 * o);  // the 8 incoming bases
    const uint32_t kv8 = kv32 >> (8 * o);
    // The eight k-mers of the group are windows of ONE (NW + 1)-word value each: XF = the state before the group with
    // the incoming bases appended above its K nibbles, YR = the reversed complements of the incoming bases below the
    // reverse-complement state.  Position jj is that value shifted by 4 (jj + 1) bits - one funnel shift per word, no
    // chain from position to position (the last one is a plain register move).
    uint32_t XF[NW + 1], YR[NW + 1];
#pragma unroll
    for (int m = 0; m + 1 < NW; ++m) XF[m] = F[m];
    XF[NW - 1] = LASTN < 8 ? (F[NW - 1] | (in32 << (4 * (LASTN & 7)))) : F[NW - 1];
    XF[NW] = LASTN < 8 ? (in32 >> (32 - 4 * LASTN)) : in32;
    if (CANON) {
      const uint32_t c = 0x55555555u - in32;  // complements (codes <= 4: no borrow between nibbles); 5 where there is no base
      const uint32_t b = prmt(c, 0u, 0x0123u);  // reverse the nibble order: bytes, then the two nibbles of every byte
      YR[0] = ((b & 0x0F0F0F0Fu) << 4) | ((b >> 4) & 0x0F0F0F0Fu);
#pragma unroll
      for (int m = 0; m < NW; ++m) YR[m + 1] = R[m];
    }
    // straight-line code for the whole group: the (rare) survivors are only flagged here and
    // inserted after the group, so the scheduler can interleave the ALU-heavy rolling/expansion
    // of one position with the multiply chains of its neighbours
    uint64_t hs[KH_GROUP];
    uint32_t min_hi = 0xFFFFFFFFu;  // smallest high word of the group's hashes: one VIMNMX per k-mer instead of a 64-bit compare
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) {
#pragma unroll
      for (int m = 0; m < NW; ++m) F[m] = jj < 7 ? funnel_r(XF[m], XF[m + 1], 4 * (jj + 1)) : XF[m + 1];
      if (LASTN < 8) F[NW - 1] &= LASTMASK;
      uint32_t C[NW];
      if (CANON) {
#pragma unroll
        for (int m = 0; m < NW; ++m) R[m] = jj < 7 ? __funnelshift_l(YR[m], YR[m + 1], 4 * (jj + 1)) : YR[m];
        if (LASTN < 8) R[NW - 1] &= LASTMASK;
        // ---- canonical = lexicographic min = numeric min of the packed states (see the code table above):
        //      borrow chain over the words, least significant first; mask = all ones iff F < R ----
        uint32_t mask;
        if (NW == 1) {
          asm("{.reg .u32 t; sub.cc.u32 t, %1, %2; subc.u32 %0, 0, 0;}" : "=r"(mask) : "r"(F[0]), "r"(R[0]));
        } else if (NW == 2) {
          asm("{.reg .u32 t; sub.cc.u32 t, %1, %2; subc.cc.u32 t, %3, %4; subc.u32 %0, 0, 0;}"
              : "=r"(mask) : "r"(F[0]), "r"(R[0]), "r"(F[1]), "r"(R[1]));
        } else if (NW == 3) {
          asm("{.reg .u32 t; sub.cc.u32 t, %1, %2; subc.cc.u32 t, %3, %4; subc.cc.u32 t, %5, %6; subc.u32 %0, 0, 0;}"
              : "=r"(mask) : "r"(F[0]), "r"(R[0]), "r"(F[1]), "r"(R[1]), "r"(F[2]), "r"(R[2]));
        } else {
          asm("{.reg .u32 t; sub.cc.u32 t, %1, %2; subc.cc.u32 t, %3, %4; subc.cc.u32 t, %5, %6; subc.cc.u32 t, %7, %8; subc.u32 %0, 0, 0;}"
              : "=r"(mask) : "r"(F[0]), "r"(R[0]), "r"(F[1]), "r"(R[1]), "r"(F[NW > 2 ? 2 : 0]), "r"(R[NW > 2 ? 2 : 0]), "r"(F[NW - 1]), "r"(R[NW - 1]));
        }
#pragma unroll
        for (int m = 0; m < NW; ++m) C[m] = (F[m] & mask) | (R[m] & ~mask);
      } else {
#pragma unroll
        for (int m = 0; m < NW; ++m) C[m] = F[m];
      }
      // ---- ASCII expansion: each nibble is a PRMT selector into {0,'A','C','G','T',0,0,0} ----
      uint64_t w[NW];
      w[0] = 0;  // (read by t1ha2_kmer only)
#pragma unroll
      for (int m = TAB ? 1 : 0; m < NW; ++m) {
        const uint32_t lo = prmt(lut_lo, lut_hi, C[m]);
        const uint32_t hi = prmt(lut_lo, lut_hi, C[m] >> 16);
        w[m] = (uint64_t)lo | ((uint64_t)hi << 32);
      }
      uint64_t h;
      if (TAB) {
        // table indices from the nibble codes: code - 1 is the 2-bit base value; x * 5 puts the values of nibbles
        // 2n and 2n + 1 side by side at bits 2-5 of byte n, and * 0x44 gathers i at bits 8-15 and j at bits 24-31
        const uint32_t z = (((C[0] - 0x11111111u) * 5u) & 0x3C3C3C3Cu) * 0x44u;
        const char *tab = reinterpret_cast<const char *>(s_tab) + (threadIdx.x & 1u) * sizeof(uint4);  // this lane's copy
        const uint4 l = *reinterpret_cast<const uint4 *>(tab + ((z >> 3) & 0x1FE0u));                 // L[i]: 32 i
        const uint4 hh = *reinterpret_cast<const uint4 *>(tab + 256 * 32 + ((z >> 19) & 0x1FE0u));    // H[j]: 32 j
        uint32_t x_w1, y_lo, y_hi;  // word 1 of the sum carries into Y1 = words 2-3 (+ Y, folded into L)
        asm("add.cc.u32 %0, %3, %4; addc.cc.u32 %1, %5, %6; addc.u32 %2, %7, %8;"
            : "=r"(x_w1), "=r"(y_lo), "=r"(y_hi) : "r"(l.y), "r"(hh.x), "r"(l.z), "r"(hh.y), "r"(l.w), "r"(hh.z));
        if (R1::x_is_seed) x_w1 ^= (uint32_t)(seed >> 32);  // X_lo is in L; X_hi is 0 when X = K
        const uint64_t x1 = (uint64_t)l.x | ((uint64_t)x_w1 << 32);
        uint64_t y1 = (uint64_t)y_lo | ((uint64_t)y_hi << 32);
        if (WRAP && (z & 0xFF00FF00u) >= wrap_at) y1 -= R1::prime;  // Y + w0 wrapped: t P is P 2^64 less
        h = R1::x_is_seed ? hg::t1ha2_kmer_rest<K>(x1, y1, w) : hg::t1ha2_kmer_rest<K>(y1, x1, w);
      } else {
        h = hg::t1ha2_kmer<K>(w, seed);
      }
      hs[jj % KH_GROUP] = h;
      min_hi = min(min_hi, (uint32_t)(h >> 32));
      if ((jj % KH_GROUP) == KH_GROUP - 1) {
        // some hash of these KH_GROUP positions may be below the threshold (1 quartet in ~375 at scaled = 1500): the exact 64-bit test
        // and the validity of the position are looked at only here
        if (min_hi <= thr_hi) {
          const uint32_t gm = kv8 >> (jj + 1 - KH_GROUP);
#pragma unroll
          for (int e = 0; e < KH_GROUP; ++e)
            if (((gm >> e) & 1u) && hs[e] < threshold) {
              const uint32_t pos = atomicAdd(s_qn, 1u);
              if (pos < KH_QCAP) s_queue[pos] = hs[e];
              else table_insert(table, gd.table_mask, hs[e], count, status);  // queue full (tiny `scaled`)
            }
        }
        min_hi = 0xFFFFFFFFu;
      }
    }
  }
  }  // kv32 != 0
  __syncwarp();
  const uint32_t qn = min(*s_qn, (uint32_t)KH_QCAP);
  for (uint32_t i = lane; i < qn; i += 32) table_insert(tables + gd.table_begin, gd.table_mask, s_queue[i], counts + g, status);
  }
}

// cta_genome[c] = genome that owns tile c * KH_WARPS: one warp per genome fills its range.  The CTAs from
// tab_cta on build the round-1 tables (one L and one H entry per thread) for X, Y, P.
__global__ void tile_map_kernel(const hg_genome_desc *__restrict__ desc, uint32_t n_genomes,
                                uint32_t *__restrict__ cta_genome, uint32_t tab_cta, uint4 *__restrict__ tab,
                                uint64_t X, uint64_t Y, uint64_t P) {
  if (blockIdx.x >= tab_cta) {
    const uint32_t e = (blockIdx.x - tab_cta) * blockDim.x + threadIdx.x;
    if (e >= 256) return;
    // L[e] = (Y + w_lo(e)) P mod 2^128; the add may carry out of 64 bits, and that carry is worth P 2^64
    const uint64_t t = Y + ascii4(e);
    const uint64_t lo = t * P, hi = __umul64hi(t, P) + (t < Y ? P : 0ull) + Y;
    tab[e] = make_uint4((uint32_t)lo ^ (uint32_t)X, (uint32_t)(lo >> 32), (uint32_t)hi, (uint32_t)(hi >> 32));
    // H[e] = w_hi(e) P < 2^96
    const uint64_t wh = ascii4(e), hlo = wh * P;
    tab[256 + e] = make_uint4((uint32_t)hlo, (uint32_t)(hlo >> 32), (uint32_t)__umul64hi(wh, P), 0u);
    return;
  }
  const uint32_t g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (g >= n_genomes) return;
  const uint32_t c0 = (desc[g].first_tile + KH_WARPS - 1) / KH_WARPS;
  const uint32_t c1 = (desc[g + 1].first_tile + KH_WARPS - 1) / KH_WARPS;
  for (uint32_t c = c0 + lane; c < c1; c += 32) cta_genome[c] = g;
}

// byte offset of the round-1 tables in HG_S_MISC, behind the CTA -> genome map
size_t kh_tab_offset(uint32_t n_tiles) { return ((size_t)(n_tiles + KH_WARPS - 1) / KH_WARPS * 4 + 255) & ~(size_t)255; }

// The smallest index j * 256 + i whose word 0 wraps Y + w0 past 2^64, in the (z & 0xFF00FF00) form the kernel
// compares (j at bits 24-31, i at bits 8-15); KH_NO_WRAP when Y + w0 wraps for no word 0.
constexpr uint32_t KH_NO_WRAP = 0xFFFFFFFFu;  // above every (z & 0xFF00FF00)
uint32_t kh_wrap_at(uint64_t Y) {
  auto w0 = [](uint32_t idx) { return (uint64_t)ascii4(idx & 0xFFu) | ((uint64_t)ascii4(idx >> 8) << 32); };
  if (Y + w0(0xFFFFu) >= Y) return KH_NO_WRAP;
  uint32_t lo = 0, hi = 0xFFFFu;  // w0 grows with the index: bisect for the first wrapping one, which is <= hi
  while (lo < hi) {
    const uint32_t mid = (lo + hi) / 2;
    if (Y + w0(mid) < Y) hi = mid;
    else lo = mid + 1;
  }
  return ((lo >> 8) << 24) | ((lo & 0xFFu) << 8);
}

template <int K, bool CANON, bool WRAP>
int launch_kc(hg_ctx *ctx, uint32_t n_tiles, const uint8_t *d_seq, const hg_genome_desc *d_desc, uint32_t n_genomes,
              const uint64_t *d_true_len, uint64_t threshold, uint64_t seed, uint64_t *d_tables, uint32_t *d_counts,
              uint32_t wrap_at) {
  using R1 = hg::t1ha2_round1<K>;
  const uint32_t grid = (n_tiles + KH_WARPS - 1) / KH_WARPS;
  void *d_map;
  int rc = hg_scratch(ctx, HG_S_MISC, hg_kmer_map_bytes(n_tiles), &d_map);
  if (rc) return rc;
  uint4 *d_tab = (uint4 *)((uint8_t *)d_map + kh_tab_offset(n_tiles));
  const uint32_t map_ctas = (n_genomes * 32 + 127) / 128, tab_ctas = K >= 8 ? 2 : 0;
  const uint64_t X = R1::x_is_seed ? seed : (uint64_t)K, Y = R1::x_is_seed ? (uint64_t)K : seed;
  tile_map_kernel<<<map_ctas + tab_ctas, 128, 0, ctx->stream>>>(d_desc, n_genomes, (uint32_t *)d_map, map_ctas, d_tab,
                                                                X, Y, R1::prime);
  kmer_hash_kernel<K, CANON, WRAP><<<grid, KH_THREADS, 0, ctx->stream>>>(
      d_seq, d_desc, n_genomes, n_tiles, threshold, seed, d_tables, d_counts, ctx->d_status, 0x47434100u, 0x00000054u,
      (const uint32_t *)d_map, d_true_len, make_uint2(0xDFDFDFDFu, 0x15060200u), d_tab, wrap_at);
  ctx->launches += 2;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

template <int K>
int launch_k(hg_ctx *ctx, bool canon, uint32_t n_tiles, const uint8_t *d_seq, const hg_genome_desc *d_desc,
             uint32_t n_genomes, const uint64_t *d_true_len, uint64_t threshold, uint64_t seed, uint64_t *d_tables,
             uint32_t *d_counts) {
  // only a seed in the Y role can wrap (K = 8 and 17..24), and only a seed near 2^64: a kernel of its own
  if constexpr (K >= 8 && !hg::t1ha2_round1<K>::x_is_seed) {
    const uint32_t wrap_at = kh_wrap_at(seed);
    if (wrap_at != KH_NO_WRAP)
      return canon ? launch_kc<K, true, true>(ctx, n_tiles, d_seq, d_desc, n_genomes, d_true_len, threshold, seed,
                                              d_tables, d_counts, wrap_at)
                   : launch_kc<K, false, true>(ctx, n_tiles, d_seq, d_desc, n_genomes, d_true_len, threshold, seed,
                                               d_tables, d_counts, wrap_at);
  }
  return canon ? launch_kc<K, true, false>(ctx, n_tiles, d_seq, d_desc, n_genomes, d_true_len, threshold, seed, d_tables,
                                           d_counts, KH_NO_WRAP)
               : launch_kc<K, false, false>(ctx, n_tiles, d_seq, d_desc, n_genomes, d_true_len, threshold, seed, d_tables,
                                            d_counts, KH_NO_WRAP);
}

}  // namespace

uint32_t hg_kmer_tile_positions() { return KH_TILE; }
size_t hg_kmer_map_bytes(uint32_t n_tiles) { return kh_tab_offset(n_tiles) + KH_TAB_BYTES; }

int hg_launch_kmer_hash(hg_ctx *ctx, const uint8_t *d_seq, const hg_genome_desc *d_desc, uint32_t n_genomes,
                        uint32_t n_tiles, const hg_sketch_params *p, const uint64_t *d_true_len, uint64_t *d_tables,
                        uint32_t *d_counts) {
  if (n_tiles == 0) return HG_OK;
  const uint64_t threshold = UINT64_MAX / p->scaled;  // sketch.rs:73
  const bool canon = p->canonical != 0;
  switch (p->ksize) {
#define HG_K(KK) \
  case KK: return launch_k<KK>(ctx, canon, n_tiles, d_seq, d_desc, n_genomes, d_true_len, threshold, p->seed, d_tables, \
                               d_counts);
#ifdef HG_KMER_ONLY_K21  // (development: one instantiation, for reading its SASS)
    HG_K(21)
#else
    HG_K(1) HG_K(2) HG_K(3) HG_K(4) HG_K(5) HG_K(6) HG_K(7) HG_K(8)
    HG_K(9) HG_K(10) HG_K(11) HG_K(12) HG_K(13) HG_K(14) HG_K(15) HG_K(16)
    HG_K(17) HG_K(18) HG_K(19) HG_K(20) HG_K(21) HG_K(22) HG_K(23) HG_K(24)
    HG_K(25) HG_K(26) HG_K(27) HG_K(28) HG_K(29) HG_K(30) HG_K(31) HG_K(32)
#endif
#undef HG_K
    default:
      hg_set_error("ksize %u unsupported (1..32)", (unsigned)p->ksize);
      return HG_E_INVALID;
  }
}
