// hg_common.cuh — shared declarations for the sm_100a HyperGen hot path.
// Arithmetic building blocks restate, for the device, the functions the reference defines in
// src/cuda_kernel.cu:71-246 (t1ha2), the wyhash crate's wyrng (call sites src/hd.rs:44,51)
// and glibc's logf (behind f32::ln in src/dist.rs:154).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "../../include/hypergen_b200.h"

#define HG_EMPTY_SLOT 0xFFFFFFFFFFFFFFFFull

// ---------------------------------------------------------------------------------------
// t1ha2_atonce (length <= 32) on pre-assembled little-endian words.
//   reference: cuda_kernel.cu:196-246 (switch), :136-141 mixup64, :149-153 final64.
// ---------------------------------------------------------------------------------------
namespace hg {

__host__ __device__ constexpr uint64_t t1_p0() { return 0xEC99BF0D8372CAABull; }
__host__ __device__ constexpr uint64_t t1_p1() { return 0x82434FE90EDCEF39ull; }
__host__ __device__ constexpr uint64_t t1_p2() { return 0xD4F06DB99D67BE4Bull; }
__host__ __device__ constexpr uint64_t t1_p3() { return 0xBD9CACC22C6E9571ull; }
__host__ __device__ constexpr uint64_t t1_p4() { return 0x9C06FAF4D023E3ABull; }
__host__ __device__ constexpr uint64_t t1_p5() { return 0xC060724A8424F345ull; }
__host__ __device__ constexpr uint64_t t1_p6() { return 0xCB5AF53AE3AAAC31ull; }

// rotate right by a compile-time amount: two funnel shifts (written out, nvcc makes four instructions of the shift-or form)
template <unsigned S>
__device__ __forceinline__ uint64_t rot64(uint64_t v) {
  static_assert(S > 0 && S < 64 && S != 32, "rot64");
  const uint32_t lo = S < 32 ? (uint32_t)v : (uint32_t)(v >> 32), hi = S < 32 ? (uint32_t)(v >> 32) : (uint32_t)v;
  const uint32_t a = __funnelshift_r(lo, hi, S & 31), b = __funnelshift_r(hi, lo, S & 31);
  return (uint64_t)a | ((uint64_t)b << 32);
}

__device__ __forceinline__ void mixup64(uint64_t &a, uint64_t &b, uint64_t v, uint64_t prime) {
  const uint64_t t = b + v;
  a ^= t * prime;
  b += __umul64hi(t, prime);
}

__device__ __forceinline__ uint64_t final64(uint64_t a, uint64_t b) {
  const uint64_t x = (a + rot64<41>(b)) * t1_p0();
  const uint64_t y = (rot64<23>(a) + b) * t1_p6();
  const uint64_t v = x ^ y;
  return (v * t1_p5()) ^ __umul64hi(v, t1_p5());
}

// NW = ceil(K / 8) words; word m holds bytes 8m..8m+7 of the k-mer, little-endian, the last
// one zero-extended (tail64_le_unaligned, cuda_kernel.cu:155-194).  Word m is mixed with prime
// p_(NW-m), alternately into (a, b) and (b, a), starting from a = seed, b = K.
//
// Round 1 (word 0) is mixup64(X, Y, w[0], P): which of a, b plays X (xored) and which Y (added
// to) depends on NW alone.  kmer_hash.cu takes this round from product tables built from these
// roles; rounds 2.. and final64 are t1ha2_kmer_rest for every caller.
template <int K>
struct t1ha2_round1 {
  static constexpr int NW = (K + 7) / 8;
  static constexpr bool x_is_seed = NW % 2 == 0;  // mixup64(a, b, ...): X = a = seed, Y = b = K
  static constexpr uint64_t prime = NW == 4 ? t1_p4() : NW == 3 ? t1_p3() : NW == 2 ? t1_p2() : t1_p1();
};

// words 1..NW-1 and final64, from the state (a, b) after round 1
template <int K>
__device__ __forceinline__ uint64_t t1ha2_kmer_rest(uint64_t a, uint64_t b, const uint64_t (&w)[(K + 7) / 8]) {
  constexpr int NW = (K + 7) / 8;
  if (NW > 3) mixup64(b, a, w[NW > 3 ? NW - 3 : 0], t1_p3());
  if (NW > 2) mixup64(a, b, w[NW > 2 ? NW - 2 : 0], t1_p2());
  if (NW > 1) mixup64(b, a, w[NW - 1], t1_p1());
  return final64(a, b);
}

template <int K>
__device__ __forceinline__ uint64_t t1ha2_kmer(const uint64_t (&w)[(K + 7) / 8], uint64_t seed) {
  uint64_t a = seed, b = (uint64_t)K;
  if (t1ha2_round1<K>::x_is_seed) mixup64(a, b, w[0], t1ha2_round1<K>::prime);
  else mixup64(b, a, w[0], t1ha2_round1<K>::prime);
  return t1ha2_kmer_rest<K>(a, b, w);
}

// ---------------------------------------------------------------------------------------
// WyRng word i (0-based) of the generator seeded with h: the state advances by a constant,
// so the i-th output is a closed form of (h, i) — no sequential dependency (hd.rs:44,51).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t wyrng_word(uint64_t h, uint32_t i) {
  const uint64_t s = h + (uint64_t)(i + 1) * 0xa0761d6478bd642full;
  const uint64_t t = s ^ 0xe7037ed1a0b428dbull;
  return (s * t) ^ __umul64hi(s, t);
}

// ---------------------------------------------------------------------------------------
// glibc logf (FMA ifunc variant), bit-for-bit: double-precision table + polynomial, one
// final rounding to float.  Restated in oracle/hg_oracle.c:hgo_logf_glibc and checked there
// against the host libm over every positive float.
// ---------------------------------------------------------------------------------------
static __device__ __constant__ double c_logf_tab[32] = {
    0x1.661ec79f8f3bep+0, -0x1.57bf7808caadep-2, 0x1.571ed4aaf883dp+0, -0x1.2bef0a7c06ddbp-2,
    0x1.49539f0f010b0p+0, -0x1.01eae7f513a67p-2, 0x1.3c995b0b80385p+0, -0x1.b31d8a68224e9p-3,
    0x1.30d190c8864a5p+0, -0x1.6574f0ac07758p-3, 0x1.25e227b0b8ea0p+0, -0x1.1aa2bc79c8100p-3,
    0x1.1bb4a4a1a343fp+0, -0x1.a4e76ce8c0e5ep-4, 0x1.12358f08ae5bap+0, -0x1.1973c5a611cccp-4,
    0x1.0953f419900a7p+0, -0x1.252f438e10c1ep-5, 0x1.0000000000000p+0, 0x0.0p+0,
    0x1.e608cfd9a47acp-1, 0x1.aa5aa5df25984p-5,  0x1.ca4b31f026aa0p-1, 0x1.c5e53aa362eb4p-4,
    0x1.b2036576afce6p-1, 0x1.526e57720db08p-3,  0x1.9c2d163a1aa2dp-1, 0x1.bc2860d224770p-3,
    0x1.886e6037841edp-1, 0x1.1058bc8a07ee1p-2,  0x1.767dcf5534862p-1, 0x1.4043057b6ee09p-2};

__device__ __forceinline__ float logf_glibc(float x) {
  uint32_t ix = __float_as_uint(x);
  if (ix == 0x3f800000u) return 0.0f;
  if (ix - 0x00800000u >= 0x7f800000u - 0x00800000u) {
    if (ix * 2 == 0) return __uint_as_float(0xff800000u);  // -inf
    if (ix == 0x7f800000u) return x;
    if ((ix & 0x80000000u) || ix * 2 >= 0xff000000u) return __uint_as_float(0x7fc00000u);
    ix = __float_as_uint(__fmul_rn(x, 8388608.0f));  // subnormal: scale by 2^23
    ix -= 23u << 23;
  }
  const uint32_t tmp = ix - 0x3f330000u;
  const uint32_t i = (tmp >> 19) & 15;
  const int k = (int)tmp >> 23;
  const uint32_t iz = ix - (tmp & 0xff800000u);
  const double z = (double)__uint_as_float(iz);
  const double invc = c_logf_tab[2 * i], logc = c_logf_tab[2 * i + 1];
  const double r = __fma_rn(z, invc, -1.0);
  const double y0 = __fma_rn((double)k, 0x1.62e42fefa39efp-1, logc);
  const double r2 = __dmul_rn(r, r);
  double y = __fma_rn(r, 0x1.5575b0be00b6ap-2, -0x1.ffffef20a4123p-2);
  y = __fma_rn(r2, -0x1.00ea348b88334p-2, y);
  y = __fma_rn(r2, y, __dadd_rn(y0, r));
  return __double2float_rn(y);
}

// compute_pairwise_ani after the dot product: src/dist.rs:153-160, every operation a
// correctly rounded f32 op exactly as rustc emits it (no contraction, no fast-math).
__device__ __forceinline__ float ani_from_dot(int32_t dot, int32_t norm2_r, int32_t norm2_q, float ksize_f) {
  const int32_t den = (int32_t)((uint32_t)norm2_r + (uint32_t)norm2_q - (uint32_t)dot);
  const float jaccard = __fdiv_rn(__int2float_rn(dot), __int2float_rn(den));
  float t = __fdiv_rn(1.0f, jaccard);
  t = __fadd_rn(t, 1.0f);
  t = __fdiv_rn(2.0f, t);
  float ani = __fadd_rn(1.0f, __fdiv_rn(logf_glibc(t), ksize_f));
  if (ani != ani) return 0.0f;
  ani = ani < 1.0f ? ani : 1.0f;  // f32::min(1.0)
  ani = ani > 0.0f ? ani : 0.0f;  // f32::max(0.0)
  return __fmul_rn(ani, 100.0f);
}

}  // namespace hg

// ---------------------------------------------------------------------------------------
// host-side plumbing shared by the .cu files
// ---------------------------------------------------------------------------------------
struct hg_ctx {
  int device;
  int sm_count;
  cudaStream_t stream;
  unsigned long long launches;
  // grow-only device scratch
  void *d_scratch[16];        // indexed by hg_scratch_slot
  size_t d_scratch_bytes[16];
  // pinned host scratch
  void *h_pinned[4];
  size_t h_pinned_bytes[4];
  // last dist decision (hg_dist_record)
  int dist_path;
  char dist_reason[288];
  // status words of the last sketch batch (device + host copy)
  uint32_t *d_status;  // [0] table overflow, [1] quant range overflow
  uint32_t h_status[4];
  // optional stage timing (hg_set_profiling): events on ctx->stream around each stage
  int prof;
  cudaEvent_t ev[8];
  int ev_used;           // which stage boundaries were recorded in the last call
  // H2D pipeline of the host-pointer sketch entry
  int tc_attr_set;
  int n1_attr_set;
  cudaStream_t copy_stream;  // created on first use, with the events below
  cudaEvent_t ev_copied[2], ev_done[2];
  cudaEvent_t ev_chunk[10];  // dist streaming: fork + query matrix + one per row chunk
  // hg_dist_dev with the single-plane path forced: the pre-pass verdict is not waited for (hg_dist_status reads it)
  const uint32_t *pending_stats[2];
  uint32_t pending_nsets[2];
  // the last search (hg_search_stats): sample rows, candidates of the floor and the main pass, reruns; with profiling
  // on, events at its step boundaries (created on first use)
  uint64_t search_stats[4];
  cudaEvent_t ev_search[5];
  int search_ev_used;
  // the last cluster run (hg_cluster_stats): windows, linked pairs, largest window's pairs, edge capacity; device ms of
  // its steps (-1: not run or profiling off)
  uint64_t cluster_stats[4];
  float cluster_ms[4];
  // the last derep run (hg_derep_stats): column chunks, windows, linked pairs, representatives; device ms of its
  // phases (-1: not run or profiling off)
  uint64_t derep_stats[4];
  float derep_ms[4];
  // the last ANI matrix run (hg_ani_matrix_stats): bands, entries, bytes copied to the host, kernel path; device ms of
  // its stages (-1: not run or profiling off)
  uint64_t matrix_stats[4];
  float matrix_ms[4];
  // the last FASTA records call (hg_fasta_records_stats): chunks, records, table slots; device ms of merge, index, hash,
  // encode and the host gap (-1: profiling off)
  uint64_t records_stats[4];
  float records_ms[5];
};

// stage boundaries: 0 start, 1 after staging/memsets, 2 after k-mer hash, 3 after encode,
// 4 dist start, 5 dist end
#define HG_PROF(ctx, idx)                                              \
  do {                                                                 \
    if ((ctx)->prof) {                                                 \
      cudaEventRecord((ctx)->ev[idx], (ctx)->stream);                  \
      (ctx)->ev_used |= 1 << (idx);                                    \
    }                                                                  \
  } while (0)

void hg_set_error(const char *fmt, ...);
int hg_cuda_fail(cudaError_t e, const char *what, const char *file, int line);
#define HG_CUDA(call)                                                   \
  do {                                                                  \
    cudaError_t e__ = (call);                                           \
    if (e__ != cudaSuccess) return hg_cuda_fail(e__, #call, __FILE__, __LINE__); \
  } while (0)

// Grow-only device scratch slots.  A slot has one tenant per entry point; entry points of one
// context never run concurrently (one stream), so slots may be shared between them.
// The FASTA records entry (hg_sketch_fasta_records) stages like the per-file one (REF_LIMBS raw, SEQ merged,
// QRY_LIMBS merge metadata, DESC, TABLES, COUNTS, MISC per chunk) and keeps its outputs for the whole call in PACKED,
// SMALL, SORT_TMP and SORT_CNT, which grow between chunks with their contents kept (hg_scratch_keep).
enum hg_scratch_slot {
  HG_S_SEQ = 0,        // staged sequence bytes (two halves when the H2D pipeline is active); search: the sample rows
  HG_S_DESC = 1,       // hg_genome_desc[] (+ sentinels); search: the per-query floors
  HG_S_TABLES = 2,     // per-genome hash tables / explicit hash sets
  HG_S_COUNTS = 3,     // distinct-hash counters; dist: the hit counter of the host entry; cluster: the edge counter and
                       // the run's linked-pair counts; derep (phase 1): the same
  HG_S_HV = 4,         // int16 HVs (sketch output staging; dist: both matrices of the host entry)
  HG_S_PACKED = 5,     // packed sketches; dist: hit records of the host entry; search: the candidates of a pass;
                       // group search: the members' results gathered on GPU 0; cluster, derep (phase 1): the edges of
                       // one window; records: the packed row of every record
  HG_S_SMALL = 6,      // norms / bits / counts per sketch; records: norm2 of every record
  HG_S_MISC = 7,       // CTA -> genome map + round-1 tables, |hv| max, probe sink, status word of a search merge; cluster: status word
                       // of a union check, root count of a flatten
  HG_S_REF_LIMBS = 8,  // s8 limb planes of the ref matrix (dist_tc)
  HG_S_QRY_LIMBS = 9,  // s8 limb planes of the query matrix (dist_tc)
  HG_S_SORT_TMP = 10,  // ping-pong buffer of the hit sort; search: the per-query segments; group search: the merged result;
                       // group cluster: the merged forest and the members' forests gathered on GPU 0; records: the
                       // quant bits of every record
  HG_S_SORT_CNT = 11,  // digit counters of the hit sort; search: per-query counts and offsets; records: n_hashes of
                       // every record
  HG_S_NARROW_META = 12,  // per-row constants + outlier lists of the single-plane dist path (dist_narrow); records:
                          // the index pass's header count per block and their prefix
  HG_S_TILES = 13,        // tile list of a multi-GPU dist launch (peer.cu); search: the results of the host entries;
                          // cluster: the forest of the packed entry; derep: its state (is_rep, rep list, order, the
                          // search result, covered flags, bitmap, counters) and the labels of the packed entry;
                          // records: one chunk's record table and the merged offsets of its headers' 'N'
  // derep: what the internal search (HG_S_SEQ, DESC, PACKED, COUNTS, SORT_*, MISC and the dist slots) and the packed
  // staging (HV, SMALL, TABLES) leave alone
  HG_S_DEREP_ROWS = 14,   // the working matrix in priority order, and its norms (when an order is given)
  HG_S_DEREP_REPS = 15,   // the representatives' rows in priority order, and their norms: the refs of the search
  HG_S_COUNT = 16
};
// scratch slot `slot` grown to at least `bytes` (contents not preserved)
int hg_scratch(hg_ctx *ctx, int slot, size_t bytes, void **out);
// the same with the slot's first `keep` bytes preserved across a growth (grows by half again, so a slot that grows a
// little per chunk is copied a logarithmic number of times)
int hg_scratch_keep(hg_ctx *ctx, int slot, size_t bytes, size_t keep, void **out);

// One context's part of a FASTA records call (api.cu): the record table on the host (file indices relative to the
// part's first file), the sketch rows in that context's HBM until hg_records_fetch copies them out.
struct hg_records_part {
  std::vector<hg_fasta_record> rec;
  const uint8_t *packed = nullptr, *bits = nullptr;
  const int32_t *norm2 = nullptr;
  const uint32_t *n_hashes = nullptr;
};
// the records of files file_off[0 .. n_files) (monotone, checked here); stops sketching once more than rec_cap
// records are found but counts them all
int hg_records_run(hg_ctx *ctx, const uint8_t *raw, const uint64_t *file_off, uint32_t n_files, const hg_sketch_params *p,
                   uint64_t rec_cap, hg_records_part &out);
// part's rows to the host outputs (any may be NULL), then the sketch status of the call (synchronises)
int hg_records_fetch(hg_ctx *ctx, const hg_records_part &part, uint32_t hv_d, uint8_t *packed, uint8_t *quant_bits,
                     int32_t *norm2, uint32_t *n_hashes);
int hg_pinned(hg_ctx *ctx, int slot, size_t bytes, void **out);

// The dist kernels, numbered as the `path` argument of the dist entries (include/hypergen_b200.h).
enum hg_dist_path { HG_PATH_AUTO = 0, HG_PATH_SIMT = 1, HG_PATH_TWO_LIMB = 2, HG_PATH_NARROW = 3 };
constexpr int32_t HG_LIMB_MAX_ABS = 8127;  // the largest |x| that splits into two s8 limbs x = 128 h + l (13 bits)
// ceil(2^31 / 3): while both rows' true norms sum x^2 stay below it, no i32 norm, dot or denominator of the pair wraps,
// and the tensor kernels' per-row / per-column candidate bounds are exact.  A row at or above it is a candidate against
// every column (DESIGN.md, dist epilogue).
constexpr uint64_t HG_NORM_WRAP_CUT = 715827883ull;
// sets what hg_dist_last_path / hg_dist_last_reason report
void hg_dist_record(hg_ctx *ctx, int path, const char *fmt, ...);

// Per-query thresholds of a search pass (hg_search_*), in place of the scalar ani_th: query column j of a launch keeps
// the pairs (i, j) whose key (ANI desc, ref index i asc) is at least (q[j].ani, q[j].imax) - ani > q[j].ani, or
// ani == q[j].ani and i <= q[j].imax - and q[j].jmin / q[j].cfrac are dist_jmin's pre-filter constants for q[j].ani.
// *cfrac_row is the smallest POSITIVE cfrac of the launch: the row term of the tensor kernels' candidate bound, valid
// for every column because cfrac_row * n_r + cfrac_j * n_q <= cfrac_j * (n_r + n_q).  A column whose cfrac is 0 (its
// floor is <= 0) is always a candidate and does not lower the row term of the others.
struct __align__(16) hg_floor { float ani, jmin, cfrac; uint32_t imax; };
struct hg_floors {
  const hg_floor *q;       // indexed like the launch's query norms
  const float *cfrac_row;  // device scalar (0: no positive cfrac)
};

// Dense output of a dist launch (hg_ani_matrix_*): the exact i32 dot of every live pair goes to its cell, in place of
// the threshold and the append (a conversion kernel turns the cells into ANI afterwards).  Cell (i, j) of global ref row
// i and query column j lies at base + hg_dense_row(i) - hg_dense_row(row_base) + j: base holds row `row_base` first.
// ld > 0: a rectangle with rows ld apart; ld == 0: the strict lower triangle (row i at i (i - 1) / 2, only j < i written).
struct hg_dense {
  int32_t *base;
  uint64_t ld;
  uint32_t row_base;
};
__host__ __device__ inline uint64_t hg_dense_row(const hg_dense &d, uint32_t i) {
  return d.ld ? (uint64_t)i * d.ld : (uint64_t)i * ((uint64_t)i - 1) / 2;
}

// ---- kernel launchers (all asynchronous on ctx->stream) ----

struct hg_genome_desc {   // per genome, device-visible
  uint64_t seq_begin;     // byte offset of the genome in the sequence buffer
  uint64_t seq_len;       // bases
  uint64_t table_begin;   // first slot of this genome's hash table
  uint32_t table_mask;    // slots - 1 (slots is a power of two) — used by the inserts
  uint32_t first_tile;    // index of this genome's first tile in the launch
  uint32_t table_slots;   // slots the encoder scans (== mask + 1, or a dense list length)
  uint32_t pad_;
};

// d_true_len (optional): per genome the bases to hash when fewer than desc.seq_len (the merged length of a FASTA file
// whose tiles were planned from its raw size)
int hg_launch_kmer_hash(hg_ctx *ctx, const uint8_t *d_seq, const hg_genome_desc *d_desc,
                        uint32_t n_genomes, uint32_t n_tiles, const hg_sketch_params *p,
                        const uint64_t *d_true_len, uint64_t *d_tables, uint32_t *d_counts);
// bytes of HG_S_MISC that hg_launch_kmer_hash over n_tiles tiles takes for its CTA -> genome map and t1ha2 round-1 tables
size_t hg_kmer_map_bytes(uint32_t n_tiles);
int hg_launch_sort_tables(hg_ctx *ctx, const hg_genome_desc *d_desc, uint32_t n_genomes,
                          uint64_t *d_tables, uint32_t max_slots);
int hg_launch_encode(hg_ctx *ctx, const hg_genome_desc *d_desc, uint32_t n_genomes,
                     const uint64_t *d_tables, const uint32_t *d_counts, uint32_t hv_d,
                     int16_t *d_hv, uint8_t *d_packed, uint8_t *d_quant_bits, int32_t *d_norm2,
                     uint32_t *d_n_hashes);
int hg_launch_unpack(hg_ctx *ctx, const uint8_t *d_packed, uint64_t row_stride,
                     const uint8_t *d_quant_bits, uint32_t n, uint32_t hv_d, int16_t *d_hv);
int hg_launch_dist_simt(hg_ctx *ctx, const int16_t *d_ref, const int32_t *d_ref_norm, uint32_t n_ref,
                        uint32_t i0, const int16_t *d_qry, const int32_t *d_qry_norm, uint32_t n_qry,
                        uint32_t j0, uint32_t hv_d, uint32_t ksize, float ani_th, int symmetric,
                        hg_hit *d_hits, uint64_t cap, unsigned long long *d_n_hits, const hg_floors *floors = nullptr,
                        const hg_dense *dense = nullptr);
// rows [a, a + h) of a dense output (every cell the launches wrote): dot -> ani_from_dot in place, f32 bits over i32.
// Rectangle rows hold n_cols cells, lower-triangle row i holds i.  Norms are indexed by global row / column.
int hg_launch_ani_convert(hg_ctx *ctx, const hg_dense &d, uint32_t a, uint32_t h, uint32_t n_cols, const int32_t *d_ref_norm,
                          const int32_t *d_qry_norm, uint32_t ksize);
// A dist launch that is one member of several GPUs (csrc/peer.cu) walks a host-built list of ITS tiles instead of the
// arithmetic enumeration, ordered by when the rows they read arrive, and its TMA producer waits for the arrival flags
// of those rows: the operand exchange over NVLink overlaps the tile computation.
// What a multi-GPU member pushes to the other members WHILE its dist kernel runs: the kernel carries extra "pusher"
// warps that copy this member's operand rows (byte ranges of its window) to the same offsets of other windows with
// 16-byte stores over NVLink.  The work is a list of UNITS, done in order: unit u sends one SET of byte ranges (set
// 0..3 = a chunk of this member's rows, set 4 = what every member needs before it starts: pre-pass statistics, outlier
// entries) to the members in its destination mask and then raises a flag in those windows - the chunk's arrival flag,
// or this member's start flag - when all pusher warps of the grid are through with it.  All-vs-all on three or more
// GPUs sends a member's rows only to the floor(N/2) members that compute tiles with them, nearest ring neighbour first
// (csrc/peer.cu); otherwise every chunk goes to everybody.  One kernel computes tiles and moves operands.
#define HG_PUSH_CHUNKS 4
#define HG_PUSH_SETS (HG_PUSH_CHUNKS + 1)
#define HG_PUSH_START_SET HG_PUSH_CHUNKS
#define HG_PUSH_RANGES 8
#define HG_PUSH_UNITS (1 + HG_PUSH_CHUNKS * (HG_MAX_PEERS / 2))
struct hg_push_plan {
  uint8_t *win[HG_MAX_PEERS];  // every member's window as this member addresses it
  int rank, world;
  uint64_t off[HG_PUSH_SETS][HG_PUSH_RANGES];   // byte ranges (relative to the window base), 4-byte granular
  uint32_t bytes[HG_PUSH_SETS][HG_PUSH_RANGES];
  int n[HG_PUSH_SETS];
  int n_units;
  uint8_t unit_set[HG_PUSH_UNITS];   // which set unit u sends
  uint8_t unit_dest[HG_PUSH_UNITS];  // bit m: to member m
  int8_t unit_stamp[HG_PUSH_UNITS];  // timeline stamp this unit's completion writes (-1: none)
  uint32_t *done;       // HG_PUSH_UNITS counters in this member's window: pusher warps through with the unit
  uint64_t ready_off;   // offset of the arrival flags in every window; chunk c raises flag rank * HG_PUSH_CHUNKS + c
  uint64_t start_off;   // offset of the start flags in every window; the start set raises flag `rank`
  const uint32_t *seq;  // the call's sequence number lives in device memory (the launch sequence is replayed as a CUDA graph)
  const uint32_t *dyn_count;  // not NULL: range 0 of the start set holds (*dyn_count - dyn_base) 4-byte entries, not its full size
  uint32_t dyn_base;
  unsigned long long *dbg;  // timeline stamps (HG_PEER_TIMELINE=1, hg_peer_timeline), else NULL
};
struct hg_tile_feed {
  const uint2 *list;        // x = tile row | tile column << 16, y = mask of the arrival flags the tile needs; NULL: arithmetic walk
  uint32_t n_list;
  const uint32_t *ready;    // 32 arrival flags (in this member's window); a flag is set when (int)(flag - seq) >= 0
  const uint32_t *seq_ptr;  // where the call's sequence number lives (device memory: the launch sequence is replayed as a CUDA graph)
  uint32_t seq;             // filled in by the kernel from *seq_ptr
  const uint32_t *start;    // HG_MAX_PEERS start flags (in this member's window): member m's start set has landed
  uint32_t start_need;      // bit m: wait for member m's start flag before anything is read (its pre-pass statistics and
                            // outlier entries are here; the root has reset its gather counter)
  uint32_t *status;         // set to 1 if a wait times out (the host turns it into an error)
  unsigned long long timeout_ns;
  unsigned long long *dbg;  // timeline stamps (HG_PEER_TIMELINE=1, hg_peer_timeline), else NULL
};

// HG_OK when both tensor kernels (two-limb and single-plane) tile this shape: hv_d % 128 == 0, hv_d <= 32768 (s32
// accumulator bound) and 16-byte aligned matrices; else HG_E_UNSUPPORTED with the reason in hg_last_error()
int hg_tensor_shape_ok(uint32_t hv_d, const void *d_a, const void *d_b);

// two s8 limb planes of one matrix (dist_tc.cu), split piecewise or at once
struct hg_tc_mat {
  const int16_t *hv;
  int8_t *planes;  // [2][n_rows][hv_d], followed by sq
  unsigned long long *sq;  // [n_rows]: sum x^2 of every row in 64 bits (the split writes it; HG_NORM_WRAP_CUT)
  uint32_t n_rows, hv_d;
};
// bytes of the planes and the row sums of an n_rows x hv_d matrix
uint64_t hg_tc_mat_bytes(uint32_t n_rows, uint32_t hv_d);
int hg_tc_setup(hg_ctx *ctx, const int16_t *d_hv, uint32_t n_rows, uint32_t hv_d, int plane_slot, hg_tc_mat *m);
int hg_tc_split_rows(hg_ctx *ctx, const hg_tc_mat *m, uint32_t row0, uint32_t rows);
int hg_tc_norm_flags(hg_ctx *ctx, const int16_t *d_hv, uint32_t n_rows, uint32_t hv_d, uint32_t *d_flags);
int hg_tc_launch(hg_ctx *ctx, const hg_tc_mat *R, uint32_t r0, uint32_t n_ref, uint32_t i0, const int32_t *d_ref_norm,
                 const hg_tc_mat *Q, uint32_t q0, uint32_t n_qry, uint32_t j0, const int32_t *d_qry_norm, uint32_t ksize,
                 float ani_th, int symmetric, hg_hit *d_hits, uint64_t cap, unsigned long long *d_n_hits,
                 const hg_floors *floors = nullptr, const hg_dense *dense = nullptr);
// `planes` holds hg_tc_mat_bytes(n_rows, hv_d)
int hg_tc_attach(hg_ctx *ctx, const int16_t *d_hv, uint32_t n_rows, uint32_t hv_d, int8_t *planes, hg_tc_mat *m);
int hg_tc_launch_ex(hg_ctx *ctx, const hg_tc_mat *R, uint32_t r0, uint32_t n_ref, uint32_t i0, const int32_t *d_ref_norm,
                    const hg_tc_mat *Q, uint32_t q0, uint32_t n_qry, uint32_t j0, const int32_t *d_qry_norm, uint32_t ksize,
                    float ani_th, int symmetric, hg_hit *d_hits, uint64_t cap, unsigned long long *d_n_hits, uint32_t walk_mul,
                    uint32_t walk_add, const hg_tile_feed *feed = nullptr, const hg_push_plan *push = nullptr,
                    const hg_floors *floors = nullptr, const hg_dense *dense = nullptr);
void hg_tc_tile_shape(uint32_t *rows, uint32_t *cols);
// single s8 plane (x = 2a + s) + sparse outlier corrections (dist_narrow.cu): one matrix in that form, prepared
// piecewise (rows as they arrive over PCIe) or at once
struct hg_narrow_mat {
  const int16_t *hv;  // the i16 matrix in HBM (n_rows x hv_d); rows need to be there only when they are prepared
  int8_t *plane;
  int32_t *s, *a2;
  uint32_t *e, *out_off, *out_cnt, *entries;
  // pre-pass statistics, 4 words per set: [0] max |x|, [1] max (|s| + 256), [2] entry cursor, [3] declined.
  // `stats` is the set THIS context's pre-pass writes; the dist kernel and the verdict reduce over the
  // n_sets sets at stats_all (one per member when the rows of the matrix were prepared on several GPUs).
  uint32_t *stats, *stats_all;
  uint32_t n_sets;
  uint32_t entry_base;  // first entry index this context's pre-pass may use ...
  uint32_t cap;         // ... and the limit (exclusive)
  uint32_t n_rows, hv_d;
};
size_t hg_narrow_meta_bytes(uint32_t n_rows);
int hg_narrow_setup(hg_ctx *ctx, const int16_t *d_hv, uint32_t n_rows, uint32_t hv_d, int plane_slot, void *meta,
                    hg_narrow_mat *m);
// the same over caller-provided memory (a peer window): nothing is allocated; entries_per_set as hg_narrow_set_cap()
size_t hg_narrow_arrays_bytes(uint32_t n_rows);  // s | a2 | e | out_off | out_cnt, n_rows words each
uint32_t hg_narrow_set_cap(uint32_t n_rows);
int hg_narrow_attach(hg_ctx *ctx, const int16_t *d_hv, uint32_t n_rows, uint32_t hv_d, int8_t *plane, void *arrays,
                     uint32_t *entries, uint32_t *stats_all, uint32_t n_sets, uint32_t my_set, uint32_t entry_base,
                     uint32_t set_cap, hg_narrow_mat *m, bool init_stats = true);
int hg_narrow_prep_rows(hg_ctx *ctx, const hg_narrow_mat *m, uint32_t row0, uint32_t rows);
int hg_narrow_norm_flags(hg_ctx *ctx, const int16_t *d_hv, uint32_t n_rows, uint32_t hv_d, uint32_t *d_flags);
int hg_narrow_launch(hg_ctx *ctx, const hg_narrow_mat *R, uint32_t r0, uint32_t n_ref, uint32_t i0, const int32_t *d_ref_norm,
                     const hg_narrow_mat *Q, uint32_t q0, uint32_t n_qry, uint32_t j0, const int32_t *d_qry_norm,
                     uint32_t ksize, float ani_th, int symmetric, hg_hit *d_hits, uint64_t cap,
                     unsigned long long *d_n_hits, const hg_floors *floors = nullptr, const hg_dense *dense = nullptr);
// as hg_narrow_launch for one member of `walk_mul` GPUs sharing the tile enumeration (takes tiles walk_add, walk_add + walk_mul, ...)
int hg_narrow_launch_ex(hg_ctx *ctx, const hg_narrow_mat *R, uint32_t r0, uint32_t n_ref, uint32_t i0, const int32_t *d_ref_norm,
                        const hg_narrow_mat *Q, uint32_t q0, uint32_t n_qry, uint32_t j0, const int32_t *d_qry_norm,
                        uint32_t ksize, float ani_th, int symmetric, hg_hit *d_hits, uint64_t cap,
                        unsigned long long *d_n_hits, uint32_t walk_mul, uint32_t walk_add, const hg_tile_feed *feed = nullptr,
                        const hg_push_plan *push = nullptr, const hg_floors *floors = nullptr, const hg_dense *dense = nullptr);
void hg_narrow_tile_shape(uint32_t *rows, uint32_t *cols);
int hg_narrow_verdict(hg_ctx *ctx, const hg_narrow_mat *A, const hg_narrow_mat *B, int32_t *absmax_out, uint64_t *outliers_out);
int hg_launch_int_peak(hg_ctx *ctx, int which, uint32_t iters, uint32_t *d_sink, uint32_t blocks);
// max |hv| over a device matrix (decides the dist path); result in *d_out (int32)
int hg_launch_sort_hits(hg_ctx *ctx, hg_hit *d_hits, uint64_t n, uint32_t *d_milli);
// top-k search (search.cu): s sample rows of the ref matrix (row t = ref row t * n_ref / s) into d_out / d_out_norm
int hg_launch_search_gather(hg_ctx *ctx, const int16_t *d_ref, const int32_t *d_ref_norm, uint32_t n_ref, uint32_t hv_d, uint32_t s,
                            int16_t *d_out, int32_t *d_out_norm);
// candidates (query indices < n_qry) -> per query the top_k best by (ANI desc, i asc): out / n_found / milli as
// hg_search_dev writes them, and the top_k-th key per query (0: fewer candidates) in d_floor_key; each may be NULL
int hg_launch_search_select(hg_ctx *ctx, const hg_hit *d_cand, uint64_t n_cand, uint32_t n_qry, uint32_t top_k, hg_hit *d_out,
                            uint32_t *d_n_found, uint32_t *d_milli, unsigned long long *d_floor_key);
// the floor pass's top_k-th keys (over s sample rows of n_ref) -> the main pass's per-query thresholds (hg_floors)
int hg_launch_search_floors(hg_ctx *ctx, const unsigned long long *d_floor_key, uint32_t n_qry, float ani_min, uint32_t ksize,
                            uint32_t n_ref, uint32_t s, hg_floor *d_floors, float *d_cfrac_row);
// n_lists (1..HG_SEARCH_MERGE_MAX_LISTS) per-block results -> one, as hg_search_merge_dev describes; *d_status |= 1 if some
// i + i0[m] does not fit 32 bits, |= 2 if some input n_found exceeds top_k (the caller zeroes it before)
int hg_launch_search_merge(hg_ctx *ctx, uint32_t n_lists, const hg_hit *d_in, const uint32_t *d_in_found, const uint32_t *i0,
                           uint32_t n_qry, uint32_t top_k, hg_hit *d_out, uint32_t *d_n_found, uint32_t *d_milli, uint32_t *d_status);
// ---- packed sketch rows from the host (api.cu), shared by the packed dist and search entries and their group forms ----

// One matrix of packed sketch rows in host memory, as the sketch file holds them: row g starts `stride` bytes after row
// g - 1, has hv_quant_bits bits[g] in 1..16 and bits[g] * hv_d / 8 live bytes.  max_bits: set by hg_packed_rows_check.
struct hg_packed_rows {
  const uint8_t *packed;
  uint64_t stride;
  const uint8_t *bits;
  const int32_t *norm;
  uint32_t n;
  uint32_t max_bits;
  uint64_t width(uint32_t hv_d) const { return (uint64_t)max_bits * hv_d / 8; }  // bytes of a row that can be live
  hg_packed_rows rows(uint32_t a, uint32_t m) const { return {packed + a * stride, stride, bits + a, norm + a, m, max_bits}; }
};
// The argument checks of a packed entry (`who` names it in the error): the pointers of a non-empty matrix, hv_d % 256
// and stride % 4.
int hg_packed_args_check(const char *who, const hg_packed_rows &R, const hg_packed_rows &Q, uint32_t hv_d);
// Every row's hv_quant_bits in 1..16 and the live width of each matrix within its stride; sets max_bits.  *same: ref and
// query are the same rows (same pointers and n); then Q becomes R.
int hg_packed_rows_check(const char *who, hg_packed_rows *R, hg_packed_rows *Q, uint32_t hv_d, bool *same);

// Host rows on their way to the device, and where they land.
struct HostRows {
  const uint8_t *base;  // first row on the host
  uint64_t stride;      // bytes between host rows
  uint64_t width;       // bytes of a row that travel (int16 rows: 2 hv_d; packed rows: max hv_quant_bits * hv_d / 8)
  const uint8_t *bits;  // packed rows: hv_quant_bits per row (host); int16 rows: NULL
  const int32_t *norm;  // host
  uint32_t n;
  uint8_t *d_stage;     // packed rows: where they land (width apart); int16 rows: the matrix itself
  uint8_t *d_bits;      // packed rows
  int16_t *d_hv;
  int32_t *d_norm;
};
// Device room for a ref block and a query block of packed rows (one block when `same`): int16 rows in HG_S_HV, each
// block 256-byte aligned; norms, then bits in HG_S_SMALL; packed bytes in HG_S_TABLES.
int hg_packed_stage(hg_ctx *ctx, const hg_packed_rows &R, const hg_packed_rows &Q, bool same, uint32_t hv_d, HostRows *hr,
                    HostRows *hq);
// One block of rows copied whole on ctx->stream (rows, norms, bits), packed rows unpacked to their int16 rows.
int hg_rows_to_device(hg_ctx *ctx, const HostRows &S, uint32_t hv_d);
// The output stage of n > 0 hits on the device: sorted into the reference's order if asked (ANI thousandths into
// ani_milli when it is not NULL), copied to the host; returns when the copies are complete.
int hg_hits_to_host(hg_ctx *ctx, hg_hit *d_hits, uint64_t n, bool sorted, hg_hit *hits, uint32_t *ani_milli);
// hg_dist_packed after its checks.
int hg_dist_packed_run(hg_ctx *ctx, const hg_packed_rows &R, const hg_packed_rows &Q, bool same, uint32_t hv_d, uint32_t ksize,
                       float ani_th, int symmetric, int path, bool sorted, hg_hit *hits, uint32_t *ani_milli, uint64_t cap,
                       uint64_t *n_hits);
// The search arguments of a search entry that do not describe rows: out / n_found, hv_d, top_k and path.
int hg_search_check(const char *who, uint32_t n_qry, const hg_hit *out, const uint32_t *n_found, uint32_t hv_d, uint32_t top_k,
                    int path);
// hg_search_packed after its argument checks (`who` names the entry that was called).
int hg_search_packed_host(hg_ctx *ctx, const char *who, hg_packed_rows R, hg_packed_rows Q, uint32_t hv_d, uint32_t ksize,
                          uint32_t top_k, float ani_min, int path, hg_hit *out, uint32_t *n_found, uint32_t *ani_milli);
// One search of checked packed rows whose result stays on the device (HG_S_TILES of the context).
int hg_search_packed_run(hg_ctx *ctx, const hg_packed_rows &R, const hg_packed_rows &Q, bool same, uint32_t hv_d, uint32_t ksize,
                         uint32_t top_k, float ani_min, int path, hg_hit **d_out, uint32_t **d_n_found, uint32_t **d_milli);
// hg_search_merge_dev after its argument checks (the context's device is current); returns with the result complete
int hg_search_merge(hg_ctx *ctx, uint32_t n_lists, const hg_hit *d_in, const uint32_t *d_in_found, const uint32_t *i0, uint32_t n_qry,
                    uint32_t top_k, hg_hit *d_out, uint32_t *d_n_found, uint32_t *d_milli);
int hg_launch_absmax(hg_ctx *ctx, const int16_t *d_hv, uint64_t n_elems, int32_t *d_out);

// ---- ANI clustering (cluster.cu, api.cu): union-find over a forest parent[0, n) with parent[x] <= x (DESIGN.md §4.9) ----
int hg_launch_cluster_iota(hg_ctx *ctx, uint32_t *d_parent, uint32_t n);
// unites (i, j) of the first min(*d_count, cap) records (d_count NULL: cap records; every index < n of the forest);
// d_stats (may be NULL): [0] += that number of records, [1] = max([1], it)
int hg_launch_cluster_hook(hg_ctx *ctx, uint32_t *d_parent, const hg_hit *d_edges, const unsigned long long *d_count, uint64_t cap,
                           unsigned long long *d_stats);
// unites (x, d_other[x]) for every x < n; d_other is a forest over at least those n nodes
int hg_launch_cluster_hook_labels(hg_ctx *ctx, uint32_t *d_parent, const uint32_t *d_other, uint32_t n);
// after every hook: d_parent[x] = the root of x for every x < n, *d_n_roots += the number of roots (the caller zeroes it)
int hg_launch_cluster_flatten(hg_ctx *ctx, uint32_t *d_parent, uint32_t n, uint32_t *d_n_roots);
// *d_status |= 1 if some edge index is >= n, |= 2 if some d_parent[x] > x (the caller zeroes it)
int hg_launch_cluster_check(hg_ctx *ctx, const uint32_t *d_parent, uint32_t n, const hg_hit *d_edges, uint64_t n_edges,
                            uint32_t *d_status);
// The arguments of a cluster entry that do not describe rows (`who` names it): rep, hv_d, ani_th and path.
int hg_cluster_check(const char *who, uint32_t n, const uint32_t *rep, uint32_t hv_d, float ani_th, int path);
// hg_cluster_packed after its argument checks (`who` names the entry that was called).
int hg_cluster_packed_host(hg_ctx *ctx, const char *who, hg_packed_rows R, uint32_t hv_d, uint32_t ksize, float ani_th, int path,
                           uint32_t *rep, uint32_t *n_clusters);
// One cluster run over checked packed rows R: the pairs whose column is in [col0, R.n), as a flattened forest over the
// R.n rows in HG_S_TILES of the context (*d_rep); rep and n_clusters as hg_cluster_finish.
int hg_cluster_packed_run(hg_ctx *ctx, const hg_packed_rows &R, uint32_t col0, uint32_t hv_d, uint32_t ksize, float ani_th, int path,
                          uint32_t **d_rep, uint32_t *rep, uint32_t *n_clusters);
// Flattens the forest d_rep[0, n) and counts its roots; rep (host, may be NULL) receives the labels and n_clusters (may be
// NULL) the count; `flattened` (may be NULL) is recorded behind the flatten.  Returns with all of it complete.
int hg_cluster_finish(hg_ctx *ctx, uint32_t *d_rep, uint32_t n, uint32_t *rep, uint32_t *n_clusters, cudaEvent_t flattened = nullptr);
void hg_cluster_stats_reset(hg_ctx *ctx);

// ---- greedy ANI dereplication (derep.cu, api.cu): DESIGN.md §4.10 ----
// The widest column chunk of the representative phase: one greedy step per chunk, w x w bits of adjacency (128 KB)
constexpr uint32_t HG_DEREP_CHUNK = 1024;
// row t of d_dst (and its norm) = row d_idx[t] of d_src, for t < m (hv_d % 256 == 0)
int hg_launch_derep_gather(hg_ctx *ctx, const int16_t *d_src, const int32_t *d_src_norm, const uint32_t *d_idx, uint32_t m,
                           uint32_t hv_d, int16_t *d_dst, int32_t *d_dst_norm);
// the first min(*d_count, cap) edges of a window of column chunk [a, a + w): covered[j - a] = 1 for an edge from an earlier
// representative i < a; bit i - a of bitmap row j - a for i >= a.  d_linked (may be NULL) += that number of edges
int hg_launch_derep_mark(hg_ctx *ctx, const hg_hit *d_edges, const unsigned long long *d_count, uint64_t cap, uint32_t a, uint32_t w,
                         const uint8_t *d_is_rep, uint8_t *d_covered, uint32_t *d_adj, unsigned long long *d_linked);
// the greedy step of chunk [a, a + w), w <= HG_DEREP_CHUNK, after its last window's marks: is_rep[a, a + w), the chunk's
// representatives appended to d_rep_list (ascending) and counted in *d_n_reps; covered and the bitmap cleared
int hg_launch_derep_greedy(hg_ctx *ctx, uint32_t a, uint32_t w, uint8_t *d_covered, uint32_t *d_adj, uint8_t *d_is_rep,
                           uint32_t *d_rep_list, uint32_t *d_n_reps);
// d_rep[order[t]] = order[t's representative] from is_rep, the rep list and a top-1 search result (d_out, d_n_found) of
// every row against the rep matrix (d_order NULL: the identity); *d_status |= 1 if a non-representative found none
int hg_launch_derep_finalize(hg_ctx *ctx, const uint8_t *d_is_rep, const uint32_t *d_rep_list, const hg_hit *d_out,
                             const uint32_t *d_n_found, const uint32_t *d_order, uint32_t n, uint32_t *d_rep, uint32_t *d_status);

// ---- the all-vs-all ANI matrix (api.cu, matrix.cu): DESIGN.md §4.11 ----
// cells of a matrix run: n_ref x n_qry, or n_ref (n_ref - 1) / 2 in lower mode
uint64_t hg_matrix_entries(uint32_t n_ref, uint32_t n_qry, int lower);
// The arguments of a matrix entry that do not describe rows (`who` names it): hv_d, path, lower (and `same` rows for it),
// ld >= n_qry for a rectangle, out when there is something to write.
int hg_matrix_check(const char *who, bool same, uint32_t n_ref, uint32_t n_qry, uint32_t hv_d, int path, int lower, const void *out,
                    uint64_t ld);
// A host output buffer page-locked for the call: kept as it is when it already is (hg_host_alloc, registered), else
// registered (portable: every context's copies see it) and unregistered when this goes out of scope.
struct HostPin {
  void *ptr = nullptr;
  int pin(void *p, uint64_t bytes);
  ~HostPin();
};
// The matrix cells of checked packed rows: ref rows [first, R.n) against Q (lower: R == Q, the strict lower triangle),
// into the page-locked host matrix `out`, which holds row `first` at offset 0 (rectangle: rows ld apart).
int hg_matrix_packed_run(hg_ctx *ctx, const hg_packed_rows &R, const hg_packed_rows &Q, bool same, uint32_t hv_d, uint32_t ksize, int path,
                         bool lower, uint32_t first, float *out, uint64_t ld);
