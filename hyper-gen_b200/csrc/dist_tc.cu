// dist_tc.cu — tensor-pipe dist path: every ref x query dot product as an exact integer
// contraction on tcgen05 (kind::i8, s32 accumulators in TMEM) fed by TMA, with the ANI /
// threshold epilogue fused behind it.
//
// Replaces the pair loop of dist::compute_hv_ani + compute_pairwise_ani (reference
// src/dist.rs:139-161,231-294).  Sketch HV elements need 9-11 bits at the BASELINE configs
// (SURVEY.md F5), which does not fit the s8 MMA input type, so every i16 value is split into
// two s8 limbs
//        x = 128 * h + l,   l = ((x + 64) mod 128) - 64 in [-64, 63],   h = (x - l) / 128
// (exact for |x| <= 8127, i.e. hv_quant_bits <= 13; wider inputs take the SIMT path), and
//        r . q = 2^14 (Hr.Hq) + 2^7 (Hr.Lq + Lr.Hq) + (Lr.Lq)
// is accumulated as three s32 accumulators (the two cross products share one), each < 2^31
// for D <= 32768.  The recombination wraps in i32 exactly like the reference's i32 sum.
//
// Kernel (dist_tc2_kernel): persistent CTA PAIRS (cluster 2 x 1, tcgen05 cta_group::2), one pair
// per TPC, each walking 256 x 128 output tiles.  Per k-block a CTA TMA-loads its own 128 ref rows and
// only HALF of the query tile (64 rows) - 48 KB instead of 64 KB for the same MMA work - because the
// pair's MMA reads the query half of both CTAs; the kernel is bound by operand bytes arriving per SM
// (L2 -> SM, ~37 B/clk/SM measured), so this is where the time goes.  10 warps per CTA: warp 0 issues
// TMA (128B-swizzled, K-major boxes) through a 4-stage mbarrier ring and runs ahead into the next
// tile while the epilogue drains, one thread of the leader CTA's warp 1 issues the tcgen05.mma stream
// (M = 256) and multicasts the stage releases to both CTAs, warps 2-9 of each CTA drain their three
// TMEM accumulators with tcgen05.ld, apply a division-free bound and run the shared exact epilogue
// (dist_common.cuh) only where a pair can reach the threshold.  The K loop always runs whole trips of the
// stage ring: when hv_d is not a multiple of 512 the tensor maps' zero fill supplies the missing columns.
#include <cuda.h>

#include <algorithm>

#include "dist_common.cuh"
#include "tc_ptx.cuh"

namespace {

using namespace hgtc;

constexpr int TC_BN = 128;
constexpr int TC_EPI_WARPS = 8;                      // two per TMEM lane quarter, half the columns each
constexpr int TC_THREADS = 64 + 32 * TC_EPI_WARPS;  // producer, MMA issuer, epilogue warps (+ 32 per pusher warp of a multi-GPU member)
constexpr int TC_PUSH_WARPS = 2;
constexpr uint32_t TC_TMEM_COLS = 512;

// ---- epilogue pieces --------------------------------------------------------------------------
// Cheap per-element test first: ani >= ani_th implies dot >= cfrac * (norm_r + norm_q)
// (dist_common.cuh), split into a per-row and a per-column integer so that an element costs
// two shift-adds, one add and one compare.  Only lanes that pass run the exact f32 ANI sequence
// and the compacted append.

// per-column bound of query column lj (INT32_MIN = always take the exact path).  QF (a search pass): the column's own
// cfrac, and the launch's smallest positive one for the rows (hg_floors).  The bound holds only while nothing of the
// pair wraps i32: a row whose true norm (qry_sq / ref_sq, 64 bits) reaches HG_NORM_WRAP_CUT is always a candidate.
template <bool QF>
__device__ __forceinline__ int32_t tc_col_bound(const hg::DistEpilogue &ep, const hg_floors &fl, const unsigned long long *qry_sq, uint32_t lj) {
  float cfrac = ep.cfrac;
  if constexpr (QF) cfrac = lj < ep.n_qry ? fl.q[lj].cfrac : 0.0f;
  if (!(cfrac > 0.0f) || lj >= ep.n_qry || qry_sq[lj] >= HG_NORM_WRAP_CUT) return INT32_MIN;
  const int32_t nq = ep.qry_norm[lj];
  return nq > 0 ? __float2int_rd(cfrac * __int2float_rz(nq)) - 1 : INT32_MIN;
}
template <bool QF>
__device__ __forceinline__ int32_t tc_row_bound(const hg::DistEpilogue &ep, const hg_floors &fl, const unsigned long long *ref_sq, uint32_t li) {
  float cfrac = ep.cfrac;
  if constexpr (QF) cfrac = *fl.cfrac_row;
  if (!(cfrac > 0.0f) || li >= ep.n_ref || ref_sq[li] >= HG_NORM_WRAP_CUT) return INT32_MIN / 2;
  const int32_t nr = ep.ref_norm[li];
  return nr > 0 ? __float2int_rd(cfrac * __int2float_rz(nr)) - 1 : INT32_MIN / 2;
}

// Candidates are not evaluated while the accumulators are being drained: each epilogue warp parks
// them (row, column, exact dot) in its own shared-memory list and runs the exact f32 ANI + append
// (dist_common.cuh) over the list afterwards, 32 candidates per round.  That second phase starts
// after TMEM has been handed back, so it overlaps the next tile's MMAs;
// it also balances the lanes (hits cluster on a few rows of the diagonal tiles).
constexpr int TC_LIST_CAP = 256;  // candidates per warp list (8 B each); a full list is evaluated in place

// pass 1: exact f32 ANI of every parked candidate; ONE atomic reserves room for the survivors (the counter may sit on
// another GPU); pass 2 writes the records
template <bool QF>
__device__ __forceinline__ void tc_process(const hg::DistEpilogue &ep, const hg_floors &fl, uint2 *list, float *anis, uint32_t n,
                                           uint32_t row0, uint32_t col0) {
  if (n == 0) return;
  const uint32_t lane = threadIdx.x & 31;
  uint32_t mine = 0;
  for (uint32_t e = lane; e < n; e += 32) {
    const uint2 c = list[e];
    const uint32_t li = row0 + (c.x >> 8), lj = col0 + (c.x & 255u);
    float ani = 0.0f;
    const bool keep = hg::dist_eval<QF>(ep, li < ep.n_ref && lj < ep.n_qry, li, lj, (int32_t)c.y, &ani, fl);
    if (keep) list[e].x = c.x | 0x80000000u;
    anis[e] = ani;
    mine += keep;
  }
  uint32_t inc = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= (uint32_t)o) inc += y;
  }
  const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
  if (total == 0) { __syncwarp(); return; }
  unsigned long long base = 0;
  if (lane == 0) base = atomicAdd(ep.n_hits, (unsigned long long)total);
  base = __shfl_sync(0xffffffffu, base, 0);
  // consecutive lanes write consecutive records: whole 64-byte+ bursts when the list may live in host memory behind PCIe
  for (uint32_t e0 = 0; e0 < n; e0 += 32) {
    const uint32_t e = e0 + lane;
    const uint2 c = e < n ? list[e] : make_uint2(0u, 0u);
    const bool keep = (c.x & 0x80000000u) != 0u;
    const uint32_t bal = __ballot_sync(0xffffffffu, keep);
    if (keep) {
      const unsigned long long idx = base + __popc(bal & ((1u << lane) - 1u));
      if (idx < ep.cap) {
        hg_hit h;
        h.i = ep.i0 + row0 + ((c.x & 0x7FFFFFFFu) >> 8);
        h.j = ep.j0 + col0 + (c.x & 255u);
        h.dot = (int32_t)c.y;
        h.ani = anis[e];
        ep.hits[idx] = h;
      }
    }
    base += __popc(bal);
  }
  __syncwarp();
}

// One epilogue warp drains columns [c_begin, c_end) of its 32 TMEM lanes (three accumulators at
// column offsets 0, BN, 2 BN from taddr): row `rowl` of the tile per lane, query columns col0 + c.
// Appends the candidates to list[0..n_list); returns the new n_list.
template <bool QF>
__device__ __forceinline__ uint32_t tc_drain(const hg::DistEpilogue &ep, const hg_floors &fl, uint32_t taddr, int c_begin, int c_end,
                                             const int32_t *s_tq, int32_t tr, bool row_live, uint32_t rowl, uint32_t row0,
                                             uint32_t col0, uint2 *list, float *anis, uint32_t n_list) {
  const uint32_t lane = threadIdx.x & 31;
  // software pipelined: the loads of chunk c + 16 are in flight while chunk c is tested
  uint32_t nh[16], nc[16], nl[16];
  tmem_ld16(taddr + 0 * TC_BN + c_begin, nh);
  tmem_ld16(taddr + 1 * TC_BN + c_begin, nc);
  tmem_ld16(taddr + 2 * TC_BN + c_begin, nl);
#pragma unroll 1
  for (int c = c_begin; c < c_end; c += 16) {
    uint32_t hh[16], cr[16], ll[16];
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    tmem_ld_fence(nh);
    tmem_ld_fence(nc);
    tmem_ld_fence(nl);
#pragma unroll
    for (int j = 0; j < 16; ++j) { hh[j] = nh[j]; cr[j] = nc[j]; ll[j] = nl[j]; }
    if (c + 16 < c_end) {
      tmem_ld16(taddr + 0 * TC_BN + c + 16, nh);
      tmem_ld16(taddr + 1 * TC_BN + c + 16, nc);
      tmem_ld16(taddr + 2 * TC_BN + c + 16, nl);
    }
    int32_t dot[16];
    uint32_t cand = 0;  // bit j: column c + j of my row can reach the threshold
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      dot[j] = (int32_t)((((hh[j] << 7) + cr[j]) << 7) + ll[j]);  // wrapping i32, as dist.rs:147-151
      const int32_t tq = s_tq[c + j];
      // tq = INT32_MIN or tr = INT32_MIN / 2 (bound off / degenerate norm) always qualify
      const bool cj = dot[j] >= (int32_t)((uint32_t)tr + (uint32_t)tq) || tq == INT32_MIN || tr == INT32_MIN / 2;
      cand |= (uint32_t)cj << j;
    }
    if (!row_live) cand = 0;
    if (!__any_sync(0xffffffffu, cand != 0)) continue;  // the common case
#pragma unroll
    for (int h = 0; h < 2; ++h) {  // 8 columns at a time: at most 256 candidates, always fits an empty list
      const uint32_t m = (cand >> (8 * h)) & 255u;
      const uint32_t cnt = __popc(m);
      uint32_t inc = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (uint32_t)o) inc += y;
      }
      const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
      if (total == 0) continue;
      if (n_list + total > TC_LIST_CAP) {  // evaluate what is parked (slow path: TMEM stays held)
        tc_process<QF>(ep, fl, list, anis, n_list, row0, col0);
        n_list = 0;
      }
      uint32_t pos = n_list + inc - cnt;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if ((m >> j) & 1u) list[pos++] = make_uint2((rowl << 8) | (uint32_t)(c + 8 * h + j), (uint32_t)dot[8 * h + j]);
      n_list += total;
      __syncwarp();
    }
  }
  return n_list;
}

// Dense mode (hg_dense): the same drain without the bound, the exact dot of each of my 16 columns stored to its cell.
__device__ __forceinline__ void tc_drain_dense(const hg::DistEpilogue &ep, const hg_dense &dn, uint32_t taddr, int c_begin, int c_end,
                                               bool row_live, uint32_t gi, uint32_t gj0) {
  uint32_t nh[16], nc[16], nl[16];
  tmem_ld16(taddr + 0 * TC_BN + c_begin, nh);
  tmem_ld16(taddr + 1 * TC_BN + c_begin, nc);
  tmem_ld16(taddr + 2 * TC_BN + c_begin, nl);
#pragma unroll 1
  for (int c = c_begin; c < c_end; c += 16) {
    uint32_t hh[16], cr[16], ll[16];
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    tmem_ld_fence(nh);
    tmem_ld_fence(nc);
    tmem_ld_fence(nl);
#pragma unroll
    for (int j = 0; j < 16; ++j) { hh[j] = nh[j]; cr[j] = nc[j]; ll[j] = nl[j]; }
    if (c + 16 < c_end) {
      tmem_ld16(taddr + 0 * TC_BN + c + 16, nh);
      tmem_ld16(taddr + 1 * TC_BN + c + 16, nc);
      tmem_ld16(taddr + 2 * TC_BN + c + 16, nl);
    }
    int32_t dot[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) dot[j] = (int32_t)((((hh[j] << 7) + cr[j]) << 7) + ll[j]);  // wrapping i32, as dist.rs:147-151
    const uint32_t n = row_live ? hg::dense_live(dn, ep, gi, gj0 + c) : 0u;
    if (n) hg::dense_store16(dn, gi, gj0 + c, n, dot);
  }
}

// ---- the kernel: persistent CTA pairs, cta_group::2, 256 x 128 tiles ---------------------------
constexpr int T2_STAGES = 4;
constexpr int T2_A_BYTES = 128 * TC_BK;               // my 128 ref rows, one limb plane
constexpr int T2_B_BYTES = 64 * TC_BK;                // my half of the 128 query rows, one limb plane
constexpr int T2_STAGE_BYTES = 2 * T2_A_BYTES + 2 * T2_B_BYTES;  // 48 KB
constexpr int T2_SMEM_BYTES = T2_STAGES * T2_STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/ + 1024 /*col bounds x 2*/ +
                              8 * 256 * 8 /*candidate lists*/ + 8 * 256 * 4 /*their ANIs*/;
// instruction descriptor, kind::i8: D = s32, A = B = signed 8-bit, both K-major, M = 256 (the pair's rows), N = 128
constexpr uint32_t T2_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((TC_BN >> 3) << 17) | ((256u >> 4) << 24);


// The pair's walk over the non-empty 256 x 128 tiles, row-block major.  Symmetric: tile (R, C) is
// empty when its largest global j is not above its smallest global i, which leaves columns
// C >= cmin(R) in row-block R.
struct PairTiles {
  uint32_t gx, gy2, R, C;
  int64_t delta;  // i0 - j0
  int sym;
  const uint2 *list;  // multi-GPU member: its tiles in the order the host chose (hg_tile_feed); NULL: the arithmetic walk below
  uint32_t n_list, cur, need;
  __device__ uint32_t cmin(uint32_t r) const {
    if (!sym) return 0;
    const int64_t v = delta + 256ll * (int64_t)r + 1;
    if (v <= 0) return 0;
    const uint64_t c = (uint64_t)v / 128u;
    return c > gx ? gx : (uint32_t)c;
  }
  __device__ void init(const hg::DistEpilogue &ep, const hg_tile_feed &f) {
    list = f.list;
    n_list = f.n_list;
    cur = 0;
    need = 0;
    gx = (ep.n_qry + TC_BN - 1) / TC_BN;
    gy2 = (ep.n_ref + 255) / 256;
    delta = (int64_t)ep.i0 - (int64_t)ep.j0;
    sym = ep.symmetric;
    R = 0;
    C = cmin(0);
  }
  __device__ bool advance(uint32_t k) {  // k non-empty tiles forward; false past the end
    if (list) {
      cur += k;
      if (cur >= n_list) return false;
      const uint2 e = list[cur];
      R = e.x & 0xFFFFu;
      C = e.x >> 16;
      need = e.y;
      return true;
    }
    while (R < gy2) {
      const uint32_t avail = gx - C;
      if (k < avail) { C += k; return true; }
      k -= avail;
      ++R;
      C = cmin(R);
    }
    return false;
  }
};

// QF: per-query thresholds (a search pass, PUSHW = 0 only); `fl` is not read otherwise.  DENSE (PUSHW = 0, no QF): every
// live pair's dot to its cell of `dn` (hg_dense) instead of the bound, the exact epilogue and the append.
template <int PUSHW, bool QF, bool DENSE>
__device__ __forceinline__ void tc2_body(const CUtensorMap &tm_ref, const CUtensorMap &tm_qry, uint32_t ref_plane_rows, uint32_t ref_row_base,
                                         uint32_t qry_plane_rows, uint32_t qry_row_base, uint32_t k_len, const hg::DistEpilogue &ep,
                                         const unsigned long long *ref_sq, const unsigned long long *qry_sq,
                                         uint32_t walk_mul, uint32_t walk_add, hg_tile_feed feed, const hg_push_plan &plan,
                                         const hg_floors &fl, const hg_dense &dn) {
  uint32_t rank;  // 0 = leader (issues the MMAs, owns the full / tmem-empty barriers), 1 = peer
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
  if (feed.seq_ptr) feed.seq = *feed.seq_ptr;
  if (blockIdx.x == 0 && threadIdx.x == 0) hg::feed_stamp(feed.dbg, 1);
  // this launch takes tiles walk_add, walk_add + walk_mul, ... of the enumeration (member walk_add of walk_mul GPUs),
  // dealt round-robin to its CTA pairs
  const uint32_t pair = (blockIdx.x >> 1) * walk_mul + walk_add, n_pairs = (gridDim.x >> 1) * walk_mul;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *aligned = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t bar_base = base + T2_STAGES * T2_STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };                  // used in the leader only
  auto empty_bar = [&](int s) { return bar_base + 8u * (T2_STAGES + s); };   // one per CTA, signalled by multicast commit
  const uint32_t accum_bar = bar_base + 8u * (2 * T2_STAGES);                // one per CTA, multicast commit
  const uint32_t tmem_empty_bar = bar_base + 8u * (2 * T2_STAGES + 1);       // leader only: both epilogues drained
  volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(aligned + T2_STAGES * T2_STAGE_BYTES + 8 * (2 * T2_STAGES + 2));
  int32_t *s_tq_all = reinterpret_cast<int32_t *>(aligned + T2_STAGES * T2_STAGE_BYTES + 256);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < T2_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    mbar_init(accum_bar, 1);
    mbar_init(tmem_empty_bar, 2 * TC_EPI_WARPS);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {  // the same warp in both CTAs
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void *)tmem_slot)),
                 "r"(TC_TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  cluster_sync_all();  // the peer's barriers are initialised before anyone signals them
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t num_kb = k_len / TC_BK;

  if (PUSHW > 0 && warp >= TC_THREADS / 32) {
    // ===== pusher warps (a member of several GPUs): my limb-plane rows to the windows of the members that compute with them, unit by unit =====
    hg::push_my_units(&plan, blockIdx.x * PUSHW + (uint32_t)(warp - TC_THREADS / 32), gridDim.x * PUSHW);
  } else {
  PairTiles tiles;
  tiles.init(ep, feed);
  bool valid = tiles.advance(pair);
  uint32_t have = 0;  // arrival flags seen so far (the producer warp)
  if (feed.start_need) {  // a member of several GPUs: nothing is appended before the root has reset its hit counter
    if (warp == 0) hg::feed_wait_start(feed);
    if (warp == 0 && blockIdx.x == 0 && lane == 0) hg::feed_stamp(feed.dbg, 2);
    asm volatile("bar.sync 2, %0;" ::"r"(TC_THREADS) : "memory");
  }

  if (warp == 0) {
    // ===== TMA producer (both CTAs; completion bytes go to the LEADER's full barrier) =====
    {
      const uint32_t on = elect_one();
      uint32_t it = 0;
      unsigned long long waited = 0;  // (timeline) ns this producer spent waiting for other members' rows
      for (; valid; valid = tiles.advance(n_pairs)) {
        const uint32_t row0 = tiles.R * 256u + rank * 128u, colh = tiles.C * TC_BN + rank * 64u;
        if (tiles.need) {  // the rows this tile reads have arrived from their owners
          const unsigned long long w0 = feed.dbg ? hg::feed_ns() : 0ull;
          hg::feed_wait(feed, tiles.need, have);
          if (feed.dbg) waited += hg::feed_ns() - w0;
        }
        for (uint32_t kb = 0; kb < num_kb; ++kb, ++it) {
          const int s = it % T2_STAGES;
          const uint32_t ph = (it / T2_STAGES) & 1u;
          mbar_wait_cluster(empty_bar(s), ph ^ 1u);
          mbar_expect_tx(full_bar(s), 2 * T2_STAGE_BYTES, rank == 0 ? on : 0u);  // the leader expects its bytes and the peer's
          const uint32_t fb = mapa_u32(full_bar(s), 0);
          const uint32_t st = base + s * T2_STAGE_BYTES;
          const int k0 = (int)(kb * TC_BK);
          tma_load_2d_pair(st, &tm_ref, fb, k0, (int)(ref_row_base + row0), on);                                  // ref hi
          tma_load_2d_pair(st + T2_A_BYTES, &tm_ref, fb, k0, (int)(ref_plane_rows + ref_row_base + row0), on);    // ref lo
          tma_load_2d_pair(st + 2 * T2_A_BYTES, &tm_qry, fb, k0, (int)(qry_row_base + colh), on);                 // qry hi, my half
          tma_load_2d_pair(st + 2 * T2_A_BYTES + T2_B_BYTES, &tm_qry, fb, k0, (int)(qry_plane_rows + qry_row_base + colh), on);  // qry lo
        }
      }
      if (feed.dbg && lane == 0) { atomicMax(feed.dbg + 5, waited); if (blockIdx.x == 0) feed.dbg[3] = waited; }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: one thread of the leader CTA drives both SMs' tensor cores =====
    if (rank == 0) {
      const uint32_t on = elect_one();
      const uint32_t d0 = umma_desc_lo(base);
      uint32_t it = 0, tile_n = 0;  // it: full trips around the stage ring
      for (; valid; valid = tiles.advance(n_pairs), ++tile_n) {
        if (tile_n) {  // both epilogues have drained the previous tile's accumulators
          mbar_wait_cluster(tmem_empty_bar, (tile_n - 1) & 1u);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        // num_kb is a multiple of T2_STAGES (k_len is), so every tile starts at stage 0 and the ring is
        // walked with a compile-time stage index: every descriptor is d0 + constant
        for (uint32_t kb0 = 0; kb0 < num_kb; kb0 += T2_STAGES, ++it) {
          const uint32_t ph = it & 1u;
#pragma unroll
          for (int s = 0; s < T2_STAGES; ++s) {
            mbar_wait(full_bar(s), ph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int ks = 0; ks < TC_BK / 32; ++ks) {
              const uint32_t off = (uint32_t)(s * T2_STAGE_BYTES + 32 * ks) >> 4;
              const uint32_t a_hi = d0 + off, a_lo = a_hi + (T2_A_BYTES >> 4);
              const uint32_t b_hi = a_hi + (2 * T2_A_BYTES >> 4), b_lo = a_hi + ((2 * T2_A_BYTES + T2_B_BYTES) >> 4);
              const uint32_t acc = (kb0 | (uint32_t)s | (uint32_t)ks) != 0u;
              umma_i8_pair(tmem_base + 0 * TC_BN, a_hi, b_hi, T2_IDESC, acc, on);  // Hr.Hq
              umma_i8_pair(tmem_base + 1 * TC_BN, a_hi, b_lo, T2_IDESC, acc, on);  // Hr.Lq
              umma_i8_pair(tmem_base + 1 * TC_BN, a_lo, b_hi, T2_IDESC, 1u, on);   //   + Lr.Hq
              umma_i8_pair(tmem_base + 2 * TC_BN, a_lo, b_lo, T2_IDESC, acc, on);  // Lr.Lq
            }
            umma_commit_pair(empty_bar(s), on);  // the stage is free in both CTAs once these MMAs have read it
          }
        }
        umma_commit_pair(accum_bar, on);       // accumulators final: wake both epilogues
      }
    }
  } else {
    // ===== epilogue (both CTAs, each its own 128 rows) =====
    const int ew = warp - 2;
    const uint32_t q = warp & 3;
    const int half = (ew >> 2);
    const uint32_t te = mapa_u32(tmem_empty_bar, 0);
    uint2 *list = reinterpret_cast<uint2 *>(aligned + T2_STAGES * T2_STAGE_BYTES + 256 + 1024) + ew * TC_LIST_CAP;
    float *anis = reinterpret_cast<float *>(aligned + T2_STAGES * T2_STAGE_BYTES + 256 + 1024 + TC_EPI_WARPS * TC_LIST_CAP * 8) + ew * TC_LIST_CAP;
    uint32_t tile_n = 0, have_e = 0, have_l = 0;
    volatile uint32_t *s_early = reinterpret_cast<volatile uint32_t *>(aligned + T2_STAGES * T2_STAGE_BYTES + 240);
    for (; valid; valid = tiles.advance(n_pairs), ++tile_n) {
      const uint32_t row0 = tiles.R * 256u + rank * 128u, col0 = tiles.C * TC_BN;
      // The bounds below read the norms of this tile's rows / columns before the accumulators are waited for - in a
      // multi-GPU launch possibly before those rows have arrived.  One epilogue warp looks at the arrival flags (no
      // spinning here: the producer does the waiting) and all eight take the same route: bounds now, or after the
      // accumulator barrier, by when the producer has seen the flags.
      bool early = true;
      if (tiles.need) {
        if (ew == 0) {
          const bool ok = hg::feed_poll(feed, tiles.need, have_e);
          if (lane == 0) *s_early = ok ? 1u : 0u;
        }
        asm volatile("bar.sync 1, %0;" ::"r"(32 * TC_EPI_WARPS) : "memory");
        early = *s_early != 0u;
      }
      int32_t *s_tq = s_tq_all + (tile_n & 1u) * TC_BN;  // double buffered: one barrier per tile is enough
      const uint32_t li = row0 + q * 32 + lane;
      int32_t tr = 0;
      auto bounds = [&]() {
        const int t = threadIdx.x - 64;
        if (t < TC_BN) s_tq[t] = tc_col_bound<QF>(ep, fl, qry_sq, col0 + t);
        asm volatile("bar.sync 1, %0;" ::"r"(32 * TC_EPI_WARPS) : "memory");
        tr = tc_row_bound<QF>(ep, fl, ref_sq, li);
      };
      if (!DENSE && early) bounds();
      // my 128 x 128 part of the tile may be empty (below the diagonal, or past the last ref row)
      const bool mine_empty = row0 >= ep.n_ref || (ep.symmetric && (uint64_t)ep.j0 + col0 + TC_BN - 1 <= (uint64_t)ep.i0 + row0);
      mbar_wait_cluster(accum_bar, tile_n & 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (!early) {  // the producer has seen this tile's arrival flags; so do we now (an acquire, returns at once)
        hg::feed_wait(feed, tiles.need, have_l);
        if (!DENSE) bounds();
      }
      uint32_t n_list = 0;
      if constexpr (DENSE) {
        if (!mine_empty)
          tc_drain_dense(ep, dn, tmem_base + ((q * 32u) << 16), half * (TC_BN / 2), (half + 1) * (TC_BN / 2), li < ep.n_ref, ep.i0 + li,
                         ep.j0 + col0);
      } else if (!mine_empty) {
        n_list = tc_drain<QF>(ep, fl, tmem_base + ((q * 32u) << 16), half * (TC_BN / 2), (half + 1) * (TC_BN / 2), s_tq, tr,
                          li < ep.n_ref, q * 32 + lane, row0, col0, list, anis, 0u);
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(te);  // this warp's TMEM reads are done: the next tile's MMAs may start
      tc_process<QF>(ep, fl, list, anis, n_list, row0, col0);  // exact ANI + append, under the next tile's mainloop
    }
  }
  }  // compute roles
  __syncthreads();
  if (threadIdx.x == 0) hg::feed_stamp_max(feed.dbg, 4);
  cluster_sync_all();  // nobody leaves while the peer may still read its smem or signal its barriers
  if (warp == 2) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TC_TMEM_COLS) : "memory");
  }
}

template <int PUSHW, bool QF = false>
__global__ void __launch_bounds__(TC_THREADS + 32 * PUSHW, 1)
dist_tc2_kernel(const __grid_constant__ CUtensorMap tm_ref, const __grid_constant__ CUtensorMap tm_qry,
                uint32_t ref_plane_rows, uint32_t ref_row_base, uint32_t qry_plane_rows, uint32_t qry_row_base, uint32_t k_len,
                hg::DistEpilogue ep, const unsigned long long *__restrict__ ref_sq, const unsigned long long *__restrict__ qry_sq,
                uint32_t walk_mul, uint32_t walk_add, hg_tile_feed feed, const __grid_constant__ hg_push_plan plan, hg_floors fl) {
  tc2_body<PUSHW, QF, false>(tm_ref, tm_qry, ref_plane_rows, ref_row_base, qry_plane_rows, qry_row_base, k_len, ep, ref_sq, qry_sq, walk_mul,
                             walk_add, feed, plan, fl, hg_dense{});
}

__global__ void __launch_bounds__(TC_THREADS, 1)
dist_tc2_dense_kernel(const __grid_constant__ CUtensorMap tm_ref, const __grid_constant__ CUtensorMap tm_qry,
                      uint32_t ref_plane_rows, uint32_t ref_row_base, uint32_t qry_plane_rows, uint32_t qry_row_base, uint32_t k_len,
                      hg::DistEpilogue ep, uint32_t walk_mul, uint32_t walk_add, hg_tile_feed feed,
                      const __grid_constant__ hg_push_plan plan, hg_dense dn) {
  tc2_body<0, false, true>(tm_ref, tm_qry, ref_plane_rows, ref_row_base, qry_plane_rows, qry_row_base, k_len, ep, nullptr, nullptr, walk_mul,
                           walk_add, feed, plan, hg_floors{}, dn);
}

// i16 -> two s8 limb planes: plane 0 = h, plane 1 = l, `plane_stride` bytes apart; `out` points at the first element
// of plane 0 that belongs to `hv`.  Also adds every row's sum x^2 into sq[row] (zeroed before): 16 consecutive lanes
// cover 128 elements, which lie in one row (hv_d % 128 == 0), and add them with one atomic.
__global__ void split_limbs_kernel(const int16_t *__restrict__ hv, uint64_t n_elems, int8_t *__restrict__ out, uint64_t plane_stride,
                                   uint32_t hv_d, unsigned long long *__restrict__ sq) {
  const uint64_t n8 = n_elems / 8;  // a multiple of 16, and so is the stride: a half-warp is in or out of the loop together
  const uint32_t lane = threadIdx.x & 31, half = 0xFFFFu << (lane & 16);
  const uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (uint64_t)gridDim.x * blockDim.x;
  // row / column of element 8 i, advanced by the stride without a division per step
  uint64_t row = i0 * 8 / hv_d;
  uint32_t col = (uint32_t)(i0 * 8 - row * hv_d);
  const uint64_t drow = stride * 8 / hv_d;
  const uint32_t dcol = (uint32_t)(stride * 8 - drow * hv_d);
  for (uint64_t i = i0; i < n8; i += stride) {
    const uint4 v = reinterpret_cast<const uint4 *>(hv)[i];
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t hi[2] = {0, 0}, lo[2] = {0, 0};
    unsigned long long s = 0;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int x = (int)(int16_t)(w[e >> 1] >> (16 * (e & 1)));
      const int l = ((x + 64) & 127) - 64;
      const int h = (x - l) >> 7;
      hi[e >> 2] |= (uint32_t)(h & 0xFF) << (8 * (e & 3));
      lo[e >> 2] |= (uint32_t)(l & 0xFF) << (8 * (e & 3));
      s += (uint32_t)(x * x);
    }
    reinterpret_cast<uint2 *>(out)[i] = make_uint2(hi[0], hi[1]);
    reinterpret_cast<uint2 *>(out + plane_stride)[i] = make_uint2(lo[0], lo[1]);
#pragma unroll
    for (int o = 8; o; o >>= 1) s += __shfl_xor_sync(half, s, o);
    if ((lane & 15) == 0) atomicAdd(sq + row, s);
    row += drow;
    col += dcol;
    if (col >= hv_d) { col -= hv_d; ++row; }
  }
}

__global__ void tc_flags_kernel(const unsigned long long *__restrict__ sq, uint32_t n, uint32_t *__restrict__ flags) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flags[i] = sq[i] >= HG_NORM_WRAP_CUT;
}

}  // namespace

void hg_tc_tile_shape(uint32_t *rows, uint32_t *cols) { *rows = 256; *cols = TC_BN; }

static int tc_attrs(hg_ctx *ctx) {
  if (!ctx->tc_attr_set) {
    HG_CUDA(cudaFuncSetAttribute(dist_tc2_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, T2_SMEM_BYTES));
    HG_CUDA(cudaFuncSetAttribute(dist_tc2_kernel<TC_PUSH_WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, T2_SMEM_BYTES));
    HG_CUDA(cudaFuncSetAttribute(dist_tc2_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, T2_SMEM_BYTES));
    HG_CUDA(cudaFuncSetAttribute(dist_tc2_dense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, T2_SMEM_BYTES));
    ctx->tc_attr_set = 1;
  }
  return HG_OK;
}

int hg_tensor_shape_ok(uint32_t hv_d, const void *d_a, const void *d_b) {
  if (hv_d % TC_BK != 0 || hv_d > 32768) {
    hg_set_error("tensor paths need hv_d %% 128 == 0 and hv_d <= 32768 (s32 accumulator bound), got %u", hv_d);
    return HG_E_UNSUPPORTED;
  }
  if (((uintptr_t)d_a | (uintptr_t)d_b) & 15) {
    hg_set_error("tensor paths need 16-byte aligned HV matrices");
    return HG_E_UNSUPPORTED;
  }
  return HG_OK;
}

// ---- one matrix as two s8 limb planes [2][n_rows][hv_d] and its row sums; its rows may be split piecewise, as they arrive ----

uint64_t hg_tc_mat_bytes(uint32_t n_rows, uint32_t hv_d) { return 2 * (uint64_t)n_rows * hv_d + 8 * (uint64_t)n_rows; }

int hg_tc_setup(hg_ctx *ctx, const int16_t *d_hv, uint32_t n_rows, uint32_t hv_d, int plane_slot, hg_tc_mat *m) {
  void *p;
  int rc;
  if ((rc = hg_scratch(ctx, plane_slot, hg_tc_mat_bytes(n_rows, hv_d) + 1024, &p))) return rc;
  return hg_tc_attach(ctx, d_hv, n_rows, hv_d, (int8_t *)p, m);
}

// limb split of rows [row0, row0 + rows) (asynchronous)
int hg_tc_split_rows(hg_ctx *ctx, const hg_tc_mat *m, uint32_t row0, uint32_t rows) {
  if (rows == 0) return HG_OK;
  const uint64_t elems = (uint64_t)rows * m->hv_d;
  uint64_t blocks = (elems / 8 + 255) / 256;
  if (blocks > (uint64_t)ctx->sm_count * 16) blocks = (uint64_t)ctx->sm_count * 16;
  HG_CUDA(cudaMemsetAsync(m->sq + row0, 0, (size_t)rows * 8, ctx->stream));
  split_limbs_kernel<<<(unsigned)blocks, 256, 0, ctx->stream>>>(m->hv + (size_t)row0 * m->hv_d, elems, m->planes + (size_t)row0 * m->hv_d,
                                                                (uint64_t)m->n_rows * m->hv_d, m->hv_d, m->sq + row0);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

// flags[i] = 1 if the limb split finds row i's true norm at or above HG_NORM_WRAP_CUT (asynchronous)
int hg_tc_norm_flags(hg_ctx *ctx, const int16_t *d_hv, uint32_t n_rows, uint32_t hv_d, uint32_t *d_flags) {
  hg_tc_mat m;
  int rc;
  if ((rc = hg_tc_setup(ctx, d_hv, n_rows, hv_d, HG_S_QRY_LIMBS, &m))) return rc;
  if ((rc = hg_tc_split_rows(ctx, &m, 0, n_rows))) return rc;
  tc_flags_kernel<<<(n_rows + 255) / 256, 256, 0, ctx->stream>>>(m.sq, n_rows, d_flags);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

// rows [r0, r0 + n_ref) of R against rows [q0, q0 + n_qry) of Q (both split); norms point at the windows' first rows
int hg_tc_launch(hg_ctx *ctx, const hg_tc_mat *R, uint32_t r0, uint32_t n_ref, uint32_t i0, const int32_t *d_ref_norm,
                 const hg_tc_mat *Q, uint32_t q0, uint32_t n_qry, uint32_t j0, const int32_t *d_qry_norm, uint32_t ksize,
                 float ani_th, int symmetric, hg_hit *d_hits, uint64_t cap, unsigned long long *d_n_hits, const hg_floors *floors,
                 const hg_dense *dense) {
  return hg_tc_launch_ex(ctx, R, r0, n_ref, i0, d_ref_norm, Q, q0, n_qry, j0, d_qry_norm, ksize, ani_th, symmetric, d_hits, cap,
                         d_n_hits, 1, 0, nullptr, nullptr, floors, dense);
}

int hg_tc_attach(hg_ctx *ctx, const int16_t *d_hv, uint32_t n_rows, uint32_t hv_d, int8_t *planes, hg_tc_mat *m) {
  m->hv = d_hv;
  m->planes = planes;
  m->sq = reinterpret_cast<unsigned long long *>(planes + 2 * (uint64_t)n_rows * hv_d);
  m->n_rows = n_rows;
  m->hv_d = hv_d;
  return tc_attrs(ctx);
}

int hg_tc_launch_ex(hg_ctx *ctx, const hg_tc_mat *R, uint32_t r0, uint32_t n_ref, uint32_t i0, const int32_t *d_ref_norm,
                    const hg_tc_mat *Q, uint32_t q0, uint32_t n_qry, uint32_t j0, const int32_t *d_qry_norm, uint32_t ksize,
                    float ani_th, int symmetric, hg_hit *d_hits, uint64_t cap, unsigned long long *d_n_hits, uint32_t walk_mul,
                    uint32_t walk_add, const hg_tile_feed *feed, const hg_push_plan *push, const hg_floors *floors, const hg_dense *dense) {
  if (n_ref == 0 || n_qry == 0) return HG_OK;
  if (floors && push) { hg_set_error("hg_tc_launch: per-query thresholds on a multi-GPU member"); return HG_E_UNSUPPORTED; }
  if (dense && (floors || push)) { hg_set_error("hg_tc_launch: dense output of a search pass or a multi-GPU member"); return HG_E_UNSUPPORTED; }
  hg_tile_feed fd = {};
  if (feed) fd = *feed;
  if (walk_mul == 0 || walk_add >= walk_mul) { hg_set_error("hg_tc_launch: tile walk %u / %u", walk_add, walk_mul); return HG_E_INVALID; }
  int rc;
  const uint32_t hv_d = R->hv_d;
  // the K loop runs whole trips of the 4-stage ring; the tensor maps end at hv_d and fill the boxes past it with zeros,
  // which add nothing to the dot products
  const uint32_t k_len = (hv_d + TC_BK * T2_STAGES - 1) / (TC_BK * T2_STAGES) * (TC_BK * T2_STAGES);
  CUtensorMap tm_ref, tm_qry;
  if ((rc = make_plane_map(&tm_qry, Q->planes, 2ull * Q->n_rows, hv_d, 64))) return rc;
  if ((rc = make_plane_map(&tm_ref, R->planes, 2ull * R->n_rows, hv_d, 128))) return rc;
  hg::DistEpilogue ep;
  ep.ref_norm = d_ref_norm;
  ep.qry_norm = d_qry_norm;
  ep.n_ref = n_ref;
  ep.n_qry = n_qry;
  ep.i0 = i0;
  ep.j0 = j0;
  ep.ksize_f = (float)ksize;
  ep.ani_th = ani_th;
  ep.jmin = hg::dist_jmin(ani_th, ksize);
  ep.cfrac = ep.jmin > 0.0f ? (float)((double)ep.jmin / (1.0 + (double)ep.jmin)) : 0.0f;
  ep.symmetric = symmetric;
  ep.hits = d_hits;
  ep.cap = cap;
  ep.n_hits = d_n_hits;
  // one CTA pair per TPC, each walking the 256 x 128 tiles with stride n_pairs
  const uint32_t gx = (n_qry + TC_BN - 1) / TC_BN;
  const uint64_t tiles = fd.list ? fd.n_list : ((uint64_t)gx * ((n_ref + 255) / 256) + walk_mul - 1) / walk_mul;
  if (tiles == 0) return HG_OK;
  const uint32_t n_pairs = (uint32_t)std::min<uint64_t>(tiles, (uint64_t)std::max(ctx->sm_count / 2, 1));
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cfg.blockDim = dim3(TC_THREADS, 1, 1);
  cfg.gridDim = dim3(2 * n_pairs, 1, 1);
  cfg.dynamicSmemBytes = T2_SMEM_BYTES;
  cfg.stream = ctx->stream;
  static const hg_push_plan no_push = {};
  const unsigned long long *rsq = R->sq + r0, *qsq = Q->sq + q0;  // indexed like the norms
  if (dense) {
    HG_CUDA(cudaLaunchKernelEx(&cfg, dist_tc2_dense_kernel, tm_ref, tm_qry, R->n_rows, r0, Q->n_rows, q0, k_len, ep, walk_mul, walk_add, fd,
                               no_push, *dense));
  } else if (push) {  // a member of several GPUs: pusher warps send my limb-plane rows while the tiles are computed
    cfg.blockDim = dim3(TC_THREADS + 32 * TC_PUSH_WARPS, 1, 1);
    HG_CUDA(cudaLaunchKernelEx(&cfg, dist_tc2_kernel<TC_PUSH_WARPS>, tm_ref, tm_qry, R->n_rows, r0, Q->n_rows, q0, k_len, ep, rsq, qsq,
                               walk_mul, walk_add, fd, *push, hg_floors{}));
  } else if (floors) {
    HG_CUDA(cudaLaunchKernelEx(&cfg, dist_tc2_kernel<0, true>, tm_ref, tm_qry, R->n_rows, r0, Q->n_rows, q0, k_len, ep, rsq, qsq,
                               walk_mul, walk_add, fd, no_push, *floors));
  } else {
    HG_CUDA(cudaLaunchKernelEx(&cfg, dist_tc2_kernel<0>, tm_ref, tm_qry, R->n_rows, r0, Q->n_rows, q0, k_len, ep, rsq, qsq, walk_mul,
                               walk_add, fd, no_push, hg_floors{}));
  }
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}
