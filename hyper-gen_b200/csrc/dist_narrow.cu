// dist_narrow.cu — single-plane tensor dist path: one tcgen05 kind::i8 MMA per K step instead of the
// four of the two-limb split (dist_tc.cu), still bit-exact.
//
// Replaces the pair loop of dist::compute_hv_ani + compute_pairwise_ani (reference
// src/dist.rs:139-161,231-294) when the sketch rows are "narrow".  A sketch HV produced by
// hd::encode_hash_hd* (src/hd.rs:15-112) is hv[d] = 2 * count[d] - n: every element of a row has the
// parity of n, and at the BASELINE configs with D = 4096 / scaled = 1500 the elements span about
// +-240 (hv_quant_bits = 9).  So with a per-row centre s (same parity)
//        x[d] = 2 a[d] + s,   a[d] in [-128, 127]          (one s8 plane, no limb split)
// and for a ref row x (centre s_r) and a query row y = 2 b + s_q
//        x . y = 4 (a . b) + s_q * sum(x~) + s_r * 2 sum(b)           (wrapping i32, like dist.rs:147-151)
// i.e. ONE s8 GEMM plus per-row / per-column constants applied in the epilogue.
//
// Rows that do not fit exactly (an element outside [s - 256, s + 254], or of the other parity) keep
// the clamped value x~ = 2 a + s in the plane and list their residuals eps[d] = x[d] - x~[d] as
// sparse "outlier" entries.  Since x . y = x~ . y~ + sum_d eps_x[d] y[d] + sum_d eps_y[d] x~[d], the
// kernel loosens the candidate bound of such a row by the largest value the correction can take and
// adds the exact correction for the (few) candidates before the exact ANI sequence.  The path is
// taken only while the outlier lists stay small (a budget per row on average); otherwise the caller
// falls back to the two-limb kernel (|hv| <= 8127) or the SIMT kernel, both exact as well.
//
// Kernel: persistent CTA pairs (cluster 2 x 1, tcgen05 cta_group::2, M = 256, N = 256, K = 32), one
// pair per TPC, 256 x 256 output tiles.  Per 128-deep K block a CTA TMA-loads its own 128 ref rows
// and its half (128 rows) of the query tile: 32 KB per stage, 6-stage mbarrier ring.  The s32
// accumulator (256 TMEM columns) is double buffered, so the epilogue of tile t (tcgen05.ld, the
// constants above, division-free ANI bound, candidate list, exact ANI + append) runs entirely under
// the MMAs of tile t + 1.  Operand bytes per MMA clock are twice those of the two-limb kernel
// (L2 -> SM is the limit), hence the 256-wide tile.
#include <cuda.h>

#include <algorithm>
#include <cstdlib>

#include "dist_common.cuh"
#include "tc_ptx.cuh"

namespace {

using namespace hgtc;

constexpr int N1_BN = 256;                              // tile columns (the pair's N)
constexpr int N1_A_BYTES = 128 * TC_BK;                 // 128 of my ref rows
constexpr int N1_B_BYTES = 128 * TC_BK;                 // my half of the 256 query rows
constexpr int N1_STAGES = 6;
constexpr int N1_STAGE_BYTES = N1_A_BYTES + N1_B_BYTES;  // 32 KB
constexpr int N1_EPI_WARPS = 8;                         // two per TMEM lane quarter, half the columns each
constexpr int N1_THREADS = 64 + 32 * N1_EPI_WARPS;      // producer, MMA issuer, epilogue warps (+ 32 per pusher warp of a multi-GPU member)
constexpr int N1_PUSH_WARPS = 2;
constexpr int N1_LIST_CAP = 256;                        // candidates per warp list (8 B each)
constexpr int N1_COL_WORDS = 3 * N1_BN;                 // per tile: bound, centre, 2 sum(b) of every column
constexpr int N1_SMEM_BYTES = N1_STAGES * N1_STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/ +
                              2 * N1_COL_WORDS * 4 /*column constants, double buffered*/ + N1_EPI_WARPS * N1_LIST_CAP * 8 +
                              N1_EPI_WARPS * N1_LIST_CAP * 4 /*ANI of the evaluated candidates*/;
constexpr uint32_t N1_TMEM_COLS = 512;                  // two accumulator buffers of 256 columns
// instruction descriptor, kind::i8: D = s32, A = B = signed 8-bit, both K-major, M = 256 (pair), N = 256
constexpr uint32_t N1_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((N1_BN >> 3) << 17) | ((256u >> 4) << 24);

constexpr int32_t ROW_ALWAYS = INT32_MIN / 2;  // row bound: every column is a candidate
constexpr int32_t COL_ALWAYS = INT32_MIN;      // column bound: every row is a candidate
constexpr int32_t COL_NEVER = INT32_MAX;       // column past the last query

struct NarrowSide {  // per-row constants of one matrix, already offset to the first row of the launch
  const int32_t *s;         // centre
  const int32_t *a2;        // 2 * sum_d a[d]
  const uint32_t *e;        // sum_d |eps[d]|  (0: the row is exactly 2 a + s; E_ALWAYS: its true norm reaches HG_NORM_WRAP_CUT)
  const uint32_t *out_off;  // first outlier entry
  const uint32_t *out_cnt;
};
struct NarrowArgs {
  NarrowSide r, q;
  const uint32_t *r_out, *q_out;  // outlier entries: (d << 16) | (eps & 0xffff)
  const int8_t *r_plane;          // s8 plane of the ref rows (first row of the launch)
  const int8_t *q_plane;          // s8 plane of the query rows (first row of the launch)
  uint32_t hv_d;
  // written by the pre-pass, one set of 4 words per contributor (a multi-GPU matrix has one per member):
  // [0] max |x|, [1] max (|s| + 256) >= max |x~|, [2] entry cursor, [3] declined
  const uint32_t *q_stats, *r_stats;
  uint32_t q_nsets, r_nsets;
  // tile walk: this launch takes the non-empty tiles walk_add, walk_add + walk_mul, ... of the row-major
  // enumeration (single GPU: 0, 1, 2, ...; member r of w GPUs: r, r + w, ...), dealt round-robin to its CTA pairs
  uint32_t walk_mul, walk_add;
};

// ---- i16 rows -> s8 plane + per-row constants + outlier lists ---------------------------------
struct PrepOut {
  int8_t *plane;
  int32_t *s, *a2;
  uint32_t *e, *out_off, *out_cnt;
  uint32_t *entries;
  uint32_t cap;     // entries available
  uint32_t *stats;  // [0] max |x|, [1] max (|s| + 256), [2] entry cursor, [3] overflow flag
};

__device__ __forceinline__ int warp_min(int v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int warp_max(int v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ uint32_t warp_sum(uint32_t v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// e of a row whose true norm sum x^2 reaches HG_NORM_WRAP_CUT: its i32 norm, dots and denominators may wrap, so the
// row / column bound is off (n1_loosen) and every pair with it takes the exact path
constexpr uint32_t E_ALWAYS = 0xFFFFFFFFu;

constexpr int PREP_THREADS = 256;  // 8 warps, one row per warp

// One warp per row, no block-level synchronisation, two int16 per instruction (VIMNMX.S16x2, VIADD.16x2,
// IDP.2A).  Pass 1: range, sum, parity count.  Pass 2 re-reads the row (L1/L2): plane, 2 sum(a), residual
// statistics, and the row's true norm sum x^2 from sum a^2 (IDP.4A on the plane bytes) and the residuals.  Pass 3, rows with outliers only: their entries.  Four 16-byte loads in flight per lane and 48
// warps per SM measured best (4.6 TB/s of HBM traffic on the 820 MB config-4 matrix); keeping the row in
// registers between the passes (116 registers, 16 warps per SM) was 8 % slower there and equal on config 3.
constexpr int PF = 4;
__global__ void __launch_bounds__(PREP_THREADS, 6)
narrow_prep_kernel(const int16_t *__restrict__ hv, uint32_t n_rows, uint32_t hv_d, PrepOut o) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t row = blockIdx.x * (PREP_THREADS / 32) + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const uint32_t nt = hv_d / 256;  // 16-byte loads per lane (hv_d is a multiple of 256)
  const uint4 *src = reinterpret_cast<const uint4 *>(hv + (size_t)row * hv_d) + lane;
  // pass 1
  uint32_t lo2 = 0x7FFF7FFFu, hi2 = 0x80008000u, n_odd = 0;
  int sum_x = 0;
  auto pass1 = [&](const uint4 &v) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      lo2 = __vmins2(lo2, w[j]);
      hi2 = __vmaxs2(hi2, w[j]);
      sum_x = __dp2a_lo((int)w[j], 0x0101, sum_x);  // both halves; |sum| <= 32768 * 32768 fits
      n_odd += __popc(w[j] & 0x00010001u);
    }
  };
  for (uint32_t t0 = 0; t0 < nt; t0 += PF) {
    uint4 v[PF];
#pragma unroll
    for (int u = 0; u < PF; ++u)
      if (t0 + u < nt) v[u] = __ldg(src + 32 * (t0 + u));
#pragma unroll
    for (int u = 0; u < PF; ++u)
      if (t0 + u < nt) pass1(v[u]);
  }
  int lo = min((int)(int16_t)(lo2 & 0xFFFFu), (int)(int16_t)(lo2 >> 16));
  int hi = max((int)(int16_t)(hi2 & 0xFFFFu), (int)(int16_t)(hi2 >> 16));
  lo = warp_min(lo);
  hi = warp_max(hi);
  sum_x = (int)warp_sum((uint32_t)sum_x);
  n_odd = warp_sum(n_odd);
  // centre with the parity of the row (hv = 2 count - n: one parity per row; the majority speaks for it):
  // the middle of the range when the whole row fits [s - 256, s + 254], else the mean (a few far
  // elements become outliers instead of dragging the window away from everything else)
  const int par = 2 * n_odd > hv_d ? 1 : 0;
  int mid = (lo + hi + 2) >> 1;
  if (hi - lo > 510) {
    const int half = (int)(hv_d / 2);
    mid = sum_x >= 0 ? (sum_x + half) / (int)hv_d : -((-sum_x + half) / (int)hv_d);
  }
  const int s = mid - ((mid - par) & 1);
  // x - s must fit 16 bits for the packed arithmetic and the outlier entries; such rows (|x - s| > 32000)
  // make the whole path decline
  const bool bad = hi - s > 32000 || s - lo > 32000;
  // pass 2
  const uint32_t ns2 = (uint32_t)(-s & 0xFFFF) * 0x00010001u;  // -s in both halves
  uint32_t cnt = 0, sum_e = 0;
  int sum_2a = 0, sum_aa = 0;  // sum a^2 <= 32768 * 128^2 = 2^29
  uint2 *dst = reinterpret_cast<uint2 *>(o.plane + (size_t)row * hv_d) + lane;
  auto pass2 = [&](const uint4 &v, uint2 *out) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t r[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t t2 = __vadd2(w[j], ns2);                                     // x - s
      const uint32_t tc = __vmaxs2(__vmins2(t2, 0x00FE00FEu), 0xFF00FF00u);      // clamped to [-256, 254]
      const uint32_t te = tc & 0xFFFEFFFEu;                                       // 2 a  (a = floor(tc / 2))
      sum_2a = __dp2a_lo((int)te, 0x0101, sum_2a);
      r[j] = tc >> 1;                                                             // a: byte 0 (low half), byte 2 (high half)
      if (t2 != te) {                                                             // rare: a residual in this pair
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int eps = (int)(int16_t)(t2 >> (16 * h)) - (int)(int16_t)(te >> (16 * h));
          if (eps != 0) { ++cnt; sum_e += (uint32_t)abs(eps); }
        }
      }
    }
    const uint2 a8 = make_uint2(__byte_perm(r[0], r[1], 0x6420), __byte_perm(r[2], r[3], 0x6420));
    sum_aa = __dp4a((int)a8.x, (int)a8.x, __dp4a((int)a8.y, (int)a8.y, sum_aa));  // signed bytes: IDP.4A.S8.S8
    *out = a8;
  };
  for (uint32_t t0 = 0; t0 < nt; t0 += PF) {
    uint4 v[PF];
#pragma unroll
    for (int u = 0; u < PF; ++u)
      if (t0 + u < nt) v[u] = __ldg(src + 32 * (t0 + u));
#pragma unroll
    for (int u = 0; u < PF; ++u)
      if (t0 + u < nt) pass2(v[u], dst + 32 * (t0 + u));
  }
  // warp totals + exclusive prefix of the outlier counts
  uint32_t inc = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= (uint32_t)d) inc += y;
  }
  const uint32_t tot_c = __shfl_sync(0xffffffffu, inc, 31);
  const uint32_t tot_2a = warp_sum((uint32_t)sum_2a), tot_e = warp_sum(sum_e), tot_aa = warp_sum((uint32_t)sum_aa);
  // the row's true norm: sum x^2 = sum x~^2 + sum (x^2 - x~^2), sum x~^2 = 4 sum a^2 + 2 s sum 2a + D s^2; the second
  // term (residuals only) is added in pass 3, before the row's `e` is written
  long long xx = 4ll * tot_aa + 2ll * s * (int32_t)tot_2a + (long long)hv_d * s * s;
  uint32_t base = 0, kept = tot_c;
  if (lane == 0) {
    if (bad) { atomicExch(&o.stats[3], 1u); kept = 0; }
    if (kept) {
      base = atomicAdd(&o.stats[2], tot_c);
      if (base > o.cap || tot_c > o.cap - base) { atomicExch(&o.stats[3], 1u); kept = 0; }
    }
    o.s[row] = s;
    o.a2[row] = (int32_t)tot_2a;
    if (!kept) o.e[row] = xx >= (long long)HG_NORM_WRAP_CUT ? E_ALWAYS : tot_e;  // no residuals (or declined)
    o.out_off[row] = base;
    o.out_cnt[row] = kept;
    const uint32_t am = (uint32_t)max(abs(lo), abs(hi)), tm = (uint32_t)abs(s) + 256u;
    if (am > *(volatile uint32_t *)&o.stats[0]) atomicMax(&o.stats[0], am);
    if (tm > *(volatile uint32_t *)&o.stats[1]) atomicMax(&o.stats[1], tm);
  }
  base = __shfl_sync(0xffffffffu, base, 0);
  kept = __shfl_sync(0xffffffffu, kept, 0);
  if (kept == 0) return;
  // pass 3 (rows with outliers only): write the entries, lane by lane in scan order
  uint32_t pos = base + inc - cnt;
  long long d_xx = 0;
  for (uint32_t t = 0; t < nt; ++t) {
    const uint4 v = __ldg(src + 32 * t);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int tt = (int)(int16_t)(w[e >> 1] >> (16 * (e & 1))) - s;
      const int a = max(-128, min(127, tt >> 1));
      const int eps = tt - 2 * a;
      if (eps != 0) {
        o.entries[pos++] = ((8u * (lane + 32 * t) + (uint32_t)e) << 16) | ((uint32_t)eps & 0xFFFFu);
        d_xx += (long long)eps * (tt + 2 * a + 2 * s);  // x^2 - x~^2 = eps (x + x~)
      }
    }
  }
#pragma unroll
  for (int m = 16; m; m >>= 1) d_xx += __shfl_xor_sync(0xffffffffu, d_xx, m);
  if (lane == 0) o.e[row] = xx + d_xx >= (long long)HG_NORM_WRAP_CUT ? E_ALWAYS : tot_e;
}

// ---- tile walk: non-empty 256 x 256 tiles, row-block major ------------------------------------------
struct N1Tiles {
  uint32_t gx, gy, R, C;
  int64_t delta;  // i0 - j0
  int sym;
  const uint2 *list;  // multi-GPU member: its tiles in the order the host chose (hg_tile_feed); NULL: the arithmetic walk below
  uint32_t n_list, cur, need;
  __device__ uint32_t cmin(uint32_t r) const {  // symmetric: tiles whose largest j is not above their smallest i are empty
    if (!sym) return 0;
    const int64_t v = delta + 256ll * (int64_t)r + 1;
    if (v <= 0) return 0;
    const uint64_t c = (uint64_t)v / (uint32_t)N1_BN;
    return c > gx ? gx : (uint32_t)c;
  }
  __device__ void init(const hg::DistEpilogue &ep, const hg_tile_feed &f) {
    list = f.list;
    n_list = f.n_list;
    cur = 0;
    need = 0;
    gx = (ep.n_qry + N1_BN - 1) / N1_BN;
    gy = (ep.n_ref + 255) / 256;
    delta = (int64_t)ep.i0 - (int64_t)ep.j0;
    sym = ep.symmetric;
    R = 0;
    C = cmin(0);
  }
  __device__ bool advance(uint32_t k) {
    if (list) {
      cur += k;
      if (cur >= n_list) return false;
      const uint2 e = list[cur];
      R = e.x & 0xFFFFu;
      C = e.x >> 16;
      need = e.y;
      return true;
    }
    while (R < gy) {
      const uint32_t avail = gx - C;
      if (k < avail) { C += k; return true; }
      k -= avail;
      ++R;
      C = cmin(R);
    }
    return false;
  }
};

// bound of a row / column lowered by the largest correction its outliers can contribute (off for an E_ALWAYS row)
__device__ __forceinline__ int32_t n1_loosen(int32_t t, uint32_t e, uint32_t m, int32_t always) {
  if (e == E_ALWAYS) return always;
  if (t == always || e == 0) return t;
  const uint64_t M = (uint64_t)e * m;
  if (M > (1ull << 29)) return always;
  return (int32_t)((int64_t)t - (int64_t)M);  // t >= -1, so this stays far above both sentinels
}

// exact i32 correction of candidate (li, lj): with x = x~ + eps_x, y = y~ + eps_y
//   x . y - x~ . y~ = sum eps_x[d] y~[d] + sum eps_y[d] x~[d] + sum eps_x[d] eps_y[d]
// from the planes and the (short) outlier lists alone - the i16 rows of a remote member are not needed
__device__ __noinline__ int32_t n1_correction(const NarrowArgs &na, uint32_t li, uint32_t lj, uint32_t er, uint32_t eq) {
  uint32_t c = 0;
  const int8_t *a = na.r_plane + (size_t)li * na.hv_d;
  const int8_t *b = na.q_plane + (size_t)lj * na.hv_d;
  const int32_t sr = na.r.s[li], sq = na.q.s[lj];
  const uint32_t roff = na.r.out_off[li], rcnt = er ? na.r.out_cnt[li] : 0u;
  const uint32_t qoff = na.q.out_off[lj], qcnt = eq ? na.q.out_cnt[lj] : 0u;
  for (uint32_t t = 0; t < rcnt; ++t) {
    const uint32_t w = na.r_out[roff + t];
    c += (uint32_t)((int32_t)(int16_t)(w & 0xFFFFu) * (2 * (int32_t)b[w >> 16] + sq));
  }
  for (uint32_t u = 0; u < qcnt; ++u) {
    const uint32_t w = na.q_out[qoff + u];
    c += (uint32_t)((int32_t)(int16_t)(w & 0xFFFFu) * (2 * (int32_t)a[w >> 16] + sr));
    for (uint32_t t = 0; t < rcnt; ++t) {  // both rows have a residual in the same dimension
      const uint32_t v = na.r_out[roff + t];
      if ((v >> 16) == (w >> 16)) c += (uint32_t)((int32_t)(int16_t)(v & 0xFFFFu) * (int32_t)(int16_t)(w & 0xFFFFu));
    }
  }
  return (int32_t)c;
}

// Evaluate a warp's parked candidates and append the survivors: pass 1 runs the exact correction + f32 ANI sequence and
// leaves (keep flag, dot, ANI) in shared memory, ONE atomic reserves room for all survivors (the counter may sit on another
// GPU), pass 2 writes the records.
template <bool QF>
__device__ __forceinline__ void n1_process(const hg::DistEpilogue &ep, const hg_floors &fl, const NarrowArgs &na, uint2 *list, float *anis,
                                           uint32_t n, uint32_t row0, uint32_t col0) {
  if (n == 0) return;
  const uint32_t lane = threadIdx.x & 31;
  uint32_t mine = 0;
  for (uint32_t e = lane; e < n; e += 32) {
    const uint2 c = list[e];
    const uint32_t li = row0 + (c.x >> 8), lj = col0 + (c.x & 255u);
    const bool live = li < ep.n_ref && lj < ep.n_qry;
    int32_t dot = (int32_t)c.y;
    if (live) {
      const uint32_t er = na.r.e[li], eq = na.q.e[lj];
      // (e alone does not say there are entries: an E_ALWAYS row may have none)
      if ((er | eq) && (na.r.out_cnt[li] | na.q.out_cnt[lj])) dot = (int32_t)((uint32_t)dot + (uint32_t)n1_correction(na, li, lj, er, eq));
    }
    float ani = 0.0f;
    const bool keep = hg::dist_eval<QF>(ep, live, li, lj, dot, &ani, fl);
    list[e] = make_uint2(c.x | (keep ? 0x80000000u : 0u), (uint32_t)dot);
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

// One epilogue warp drains columns [c_begin, c_end) of its 32 TMEM lanes: row `rowl` of the CTA's
// 128 rows per lane.  x~ . y~ = 4 acc + s_q * X_r + s_r * T_q with X_r = sum x~ of my row and, per
// column, the centre s_q and T_q = 2 sum(b).  Candidates (rowl, column, x~ . y~) go to `list`.
template <bool QF>
__device__ __forceinline__ uint32_t n1_drain(const hg::DistEpilogue &ep, const hg_floors &fl, const NarrowArgs &na, uint32_t taddr, int c_begin,
                                             int c_end, const int32_t *s_col, int32_t tr, int32_t sr, int32_t xr, bool row_live,
                                             uint32_t rowl, uint32_t row0, uint32_t col0, uint2 *list, float *anis, uint32_t n_list) {
  const uint32_t lane = threadIdx.x & 31;
  const bool row_always = tr == ROW_ALWAYS;
  uint32_t nx[16];
  tmem_ld16(taddr + c_begin, nx);
#pragma unroll 1
  for (int c = c_begin; c < c_end; c += 16) {
    uint32_t ac[16];
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    tmem_ld_fence(nx);
#pragma unroll
    for (int j = 0; j < 16; ++j) ac[j] = nx[j];
    if (c + 16 < c_end) tmem_ld16(taddr + c + 16, nx);
    int32_t dot[16];
    uint32_t cand = 0;
#pragma unroll
    for (int j4 = 0; j4 < 16; j4 += 4) {
      const int4 tq4 = *reinterpret_cast<const int4 *>(s_col + c + j4);
      const int4 sq4 = *reinterpret_cast<const int4 *>(s_col + N1_BN + c + j4);
      const int4 tt4 = *reinterpret_cast<const int4 *>(s_col + 2 * N1_BN + c + j4);
      const int32_t tq[4] = {tq4.x, tq4.y, tq4.z, tq4.w}, sq[4] = {sq4.x, sq4.y, sq4.z, sq4.w}, tt[4] = {tt4.x, tt4.y, tt4.z, tt4.w};
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = j4 + u;
        dot[j] = (int32_t)(4u * ac[j] + (uint32_t)sq[u] * (uint32_t)xr + (uint32_t)sr * (uint32_t)tt[u]);  // wrapping i32
        const bool cj = (dot[j] >= (int32_t)((uint32_t)tr + (uint32_t)tq[u]) || tq[u] == COL_ALWAYS || row_always) && tq[u] != COL_NEVER;
        cand |= (uint32_t)cj << j;
      }
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
      if (n_list + total > N1_LIST_CAP) {  // evaluate what is parked (slow path: the accumulator stays held)
        n1_process<QF>(ep, fl, na, list, anis, n_list, row0, col0);
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

// Dense mode (hg_dense): the same drain without the bound; every live element gets its outlier correction when its row
// or column has entries (`rcorr`, and the column flags in place of the bounds in s_col), and the exact dot goes to its cell.
__device__ __forceinline__ void n1_drain_dense(const hg::DistEpilogue &ep, const hg_dense &dn, const NarrowArgs &na, uint32_t taddr,
                                               int c_begin, int c_end, const int32_t *s_col, int32_t sr, int32_t xr, bool row_live,
                                               bool rcorr, uint32_t li, uint32_t col0) {
  const uint32_t gi = ep.i0 + li;
  uint32_t nx[16];
  tmem_ld16(taddr + c_begin, nx);
#pragma unroll 1
  for (int c = c_begin; c < c_end; c += 16) {
    uint32_t ac[16];
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    tmem_ld_fence(nx);
#pragma unroll
    for (int j = 0; j < 16; ++j) ac[j] = nx[j];
    if (c + 16 < c_end) tmem_ld16(taddr + c + 16, nx);
    const uint32_t gj = ep.j0 + col0 + c;
    const uint32_t n = row_live ? hg::dense_live(dn, ep, gi, gj) : 0u;
    if (n) {  // (no `continue`: the warp stays converged for the next tcgen05.wait)
      int32_t dot[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        dot[j] = (int32_t)(4u * ac[j] + (uint32_t)s_col[N1_BN + c + j] * (uint32_t)xr + (uint32_t)sr * (uint32_t)s_col[2 * N1_BN + c + j]);
        if ((uint32_t)j < n && (rcorr || s_col[c + j])) {
          const uint32_t lj = col0 + c + j;
          dot[j] = (int32_t)((uint32_t)dot[j] + (uint32_t)n1_correction(na, li, lj, na.r.e[li], na.q.e[lj]));
        }
      }
      hg::dense_store16(dn, gi, gj, n, dot);
    }
  }
}

// QF: per-query thresholds (a search pass, PUSHW = 0 only); `fl` is not read otherwise.  DENSE (PUSHW = 0, no QF): every
// live pair's dot to its cell of `dn` (hg_dense) instead of the bound, the exact epilogue and the append.
template <int PUSHW, bool QF, bool DENSE>
__device__ __forceinline__ void n1_body(const CUtensorMap &tm_ref, const CUtensorMap &tm_qry, uint32_t ref_row_base, uint32_t qry_row_base,
                                        const hg::DistEpilogue &ep, const NarrowArgs &na, hg_tile_feed feed, const hg_push_plan &plan,
                                        const hg_floors &fl, const hg_dense &dn) {
  constexpr int STAGES = N1_STAGES, STAGE_BYTES = N1_STAGE_BYTES;
  uint32_t rank;  // 0 = leader (issues the MMAs, owns the full / tmem-empty barriers), 1 = peer
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
  if (feed.seq_ptr) feed.seq = *feed.seq_ptr;
  if (blockIdx.x == 0 && threadIdx.x == 0) hg::feed_stamp(feed.dbg, 1);
  // this pair's tiles: first, first + n_pairs, ... of the launch's share of the tile enumeration
  const uint32_t pair = (blockIdx.x >> 1) * na.walk_mul + na.walk_add, n_pairs = (gridDim.x >> 1) * na.walk_mul;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;  // 128B swizzle wants 1024 B alignment
  uint8_t *aligned = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t bar_base = base + STAGES * STAGE_BYTES;
  auto full_bar = [&](uint32_t s) { return bar_base + 8u * s; };                       // used in the leader only
  auto empty_bar = [&](uint32_t s) { return bar_base + 8u * (STAGES + s); };           // one per CTA, multicast commit
  auto accum_bar = [&](uint32_t b) { return bar_base + 8u * (2 * STAGES + b); };       // one per CTA and buffer, multicast commit
  auto tmem_empty_bar = [&](uint32_t b) { return bar_base + 8u * (2 * STAGES + 2 + b); };  // leader only: both epilogues drained
  volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(aligned + STAGES * STAGE_BYTES + 8 * (2 * STAGES + 4));
  int32_t *s_col_all = reinterpret_cast<int32_t *>(aligned + STAGES * STAGE_BYTES + 256);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(accum_bar(b), 1); mbar_init(tmem_empty_bar(b), 2 * N1_EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {  // the same warp in both CTAs
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void *)tmem_slot)),
                 "r"(N1_TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  cluster_sync_all();  // the peer's barriers are initialised before anyone signals them
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t num_kb = na.hv_d / TC_BK;

  if (PUSHW > 0 && warp >= N1_THREADS / 32) {
    // ===== pusher warps (a member of several GPUs): my operand rows to the windows of the members that compute with them, unit by unit =====
    hg::push_my_units(&plan, blockIdx.x * PUSHW + (uint32_t)(warp - N1_THREADS / 32), gridDim.x * PUSHW);
  } else {
  uint32_t have = 0;  // arrival flags seen so far (warp 0)
  if (feed.start_need) {  // the other members' pre-pass statistics have arrived, the root has reset its hit counter
    if (warp == 0) hg::feed_wait_start(feed);
    if (warp == 0 && blockIdx.x == 0 && lane == 0) hg::feed_stamp(feed.dbg, 2);
    asm volatile("bar.sync 2, %0;" ::"r"(N1_THREADS) : "memory");
  }
  // the pre-passes ran before this kernel (on this GPU, and on the others before their statistics were pushed): if they
  // found the rows not narrow (outlier budget exceeded) nothing is computed here and the host, which reads the same
  // flags after this launch, takes another path
  uint32_t declined = 0, q_absmax = 0, r_tmax = 0;
  for (uint32_t t = 0; t < na.q_nsets; ++t) { declined |= na.q_stats[4 * t + 3]; q_absmax = max(q_absmax, na.q_stats[4 * t]); }
  for (uint32_t t = 0; t < na.r_nsets; ++t) { declined |= na.r_stats[4 * t + 3]; r_tmax = max(r_tmax, na.r_stats[4 * t + 1]); }

  N1Tiles tiles;
  tiles.init(ep, feed);
  bool valid = !declined && tiles.advance(pair);

  if (warp == 0) {
    // ===== TMA producer (both CTAs; completion bytes go to the LEADER's full barrier) =====
    const uint32_t on = elect_one();
    uint32_t s = 0, ph = 0;
    unsigned long long waited = 0;  // (timeline) ns this producer spent waiting for other members' rows
    for (; valid; valid = tiles.advance(n_pairs)) {
      const uint32_t row0 = tiles.R * 256u + rank * 128u, colh = tiles.C * N1_BN + rank * 128u;
      if (tiles.need) {  // the rows this tile reads have arrived from their owners
        const unsigned long long w0 = feed.dbg ? hg::feed_ns() : 0ull;
        hg::feed_wait(feed, tiles.need, have);
        if (feed.dbg) waited += hg::feed_ns() - w0;
      }
      for (uint32_t kb = 0; kb < num_kb; ++kb) {
        mbar_wait_cluster(empty_bar(s), ph ^ 1u);
        mbar_expect_tx(full_bar(s), 2 * STAGE_BYTES, rank == 0 ? on : 0u);  // the leader expects its bytes and the peer's
        const uint32_t fb = mapa_u32(full_bar(s), 0);
        const uint32_t st = base + s * STAGE_BYTES;
        const int k0 = (int)(kb * TC_BK);
        tma_load_2d_pair(st, &tm_ref, fb, k0, (int)(ref_row_base + row0), on);                     // my 128 ref rows
        tma_load_2d_pair(st + N1_A_BYTES, &tm_qry, fb, k0, (int)(qry_row_base + colh), on);      // my half of the query rows
        if (++s == STAGES) { s = 0; ph ^= 1u; }
      }
    }
    if (feed.dbg && lane == 0) { atomicMax(feed.dbg + 5, waited); if (blockIdx.x == 0) feed.dbg[3] = waited; }
  } else if (warp == 1) {
    // ===== MMA issuer: one thread of the leader CTA drives both SMs' tensor cores =====
    if (rank == 0) {
      const uint32_t on = elect_one();
      const uint32_t d0 = umma_desc_lo(base);
      uint32_t s = 0, ph = 0, tile_n = 0;
      for (; valid; valid = tiles.advance(n_pairs), ++tile_n) {
        const uint32_t b = tile_n & 1u, use = tile_n >> 1;  // accumulator buffer, and how often it was used before
        // both epilogues have drained this buffer's previous tile (passes at once for its first use)
        mbar_wait_cluster(tmem_empty_bar(b), (use & 1u) ^ 1u);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t tacc = tmem_base + b * N1_BN;
        for (uint32_t kb = 0; kb < num_kb; ++kb) {
          mbar_wait(full_bar(s), ph);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t a0 = d0 + s * (uint32_t)(STAGE_BYTES >> 4);
#pragma unroll
          for (int ks = 0; ks < TC_BK / 32; ++ks)  // one MMA covers K = 32 int8
            umma_i8_pair(tacc, a0 + (uint32_t)((32 * ks) >> 4), a0 + (uint32_t)((N1_A_BYTES + 32 * ks) >> 4), N1_IDESC,
                         (kb | (uint32_t)ks) != 0u, on);
          umma_commit_pair(empty_bar(s), on);  // the stage is free in both CTAs once these MMAs have read it
          if (++s == STAGES) { s = 0; ph ^= 1u; }
        }
        umma_commit_pair(accum_bar(b), on);  // accumulators final: wake both epilogues
      }
    }
  } else {
    // ===== epilogue (both CTAs, each its own 128 rows of the accumulator) =====
    const int ew = warp - 2;
    const uint32_t q = warp & 3;  // TMEM lane quarter this warp may read
    const int half = (ew >> 2);   // which 128 columns this warp drains
    uint2 *list = reinterpret_cast<uint2 *>(aligned + STAGES * STAGE_BYTES + 256 + 2 * N1_COL_WORDS * 4) + ew * N1_LIST_CAP;
    float *anis = reinterpret_cast<float *>(aligned + STAGES * STAGE_BYTES + 256 + 2 * N1_COL_WORDS * 4 + N1_EPI_WARPS * N1_LIST_CAP * 8) +
                  ew * N1_LIST_CAP;
    uint32_t tile_n = 0, have_e = 0, have_l = 0;
    volatile uint32_t *s_early = reinterpret_cast<volatile uint32_t *>(aligned + STAGES * STAGE_BYTES + 240);
    for (; valid; valid = tiles.advance(n_pairs), ++tile_n) {
      const uint32_t b = tile_n & 1u, use = tile_n >> 1;
      const uint32_t row0 = tiles.R * 256u + rank * 128u, col0 = tiles.C * N1_BN;
      // The per-row / per-column constants are read BEFORE the accumulator is waited for, to hide their latency - in a
      // multi-GPU launch possibly before the rows they belong to have arrived.  One epilogue warp looks at the arrival
      // flags (no spinning here: the producer does the waiting) and all eight take the same route: constants now, or
      // after the accumulator barrier, by when the producer has seen the flags.
      bool early = true;
      if (tiles.need) {
        if (ew == 0) {
          const bool ok = hg::feed_poll(feed, tiles.need, have_e);
          if (lane == 0) *s_early = ok ? 1u : 0u;
        }
        asm volatile("bar.sync 1, %0;" ::"r"(32 * N1_EPI_WARPS) : "memory");
        early = *s_early != 0u;
      }
      int32_t *s_col = s_col_all + (tile_n & 1u) * N1_COL_WORDS;  // double buffered: one barrier per tile is enough
      int32_t tr, sr, xr;
      bool live, rcorr;
      auto constants = [&]() {
        {
          const uint32_t t = threadIdx.x - 64, lj = col0 + t;  // one column per epilogue thread
          int32_t tq = COL_NEVER, sq = 0, tt = 0;
          if (DENSE) {  // the column's outlier flag
            tq = lj < ep.n_qry && na.q.e[lj] && na.q.out_cnt[lj];
            if (lj < ep.n_qry) { sq = na.q.s[lj]; tt = na.q.a2[lj]; }
          } else if (lj < ep.n_qry) {
            tq = COL_ALWAYS;
            float cq = ep.cfrac;
            if constexpr (QF) cq = fl.q[lj].cfrac;
            if (cq > 0.0f) {
              const int32_t nq = ep.qry_norm[lj];
              if (nq > 0) tq = n1_loosen(__float2int_rd(cq * __int2float_rz(nq)) - 1, na.q.e[lj], r_tmax, COL_ALWAYS);
            }
            sq = na.q.s[lj];
            tt = na.q.a2[lj];
          }
          s_col[t] = tq;
          s_col[N1_BN + t] = sq;
          s_col[2 * N1_BN + t] = tt;
        }
        asm volatile("bar.sync 1, %0;" ::"r"(32 * N1_EPI_WARPS) : "memory");  // epilogue warps only
        // row constants of my row
        const uint32_t li = row0 + q * 32 + lane;
        tr = ROW_ALWAYS; sr = 0; xr = 0;
        live = li < ep.n_ref;
        rcorr = DENSE && live && na.r.e[li] && na.r.out_cnt[li];
        if (live) {
          float cr = ep.cfrac;
          if constexpr (QF) cr = *fl.cfrac_row;
          if (cr > 0.0f) {
            const int32_t nr = ep.ref_norm[li];
            if (nr > 0) tr = n1_loosen(__float2int_rd(cr * __int2float_rz(nr)) - 1, na.r.e[li], q_absmax, ROW_ALWAYS);
          }
          sr = na.r.s[li];
          xr = (int32_t)((uint32_t)na.r.a2[li] + na.hv_d * (uint32_t)sr);  // sum x~ = 2 sum a + D s
        }
      };
      if (early) constants();
      mbar_wait_cluster(accum_bar(b), use & 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (!early) {  // the producer has seen this tile's arrival flags; so do we now (an acquire, returns at once)
        hg::feed_wait(feed, tiles.need, have_l);
        constants();
      }
      uint32_t n_list = 0;
      // my 128 x 256 part of the tile may be empty (below the diagonal, or past the last ref row)
      const bool mine_empty = row0 >= ep.n_ref || (ep.symmetric && (uint64_t)ep.j0 + col0 + N1_BN - 1 <= (uint64_t)ep.i0 + row0);
      if constexpr (DENSE) {
        if (!mine_empty)
          n1_drain_dense(ep, dn, na, tmem_base + ((q * 32u) << 16) + b * N1_BN, half * (N1_BN / 2), (half + 1) * (N1_BN / 2), s_col, sr, xr,
                         live, rcorr, row0 + q * 32 + lane, col0);
      } else if (!mine_empty) {
        n_list = n1_drain<QF>(ep, fl, na, tmem_base + ((q * 32u) << 16) + b * N1_BN, half * (N1_BN / 2), (half + 1) * (N1_BN / 2), s_col, tr,
                          sr, xr, live, q * 32 + lane, row0, col0, list, anis, 0u);
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(mapa_u32(tmem_empty_bar(b), 0));  // this warp's TMEM reads of buffer b are done
      n1_process<QF>(ep, fl, na, list, anis, n_list, row0, col0);          // exact ANI + append, under the next tiles' MMAs
    }
  }
  }  // compute roles
  __syncthreads();
  if (threadIdx.x == 0) hg::feed_stamp_max(feed.dbg, 4);
  cluster_sync_all();  // nobody leaves while the peer may still read its smem or signal its barriers
  if (warp == 2) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(N1_TMEM_COLS) : "memory");
  }
}

template <int PUSHW, bool QF = false>
__global__ void __launch_bounds__(N1_THREADS + 32 * PUSHW, 1)
dist_n1_kernel(const __grid_constant__ CUtensorMap tm_ref, const __grid_constant__ CUtensorMap tm_qry, uint32_t ref_row_base,
               uint32_t qry_row_base, hg::DistEpilogue ep, NarrowArgs na, hg_tile_feed feed, const __grid_constant__ hg_push_plan plan,
               hg_floors fl) {
  n1_body<PUSHW, QF, false>(tm_ref, tm_qry, ref_row_base, qry_row_base, ep, na, feed, plan, fl, hg_dense{});
}

__global__ void __launch_bounds__(N1_THREADS, 1)
dist_n1_dense_kernel(const __grid_constant__ CUtensorMap tm_ref, const __grid_constant__ CUtensorMap tm_qry, uint32_t ref_row_base,
                     uint32_t qry_row_base, hg::DistEpilogue ep, NarrowArgs na, hg_tile_feed feed,
                     const __grid_constant__ hg_push_plan plan, hg_dense dn) {
  n1_body<0, false, true>(tm_ref, tm_qry, ref_row_base, qry_row_base, ep, na, feed, plan, hg_floors{}, dn);
}

void carve_arrays(hg_narrow_mat &m, void *arrays) {
  uint32_t *w = (uint32_t *)arrays;
  const size_t n = m.n_rows;
  m.s = (int32_t *)w;
  m.a2 = (int32_t *)(w + n);
  m.e = w + 2 * n;
  m.out_off = w + 3 * n;
  m.out_cnt = w + 4 * n;
}

PrepOut prep_out(const hg_narrow_mat &m, uint32_t row0) {
  PrepOut o;
  o.plane = m.plane + (size_t)row0 * m.hv_d;
  o.s = m.s + row0;
  o.a2 = m.a2 + row0;
  o.e = m.e + row0;
  o.out_off = m.out_off + row0;
  o.out_cnt = m.out_cnt + row0;
  o.entries = m.entries;
  o.cap = m.cap;
  o.stats = m.stats;
  return o;
}

__global__ void narrow_stats_init_kernel(uint32_t *stats, uint32_t entry_base) {
  if (threadIdx.x < 4) stats[threadIdx.x] = threadIdx.x == 2 ? entry_base : 0u;
}

__global__ void narrow_flags_kernel(const uint32_t *__restrict__ e, uint32_t n, uint32_t *__restrict__ flags) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flags[i] = e[i] == E_ALWAYS;
}

uint32_t narrow_budget() {  // outlier entries per row on average (HG_NARROW_BUDGET overrides; tests use it to force the correction path)
  uint32_t per_row = 4;
  if (const char *e = getenv("HG_NARROW_BUDGET")) per_row = (uint32_t)std::max(0, atoi(e));
  return per_row;
}

}  // namespace

void hg_narrow_tile_shape(uint32_t *rows, uint32_t *cols) { *rows = 256; *cols = N1_BN; }

// ---- one matrix in single-plane form; its rows may be prepared piecewise, as they arrive ------
size_t hg_narrow_meta_bytes(uint32_t n_rows) {
  return ((((size_t)n_rows * 5 + ((size_t)n_rows * narrow_budget() + 1024) + 4) * 4 + 256) + 255) & ~(size_t)255;
}
size_t hg_narrow_arrays_bytes(uint32_t n_rows) { return (size_t)n_rows * 5 * 4; }
uint32_t hg_narrow_set_cap(uint32_t n_rows) { return (uint32_t)std::min<uint64_t>((uint64_t)n_rows * narrow_budget() + 1024, 0x0FFFFFFFull); }

static int narrow_attrs(hg_ctx *ctx) {
  if (!ctx->n1_attr_set) {
    HG_CUDA(cudaFuncSetAttribute(dist_n1_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, N1_SMEM_BYTES));
    HG_CUDA(cudaFuncSetAttribute(dist_n1_kernel<N1_PUSH_WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, N1_SMEM_BYTES));
    HG_CUDA(cudaFuncSetAttribute(dist_n1_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, N1_SMEM_BYTES));
    HG_CUDA(cudaFuncSetAttribute(dist_n1_dense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, N1_SMEM_BYTES));
    ctx->n1_attr_set = 1;
  }
  return HG_OK;
}

// the matrix lives in caller-provided memory (a peer window shared by `n_sets` members); this context prepares some of
// its rows, records its statistics in set `my_set` and may use entries [entry_base, entry_base + set_cap)
int hg_narrow_attach(hg_ctx *ctx, const int16_t *d_hv, uint32_t n_rows, uint32_t hv_d, int8_t *plane, void *arrays,
                     uint32_t *entries, uint32_t *stats_all, uint32_t n_sets, uint32_t my_set, uint32_t entry_base,
                     uint32_t set_cap, hg_narrow_mat *m, bool init_stats) {
  m->hv = d_hv;
  m->n_rows = n_rows;
  m->hv_d = hv_d;
  m->plane = plane;
  carve_arrays(*m, arrays);
  m->entries = entries;
  m->stats_all = stats_all;
  m->stats = stats_all + 4 * my_set;
  m->n_sets = n_sets;
  m->entry_base = entry_base;
  m->cap = entry_base + set_cap;
  if (init_stats) {  // (peer.cu resets the statistics in the first node of its launch sequence instead)
    narrow_stats_init_kernel<<<1, 32, 0, ctx->stream>>>(m->stats, entry_base);
    ctx->launches++;
    HG_CUDA(cudaGetLastError());
  }
  return narrow_attrs(ctx);
}

// plane in scratch slot `plane_slot`, constants at `meta` (hg_narrow_meta_bytes); the statistics are zeroed on the stream
int hg_narrow_setup(hg_ctx *ctx, const int16_t *d_hv, uint32_t n_rows, uint32_t hv_d, int plane_slot, void *meta,
                    hg_narrow_mat *m) {
  const uint64_t cap64 = (uint64_t)n_rows * narrow_budget() + 1024;
  if (cap64 > 0x7FFFFFFFull) { hg_set_error("narrow tensor path: outlier budget too large"); return HG_E_UNSUPPORTED; }
  void *plane;
  int rc;
  if ((rc = hg_scratch(ctx, plane_slot, (uint64_t)n_rows * hv_d + 1024, &plane))) return rc;
  m->hv = d_hv;
  m->n_rows = n_rows;
  m->hv_d = hv_d;
  m->plane = (int8_t *)plane;
  uint32_t *w = (uint32_t *)meta;  // 4 statistics words | the five per-row arrays | entries
  m->stats = m->stats_all = w;
  m->n_sets = 1;
  m->entry_base = 0;
  m->cap = (uint32_t)cap64;
  carve_arrays(*m, w + 4);
  m->entries = w + 4 + 5 * (size_t)n_rows;
  HG_CUDA(cudaMemsetAsync(m->stats, 0, 16, ctx->stream));
  return narrow_attrs(ctx);
}

// pre-pass over rows [row0, row0 + rows) of the matrix (asynchronous)
int hg_narrow_prep_rows(hg_ctx *ctx, const hg_narrow_mat *m, uint32_t row0, uint32_t rows) {
  if (rows == 0) return HG_OK;
  const uint32_t blocks = (rows + PREP_THREADS / 32 - 1) / (PREP_THREADS / 32);
  narrow_prep_kernel<<<blocks, PREP_THREADS, 0, ctx->stream>>>(m->hv + (size_t)row0 * m->hv_d, rows, m->hv_d, prep_out(*m, row0));
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

// rows [r0, r0 + n_ref) of R against rows [q0, q0 + n_qry) of Q (both prepared); norms point at the windows' first rows.
// Asynchronous; the kernel does nothing if a pre-pass so far has declined (hg_narrow_verdict tells the host).
int hg_narrow_launch(hg_ctx *ctx, const hg_narrow_mat *R, uint32_t r0, uint32_t n_ref, uint32_t i0, const int32_t *d_ref_norm,
                     const hg_narrow_mat *Q, uint32_t q0, uint32_t n_qry, uint32_t j0, const int32_t *d_qry_norm,
                     uint32_t ksize, float ani_th, int symmetric, hg_hit *d_hits, uint64_t cap,
                     unsigned long long *d_n_hits, const hg_floors *floors, const hg_dense *dense) {
  return hg_narrow_launch_ex(ctx, R, r0, n_ref, i0, d_ref_norm, Q, q0, n_qry, j0, d_qry_norm, ksize, ani_th, symmetric, d_hits, cap,
                             d_n_hits, 1, 0, nullptr, nullptr, floors, dense);
}

int hg_narrow_launch_ex(hg_ctx *ctx, const hg_narrow_mat *R, uint32_t r0, uint32_t n_ref, uint32_t i0, const int32_t *d_ref_norm,
                        const hg_narrow_mat *Q, uint32_t q0, uint32_t n_qry, uint32_t j0, const int32_t *d_qry_norm,
                        uint32_t ksize, float ani_th, int symmetric, hg_hit *d_hits, uint64_t cap,
                        unsigned long long *d_n_hits, uint32_t walk_mul, uint32_t walk_add, const hg_tile_feed *feed,
                        const hg_push_plan *push, const hg_floors *floors, const hg_dense *dense) {
  if (n_ref == 0 || n_qry == 0) return HG_OK;
  if (floors && push) { hg_set_error("hg_narrow_launch: per-query thresholds on a multi-GPU member"); return HG_E_UNSUPPORTED; }
  if (dense && (floors || push)) { hg_set_error("hg_narrow_launch: dense output of a search pass or a multi-GPU member"); return HG_E_UNSUPPORTED; }
  if (walk_mul == 0 || walk_add >= walk_mul) { hg_set_error("hg_narrow_launch: tile walk %u / %u", walk_add, walk_mul); return HG_E_INVALID; }
  int rc;
  const uint32_t hv_d = R->hv_d;
  CUtensorMap tm_ref, tm_qry;
  if ((rc = make_plane_map(&tm_qry, Q->plane, Q->n_rows, hv_d, 128))) return rc;
  if (R == Q || R->plane == Q->plane) tm_ref = tm_qry;
  else if ((rc = make_plane_map(&tm_ref, R->plane, R->n_rows, hv_d, 128))) return rc;
  NarrowArgs na;
  na.r = {R->s + r0, R->a2 + r0, R->e + r0, R->out_off + r0, R->out_cnt + r0};
  na.q = {Q->s + q0, Q->a2 + q0, Q->e + q0, Q->out_off + q0, Q->out_cnt + q0};
  na.r_out = R->entries;
  na.q_out = Q->entries;
  na.r_plane = R->plane + (size_t)r0 * hv_d;
  na.q_plane = Q->plane + (size_t)q0 * hv_d;
  na.hv_d = hv_d;
  na.q_stats = Q->stats_all;
  na.r_stats = R->stats_all;
  na.q_nsets = Q->n_sets;
  na.r_nsets = R->n_sets;
  na.walk_mul = walk_mul;
  na.walk_add = walk_add;

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

  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cfg.blockDim = dim3(N1_THREADS, 1, 1);
  cfg.stream = ctx->stream;
  // one CTA pair per TPC, each walking its 256 x 256 tiles with stride n_pairs
  const uint64_t tiles_all = (uint64_t)((n_qry + N1_BN - 1) / N1_BN) * ((n_ref + 255) / 256);
  hg_tile_feed fd = {};
  if (feed) fd = *feed;
  // this launch's share of the tiles (an upper bound when symmetric)
  const uint64_t tiles = fd.list ? fd.n_list : (tiles_all + walk_mul - 1) / walk_mul;
  if (tiles == 0) return HG_OK;
  const uint32_t n_pairs = (uint32_t)std::min<uint64_t>(tiles, (uint64_t)std::max(ctx->sm_count / 2, 1));
  cfg.gridDim = dim3(2 * n_pairs, 1, 1);
  cfg.dynamicSmemBytes = N1_SMEM_BYTES;
  static const hg_push_plan no_push = {};
  if (dense) {
    HG_CUDA(cudaLaunchKernelEx(&cfg, dist_n1_dense_kernel, tm_ref, tm_qry, r0, q0, ep, na, fd, no_push, *dense));
  } else if (push) {  // a member of several GPUs: the launch carries pusher warps that send my operand rows while the tiles are computed
    cfg.blockDim = dim3(N1_THREADS + 32 * N1_PUSH_WARPS, 1, 1);
    HG_CUDA(cudaLaunchKernelEx(&cfg, dist_n1_kernel<N1_PUSH_WARPS>, tm_ref, tm_qry, r0, q0, ep, na, fd, *push, hg_floors{}));
  } else if (floors) {
    HG_CUDA(cudaLaunchKernelEx(&cfg, dist_n1_kernel<0, true>, tm_ref, tm_qry, r0, q0, ep, na, fd, no_push, *floors));
  } else {
    HG_CUDA(cudaLaunchKernelEx(&cfg, dist_n1_kernel<0>, tm_ref, tm_qry, r0, q0, ep, na, fd, no_push, hg_floors{}));
  }
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}

// flags[i] = 1 if the pre-pass marks row i E_ALWAYS (its true norm reaches HG_NORM_WRAP_CUT); HG_E_UNSUPPORTED if the
// pre-pass declines the rows (synchronises the stream)
int hg_narrow_norm_flags(hg_ctx *ctx, const int16_t *d_hv, uint32_t n_rows, uint32_t hv_d, uint32_t *d_flags) {
  void *meta;
  int rc;
  hg_narrow_mat m;
  if ((rc = hg_scratch(ctx, HG_S_NARROW_META, hg_narrow_meta_bytes(n_rows), &meta))) return rc;
  if ((rc = hg_narrow_setup(ctx, d_hv, n_rows, hv_d, HG_S_QRY_LIMBS, meta, &m))) return rc;
  if ((rc = hg_narrow_prep_rows(ctx, &m, 0, n_rows))) return rc;
  narrow_flags_kernel<<<(n_rows + 255) / 256, 256, 0, ctx->stream>>>(m.e, n_rows, d_flags);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return hg_narrow_verdict(ctx, &m, nullptr, nullptr, nullptr);
}

// Reads the pre-pass statistics (synchronises the stream): HG_OK if every row prepared so far fits the single
// plane within the budget, else HG_E_UNSUPPORTED, a result that sets no error (then the kernels launched so far
// have done nothing useful and the caller must discard their hits).  B may be NULL or equal to A.
int hg_narrow_verdict(hg_ctx *ctx, const hg_narrow_mat *A, const hg_narrow_mat *B, int32_t *absmax_out, uint64_t *outliers_out) {
  uint32_t sa[4 * 8] = {0}, sb[4 * 8] = {0};
  if (A->n_sets > 8 || (B && B->n_sets > 8)) { hg_set_error("hg_narrow_verdict: more than 8 statistic sets"); return HG_E_INVALID; }
  HG_CUDA(cudaMemcpyAsync(sa, A->stats_all, 16 * A->n_sets, cudaMemcpyDeviceToHost, ctx->stream));
  const bool two = B && B != A && B->stats_all != A->stats_all;
  if (two) HG_CUDA(cudaMemcpyAsync(sb, B->stats_all, 16 * B->n_sets, cudaMemcpyDeviceToHost, ctx->stream));
  HG_CUDA(cudaStreamSynchronize(ctx->stream));
  uint32_t amax = 0, declined = 0;
  uint64_t used = 0;
  for (uint32_t t = 0; t < A->n_sets; ++t) { amax = std::max(amax, sa[4 * t]); declined |= sa[4 * t + 3]; }
  for (uint32_t t = 0; two && t < B->n_sets; ++t) { amax = std::max(amax, sb[4 * t]); declined |= sb[4 * t + 3]; }
  // entries used: the cursors start at each set's base (a single-set matrix: 0)
  used += A->n_sets == 1 ? sa[2] - A->entry_base : 0;
  used += two && B->n_sets == 1 ? sb[2] - B->entry_base : 0;
  if (absmax_out) *absmax_out = (int32_t)amax;
  if (outliers_out) *outliers_out = used;
  return declined ? HG_E_UNSUPPORTED : HG_OK;
}
