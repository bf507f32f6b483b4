// dist_common.cuh — the fused epilogue shared by both dist kernels: exact i32 dot ->
// Jaccard -> ANI (reference src/dist.rs:153-160) -> `ani >= ani_th` filter
// (src/utils.rs:274-285) -> compacted append of (i, j, dot, ani).
#pragma once
#include <math.h>

#include "hg_common.cuh"

namespace hg {

struct DistEpilogue {
  const int32_t *__restrict__ ref_norm;
  const int32_t *__restrict__ qry_norm;
  uint32_t n_ref, n_qry;
  uint32_t i0, j0;  // global index offsets of this shard
  float ksize_f;
  float ani_th;
  float jmin;  // conservative Jaccard pre-filter (0 = off): pairs below it (and above -1) cannot reach ani_th
  float cfrac; // jmin / (1 + jmin): dot >= cfrac * (norm_r + norm_q) is the same bound, division-free
  int symmetric;
  hg_hit *__restrict__ hits;
  unsigned long long cap;
  unsigned long long *__restrict__ n_hits;
};

// Called by every lane of a warp (converged) with its own candidate; `live` marks lanes
// whose (li, lj) is inside the matrices.  Survivors are appended with one atomic per warp.
// QF: the threshold, its ref-index tie bound and the pre-filter of query column lj come from fl (a search pass,
// hg_floor) instead of e.ani_th / e.jmin.
template <bool QF = false>
__device__ __forceinline__ void dist_emit(const DistEpilogue &e, bool live, uint32_t li, uint32_t lj, int32_t dot,
                                          const hg_floors &fl = {}) {
  bool keep = false;
  float ani = 0.0f;
  uint32_t gi = 0, gj = 0;
  if (live) {
    gi = e.i0 + li;
    gj = e.j0 + lj;
    if (!e.symmetric || gj > gi) {  // dist.rs:253-265: only j > i when ref == query
      const int32_t nr = e.ref_norm[li], nq = e.qry_norm[lj];
      float th = e.ani_th, jmin = e.jmin;
      uint32_t imax = 0;
      if constexpr (QF) { const hg_floor f = fl.q[lj]; th = f.ani; jmin = f.jmin; imax = f.imax; }
      bool cand = true;
      if (jmin > 0.0f) {  // cheap monotone bound first; the exact f32 sequence decides
        const int32_t den = (int32_t)((uint32_t)nr + (uint32_t)nq - (uint32_t)dot);
        const float fd = __int2float_rn(dot), fn = __int2float_rn(den);
        cand = den <= 0 || fd >= jmin * fn || fd <= -fn;  // the last: J <= -1, ANI 100 (DESIGN.md, dist epilogue)
      }
      if (cand) {
        ani = ani_from_dot(dot, nr, nq, e.ksize_f);
        if constexpr (QF) keep = ani > th || (ani == th && gi <= imax);
        else keep = ani >= th;
      }
    }
  }
  const uint32_t bal = __ballot_sync(0xffffffffu, keep);
  if (bal == 0) return;
  const uint32_t lane = threadIdx.x & 31;
  unsigned long long base = 0;
  if (lane == (uint32_t)(__ffs(bal) - 1)) base = atomicAdd(e.n_hits, (unsigned long long)__popc(bal));
  base = __shfl_sync(0xffffffffu, base, __ffs(bal) - 1);
  if (keep) {
    const unsigned long long idx = base + __popc(bal & ((1u << lane) - 1u));
    if (idx < e.cap) {
      hg_hit h;
      h.i = gi; h.j = gj; h.dot = dot; h.ani = ani;
      e.hits[idx] = h;
    }
  }
}

// The same decision without the append: used by the tensor kernels' candidate lists, which evaluate a whole list first
// and then reserve room for all its survivors with ONE atomic (the counter may live on another GPU: a round trip over
// NVLink per 32 candidates is what made remote members slow).
template <bool QF = false>
__device__ __forceinline__ bool dist_eval(const DistEpilogue &e, bool live, uint32_t li, uint32_t lj, int32_t dot, float *ani_out,
                                          const hg_floors &fl = {}) {
  if (!live) return false;
  const uint32_t gi = e.i0 + li, gj = e.j0 + lj;
  if (e.symmetric && gj <= gi) return false;
  const int32_t nr = e.ref_norm[li], nq = e.qry_norm[lj];
  float th = e.ani_th, jmin = e.jmin;
  uint32_t imax = 0;
  if constexpr (QF) { const hg_floor f = fl.q[lj]; th = f.ani; jmin = f.jmin; imax = f.imax; }
  if (jmin > 0.0f) {
    const int32_t den = (int32_t)((uint32_t)nr + (uint32_t)nq - (uint32_t)dot);
    const float fd = __int2float_rn(dot), fn = __int2float_rn(den);
    if (!(den <= 0 || fd >= jmin * fn || fd <= -fn)) return false;
  }
  const float ani = ani_from_dot(dot, nr, nq, e.ksize_f);
  *ani_out = ani;
  if constexpr (QF) return ani > th || (ani == th && gi <= imax);
  return ani >= th;
}

// ---- dense output (hg_dense): the exact dot of every live pair, no threshold ----
// cells of global row gi owned by query columns gj, gj + 1, ... up to 16: how many are live (inside the launch's
// columns, and below the diagonal in a lower triangle)
__device__ __forceinline__ uint32_t dense_live(const hg_dense &d, const DistEpilogue &e, uint32_t gi, uint32_t gj) {
  uint32_t end = e.j0 + e.n_qry;
  if (!d.ld && gi < end) end = gi;
  return gj >= end ? 0u : min(16u, end - gj);
}
__device__ __forceinline__ int32_t *dense_cell(const hg_dense &d, uint32_t gi, uint32_t gj) {
  return d.base + (hg_dense_row(d, gi) - hg_dense_row(d, d.row_base)) + gj;
}
// the first n of 16 consecutive cells of row gi from column gj: four 16-byte stores when all 16 are live and aligned
__device__ __forceinline__ void dense_store16(const hg_dense &d, uint32_t gi, uint32_t gj, uint32_t n, const int32_t (&v)[16]) {
  int32_t *p = dense_cell(d, gi, gj);
  if (n == 16 && ((uintptr_t)p & 15) == 0) {
#pragma unroll
    for (int t = 0; t < 4; ++t) reinterpret_cast<int4 *>(p)[t] = make_int4(v[4 * t], v[4 * t + 1], v[4 * t + 2], v[4 * t + 3]);
    return;
  }
#pragma unroll
  for (int j = 0; j < 16; ++j)
    if ((uint32_t)j < n) p[j] = v[j];
}

// ---- arrival flags of a multi-GPU launch (hg_tile_feed) ----
__device__ __forceinline__ unsigned long long feed_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// timeline stamp i of a multi-GPU launch (measurement support): first writer wins for "first", atomicMax for "last"
__device__ __forceinline__ void feed_stamp(unsigned long long *dbg, int i) {
  if (dbg) dbg[i] = feed_ns();
}
__device__ __forceinline__ void feed_stamp_max(unsigned long long *dbg, int i) {
  if (dbg) atomicMax(dbg + i, feed_ns());
}
// whole warp, converged: returns once every flag in `need` is set (`have` caches what has been seen)
__device__ __forceinline__ void feed_wait(const hg_tile_feed &f, uint32_t need, uint32_t &have) {
  if ((have & need) == need) return;
  const uint32_t lane = threadIdx.x & 31;
  const unsigned long long t0 = feed_ns();
  for (;;) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f.ready + lane) : "memory");
    have |= __ballot_sync(0xffffffffu, (int32_t)(v - f.seq) >= 0);
    if ((have & need) == need) break;
    if (feed_ns() - t0 > f.timeout_ns) {  // a member never delivered: flag the error, stop waiting for good
      if (lane == 0) atomicExch(f.status, 1u);
      have = 0xffffffffu;
      break;
    }
    __nanosleep(200);
  }
  asm volatile("fence.proxy.async;" ::: "memory");  // the TMA (async proxy) reads that follow see what the flags published
}
// whole warp, converged: one look at the flags, no waiting
__device__ __forceinline__ bool feed_poll(const hg_tile_feed &f, uint32_t need, uint32_t &have) {
  if ((have & need) == need) return true;
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f.ready + (threadIdx.x & 31)) : "memory");
  have |= __ballot_sync(0xffffffffu, (int32_t)(v - f.seq) >= 0);
  return (have & need) == need;
}

// whole warp, converged: returns once every member in f.start_need has raised its start flag
__device__ __forceinline__ void feed_wait_start(const hg_tile_feed &f) {
  const uint32_t lane = threadIdx.x & 31;
  const unsigned long long t0 = feed_ns();
  for (;;) {
    uint32_t v = f.seq;
    if (lane < HG_MAX_PEERS) asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f.start + lane) : "memory");
    const uint32_t have = __ballot_sync(0xffffffffu, (int32_t)(v - f.seq) >= 0);
    if ((have & f.start_need) == f.start_need) break;
    if (feed_ns() - t0 > f.timeout_ns) {
      if (lane == 0) atomicExch(f.status, 1u);
      break;
    }
    __nanosleep(200);
  }
}

// One pusher warp's share of this member's pushes (hg_push_plan); `me` of `n_pushers` warps in the grid.
__device__ __forceinline__ void push_my_units(const hg_push_plan *__restrict__ pp, uint32_t me, uint32_t n_pushers) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t seq = *pp->seq;
  const int rank = pp->rank, world = pp->world;
  const size_t tid = (size_t)me * 32 + lane, nth = (size_t)n_pushers * 32;
  for (int u = 0; u < pp->n_units; ++u) {
    const int set = pp->unit_set[u];
    const uint32_t dest = pp->unit_dest[u];
    for (int k = 0; k < pp->n[set]; ++k) {
      const uint64_t off = pp->off[set][k];
      uint32_t bytes = pp->bytes[set][k];
      if (set == HG_PUSH_START_SET && k == 0 && pp->dyn_count) {  // only the outlier entries that exist (usually a handful)
        const uint32_t used = *pp->dyn_count - pp->dyn_base;      // (a cursor past the capacity means "declined": nothing to send)
        bytes = used * 4u <= bytes ? ((used * 4u + 15u) & ~15u) : 0u;
      }
      if (((off | bytes) & 15) == 0) {
        const uint4 *src = reinterpret_cast<const uint4 *>(pp->win[rank] + off);
        const size_t n16 = bytes / 16;
        for (size_t i = tid; i < n16; i += 12 * nth) {  // twelve loads in flight per lane, then their stores to the destinations
          uint4 v[12];
#pragma unroll
          for (int t = 0; t < 12; ++t)
            if (i + t * nth < n16) v[t] = src[i + t * nth];
#pragma unroll
          for (int t = 0; t < 12; ++t)
            if (i + t * nth < n16)
              for (int m = 0; m < world; ++m)
                if (dest >> m & 1u) reinterpret_cast<uint4 *>(pp->win[m] + off)[i + t * nth] = v[t];
        }
      } else {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(pp->win[rank] + off);
        for (size_t i = tid; i < bytes / 4; i += nth) {
          const uint32_t v = src[i];
          for (int m = 0; m < world; ++m)
            if (dest >> m & 1u) reinterpret_cast<uint32_t *>(pp->win[m] + off)[i] = v;
        }
      }
    }
    // the last pusher warp of the grid through with this unit raises its flag in the destination windows: one lane per
    // window, all release stores in flight together (one after the other they cost an NVLink round trip each)
    __threadfence_system();
    __syncwarp();
    uint32_t prev = 0;
    if (lane == 0) prev = atomicAdd(pp->done + u, 1u);
    prev = __shfl_sync(0xffffffffu, prev, 0);
    if (prev == n_pushers - 1) {
      __threadfence_system();  // (acquire side of the counter: the other warps' stores are ordered before the flags below)
      if (lane == 0) {
        pp->done[u] = 0;
        if (pp->unit_stamp[u] >= 0) feed_stamp(pp->dbg, pp->unit_stamp[u]);
      }
      if ((int)lane < world && (dest >> lane & 1u)) {
        uint32_t *f = set == HG_PUSH_START_SET ? reinterpret_cast<uint32_t *>(pp->win[lane] + pp->start_off) + rank
                                               : reinterpret_cast<uint32_t *>(pp->win[lane] + pp->ready_off) + (rank * HG_PUSH_CHUNKS + set);
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(seq) : "memory");
      }
    }
    __syncwarp();
  }
}

// The Jaccard value below which ANI (dist.rs:154) cannot reach ani_th, lowered by a safety
// margin (0.01 ANI points and 0.1 % relative) that dwarfs every f32 rounding in the exact path.
// Host for a scalar threshold; device for the per-query floors of a search pass.
__host__ __device__ inline float dist_jmin(float ani_th, uint32_t ksize) {
  const double a = (double)ani_th / 100.0 - 1e-4;
  if (!(a > 0.0)) return 0.0f;            // everything (ani >= 0 always) must be evaluated exactly
  if (a >= 1.0) return 1e30f;             // ani is clamped to 100: nothing can pass, J bound irrelevant
  const double E = exp((double)ksize * (a - 1.0));  // 2J/(1+J) = E
  const double J = E / (2.0 - E);
  return (float)(J * (1.0 - 1e-3));
}

}  // namespace hg
