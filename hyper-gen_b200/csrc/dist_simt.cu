// dist_simt.cu — CUDA-core dist path: exact i16 x i16 -> i32 dot products of every
// ref x query pair with the fused ANI / threshold epilogue.
//
// Replaces the pair loop of dist::compute_hv_ani + compute_pairwise_ani (reference
// src/dist.rs:139-161,231-294).  This is the path taken when an HV element does not fit the
// 13-bit budget of the int8 limb split used on the tensor pipe (dist_tc.cu), when the
// problem is too small to fill a tensor tile, or when the caller forces it (path = 1); the
// reason is recorded in hg_dist_last_reason().  Exact for any i16 input: accumulation is
// wrapping i32 like the reference's `i32` sum (dist.rs:147-151).
//
// 64 x 64 output tile per CTA (256 threads, 4 x 4 outputs each), 64-deep K slabs staged in
// padded shared memory (144-byte rows: conflict-free 16-byte reads for 8-lane phases).
#include "dist_common.cuh"

namespace {

constexpr int DS_TILE = 64;
constexpr int DS_KS = 64;                 // int16 per K slab
constexpr int DS_ROW_BYTES = DS_KS * 2 + 16;
constexpr int DS_THREADS = 256;

__device__ __forceinline__ void mac8(int32_t &acc, const uint4 &a, const uint4 &b) {
  const uint32_t av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int32_t alo = (int32_t)(int16_t)(av[i] & 0xFFFFu), ahi = (int32_t)av[i] >> 16;
    const int32_t blo = (int32_t)(int16_t)(bv[i] & 0xFFFFu), bhi = (int32_t)bv[i] >> 16;
    acc += alo * blo;  // wraps like the reference's i32 accumulator
    acc += ahi * bhi;
  }
}

// QF: per-query thresholds (a search pass); `fl` is not read otherwise.  DENSE: every live pair's dot to its cell of `dn`
// (hg_dense), no threshold; `fl` and the hit fields of `ep` are not read.
template <bool QF, bool DENSE>
__device__ __forceinline__ void simt_body(const int16_t *__restrict__ ref, const int16_t *__restrict__ qry, uint32_t hv_d,
                                          hg::DistEpilogue ep, hg_floors fl, hg_dense dn) {
  __shared__ __align__(16) unsigned char s_a[DS_TILE * DS_ROW_BYTES];
  __shared__ __align__(16) unsigned char s_b[DS_TILE * DS_ROW_BYTES];

  const uint32_t row0 = blockIdx.y * DS_TILE, col0 = blockIdx.x * DS_TILE;
  // symmetric: a tile whose largest global j is not above its smallest global i is empty
  if (ep.symmetric && (uint64_t)ep.j0 + col0 + DS_TILE - 1 <= (uint64_t)ep.i0 + row0) return;
  // lower triangle: a tile with no j < i
  if (DENSE && !dn.ld && (uint64_t)ep.j0 + col0 >= (uint64_t)ep.i0 + row0 + DS_TILE - 1) return;

  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  int32_t acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0;

  // loader mapping: 8 threads per row (16 B each = 128 B of K), 32 rows per pass, 2 passes
  const int lrow = tid >> 3, lseg = tid & 7;

  for (uint32_t k0 = 0; k0 < hv_d; k0 += DS_KS) {
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const int r = lrow + 32 * pass;
      uint4 va = make_uint4(0, 0, 0, 0), vb = make_uint4(0, 0, 0, 0);
      if (row0 + r < ep.n_ref)
        va = *reinterpret_cast<const uint4 *>(ref + (size_t)(row0 + r) * hv_d + k0 + lseg * 8);
      if (col0 + r < ep.n_qry)
        vb = *reinterpret_cast<const uint4 *>(qry + (size_t)(col0 + r) * hv_d + k0 + lseg * 8);
      *reinterpret_cast<uint4 *>(s_a + r * DS_ROW_BYTES + lseg * 16) = va;
      *reinterpret_cast<uint4 *>(s_b + r * DS_ROW_BYTES + lseg * 16) = vb;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < DS_KS / 8; ++kk) {
      uint4 a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const uint4 *>(s_a + (ty + 16 * i) * DS_ROW_BYTES + kk * 16);
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = *reinterpret_cast<const uint4 *>(s_b + (tx + 16 * j) * DS_ROW_BYTES + kk * 16);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) mac8(acc[i][j], a[i], b[j]);
    }
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t li = row0 + ty + 16 * i, lj = col0 + tx + 16 * j;
      if constexpr (DENSE) {
        const uint32_t gi = ep.i0 + li, gj = ep.j0 + lj;
        if (li < ep.n_ref && lj < ep.n_qry && (dn.ld || gj < gi)) *hg::dense_cell(dn, gi, gj) = acc[i][j];
      } else {
        hg::dist_emit<QF>(ep, li < ep.n_ref && lj < ep.n_qry, li, lj, acc[i][j], fl);
      }
    }
}

template <bool QF>
__global__ void __launch_bounds__(DS_THREADS)
dist_simt_kernel(const int16_t *__restrict__ ref, const int16_t *__restrict__ qry, uint32_t hv_d,
                 hg::DistEpilogue ep, hg_floors fl) {
  simt_body<QF, false>(ref, qry, hv_d, ep, fl, hg_dense{});
}

__global__ void __launch_bounds__(DS_THREADS)
dist_simt_dense_kernel(const int16_t *__restrict__ ref, const int16_t *__restrict__ qry, uint32_t hv_d, hg::DistEpilogue ep,
                       hg_dense dn) {
  simt_body<false, true>(ref, qry, hv_d, ep, hg_floors{}, dn);
}

}  // namespace

int hg_launch_dist_simt(hg_ctx *ctx, const int16_t *d_ref, const int32_t *d_ref_norm, uint32_t n_ref, uint32_t i0,
                        const int16_t *d_qry, const int32_t *d_qry_norm, uint32_t n_qry, uint32_t j0,
                        uint32_t hv_d, uint32_t ksize, float ani_th, int symmetric, hg_hit *d_hits, uint64_t cap,
                        unsigned long long *d_n_hits, const hg_floors *floors, const hg_dense *dense) {
  if (n_ref == 0 || n_qry == 0) return HG_OK;
  if (hv_d % DS_KS != 0) {
    hg_set_error("hv_d %u must be a multiple of %d", hv_d, DS_KS);
    return HG_E_INVALID;
  }
  hg::DistEpilogue ep;
  ep.ref_norm = d_ref_norm; ep.qry_norm = d_qry_norm;
  ep.n_ref = n_ref; ep.n_qry = n_qry; ep.i0 = i0; ep.j0 = j0;
  ep.ksize_f = (float)ksize; ep.ani_th = ani_th; ep.symmetric = symmetric;
  ep.jmin = hg::dist_jmin(ani_th, ksize);
  ep.cfrac = ep.jmin > 0.0f ? (float)((double)ep.jmin / (1.0 + (double)ep.jmin)) : 0.0f;
  ep.hits = d_hits; ep.cap = cap; ep.n_hits = d_n_hits;
  const uint32_t gx = (n_qry + DS_TILE - 1) / DS_TILE, gy_total = (n_ref + DS_TILE - 1) / DS_TILE;
  // gridDim.y <= 65535: slice the rows if a shard is taller than 4.19 M sketches
  for (uint32_t y0 = 0; y0 < gy_total; y0 += 65535) {
    const uint32_t gy = gy_total - y0 < 65535 ? gy_total - y0 : 65535;
    hg::DistEpilogue e2 = ep;
    e2.ref_norm = d_ref_norm + (size_t)y0 * DS_TILE;
    e2.n_ref = n_ref - y0 * DS_TILE;
    e2.i0 = i0 + y0 * DS_TILE;
    if (dense)
      dist_simt_dense_kernel<<<dim3(gx, gy), DS_THREADS, 0, ctx->stream>>>(d_ref + (size_t)y0 * DS_TILE * hv_d, d_qry, hv_d, e2, *dense);
    else if (floors)
      dist_simt_kernel<true><<<dim3(gx, gy), DS_THREADS, 0, ctx->stream>>>(d_ref + (size_t)y0 * DS_TILE * hv_d, d_qry, hv_d, e2,
                                                                           *floors);
    else
      dist_simt_kernel<false><<<dim3(gx, gy), DS_THREADS, 0, ctx->stream>>>(d_ref + (size_t)y0 * DS_TILE * hv_d, d_qry, hv_d, e2,
                                                                            hg_floors{});
    ctx->launches++;
  }
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}
