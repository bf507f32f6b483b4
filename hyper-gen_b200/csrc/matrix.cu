// matrix.cu — the second half of an ANI matrix band (hg_ani_matrix_*, DESIGN.md §4.11): the dist kernels' dense mode
// left the exact i32 dot of every pair in its cell; this turns each cell into ani_from_dot in place (f32 and i32 have
// the same width).  One code path for every kernel, so the matrix is bit for bit what hg_dist reports at ani_th = 0.
#include "dist_common.cuh"

namespace {

constexpr int CV_THREADS = 256;
constexpr uint32_t CV_CHUNK = 4 * CV_THREADS;  // cells of one row one block converts in one pass

// The band's rows cut into chunks of CV_CHUNK cells (rows of a lower triangle grow by one cell each: the chunks past a
// row's end are empty), chunks dealt to the blocks in turn, consecutive threads on consecutive cells.  So a band of a
// few very wide rows spreads over every block as a band of many short ones does.
__global__ void __launch_bounds__(CV_THREADS)
ani_convert_kernel(hg_dense d, uint32_t a, uint32_t h, uint32_t n_cols, uint32_t chunks_per_row, const int32_t *__restrict__ ref_norm,
                   const int32_t *__restrict__ qry_norm, float ksize_f) {
  const uint64_t total = (uint64_t)h * chunks_per_row;
  for (uint64_t t = blockIdx.x; t < total; t += gridDim.x) {
    const uint32_t i = a + (uint32_t)(t / chunks_per_row), len = d.ld ? n_cols : i;
    const uint32_t j0 = (uint32_t)(t % chunks_per_row) * CV_CHUNK;
    if (j0 >= len) continue;
    const uint32_t j1 = len - j0 < CV_CHUNK ? len : j0 + CV_CHUNK;
    int32_t *p = hg::dense_cell(d, i, 0);
    const int32_t nr = ref_norm[i];
    for (uint32_t j = j0 + threadIdx.x; j < j1; j += CV_THREADS) p[j] = __float_as_int(hg::ani_from_dot(p[j], nr, qry_norm[j], ksize_f));
  }
}

}  // namespace

int hg_launch_ani_convert(hg_ctx *ctx, const hg_dense &d, uint32_t a, uint32_t h, uint32_t n_cols, const int32_t *d_ref_norm,
                          const int32_t *d_qry_norm, uint32_t ksize) {
  if (h == 0) return HG_OK;
  const uint32_t widest = d.ld ? n_cols : a + h - 1;
  if (widest == 0) return HG_OK;
  const uint32_t chunks = (widest + CV_CHUNK - 1) / CV_CHUNK;
  const uint64_t total = (uint64_t)h * chunks, cap = (uint64_t)ctx->sm_count * 8;
  ani_convert_kernel<<<(unsigned)(total < cap ? total : cap), CV_THREADS, 0, ctx->stream>>>(d, a, h, n_cols, chunks, d_ref_norm, d_qry_norm,
                                                                                           (float)ksize);
  ctx->launches++;
  HG_CUDA(cudaGetLastError());
  return HG_OK;
}
