// api.cu — the extern "C" boundary declared in include/hypergen_b200.h: context, host-buffer
// entry points (H2D / D2H inside), device-pointer entry points (inputs resident in HBM).
// Replaces the cudarc plumbing of reference src/sketch_cuda.rs:52-60,119-166.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <functional>
#include <vector>

#include "hg_common.cuh"

uint32_t hg_kmer_tile_positions();

// ---------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

void hg_set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int hg_cuda_fail(cudaError_t e, const char *what, const char *file, int line) {
  hg_set_error("CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
  return HG_E_CUDA;
}

extern "C" const char *hg_last_error(void) { return g_err; }
extern "C" const char *hg_version(void) { return "hypergen_b200 0.1 (sm_100a)"; }

// ---------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------
extern "C" int hg_init(int device, hg_ctx **out) {
  if (!out) { hg_set_error("hg_init: out is NULL"); return HG_E_INVALID; }
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    hg_set_error("hg_init: no CUDA device (%s); this library has no CPU fallback",
                 e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    return HG_E_CUDA;
  }
  if (device < 0 || device >= n) { hg_set_error("hg_init: device %d out of range (%d)", device, n); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(device));
  hg_ctx *c = new hg_ctx();
  memset(c, 0, sizeof(*c));
  c->device = device;
  hg_cluster_stats_reset(c);
  for (int i = 0; i < 5; i++) c->records_ms[i] = -1.0f;
  struct Guard { hg_ctx *c; ~Guard() { if (c) hg_destroy(c); } } guard{c};  // nothing leaks when a step below fails
  cudaDeviceProp prop;
  HG_CUDA(cudaGetDeviceProperties(&prop, device));
  c->sm_count = prop.multiProcessorCount;
  {  // highest priority: work on other streams running next to this one (the H2D copy stream of the host entries, or the
     // caller's own) must not get in front of the kernels launched here
    int lo = 0, hi = 0;
    HG_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    HG_CUDA(cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, hi));
  }
  HG_CUDA(cudaMalloc(&c->d_status, 4 * sizeof(uint32_t)));
  HG_CUDA(cudaMemset(c->d_status, 0, 4 * sizeof(uint32_t)));
  for (int i = 0; i < 8; i++) HG_CUDA(cudaEventCreate(&c->ev[i]));
  guard.c = nullptr;
  *out = c;
  return HG_OK;
}

extern "C" void hg_destroy(hg_ctx *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  for (int i = 0; i < 10; i++) if (c->ev_chunk[i]) cudaEventDestroy(c->ev_chunk[i]);
  for (int i = 0; i < 5; i++) if (c->ev_search[i]) cudaEventDestroy(c->ev_search[i]);
  for (int i = 0; i < HG_S_COUNT; i++) if (c->d_scratch[i]) cudaFree(c->d_scratch[i]);
  for (int i = 0; i < 4; i++) if (c->h_pinned[i]) cudaFreeHost(c->h_pinned[i]);
  if (c->d_status) cudaFree(c->d_status);
  for (int i = 0; i < 8; i++) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
  if (c->copy_stream) {
    cudaStreamDestroy(c->copy_stream);
    for (int i = 0; i < 2; i++) { cudaEventDestroy(c->ev_copied[i]); cudaEventDestroy(c->ev_done[i]); }
  }
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

extern "C" int hg_sync(hg_ctx *c) {
  if (!c) { hg_set_error("hg_sync: ctx is NULL"); return HG_E_INVALID; }
  HG_CUDA(cudaStreamSynchronize(c->stream));
  return HG_OK;
}

extern "C" uint64_t hg_stream_handle(hg_ctx *c) { return c ? (uint64_t)(uintptr_t)c->stream : 0; }
extern "C" uint64_t hg_launch_count(hg_ctx *c) { return c ? c->launches : 0; }

extern "C" int hg_set_profiling(hg_ctx *c, int enabled) {
  if (!c) { hg_set_error("ctx is NULL"); return HG_E_INVALID; }
  c->prof = enabled != 0;
  c->ev_used = 0;
  return HG_OK;
}

extern "C" int hg_stage_ms(hg_ctx *c, float out_ms[4]) {
  if (!c || !out_ms) { hg_set_error("hg_stage_ms: NULL argument"); return HG_E_INVALID; }
  HG_CUDA(cudaStreamSynchronize(c->stream));
  const int pairs[4][2] = {{0, 1}, {1, 2}, {2, 3}, {4, 5}};
  for (int s = 0; s < 4; s++) {
    out_ms[s] = -1.0f;
    const int a = pairs[s][0], b = pairs[s][1];
    if ((c->ev_used >> a & 1) && (c->ev_used >> b & 1)) HG_CUDA(cudaEventElapsedTime(&out_ms[s], c->ev[a], c->ev[b]));
  }
  return HG_OK;
}

extern "C" int hg_int_peak(hg_ctx *c, int which, double *lane_ops_per_s) {
  if (!c || !lane_ops_per_s) { hg_set_error("hg_int_peak: NULL argument"); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(c->device));
  void *d_sink;
  int rc;
  if ((rc = hg_scratch(c, HG_S_MISC, 256, &d_sink))) return rc;
  const uint32_t blocks = (uint32_t)c->sm_count * 8, iters = 4096;
  if ((rc = hg_launch_int_peak(c, which, 64, (uint32_t *)d_sink, blocks))) return rc;  // warm-up
  cudaEvent_t e0, e1;
  HG_CUDA(cudaEventCreate(&e0));
  HG_CUDA(cudaEventCreate(&e1));
  float best = 1e30f;
  for (int rep = 0; rep < 5; rep++) {
    HG_CUDA(cudaEventRecord(e0, c->stream));
    if ((rc = hg_launch_int_peak(c, which, iters, (uint32_t *)d_sink, blocks))) return rc;
    HG_CUDA(cudaEventRecord(e1, c->stream));
    HG_CUDA(cudaEventSynchronize(e1));
    float ms;
    HG_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    if (ms < best) best = ms;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  const double per_thread = (double)iters * 64.0 * (which == 2 ? 2.0 : 1.0);
  *lane_ops_per_s = per_thread * 256.0 * blocks / (best * 1e-3);
  return HG_OK;
}

extern "C" int hg_host_alloc(uint64_t bytes, void **out) {
  if (!out) { hg_set_error("hg_host_alloc: out is NULL"); return HG_E_INVALID; }
  *out = nullptr;
  if (bytes == 0) return HG_OK;
  HG_CUDA(cudaHostAlloc(out, bytes, cudaHostAllocPortable));
  return HG_OK;
}

extern "C" int hg_host_free(void *p) {
  if (p) HG_CUDA(cudaFreeHost(p));
  return HG_OK;
}

extern "C" int hg_host_register(void *p, uint64_t bytes, void **dev_ptr) {
  if (!p || !dev_ptr) { hg_set_error("hg_host_register: NULL argument"); return HG_E_INVALID; }
  *dev_ptr = nullptr;
  HG_CUDA(cudaHostRegister(p, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped));
  HG_CUDA(cudaHostGetDevicePointer(dev_ptr, p, 0));
  return HG_OK;
}

extern "C" int hg_host_unregister(void *p) {
  if (p) HG_CUDA(cudaHostUnregister(p));
  return HG_OK;
}

int hg_scratch(hg_ctx *c, int slot, size_t bytes, void **out) {
  if (bytes == 0) bytes = 256;
  if (c->d_scratch_bytes[slot] < bytes) {
    HG_CUDA(cudaStreamSynchronize(c->stream));
    if (c->d_scratch[slot]) HG_CUDA(cudaFree(c->d_scratch[slot]));
    c->d_scratch[slot] = nullptr;
    c->d_scratch_bytes[slot] = 0;
    size_t want = bytes + bytes / 8 + 4096;
    HG_CUDA(cudaMalloc(&c->d_scratch[slot], want));
    c->d_scratch_bytes[slot] = want;
  }
  *out = c->d_scratch[slot];
  return HG_OK;
}

int hg_scratch_keep(hg_ctx *c, int slot, size_t bytes, size_t keep, void **out) {
  if (c->d_scratch_bytes[slot] < bytes) {
    void *p = nullptr;
    const size_t want = bytes + bytes / 2 + 4096;
    HG_CUDA(cudaMalloc(&p, want));
    if (keep) HG_CUDA(cudaMemcpyAsync(p, c->d_scratch[slot], keep, cudaMemcpyDeviceToDevice, c->stream));
    HG_CUDA(cudaStreamSynchronize(c->stream));
    if (c->d_scratch[slot]) HG_CUDA(cudaFree(c->d_scratch[slot]));
    c->d_scratch[slot] = p;
    c->d_scratch_bytes[slot] = want;
  }
  *out = c->d_scratch[slot];
  return HG_OK;
}

int hg_pinned(hg_ctx *c, int slot, size_t bytes, void **out) {
  if (bytes == 0) bytes = 256;
  if (c->h_pinned_bytes[slot] < bytes) {
    HG_CUDA(cudaStreamSynchronize(c->stream));
    if (c->h_pinned[slot]) HG_CUDA(cudaFreeHost(c->h_pinned[slot]));
    c->h_pinned[slot] = nullptr;
    c->h_pinned_bytes[slot] = 0;
    size_t want = bytes + bytes / 8 + 4096;
    HG_CUDA(cudaMallocHost(&c->h_pinned[slot], want));
    c->h_pinned_bytes[slot] = want;
  }
  *out = c->h_pinned[slot];
  return HG_OK;
}

// the copy stream of the host-pointer entries (H2D next to the compute stream) and its events, created on first use
static int ensure_copy_stream(hg_ctx *c) {
  if (c->copy_stream) return HG_OK;
  HG_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; i++) {
    HG_CUDA(cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming));
    HG_CUDA(cudaEventCreateWithFlags(&c->ev_done[i], cudaEventDisableTiming));
  }
  for (int i = 0; i < 10; i++) HG_CUDA(cudaEventCreateWithFlags(&c->ev_chunk[i], cudaEventDisableTiming));
  return HG_OK;
}

// ---------------------------------------------------------------------------------------
// sketch
// ---------------------------------------------------------------------------------------
static int check_params(const hg_sketch_params *p) {
  if (!p) { hg_set_error("params is NULL"); return HG_E_INVALID; }
  if (p->ksize == 0 || p->ksize > 32) { hg_set_error("ksize %u out of range 1..32", (unsigned)p->ksize); return HG_E_INVALID; }
  if (p->scaled == 0) { hg_set_error("scaled must be >= 1"); return HG_E_INVALID; }
  if (p->hv_d == 0 || p->hv_d % 256 != 0) {
    hg_set_error("hv_d %u must be a positive multiple of 256 (BitPacker8x block, src/hd.rs:147)", p->hv_d);
    return HG_E_INVALID;
  }
  return HG_OK;
}

static int check_offsets(const uint64_t *off, uint32_t n, const char *name) {
  for (uint32_t g = 0; g < n; g++)
    if (off[g + 1] < off[g]) { hg_set_error("%s not monotone at %u", name, g); return HG_E_INVALID; }
  return HG_OK;
}

struct SketchPlan {
  std::vector<hg_genome_desc> desc;
  uint64_t total_slots = 0;
  uint32_t n_tiles = 0;
  uint32_t max_slots = 0;
};

// genome g = bytes [r[g].begin, r[g].begin + r[g].len) of the device sequence buffer
struct SeqRange { uint64_t begin, len; };

// the ranges of genomes that lie back to back: genome g = bytes [off[g], off[g + 1]) of a buffer whose byte off[0] sits
// at byte `base` of the device sequence buffer; off is monotone
static std::vector<SeqRange> back_to_back(const uint64_t *off, uint32_t n, uint64_t base) {
  std::vector<SeqRange> r(n);
  for (uint32_t g = 0; g < n; g++) r[g] = {off[g] - off[0] + base, off[g + 1] - off[g]};
  return r;
}

static int make_plan(const SeqRange *r, uint32_t n, const hg_sketch_params *p, SketchPlan &pl) {
  const uint32_t tile = hg_kmer_tile_positions();
  pl.desc.resize(n + 1);  // + sentinel
  pl.max_slots = 0;
  uint64_t slots_total = 0, tiles_total = 0;
  for (uint32_t g = 0; g < n; g++) {
    const uint64_t len = r[g].len;
    const uint64_t n_kmers = len >= p->ksize ? len - p->ksize + 1 : 0;
    // open-addressing table at <= 50 % load for the expected FracMinHash sample size
    uint64_t want = 2 * (len / p->scaled + 1) + 32, slots = 64;
    while (slots < want) slots <<= 1;
    if (slots > (1ull << 31)) { hg_set_error("genome %u too large for one table", g); return HG_E_UNSUPPORTED; }
    hg_genome_desc &d = pl.desc[g];
    d.seq_begin = r[g].begin;
    d.seq_len = len;
    d.table_begin = slots_total;
    d.table_mask = (uint32_t)(slots - 1);
    d.first_tile = (uint32_t)tiles_total;
    d.table_slots = (uint32_t)slots;
    d.pad_ = 0;
    slots_total += slots;
    tiles_total += (n_kmers + tile - 1) / tile;
    if (slots > pl.max_slots) pl.max_slots = (uint32_t)slots;
    if (tiles_total > 0x7fffffffull) { hg_set_error("batch too large: split it"); return HG_E_UNSUPPORTED; }
  }
  memset(&pl.desc[n], 0, sizeof(hg_genome_desc));
  pl.desc[n].first_tile = (uint32_t)tiles_total;  // sentinel: ends the kernel's forward walk
  pl.total_slots = slots_total;
  pl.n_tiles = (uint32_t)tiles_total;
  return HG_OK;
}

// stage the plan, clear the tables and hash every genome; tables/counts stay in scratch 2/3
static int run_hash_stage(hg_ctx *c, const uint8_t *d_seq, const SketchPlan &pl, uint32_t n,
                          const hg_sketch_params *p, hg_genome_desc **d_desc_out, uint64_t **d_tables_out,
                          uint32_t **d_counts_out) {
  void *d_desc, *d_tables, *d_counts, *h_desc;
  int rc;
  if ((rc = hg_scratch(c, HG_S_DESC, sizeof(hg_genome_desc) * (n + 1), &d_desc))) return rc;
  if ((rc = hg_scratch(c, HG_S_TABLES, pl.total_slots * 8, &d_tables))) return rc;
  if ((rc = hg_scratch(c, HG_S_COUNTS, sizeof(uint32_t) * n, &d_counts))) return rc;
  if ((rc = hg_pinned(c, 0, sizeof(hg_genome_desc) * (n + 1), &h_desc))) return rc;
  memcpy(h_desc, pl.desc.data(), sizeof(hg_genome_desc) * (n + 1));
  c->ev_used = 0;
  HG_PROF(c, 0);
  HG_CUDA(cudaMemcpyAsync(d_desc, h_desc, sizeof(hg_genome_desc) * (n + 1), cudaMemcpyHostToDevice, c->stream));
  HG_CUDA(cudaMemsetAsync(d_tables, 0xFF, pl.total_slots * 8, c->stream));
  HG_CUDA(cudaMemsetAsync(d_counts, 0, sizeof(uint32_t) * n, c->stream));
  HG_CUDA(cudaMemsetAsync(c->d_status, 0, 4 * sizeof(uint32_t), c->stream));
  HG_PROF(c, 1);
  if ((rc = hg_launch_kmer_hash(c, d_seq, (const hg_genome_desc *)d_desc, n, pl.n_tiles, p, nullptr,
                                (uint64_t *)d_tables, (uint32_t *)d_counts)))
    return rc;
  HG_PROF(c, 2);
  *d_desc_out = (hg_genome_desc *)d_desc;
  *d_tables_out = (uint64_t *)d_tables;
  *d_counts_out = (uint32_t *)d_counts;
  return HG_OK;
}

static int status_to_rc(const uint32_t *st) {
  if (st[0]) { hg_set_error("a genome's hash table overflowed (more distinct sampled hashes than 2x the FracMinHash expectation)"); return HG_E_CAPACITY; }
  if (st[1]) { hg_set_error("a sketch needs hv_quant_bits = 16: outside the reference's representable range (src/hd.rs:140)"); return HG_E_RANGE; }
  return HG_OK;
}

extern "C" int hg_sketch_batch_dev(hg_ctx *c, const uint8_t *d_seq, const uint64_t *seg_off, uint32_t n,
                                   const hg_sketch_params *p, int16_t *d_hv, uint8_t *d_packed,
                                   uint8_t *d_quant_bits, int32_t *d_norm2, uint32_t *d_n_hashes) {
  if (!c || !seg_off || (!d_seq && n && seg_off[n] > 0)) { hg_set_error("hg_sketch_batch_dev: NULL argument"); return HG_E_INVALID; }
  if (!d_quant_bits || !d_norm2 || !d_n_hashes) { hg_set_error("hg_sketch_batch_dev: quant_bits/norm2/n_hashes are required"); return HG_E_INVALID; }
  int rc = check_params(p);
  if (rc) return rc;
  if (n == 0) return HG_OK;
  HG_CUDA(cudaSetDevice(c->device));
  SketchPlan pl;
  if ((rc = check_offsets(seg_off, n, "seg_off")) || (rc = make_plan(back_to_back(seg_off, n, seg_off[0]).data(), n, p, pl)))
    return rc;
  hg_genome_desc *d_desc; uint64_t *d_tables; uint32_t *d_counts;
  if ((rc = run_hash_stage(c, d_seq, pl, n, p, &d_desc, &d_tables, &d_counts))) return rc;
  rc = hg_launch_encode(c, d_desc, n, d_tables, d_counts, p->hv_d, d_hv, d_packed, d_quant_bits, d_norm2, d_n_hashes);
  HG_PROF(c, 3);
  return rc;
}

// ---- stage hook: encode from explicit hash sets (hd.rs:15 takes a HashSet) ----
extern "C" int hg_encode_sets_dev(hg_ctx *c, const uint64_t *d_hashes, const uint64_t *hash_off, uint32_t n,
                                  uint32_t hv_d, int16_t *d_hv, uint8_t *d_packed, uint8_t *d_quant_bits,
                                  int32_t *d_norm2) {
  if (!c || !hash_off || !d_quant_bits || !d_norm2) { hg_set_error("hg_encode_sets_dev: NULL argument"); return HG_E_INVALID; }
  if (hv_d == 0 || hv_d % 256 != 0) { hg_set_error("hv_d %u must be a positive multiple of 256", hv_d); return HG_E_INVALID; }
  if (n == 0) return HG_OK;
  HG_CUDA(cudaSetDevice(c->device));
  std::vector<hg_genome_desc> desc(n);
  for (uint32_t g = 0; g < n; g++) {
    if (hash_off[g + 1] < hash_off[g] || hash_off[g + 1] - hash_off[g] > 0x7fffffffull) { hg_set_error("hash_off invalid at %u", g); return HG_E_INVALID; }
    memset(&desc[g], 0, sizeof(hg_genome_desc));
    desc[g].table_begin = hash_off[g];
    desc[g].table_slots = (uint32_t)(hash_off[g + 1] - hash_off[g]);
  }
  void *d_desc, *h_desc;
  int rc;
  if ((rc = hg_scratch(c, HG_S_DESC, sizeof(hg_genome_desc) * n, &d_desc))) return rc;
  if ((rc = hg_pinned(c, 0, sizeof(hg_genome_desc) * n, &h_desc))) return rc;
  memcpy(h_desc, desc.data(), sizeof(hg_genome_desc) * n);
  c->ev_used = 0;
  HG_CUDA(cudaMemcpyAsync(d_desc, h_desc, sizeof(hg_genome_desc) * n, cudaMemcpyHostToDevice, c->stream));
  HG_CUDA(cudaMemsetAsync(c->d_status, 0, 4 * sizeof(uint32_t), c->stream));
  HG_PROF(c, 2);
  rc = hg_launch_encode(c, (const hg_genome_desc *)d_desc, n, d_hashes, nullptr, hv_d, d_hv, d_packed, d_quant_bits,
                        d_norm2, nullptr);
  HG_PROF(c, 3);
  return rc;
}

// Device staging of the sketches of a host entry: hv and packed in their own slots, norm2 | n_hashes | quant_bits in
// HG_S_SMALL.  hv and packed exist only when asked for.
struct SketchOut {
  int16_t *hv = nullptr;
  uint8_t *packed = nullptr, *bits = nullptr;
  int32_t *norm2 = nullptr;
  uint32_t *n_hashes = nullptr;
};

static int sketch_out_alloc(hg_ctx *c, uint32_t n, uint32_t hv_d, bool hv, bool packed, SketchOut &o) {
  void *d_hv = nullptr, *d_packed = nullptr, *d_small;
  int rc;
  if (hv && (rc = hg_scratch(c, HG_S_HV, (size_t)n * hv_d * 2, &d_hv))) return rc;
  if (packed && (rc = hg_scratch(c, HG_S_PACKED, (size_t)n * hv_d * 2, &d_packed))) return rc;
  if ((rc = hg_scratch(c, HG_S_SMALL, (size_t)n * 12, &d_small))) return rc;
  o.hv = (int16_t *)d_hv;
  o.packed = (uint8_t *)d_packed;
  o.norm2 = (int32_t *)d_small;
  o.n_hashes = (uint32_t *)d_small + n;
  o.bits = (uint8_t *)d_small + (size_t)n * 8;
  return HG_OK;
}

// D2H of every output the caller passed a buffer for, then the batch's status (synchronises)
static int sketch_out_fetch(hg_ctx *c, const SketchOut &o, uint32_t n, uint32_t hv_d, int16_t *hv, uint8_t *packed,
                            uint8_t *quant_bits, int32_t *norm2, uint32_t *n_hashes) {
  if (hv) HG_CUDA(cudaMemcpyAsync(hv, o.hv, (size_t)n * hv_d * 2, cudaMemcpyDeviceToHost, c->stream));
  if (packed) HG_CUDA(cudaMemcpyAsync(packed, o.packed, (size_t)n * hv_d * 2, cudaMemcpyDeviceToHost, c->stream));
  if (quant_bits) HG_CUDA(cudaMemcpyAsync(quant_bits, o.bits, n, cudaMemcpyDeviceToHost, c->stream));
  if (norm2) HG_CUDA(cudaMemcpyAsync(norm2, o.norm2, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (n_hashes) HG_CUDA(cudaMemcpyAsync(n_hashes, o.n_hashes, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  return hg_sketch_status(c);
}

extern "C" int hg_encode_sets(hg_ctx *c, const uint64_t *hashes, const uint64_t *hash_off, uint32_t n, uint32_t hv_d,
                              int16_t *hv, uint8_t *packed, uint8_t *quant_bits, int32_t *norm2) {
  if (!c || !hash_off) { hg_set_error("hg_encode_sets: NULL argument"); return HG_E_INVALID; }
  if (n == 0) return HG_OK;
  if (hv_d == 0 || hv_d % 256 != 0) { hg_set_error("hv_d %u must be a positive multiple of 256", hv_d); return HG_E_INVALID; }
  const uint64_t total = hash_off[n] - hash_off[0];
  if (total && !hashes) { hg_set_error("hg_encode_sets: hashes is NULL"); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(c->device));
  int rc;
  void *d_hashes;
  SketchOut o;
  if ((rc = hg_scratch(c, HG_S_TABLES, total * 8 + 64, &d_hashes))) return rc;
  if ((rc = sketch_out_alloc(c, n, hv_d, hv != nullptr, packed != nullptr, o))) return rc;
  HG_CUDA(cudaMemcpyAsync(d_hashes, hashes + hash_off[0], total * 8, cudaMemcpyHostToDevice, c->stream));
  std::vector<uint64_t> rel(n + 1);
  for (uint32_t g = 0; g <= n; g++) rel[g] = hash_off[g] - hash_off[0];
  if ((rc = hg_encode_sets_dev(c, (const uint64_t *)d_hashes, rel.data(), n, hv_d, o.hv, o.packed, o.bits, o.norm2)))
    return rc;
  return sketch_out_fetch(c, o, n, hv_d, hv, packed, quant_bits, norm2, nullptr);
}

extern "C" int hg_sketch_status(hg_ctx *c) {
  if (!c) { hg_set_error("ctx is NULL"); return HG_E_INVALID; }
  HG_CUDA(cudaMemcpyAsync(c->h_status, c->d_status, sizeof(c->h_status), cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaStreamSynchronize(c->stream));
  return status_to_rc(c->h_status);
}

// ---------------------------------------------------------------------------------------
// FASTA file bytes in (fastx_reader::read_merge_seq on the GPU)
// ---------------------------------------------------------------------------------------
uint32_t hg_fasta_block_bytes();
int hg_launch_fasta_merge(hg_ctx *ctx, const uint8_t *d_raw, const uint64_t *d_file_off, const uint64_t *d_blk_off,
                          uint32_t n_files, uint32_t max_blocks, void *d_sums, uint8_t *d_carry, uint64_t *d_out_off,
                          uint8_t *d_merged, uint64_t *d_merged_len);

// The merge of files that lie back to back in a device buffer, as in the host buffer (one copy; the kernels take any
// byte phase): per file (+ end) its offset there and its block prefix.  The merged bytes of a file land at its offset.
struct MergePlan {
  std::vector<uint64_t> off, blk;
  uint64_t max_blocks = 0;
};

// file_off is monotone
static int make_merge_plan(const uint64_t *file_off, uint32_t n, MergePlan &mp) {
  const uint32_t B = hg_fasta_block_bytes();
  mp.off.assign(n + 1, 0);
  mp.blk.assign(n + 1, 0);
  mp.max_blocks = 0;
  for (uint32_t f = 0; f < n; f++) {
    const uint64_t len = file_off[f + 1] - file_off[f];
    mp.off[f + 1] = mp.off[f] + len;
    const uint64_t nb = (len + B - 1) / B;
    mp.blk[f + 1] = mp.blk[f] + nb;
    mp.max_blocks = std::max(mp.max_blocks, nb);
  }
  if (mp.max_blocks > 0x7fffffffull) { hg_set_error("file too large"); return HG_E_UNSUPPORTED; }
  return HG_OK;
}

// Byte offsets of a merge's device metadata for up to n files and nblk blocks, in one buffer: file offsets (n+1) at 0 |
// block prefix (n+1) | out_off (nblk) | sums (16 B a block) | carry (1 B a block), then the merged lengths.  The host
// writes the first two arrays, bytes [0, out).
struct MergeLayout { size_t blk, out, sums, carry, len; };

static MergeLayout merge_layout(uint32_t n, uint64_t nblk) {
  MergeLayout L;
  L.blk = (size_t)(n + 1) * 8;
  L.out = 2 * L.blk;
  L.sums = L.out + nblk * 8;
  L.carry = L.sums + nblk * 16;
  L.len = (L.carry + nblk + 256 + 15) & ~(size_t)15;
  return L;
}

// mp's file offsets and block prefix through pinned h_meta to the head of d_meta, on the compute stream
static int put_merge_meta(hg_ctx *c, const MergePlan &mp, const MergeLayout &L, uint8_t *h_meta, uint8_t *d_meta) {
  memcpy(h_meta, mp.off.data(), mp.off.size() * 8);
  memcpy(h_meta + L.blk, mp.blk.data(), mp.blk.size() * 8);
  HG_CUDA(cudaMemcpyAsync(d_meta, h_meta, L.out, cudaMemcpyHostToDevice, c->stream));
  return HG_OK;
}

static int launch_merge(hg_ctx *c, const uint8_t *d_raw, const MergePlan &mp, const MergeLayout &L, uint8_t *d_meta,
                        uint8_t *d_merged, uint64_t *d_merged_len) {
  return hg_launch_fasta_merge(c, d_raw, (const uint64_t *)d_meta, (const uint64_t *)(d_meta + L.blk),
                               (uint32_t)(mp.off.size() - 1), (uint32_t)mp.max_blocks, d_meta + L.sums,
                               d_meta + L.carry, (uint64_t *)(d_meta + L.out), d_merged, d_merged_len);
}

// H2D of the raw files (one copy on the compute stream), merge on the device, lengths back, merged bytes back.
extern "C" int hg_fasta_merge(hg_ctx *c, const uint8_t *raw, const uint64_t *file_off, uint32_t n, uint8_t *merged,
                              uint64_t cap, uint64_t *merged_off) {
  if (!c || !file_off || !merged_off) { hg_set_error("hg_fasta_merge: NULL argument"); return HG_E_INVALID; }
  merged_off[0] = 0;
  if (n == 0) return HG_OK;
  if (!raw && file_off[n] > file_off[0]) { hg_set_error("hg_fasta_merge: raw is NULL"); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(c->device));
  MergePlan mp;
  int rc;
  if ((rc = check_offsets(file_off, n, "file_off")) || (rc = make_merge_plan(file_off, n, mp))) return rc;
  const uint64_t total = mp.off[n];
  const MergeLayout L = merge_layout(n, mp.blk[n]);
  void *d_raw, *d_merged, *d_meta, *h_meta;
  if ((rc = hg_scratch(c, HG_S_PACKED, total + 64, &d_raw))) return rc;      // raw bytes (free until the sketches are packed)
  if ((rc = hg_scratch(c, HG_S_SEQ, total + 64, &d_merged))) return rc;      // merged sequences
  if ((rc = hg_scratch(c, HG_S_MISC, L.len + (size_t)n * 8, &d_meta))) return rc;
  if ((rc = hg_pinned(c, 1, L.out + (size_t)n * 8, &h_meta))) return rc;
  uint64_t *h_len = (uint64_t *)((uint8_t *)h_meta + L.out), *d_len = (uint64_t *)((uint8_t *)d_meta + L.len);
  if ((rc = put_merge_meta(c, mp, L, (uint8_t *)h_meta, (uint8_t *)d_meta))) return rc;
  if (total) HG_CUDA(cudaMemcpyAsync(d_raw, raw + file_off[0], total, cudaMemcpyHostToDevice, c->stream));
  if ((rc = launch_merge(c, (const uint8_t *)d_raw, mp, L, (uint8_t *)d_meta, (uint8_t *)d_merged, d_len))) return rc;
  HG_CUDA(cudaMemcpyAsync(h_len, d_len, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaStreamSynchronize(c->stream));
  for (uint32_t f = 0; f < n; f++) merged_off[f + 1] = merged_off[f] + h_len[f];
  if (merged_off[n] > cap || (!merged && merged_off[n])) { hg_set_error("hg_fasta_merge: need room for %llu bytes", (unsigned long long)merged_off[n]); return HG_E_CAPACITY; }
  for (uint32_t f = 0; f < n; f++)
    if (h_len[f])
      HG_CUDA(cudaMemcpyAsync(merged + merged_off[f], (uint8_t *)d_merged + mp.off[f], h_len[f], cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaStreamSynchronize(c->stream));
  return HG_OK;
}

// ---------------------------------------------------------------------------------------
// host-pointer sketch entries: sequences or raw FASTA files in, sketches out
// ---------------------------------------------------------------------------------------
enum class Input { SEQUENCES, FASTA_FILES, FASTA_RECORDS };  // records: planned per chunk, once its records are known

// genomes [g0, g1), whose host bytes [lo, hi) are copied to byte `shift` of a staging slot
struct Chunk {
  uint32_t g0, g1;
  uint64_t lo, hi, shift;
  SketchPlan pl;
  MergePlan merge;  // FASTA files only
};

// The batch cut on genome boundaries into chunks of at most `limit` bytes (or one genome).  Sequences keep the
// caller's alignment modulo 16; FASTA files go back to back from the start of the slot, and their tiles and tables
// are planned from the raw sizes, an upper bound of the merged lengths.
static int plan_chunks(const uint8_t *host, const uint64_t *off, uint32_t n, const hg_sketch_params *p, Input in,
                       uint64_t limit, std::vector<Chunk> &chunks) {
  const bool fasta = in != Input::SEQUENCES;
  int rc = check_offsets(off, n, fasta ? "file_off" : "seg_off");
  if (rc) return rc;
  for (uint32_t g = 0; g < n;) {
    Chunk ch;
    ch.g0 = g;
    ch.lo = off[g];
    do { ++g; } while (g < n && off[g + 1] - ch.lo <= limit);
    ch.g1 = g;
    ch.hi = off[g];
    ch.shift = fasta ? 0 : (uint64_t)((uintptr_t)(host + ch.lo) & 15);
    if (fasta && (rc = make_merge_plan(off + ch.g0, ch.g1 - ch.g0, ch.merge))) return rc;
    if (in != Input::FASTA_RECORDS && (rc = make_plan(back_to_back(off + ch.g0, ch.g1 - ch.g0, ch.shift).data(), ch.g1 - ch.g0, p, ch.pl)))
      return rc;
    chunks.push_back(std::move(ch));
  }
  return HG_OK;
}

// The batch is cut into ~64 MB chunks and pipelined: chunk c+1 crosses PCIe on a copy stream (double-buffered device
// staging) while chunk c is (merged,) hashed and encoded on the compute stream; the sketches come back in one D2H at
// the end.  (Measured on B200: 32-64 MB chunks sustain the full 55 GB/s PCIe rate; 256 MB chunks drop it to 43 GB/s.)
static uint64_t hg_chunk_bytes() {
  const char *e = getenv("HG_CHUNK_MB");
  const uint64_t mb = e ? strtoull(e, nullptr, 10) : 64;
  return (mb ? mb : 64) << 20;
}

// Nothing comes back to the host between the stages of a FASTA chunk: the hash kernel reads the true merged lengths
// the merge left in HBM.
static int sketch_pipeline(hg_ctx *c, const uint8_t *host, const uint64_t *off, uint32_t n, const hg_sketch_params *p,
                           Input in, int16_t *hv, uint8_t *packed, uint8_t *quant_bits, int32_t *norm2,
                           uint32_t *n_hashes) {
  HG_CUDA(cudaSetDevice(c->device));
  const uint32_t D = p->hv_d;
  const bool fasta = in == Input::FASTA_FILES;
  std::vector<Chunk> chunks;
  int rc = plan_chunks(host, off, n, p, in, hg_chunk_bytes(), chunks);
  if (rc) return rc;
  uint64_t max_bytes = 0, max_slots = 0, max_tiles = 0, max_blk = 0;
  uint32_t max_m = 0;
  for (const Chunk &ch : chunks) {
    max_bytes = std::max(max_bytes, ch.hi - ch.lo);
    max_slots = std::max<uint64_t>(max_slots, ch.pl.total_slots);
    max_tiles = std::max<uint64_t>(max_tiles, ch.pl.n_tiles);
    max_m = std::max(max_m, ch.g1 - ch.g0);
    if (fasta) max_blk = std::max(max_blk, ch.merge.blk.back());
  }
  const uint64_t slot_bytes = (max_bytes + 64 + 255) & ~255ull;
  const size_t n_desc = (size_t)n + chunks.size();  // one sentinel per chunk
  const MergeLayout L = merge_layout(max_m, max_blk);  // one region for every chunk's merge

  // size every scratch buffer before anything is enqueued (growing one synchronises); FASTA files are staged in
  // HG_S_REF_LIMBS and merged into HG_S_SEQ
  void *d_stage, *d_merged = nullptr, *d_meta = nullptr, *d_desc, *d_tables, *d_counts, *d_map, *h_desc, *h_meta = nullptr;
  SketchOut o;
  if ((rc = hg_scratch(c, fasta ? HG_S_REF_LIMBS : HG_S_SEQ, 2 * slot_bytes, &d_stage))) return rc;
  if (fasta && (rc = hg_scratch(c, HG_S_SEQ, slot_bytes, &d_merged))) return rc;
  if (fasta && (rc = hg_scratch(c, HG_S_QRY_LIMBS, L.len + (size_t)n * 8, &d_meta))) return rc;
  if ((rc = hg_scratch(c, HG_S_DESC, sizeof(hg_genome_desc) * n_desc, &d_desc))) return rc;
  if ((rc = hg_scratch(c, HG_S_TABLES, max_slots * 8, &d_tables))) return rc;
  if ((rc = hg_scratch(c, HG_S_COUNTS, sizeof(uint32_t) * n, &d_counts))) return rc;
  if ((rc = sketch_out_alloc(c, n, D, hv != nullptr, true, o))) return rc;
  if ((rc = hg_scratch(c, HG_S_MISC, hg_kmer_map_bytes((uint32_t)max_tiles), &d_map))) return rc;
  if ((rc = hg_pinned(c, 0, sizeof(hg_genome_desc) * n_desc, &h_desc))) return rc;
  if (fasta && (rc = hg_pinned(c, 1, L.out * chunks.size(), &h_meta))) return rc;
  uint64_t *d_len = fasta ? (uint64_t *)((uint8_t *)d_meta + L.len) : nullptr;  // true merged lengths, all files
  if ((rc = ensure_copy_stream(c))) return rc;
  c->ev_used = 0;
  HG_CUDA(cudaMemsetAsync(c->d_status, 0, 4 * sizeof(uint32_t), c->stream));
  HG_CUDA(cudaMemsetAsync(d_counts, 0, sizeof(uint32_t) * n, c->stream));
  // the copy stream may not overwrite a staging slot before everything already queued is done with it
  HG_CUDA(cudaEventRecord(c->ev_done[0], c->stream));
  HG_CUDA(cudaEventRecord(c->ev_done[1], c->stream));

  size_t desc_pos = 0;
  for (size_t ci = 0; ci < chunks.size(); ci++) {
    const Chunk &ch = chunks[ci];
    const int slot = (int)(ci & 1);
    const uint32_t m = ch.g1 - ch.g0;
    uint8_t *d_in = (uint8_t *)d_stage + slot * slot_bytes;
    // ---- copy stream: the chunk in one copy (per-genome copies cost ~6 us each of PCIe idle time), once the slot's
    // previous tenant has been consumed ----
    HG_CUDA(cudaStreamWaitEvent(c->copy_stream, c->ev_done[slot], 0));
    if (ch.hi > ch.lo)
      HG_CUDA(cudaMemcpyAsync(d_in + ch.shift, host + ch.lo, ch.hi - ch.lo, cudaMemcpyHostToDevice, c->copy_stream));
    HG_CUDA(cudaEventRecord(c->ev_copied[slot], c->copy_stream));
    // ---- compute stream: merge metadata, descriptors, table clear, merge, hash, encode ----
    if (fasta && (rc = put_merge_meta(c, ch.merge, L, (uint8_t *)h_meta + ci * L.out, (uint8_t *)d_meta))) return rc;
    hg_genome_desc *hd = (hg_genome_desc *)h_desc + desc_pos, *dd = (hg_genome_desc *)d_desc + desc_pos;
    memcpy(hd, ch.pl.desc.data(), sizeof(hg_genome_desc) * (m + 1));
    desc_pos += m + 1;
    HG_CUDA(cudaMemcpyAsync(dd, hd, sizeof(hg_genome_desc) * (m + 1), cudaMemcpyHostToDevice, c->stream));
    HG_CUDA(cudaMemsetAsync(d_tables, 0xFF, ch.pl.total_slots * 8, c->stream));
    HG_CUDA(cudaStreamWaitEvent(c->stream, c->ev_copied[slot], 0));
    const uint8_t *d_seq = d_in;
    const uint64_t *d_true_len = nullptr;
    if (fasta) {
      if ((rc = launch_merge(c, d_in, ch.merge, L, (uint8_t *)d_meta, (uint8_t *)d_merged, d_len + ch.g0))) return rc;
      HG_CUDA(cudaEventRecord(c->ev_done[slot], c->stream));  // the raw slot may be overwritten now
      d_seq = (const uint8_t *)d_merged;
      d_true_len = d_len + ch.g0;
    }
    if ((rc = hg_launch_kmer_hash(c, d_seq, dd, m, ch.pl.n_tiles, p, d_true_len, (uint64_t *)d_tables,
                                  (uint32_t *)d_counts + ch.g0)))
      return rc;
    if (!fasta) HG_CUDA(cudaEventRecord(c->ev_done[slot], c->stream));
    if ((rc = hg_launch_encode(c, dd, m, (const uint64_t *)d_tables, (const uint32_t *)d_counts + ch.g0, D,
                               o.hv ? o.hv + (size_t)ch.g0 * D : nullptr, o.packed + (size_t)ch.g0 * 2 * D,
                               o.bits + ch.g0, o.norm2 + ch.g0, o.n_hashes + ch.g0)))
      return rc;
  }
  return sketch_out_fetch(c, o, n, D, hv, packed, quant_bits, norm2, n_hashes);
}

extern "C" int hg_sketch_batch(hg_ctx *c, const uint8_t *seq, const uint64_t *seg_off, uint32_t n,
                               const hg_sketch_params *p, int16_t *hv, uint8_t *packed, uint8_t *quant_bits,
                               int32_t *norm2, uint32_t *n_hashes) {
  if (!c || !seg_off) { hg_set_error("hg_sketch_batch: NULL argument"); return HG_E_INVALID; }
  int rc = check_params(p);
  if (rc) return rc;
  if (n == 0) return HG_OK;
  if (!seq && seg_off[n] > seg_off[0]) { hg_set_error("hg_sketch_batch: seq is NULL"); return HG_E_INVALID; }
  return sketch_pipeline(c, seq, seg_off, n, p, Input::SEQUENCES, hv, packed, quant_bits, norm2, n_hashes);
}

extern "C" int hg_sketch_fasta_batch(hg_ctx *c, const uint8_t *raw, const uint64_t *file_off, uint32_t n,
                                     const hg_sketch_params *p, int16_t *hv, uint8_t *packed, uint8_t *quant_bits,
                                     int32_t *norm2, uint32_t *n_hashes) {
  if (!c || !file_off) { hg_set_error("hg_sketch_fasta_batch: NULL argument"); return HG_E_INVALID; }
  int rc = check_params(p);
  if (rc) return rc;
  if (n == 0) return HG_OK;
  if (!raw && file_off[n] > file_off[0]) { hg_set_error("hg_sketch_fasta_batch: raw is NULL"); return HG_E_INVALID; }
  return sketch_pipeline(c, raw, file_off, n, p, Input::FASTA_FILES, hv, packed, quant_bits, norm2, n_hashes);
}

// ---------------------------------------------------------------------------------------
// FASTA records in: one sketch per record
// ---------------------------------------------------------------------------------------
int hg_launch_fasta_rec_count(hg_ctx *ctx, const uint8_t *d_raw, const uint64_t *d_file_off, const uint64_t *d_blk_off,
                              uint32_t n_files, uint32_t max_blocks, uint64_t n_blocks, uint32_t *d_cnt, uint64_t *d_first);
int hg_launch_fasta_rec_table(hg_ctx *ctx, const uint8_t *d_raw, const uint64_t *d_file_off, const uint64_t *d_blk_off,
                              uint32_t n_files, uint32_t max_blocks, const uint8_t *d_carry, const uint64_t *d_out_off,
                              const uint64_t *d_merged_len, const uint32_t *d_cnt, const uint64_t *d_first, uint64_t n_slots,
                              hg_fasta_record *d_rec, uint64_t *d_rec_n);

// The chunked pipeline of the per-file entry with the record index behind the merge.  A chunk's hash plan needs its
// records, so each chunk makes two round trips to the host (the header count, then the record table); the next
// chunk's H2D is queued on the copy stream before them, so PCIe stays busy.  The raw slot is released after the index
// pass, which reads the raw bytes too.  A record's range starts at its header's 'N', which adds no k-mer.
int hg_records_run(hg_ctx *c, const uint8_t *raw, const uint64_t *off, uint32_t n, const hg_sketch_params *p,
                   uint64_t rec_cap, hg_records_part &out) {
  out = hg_records_part();
  int rc = check_params(p);
  if (rc) return rc;
  for (int i = 0; i < 4; i++) c->records_stats[i] = 0;
  for (int i = 0; i < 5; i++) c->records_ms[i] = -1.0f;
  HG_CUDA(cudaSetDevice(c->device));
  const uint32_t D = p->hv_d;
  std::vector<Chunk> chunks;
  if ((rc = plan_chunks(raw, off, n, p, Input::FASTA_RECORDS, hg_chunk_bytes(), chunks))) return rc;
  uint64_t max_bytes = 0, max_blk = 0;
  uint32_t max_m = 0;
  for (const Chunk &ch : chunks) {
    max_bytes = std::max(max_bytes, ch.hi - ch.lo);
    max_m = std::max(max_m, ch.g1 - ch.g0);
    max_blk = std::max(max_blk, ch.merge.blk.back());
  }
  const uint64_t slot_bytes = (max_bytes + 64 + 255) & ~255ull;
  const MergeLayout L = merge_layout(max_m, max_blk);
  void *d_stage, *d_merged, *d_meta, *d_idx, *h_meta;
  if ((rc = hg_scratch(c, HG_S_REF_LIMBS, 2 * slot_bytes, &d_stage))) return rc;
  if ((rc = hg_scratch(c, HG_S_SEQ, slot_bytes, &d_merged))) return rc;
  if ((rc = hg_scratch(c, HG_S_QRY_LIMBS, L.len + (size_t)n * 8, &d_meta))) return rc;
  if ((rc = hg_scratch(c, HG_S_NARROW_META, (max_blk + 1) * 8 + max_blk * 4, &d_idx))) return rc;
  if ((rc = hg_pinned(c, 1, L.out * chunks.size(), &h_meta))) return rc;
  if ((rc = ensure_copy_stream(c))) return rc;
  uint8_t *meta = (uint8_t *)d_meta;
  const uint64_t *d_foff = (const uint64_t *)meta, *d_boff = (const uint64_t *)(meta + L.blk);
  uint64_t *d_len = (uint64_t *)(meta + L.len);  // merged lengths, all files
  uint64_t *d_first = (uint64_t *)d_idx;
  uint32_t *d_cnt = (uint32_t *)(d_first + max_blk + 1);
  c->ev_used = 0;
  HG_CUDA(cudaMemsetAsync(c->d_status, 0, 4 * sizeof(uint32_t), c->stream));
  HG_CUDA(cudaEventRecord(c->ev_done[0], c->stream));
  HG_CUDA(cudaEventRecord(c->ev_done[1], c->stream));
  auto copy = [&](size_t ci) -> int {
    const Chunk &ch = chunks[ci];
    const int slot = (int)(ci & 1);
    HG_CUDA(cudaStreamWaitEvent(c->copy_stream, c->ev_done[slot], 0));
    if (ch.hi > ch.lo)
      HG_CUDA(cudaMemcpyAsync((uint8_t *)d_stage + slot * slot_bytes, raw + ch.lo, ch.hi - ch.lo, cudaMemcpyHostToDevice, c->copy_stream));
    HG_CUDA(cudaEventRecord(c->ev_copied[slot], c->copy_stream));
    return HG_OK;
  };
  // Profiling: ev[0] merge [1] count pass [2] (host) [3] table pass [4] (host) [5] hash [6] encode [7].  A chunk's
  // hash and encode are read at the next chunk's first synchronisation.
  const bool prof = c->prof != 0;
  float ms[5] = {0, 0, 0, 0, 0};  // merge, index, hash, encode, host gap
  bool hash_pending = false;
  auto mark = [&](int i) { if (prof) cudaEventRecord(c->ev[i], c->stream); };
  auto span = [&](int a, int b) { float t = 0; cudaEventElapsedTime(&t, c->ev[a], c->ev[b]); return t; };
  auto read_hash = [&]() {
    if (!hash_pending) return;
    ms[4] += span(4, 5); ms[2] += span(5, 6); ms[3] += span(6, 7);
    hash_pending = false;
  };

  if ((rc = copy(0))) return rc;
  uint64_t rows = 0, slots = 0;
  std::vector<SeqRange> rng;
  for (size_t ci = 0; ci < chunks.size(); ci++) {
    const Chunk &ch = chunks[ci];
    const int slot = (int)(ci & 1);
    const uint32_t m = ch.g1 - ch.g0, max_blocks = (uint32_t)ch.merge.max_blocks;
    const uint64_t nblk = ch.merge.blk.back();
    const uint8_t *d_in = (const uint8_t *)d_stage + slot * slot_bytes;
    if (ci + 1 < chunks.size() && (rc = copy(ci + 1))) return rc;
    // ---- merge and index pass 1; the header count to the host ----
    if ((rc = put_merge_meta(c, ch.merge, L, (uint8_t *)h_meta + ci * L.out, meta))) return rc;
    HG_CUDA(cudaStreamWaitEvent(c->stream, c->ev_copied[slot], 0));
    mark(0);
    if ((rc = launch_merge(c, d_in, ch.merge, L, meta, (uint8_t *)d_merged, d_len + ch.g0))) return rc;
    mark(1);
    if ((rc = hg_launch_fasta_rec_count(c, d_in, d_foff, d_boff, m, max_blocks, nblk, d_cnt, d_first))) return rc;
    mark(2);
    void *h_x;
    if ((rc = hg_pinned(c, 3, 64, &h_x))) return rc;
    HG_CUDA(cudaMemcpyAsync(h_x, d_first + nblk, 8, cudaMemcpyDeviceToHost, c->stream));
    HG_CUDA(cudaStreamSynchronize(c->stream));
    read_hash();
    const uint64_t n_slots = *(const uint64_t *)h_x + m;
    // ---- index pass 2; the table to the host ----
    void *d_tab, *h_tab;
    if ((rc = hg_scratch(c, HG_S_TILES, n_slots * (sizeof(hg_fasta_record) + 8), &d_tab))) return rc;
    if ((rc = hg_pinned(c, 3, n_slots * sizeof(hg_fasta_record), &h_tab))) return rc;
    hg_fasta_record *d_rec = (hg_fasta_record *)d_tab;
    mark(3);
    if ((rc = hg_launch_fasta_rec_table(c, d_in, d_foff, d_boff, m, max_blocks, meta + L.carry, (const uint64_t *)(meta + L.out),
                                        d_len + ch.g0, d_cnt, d_first, n_slots, d_rec, (uint64_t *)(d_rec + n_slots))))
      return rc;
    mark(4);
    HG_CUDA(cudaEventRecord(c->ev_done[slot], c->stream));  // the raw slot may be overwritten now
    HG_CUDA(cudaMemcpyAsync(h_tab, d_rec, n_slots * sizeof(hg_fasta_record), cudaMemcpyDeviceToHost, c->stream));
    HG_CUDA(cudaStreamSynchronize(c->stream));
    if (prof) { ms[0] += span(0, 1); ms[1] += span(1, 2) + span(3, 4); ms[4] += span(2, 3); }
    slots += n_slots;
    // ---- the chunk's records (empty leading slots dropped) and their ranges in the merged bytes ----
    rng.clear();
    const hg_fasta_record *hr = (const hg_fasta_record *)h_tab;
    uint64_t pos = 0;  // merged offset of the slot inside its file
    for (uint64_t s = 0; s < n_slots; s++) {
      hg_fasta_record r = hr[s];
      if (!r.has_header) pos = 0;
      const uint64_t begin = ch.merge.off[r.file] + pos, len = r.seq_len + r.has_header;
      pos += len;
      if (!r.has_header && r.seq_len == 0) continue;
      r.file += ch.g0;
      r.name_off += ch.lo;
      out.rec.push_back(r);
      rng.push_back({begin, len});
    }
    if (out.rec.size() > 0xFFFFFFFFull) { hg_set_error("more than 2^32 - 1 records in one call"); return HG_E_UNSUPPORTED; }
    const uint32_t mr = (uint32_t)rng.size();
    if (out.rec.size() > rec_cap || mr == 0) continue;  // over capacity: count the rest, sketch nothing more
    // ---- hash and encode the chunk's records into rows [rows, rows + mr) ----
    SketchPlan pl;
    if ((rc = make_plan(rng.data(), mr, p, pl))) return rc;
    const uint64_t need = rows + mr;
    void *d_packed, *d_norm2, *d_nh, *d_bits, *d_desc, *d_tables, *d_counts, *h_desc;
    if ((rc = hg_scratch_keep(c, HG_S_PACKED, need * 2 * D, rows * 2 * D, &d_packed))) return rc;
    if ((rc = hg_scratch_keep(c, HG_S_SMALL, need * 4, rows * 4, &d_norm2))) return rc;
    if ((rc = hg_scratch_keep(c, HG_S_SORT_CNT, need * 4, rows * 4, &d_nh))) return rc;
    if ((rc = hg_scratch_keep(c, HG_S_SORT_TMP, need, rows, &d_bits))) return rc;
    if ((rc = hg_scratch(c, HG_S_DESC, sizeof(hg_genome_desc) * (mr + 1), &d_desc))) return rc;
    if ((rc = hg_scratch(c, HG_S_TABLES, pl.total_slots * 8, &d_tables))) return rc;
    if ((rc = hg_scratch(c, HG_S_COUNTS, sizeof(uint32_t) * mr, &d_counts))) return rc;
    if ((rc = hg_pinned(c, 0, sizeof(hg_genome_desc) * (mr + 1), &h_desc))) return rc;
    memcpy(h_desc, pl.desc.data(), sizeof(hg_genome_desc) * (mr + 1));
    mark(5);
    HG_CUDA(cudaMemcpyAsync(d_desc, h_desc, sizeof(hg_genome_desc) * (mr + 1), cudaMemcpyHostToDevice, c->stream));
    HG_CUDA(cudaMemsetAsync(d_tables, 0xFF, pl.total_slots * 8, c->stream));
    HG_CUDA(cudaMemsetAsync(d_counts, 0, sizeof(uint32_t) * mr, c->stream));
    const hg_genome_desc *dd = (const hg_genome_desc *)d_desc;
    if ((rc = hg_launch_kmer_hash(c, (const uint8_t *)d_merged, dd, mr, pl.n_tiles, p, nullptr, (uint64_t *)d_tables,
                                  (uint32_t *)d_counts)))
      return rc;
    mark(6);
    if ((rc = hg_launch_encode(c, dd, mr, (const uint64_t *)d_tables, (const uint32_t *)d_counts, D, nullptr,
                               (uint8_t *)d_packed + rows * 2 * D, (uint8_t *)d_bits + rows, (int32_t *)d_norm2 + rows,
                               (uint32_t *)d_nh + rows)))
      return rc;
    mark(7);
    hash_pending = prof;
    rows = need;
  }
  if (prof) {
    HG_CUDA(cudaStreamSynchronize(c->stream));
    read_hash();
    for (int i = 0; i < 5; i++) c->records_ms[i] = ms[i];
  }
  c->records_stats[0] = chunks.size();
  c->records_stats[1] = out.rec.size();
  c->records_stats[2] = slots;
  if (rows) {  // the slots hold this call's rows until the context's next entry
    out.packed = (const uint8_t *)c->d_scratch[HG_S_PACKED];
    out.norm2 = (const int32_t *)c->d_scratch[HG_S_SMALL];
    out.n_hashes = (const uint32_t *)c->d_scratch[HG_S_SORT_CNT];
    out.bits = (const uint8_t *)c->d_scratch[HG_S_SORT_TMP];
  }
  return HG_OK;
}

int hg_records_fetch(hg_ctx *c, const hg_records_part &o, uint32_t D, uint8_t *packed, uint8_t *quant_bits, int32_t *norm2,
                     uint32_t *n_hashes) {
  HG_CUDA(cudaSetDevice(c->device));
  const size_t n = o.rec.size();
  if (n && packed) HG_CUDA(cudaMemcpyAsync(packed, o.packed, n * 2 * D, cudaMemcpyDeviceToHost, c->stream));
  if (n && quant_bits) HG_CUDA(cudaMemcpyAsync(quant_bits, o.bits, n, cudaMemcpyDeviceToHost, c->stream));
  if (n && norm2) HG_CUDA(cudaMemcpyAsync(norm2, o.norm2, n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (n && n_hashes) HG_CUDA(cudaMemcpyAsync(n_hashes, o.n_hashes, n * 4, cudaMemcpyDeviceToHost, c->stream));
  return hg_sketch_status(c);
}

extern "C" int hg_sketch_fasta_records(hg_ctx *c, const uint8_t *raw, const uint64_t *file_off, uint32_t n,
                                       const hg_sketch_params *p, uint32_t rec_cap, hg_fasta_record *records,
                                       uint8_t *packed, uint8_t *quant_bits, int32_t *norm2, uint32_t *n_hashes,
                                       uint32_t *n_records) {
  if (!c || !file_off || !n_records) { hg_set_error("hg_sketch_fasta_records: NULL argument"); return HG_E_INVALID; }
  *n_records = 0;
  int rc = check_params(p);
  if (rc) return rc;
  if (n == 0) return HG_OK;
  if (!raw && file_off[n] > file_off[0]) { hg_set_error("hg_sketch_fasta_records: raw is NULL"); return HG_E_INVALID; }
  hg_records_part part;
  if ((rc = hg_records_run(c, raw, file_off, n, p, rec_cap, part))) return rc;
  *n_records = (uint32_t)part.rec.size();
  if (part.rec.size() > rec_cap) {
    hg_set_error("hg_sketch_fasta_records: %u records, rec_cap is %u", *n_records, rec_cap);
    return HG_E_CAPACITY;
  }
  if (records && !part.rec.empty()) memcpy(records, part.rec.data(), part.rec.size() * sizeof(hg_fasta_record));
  return hg_records_fetch(c, part, p->hv_d, packed, quant_bits, norm2, n_hashes);
}

extern "C" int hg_fasta_records_stats(hg_ctx *c, uint64_t counts[4], float ms[4], float *host_gap_ms) {
  if (!c || !counts || !ms || !host_gap_ms) { hg_set_error("hg_fasta_records_stats: NULL argument"); return HG_E_INVALID; }
  for (int i = 0; i < 4; i++) { counts[i] = c->records_stats[i]; ms[i] = c->records_ms[i]; }
  *host_gap_ms = c->records_ms[4];
  return HG_OK;
}

extern "C" int hg_kmer_hash(hg_ctx *c, const uint8_t *seq, const uint64_t *seg_off, uint32_t n,
                            const hg_sketch_params *p, uint64_t *hashes, uint64_t cap, uint64_t *hash_off) {
  if (!c || !seg_off || !hash_off) { hg_set_error("hg_kmer_hash: NULL argument"); return HG_E_INVALID; }
  int rc = check_params(p);
  if (rc) return rc;
  hash_off[0] = 0;
  if (n == 0) return HG_OK;
  if (!seq && seg_off[n] > 0) { hg_set_error("hg_kmer_hash: seq is NULL"); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(c->device));
  std::vector<Chunk> one;  // the whole batch, staged at once
  if ((rc = plan_chunks(seq, seg_off, n, p, Input::SEQUENCES, UINT64_MAX, one))) return rc;
  const Chunk &ch = one[0];
  void *d_seq;
  if ((rc = hg_scratch(c, HG_S_SEQ, ch.hi - ch.lo + 64, &d_seq))) return rc;
  HG_CUDA(cudaMemcpyAsync((uint8_t *)d_seq + ch.shift, seq + ch.lo, ch.hi - ch.lo, cudaMemcpyHostToDevice, c->stream));
  hg_genome_desc *d_desc; uint64_t *d_tables; uint32_t *d_counts;
  if ((rc = run_hash_stage(c, (const uint8_t *)d_seq, ch.pl, n, p, &d_desc, &d_tables, &d_counts))) return rc;
  if ((rc = hg_launch_sort_tables(c, d_desc, n, d_tables, ch.pl.max_slots))) return rc;
  std::vector<uint32_t> counts(n);
  HG_CUDA(cudaMemcpyAsync(counts.data(), d_counts, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if ((rc = hg_sketch_status(c))) return rc;  // synchronises
  uint64_t total = 0;
  for (uint32_t g = 0; g < n; g++) { total += counts[g]; hash_off[g + 1] = total; }
  if (total > cap || (!hashes && total)) { hg_set_error("hg_kmer_hash: need room for %llu hashes", (unsigned long long)total); return HG_E_CAPACITY; }
  for (uint32_t g = 0; g < n; g++)
    if (counts[g])
      HG_CUDA(cudaMemcpyAsync(hashes + hash_off[g], d_tables + ch.pl.desc[g].table_begin, (size_t)counts[g] * 8,
                              cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaStreamSynchronize(c->stream));
  return HG_OK;
}

// ---------------------------------------------------------------------------------------
// sketch format
// ---------------------------------------------------------------------------------------
extern "C" int hg_unpack_dev(hg_ctx *c, const uint8_t *d_packed, uint64_t row_stride, const uint8_t *d_bits,
                             uint32_t n, uint32_t hv_d, int16_t *d_hv) {
  if (!c || !d_packed || !d_bits || !d_hv) { hg_set_error("hg_unpack_dev: NULL argument"); return HG_E_INVALID; }
  if (hv_d == 0 || hv_d % 256 != 0 || row_stride % 4 != 0) { hg_set_error("hg_unpack_dev: hv_d %% 256 or row_stride %% 4"); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(c->device));
  return hg_launch_unpack(c, d_packed, row_stride, d_bits, n, hv_d, d_hv);
}

extern "C" int hg_unpack(hg_ctx *c, const uint8_t *packed, uint64_t row_stride, const uint8_t *bits, uint32_t n,
                         uint32_t hv_d, int16_t *hv) {
  if (!c || !packed || !bits || !hv) { hg_set_error("hg_unpack: NULL argument"); return HG_E_INVALID; }
  if (n == 0) return HG_OK;
  for (uint32_t g = 0; g < n; g++)
    if (bits[g] < 1 || bits[g] > 16 || (uint64_t)bits[g] * hv_d / 8 > row_stride) {
      hg_set_error("hg_unpack: sketch %u has hv_quant_bits %u (row_stride %llu)", g, (unsigned)bits[g], (unsigned long long)row_stride);
      return HG_E_INVALID;
    }
  HG_CUDA(cudaSetDevice(c->device));
  int rc;
  void *d_p, *d_b, *d_h;
  if ((rc = hg_scratch(c, HG_S_PACKED, (size_t)n * row_stride, &d_p))) return rc;
  if ((rc = hg_scratch(c, HG_S_SMALL, n, &d_b))) return rc;
  if ((rc = hg_scratch(c, HG_S_HV, (size_t)n * hv_d * 2, &d_h))) return rc;
  HG_CUDA(cudaMemcpyAsync(d_p, packed, (size_t)n * row_stride, cudaMemcpyHostToDevice, c->stream));
  HG_CUDA(cudaMemcpyAsync(d_b, bits, n, cudaMemcpyHostToDevice, c->stream));
  if ((rc = hg_unpack_dev(c, (const uint8_t *)d_p, row_stride, (const uint8_t *)d_b, n, hv_d, (int16_t *)d_h))) return rc;
  HG_CUDA(cudaMemcpyAsync(hv, d_h, (size_t)n * hv_d * 2, cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaStreamSynchronize(c->stream));
  return HG_OK;
}

// ---------------------------------------------------------------------------------------
// dist
// ---------------------------------------------------------------------------------------
void hg_dist_record(hg_ctx *c, int path, const char *fmt, ...) {
  c->dist_path = path;
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(c->dist_reason, sizeof(c->dist_reason), fmt, ap);
  va_end(ap);
}

// A window of a dist call's pairs: ref rows [r0, r0 + h) x query rows [c0, c0 + w) (indices into the call's ref and
// query blocks), reported with the call's global offsets (i0 + r, j0 + c).
struct DistWindow { uint32_t r0, h, c0, w; };
// A dist call that runs only these windows (a cluster or derep run, hg_cluster_* / hg_derep_*): every row is prepared
// once, then each window is launched and `after(k)` is enqueued behind the launch of window k - by every kernel branch,
// the two-limb rerun after a declined single plane included.
struct DistWindows {
  std::vector<DistWindow> win;
  std::function<int(size_t)> after;
  cudaEvent_t prepared = nullptr;  // if set: recorded once the rows are prepared, before the first window
  // The single plane's verdict is read once the rows are prepared, before the first window: a declined plane then
  // launches no window and no `after`, and the rerun starts from the state the caller left.  For hooks that are not
  // idempotent (the greedy steps of a derep run); without it the declined windows run their hooks on empty edge lists.
  bool decide_first = false;
  // An ANI matrix run (hg_ani_matrix_*): window k writes the exact dot of every pair to dense[k] (hg_dense) instead of
  // appending hits, and `before(k)` is enqueued ahead of its launch.
  const hg_dense *dense = nullptr;
  std::function<int(size_t)> before;
};

// one dist call: ref rows [i0, i0 + n_ref) against query rows [j0, j0 + n_qry), both matrices in HBM (or arriving there)
struct DistOp {
  const int16_t *ref;
  const int32_t *ref_norm;
  uint32_t n_ref, i0;
  const int16_t *qry;
  const int32_t *qry_norm;
  uint32_t n_qry, j0;
  uint32_t hv_d, ksize;
  float ani_th;
  int symmetric;
  hg_hit *hits;
  uint64_t cap;
  unsigned long long *n_hits;
  const hg_floor *floors = nullptr;  // a search's main pass: per-query thresholds in place of ani_th (hg_floors)
  const float *cfrac_row = nullptr;
  const DistWindows *windows = nullptr;  // only these windows (the ref block may lie inside the query matrix, as anywhere)
};

// The kernel a dist call tries first, chosen before anything runs.
struct DistChoice {
  int kernel;     // HG_PATH_SIMT, HG_PATH_TWO_LIMB or HG_PATH_NARROW
  bool fallback;  // the single plane may decline the rows: then two-limb if max |hv| fits the limb split, else SIMT
  char why[96];   // why this kernel (the reason of a run that had no facts to report)
};

// What a run found out on the way (the reason reports it).
struct DistFacts {
  int32_t absmax = -1;    // max |hv| once a pre-pass or a scan has produced it
  uint64_t outliers = 0;  // outlier elements the single-plane run corrects per candidate
  uint32_t chunks = 0;    // row chunks streamed from the host (0: the rows were in HBM)
};

// path: as requested (0 auto).  shape_ok: hg_tensor_shape_ok.  bits: what the caller knows about the rows - 0 for i16
// rows, the largest hv_quant_bits for packed rows.  b-bit two's-complement values are below 2^(b-1): above 10 bits no
// row fits the single s8 plane (x = 2a + s spans 510), and up to 13 bits every element fits the int8 limb split.
static int dist_choose(int path, uint32_t n_ref, uint32_t n_qry, bool shape_ok, uint32_t bits, DistChoice *ch) {
  ch->kernel = path;
  ch->fallback = false;
  snprintf(ch->why, sizeof(ch->why), "forced by caller");
  if (path != HG_PATH_AUTO) return path == HG_PATH_SIMT || shape_ok ? HG_OK : HG_E_UNSUPPORTED;  // (error set by the predicate)
  if ((uint64_t)n_ref * n_qry < 128ull * 128ull) {
    ch->kernel = HG_PATH_SIMT;
    snprintf(ch->why, sizeof(ch->why), "%u x %u pairs do not fill one 128x128 tensor tile", n_ref, n_qry);
  } else if (!shape_ok) {
    ch->kernel = HG_PATH_SIMT;
    snprintf(ch->why, sizeof(ch->why), "the tensor kernels declined this shape (hv_d <= 32768, 16-byte aligned matrices)");
  } else if (bits > 10 && bits <= 13) {
    ch->kernel = HG_PATH_TWO_LIMB;
    snprintf(ch->why, sizeof(ch->why), "hv_quant_bits <= %u fits two s8 limbs; tcgen05 kind::i8", bits);
  } else {
    ch->kernel = HG_PATH_NARROW;  // its pre-pass (one read of both matrices) tells whether the rows fit one s8 plane
    ch->fallback = true;
  }
  return HG_OK;
}

// dist_path and dist_reason of a finished run; `ran` is the kernel whose hits the call returns
static void dist_note(hg_ctx *c, const DistChoice &ch, int ran, const DistFacts &f, bool deferred) {
  static const char *const name[4] = {"", "SIMT", "tensor", "tensor-narrow"};
  char chunks[64] = "";
  if (f.chunks) snprintf(chunks, sizeof(chunks), "; %u row chunk(s) overlapping their H2D", f.chunks);
  if (ran != ch.kernel && ran == HG_PATH_TWO_LIMB)
    hg_dist_record(c, ran, "tensor: max |hv| = %d fits two s8 limbs, tcgen05 kind::i8 (one s8 plane declined: rows are not narrow)",
                   f.absmax);
  else if (ran != ch.kernel)
    hg_dist_record(c, ran, "SIMT: max |hv| = %d exceeds the 13-bit budget (%d) of the int8 limb split (one s8 plane declined)",
                   f.absmax, HG_LIMB_MAX_ABS);
  else if (ran == HG_PATH_NARROW && !deferred)
    hg_dist_record(c, ran,
                   "tensor-narrow%s: rows fit one s8 plane as x = 2a + s (max |hv| = %d, %llu outlier elements corrected per "
                   "candidate); tcgen05 kind::i8, one MMA per K step%s",
                   ch.fallback ? "" : " (forced)", f.absmax, (unsigned long long)f.outliers, chunks);
  else
    hg_dist_record(c, ran, "%s: %s%s%s", name[ran], ch.why, deferred ? " (verdict deferred to hg_dist_status)" : "", chunks);
}

// ---- host matrices streamed in row chunks: H2D of chunk c + 1 under unpack / pre-pass / dist kernel of chunk c ----
static uint32_t dist_chunk_rows(uint32_t n) {
  uint32_t rows = 0;
  if (const char *e = getenv("HG_DIST_CHUNK_ROWS")) rows = (uint32_t)std::max(0, atoi(e));
  if (rows == 0) {
    const uint32_t want = std::min<uint32_t>(8, std::max<uint32_t>(1, n / 1280));  // measured on config 3: 6-8 chunks beat 2-4
    rows = (n + want - 1) / want;
  }
  rows = std::max<uint32_t>(256, (rows + 255) & ~255u);
  if ((uint64_t)rows * 8 < n) rows = (uint32_t)((((uint64_t)n + 7) / 8 + 255) & ~255ull);  // at most 8 chunks
  return rows;
}

// The tensor dist (two-limb or single-plane kernel): the query matrix is prepared (limb split or pre-pass), then the
// ref rows chunk by chunk, each chunk launched against the query rows.  Rows already in HBM are one chunk and no
// copies.  With hr / hq the rows arrive from the host: all copies are queued first on the copy stream, so that chunk
// k + 1 crosses PCIe under the kernels of chunk k.  The ref block may lie inside the query matrix (all-vs-all on one
// matrix, or a row shard of it as hg_dist_dev gets it): then it shares the query's preparation.  When it IS the query
// matrix, chunk k is compared against the rows up to its own end (j in the chunk, i < j): the later rows are still
// on their way.  Single plane: HG_E_UNSUPPORTED, with max |hv| in f, if the rows turn out not to be narrow - unless
// `defer`: then nothing waits and hg_dist_status reads the verdict.
static int dist_tensor(hg_ctx *c, const DistOp &op, bool narrow, HostRows *hr, HostRows *hq, bool defer, DistFacts *f) {
  int rc;
  const uint32_t hv_d = op.hv_d;
  const bool in_q = op.ref >= op.qry && op.ref + (uint64_t)op.n_ref * hv_d <= op.qry + (uint64_t)op.n_qry * hv_d &&
                    (op.ref - op.qry) % hv_d == 0;
  const uint32_t r_off = in_q ? (uint32_t)((op.ref - op.qry) / hv_d) : 0u;
  const bool one = in_q && r_off == 0 && op.n_ref == op.n_qry;
  if (hr && (rc = ensure_copy_stream(c))) return rc;
  hg_narrow_mat Qm, Rm;
  hg_tc_mat Qt, Rt;
  if (narrow) {
    const size_t mq = hg_narrow_meta_bytes(op.n_qry), mr = in_q ? 0 : hg_narrow_meta_bytes(op.n_ref);
    void *meta;
    if ((rc = hg_scratch(c, HG_S_NARROW_META, mq + mr, &meta))) return rc;
    if ((rc = hg_narrow_setup(c, op.qry, op.n_qry, hv_d, HG_S_QRY_LIMBS, meta, &Qm))) return rc;
    if (!in_q && (rc = hg_narrow_setup(c, op.ref, op.n_ref, hv_d, HG_S_REF_LIMBS, (uint8_t *)meta + mq, &Rm))) return rc;
  } else {
    if ((rc = hg_tc_setup(c, op.qry, op.n_qry, hv_d, HG_S_QRY_LIMBS, &Qt))) return rc;
    if (!in_q && (rc = hg_tc_setup(c, op.ref, op.n_ref, hv_d, HG_S_REF_LIMBS, &Rt))) return rc;
  }
  const hg_narrow_mat *Rn = in_q ? &Qm : &Rm;
  const hg_tc_mat *Rl = in_q ? &Qt : &Rt;
  std::vector<std::pair<uint32_t, uint32_t>> chunks;
  const uint32_t step = hr ? dist_chunk_rows(op.n_ref) : op.n_ref;
  for (uint32_t a = 0; a < op.n_ref; a += step) chunks.push_back({a, std::min(step, op.n_ref - a)});
  if (hr) {
    auto small = [&](HostRows &S) -> int {
      HG_CUDA(cudaMemcpyAsync(S.d_norm, S.norm, (size_t)S.n * 4, cudaMemcpyHostToDevice, c->stream));
      if (S.bits) HG_CUDA(cudaMemcpyAsync(S.d_bits, S.bits, S.n, cudaMemcpyHostToDevice, c->stream));
      return HG_OK;
    };
    auto stage = [&](HostRows &S, uint32_t a, uint32_t rows, cudaEvent_t ev) -> int {
      HG_CUDA(cudaMemcpy2DAsync(S.d_stage + (size_t)a * S.width, S.width, S.base + (size_t)a * S.stride, S.stride, S.width, rows,
                                cudaMemcpyHostToDevice, c->copy_stream));
      HG_CUDA(cudaEventRecord(ev, c->copy_stream));
      return HG_OK;
    };
    if ((rc = small(*hr))) return rc;
    if (!in_q && (rc = small(*hq))) return rc;
    // the copy stream starts once the compute stream has got here (the buffers may still be in use by an earlier call)
    HG_CUDA(cudaEventRecord(c->ev_chunk[0], c->stream));
    HG_CUDA(cudaStreamWaitEvent(c->copy_stream, c->ev_chunk[0], 0));
    if (!in_q && (rc = stage(*hq, 0, op.n_qry, c->ev_chunk[1]))) return rc;
    for (size_t k = 0; k < chunks.size(); k++)
      if ((rc = stage(*hr, chunks[k].first, chunks[k].second, c->ev_chunk[2 + k]))) return rc;
  } else {
    HG_PROF(c, 4);
  }
  // rows [a, a + rows) of one matrix: once they have arrived (and packed rows are unpacked), split or pre-passed
  auto prep = [&](HostRows *S, const hg_narrow_mat *M, const hg_tc_mat *T, uint32_t a, uint32_t rows, cudaEvent_t ev) -> int {
    if (S) {
      HG_CUDA(cudaStreamWaitEvent(c->stream, ev, 0));
      int r2 = S->bits ? hg_launch_unpack(c, S->d_stage + (size_t)a * S->width, S->width, S->d_bits + a, rows, hv_d, S->d_hv + (size_t)a * hv_d)
                       : HG_OK;
      if (r2) return r2;
    }
    return narrow ? hg_narrow_prep_rows(c, M, a, rows) : hg_tc_split_rows(c, T, a, rows);
  };
  auto launch = [&](uint32_t r0, uint32_t nr, uint32_t i0, const int32_t *rn, uint32_t q0, uint32_t nq, uint32_t j0, const int32_t *qn,
                    const hg_dense *dn = nullptr) {
    const hg_floors fl = {op.floors ? op.floors + q0 : nullptr, op.cfrac_row};  // indexed like qn = qry_norm + q0
    const hg_floors *flp = op.floors ? &fl : nullptr;
    return narrow ? hg_narrow_launch(c, Rn, r0, nr, i0, rn, &Qm, q0, nq, j0, qn, op.ksize, op.ani_th, op.symmetric, op.hits, op.cap, op.n_hits, flp, dn)
                  : hg_tc_launch(c, Rl, r0, nr, i0, rn, &Qt, q0, nq, j0, qn, op.ksize, op.ani_th, op.symmetric, op.hits, op.cap, op.n_hits, flp, dn);
  };
  if (!one && (rc = prep(hq, &Qm, &Qt, 0, op.n_qry, c->ev_chunk[1]))) return rc;
  for (size_t k = 0; k < chunks.size(); k++) {
    const uint32_t a = chunks[k].first, rows = chunks[k].second;
    if ((!in_q || one) && (rc = prep(hr, Rn, Rl, a, rows, c->ev_chunk[2 + k]))) return rc;
    if (op.windows) continue;  // they run below, once every row is prepared
    rc = one ? launch(0, a + rows, op.i0, op.ref_norm, a, rows, op.j0 + a, op.qry_norm + a)
             : launch(r_off + a, rows, op.i0 + a, op.ref_norm + a, 0, op.n_qry, op.j0, op.qry_norm);
    if (rc) return rc;
  }
  const bool first = narrow && op.windows && op.windows->decide_first;
  if (op.windows) {
    if (op.windows->prepared) HG_CUDA(cudaEventRecord(op.windows->prepared, c->stream));
    if (first && (rc = hg_narrow_verdict(c, &Qm, in_q ? nullptr : &Rm, &f->absmax, &f->outliers))) return rc;
    for (size_t k = 0; k < op.windows->win.size(); k++) {
      const DistWindow &w = op.windows->win[k];
      if ((op.windows->before && (rc = op.windows->before(k))) ||
          (rc = launch(r_off + w.r0, w.h, op.i0 + w.r0, op.ref_norm + w.r0, w.c0, w.w, op.j0 + w.c0, op.qry_norm + w.c0,
                       op.windows->dense ? &op.windows->dense[k] : nullptr)) ||
          (rc = op.windows->after(k)))
        return rc;
    }
  }
  if (!hr) HG_PROF(c, 5);
  f->chunks = hr ? (uint32_t)chunks.size() : 0;
  if (!narrow || first) return HG_OK;
  if (defer) {  // the kernel itself honours the pre-pass's verdict (it does nothing when the rows are not narrow)
    c->pending_stats[0] = Qm.stats_all;
    c->pending_nsets[0] = Qm.n_sets;
    c->pending_stats[1] = in_q ? nullptr : Rm.stats_all;
    c->pending_nsets[1] = in_q ? 0 : Rm.n_sets;
    return HG_OK;
  }
  return hg_narrow_verdict(c, &Qm, in_q ? nullptr : &Rm, &f->absmax, &f->outliers);
}

// max |hv| over both matrices when no pre-pass has produced it: one read of each and one 4-byte D2H each
static int dist_absmax(hg_ctx *c, const DistOp &op, int32_t *absmax) {
  void *d_max;
  int rc;
  if ((rc = hg_scratch(c, HG_S_MISC, 256, &d_max))) return rc;
  int32_t m[2] = {0, 0};
  for (int k = 0; k < (op.qry == op.ref ? 1 : 2); ++k) {
    if ((rc = hg_launch_absmax(c, k ? op.qry : op.ref, (uint64_t)(k ? op.n_qry : op.n_ref) * op.hv_d, (int32_t *)d_max))) return rc;
    HG_CUDA(cudaMemcpyAsync(&m[k], d_max, 4, cudaMemcpyDeviceToHost, c->stream));
    HG_CUDA(cudaStreamSynchronize(c->stream));
  }
  *absmax = std::max(m[0], m[1]);
  return HG_OK;
}

// Runs the chosen kernel (streaming the rows from the host when hr / hq are given).  When the single plane declines
// and the choice allows it, the kernel max |hv| calls for runs on the same rows, complete in HBM by then.
static int dist_run(hg_ctx *c, const DistOp &op, const DistChoice &ch, HostRows *hr, HostRows *hq, bool defer) {
  DistFacts f;
  int ran = ch.kernel, rc;
  if (ran != HG_PATH_SIMT) {
    rc = dist_tensor(c, op, ran == HG_PATH_NARROW, hr, hq, defer, &f);
    if (rc == HG_E_UNSUPPORTED && ran == HG_PATH_NARROW && ch.fallback) {
      if (f.absmax < 0 && (rc = dist_absmax(c, op, &f.absmax))) return rc;  // declined before its pre-pass
      ran = f.absmax > HG_LIMB_MAX_ABS ? HG_PATH_SIMT : HG_PATH_TWO_LIMB;
      HG_CUDA(cudaMemsetAsync(op.n_hits, 0, sizeof(unsigned long long), c->stream));  // what the declined chunks appended
      rc = ran == HG_PATH_TWO_LIMB ? dist_tensor(c, op, false, nullptr, nullptr, false, &f) : HG_OK;
    } else if (rc == HG_E_UNSUPPORTED && ran == HG_PATH_NARROW && f.absmax >= 0) {
      hg_set_error("rows are not narrow (max |hv| = %d): more outlier entries than the single-plane path's budget", f.absmax);
    }
    if (rc) return rc;
  }
  if (ran == HG_PATH_SIMT) {
    HG_PROF(c, 4);
    const hg_floors fl = {op.floors, op.cfrac_row};
    const DistWindow all = {0, op.n_ref, 0, op.n_qry};
    const size_t n_win = op.windows ? op.windows->win.size() : 1;
    rc = HG_OK;
    for (size_t k = 0; k < n_win && !rc; k++) {
      const DistWindow &w = op.windows ? op.windows->win[k] : all;
      if (op.windows && op.windows->before && (rc = op.windows->before(k))) break;
      rc = hg_launch_dist_simt(c, op.ref + (size_t)w.r0 * op.hv_d, op.ref_norm + w.r0, w.h, op.i0 + w.r0, op.qry + (size_t)w.c0 * op.hv_d,
                               op.qry_norm + w.c0, w.w, op.j0 + w.c0, op.hv_d, op.ksize, op.ani_th, op.symmetric, op.hits, op.cap, op.n_hits,
                               op.floors ? &fl : nullptr, op.windows && op.windows->dense ? &op.windows->dense[k] : nullptr);
      if (!rc && op.windows) rc = op.windows->after(k);
    }
    HG_PROF(c, 5);
    if (rc) return rc;
  }
  dist_note(c, ch, ran, f, defer);
  return HG_OK;
}

extern "C" int hg_dist_dev(hg_ctx *c, const int16_t *d_ref, const int32_t *d_ref_norm, uint32_t n_ref, uint32_t i0,
                           const int16_t *d_qry, const int32_t *d_qry_norm, uint32_t n_qry, uint32_t j0,
                           uint32_t hv_d, uint32_t ksize, float ani_th, int symmetric, int path, hg_hit *d_hits,
                           uint64_t cap, unsigned long long *d_n_hits) {
  if (!c || !d_n_hits) { hg_set_error("hg_dist_dev: NULL argument"); return HG_E_INVALID; }
  c->pending_stats[0] = c->pending_stats[1] = nullptr;
  if ((n_ref && (!d_ref || !d_ref_norm)) || (n_qry && (!d_qry || !d_qry_norm)) || (cap && !d_hits)) {
    hg_set_error("hg_dist_dev: NULL argument"); return HG_E_INVALID;
  }
  if (hv_d == 0 || hv_d % 256 != 0) { hg_set_error("hg_dist_dev: hv_d %u must be a multiple of 256", hv_d); return HG_E_INVALID; }
  if (path < HG_PATH_AUTO || path > HG_PATH_NARROW) { hg_set_error("hg_dist_dev: path %d", path); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(c->device));
  HG_CUDA(cudaMemsetAsync(d_n_hits, 0, sizeof(unsigned long long), c->stream));
  if (n_ref == 0 || n_qry == 0) return HG_OK;
  c->ev_used &= ~(3 << 4);
  int rc;
  DistChoice ch;
  if ((rc = dist_choose(path, n_ref, n_qry, hg_tensor_shape_ok(hv_d, d_ref, d_qry) == HG_OK, 0, &ch))) return rc;
  const DistOp op = {d_ref, d_ref_norm, n_ref, i0, d_qry, d_qry_norm, n_qry, j0, hv_d, ksize, ani_th, symmetric, d_hits, cap, d_n_hits};
  // a caller that forces the single plane on device rows does not wait for its verdict here
  return dist_run(c, op, ch, nullptr, nullptr, path == HG_PATH_NARROW);
}

extern "C" int hg_dist_norm_flags(hg_ctx *c, const int16_t *d_hv, uint32_t n_rows, uint32_t hv_d, int path, uint32_t *d_flags) {
  if (!c || (n_rows && (!d_hv || !d_flags))) { hg_set_error("hg_dist_norm_flags: NULL argument"); return HG_E_INVALID; }
  if (path != HG_PATH_TWO_LIMB && path != HG_PATH_NARROW) { hg_set_error("hg_dist_norm_flags: path %d (2 or 3)", path); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(c->device));
  if (n_rows == 0) return HG_OK;
  int rc;
  if ((rc = hg_tensor_shape_ok(hv_d, d_hv, d_hv))) return rc;
  rc = path == HG_PATH_NARROW ? hg_narrow_norm_flags(c, d_hv, n_rows, hv_d, d_flags) : hg_tc_norm_flags(c, d_hv, n_rows, hv_d, d_flags);
  if (rc) return rc;
  HG_CUDA(cudaStreamSynchronize(c->stream));
  return HG_OK;
}

// After hg_dist_dev(path = 3): the pre-pass verdict that call did not wait for.
extern "C" int hg_dist_status(hg_ctx *c) {
  if (!c) { hg_set_error("ctx is NULL"); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(c->device));
  uint32_t st[2][4 * HG_MAX_PEERS] = {{0}, {0}};
  for (int k = 0; k < 2; ++k)
    if (c->pending_stats[k] && c->pending_nsets[k] <= HG_MAX_PEERS)
      HG_CUDA(cudaMemcpyAsync(st[k], c->pending_stats[k], 16 * c->pending_nsets[k], cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaStreamSynchronize(c->stream));
  for (int k = 0; k < 2; ++k)
    for (uint32_t t = 0; c->pending_stats[k] && t < c->pending_nsets[k]; ++t)
      if (st[k][4 * t + 3]) {
        hg_set_error("the forced single-plane dist did nothing: its rows are not narrow (outlier budget exceeded)");
        return HG_E_UNSUPPORTED;
      }
  return HG_OK;
}

extern "C" int hg_dist_last_path(hg_ctx *c) { return c ? c->dist_path : 0; }
extern "C" const char *hg_dist_last_reason(hg_ctx *c) { return c ? c->dist_reason : ""; }

int hg_hits_to_host(hg_ctx *c, hg_hit *d_hits, uint64_t n, bool sorted, hg_hit *hits, uint32_t *ani_milli) {
  int rc;
  void *d_milli = nullptr;
  if (sorted) {  // output stage on the device (src/utils.rs:262-269); unsorted: append order is unspecified
    if (ani_milli && (rc = hg_scratch(c, HG_S_MISC, n * 4 + 256, &d_milli))) return rc;
    if ((rc = hg_launch_sort_hits(c, d_hits, n, (uint32_t *)d_milli))) return rc;
  }
  HG_CUDA(cudaMemcpyAsync(hits, d_hits, n * sizeof(hg_hit), cudaMemcpyDeviceToHost, c->stream));
  if (d_milli) HG_CUDA(cudaMemcpyAsync(ani_milli, d_milli, n * 4, cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaStreamSynchronize(c->stream));
  return HG_OK;
}

// shared tail of the host-pointer dist entries: hit count back, then the output stage
static int dist_tail(hg_ctx *c, void *d_hits, void *d_cnt, hg_hit *hits, uint64_t cap, uint64_t *n_hits, bool sorted,
                     uint32_t *ani_milli) {
  unsigned long long cnt = 0;
  HG_CUDA(cudaMemcpyAsync(&cnt, d_cnt, sizeof(cnt), cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaStreamSynchronize(c->stream));
  *n_hits = cnt;
  if (cnt > cap) {
    hg_set_error("hg_dist: %llu pairs pass the threshold, capacity is %llu", cnt, (unsigned long long)cap);
    return HG_E_CAPACITY;
  }
  return cnt ? hg_hits_to_host(c, (hg_hit *)d_hits, cnt, sorted, hits, ani_milli) : HG_OK;
}

int hg_rows_to_device(hg_ctx *c, const HostRows &S, uint32_t hv_d) {
  if (S.n == 0) return HG_OK;
  HG_CUDA(cudaMemcpy2DAsync(S.d_stage, S.width, S.base, S.stride, S.width, S.n, cudaMemcpyHostToDevice, c->stream));
  HG_CUDA(cudaMemcpyAsync(S.d_norm, S.norm, (size_t)S.n * 4, cudaMemcpyHostToDevice, c->stream));
  if (!S.bits) return HG_OK;
  HG_CUDA(cudaMemcpyAsync(S.d_bits, S.bits, S.n, cudaMemcpyHostToDevice, c->stream));
  return hg_launch_unpack(c, S.d_stage, S.width, S.d_bits, S.n, hv_d, S.d_hv);
}

// Common driver of the host entries: the kernel chosen for these rows, streamed from the host when it can be, else
// after whole copies on the compute stream; then the tail.  bits: as dist_choose.
static int dist_from_host(hg_ctx *c, HostRows &R, HostRows &Q, bool same, uint32_t hv_d, uint32_t ksize, float ani_th, int symmetric,
                          int path, uint32_t bits, hg_hit *hits, uint64_t cap, uint64_t *n_hits, bool sorted, uint32_t *ani_milli) {
  int rc;
  DistChoice ch;
  if ((rc = dist_choose(path, R.n, Q.n, hg_tensor_shape_ok(hv_d, R.d_hv, Q.d_hv) == HG_OK, bits, &ch))) return rc;
  void *d_hits, *d_cnt;
  if ((rc = hg_scratch(c, HG_S_PACKED, cap * sizeof(hg_hit) + 256, &d_hits))) return rc;
  if ((rc = hg_scratch(c, HG_S_COUNTS, 256, &d_cnt))) return rc;
  bool stream_on = true;
  if (const char *e = getenv("HG_DIST_STREAM")) stream_on = atoi(e) != 0;
  // Streamed: the single plane on rows that may be narrow, and the two-limb kernel that packed rows of 11..13 bits
  // chose.  The full n x n of one matrix (both (i, j) and (j, i)) is not worth a special walk.
  const bool stream = stream_on && !(same && !symmetric) &&
                      (ch.kernel == HG_PATH_NARROW ? bits <= 10
                                                   : ch.kernel == HG_PATH_TWO_LIMB && path == HG_PATH_AUTO && hv_d % 512 == 0);
  c->pending_stats[0] = c->pending_stats[1] = nullptr;
  c->ev_used &= ~(3 << 4);
  HG_CUDA(cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long), c->stream));
  if (!stream && ((rc = hg_rows_to_device(c, R, hv_d)) || (!same && (rc = hg_rows_to_device(c, Q, hv_d))))) return rc;
  const DistOp op = {R.d_hv, R.d_norm, R.n, 0, Q.d_hv, Q.d_norm, Q.n, 0, hv_d, ksize, ani_th, symmetric, (hg_hit *)d_hits, cap,
                     (unsigned long long *)d_cnt};
  if ((rc = dist_run(c, op, ch, stream ? &R : nullptr, stream ? &Q : nullptr, false))) return rc;
  return dist_tail(c, d_hits, d_cnt, hits, cap, n_hits, sorted, ani_milli);
}

static int dist_host(hg_ctx *c, const int16_t *ref, const int32_t *ref_norm, uint32_t n_ref, const int16_t *qry,
                     const int32_t *qry_norm, uint32_t n_qry, uint32_t hv_d, uint32_t ksize, float ani_th, int symmetric,
                     int path, hg_hit *hits, uint64_t cap, uint64_t *n_hits, bool sorted, uint32_t *ani_milli) {
  if (!c || !n_hits) { hg_set_error("hg_dist: NULL argument"); return HG_E_INVALID; }
  *n_hits = 0;
  if ((n_ref && (!ref || !ref_norm)) || (n_qry && (!qry || !qry_norm)) || (cap && !hits)) {
    hg_set_error("hg_dist: NULL argument"); return HG_E_INVALID;
  }
  if (n_ref == 0 || n_qry == 0) return HG_OK;
  HG_CUDA(cudaSetDevice(c->device));
  int rc;
  const bool same = (ref == qry && ref_norm == qry_norm && n_ref == n_qry);
  const size_t rb = (size_t)n_ref * hv_d * 2, qb = same ? 0 : (size_t)n_qry * hv_d * 2;
  void *d_mat, *d_norm;
  if ((rc = hg_scratch(c, HG_S_HV, rb + qb + 512, &d_mat))) return rc;
  if ((rc = hg_scratch(c, HG_S_SMALL, ((size_t)n_ref + n_qry) * 4 + 256, &d_norm))) return rc;
  int16_t *d_ref = (int16_t *)d_mat;
  const size_t rb_al = (rb + 255) & ~(size_t)255;
  int16_t *d_qry = same ? d_ref : (int16_t *)((uint8_t *)d_mat + rb_al);
  int32_t *d_rn = (int32_t *)d_norm, *d_qn = same ? d_rn : d_rn + n_ref;
  HostRows R = {(const uint8_t *)ref, (uint64_t)hv_d * 2, (uint64_t)hv_d * 2, nullptr, ref_norm, n_ref, (uint8_t *)d_ref, nullptr, d_ref, d_rn};
  HostRows Q = {(const uint8_t *)qry, (uint64_t)hv_d * 2, (uint64_t)hv_d * 2, nullptr, qry_norm, n_qry, (uint8_t *)d_qry, nullptr, d_qry, d_qn};
  return dist_from_host(c, R, same ? R : Q, same, hv_d, ksize, ani_th, symmetric, path, 0, hits, cap, n_hits, sorted, ani_milli);
}

int hg_packed_args_check(const char *who, const hg_packed_rows &R, const hg_packed_rows &Q, uint32_t hv_d) {
  for (const hg_packed_rows *S : {&R, &Q})
    if (S->n && (!S->packed || !S->bits || !S->norm)) { hg_set_error("%s: NULL argument", who); return HG_E_INVALID; }
  if (hv_d == 0 || hv_d % 256 != 0) { hg_set_error("%s: hv_d %u must be a multiple of 256", who, hv_d); return HG_E_INVALID; }
  if (R.stride % 4 != 0 || Q.stride % 4 != 0) { hg_set_error("%s: row stride %% 4", who); return HG_E_INVALID; }
  return HG_OK;
}

int hg_packed_rows_check(const char *who, hg_packed_rows *R, hg_packed_rows *Q, uint32_t hv_d, bool *same) {
  *same = R->packed == Q->packed && R->bits == Q->bits && R->norm == Q->norm && R->n == Q->n;
  for (int k = 0; k < (*same ? 1 : 2); ++k) {
    hg_packed_rows &S = k ? *Q : *R;
    S.max_bits = 0;
    for (uint32_t g = 0; g < S.n; g++) {
      if (S.bits[g] < 1 || S.bits[g] > 16) {
        hg_set_error("%s: %s sketch %u has hv_quant_bits %u", who, k ? "query" : "ref", g, (unsigned)S.bits[g]);
        return HG_E_INVALID;
      }
      S.max_bits = std::max<uint32_t>(S.max_bits, S.bits[g]);
    }
  }
  if (*same) *Q = *R;
  if (R->width(hv_d) > R->stride || Q->width(hv_d) > Q->stride) {
    hg_set_error("%s: row stride below hv_quant_bits * hv_d / 8", who); return HG_E_INVALID;
  }
  return HG_OK;
}

int hg_packed_stage(hg_ctx *c, const hg_packed_rows &R, const hg_packed_rows &Q, bool same, uint32_t hv_d, HostRows *hr,
                    HostRows *hq) {
  const uint64_t rw = R.width(hv_d), qw = Q.width(hv_d);
  const uint32_t nq = same ? 0 : Q.n;  // rows of a second block
  const size_t rb = (size_t)R.n * hv_d * 2, rb_al = (rb + 255) & ~(size_t)255, qb = (size_t)nq * hv_d * 2;
  const size_t rp = ((size_t)R.n * rw + 255) & ~(size_t)255, qp = (size_t)nq * qw;
  int rc;
  void *d_mat, *d_small, *d_pk;
  if ((rc = hg_scratch(c, HG_S_HV, rb + qb + 512, &d_mat))) return rc;
  if ((rc = hg_scratch(c, HG_S_SMALL, ((size_t)R.n + nq) * 5 + 512, &d_small))) return rc;
  if ((rc = hg_scratch(c, HG_S_TABLES, rp + qp + 256, &d_pk))) return rc;
  int32_t *d_norm = (int32_t *)d_small;
  uint8_t *d_bits = (uint8_t *)(d_norm + R.n + nq);
  *hr = {R.packed, R.stride, rw, R.bits, R.norm, R.n, (uint8_t *)d_pk, d_bits, (int16_t *)d_mat, d_norm};
  *hq = same ? *hr
             : HostRows{Q.packed, Q.stride, qw, Q.bits, Q.norm, Q.n, (uint8_t *)d_pk + rp, d_bits + R.n,
                        (int16_t *)((uint8_t *)d_mat + rb_al), d_norm + R.n};
  return HG_OK;
}

int hg_dist_packed_run(hg_ctx *c, const hg_packed_rows &R, const hg_packed_rows &Q, bool same, uint32_t hv_d, uint32_t ksize,
                       float ani_th, int symmetric, int path, bool sorted, hg_hit *hits, uint32_t *ani_milli, uint64_t cap,
                       uint64_t *n_hits) {
  HG_CUDA(cudaSetDevice(c->device));
  int rc;
  HostRows hr, hq;
  if ((rc = hg_packed_stage(c, R, Q, same, hv_d, &hr, &hq))) return rc;
  return dist_from_host(c, hr, hq, same, hv_d, ksize, ani_th, symmetric, path, std::max(R.max_bits, Q.max_bits), hits, cap, n_hits,
                        sorted, ani_milli);
}

// `dist` straight from what the sketch file holds (FileSketch.hv bit-packed + hv_quant_bits + hv_norm_2,
// src/types.rs:224-235): only the packed bytes cross PCIe (b/16 of the i16 matrix), decompress_file_sketch
// (src/hd.rs:171-232) runs on the device, then the dist kernel and, if asked, the output-stage sort.
extern "C" int hg_dist_packed(hg_ctx *c, const uint8_t *ref_packed, uint64_t ref_stride, const uint8_t *ref_bits,
                              const int32_t *ref_norm, uint32_t n_ref, const uint8_t *qry_packed, uint64_t qry_stride,
                              const uint8_t *qry_bits, const int32_t *qry_norm, uint32_t n_qry, uint32_t hv_d, uint32_t ksize,
                              float ani_th, int symmetric, int path, int sorted, hg_hit *hits, uint32_t *ani_milli, uint64_t cap,
                              uint64_t *n_hits) {
  if (!c || !n_hits) { hg_set_error("hg_dist_packed: NULL argument"); return HG_E_INVALID; }
  *n_hits = 0;
  hg_packed_rows R = {ref_packed, ref_stride, ref_bits, ref_norm, n_ref}, Q = {qry_packed, qry_stride, qry_bits, qry_norm, n_qry};
  int rc;
  if (cap && !hits) { hg_set_error("hg_dist_packed: NULL argument"); return HG_E_INVALID; }
  if ((rc = hg_packed_args_check("hg_dist_packed", R, Q, hv_d))) return rc;
  if (n_ref == 0 || n_qry == 0) return HG_OK;
  bool same;
  if ((rc = hg_packed_rows_check("hg_dist_packed", &R, &Q, hv_d, &same))) return rc;
  return hg_dist_packed_run(c, R, Q, same, hv_d, ksize, ani_th, symmetric, path, sorted != 0, hits, ani_milli, cap, n_hits);
}

extern "C" int hg_dist(hg_ctx *c, const int16_t *ref, const int32_t *ref_norm, uint32_t n_ref, const int16_t *qry,
                       const int32_t *qry_norm, uint32_t n_qry, uint32_t hv_d, uint32_t ksize, float ani_th,
                       int symmetric, int path, hg_hit *hits, uint64_t cap, uint64_t *n_hits) {
  return dist_host(c, ref, ref_norm, n_ref, qry, qry_norm, n_qry, hv_d, ksize, ani_th, symmetric, path, hits, cap, n_hits,
                   false, nullptr);
}

extern "C" int hg_dist_sorted(hg_ctx *c, const int16_t *ref, const int32_t *ref_norm, uint32_t n_ref, const int16_t *qry,
                              const int32_t *qry_norm, uint32_t n_qry, uint32_t hv_d, uint32_t ksize, float ani_th,
                              int symmetric, int path, hg_hit *hits, uint32_t *ani_milli, uint64_t cap, uint64_t *n_hits) {
  return dist_host(c, ref, ref_norm, n_ref, qry, qry_norm, n_qry, hv_d, ksize, ani_th, symmetric, path, hits, cap, n_hits,
                   true, ani_milli);
}

extern "C" int hg_sort_hits_dev(hg_ctx *c, hg_hit *d_hits, uint64_t n, uint32_t *d_ani_milli) {
  if (!c || (n && !d_hits)) { hg_set_error("hg_sort_hits_dev: NULL argument"); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(c->device));
  return hg_launch_sort_hits(c, d_hits, n, d_ani_milli);
}

// ---------------------------------------------------------------------------------------
// search: the top_k best refs of every query (DESIGN.md §4, "Top-k search")
// ---------------------------------------------------------------------------------------

// rows of the floor pass's sample: about sqrt(top_k * n_ref) in [1024, 16384], a multiple of 256 and at least top_k;
// all of them (one pass) when that is not fewer than n_ref
static uint32_t search_sample_rows(uint32_t top_k, uint32_t n_ref) {
  const double want = std::min(16384.0, std::max(1024.0, std::sqrt((double)top_k * (double)n_ref)));
  const uint32_t s = std::max(((uint32_t)want + 255u) & ~255u, (top_k + 255u) & ~255u);
  return s < n_ref ? s : n_ref;
}

static void search_mark(hg_ctx *c, int k) {
  if (!c->prof) return;
  cudaEventRecord(c->ev_search[k], c->stream);
  c->search_ev_used |= 1 << k;
}

// One dist pass of a search: every pair that passes op's threshold(s), into the candidate scratch.  When they do not
// fit, the scratch grows to their count and the pass reruns: no candidate is dropped.
static int search_pass(hg_ctx *c, DistOp op, int path, uint32_t bits, uint64_t want, hg_hit **cand, uint64_t *n_cand) {
  int rc;
  DistChoice ch;
  if ((rc = dist_choose(path, op.n_ref, op.n_qry, hg_tensor_shape_ok(op.hv_d, op.ref, op.qry) == HG_OK, bits, &ch))) return rc;
  void *d_cnt, *d_hits;
  if ((rc = hg_scratch(c, HG_S_COUNTS, 256, &d_cnt))) return rc;
  for (;;) {
    if ((rc = hg_scratch(c, HG_S_PACKED, want * sizeof(hg_hit), &d_hits))) return rc;
    op.hits = (hg_hit *)d_hits;
    op.cap = c->d_scratch_bytes[HG_S_PACKED] / sizeof(hg_hit);
    op.n_hits = (unsigned long long *)d_cnt;
    HG_CUDA(cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long), c->stream));
    if ((rc = dist_run(c, op, ch, nullptr, nullptr, false))) return rc;
    unsigned long long cnt = 0;
    HG_CUDA(cudaMemcpyAsync(&cnt, d_cnt, sizeof(cnt), cudaMemcpyDeviceToHost, c->stream));
    HG_CUDA(cudaStreamSynchronize(c->stream));
    if (cnt <= op.cap) {
      *cand = op.hits;
      *n_cand = cnt;
      return HG_OK;
    }
    want = cnt;
    c->search_stats[3]++;
  }
}

// Exact by construction.  Floor pass: the dist kernel on s sample rows S x Q at ani_min, and per query the top_k-th
// key (ANI desc, i asc) of the sample.  S is a subset of the refs, so every member of the true top_k of query j has a
// key at least that large: the main pass over R x Q keeps exactly those pairs (hg_floors) - a superset of the answer -
// and the select kernel takes the top_k of each query from them.  With s = n_ref the first pass is the answer.
static int search_run(hg_ctx *c, const int16_t *d_ref, const int32_t *d_ref_norm, uint32_t n_ref, const int16_t *d_qry,
                      const int32_t *d_qry_norm, uint32_t n_qry, uint32_t hv_d, uint32_t ksize, uint32_t top_k, float ani_min,
                      int path, uint32_t bits, hg_hit *d_out, uint32_t *d_n_found, uint32_t *d_milli) {
  int rc;
  memset(c->search_stats, 0, sizeof(c->search_stats));
  c->search_ev_used = 0;
  c->pending_stats[0] = c->pending_stats[1] = nullptr;
  c->ev_used &= ~(3 << 4);
  if (n_qry == 0) return HG_OK;
  if (n_ref == 0) {
    HG_CUDA(cudaMemsetAsync(d_out, 0, (size_t)n_qry * top_k * sizeof(hg_hit), c->stream));
    HG_CUDA(cudaMemsetAsync(d_n_found, 0, (size_t)n_qry * 4, c->stream));
    if (d_milli) HG_CUDA(cudaMemsetAsync(d_milli, 0, (size_t)n_qry * top_k * 4, c->stream));
    HG_CUDA(cudaStreamSynchronize(c->stream));
    return HG_OK;
  }
  if (c->prof && !c->ev_search[0])
    for (int k = 0; k < 5; k++) HG_CUDA(cudaEventCreate(&c->ev_search[k]));
  const uint32_t s = search_sample_rows(top_k, n_ref);
  c->search_stats[0] = s;
  const uint64_t want = 4096 + 4ull * n_qry * top_k;  // initial candidate room; grows as the passes need
  DistOp op = {d_ref, d_ref_norm, n_ref, 0, d_qry, d_qry_norm, n_qry, 0, hv_d, ksize, ani_min, 0, nullptr, 0, nullptr};
  hg_hit *cand;
  uint64_t n_cand;
  search_mark(c, 0);
  if (s < n_ref) {
    void *d_sample, *d_fl;
    const size_t sb = ((size_t)s * hv_d * 2 + 255) & ~(size_t)255;
    if ((rc = hg_scratch(c, HG_S_SEQ, sb + (size_t)s * 4, &d_sample))) return rc;
    if ((rc = hg_scratch(c, HG_S_DESC, (size_t)n_qry * (sizeof(hg_floor) + 8) + 256, &d_fl))) return rc;
    hg_floor *floors = (hg_floor *)d_fl;
    unsigned long long *fkey = (unsigned long long *)(floors + n_qry);
    float *cfrac_row = (float *)(fkey + n_qry);
    int16_t *S = (int16_t *)d_sample;
    int32_t *Sn = (int32_t *)((uint8_t *)d_sample + sb);
    if ((rc = hg_launch_search_gather(c, d_ref, d_ref_norm, n_ref, hv_d, s, S, Sn))) return rc;
    DistOp fo = op;
    fo.ref = S;
    fo.ref_norm = Sn;
    fo.n_ref = s;
    if ((rc = search_pass(c, fo, path, bits, want, &cand, &n_cand))) return rc;
    c->search_stats[1] = n_cand;
    search_mark(c, 1);
    if ((rc = hg_launch_search_select(c, cand, n_cand, n_qry, top_k, nullptr, nullptr, nullptr, fkey))) return rc;
    if ((rc = hg_launch_search_floors(c, fkey, n_qry, ani_min, ksize, n_ref, s, floors, cfrac_row))) return rc;
    search_mark(c, 2);
    op.floors = floors;
    op.cfrac_row = cfrac_row;
  }
  if ((rc = search_pass(c, op, path, bits, want, &cand, &n_cand))) return rc;
  c->search_stats[2] = n_cand;
  search_mark(c, 3);
  if ((rc = hg_launch_search_select(c, cand, n_cand, n_qry, top_k, d_out, d_n_found, d_milli, nullptr))) return rc;
  search_mark(c, 4);
  HG_CUDA(cudaStreamSynchronize(c->stream));
  return HG_OK;
}

int hg_search_check(const char *who, uint32_t n_qry, const hg_hit *out, const uint32_t *n_found, uint32_t hv_d, uint32_t top_k,
                    int path) {
  if (n_qry && (!out || !n_found)) { hg_set_error("%s: NULL argument", who); return HG_E_INVALID; }
  if (hv_d == 0 || hv_d % 256 != 0) { hg_set_error("%s: hv_d %u must be a multiple of 256", who, hv_d); return HG_E_INVALID; }
  if (top_k < 1 || top_k > 1024) { hg_set_error("%s: top_k %u outside 1..1024", who, top_k); return HG_E_INVALID; }
  if (path < HG_PATH_AUTO || path > HG_PATH_NARROW) { hg_set_error("%s: path %d", who, path); return HG_E_INVALID; }
  return HG_OK;
}

extern "C" int hg_search_dev(hg_ctx *c, const int16_t *d_ref, const int32_t *d_ref_norm2, uint32_t n_ref, const int16_t *d_qry,
                             const int32_t *d_qry_norm2, uint32_t n_qry, uint32_t hv_d, uint32_t ksize, uint32_t top_k, float ani_min,
                             int path, hg_hit *d_out, uint32_t *d_n_found, uint32_t *d_ani_milli) {
  if (!c || (n_ref && (!d_ref || !d_ref_norm2)) || (n_qry && (!d_qry || !d_qry_norm2))) {
    hg_set_error("hg_search_dev: NULL argument"); return HG_E_INVALID;
  }
  int rc;
  if ((rc = hg_search_check("hg_search_dev", n_qry, d_out, d_n_found, hv_d, top_k, path))) return rc;
  HG_CUDA(cudaSetDevice(c->device));
  return search_run(c, d_ref, d_ref_norm2, n_ref, d_qry, d_qry_norm2, n_qry, hv_d, ksize, top_k, ani_min, path, 0, d_out, d_n_found,
                    d_ani_milli);
}

// The rows as the sketch files hold them: whole copies of the packed bytes (the live width of every row),
// decompress_file_sketch on the device (as hg_dist_packed), then the search.
int hg_search_packed_run(hg_ctx *c, const hg_packed_rows &R, const hg_packed_rows &Q, bool same, uint32_t hv_d, uint32_t ksize,
                         uint32_t top_k, float ani_min, int path, hg_hit **d_out_p, uint32_t **d_nf_p, uint32_t **d_milli_p) {
  int rc;
  HostRows hr, hq;
  if ((rc = hg_packed_stage(c, R, Q, same, hv_d, &hr, &hq))) return rc;
  const size_t n_out = (size_t)Q.n * top_k;
  void *d_res;
  if ((rc = hg_scratch(c, HG_S_TILES, n_out * (sizeof(hg_hit) + 4) + (size_t)Q.n * 4 + 256, &d_res))) return rc;
  hg_hit *d_out = (hg_hit *)d_res;
  uint32_t *d_milli = (uint32_t *)(d_out + n_out), *d_nf = d_milli + n_out;
  if ((rc = hg_rows_to_device(c, hr, hv_d)) || (!same && (rc = hg_rows_to_device(c, hq, hv_d)))) return rc;
  if ((rc = search_run(c, hr.d_hv, hr.d_norm, R.n, hq.d_hv, hq.d_norm, Q.n, hv_d, ksize, top_k, ani_min, path,
                       std::max(R.max_bits, Q.max_bits), d_out, d_nf, d_milli)))
    return rc;
  *d_out_p = d_out;
  *d_nf_p = d_nf;
  *d_milli_p = d_milli;
  return HG_OK;
}

int hg_search_packed_host(hg_ctx *c, const char *who, hg_packed_rows R, hg_packed_rows Q, uint32_t hv_d, uint32_t ksize,
                          uint32_t top_k, float ani_min, int path, hg_hit *out, uint32_t *n_found, uint32_t *ani_milli) {
  memset(c->search_stats, 0, sizeof(c->search_stats));
  const size_t n_out = (size_t)Q.n * top_k;
  if (Q.n == 0) return HG_OK;
  if (R.n == 0) {
    memset(out, 0, n_out * sizeof(hg_hit));
    memset(n_found, 0, (size_t)Q.n * 4);
    if (ani_milli) memset(ani_milli, 0, n_out * 4);
    return HG_OK;
  }
  int rc;
  bool same;
  if ((rc = hg_packed_rows_check(who, &R, &Q, hv_d, &same))) return rc;
  HG_CUDA(cudaSetDevice(c->device));
  hg_hit *d_out;
  uint32_t *d_nf, *d_milli;
  if ((rc = hg_search_packed_run(c, R, Q, same, hv_d, ksize, top_k, ani_min, path, &d_out, &d_nf, &d_milli))) return rc;
  HG_CUDA(cudaMemcpyAsync(out, d_out, n_out * sizeof(hg_hit), cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaMemcpyAsync(n_found, d_nf, (size_t)Q.n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (ani_milli) HG_CUDA(cudaMemcpyAsync(ani_milli, d_milli, n_out * 4, cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaStreamSynchronize(c->stream));
  return HG_OK;
}

extern "C" int hg_search_packed(hg_ctx *c, const uint8_t *ref_packed, uint64_t ref_stride, const uint8_t *ref_bits, const int32_t *ref_norm,
                                uint32_t n_ref, const uint8_t *qry_packed, uint64_t qry_stride, const uint8_t *qry_bits,
                                const int32_t *qry_norm, uint32_t n_qry, uint32_t hv_d, uint32_t ksize, uint32_t top_k, float ani_min,
                                int path, hg_hit *out, uint32_t *n_found, uint32_t *ani_milli) {
  if (!c) { hg_set_error("hg_search_packed: NULL argument"); return HG_E_INVALID; }
  const hg_packed_rows R = {ref_packed, ref_stride, ref_bits, ref_norm, n_ref}, Q = {qry_packed, qry_stride, qry_bits, qry_norm, n_qry};
  int rc;
  if ((rc = hg_packed_args_check("hg_search_packed", R, Q, hv_d)) ||
      (rc = hg_search_check("hg_search_packed", n_qry, out, n_found, hv_d, top_k, path)))
    return rc;
  return hg_search_packed_host(c, "hg_search_packed", R, Q, hv_d, ksize, top_k, ani_min, path, out, n_found, ani_milli);
}

int hg_search_merge(hg_ctx *c, uint32_t n_lists, const hg_hit *d_in, const uint32_t *d_in_found, const uint32_t *i0, uint32_t n_qry,
                    uint32_t top_k, hg_hit *d_out, uint32_t *d_n_found, uint32_t *d_milli) {
  if (n_qry == 0) return HG_OK;
  int rc;
  void *d_status;
  if ((rc = hg_scratch(c, HG_S_MISC, 256, &d_status))) return rc;
  HG_CUDA(cudaMemsetAsync(d_status, 0, 4, c->stream));
  if ((rc = hg_launch_search_merge(c, n_lists, d_in, d_in_found, i0, n_qry, top_k, d_out, d_n_found, d_milli, (uint32_t *)d_status)))
    return rc;
  uint32_t status = 0;
  HG_CUDA(cudaMemcpyAsync(&status, d_status, 4, cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaStreamSynchronize(c->stream));
  if (status & 1) { hg_set_error("hg_search_merge_dev: a ref index i + i0 does not fit 32 bits"); return HG_E_INVALID; }
  if (status & 2) { hg_set_error("hg_search_merge_dev: an input n_found exceeds top_k %u", top_k); return HG_E_INVALID; }
  return HG_OK;
}

extern "C" int hg_search_merge_dev(hg_ctx *c, uint32_t n_lists, const hg_hit *d_in, const uint32_t *d_in_found, const uint32_t *i0,
                                   uint32_t n_qry, uint32_t top_k, hg_hit *d_out, uint32_t *d_n_found, uint32_t *d_ani_milli) {
  if (!c || !i0 || (n_qry && (!d_in || !d_in_found || !d_out || !d_n_found))) { hg_set_error("hg_search_merge_dev: NULL argument"); return HG_E_INVALID; }
  if (n_lists < 1 || n_lists > HG_SEARCH_MERGE_MAX_LISTS) {
    hg_set_error("hg_search_merge_dev: n_lists %u outside 1..%d", n_lists, HG_SEARCH_MERGE_MAX_LISTS); return HG_E_INVALID;
  }
  if (top_k < 1 || top_k > 1024) { hg_set_error("hg_search_merge_dev: top_k %u outside 1..1024", top_k); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(c->device));
  return hg_search_merge(c, n_lists, d_in, d_in_found, i0, n_qry, top_k, d_out, d_n_found, d_ani_milli);
}

extern "C" int hg_search_stats(hg_ctx *c, uint64_t counts[4], float ms[4]) {
  if (!c || !counts || !ms) { hg_set_error("hg_search_stats: NULL argument"); return HG_E_INVALID; }
  memcpy(counts, c->search_stats, sizeof(c->search_stats));
  // floor pass (gather + dist), its select, main pass, its select; the main pass of a one-pass search starts at mark 0
  const int from[4] = {0, 1, (c->search_ev_used >> 2 & 1) ? 2 : 0, 3};
  for (int k = 0; k < 4; k++) {
    ms[k] = -1.0f;
    if ((c->search_ev_used >> from[k] & 1) && (c->search_ev_used >> (k + 1) & 1))
      HG_CUDA(cudaEventElapsedTime(&ms[k], c->ev_search[from[k]], c->ev_search[k + 1]));
  }
  return HG_OK;
}

// ---------------------------------------------------------------------------------------
// cluster: single-linkage ANI clusters of one sketch set (DESIGN.md §4.9)
// ---------------------------------------------------------------------------------------

// edge records one window of a cluster or derep run may hold: 2^26 (1 GiB of hg_hit), or HG_CLUSTER_EDGE_CAP, read at
// every call (at least 256 x 256)
static uint64_t cluster_edge_cap() {
  uint64_t cap = 0;
  if (const char *e = getenv("HG_CLUSTER_EDGE_CAP")) cap = strtoull(e, nullptr, 10);
  return std::max<uint64_t>(cap ? cap : 1ull << 26, 256ull * 256ull);
}

// The upper triangle of n rows, columns [c0, n), cut into windows of at most cap pairs j > i.  Column chunks [a, a + w)
// of a multiple of 256 columns (the last one ends at n) run against refs [0, a + w), each chunk as wide as keeps its
// a w + w (w - 1) / 2 pairs within cap and w within max_w (a multiple of 256); where even 256 columns have more, the
// refs of a 256-column chunk are split into blocks of floor(cap / 256) rows rounded down to a multiple of 256.  So no
// window's hits can overflow the edge buffer.
static std::vector<DistWindow> cluster_windows(uint32_t n, uint32_t c0, uint64_t cap, uint64_t max_w = UINT32_MAX) {
  std::vector<DistWindow> out;
  auto pairs = [](uint64_t a, uint64_t w) { return a * w + w * (w - 1) / 2; };
  for (uint32_t a = c0; a < n;) {
    uint32_t w = std::min<uint32_t>(256, n - a);
    if (pairs(a, w) <= cap) {
      while (w < n - a && (uint64_t)w + 256 <= max_w && pairs(a, std::min<uint32_t>(w + 256, n - a)) <= cap)
        w = std::min<uint32_t>(w + 256, n - a);
      out.push_back({0, a + w, a, w});
    } else {
      const uint32_t h = (uint32_t)std::min<uint64_t>(cap / 256 / 256 * 256, a + w);
      for (uint32_t r0 = 0; r0 < a + w; r0 += h) out.push_back({r0, std::min(h, a + w - r0), a, w});
    }
    a += w;
  }
  return out;
}

void hg_cluster_stats_reset(hg_ctx *c) {
  memset(c->cluster_stats, 0, sizeof(c->cluster_stats));
  for (float &m : c->cluster_ms) m = -1.0f;
}

int hg_cluster_finish(hg_ctx *c, uint32_t *d_rep, uint32_t n, uint32_t *rep, uint32_t *n_clusters, cudaEvent_t flattened) {
  int rc;
  void *d_misc;
  if ((rc = hg_scratch(c, HG_S_MISC, 256, &d_misc))) return rc;
  uint32_t *d_count = (uint32_t *)d_misc + 1;
  HG_CUDA(cudaMemsetAsync(d_count, 0, 4, c->stream));
  if ((rc = hg_launch_cluster_flatten(c, d_rep, n, d_count))) return rc;
  if (flattened) HG_CUDA(cudaEventRecord(flattened, c->stream));
  uint32_t count = 0;
  HG_CUDA(cudaMemcpyAsync(&count, d_count, 4, cudaMemcpyDeviceToHost, c->stream));
  if (rep && n) HG_CUDA(cudaMemcpyAsync(rep, d_rep, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaStreamSynchronize(c->stream));
  if (n_clusters) *n_clusters = count;
  return HG_OK;
}

// Device events of a cluster run with profiling on: [0] start, [1] rows prepared, then per window before / after its hook,
// then the end.  Destroyed with the run.
struct ClusterEvents {
  std::vector<cudaEvent_t> ev;
  ~ClusterEvents() { for (cudaEvent_t e : ev) cudaEventDestroy(e); }
  int ms(int a, int b, float *out) const {  // both recorded
    HG_CUDA(cudaEventElapsedTime(out, ev[a], ev[b]));
    return HG_OK;
  }
};

// The single-linkage clusters of rows [0, n) over the linked pairs whose column is in [c0, n) (all of them when c0 = 0):
// the kernel is chosen once for the whole matrix, every row prepared once, and the windows of cluster_windows launched one
// after another, each followed on the stream by the hook kernel on its edges and a reset of the edge counter.  d_rep ends
// as a flattened forest (rep[x] = the smallest index of x's cluster); rep / n_clusters as hg_cluster_finish.  bits: as
// dist_choose.  Synchronises once, at the end (and where the single-plane verdict is read, as every dist run does).
static int cluster_run(hg_ctx *c, const int16_t *d_hv, const int32_t *d_norm, uint32_t n, uint32_t c0, uint32_t hv_d, uint32_t ksize,
                       float ani_th, int path, uint32_t bits, uint32_t *d_rep, uint32_t *rep, uint32_t *n_clusters) {
  hg_cluster_stats_reset(c);
  c->pending_stats[0] = c->pending_stats[1] = nullptr;
  c->ev_used &= ~(3 << 4);
  if (n == 0) {
    if (n_clusters) *n_clusters = 0;
    return HG_OK;
  }
  int rc;
  DistChoice ch;
  if ((rc = dist_choose(path, n, n, hg_tensor_shape_ok(hv_d, d_hv, d_hv) == HG_OK, bits, &ch))) return rc;
  const uint64_t cap = cluster_edge_cap();
  const uint64_t room = std::max<uint64_t>(1, std::min<uint64_t>(cap, (uint64_t)n * (n - 1) / 2));  // no window has more pairs
  void *d_edges, *d_cnt;
  if ((rc = hg_scratch(c, HG_S_PACKED, room * sizeof(hg_hit), &d_edges))) return rc;
  if ((rc = hg_scratch(c, HG_S_COUNTS, 256, &d_cnt))) return rc;
  unsigned long long *cnt = (unsigned long long *)d_cnt, *linked = cnt + 1;  // edge counter; linked pairs and the largest window's
  DistWindows W;
  W.win = cluster_windows(n, c0, cap);
  ClusterEvents E;
  if (c->prof) {
    E.ev.resize(3 + 2 * W.win.size(), nullptr);
    for (cudaEvent_t &e : E.ev) HG_CUDA(cudaEventCreate(&e));
    W.prepared = E.ev[1];
  }
  auto mark = [&](size_t k) -> int {
    if (c->prof) HG_CUDA(cudaEventRecord(E.ev[k], c->stream));
    return HG_OK;
  };
  HG_CUDA(cudaMemsetAsync(d_cnt, 0, 3 * sizeof(unsigned long long), c->stream));
  if ((rc = hg_launch_cluster_iota(c, d_rep, n)) || (rc = mark(0))) return rc;
  W.after = [&](size_t k) -> int {
    int r2;
    if ((r2 = mark(2 + 2 * k)) || (r2 = hg_launch_cluster_hook(c, d_rep, (const hg_hit *)d_edges, cnt, room, linked))) return r2;
    HG_CUDA(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), c->stream));
    return mark(3 + 2 * k);
  };
  DistOp op = {d_hv, d_norm, n, 0, d_hv, d_norm, n, 0, hv_d, ksize, ani_th, 1, (hg_hit *)d_edges, room, cnt};
  op.windows = &W;
  if ((rc = dist_run(c, op, ch, nullptr, nullptr, false))) return rc;
  unsigned long long h_linked[2] = {0, 0};
  HG_CUDA(cudaMemcpyAsync(h_linked, linked, sizeof(h_linked), cudaMemcpyDeviceToHost, c->stream));
  if ((rc = hg_cluster_finish(c, d_rep, n, rep, n_clusters, c->prof ? E.ev.back() : nullptr))) return rc;
  c->cluster_stats[0] = W.win.size();
  c->cluster_stats[1] = h_linked[0];
  c->cluster_stats[2] = h_linked[1];
  c->cluster_stats[3] = cap;
  if (c->prof && !W.win.empty()) {
    const int last = (int)(3 + 2 * (W.win.size() - 1)), end = (int)E.ev.size() - 1;
    const bool prepared = c->dist_path != HG_PATH_SIMT;  // the SIMT kernel prepares nothing: ms[0] stays -1
    float hooks = 0.0f, t, windows, flatten, prep = -1.0f;
    for (size_t k = 0; k < W.win.size(); k++) {
      if ((rc = E.ms((int)(2 + 2 * k), (int)(3 + 2 * k), &t))) return rc;
      hooks += t;
    }
    if ((prepared && (rc = E.ms(0, 1, &prep))) || (rc = E.ms(prepared ? 1 : 0, last, &windows)) || (rc = E.ms(last, end, &flatten))) return rc;
    c->cluster_ms[0] = prep;
    c->cluster_ms[1] = windows - hooks;
    c->cluster_ms[2] = hooks;
    c->cluster_ms[3] = flatten;
  }
  return HG_OK;
}

int hg_cluster_check(const char *who, uint32_t n, const uint32_t *rep, uint32_t hv_d, float ani_th, int path) {
  if (n && !rep) { hg_set_error("%s: NULL argument", who); return HG_E_INVALID; }
  if (hv_d == 0 || hv_d % 256 != 0) { hg_set_error("%s: hv_d %u must be a multiple of 256", who, hv_d); return HG_E_INVALID; }
  if (path < HG_PATH_AUTO || path > HG_PATH_NARROW) { hg_set_error("%s: path %d", who, path); return HG_E_INVALID; }
  if (ani_th != ani_th) { hg_set_error("%s: ani_th is NaN", who); return HG_E_INVALID; }
  return HG_OK;
}

extern "C" int hg_cluster_dev(hg_ctx *c, const int16_t *d_hv, const int32_t *d_norm2, uint32_t n, uint32_t hv_d, uint32_t ksize,
                              float ani_th, int path, uint32_t *d_rep, uint32_t *n_clusters) {
  if (!c || (n && (!d_hv || !d_norm2))) { hg_set_error("hg_cluster_dev: NULL argument"); return HG_E_INVALID; }
  int rc;
  if ((rc = hg_cluster_check("hg_cluster_dev", n, d_rep, hv_d, ani_th, path))) return rc;
  HG_CUDA(cudaSetDevice(c->device));
  return cluster_run(c, d_hv, d_norm2, n, 0, hv_d, ksize, ani_th, path, 0, d_rep, nullptr, n_clusters);
}

int hg_cluster_packed_run(hg_ctx *c, const hg_packed_rows &R, uint32_t col0, uint32_t hv_d, uint32_t ksize, float ani_th, int path,
                          uint32_t **d_rep, uint32_t *rep, uint32_t *n_clusters) {
  int rc;
  HostRows hr, hq;
  if ((rc = hg_packed_stage(c, R, R, true, hv_d, &hr, &hq))) return rc;
  void *d_f;
  if ((rc = hg_scratch(c, HG_S_TILES, (size_t)R.n * 4, &d_f))) return rc;
  *d_rep = (uint32_t *)d_f;
  if ((rc = hg_rows_to_device(c, hr, hv_d))) return rc;
  return cluster_run(c, hr.d_hv, hr.d_norm, R.n, col0, hv_d, ksize, ani_th, path, R.max_bits, *d_rep, rep, n_clusters);
}

int hg_cluster_packed_host(hg_ctx *c, const char *who, hg_packed_rows R, uint32_t hv_d, uint32_t ksize, float ani_th, int path,
                           uint32_t *rep, uint32_t *n_clusters) {
  hg_cluster_stats_reset(c);
  if (R.n == 0) {
    if (n_clusters) *n_clusters = 0;
    return HG_OK;
  }
  int rc;
  bool same;
  hg_packed_rows Q = R;
  if ((rc = hg_packed_rows_check(who, &R, &Q, hv_d, &same))) return rc;
  HG_CUDA(cudaSetDevice(c->device));
  uint32_t *d_rep;
  return hg_cluster_packed_run(c, R, 0, hv_d, ksize, ani_th, path, &d_rep, rep, n_clusters);
}

extern "C" int hg_cluster_packed(hg_ctx *c, const uint8_t *packed, uint64_t stride, const uint8_t *quant_bits, const int32_t *norm2,
                                 uint32_t n, uint32_t hv_d, uint32_t ksize, float ani_th, int path, uint32_t *rep, uint32_t *n_clusters) {
  if (!c) { hg_set_error("hg_cluster_packed: NULL argument"); return HG_E_INVALID; }
  const hg_packed_rows R = {packed, stride, quant_bits, norm2, n};
  int rc;
  if ((rc = hg_packed_args_check("hg_cluster_packed", R, R, hv_d)) || (rc = hg_cluster_check("hg_cluster_packed", n, rep, hv_d, ani_th, path)))
    return rc;
  return hg_cluster_packed_host(c, "hg_cluster_packed", R, hv_d, ksize, ani_th, path, rep, n_clusters);
}

extern "C" int hg_cluster_union_dev(hg_ctx *c, uint32_t n, uint32_t *d_rep, const hg_hit *d_edges, uint64_t n_edges, uint32_t *n_clusters) {
  if (!c || (n && !d_rep) || (n_edges && !d_edges)) { hg_set_error("hg_cluster_union_dev: NULL argument"); return HG_E_INVALID; }
  HG_CUDA(cudaSetDevice(c->device));
  int rc;
  void *d_misc;
  if ((rc = hg_scratch(c, HG_S_MISC, 256, &d_misc))) return rc;
  uint32_t *d_status = (uint32_t *)d_misc, status = 0;
  // nothing may reach a find before this: an index >= n would be an access out of bounds, a rep[x] > x a possible cycle
  HG_CUDA(cudaMemsetAsync(d_status, 0, 4, c->stream));
  if ((rc = hg_launch_cluster_check(c, d_rep, n, d_edges, n_edges, d_status))) return rc;
  HG_CUDA(cudaMemcpyAsync(&status, d_status, 4, cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaStreamSynchronize(c->stream));
  if (status & 1) { hg_set_error("hg_cluster_union_dev: an edge index is >= n (%u)", n); return HG_E_INVALID; }
  if (status & 2) { hg_set_error("hg_cluster_union_dev: rep[x] > x for some x: not a forest this union accepts"); return HG_E_INVALID; }
  if ((rc = hg_launch_cluster_hook(c, d_rep, d_edges, nullptr, n_edges, nullptr))) return rc;
  return hg_cluster_finish(c, d_rep, n, nullptr, n_clusters);
}

extern "C" int hg_cluster_stats(hg_ctx *c, uint64_t counts[4], float ms[4]) {
  if (!c || !counts || !ms) { hg_set_error("hg_cluster_stats: NULL argument"); return HG_E_INVALID; }
  memcpy(counts, c->cluster_stats, sizeof(c->cluster_stats));
  memcpy(ms, c->cluster_ms, sizeof(c->cluster_ms));
  return HG_OK;
}

// ---------------------------------------------------------------------------------------
// derep: greedy ANI dereplication of one sketch set (DESIGN.md §4.10)
// ---------------------------------------------------------------------------------------

static void derep_stats_reset(hg_ctx *c) {
  memset(c->derep_stats, 0, sizeof(c->derep_stats));
  for (float &m : c->derep_ms) m = -1.0f;
}

// The state of a derep run, carved from HG_S_TILES (which neither the dist windows nor the internal search touch):
// per row of the permuted space is_rep, the rep list (ascending), the order, the search's top-1 result and the labels;
// the covered flags and adjacency bitmap of one column chunk; the rep count, a status word and the linked pairs.
struct DerepState {
  uint8_t *is_rep, *covered;
  uint32_t *rep_list, *order, *n_found, *rep, *adj;
  uint32_t *count;  // [0] representatives so far, [1] status
  hg_hit *out;
  unsigned long long *linked;
};

static int derep_state(hg_ctx *c, uint32_t n, DerepState *S) {
  const size_t sizes[] = {(size_t)n, (size_t)HG_DEREP_CHUNK, (size_t)n * 4, (size_t)n * 4, (size_t)n * 4, (size_t)n * 4,
                          (size_t)HG_DEREP_CHUNK * HG_DEREP_CHUNK / 8, 16, (size_t)n * sizeof(hg_hit), 8};
  size_t off[10], total = 0;
  for (int k = 0; k < 10; k++) {
    off[k] = total;
    total += (sizes[k] + 255) & ~(size_t)255;
  }
  void *p;
  int rc;
  if ((rc = hg_scratch(c, HG_S_TILES, total, &p))) return rc;
  uint8_t *b = (uint8_t *)p;
  *S = {b + off[0], b + off[1], (uint32_t *)(b + off[2]), (uint32_t *)(b + off[3]), (uint32_t *)(b + off[4]), (uint32_t *)(b + off[5]),
        (uint32_t *)(b + off[6]), (uint32_t *)(b + off[7]), (hg_hit *)(b + off[8]), (unsigned long long *)(b + off[9])};
  // the chunk state starts clear (each greedy step leaves it so), and the counters at 0
  HG_CUDA(cudaMemsetAsync(S->covered, 0, HG_DEREP_CHUNK, c->stream));
  HG_CUDA(cudaMemsetAsync(S->adj, 0, (size_t)HG_DEREP_CHUNK * HG_DEREP_CHUNK / 8, c->stream));
  HG_CUDA(cudaMemsetAsync(S->count, 0, 16, c->stream));
  HG_CUDA(cudaMemsetAsync(S->linked, 0, 8, c->stream));
  return HG_OK;
}

// Greedy dereplication of rows [0, n) at ani_th in the priority order `order` (host; NULL: file order), in two phases.
//   1. Representatives: the rows in priority order (gathered into HG_S_DEREP_ROWS when an order is given), the kernel
//      chosen once and every row prepared once, then the upper triangle in the windows of cluster_windows with column
//      chunks of at most HG_DEREP_CHUNK; behind each window a mark hook, behind a chunk's last window its greedy step.
//      The single plane's verdict is read before the first window (DistWindows::decide_first): a greedy step marks
//      every uncovered node of its chunk, so it must never run on the empty edges of a declined plane.
//   2. Assignment: the representatives' rows gathered (ascending, so in priority order) into HG_S_DEREP_REPS, a top-1
//      search of every row against them at ani_min = ani_th (ties to the smaller ref index: the first in the order),
//      and the finalize kernel, which maps the labels back to file indices in d_rep.
// hg_dist_last_path / reason report phase 1; hg_search_stats the search of phase 2 (zeros when every row is a
// representative and no search runs).  bits: as dist_choose.  d_rep: the labels on the device (NULL: in the state);
// rep (host, may be NULL) receives them.
static int derep_run(hg_ctx *c, const int16_t *d_hv, const int32_t *d_norm, uint32_t n, uint32_t hv_d, uint32_t ksize, float ani_th,
                     int path, uint32_t bits, const uint32_t *order, uint32_t *d_rep, uint32_t *rep, uint32_t *n_reps) {
  derep_stats_reset(c);
  memset(c->search_stats, 0, sizeof(c->search_stats));
  c->search_ev_used = 0;
  c->pending_stats[0] = c->pending_stats[1] = nullptr;
  c->ev_used &= ~(3 << 4);
  if (n == 0) {
    if (n_reps) *n_reps = 0;
    return HG_OK;
  }
  int rc;
  DerepState S;
  if ((rc = derep_state(c, n, &S))) return rc;
  if (!d_rep) d_rep = S.rep;  // the packed entry: labels on the device before their copy to `rep`
  const int16_t *W = d_hv;
  const int32_t *Wn = d_norm;
  ClusterEvents E;  // [0] start, [1] permuted, [2] rows prepared, per window before / after its hook, phase 2 start, end
  DistWindows DW;
  DW.win = cluster_windows(n, 0, cluster_edge_cap(), HG_DEREP_CHUNK);
  DW.decide_first = true;
  const size_t n_ev = 5 + 2 * DW.win.size();
  if (c->prof) {
    E.ev.resize(n_ev, nullptr);
    for (cudaEvent_t &e : E.ev) HG_CUDA(cudaEventCreate(&e));
    DW.prepared = E.ev[2];
  }
  auto mark = [&](size_t k) -> int {
    if (c->prof) HG_CUDA(cudaEventRecord(E.ev[k], c->stream));
    return HG_OK;
  };
  if ((rc = mark(0))) return rc;
  if (order) {
    const size_t mb = ((size_t)n * hv_d * 2 + 255) & ~(size_t)255;
    void *d_w;
    if ((rc = hg_scratch(c, HG_S_DEREP_ROWS, mb + (size_t)n * 4, &d_w))) return rc;
    HG_CUDA(cudaMemcpyAsync(S.order, order, (size_t)n * 4, cudaMemcpyHostToDevice, c->stream));
    W = (const int16_t *)d_w;
    Wn = (const int32_t *)((uint8_t *)d_w + mb);
    if ((rc = hg_launch_derep_gather(c, d_hv, d_norm, S.order, n, hv_d, (int16_t *)W, (int32_t *)Wn))) return rc;
  }
  if ((rc = mark(1))) return rc;

  // ---- phase 1: the representatives ----
  DistChoice ch;
  if ((rc = dist_choose(path, n, n, hg_tensor_shape_ok(hv_d, W, W) == HG_OK, bits, &ch))) return rc;
  const uint64_t room = std::max<uint64_t>(1, std::min<uint64_t>(cluster_edge_cap(), (uint64_t)n * (n - 1) / 2));
  void *d_edges, *d_cnt;
  if ((rc = hg_scratch(c, HG_S_PACKED, room * sizeof(hg_hit), &d_edges))) return rc;
  if ((rc = hg_scratch(c, HG_S_COUNTS, 256, &d_cnt))) return rc;
  unsigned long long *cnt = (unsigned long long *)d_cnt;
  HG_CUDA(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), c->stream));
  DW.after = [&](size_t k) -> int {
    const DistWindow &w = DW.win[k];
    int r2;
    if ((r2 = mark(3 + 2 * k)) ||
        (r2 = hg_launch_derep_mark(c, (const hg_hit *)d_edges, cnt, room, w.c0, w.w, S.is_rep, S.covered, S.adj, S.linked)))
      return r2;
    HG_CUDA(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), c->stream));
    const bool last = k + 1 == DW.win.size() || DW.win[k + 1].c0 != w.c0;  // the chunk's refs may span several windows
    if (last && (r2 = hg_launch_derep_greedy(c, w.c0, w.w, S.covered, S.adj, S.is_rep, S.rep_list, S.count))) return r2;
    return mark(4 + 2 * k);
  };
  DistOp op = {W, Wn, n, 0, W, Wn, n, 0, hv_d, ksize, ani_th, 1, (hg_hit *)d_edges, room, cnt};
  op.windows = &DW;
  if ((rc = dist_run(c, op, ch, nullptr, nullptr, false))) return rc;
  const int p1_path = c->dist_path;
  char p1_reason[sizeof(c->dist_reason)];
  memcpy(p1_reason, c->dist_reason, sizeof(p1_reason));
  uint32_t h_count[2] = {0, 0};
  unsigned long long linked = 0;
  HG_CUDA(cudaMemcpyAsync(h_count, S.count, 8, cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaMemcpyAsync(&linked, S.linked, 8, cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaStreamSynchronize(c->stream));
  const uint32_t k_reps = h_count[0];

  // ---- phase 2: every other row to its closest representative ----
  if ((rc = mark(n_ev - 2))) return rc;
  if (k_reps < n) {  // (all rows representatives: nothing to assign)
    const size_t rb = ((size_t)k_reps * hv_d * 2 + 255) & ~(size_t)255;
    void *d_r;
    if ((rc = hg_scratch(c, HG_S_DEREP_REPS, rb + (size_t)k_reps * 4, &d_r))) return rc;
    int16_t *R = (int16_t *)d_r;
    int32_t *Rn = (int32_t *)((uint8_t *)d_r + rb);
    if ((rc = hg_launch_derep_gather(c, W, Wn, S.rep_list, k_reps, hv_d, R, Rn))) return rc;
    rc = search_run(c, R, Rn, k_reps, W, Wn, n, hv_d, ksize, 1, ani_th, path, bits, S.out, S.n_found, nullptr);
    hg_dist_record(c, p1_path, "%s", p1_reason);  // in auto mode a small rep set may have made the search pick SIMT
    if (rc) return rc;
  }
  if ((rc = hg_launch_derep_finalize(c, S.is_rep, S.rep_list, S.out, S.n_found, order ? S.order : nullptr, n, d_rep, S.count + 1)) ||
      (rc = mark(n_ev - 1)))
    return rc;
  HG_CUDA(cudaMemcpyAsync(h_count + 1, S.count + 1, 4, cudaMemcpyDeviceToHost, c->stream));
  if (rep) HG_CUDA(cudaMemcpyAsync(rep, d_rep, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  HG_CUDA(cudaStreamSynchronize(c->stream));
  if (h_count[1]) {
    hg_set_error("hg_derep: internal error: a sketch that is not a representative matched none at ANI >= %g", (double)ani_th);
    return HG_E_CUDA;
  }
  if (n_reps) *n_reps = k_reps;
  uint64_t chunks = 0;
  for (size_t k = 0; k < DW.win.size(); k++) chunks += k == 0 || DW.win[k].c0 != DW.win[k - 1].c0;
  c->derep_stats[0] = chunks;
  c->derep_stats[1] = DW.win.size();
  c->derep_stats[2] = linked;
  c->derep_stats[3] = k_reps;
  if (c->prof) {
    const int last = (int)(4 + 2 * (DW.win.size() - 1)), p2 = (int)n_ev - 2, end = (int)n_ev - 1;
    const int prep_end = p1_path != HG_PATH_SIMT ? 2 : 1;  // the SIMT kernel prepares nothing
    float hooks = 0.0f, t, windows;
    for (size_t k = 0; k < DW.win.size(); k++) {
      if ((rc = E.ms((int)(3 + 2 * k), (int)(4 + 2 * k), &t))) return rc;
      hooks += t;
    }
    if ((rc = E.ms(0, prep_end, &c->derep_ms[0])) || (rc = E.ms(prep_end, last, &windows)) || (rc = E.ms(p2, end, &c->derep_ms[3])))
      return rc;
    c->derep_ms[1] = windows - hooks;
    c->derep_ms[2] = hooks;
  }
  return HG_OK;
}

// order: NULL, or a permutation of [0, n) - checked whole before anything runs
static int derep_order_check(const char *who, const uint32_t *order, uint32_t n) {
  if (!order) return HG_OK;
  std::vector<uint8_t> seen(n, 0);
  for (uint32_t t = 0; t < n; t++) {
    if (order[t] >= n) { hg_set_error("%s: order[%u] = %u is not below n = %u", who, t, order[t], n); return HG_E_INVALID; }
    if (seen[order[t]]++) { hg_set_error("%s: order[%u] = %u repeats an earlier entry", who, t, order[t]); return HG_E_INVALID; }
  }
  return HG_OK;
}

extern "C" int hg_derep_dev(hg_ctx *c, const int16_t *d_hv, const int32_t *d_norm2, uint32_t n, uint32_t hv_d, uint32_t ksize,
                            float ani_th, int path, const uint32_t *order, uint32_t *d_rep, uint32_t *n_reps) {
  if (!c || (n && (!d_hv || !d_norm2))) { hg_set_error("hg_derep_dev: NULL argument"); return HG_E_INVALID; }
  int rc;
  if ((rc = hg_cluster_check("hg_derep_dev", n, d_rep, hv_d, ani_th, path)) || (rc = derep_order_check("hg_derep_dev", order, n)))
    return rc;
  HG_CUDA(cudaSetDevice(c->device));
  return derep_run(c, d_hv, d_norm2, n, hv_d, ksize, ani_th, path, 0, order, d_rep, nullptr, n_reps);
}

extern "C" int hg_derep_packed(hg_ctx *c, const uint8_t *packed, uint64_t stride, const uint8_t *quant_bits, const int32_t *norm2,
                               uint32_t n, uint32_t hv_d, uint32_t ksize, float ani_th, int path, const uint32_t *order, uint32_t *rep,
                               uint32_t *n_reps) {
  if (!c) { hg_set_error("hg_derep_packed: NULL argument"); return HG_E_INVALID; }
  hg_packed_rows R = {packed, stride, quant_bits, norm2, n}, Q = R;
  int rc;
  if ((rc = hg_packed_args_check("hg_derep_packed", R, R, hv_d)) || (rc = hg_cluster_check("hg_derep_packed", n, rep, hv_d, ani_th, path)) ||
      (rc = derep_order_check("hg_derep_packed", order, n)))
    return rc;
  if (n == 0) {
    derep_stats_reset(c);
    if (n_reps) *n_reps = 0;
    return HG_OK;
  }
  bool same;
  if ((rc = hg_packed_rows_check("hg_derep_packed", &R, &Q, hv_d, &same))) return rc;
  HG_CUDA(cudaSetDevice(c->device));
  HostRows hr, hq;
  if ((rc = hg_packed_stage(c, R, R, true, hv_d, &hr, &hq)) || (rc = hg_rows_to_device(c, hr, hv_d))) return rc;
  return derep_run(c, hr.d_hv, hr.d_norm, n, hv_d, ksize, ani_th, path, R.max_bits, order, nullptr, rep, n_reps);
}

extern "C" int hg_derep_stats(hg_ctx *c, uint64_t counts[4], float ms[4]) {
  if (!c || !counts || !ms) { hg_set_error("hg_derep_stats: NULL argument"); return HG_E_INVALID; }
  memcpy(counts, c->derep_stats, sizeof(c->derep_stats));
  memcpy(ms, c->derep_ms, sizeof(c->derep_ms));
  return HG_OK;
}

// ---------------------------------------------------------------------------------------
// ANI matrix: every pair, dense (DESIGN.md §4.11)
// ---------------------------------------------------------------------------------------

// output bytes one band may hold: 64 MiB (16 M cells: a 256-row band of 65 536 columns, and far more than the 74 CTA
// pairs' 4.8 M cells of one wave of tiles), or HG_MATRIX_BAND_BYTES, read at every call
static uint64_t matrix_band_bytes() {
  uint64_t b = 0;
  if (const char *e = getenv("HG_MATRIX_BAND_BYTES")) b = strtoull(e, nullptr, 10);
  return b ? b : 64ull << 20;
}

// cell offset of row i's first cell (hg_dense_row of the caller's layout)
static uint64_t matrix_row(bool lower, uint64_t ld, uint32_t i) { return lower ? (uint64_t)i * ((uint64_t)i - 1) / 2 : (uint64_t)i * ld; }

// Bands of ref rows [first, n_ref): rows [a, a + h) against the query columns [0, a + h) (lower) or [0, n_qry), each
// the most rows whose cells fit `bytes` (at least one row), cut to a multiple of 256 rows where that many fit.
static std::vector<DistWindow> matrix_bands(uint32_t first, uint32_t n_ref, uint32_t n_qry, bool lower, uint64_t bytes) {
  const uint64_t cap = std::max<uint64_t>(1, bytes / 4);
  std::vector<DistWindow> out;
  for (uint32_t a = first; a < n_ref;) {
    auto cells = [&](uint64_t h) { return lower ? h * a + h * (h - 1) / 2 : h * n_qry; };
    uint64_t lo = 1, hi = n_ref - a;
    while (lo < hi) {
      const uint64_t m = (lo + hi + 1) / 2;
      if (cells(m) <= cap) lo = m; else hi = m - 1;
    }
    if (lo >= 256 && lo < n_ref - a) lo &= ~255ull;
    out.push_back({a, (uint32_t)lo, 0, lower ? a + (uint32_t)lo : n_qry});
    a += (uint32_t)lo;
  }
  return out;
}

static void matrix_stats_reset(hg_ctx *c) {
  memset(c->matrix_stats, 0, sizeof(c->matrix_stats));
  for (float &m : c->matrix_ms) m = -1.0f;
}

// The matrix cells of ref rows [first, n_ref) - of the one matrix ref = qry in lower mode, else against every query row:
// the kernel chosen once and every row prepared once, then the bands of matrix_bands, each launched in dense mode and
// converted in place behind its launch (DistWindows::after).  d_out: the bands write straight into the caller's device
// matrix.  h_out: they alternate between two band buffers; band k is copied to the host on the copy stream under band
// k + 1's kernel, and band k + 2 (same buffer) waits for that copy.  The single plane's verdict is read before band 0
// (decide_first), so a declined attempt writes and copies nothing.  d_out / h_out hold row `first` at offset 0.
// `upload` (may be empty) brings the rows to the device first; profiling counts it with the row preparation.  Returns
// with everything complete.
static int matrix_run(hg_ctx *c, const int16_t *d_ref, const int32_t *d_rn, uint32_t n_ref, const int16_t *d_qry, const int32_t *d_qn,
                      uint32_t n_qry, uint32_t hv_d, uint32_t ksize, int path, uint32_t bits, bool lower, uint32_t first, float *d_out,
                      float *h_out, uint64_t ld, const std::function<int()> &upload = nullptr) {
  int rc;
  DistChoice ch;
  if ((rc = dist_choose(path, n_ref, n_qry, hg_tensor_shape_ok(hv_d, d_ref, d_qry) == HG_OK, bits, &ch))) return rc;
  DistWindows W;
  W.win = matrix_bands(first, n_ref, n_qry, lower, matrix_band_bytes());
  W.decide_first = true;
  const size_t nb = W.win.size();
  auto cells = [&](const DistWindow &w) { return matrix_row(lower, n_qry, w.r0 + w.h) - matrix_row(lower, n_qry, w.r0); };
  uint64_t band_max = 0;
  for (const DistWindow &w : W.win) band_max = std::max(band_max, cells(w));
  int32_t *buf[2] = {nullptr, nullptr};
  if (h_out) {
    void *p;
    const uint64_t bb = (band_max * 4 + 255) & ~255ull;
    if ((rc = hg_scratch(c, HG_S_PACKED, 2 * bb, &p)) || (rc = ensure_copy_stream(c))) return rc;
    buf[0] = (int32_t *)p;
    buf[1] = (int32_t *)((uint8_t *)p + bb);
  }
  std::vector<hg_dense> D(nb);
  for (size_t k = 0; k < nb; k++)
    D[k] = h_out ? hg_dense{buf[k & 1], lower ? 0 : (uint64_t)n_qry, W.win[k].r0} : hg_dense{(int32_t *)d_out, lower ? 0 : ld, first};
  W.dense = D.data();
  // [0] converted, [1..2] band buffer copied; then with profiling: [3] start, [4] rows prepared, per band: kernel start,
  // kernel end, converted, copy start, copy end
  ClusterEvents E;
  E.ev.resize(c->prof ? 5 + 5 * nb : 3, nullptr);
  for (size_t t = 0; t < E.ev.size(); t++) HG_CUDA(cudaEventCreateWithFlags(&E.ev[t], t < 3 ? cudaEventDisableTiming : cudaEventDefault));
  auto mark = [&](size_t t, cudaStream_t s) -> int {
    if (c->prof) HG_CUDA(cudaEventRecord(E.ev[t], s));
    return HG_OK;
  };
  if (c->prof) W.prepared = E.ev[4];
  uint64_t entries = 0, bytes = 0;
  W.before = [&](size_t k) -> int {
    if (h_out && k >= 2) HG_CUDA(cudaStreamWaitEvent(c->stream, E.ev[1 + (k & 1)], 0));  // its buffer's last band is on the host
    return mark(5 + 5 * k, c->stream);
  };
  W.after = [&](size_t k) -> int {
    const DistWindow &w = W.win[k];
    int r2;
    if ((r2 = mark(6 + 5 * k, c->stream)) || (r2 = hg_launch_ani_convert(c, D[k], w.r0, w.h, n_qry, d_rn, d_qn, ksize)) ||
        (r2 = mark(7 + 5 * k, c->stream)))
      return r2;
    const uint64_t n_cells = cells(w);
    entries += n_cells;
    if (!h_out) return HG_OK;
    HG_CUDA(cudaEventRecord(E.ev[0], c->stream));
    HG_CUDA(cudaStreamWaitEvent(c->copy_stream, E.ev[0], 0));
    if ((r2 = mark(8 + 5 * k, c->copy_stream))) return r2;
    float *dst = h_out + (matrix_row(lower, ld, w.r0) - matrix_row(lower, ld, first));
    if (lower || ld == n_qry)
      HG_CUDA(cudaMemcpyAsync(dst, buf[k & 1], n_cells * 4, cudaMemcpyDeviceToHost, c->copy_stream));
    else
      HG_CUDA(cudaMemcpy2DAsync(dst, ld * 4, buf[k & 1], (size_t)n_qry * 4, (size_t)n_qry * 4, w.h, cudaMemcpyDeviceToHost, c->copy_stream));
    HG_CUDA(cudaEventRecord(E.ev[1 + (k & 1)], c->copy_stream));
    bytes += n_cells * 4;
    return mark(9 + 5 * k, c->copy_stream);
  };
  void *d_cnt;
  if ((rc = hg_scratch(c, HG_S_COUNTS, 256, &d_cnt))) return rc;  // (no hits: the counter a declined attempt resets)
  if ((rc = mark(3, c->stream)) || (upload && (rc = upload()))) return rc;
  DistOp op = {d_ref, d_rn, n_ref, 0, d_qry, d_qn, n_qry, 0, hv_d, ksize, 0.0f, 0, nullptr, 0, (unsigned long long *)d_cnt};
  op.windows = &W;
  rc = dist_run(c, op, ch, nullptr, nullptr, false);
  if (h_out) HG_CUDA(cudaStreamSynchronize(c->copy_stream));  // (also on an error: no copy may outlive the call)
  HG_CUDA(cudaStreamSynchronize(c->stream));
  if (rc) return rc;
  c->matrix_stats[0] = nb;
  c->matrix_stats[1] = entries;
  c->matrix_stats[2] = bytes;
  c->matrix_stats[3] = (uint64_t)c->dist_path;
  if (c->prof && nb) {
    float t, kern = 0.0f, conv = 0.0f, copy = 0.0f;
    for (size_t k = 0; k < nb; k++) {
      if ((rc = E.ms((int)(5 + 5 * k), (int)(6 + 5 * k), &t))) return rc;
      kern += t;
      if ((rc = E.ms((int)(6 + 5 * k), (int)(7 + 5 * k), &t))) return rc;
      conv += t;
      if (h_out) {
        if ((rc = E.ms((int)(8 + 5 * k), (int)(9 + 5 * k), &t))) return rc;
        copy += t;
      }
    }
    if (c->dist_path != HG_PATH_SIMT && (rc = E.ms(3, 4, &c->matrix_ms[0]))) return rc;  // the SIMT kernel prepares nothing
    c->matrix_ms[1] = kern;
    c->matrix_ms[2] = conv;
    if (h_out) c->matrix_ms[3] = copy;
  }
  return HG_OK;
}

int hg_matrix_check(const char *who, bool same, uint32_t n_ref, uint32_t n_qry, uint32_t hv_d, int path, int lower, const void *out,
                    uint64_t ld) {
  if (hv_d == 0 || hv_d % 256 != 0) { hg_set_error("%s: hv_d %u must be a multiple of 256", who, hv_d); return HG_E_INVALID; }
  if (path < HG_PATH_AUTO || path > HG_PATH_NARROW) { hg_set_error("%s: path %d", who, path); return HG_E_INVALID; }
  if (lower != 0 && lower != 1) { hg_set_error("%s: lower %d (0 or 1)", who, lower); return HG_E_INVALID; }
  if (lower && !same) { hg_set_error("%s: the lower triangle needs the same rows as ref and query", who); return HG_E_INVALID; }
  if (!lower && ld < n_qry) { hg_set_error("%s: ld %llu < n_qry %u", who, (unsigned long long)ld, n_qry); return HG_E_INVALID; }
  if (!out && hg_matrix_entries(n_ref, n_qry, lower)) { hg_set_error("%s: NULL argument", who); return HG_E_INVALID; }
  return HG_OK;
}

uint64_t hg_matrix_entries(uint32_t n_ref, uint32_t n_qry, int lower) {
  return lower ? (n_ref ? (uint64_t)n_ref * (n_ref - 1) / 2 : 0) : (uint64_t)n_ref * n_qry;
}

int HostPin::pin(void *p, uint64_t bytes) {
  cudaPointerAttributes a;
  const uint8_t *last = (const uint8_t *)p + bytes - 1;
  bool locked = cudaPointerGetAttributes(&a, p) == cudaSuccess && a.type == cudaMemoryTypeHost;
  locked = locked && cudaPointerGetAttributes(&a, last) == cudaSuccess && a.type == cudaMemoryTypeHost;
  cudaGetLastError();  // (an unregistered pointer is not an error to keep)
  if (locked || bytes == 0) return HG_OK;
  HG_CUDA(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
  ptr = p;
  return HG_OK;
}
HostPin::~HostPin() {
  if (ptr) cudaHostUnregister(ptr);
}

int hg_matrix_packed_run(hg_ctx *c, const hg_packed_rows &R, const hg_packed_rows &Q, bool same, uint32_t hv_d, uint32_t ksize, int path,
                         bool lower, uint32_t first, float *out, uint64_t ld) {
  HG_CUDA(cudaSetDevice(c->device));
  matrix_stats_reset(c);
  int rc;
  HostRows hr, hq;
  if ((rc = hg_packed_stage(c, R, Q, same, hv_d, &hr, &hq))) return rc;
  auto upload = [&]() -> int {
    int r2 = hg_rows_to_device(c, hr, hv_d);
    return r2 || same ? r2 : hg_rows_to_device(c, hq, hv_d);
  };
  return matrix_run(c, hr.d_hv, hr.d_norm, R.n, hq.d_hv, hq.d_norm, Q.n, hv_d, ksize, path, std::max(R.max_bits, Q.max_bits), lower, first,
                    nullptr, out, ld, upload);
}

extern "C" int hg_ani_matrix_dev(hg_ctx *c, const int16_t *d_ref, const int32_t *d_ref_norm2, uint32_t n_ref, const int16_t *d_qry,
                                 const int32_t *d_qry_norm2, uint32_t n_qry, uint32_t hv_d, uint32_t ksize, int path, int lower,
                                 float *d_out, uint64_t ld) {
  const char *who = "hg_ani_matrix_dev";
  if (!c || (n_ref && (!d_ref || !d_ref_norm2)) || (n_qry && (!d_qry || !d_qry_norm2))) { hg_set_error("%s: NULL argument", who); return HG_E_INVALID; }
  const bool same = d_ref == d_qry && d_ref_norm2 == d_qry_norm2 && n_ref == n_qry;
  int rc;
  if ((rc = hg_matrix_check(who, same, n_ref, n_qry, hv_d, path, lower, d_out, ld))) return rc;
  matrix_stats_reset(c);
  if (hg_matrix_entries(n_ref, n_qry, lower) == 0) return HG_OK;
  HG_CUDA(cudaSetDevice(c->device));
  return matrix_run(c, d_ref, d_ref_norm2, n_ref, d_qry, d_qry_norm2, n_qry, hv_d, ksize, path, 0, lower != 0, 0, d_out, nullptr, ld);
}

extern "C" int hg_ani_matrix_packed(hg_ctx *c, const uint8_t *ref_packed, uint64_t ref_stride, const uint8_t *ref_bits,
                                    const int32_t *ref_norm2, uint32_t n_ref, const uint8_t *qry_packed, uint64_t qry_stride,
                                    const uint8_t *qry_bits, const int32_t *qry_norm2, uint32_t n_qry, uint32_t hv_d, uint32_t ksize,
                                    int path, int lower, float *out, uint64_t ld) {
  const char *who = "hg_ani_matrix_packed";
  if (!c) { hg_set_error("%s: NULL argument", who); return HG_E_INVALID; }
  hg_packed_rows R = {ref_packed, ref_stride, ref_bits, ref_norm2, n_ref}, Q = {qry_packed, qry_stride, qry_bits, qry_norm2, n_qry};
  const bool same = R.packed == Q.packed && R.bits == Q.bits && R.norm == Q.norm && R.n == Q.n;
  int rc;
  if ((rc = hg_packed_args_check(who, R, Q, hv_d)) || (rc = hg_matrix_check(who, same, n_ref, n_qry, hv_d, path, lower, out, ld))) return rc;
  matrix_stats_reset(c);
  const uint64_t entries = hg_matrix_entries(n_ref, n_qry, lower);
  if (entries == 0) return HG_OK;
  bool same2;
  if ((rc = hg_packed_rows_check(who, &R, &Q, hv_d, &same2))) return rc;
  HostPin pin;
  const uint64_t span = lower ? entries : (uint64_t)(n_ref - 1) * ld + n_qry;
  if ((rc = pin.pin(out, span * 4))) return rc;
  return hg_matrix_packed_run(c, R, Q, same2, hv_d, ksize, path, lower != 0, 0, out, ld);
}

extern "C" int hg_ani_matrix_stats(hg_ctx *c, uint64_t counts[4], float ms[4]) {
  if (!c || !counts || !ms) { hg_set_error("hg_ani_matrix_stats: NULL argument"); return HG_E_INVALID; }
  memcpy(counts, c->matrix_stats, sizeof(c->matrix_stats));
  memcpy(ms, c->matrix_ms, sizeof(c->matrix_ms));
  return HG_OK;
}
