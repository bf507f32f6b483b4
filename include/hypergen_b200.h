/*
 * hypergen_b200.h — C ABI of the B200-native (sm_100a) HyperGen sketch -> dist hot path.
 *
 * This header takes the place of the reference's src/cuda_kernel.h (an empty include
 * guard, cuda_kernel.h:1-4) and the library behind it replaces the PTX-JIT boundary of
 * src/sketch_cuda.rs:52-60,119-166 (cudarc htod_copy / launch / sync_reclaim) plus the CPU
 * stages that followed it.  Every entry point names the reference interface it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; the caller owns every buffer it passes in;
 *   - every function returns HG_OK (0) or a negative hg_status, never throws or aborts
 *     (the reference panics: `unwrap()` + panic="abort", Cargo.toml:67-70);
 *     hg_last_error() returns a thread-local message for the last failure;
 *   - "_dev" variants take DEVICE pointers (inputs/outputs resident in HBM) and run
 *     asynchronously on the context's stream — call hg_sync() before reading results;
 *     the plain variants take HOST pointers and include the H2D / D2H copies;
 *   - there is no CPU fallback: without a CUDA device hg_init fails with HG_E_CUDA.
 */
#ifndef HYPERGEN_B200_H
#define HYPERGEN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define HG_API
#else
#define HG_API __attribute__((visibility("default")))
#endif

typedef enum hg_status {
  HG_OK = 0,
  HG_E_INVALID = -1,     /* bad argument (NULL pointer, k = 0 or > 32, hv_d % 256 != 0 ...) */
  HG_E_CUDA = -2,        /* CUDA runtime / driver error, message in hg_last_error()        */
  HG_E_CAPACITY = -3,    /* caller's output buffer too small; required size is reported    */
  HG_E_RANGE = -4,       /* a sketch needs hv_quant_bits = 16, which the reference's own
                            offset arithmetic cannot represent (src/hd.rs:140)              */
  HG_E_UNSUPPORTED = -5  /* valid for the reference but outside this build (see DESIGN.md)  */
} hg_status;

typedef struct hg_ctx hg_ctx; /* one CUDA device, one stream, grow-only device scratch */

/* The knobs that reach the kernels: FileSketch fields ksize/scaled/canonical/seed/hv_d
 * (src/types.rs:224-235; defaults src/types.rs:97-113: k=21 seed=123 scaled=1500 hv_d=4096). */
typedef struct hg_sketch_params {
  uint64_t scaled;   /* FracMinHash: keep h < u64::MAX / scaled (src/sketch.rs:73)          */
  uint64_t seed;     /* t1ha2 seed (src/sketch.rs:74)                                       */
  uint32_t hv_d;     /* HV dimension, multiple of 256 (BitPacker8x block, src/hd.rs:147)    */
  uint8_t ksize;     /* 1..32 (t1ha2_atonce in src/cuda_kernel.cu:196-246 covers <= 32)     */
  uint8_t canonical; /* as the reference GPU path (src/cuda_kernel.cu:306-314); the CPU path
                        is always canonical (src/sketch.rs:89)                              */
  uint8_t reserved[2];
} hg_sketch_params;

/* One reported pair: indices into the ref / query arrays, the exact i32 dot product and
 * the f32 ANI of src/dist.rs:139-161. */
typedef struct hg_hit {
  uint32_t i;
  uint32_t j;
  int32_t dot;
  float ani;
} hg_hit;

/* ---- context ---------------------------------------------------------------------- */

/* Replaces CudaDevice::new(0) + load_ptx (src/sketch_cuda.rs:52-60).  `device` is a CUDA
 * ordinal; multi-GPU hosts create one context per device (one process per GPU). */
HG_API int hg_init(int device, hg_ctx **out);
HG_API void hg_destroy(hg_ctx *ctx);
HG_API int hg_sync(hg_ctx *ctx);

/* Page-locked host memory for the buffers the host entries read from / write to (FASTA bytes, sequences, packed
 * sketches, hits): from such memory the H2D copies run at the PCIe rate and overlap with the kernels; from
 * ordinary (pageable) memory they are staged by the driver at a fraction of it.  A Rust host reads its files
 * straight into a buffer from hg_host_alloc instead of a Vec.  hg_host_free(NULL) is a no-op. */
HG_API int hg_host_alloc(uint64_t bytes, void **out);
HG_API int hg_host_free(void *p);
/* Page-lock and map memory the caller already owns (e.g. a POSIX shared-memory segment several processes have
 * mmap'ed) so that this process's GPU can write into it; *dev_ptr is the pointer kernels use. */
HG_API int hg_host_register(void *p, uint64_t bytes, void **dev_ptr);
HG_API int hg_host_unregister(void *p);
HG_API const char *hg_last_error(void);
HG_API const char *hg_version(void);
/* cudaStream_t of the context as an integer handle, so a host framework (torch) can order
 * its own work against it. */
HG_API uint64_t hg_stream_handle(hg_ctx *ctx);
/* number of kernel launches issued through this context so far (bench `gpu_launches`) */
HG_API uint64_t hg_launch_count(hg_ctx *ctx);
/* Measurement support.  hg_set_profiling(ctx, 1) records CUDA events on the context stream
 * around every stage; after hg_sync(), hg_stage_ms() returns the device time of the last
 * call's stages in ms: [0] staging + table clears, [1] k-mer hash kernel, [2] encode kernel,
 * [3] dist kernel(s).  Entries that did not run are -1. */
HG_API int hg_set_profiling(hg_ctx *ctx, int enabled);
HG_API int hg_stage_ms(hg_ctx *ctx, float out_ms[4]);
/* Dependent-free integer issue-rate probe used as the INT32 roofline denominator:
 * which = 0 IMAD chain mix, 1 LOP3/IADD3/SHF mix, 2 both interleaved.  Returns lane-ops/s. */
HG_API int hg_int_peak(hg_ctx *ctx, int which, double *lane_ops_per_s);
/* tcgen05 kind::i8 issue-rate probe used as the dist roofline denominator: the dist kernels' MMA shape (cta_group::2,
 * 256 x 256 x 32) back to back from resident shared-memory operands on every TPC.  Returns integer ops / s (2 per MAC).
 * Both probes are measurement hooks of this build, not part of the interface a host binds. */
HG_API int hg_tensor_peak(hg_ctx *ctx, double *ops_per_s);
/* Which rows of d_hv (n_rows x hv_d, on the device) the tensor kernel `path` (2 two-limb, 3 single plane) takes as
 * rows whose true norm sum x^2 reaches ceil(2^31 / 3), i.e. rows whose every pair skips the candidate bound:
 * d_flags[i] = 1 or 0, from the kernel's own row preparation.  HG_E_UNSUPPORTED for path 3 if its pre-pass declines
 * the rows.  Synchronous.  A measurement hook like the probes above. */
HG_API int hg_dist_norm_flags(hg_ctx *ctx, const int16_t *d_hv, uint32_t n_rows, uint32_t hv_d, int path, uint32_t *d_flags);

/* ---- stage 1: sketch -------------------------------------------------------------- */

/* Stage hook = extract_kmer_t1ha2_cuda (src/sketch_cuda.rs:119-166) for a batch: the set of
 * sampled canonical k-mer hashes of each genome, SORTED ascending and de-duplicated (the
 * reference builds a HashSet, src/sketch_cuda.rs:158-163; unlike it, nothing is dropped
 * when a 512-k-mer chunk yields more than 8 samples, and h == 0 is kept).
 *   seq      concatenated sequence bytes, genome g = seq[seg_off[g] .. seg_off[g+1])
 *            (what fastx_reader::read_merge_seq returns, src/fastx_reader.rs:6-29)
 *   hash_off n_genomes+1 prefix offsets into `hashes` (written)
 *   hashes   capacity `cap` u64; on HG_E_CAPACITY hash_off[n_genomes] holds the need. */
HG_API int hg_kmer_hash(hg_ctx *ctx, const uint8_t *seq, const uint64_t *seg_off, uint32_t n_genomes,
                        const hg_sketch_params *p, uint64_t *hashes, uint64_t cap, uint64_t *hash_off);

/* The whole per-file body of sketch_cuda (src/sketch_cuda.rs:79-100) for a batch of files:
 * k-mer hash set -> encode_hash_hd_avx2 layout (src/hd.rs:15-92) -> compute_hv_l2_norm
 * (src/dist.rs:132-137) -> compress_hd_sketch (src/hd.rs:116-157).
 *   hv         optional (NULL ok) n_genomes x hv_d int16, the uncompressed sketch HVs
 *   packed     n_genomes rows of 2*hv_d bytes; row g holds quant_bits[g]*hv_d/8 valid
 *              bytes = FileSketch.hv reinterpreted as bytes (src/hd.rs:155-157)
 *   quant_bits FileSketch.hv_quant_bits, norm2 FileSketch.hv_norm_2, n_hashes set sizes */
HG_API int hg_sketch_batch(hg_ctx *ctx, const uint8_t *seq, const uint64_t *seg_off, uint32_t n_genomes,
                           const hg_sketch_params *p, int16_t *hv, uint8_t *packed,
                           uint8_t *quant_bits, int32_t *norm2, uint32_t *n_hashes);

/* Same with `d_seq` and every output in device memory; seg_off stays a HOST array (the
 * tile schedule is built from it).  Asynchronous on the context stream. */
HG_API int hg_sketch_batch_dev(hg_ctx *ctx, const uint8_t *d_seq, const uint64_t *seg_off,
                               uint32_t n_genomes, const hg_sketch_params *p, int16_t *d_hv,
                               uint8_t *d_packed, uint8_t *d_quant_bits, int32_t *d_norm2,
                               uint32_t *d_n_hashes);
/* After hg_sync(): HG_OK, or HG_E_RANGE / HG_E_CAPACITY if any genome of the last
 * hg_sketch_batch_dev overflowed (never silently truncated). */
HG_API int hg_sketch_status(hg_ctx *ctx);

/* Stage hook = hd::encode_hash_hd_avx2 + compute_hv_l2_norm + compress_hd_sketch
 * (src/hd.rs:15-92,116-157, src/dist.rs:132-137) from explicit hash SETS (unique values,
 * as the reference's HashSet argument): set g = hashes[hash_off[g] .. hash_off[g+1]).
 * Every element is a hash, 0 and u64::MAX included.  hv_d <= 32000 (HG_E_UNSUPPORTED above).
 * Host pointers; outputs as hg_sketch_batch. */
HG_API int hg_encode_sets(hg_ctx *ctx, const uint64_t *hashes, const uint64_t *hash_off, uint32_t n_sets,
                          uint32_t hv_d, int16_t *hv, uint8_t *packed, uint8_t *quant_bits, int32_t *norm2);
/* Same with `d_hashes` and the outputs in device memory (hash_off stays on the host). */
HG_API int hg_encode_sets_dev(hg_ctx *ctx, const uint64_t *d_hashes, const uint64_t *hash_off,
                              uint32_t n_sets, uint32_t hv_d, int16_t *d_hv, uint8_t *d_packed,
                              uint8_t *d_quant_bits, int32_t *d_norm2);

/* ---- FASTA file bytes in -------------------------------------------------------------- */

/* fastx_reader::read_merge_seq (src/fastx_reader.rs:6-29) for a batch of files, on the GPU:
 * file f = raw[file_off[f] .. file_off[f+1]) exactly as read from disk.  Every line starting
 * with '>' becomes one 'N', every other line loses its trailing '\n' and one '\r' before it.
 * merged_off (n_files + 1) receives the prefix offsets of the merged sequences in `merged`
 * (capacity `cap`; HG_E_CAPACITY reports the need in merged_off[n_files]).  Stage hook. */
HG_API int hg_fasta_merge(hg_ctx *ctx, const uint8_t *raw, const uint64_t *file_off, uint32_t n_files,
                          uint8_t *merged, uint64_t cap, uint64_t *merged_off);

/* hg_sketch_batch fed with raw FASTA files: the merge above, then the sketch pipeline, without
 * the merged sequences ever visiting the host.  Outputs as hg_sketch_batch. */
HG_API int hg_sketch_fasta_batch(hg_ctx *ctx, const uint8_t *raw, const uint64_t *file_off, uint32_t n_files,
                                 const hg_sketch_params *p, int16_t *hv, uint8_t *packed,
                                 uint8_t *quant_bits, int32_t *norm2, uint32_t *n_hashes);

/* One record of a FASTA file, as hg_sketch_fasta_records reports it.  A file's records, in file
 * order: every line that starts with '>' opens one; its sequence is the merged bytes (as
 * hg_fasta_merge merges them) of its sequence lines up to the next header or the end of the file,
 * without the header's own 'N'.  Merged bytes before a file's first header (or of a file without
 * one) form one leading record first, with has_header = 0; a file with no such byte has none. */
typedef struct hg_fasta_record {
  uint64_t name_off;   /* index into raw (the indexing of file_off) of the first byte after '>'          */
  uint64_t name_len;   /* header text bytes, without the line's '\n' and one '\r' before it              */
  uint64_t seq_len;    /* bases of the record's merged sequence: what was hashed                          */
  uint32_t file;       /* index of the record's file in this call                                         */
  uint32_t has_header; /* 0 only for the leading record of a file (sequence before its first header)     */
} hg_fasta_record;     /* 32 bytes */

/* hg_sketch_fasta_batch with one sketch per record instead of one per file.  Record r's row of
 * packed, quant_bits, norm2 and n_hashes is what hg_sketch_fasta_batch returns for a file holding
 * that record alone (its header line, if any, and its sequence lines).  Records go out in file
 * order, then record order; *n_records always receives their count.  A file that contains c '>'
 * bytes holds at most c + 1 records, so rec_cap = (the '>' bytes of all files) + n_files always
 * suffices.  More records than rec_cap: HG_E_CAPACITY and nothing else is written; more than
 * 2^32 - 1: HG_E_UNSUPPORTED.  Any output pointer but n_records may be NULL (not copied). */
HG_API int hg_sketch_fasta_records(hg_ctx *ctx, const uint8_t *raw, const uint64_t *file_off, uint32_t n_files,
                                   const hg_sketch_params *p, uint32_t rec_cap, hg_fasta_record *records,
                                   uint8_t *packed /* rec_cap rows of 2 * hv_d bytes */, uint8_t *quant_bits,
                                   int32_t *norm2, uint32_t *n_hashes, uint32_t *n_records);
/* The last hg_sketch_fasta_records call on this context: counts = [chunks, records, record table slots (one
 * leading slot per file included), 0]; with hg_set_profiling on, ms = device ms of [merge, record index, k-mer
 * hash, encode] summed over the chunks and host_gap_ms = the device time between the index pass and the hash
 * stage spent waiting for the host (the two record table round trips and the planning); -1 otherwise. */
HG_API int hg_fasta_records_stats(hg_ctx *ctx, uint64_t counts[4], float ms[4], float *host_gap_ms);

/* ---- sketch format ---------------------------------------------------------------- */

/* decompress_hd_sketch (src/hd.rs:184-212) for n sketches on the GPU: packed rows of
 * `row_stride` bytes -> n x hv_d int16.  Host pointers. */
HG_API int hg_unpack(hg_ctx *ctx, const uint8_t *packed, uint64_t row_stride, const uint8_t *quant_bits,
                     uint32_t n, uint32_t hv_d, int16_t *hv);
HG_API int hg_unpack_dev(hg_ctx *ctx, const uint8_t *d_packed, uint64_t row_stride,
                         const uint8_t *d_quant_bits, uint32_t n, uint32_t hv_d, int16_t *d_hv);

/* ---- stage 2: dist ---------------------------------------------------------------- */

/* compute_hv_ani + the threshold filter of dump_ani_file (src/dist.rs:231-294,
 * src/utils.rs:274-285): every (ref i, query j) pair — only j > i when `symmetric`
 * (same ref/query sketch file, src/dist.rs:13,253-265) — gets the exact i32 dot, the ANI
 * of src/dist.rs:153-160, and is reported iff ani >= ani_th.  The order of the hits is
 * unspecified (the reference sorts by ANI when it writes its output, src/utils.rs:262-269).
 * If more than `cap` pairs pass, returns HG_E_CAPACITY with *n_hits = need.
 *   path: 0 = auto: the single-plane tcgen05 int8 kernel when the rows are narrow (sketch rows are
 *             hv = 2 count - n, one parity per row; x = 2a + s with a in s8 when the row spans
 *             <= 510 — every hv_quant_bits = 9 sketch — plus sparse exact corrections for the odd
 *             element outside), else the two-limb tcgen05 int8 kernel when every |hv| fits 13
 *             bits, else SIMT; fewer than 128 x 128 pairs go to SIMT directly,
 *         1 = force SIMT (CUDA-core) path, 2 = force the two-limb tensor path,
 *         3 = force the single-plane tensor path (HG_E_UNSUPPORTED if the rows are not narrow).
 *   Every path is exact: identical i32 dots and f32 ANI bits.
 *   The host-pointer entries (hg_dist, hg_dist_sorted, hg_dist_packed) with path 0 or 3 stream the rows
 *   in chunks: the H2D copy of one chunk runs under the unpack / pre-pass / kernel of the previous ones. */
HG_API int hg_dist(hg_ctx *ctx, const int16_t *ref_hv, const int32_t *ref_norm2, uint32_t n_ref,
                   const int16_t *qry_hv, const int32_t *qry_norm2, uint32_t n_qry, uint32_t hv_d,
                   uint32_t ksize, float ani_th, int symmetric, int path, hg_hit *hits, uint64_t cap,
                   uint64_t *n_hits);

/* Device-resident variant: HVs/norms/hits in HBM, hit order unspecified (atomic append),
 * *d_n_hits counts every passing pair even beyond cap.  (i, j) are offset by i0 / j0 so a
 * row shard of a larger ref matrix reports global indices; with `symmetric` the filter is
 * global_j > global_i.  Work is enqueued on the context stream; paths 1, 2 and 3 return without waiting
 * for it; path 0 waits once at the end (the host reads the single-plane pre-pass's verdict there, after
 * the kernel has been enqueued behind it, so the GPU never idles on that read).  With path 3 the caller
 * asserts that the rows are narrow: if they are not, the kernel does nothing and hg_dist_status() says so. */
HG_API int hg_dist_dev(hg_ctx *ctx, const int16_t *d_ref_hv, const int32_t *d_ref_norm2, uint32_t n_ref,
                       uint32_t i0, const int16_t *d_qry_hv, const int32_t *d_qry_norm2,
                       uint32_t n_qry, uint32_t j0, uint32_t hv_d, uint32_t ksize, float ani_th,
                       int symmetric, int path, hg_hit *d_hits, uint64_t cap,
                       unsigned long long *d_n_hits);

/* After hg_dist_dev(path = 3) (synchronises the stream): HG_OK, or HG_E_UNSUPPORTED if the rows were not
 * narrow - the forced call then produced no hits and the caller must use path 0 / 2 / 1. */
HG_API int hg_dist_status(hg_ctx *ctx);

/* ---- output stage ------------------------------------------------------------------ */

/* The order of utils::dump_ani_file (src/utils.rs:262-285): a stable ascending sort by ANI,
 * reversed - i.e. ANI descending, equal ANIs in DESCENDING pair-enumeration index, which for
 * both enumerations (src/dist.rs:243-265) is (i descending, j descending).  Sorts the n device
 * records in place with an on-device radix sort.  If d_ani_milli is not NULL it also receives,
 * per sorted record, the ANI in thousandths rounded exactly as the `{:.3}` of src/utils.rs:280
 * prints it (so the host writes "%u.%03u"). */
HG_API int hg_sort_hits_dev(hg_ctx *ctx, hg_hit *d_hits, uint64_t n, uint32_t *d_ani_milli);

/* hg_dist followed by hg_sort_hits_dev: host pointers in, the hits in the reference's output
 * order out (ani_milli may be NULL).  Same capacity contract as hg_dist. */
HG_API int hg_dist_sorted(hg_ctx *ctx, const int16_t *ref_hv, const int32_t *ref_norm2, uint32_t n_ref,
                          const int16_t *qry_hv, const int32_t *qry_norm2, uint32_t n_qry, uint32_t hv_d,
                          uint32_t ksize, float ani_th, int symmetric, int path, hg_hit *hits,
                          uint32_t *ani_milli, uint64_t cap, uint64_t *n_hits);

/* `dist` straight from the sketch-file payload: bit-packed rows (FileSketch.hv as bytes,
 * src/types.rs:224-235; row g holds quant_bits[g] * hv_d / 8 live bytes, rows `*_stride` bytes
 * apart), hv_quant_bits and hv_norm_2.  Only the live bytes cross PCIe; decompress_file_sketch
 * (src/hd.rs:171-232) runs on the device in front of the dist kernel.  sorted != 0: the hits
 * come back in dump_ani_file's order as from hg_dist_sorted (ani_milli may be NULL); otherwise
 * as from hg_dist and ani_milli is NOT written (the output-stage sort produces it).  Pass the same pointers for ref and query for the symmetric all-vs-all. */
HG_API int hg_dist_packed(hg_ctx *ctx, const uint8_t *ref_packed, uint64_t ref_stride, const uint8_t *ref_quant_bits,
                          const int32_t *ref_norm2, uint32_t n_ref, const uint8_t *qry_packed,
                          uint64_t qry_stride, const uint8_t *qry_quant_bits, const int32_t *qry_norm2,
                          uint32_t n_qry, uint32_t hv_d, uint32_t ksize, float ani_th, int symmetric, int path,
                          int sorted, hg_hit *hits, uint32_t *ani_milli, uint64_t cap, uint64_t *n_hits);

/* ---- several GPUs of one box ---------------------------------------------------------- */

/* The reference drives one GPU (CudaDevice::new(0), src/sketch_cuda.rs:52) and has no GPU dist at all
 * (src/dist.rs:231-294 is a rayon loop); SURVEY.md 8e shards the path over the GPUs of one box:
 * genome files split across GPUs for sketching (no exchange), ref rows sharded / queries broadcast /
 * hits gathered for dist.  The exchange runs over NVLink windows owned by the library (no collective
 * library on the data path, see csrc/peer.cu).
 *
 * hg_group: ONE process driving all GPUs - what `hyper-gen sketch -D gpu` and `hyper-gen dist` call. */
typedef struct hg_group hg_group;
#define HG_MAX_PEERS 8
/* n_devices <= 0: every visible GPU (at most HG_MAX_PEERS); ordinals may be NULL (0 .. n-1). */
HG_API int hg_group_create(int n_devices, const int *ordinals, hg_group **out);
HG_API void hg_group_destroy(hg_group *g);
HG_API int hg_group_size(const hg_group *g);
HG_API hg_ctx *hg_group_ctx(hg_group *g, int i);
/* hg_sketch_fasta_batch with the files split into one contiguous run per GPU of about equal bytes
 * (sketch_cuda's par_iter over files, src/sketch_cuda.rs:79, across GPUs); same arguments and outputs. */
HG_API int hg_group_sketch_fasta_batch(hg_group *g, const uint8_t *raw, const uint64_t *file_off, uint32_t n_files,
                                       const hg_sketch_params *p, int16_t *hv, uint8_t *packed, uint8_t *quant_bits,
                                       int32_t *norm2, uint32_t *n_hashes);
/* hg_sketch_fasta_records with the files split as hg_group_sketch_fasta_batch splits them; every GPU keeps its
 * rows until the group has checked the total against rec_cap.  Same arguments, outputs and bytes as one GPU. */
HG_API int hg_group_sketch_fasta_records(hg_group *g, const uint8_t *raw, const uint64_t *file_off, uint32_t n_files,
                                         const hg_sketch_params *p, uint32_t rec_cap, hg_fasta_record *records,
                                         uint8_t *packed, uint8_t *quant_bits, int32_t *norm2, uint32_t *n_hashes,
                                         uint32_t *n_records);
/* hg_dist_packed with the rows of both sketch files split into one block per GPU: each block crosses its
 * own GPU's PCIe link, is unpacked and brought into operand form there, the query operands are pushed to
 * every GPU, the output tiles are shared out, the hits land on GPU 0 (sorted there if asked).  Results are
 * identical to hg_dist_packed (the unsorted order is unspecified in both). */
HG_API int hg_group_dist_packed(hg_group *g, const uint8_t *ref_packed, uint64_t ref_stride, const uint8_t *ref_quant_bits,
                                const int32_t *ref_norm2, uint32_t n_ref, const uint8_t *qry_packed, uint64_t qry_stride,
                                const uint8_t *qry_quant_bits, const int32_t *qry_norm2, uint32_t n_qry, uint32_t hv_d,
                                uint32_t ksize, float ani_th, int symmetric, int sorted, hg_hit *hits, uint32_t *ani_milli,
                                uint64_t cap, uint64_t *n_hits);
/* hg_search_packed with the refs split into contiguous blocks of about equal size, one per GPU (as many GPUs as give
 * every block at least 1024 refs): each GPU receives its ref block and all query rows over its own PCIe link and
 * searches them; the per-block results are copied to GPU 0 and merged there (hg_search_merge_dev).  Same arguments,
 * results identical to hg_search_packed.  One GPU in use (g has one member, or fewer than 2048 refs): hg_search_packed
 * on member 0.  Members that share a device ordinal run one after another.  hg_search_stats on hg_group_ctx(g, m)
 * reports member m's passes (all zero for a member without a block). */
HG_API int hg_group_search_packed(hg_group *g, const uint8_t *ref_packed, uint64_t ref_stride, const uint8_t *ref_quant_bits,
                                  const int32_t *ref_norm2, uint32_t n_ref, const uint8_t *qry_packed, uint64_t qry_stride,
                                  const uint8_t *qry_quant_bits, const int32_t *qry_norm2, uint32_t n_qry, uint32_t hv_d,
                                  uint32_t ksize, uint32_t top_k, float ani_min, int path,
                                  hg_hit *out, uint32_t *n_found, uint32_t *ani_milli /* may be NULL */);

/* hg_peer: one member of a group of GPUs, for hosts that run ONE PROCESS PER GPU.  Every member
 * allocates a window (hg_peer_create), the host exchanges the HG_IPC_HANDLE_BYTES-byte handles by its
 * own means (an all-gather), and every member maps the others' windows (hg_peer_connect). */
typedef struct hg_peer hg_peer;
#define HG_IPC_HANDLE_BYTES 64
/* bytes a window needs for a sharded dist whose gathered (query) matrix has `gathered_rows` rows */
HG_API uint64_t hg_peer_window_need(uint32_t gathered_rows, uint32_t hv_d, uint64_t hit_cap);
HG_API int hg_peer_create(hg_ctx *ctx, int rank, int world, uint64_t window_bytes, uint8_t handle_out[HG_IPC_HANDLE_BYTES],
                          hg_peer **out);
HG_API int hg_peer_connect(hg_peer *p, const uint8_t *handles /* world x HG_IPC_HANDLE_BYTES, rank order */);
/* members of one process instead (what hg_group uses): out[0 .. world) */
HG_API int hg_peer_create_local(hg_ctx *const *ctxs, int world, uint64_t window_bytes, hg_peer **out);
HG_API void hg_peer_destroy(hg_peer *p);
HG_API int hg_peer_rank(const hg_peer *p);
HG_API int hg_peer_world(const hg_peer *p);
/* enqueue a barrier among the members on this member's stream (bounded wait: HG_PEER_TIMEOUT_MS, default 10 s) */
HG_API int hg_peer_barrier(hg_peer *p);
/* Collective sharded dist, rows resident in HBM (compute_hv_ani, src/dist.rs:231-294, over several GPUs).
 * Every member calls it with the same scalars and ITS rows.  qry_bounds (world + 1 entries, [0] = 0) says which rows
 * of the gathered ("query") matrix each member holds: member m has rows [qry_bounds[m], qry_bounds[m + 1]) - d_qry_hv /
 * d_qry_norm2 point at this member's block (it may be empty; one member may hold everything: a broadcast).
 *   symmetric != 0  all-vs-all (j > i, src/dist.rs:253-265) over that ONE matrix; the ref arguments are ignored.  With
 *                   block boundaries that are multiples of 256 rows a block pair is computed by the member from which
 *                   the other block is at most world / 2 steps ahead on the ring, and a member's rows travel only to
 *                   those world / 2 members; otherwise the non-empty output tiles are dealt round-robin and every row
 *                   goes to every member (hg_peer_plan_tiles / hg_peer_plan_push show the plan);
 *   symmetric == 0  this member's n_ref_local resident ref rows (global index ref_row0 + row) against ALL gathered rows.
 *   path  0 auto (one host read of all members' pre-pass verdict; two-limb kernel if the rows are not narrow),
 *         3 / 2 single-plane / two-limb tensor kernel asserted by the caller: the call only enqueues.
 * Hits carry global (i, j) and go to member `root`: into its window (capacity `cap`, same on every member), or - if
 * mapped_hits is not NULL - into a HOST buffer of `cap` records that every member has mapped (the same physical
 * memory: hg_host_alloc in a one-process group, a shared-memory segment passed through hg_host_register by every
 * process otherwise; each member passes ITS device pointer to it).  Every member collects its hits in its own window
 * and moves them to the root's list / the host buffer in one piece after its kernel (over NVLink / its own PCIe link). */
HG_API int hg_dist_sharded_dev(hg_peer *p, const int16_t *d_ref_hv, const int32_t *d_ref_norm2, uint32_t n_ref_local,
                               uint32_t ref_row0, const int16_t *d_qry_hv, const int32_t *d_qry_norm2, const uint32_t *qry_bounds,
                               uint32_t hv_d, uint32_t ksize, float ani_th, int symmetric, int path, int root, uint64_t cap,
                               hg_hit *mapped_hits);
/* Waits for this member's part.  On the root: *n_hits and the hits copied to HOST memory, in dump_ani_file's
 * order if `sorted` (ani_milli as in hg_dist_sorted; may be NULL); HG_E_CAPACITY with the need if they exceed
 * cap.  After a call with mapped_hits the records already are in that buffer: nothing is copied (hits may be NULL,
 * `sorted` is not available).  On the other members *n_hits = 0 and hits may be NULL. */
HG_API int hg_dist_sharded_hits(hg_peer *p, int sorted, hg_hit *hits, uint32_t *ani_milli, uint64_t cap, uint64_t *n_hits);
/* Host logic of the sharded dist, no GPU involved: the tiles member `rank` of `world` computes (path 3: 256 x 256
 * tiles, path 2: 256 x 128), in the order it walks them - tiles_out[2 t] = tile row | tile column << 16,
 * tiles_out[2 t + 1] = mask of the arrival flags (member m, chunk c -> bit 4 m + c) the tile waits for. */
HG_API int hg_peer_plan_tiles(int world, int rank, int symmetric, int path, uint32_t hv_d, uint32_t n_ref_local,
                              const uint32_t *qry_bounds, uint32_t *tiles_out, uint64_t cap, uint64_t *n_tiles);
/* ... and what the member sends: chunk_rows_out[c .. c + 1] = the rows of its chunk c (a block is cut into 1..4 chunks
 * of about 2 MB of operand bytes or more), units_out[2 u] = what push unit u sends (chunk index, or 4 = the start set:
 * pre-pass statistics and outlier entries), units_out[2 u + 1] = mask of the members it goes to, in sending order;
 * *ring = 1 when rows go only to the floor(world / 2) members that compute with them (all-vs-all, block boundaries
 * multiples of 256 rows). */
HG_API int hg_peer_plan_push(int world, int rank, int symmetric, int path, uint32_t hv_d, const uint32_t *qry_bounds,
                             uint32_t chunk_rows_out[5], uint32_t *units_out, uint64_t cap, uint64_t *n_units, int *ring);
/* Measurement support (hg_set_profiling on the member's context): device ms of the last sharded dist's stages -
 * [0] operand form of this member's rows, [1] chunked push to the peers, [2] dist kernel (with its waits for the
 * peers' chunks), [3] final barrier.  Synchronises the member's stream. */
HG_API int hg_peer_stage_ms(hg_peer *p, float out_ms[4]);
/* Measurement support, with HG_PEER_TIMELINE=1 in the environment when the member is created: %globaltimer stamps (ns) the
 * kernels of the last sharded dist left in the member's window: [0] first node, [1] dist kernel entry, [2] start flags seen,
 * [3] ns CTA 0's producer waited for other members' rows, [4] last CTA done, [5] longest producer wait, [8..11] chunk c pushed,
 * [12] hit flush, [13] barrier entry, [14] barrier exit, [16] barrier exit of the call before (the members' common time
 * base).  Synchronises the member's stream.  No counterpart in the reference. */
HG_API int hg_peer_timeline(hg_peer *p, unsigned long long out_ns[32]);
/* the root's hit list and counter as this member addresses them (device pointers) */
HG_API int hg_peer_hit_buffers(hg_peer *p, int root, hg_hit **d_hits, unsigned long long **d_count);

/* ---- top-k search: the best-matching refs of every query ------------------------------------------
 * Every (i, j) of ref rows R x query rows Q, as hg_dist with symmetric = 0 (the same pointers for ref and
 * query are a plain R x R search, self hits included).  For query j the result is the refs with the top_k
 * largest ANIs among those with ani >= ani_min, ordered by ANI descending and, for equal ANIs, by ascending
 * ref index i; the tie rule also decides membership at the top_k-th place, so the set is exact.  Every
 * record's dot and ANI are bit-identical to hg_dist's.
 *   out        n_qry * top_k records: query j's are out[j * top_k .. j * top_k + n_found[j]), with i = ref
 *              index and j = query index; the unused slots are zeroed
 *   n_found[j] = min(top_k, number of refs with ani >= ani_min)
 *   ani_milli  may be NULL: each record's ANI in thousandths, rounded as hg_sort_hits_dev rounds it (0 in
 *              the unused slots)
 *   top_k      1..1024, else HG_E_INVALID.  n_ref == 0 or n_qry == 0: HG_OK with every n_found 0.
 *   path       as hg_dist (0 auto, 1 SIMT, 2 two-limb, 3 single plane) with the same choice and fallbacks;
 *              hg_dist_last_path / hg_dist_last_reason report the main pass.
 * Both entries return with the result complete.  The candidate lists between the passes are library scratch
 * that grows as a pass needs it (DESIGN.md §4, "Top-k search"); no candidate is dropped. */
HG_API int hg_search_dev(hg_ctx *ctx, const int16_t *d_ref, const int32_t *d_ref_norm2, uint32_t n_ref,
                         const int16_t *d_qry, const int32_t *d_qry_norm2, uint32_t n_qry, uint32_t hv_d,
                         uint32_t ksize, uint32_t top_k, float ani_min, int path,
                         hg_hit *d_out, uint32_t *d_n_found, uint32_t *d_ani_milli /* may be NULL */);
/* The same from the rows as the sketch files hold them (as hg_dist_packed: packed bytes + hv_quant_bits +
 * norms, unpacked on the device); results in host memory. */
HG_API int hg_search_packed(hg_ctx *ctx, const uint8_t *ref_packed, uint64_t ref_stride, const uint8_t *ref_quant_bits,
                            const int32_t *ref_norm2, uint32_t n_ref, const uint8_t *qry_packed, uint64_t qry_stride,
                            const uint8_t *qry_quant_bits, const int32_t *qry_norm2, uint32_t n_qry, uint32_t hv_d,
                            uint32_t ksize, uint32_t top_k, float ani_min, int path,
                            hg_hit *out, uint32_t *n_found, uint32_t *ani_milli /* may be NULL */);
/* Measurement hook of the last search: counts = {sample rows s (= n_ref: one pass), floor-pass candidates,
 * main-pass candidates, reruns after a candidate list outgrew its scratch}; ms = device time of the floor
 * pass (gather + dist), its select, the main pass, its select (-1 where not run or profiling is off, see
 * hg_set_profiling). */
HG_API int hg_search_stats(hg_ctx *ctx, uint64_t counts[4], float ms[4]);
/* The search over refs cut into contiguous blocks, from the search of each block: list m (m < n_lists) is what
 * hg_search_dev wrote for block m, which starts at global ref index i0[m] - records d_in[(m * n_qry + j) * top_k ..],
 * counts d_in_found[m * n_qry + j].  The result is what one search over all blocks writes (d_out, d_n_found,
 * d_ani_milli as hg_search_dev), with i = block index + i0[m].  Exact: the global top_k of a query is a subset of the
 * union of the blocks' top_k, and within a contiguous block the ref order is the global order, so ties come out by
 * ascending global index.  Device pointers; returns with the result complete.  A host that runs one process per GPU
 * searches its own ref block, gathers the ranks' lists into one device buffer by its own means and calls this.
 *   n_lists 1..HG_SEARCH_MERGE_MAX_LISTS, top_k 1..1024; an i + i0[m] beyond 32 bits or an input count above top_k:
 *   HG_E_INVALID. */
#define HG_SEARCH_MERGE_MAX_LISTS 64
HG_API int hg_search_merge_dev(hg_ctx *ctx, uint32_t n_lists, const hg_hit *d_in, const uint32_t *d_in_found,
                               const uint32_t *i0 /* host, n_lists entries */, uint32_t n_qry, uint32_t top_k, hg_hit *d_out,
                               uint32_t *d_n_found, uint32_t *d_ani_milli /* may be NULL */);

/* ---- ANI clustering: which sketches of one set belong together ---------------------------------------------------
 * Single linkage over one sketch set of n rows, all against all: sketches i < j are linked when ani(i, j) >= ani_th -
 * exactly the pairs hg_dist(..., symmetric = 1, ani_th) reports - and a cluster is a connected component of that graph.
 * rep[i] = the smallest index in i's cluster (so rep[i] <= i, and rep[i] == i marks a representative); *n_clusters
 * (host, may be NULL) = the number of representatives.  The result does not depend on the kernel, the window plan, the
 * thread schedule or the number of GPUs.  n == 0: HG_OK with n_clusters = 0; ani_th <= 0 links everything (every ANI
 * is >= 0); a sketch with norm 0 has ANI 0 to everything; a NaN ani_th is HG_E_INVALID.
 *   path   as hg_search_dev (0 auto, 1 SIMT, 2 two-limb, 3 single plane) with the same choice and fallbacks;
 *          hg_dist_last_path / hg_dist_last_reason report the run.
 * The linked pairs never leave the device: the dist kernels emit them window by window (at most HG_CLUSTER_EDGE_CAP
 * records each, default 2^26, read at every call) into library scratch, and a lock-free union-find unites each window's
 * pairs behind it (DESIGN.md §4.9).  Every entry returns with its result complete. */
HG_API int hg_cluster_dev(hg_ctx *ctx, const int16_t *d_hv, const int32_t *d_norm2, uint32_t n, uint32_t hv_d,
                          uint32_t ksize, float ani_th, int path, uint32_t *d_rep, uint32_t *n_clusters /* host, may be NULL */);
/* The same from the rows as the sketch file holds them (as hg_dist_packed: packed bytes + hv_quant_bits + norms,
 * unpacked on the device); rep in host memory. */
HG_API int hg_cluster_packed(hg_ctx *ctx, const uint8_t *packed, uint64_t stride, const uint8_t *quant_bits,
                             const int32_t *norm2, uint32_t n, uint32_t hv_d, uint32_t ksize, float ani_th, int path,
                             uint32_t *rep, uint32_t *n_clusters /* may be NULL */);
/* hg_cluster_packed over the GPUs of the group: the upper triangle cut by query column into one range per GPU of about
 * equal pairs (as many GPUs as give each at least 2^23 pairs); each GPU receives the packed rows up to the end of its
 * range over its own PCIe link and builds a forest of its pairs; the forests are united on GPU 0.  Same arguments,
 * result identical to hg_cluster_packed.  One GPU in use: hg_cluster_packed on member 0.  Members that share a device
 * ordinal run one after another.  hg_cluster_stats on hg_group_ctx(g, m) reports member m's run. */
HG_API int hg_group_cluster_packed(hg_group *g, const uint8_t *packed, uint64_t stride, const uint8_t *quant_bits,
                                   const int32_t *norm2, uint32_t n, uint32_t hv_d, uint32_t ksize, float ani_th, int path,
                                   uint32_t *rep, uint32_t *n_clusters /* may be NULL */);
/* Unites the edges (i, j of each record) into an existing forest d_rep (every rep[x] <= x: iota, or a cluster result),
 * then flattens it, so that rep[x] is the smallest index of x's component; device pointers.  An index >= n or a
 * rep[x] > x: HG_E_INVALID before anything is written.  The merge step for a host that runs one process per GPU. */
HG_API int hg_cluster_union_dev(hg_ctx *ctx, uint32_t n, uint32_t *d_rep, const hg_hit *d_edges, uint64_t n_edges,
                                uint32_t *n_clusters /* host, may be NULL */);
/* Measurement hook of the last cluster run: counts = {windows, linked pairs, largest window's pairs, edge capacity};
 * ms = device time of {preparing the rows, the dist windows, the hooks, flatten + count} (-1 where not run or profiling
 * is off, see hg_set_profiling). */
HG_API int hg_cluster_stats(hg_ctx *ctx, uint64_t counts[4], float ms[4]);

/* ---- greedy ANI dereplication: one representative per group, every other sketch assigned to one -----------------
 * Over one sketch set of n rows at ani_th, in the priority order `order` (host, n entries, a permutation of [0, n);
 * NULL: file order, order[t] = t).  Every ANI is the exact value hg_dist computes.
 *   1. Sketch order[t] is a representative iff no earlier representative order[s] (s < t) has
 *      ani(order[s], order[t]) >= ani_th.
 *   2. A representative's rep is itself.  Any other sketch g goes to the representative r with the largest ani(r, g)
 *      among those with ani(r, g) >= ani_th (never empty: the one that excluded g is there); ties go to the
 *      representative first in `order`.  It may come before or after g in the order.
 * rep[i] = the index of sketch i's representative (rep[r] == r exactly for representatives); *n_reps (host, may be
 * NULL) = the number of representatives.  The result does not depend on the kernel, the window plan or the thread
 * schedule.  n == 0: HG_OK with n_reps = 0; ani_th <= 0: order[0] is the only representative; a sketch with norm 0 is
 * its own representative when ani_th > 0.  A NaN ani_th, or an order with an index >= n or a repeat, is HG_E_INVALID
 * before anything runs; HG_E_CUDA with "internal error" if a non-representative matched no representative.
 *   path   as hg_cluster_dev; hg_dist_last_path / hg_dist_last_reason report the representative phase, and
 *          hg_search_stats the top-1 search of the assignment phase (zeros when every sketch is a representative).
 * On one GPU: the representatives come from the dist windows of hg_cluster_dev (at most HG_CLUSTER_EDGE_CAP pairs
 * each, and at most 1024 columns) with a greedy step on the device behind each column chunk; then one top-1 search of
 * every sketch against the representatives (DESIGN.md §4.10).  Every entry returns with its result complete. */
HG_API int hg_derep_dev(hg_ctx *ctx, const int16_t *d_hv, const int32_t *d_norm2, uint32_t n, uint32_t hv_d, uint32_t ksize,
                        float ani_th, int path, const uint32_t *order /* host, n entries, may be NULL */,
                        uint32_t *d_rep, uint32_t *n_reps /* host, may be NULL */);
/* The same from the rows as the sketch file holds them (as hg_cluster_packed); rep in host memory. */
HG_API int hg_derep_packed(hg_ctx *ctx, const uint8_t *packed, uint64_t stride, const uint8_t *quant_bits, const int32_t *norm2,
                           uint32_t n, uint32_t hv_d, uint32_t ksize, float ani_th, int path, const uint32_t *order,
                           uint32_t *rep, uint32_t *n_reps /* may be NULL */);
/* Measurement hook of the last derep run: counts = {column chunks, windows, linked pairs, representatives};
 * ms = device time of {preparing the rows (the permutation included), the dist windows, the mark hooks + greedy
 * steps, the assignment (gather + search + finalize)} (-1 where not run or profiling is off, see hg_set_profiling). */
HG_API int hg_derep_stats(hg_ctx *ctx, uint64_t counts[4], float ms[4]);

/* ---- the all-vs-all ANI matrix ----------------------------------------------------------------------------------
 * Entry (i, j) is bit for bit the `ani` that hg_dist(..., ani_th = 0, symmetric = 0) reports for ref row i and query row
 * j (clamped to [0, 100], NaN as 0: that call reports every pair), through every kernel and where the i32 norms and
 * denominators wrap.  f32 values.  Two layouts, chosen by `lower`:
 *   lower = 0, rectangle: out[i * ld + j] for every i < n_ref, j < n_qry, with ld >= n_qry; the cells between rows are
 *     never written.  With the same rows as ref and query it is the full square; the diagonal is whatever the kernel
 *     gives the self pair.
 *   lower = 1, strict lower triangle of one set: ref and query must be the same rows (same pointers and n), else
 *     HG_E_INVALID.  Row i holds j < i at out[i (i - 1) / 2 + j]: n (n - 1) / 2 entries, the PHYLIP lower-triangular
 *     order.  Only these pairs are copied, and only the band's diagonal block computes more.
 * n = 0, n = 1 in lower mode, or an empty rectangle: HG_OK, nothing written.  Every offset is 64-bit.
 *   path   as hg_cluster_dev (0 auto, 1 SIMT, 2 two-limb, 3 single plane) with the same choice and fallbacks;
 *          hg_dist_last_path / hg_dist_last_reason report the run.
 * The rows are computed in bands of ref rows (HG_MATRIX_BAND_BYTES of output each, read at every call; default 64 MiB):
 * band k + 1's kernel runs while band k's cells are converted and copied (DESIGN.md §4.11).  Every entry returns with
 * its result complete. */
/* Rows, norms and output in HBM; the whole output must fit on the device. */
HG_API int hg_ani_matrix_dev(hg_ctx *ctx, const int16_t *d_ref, const int32_t *d_ref_norm2, uint32_t n_ref, const int16_t *d_qry,
                             const int32_t *d_qry_norm2, uint32_t n_qry, uint32_t hv_d, uint32_t ksize, int path, int lower,
                             float *d_out, uint64_t ld);
/* Rows as the sketch file holds them (as hg_dist_packed), output in host memory; the output never has to fit on the
 * device.  A page-locked `out` (hg_host_alloc or registered) is copied into directly; any other is registered for the
 * call. */
HG_API int hg_ani_matrix_packed(hg_ctx *ctx, const uint8_t *ref_packed, uint64_t ref_stride, const uint8_t *ref_bits,
                                const int32_t *ref_norm2, uint32_t n_ref, const uint8_t *qry_packed, uint64_t qry_stride,
                                const uint8_t *qry_bits, const int32_t *qry_norm2, uint32_t n_qry, uint32_t hv_d, uint32_t ksize,
                                int path, int lower, float *out, uint64_t ld);
/* hg_ani_matrix_packed over the GPUs of the group: the ref rows cut into one contiguous range per member with about the
 * same number of output entries (in lower mode the boundaries grow like sqrt).  A member copies the packed rows it needs
 * over its own link (lower: rows [0, end of its range); rectangle: its range and every query row) and writes its bands
 * straight into `out`.  As many members as give each at least 2^23 entries take part; with one, hg_ani_matrix_packed on
 * member 0.  Members that share a device ordinal run one after another.  The result is byte-identical to
 * hg_ani_matrix_packed; hg_ani_matrix_stats on hg_group_ctx(g, m) reports member m's part. */
HG_API int hg_group_ani_matrix_packed(hg_group *g, const uint8_t *ref_packed, uint64_t ref_stride, const uint8_t *ref_bits,
                                      const int32_t *ref_norm2, uint32_t n_ref, const uint8_t *qry_packed, uint64_t qry_stride,
                                      const uint8_t *qry_bits, const int32_t *qry_norm2, uint32_t n_qry, uint32_t hv_d,
                                      uint32_t ksize, int path, int lower, float *out, uint64_t ld);
/* Measurement hook of the last matrix run: counts = {bands, entries written, bytes copied to the host, the kernel path
 * that produced them}; ms = device time of {row preparation (the packed entries: with the rows' upload and unpack), band
 * kernels, dot-to-ANI conversion, copies to the host}
 * (-1 where a stage did not run or profiling is off, see hg_set_profiling). */
HG_API int hg_ani_matrix_stats(hg_ctx *ctx, uint64_t counts[4], float ms[4]);

/* Which path the last hg_dist / hg_dist_dev took (1 SIMT, 2 two-limb tensor, 3 single-plane tensor) and why. */
HG_API int hg_dist_last_path(hg_ctx *ctx);
HG_API const char *hg_dist_last_reason(hg_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* HYPERGEN_B200_H */
