//! `extern "C"` surface of libhypergen_b200 (include/hypergen_b200.h) as bindgen emits it, written out by hand so the
//! shim reads without a build.  Takes the place of the cudarc calls of src/sketch_cuda.rs:52-60,134-156.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] pub struct hg_ctx { _private: [u8; 0] }
#[repr(C)] pub struct hg_group { _private: [u8; 0] }

/// FileSketch knobs that reach the kernels (src/types.rs:224-235; defaults src/types.rs:97-113)
#[repr(C)] #[derive(Clone, Copy)]
pub struct hg_sketch_params { pub scaled: u64, pub seed: u64, pub hv_d: u32, pub ksize: u8, pub canonical: u8, pub reserved: [u8; 2] }

/// one reported pair: indices into the ref / query records, exact i32 dot, f32 ANI of src/dist.rs:139-161
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct hg_hit { pub i: u32, pub j: u32, pub dot: i32, pub ani: f32 }

/// one FASTA record of hg_sketch_fasta_records: header text span in raw, merged sequence length, file, 0 for the
/// sequence before a file's first header
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct hg_fasta_record { pub name_off: u64, pub name_len: u64, pub seq_len: u64, pub file: u32, pub has_header: u32 }

pub const HG_OK: c_int = 0;
pub const HG_E_CAPACITY: c_int = -3;

extern "C" {
    pub fn hg_last_error() -> *const c_char;
    pub fn hg_host_alloc(bytes: u64, out: *mut *mut c_void) -> c_int;
    pub fn hg_host_free(p: *mut c_void) -> c_int;
    // every GPU of the box behind one handle (the reference drives CudaDevice::new(0) only, src/sketch_cuda.rs:52)
    pub fn hg_group_create(n_devices: c_int, ordinals: *const c_int, out: *mut *mut hg_group) -> c_int;
    pub fn hg_group_destroy(g: *mut hg_group);
    pub fn hg_group_size(g: *const hg_group) -> c_int;
    pub fn hg_group_sketch_fasta_batch(g: *mut hg_group, raw: *const u8, file_off: *const u64, n_files: u32,
        p: *const hg_sketch_params, hv: *mut i16, packed: *mut u8, quant_bits: *mut u8, norm2: *mut i32,
        n_hashes: *mut u32) -> c_int;
    // one sketch per FASTA record (`sketch -i`); rec_cap = the '>' bytes of all files + n_files always suffices
    pub fn hg_sketch_fasta_records(ctx: *mut hg_ctx, raw: *const u8, file_off: *const u64, n_files: u32,
        p: *const hg_sketch_params, rec_cap: u32, records: *mut hg_fasta_record, packed: *mut u8, quant_bits: *mut u8,
        norm2: *mut i32, n_hashes: *mut u32, n_records: *mut u32) -> c_int;
    pub fn hg_group_sketch_fasta_records(g: *mut hg_group, raw: *const u8, file_off: *const u64, n_files: u32,
        p: *const hg_sketch_params, rec_cap: u32, records: *mut hg_fasta_record, packed: *mut u8, quant_bits: *mut u8,
        norm2: *mut i32, n_hashes: *mut u32, n_records: *mut u32) -> c_int;
    pub fn hg_group_dist_packed(g: *mut hg_group, ref_packed: *const u8, ref_stride: u64, ref_quant_bits: *const u8,
        ref_norm2: *const i32, n_ref: u32, qry_packed: *const u8, qry_stride: u64, qry_quant_bits: *const u8,
        qry_norm2: *const i32, n_qry: u32, hv_d: u32, ksize: u32, ani_th: f32, symmetric: c_int, sorted: c_int,
        hits: *mut hg_hit, ani_milli: *mut u32, cap: u64, n_hits: *mut u64) -> c_int;
    // top-k search with one contiguous ref block per GPU; results identical to hg_search_packed
    pub fn hg_group_search_packed(g: *mut hg_group, ref_packed: *const u8, ref_stride: u64, ref_quant_bits: *const u8,
        ref_norm2: *const i32, n_ref: u32, qry_packed: *const u8, qry_stride: u64, qry_quant_bits: *const u8,
        qry_norm2: *const i32, n_qry: u32, hv_d: u32, ksize: u32, top_k: u32, ani_min: f32, path: c_int,
        out: *mut hg_hit, n_found: *mut u32, ani_milli: *mut u32) -> c_int;
    // the per-block top-k lists (device memory, block m starting at global ref i0[m]) merged into one
    pub fn hg_search_merge_dev(ctx: *mut hg_ctx, n_lists: u32, d_in: *const hg_hit, d_in_found: *const u32, i0: *const u32,
        n_qry: u32, top_k: u32, d_out: *mut hg_hit, d_n_found: *mut u32, d_ani_milli: *mut u32) -> c_int;
    // single-linkage ANI clusters of one sketch set: rep[i] = the smallest index of i's cluster
    pub fn hg_cluster_dev(ctx: *mut hg_ctx, d_hv: *const i16, d_norm2: *const i32, n: u32, hv_d: u32, ksize: u32, ani_th: f32,
        path: c_int, d_rep: *mut u32, n_clusters: *mut u32) -> c_int;
    pub fn hg_cluster_packed(ctx: *mut hg_ctx, packed: *const u8, stride: u64, quant_bits: *const u8, norm2: *const i32, n: u32,
        hv_d: u32, ksize: u32, ani_th: f32, path: c_int, rep: *mut u32, n_clusters: *mut u32) -> c_int;
    // the same with one range of query columns per GPU, the forests united on GPU 0; result identical to hg_cluster_packed
    pub fn hg_group_cluster_packed(g: *mut hg_group, packed: *const u8, stride: u64, quant_bits: *const u8, norm2: *const i32,
        n: u32, hv_d: u32, ksize: u32, ani_th: f32, path: c_int, rep: *mut u32, n_clusters: *mut u32) -> c_int;
    // edge records united into a forest with rep[x] <= x (device memory), then flattened
    pub fn hg_cluster_union_dev(ctx: *mut hg_ctx, n: u32, d_rep: *mut u32, d_edges: *const hg_hit, n_edges: u64,
        n_clusters: *mut u32) -> c_int;
    // counts = {windows, linked pairs, largest window's pairs, edge capacity}; ms of its steps (-1: not run / not profiled)
    pub fn hg_cluster_stats(ctx: *mut hg_ctx, counts: *mut u64, ms: *mut f32) -> c_int;
    // greedy ANI dereplication: representatives in priority order (order: n entries, or null for file order), every
    // other sketch with its closest representative; rep[i] = the index of i's representative
    pub fn hg_derep_dev(ctx: *mut hg_ctx, d_hv: *const i16, d_norm2: *const i32, n: u32, hv_d: u32, ksize: u32, ani_th: f32,
        path: c_int, order: *const u32, d_rep: *mut u32, n_reps: *mut u32) -> c_int;
    pub fn hg_derep_packed(ctx: *mut hg_ctx, packed: *const u8, stride: u64, quant_bits: *const u8, norm2: *const i32, n: u32,
        hv_d: u32, ksize: u32, ani_th: f32, path: c_int, order: *const u32, rep: *mut u32, n_reps: *mut u32) -> c_int;
    // counts = {column chunks, windows, linked pairs, representatives}; ms of its phases (-1: not run / not profiled)
    pub fn hg_derep_stats(ctx: *mut hg_ctx, counts: *mut u64, ms: *mut f32) -> c_int;
    // the ANI of every pair as f32: lower = 1 the strict lower triangle of one set (row i at i (i - 1) / 2), lower = 0
    // the n_ref x n_qry rectangle with rows ld apart; bit for bit hg_dist's ani at ani_th = 0
    pub fn hg_ani_matrix_dev(ctx: *mut hg_ctx, d_ref: *const i16, d_ref_norm2: *const i32, n_ref: u32, d_qry: *const i16,
        d_qry_norm2: *const i32, n_qry: u32, hv_d: u32, ksize: u32, path: c_int, lower: c_int, d_out: *mut f32, ld: u64) -> c_int;
    pub fn hg_ani_matrix_packed(ctx: *mut hg_ctx, ref_packed: *const u8, ref_stride: u64, ref_bits: *const u8, ref_norm2: *const i32,
        n_ref: u32, qry_packed: *const u8, qry_stride: u64, qry_bits: *const u8, qry_norm2: *const i32, n_qry: u32, hv_d: u32,
        ksize: u32, path: c_int, lower: c_int, out: *mut f32, ld: u64) -> c_int;
    pub fn hg_group_ani_matrix_packed(g: *mut hg_group, ref_packed: *const u8, ref_stride: u64, ref_bits: *const u8,
        ref_norm2: *const i32, n_ref: u32, qry_packed: *const u8, qry_stride: u64, qry_bits: *const u8, qry_norm2: *const i32,
        n_qry: u32, hv_d: u32, ksize: u32, path: c_int, lower: c_int, out: *mut f32, ld: u64) -> c_int;
    // counts = {bands, entries, bytes copied to the host, kernel path}; ms of its stages (-1: not run / not profiled)
    pub fn hg_ani_matrix_stats(ctx: *mut hg_ctx, counts: *mut u64, ms: *mut f32) -> c_int;
}

/// status -> panic with the library's message, the reference's error style (`unwrap()`, Cargo.toml:67-70)
pub fn check(rc: c_int) {
    if rc != HG_OK {
        let msg = unsafe { std::ffi::CStr::from_ptr(hg_last_error()) }.to_string_lossy().into_owned();
        panic!("hypergen_b200 error {}: {}", rc, msg);
    }
}
