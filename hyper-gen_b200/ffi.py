"""ctypes binding of include/hypergen_b200.h — the stub a host language adds on its side.

Every function here is a 1:1 call into the C ABI; there is no Python or CPU implementation
of the hot path behind it.  If the shared library (or a CUDA device) is missing the calls
fail loudly.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref

import numpy as np

from . import _build

HG_OK, HG_E_INVALID, HG_E_CUDA, HG_E_CAPACITY, HG_E_RANGE, HG_E_UNSUPPORTED = 0, -1, -2, -3, -4, -5

EXPORTS = [
    "hg_init", "hg_destroy", "hg_sync", "hg_host_alloc", "hg_host_free", "hg_host_register", "hg_host_unregister", "hg_last_error", "hg_version", "hg_stream_handle", "hg_launch_count",
    "hg_set_profiling", "hg_stage_ms", "hg_int_peak", "hg_tensor_peak", "hg_dist_norm_flags", "hg_encode_sets", "hg_encode_sets_dev",
    "hg_fasta_merge", "hg_sketch_fasta_batch", "hg_sketch_fasta_records", "hg_fasta_records_stats",
    "hg_kmer_hash", "hg_sketch_batch", "hg_sketch_batch_dev", "hg_sketch_status", "hg_unpack", "hg_unpack_dev",
    "hg_dist", "hg_dist_dev", "hg_dist_status", "hg_dist_last_path", "hg_dist_last_reason", "hg_sort_hits_dev", "hg_dist_sorted", "hg_dist_packed",
    "hg_search_dev", "hg_search_packed", "hg_search_stats", "hg_search_merge_dev",
    "hg_cluster_dev", "hg_cluster_packed", "hg_cluster_union_dev", "hg_cluster_stats",
    "hg_derep_dev", "hg_derep_packed", "hg_derep_stats",
    "hg_ani_matrix_dev", "hg_ani_matrix_packed", "hg_group_ani_matrix_packed", "hg_ani_matrix_stats",
    "hg_group_create", "hg_group_destroy", "hg_group_size", "hg_group_ctx", "hg_group_sketch_fasta_batch", "hg_group_sketch_fasta_records",
    "hg_group_dist_packed",
    "hg_group_search_packed", "hg_group_cluster_packed",
    "hg_peer_window_need", "hg_peer_create", "hg_peer_connect", "hg_peer_create_local", "hg_peer_destroy", "hg_peer_rank",
    "hg_peer_world", "hg_peer_barrier", "hg_peer_stage_ms", "hg_peer_timeline", "hg_peer_plan_tiles", "hg_peer_plan_push", "hg_dist_sharded_dev", "hg_dist_sharded_hits", "hg_peer_hit_buffers",
]
HG_MAX_PEERS, HG_IPC_HANDLE_BYTES = 8, 64


class SketchParams(C.Structure):
    """struct hg_sketch_params (reference knobs: src/types.rs:97-113, FileSketch fields)."""
    _fields_ = [("scaled", C.c_uint64), ("seed", C.c_uint64), ("hv_d", C.c_uint32), ("ksize", C.c_uint8),
                ("canonical", C.c_uint8), ("reserved", C.c_uint8 * 2)]


HIT_DTYPE = np.dtype([("i", np.uint32), ("j", np.uint32), ("dot", np.int32), ("ani", np.float32)])
# struct hg_fasta_record
RECORD_DTYPE = np.dtype([("name_off", np.uint64), ("name_len", np.uint64), ("seq_len", np.uint64), ("file", np.uint32),
                         ("has_header", np.uint32)])


class HyperGenError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("hypergen_b200 error %d: %s" % (code, msg))
        self.code = code


_lib = None


def lib_path() -> str:
    return _build.LIB


def load() -> C.CDLL:
    """dlopen the in-tree library (building it first if the sources are newer)."""
    global _lib
    if _lib is not None:
        return _lib
    override = os.environ.get("HG_LIB")  # kernel-variant experiments only
    if override:
        L = C.CDLL(override)
    else:
        if _build.needs_build():
            _build.build()
        L = C.CDLL(lib_path())
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
    pp = C.POINTER(SketchParams)
    L.hg_init.restype = i32; L.hg_init.argtypes = [i32, C.POINTER(vp)]
    L.hg_destroy.restype = None; L.hg_destroy.argtypes = [vp]
    L.hg_sync.restype = i32; L.hg_sync.argtypes = [vp]
    L.hg_host_alloc.restype = i32; L.hg_host_alloc.argtypes = [C.c_uint64, C.POINTER(C.c_void_p)]
    L.hg_host_free.restype = i32; L.hg_host_free.argtypes = [vp]
    L.hg_host_register.restype = i32; L.hg_host_register.argtypes = [vp, C.c_uint64, C.POINTER(C.c_void_p)]
    L.hg_host_unregister.restype = i32; L.hg_host_unregister.argtypes = [vp]
    L.hg_last_error.restype = C.c_char_p; L.hg_last_error.argtypes = []
    L.hg_version.restype = C.c_char_p; L.hg_version.argtypes = []
    L.hg_stream_handle.restype = u64; L.hg_stream_handle.argtypes = [vp]
    L.hg_launch_count.restype = u64; L.hg_launch_count.argtypes = [vp]
    L.hg_set_profiling.restype = i32; L.hg_set_profiling.argtypes = [vp, i32]
    L.hg_stage_ms.restype = i32; L.hg_stage_ms.argtypes = [vp, C.POINTER(C.c_float)]
    L.hg_int_peak.restype = i32; L.hg_int_peak.argtypes = [vp, i32, C.POINTER(C.c_double)]
    L.hg_tensor_peak.restype = i32; L.hg_tensor_peak.argtypes = [vp, C.POINTER(C.c_double)]
    L.hg_dist_norm_flags.restype = i32; L.hg_dist_norm_flags.argtypes = [vp, vp, u32, u32, i32, vp]
    L.hg_encode_sets.restype = i32; L.hg_encode_sets.argtypes = [vp, vp, vp, u32, u32, vp, vp, vp, vp]
    L.hg_encode_sets_dev.restype = i32; L.hg_encode_sets_dev.argtypes = [vp, vp, vp, u32, u32, vp, vp, vp, vp]
    L.hg_fasta_merge.restype = i32; L.hg_fasta_merge.argtypes = [vp, vp, vp, u32, vp, u64, vp]
    L.hg_sketch_fasta_batch.restype = i32; L.hg_sketch_fasta_batch.argtypes = [vp, vp, vp, u32, pp, vp, vp, vp, vp, vp]
    L.hg_sketch_fasta_records.restype = i32
    L.hg_sketch_fasta_records.argtypes = [vp, vp, vp, u32, pp, u32, vp, vp, vp, vp, vp, C.POINTER(u32)]
    L.hg_fasta_records_stats.restype = i32
    L.hg_fasta_records_stats.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_float), C.POINTER(C.c_float)]
    L.hg_kmer_hash.restype = i32; L.hg_kmer_hash.argtypes = [vp, vp, vp, u32, pp, vp, u64, vp]
    L.hg_sketch_batch.restype = i32; L.hg_sketch_batch.argtypes = [vp, vp, vp, u32, pp, vp, vp, vp, vp, vp]
    L.hg_sketch_batch_dev.restype = i32; L.hg_sketch_batch_dev.argtypes = [vp, vp, vp, u32, pp, vp, vp, vp, vp, vp]
    L.hg_sketch_status.restype = i32; L.hg_sketch_status.argtypes = [vp]
    L.hg_unpack.restype = i32; L.hg_unpack.argtypes = [vp, vp, u64, vp, u32, u32, vp]
    L.hg_unpack_dev.restype = i32; L.hg_unpack_dev.argtypes = [vp, vp, u64, vp, u32, u32, vp]
    L.hg_dist.restype = i32
    L.hg_dist.argtypes = [vp, vp, vp, u32, vp, vp, u32, u32, u32, C.c_float, i32, i32, vp, u64, C.POINTER(u64)]
    L.hg_dist_dev.restype = i32
    L.hg_dist_dev.argtypes = [vp, vp, vp, u32, u32, vp, vp, u32, u32, u32, u32, C.c_float, i32, i32, vp, u64, vp]
    L.hg_dist_status.restype = i32; L.hg_dist_status.argtypes = [vp]
    L.hg_sort_hits_dev.restype = i32; L.hg_sort_hits_dev.argtypes = [vp, vp, u64, vp]
    L.hg_dist_sorted.restype = i32
    L.hg_dist_sorted.argtypes = [vp, vp, vp, u32, vp, vp, u32, u32, u32, C.c_float, i32, i32, vp, vp, u64, C.POINTER(u64)]
    L.hg_dist_packed.restype = i32
    L.hg_dist_packed.argtypes = [vp, vp, u64, vp, vp, u32, vp, u64, vp, vp, u32, u32, u32, C.c_float, i32, i32, i32, vp, vp,
                                 u64, C.POINTER(u64)]
    L.hg_search_dev.restype = i32
    L.hg_search_dev.argtypes = [vp, vp, vp, u32, vp, vp, u32, u32, u32, u32, C.c_float, i32, vp, vp, vp]
    L.hg_search_packed.restype = i32
    L.hg_search_packed.argtypes = [vp, vp, u64, vp, vp, u32, vp, u64, vp, vp, u32, u32, u32, u32, C.c_float, i32, vp, vp, vp]
    L.hg_search_stats.restype = i32; L.hg_search_stats.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_float)]
    L.hg_search_merge_dev.restype = i32; L.hg_search_merge_dev.argtypes = [vp, u32, vp, vp, vp, u32, u32, vp, vp, vp]
    L.hg_cluster_dev.restype = i32
    L.hg_cluster_dev.argtypes = [vp, vp, vp, u32, u32, u32, C.c_float, i32, vp, C.POINTER(u32)]
    L.hg_cluster_packed.restype = i32
    L.hg_cluster_packed.argtypes = [vp, vp, u64, vp, vp, u32, u32, u32, C.c_float, i32, vp, C.POINTER(u32)]
    L.hg_cluster_union_dev.restype = i32; L.hg_cluster_union_dev.argtypes = [vp, u32, vp, vp, u64, C.POINTER(u32)]
    L.hg_cluster_stats.restype = i32; L.hg_cluster_stats.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_float)]
    L.hg_derep_dev.restype = i32
    L.hg_derep_dev.argtypes = [vp, vp, vp, u32, u32, u32, C.c_float, i32, vp, vp, C.POINTER(u32)]
    L.hg_derep_packed.restype = i32
    L.hg_derep_packed.argtypes = [vp, vp, u64, vp, vp, u32, u32, u32, C.c_float, i32, vp, vp, C.POINTER(u32)]
    L.hg_derep_stats.restype = i32; L.hg_derep_stats.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_float)]
    L.hg_ani_matrix_dev.restype = i32
    L.hg_ani_matrix_dev.argtypes = [vp, vp, vp, u32, vp, vp, u32, u32, u32, i32, i32, vp, u64]
    L.hg_ani_matrix_packed.restype = i32
    L.hg_ani_matrix_packed.argtypes = [vp, vp, u64, vp, vp, u32, vp, u64, vp, vp, u32, u32, u32, i32, i32, vp, u64]
    L.hg_group_ani_matrix_packed.restype = i32
    L.hg_group_ani_matrix_packed.argtypes = [vp, vp, u64, vp, vp, u32, vp, u64, vp, vp, u32, u32, u32, i32, i32, vp, u64]
    L.hg_ani_matrix_stats.restype = i32; L.hg_ani_matrix_stats.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_float)]
    L.hg_group_create.restype = i32; L.hg_group_create.argtypes = [i32, vp, C.POINTER(vp)]
    L.hg_group_destroy.restype = None; L.hg_group_destroy.argtypes = [vp]
    L.hg_group_size.restype = i32; L.hg_group_size.argtypes = [vp]
    L.hg_group_ctx.restype = vp; L.hg_group_ctx.argtypes = [vp, i32]
    L.hg_group_sketch_fasta_batch.restype = i32; L.hg_group_sketch_fasta_batch.argtypes = [vp, vp, vp, u32, pp, vp, vp, vp, vp, vp]
    L.hg_group_sketch_fasta_records.restype = i32
    L.hg_group_sketch_fasta_records.argtypes = [vp, vp, vp, u32, pp, u32, vp, vp, vp, vp, vp, C.POINTER(u32)]
    L.hg_group_dist_packed.restype = i32
    L.hg_group_dist_packed.argtypes = [vp, vp, u64, vp, vp, u32, vp, u64, vp, vp, u32, u32, u32, C.c_float, i32, i32, vp, vp, u64,
                                       C.POINTER(u64)]
    L.hg_group_search_packed.restype = i32
    L.hg_group_search_packed.argtypes = [vp, vp, u64, vp, vp, u32, vp, u64, vp, vp, u32, u32, u32, u32, C.c_float, i32, vp, vp, vp]
    L.hg_group_cluster_packed.restype = i32
    L.hg_group_cluster_packed.argtypes = [vp, vp, u64, vp, vp, u32, u32, u32, C.c_float, i32, vp, C.POINTER(u32)]
    L.hg_peer_window_need.restype = u64; L.hg_peer_window_need.argtypes = [u32, u32, u64]
    L.hg_peer_create.restype = i32; L.hg_peer_create.argtypes = [vp, i32, i32, u64, vp, C.POINTER(vp)]
    L.hg_peer_connect.restype = i32; L.hg_peer_connect.argtypes = [vp, vp]
    L.hg_peer_create_local.restype = i32; L.hg_peer_create_local.argtypes = [vp, i32, u64, vp]
    L.hg_peer_destroy.restype = None; L.hg_peer_destroy.argtypes = [vp]
    L.hg_peer_rank.restype = i32; L.hg_peer_rank.argtypes = [vp]
    L.hg_peer_world.restype = i32; L.hg_peer_world.argtypes = [vp]
    L.hg_peer_barrier.restype = i32; L.hg_peer_barrier.argtypes = [vp]
    L.hg_peer_plan_tiles.restype = i32; L.hg_peer_plan_tiles.argtypes = [i32, i32, i32, i32, u32, u32, vp, vp, u64, C.POINTER(u64)]
    L.hg_peer_plan_push.restype = i32; L.hg_peer_plan_push.argtypes = [i32, i32, i32, i32, u32, vp, vp, vp, u64, C.POINTER(u64), C.POINTER(C.c_int)]
    L.hg_peer_stage_ms.restype = i32; L.hg_peer_stage_ms.argtypes = [vp, C.POINTER(C.c_float)]
    L.hg_peer_timeline.restype = i32; L.hg_peer_timeline.argtypes = [vp, C.POINTER(C.c_uint64)]
    L.hg_dist_sharded_dev.restype = i32
    L.hg_dist_sharded_dev.argtypes = [vp, vp, vp, u32, u32, vp, vp, vp, u32, u32, C.c_float, i32, i32, i32, u64, vp]
    L.hg_dist_sharded_hits.restype = i32; L.hg_dist_sharded_hits.argtypes = [vp, i32, vp, vp, u64, C.POINTER(u64)]
    L.hg_peer_hit_buffers.restype = i32; L.hg_peer_hit_buffers.argtypes = [vp, i32, C.POINTER(vp), C.POINTER(vp)]
    L.hg_dist_last_path.restype = i32; L.hg_dist_last_path.argtypes = [vp]
    L.hg_dist_last_reason.restype = C.c_char_p; L.hg_dist_last_reason.argtypes = [vp]
    _lib = L
    return L


def _check(rc: int) -> None:
    if rc != HG_OK:
        raise HyperGenError(rc, load().hg_last_error().decode("utf-8", "replace"))


def _ptr(a) -> int:
    """host numpy array / device pointer int / None -> void*"""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    return a.ctypes.data


def _sketch_out(n: int, hv_d: int, want_hv: bool, n_hashes: bool = True) -> dict:
    """The host arrays of n sketches, in the order the C entries take them: hv (None unless wanted), packed,
    quant_bits, norm2 and, unless n_hashes is False, n_hashes.  Pass them on as *map(_ptr, out.values())."""
    out = dict(hv=np.empty((n, hv_d), np.int16) if want_hv else None, packed=np.empty((n, 2 * hv_d), np.uint8),
               quant_bits=np.empty(n, np.uint8), norm2=np.empty(n, np.int32))
    if n_hashes:
        out["n_hashes"] = np.empty(n, np.uint32)
    return out


def make_params(k=21, scaled=1500, seed=123, canonical=True, hv_d=4096) -> SketchParams:
    return SketchParams(scaled=scaled, seed=seed, hv_d=hv_d, ksize=k, canonical=int(bool(canonical)))


def _packed_rows(ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits, qry_norm2):
    """the ref and the query rows of an hg_*_packed call as contiguous (packed, bits, norm2) arrays; when qry_packed is
    ref_packed the query side is the ref's own arrays, so that the library compares one matrix with itself"""
    r = (np.ascontiguousarray(ref_packed, np.uint8), np.ascontiguousarray(ref_bits, np.uint8), np.ascontiguousarray(ref_norm2, np.int32))
    if qry_packed is ref_packed:
        return r, r
    return r, (np.ascontiguousarray(qry_packed, np.uint8), np.ascontiguousarray(qry_bits, np.uint8),
               np.ascontiguousarray(qry_norm2, np.int32))


def _row_args(rows):
    """(packed, stride, bits, norm2, n) of one matrix, as the hg_*_packed entries take them"""
    p, b, n = rows
    return _ptr(p), p.strides[0] if p.shape[0] else 0, _ptr(b), _ptr(n), p.shape[0]


def _dist_packed(fn, h, ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits, qry_norm2, hv_d, ksize, ani_th, mode, sorted_output,
                 cap):
    """hg_dist_packed / hg_group_dist_packed (fn) on the context / group h; mode: the arguments between ani_th and
    sorted ((symmetric, path), or (symmetric,) for the group)"""
    r, q = _packed_rows(ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits, qry_norm2)
    if cap is None:
        cap = max(1024, r[0].shape[0] * q[0].shape[0] // 64)
    while True:
        hits = np.empty(cap, HIT_DTYPE)
        milli = np.empty(cap, np.uint32)
        n_hits = C.c_uint64(0)
        rc = fn(h, *_row_args(r), *_row_args(q), hv_d, ksize, ani_th, *mode, int(sorted_output), _ptr(hits), _ptr(milli), cap,
                C.byref(n_hits))
        if rc == HG_E_CAPACITY and n_hits.value > cap:
            cap = int(n_hits.value)
            continue
        _check(rc)
        # ani_milli is written by the output-stage sort only (hypergen_b200.h): unsorted calls get None
        return hits[: n_hits.value].copy(), (milli[: n_hits.value].copy() if sorted_output else None)


def _search_packed(fn, h, ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits, qry_norm2, hv_d, ksize, top_k, ani_min, path):
    """hg_search_packed / hg_group_search_packed (fn) on the context / group h"""
    r, q = _packed_rows(ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits, qry_norm2)
    Q = q[0].shape[0]
    hits = np.zeros((Q, top_k), HIT_DTYPE)
    n_found = np.zeros(Q, np.uint32)
    milli = np.zeros((Q, top_k), np.uint32)
    _check(fn(h, *_row_args(r), *_row_args(q), hv_d, ksize, top_k, ani_min, path, _ptr(hits), _ptr(n_found), _ptr(milli)))
    return hits, n_found, milli


def _search_stats(ctx_handle):
    counts, ms = (C.c_uint64 * 4)(), (C.c_float * 4)()
    _check(load().hg_search_stats(ctx_handle, counts, ms))
    return [int(x) for x in counts], [float(x) for x in ms]


def _cluster_packed(fn, h, packed, bits, norm2, hv_d, ksize, ani_th, path):
    """hg_cluster_packed / hg_group_cluster_packed (fn) on the context / group h"""
    p, b, nm = _packed_rows(packed, bits, norm2, packed, bits, norm2)[0]
    rep = np.zeros(p.shape[0], np.uint32)
    n_clusters = C.c_uint32(0)
    _check(fn(h, *_row_args((p, b, nm)), hv_d, ksize, ani_th, path, _ptr(rep), C.byref(n_clusters)))
    return rep, int(n_clusters.value)


def _cluster_stats(ctx_handle):
    counts, ms = (C.c_uint64 * 4)(), (C.c_float * 4)()
    _check(load().hg_cluster_stats(ctx_handle, counts, ms))
    return [int(x) for x in counts], [float(x) for x in ms]


def _sketch_records(fn, h, files, params):
    """hg_sketch_fasta_records / hg_group_sketch_fasta_records (fn) on the context / group h: raw FASTA file contents in,
    dict(packed, quant_bits, norm2, n_hashes, records) out, one row per record.  rec_cap is the '>' bytes of all files
    plus one per file, which no call can exceed."""
    raw, off = Context._concat_files(files)
    n = len(files)
    cap = sum(bytes(f).count(b">") for f in files) + n
    out = _sketch_out(cap, int(params.hv_d), False)
    del out["hv"]
    records = np.empty(cap, RECORD_DTYPE)
    n_rec = C.c_uint32(0)
    _check(fn(h, _ptr(raw) if raw.size else None, _ptr(off), n, C.byref(params), cap, _ptr(records), *map(_ptr, out.values()),
              C.byref(n_rec)))
    out = {k: v[: n_rec.value] for k, v in out.items()}
    out["records"] = records[: n_rec.value]
    return out


def pinned_empty(shape, dtype) -> np.ndarray:
    """an uninitialised numpy array in page-locked host memory (hg_host_alloc), freed (hg_host_free) with its last view:
    the GPU copies into it at link rate, where a pageable array has to be page-locked for every call"""
    dtype = np.dtype(dtype)
    count = int(np.prod(shape))
    nbytes = max(1, count * dtype.itemsize)
    p = C.c_void_p()
    _check(load().hg_host_alloc(nbytes, C.byref(p)))
    raw = (C.c_uint8 * nbytes).from_address(p.value)
    weakref.finalize(raw, load().hg_host_free, p.value).atexit = False  # the numpy array below keeps `raw` alive
    return np.frombuffer(raw, np.uint8, count * dtype.itemsize).view(dtype).reshape(shape)


def _ani_matrix_packed(fn, h, ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits, qry_norm2, hv_d, ksize, path, lower, out):
    """hg_ani_matrix_packed / hg_group_ani_matrix_packed (fn) on the context / group h.  lower: the strict lower triangle
    of the ref rows (the query must be the same arrays; n (n - 1) / 2 float32), else the n_ref x n_qry rectangle.  out: None, or a float32
    array to write into (lower: 1-D, at least n (n - 1) / 2 entries; rectangle: 1-D with rows n_qry apart, or 2-D with
    n_ref rows of at least n_qry contiguous entries, rows its ld apart).  None: a new page-locked array (pinned_empty)."""
    r, q = _packed_rows(ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits, qry_norm2)
    n_ref, n_qry = r[0].shape[0], q[0].shape[0]
    if out is None:
        out = pinned_empty(n_ref * (n_ref - 1) // 2 if lower else (n_ref, n_qry), np.float32)
    if out.dtype != np.float32 or not (out.flags.c_contiguous or (out.ndim == 2 and out.strides[1] == 4)):
        raise ValueError("out must be float32 with contiguous rows")
    if lower:
        if out.ndim != 1 or out.size < n_ref * (n_ref - 1) // 2:
            raise ValueError("out must be 1-D with at least %d entries" % (n_ref * (n_ref - 1) // 2))
        ld = 0
    elif out.ndim == 2:
        ld = out.strides[0] // 4
        if out.shape[0] < n_ref or out.shape[1] < n_qry or out.strides[0] % 4 or out.strides[0] < 0:
            raise ValueError("out must have at least %d rows of %d entries" % (n_ref, n_qry))
    else:
        ld = n_qry
        if out.ndim != 1 or out.size < n_ref * n_qry:
            raise ValueError("out must be 1-D with at least %d entries, or 2-D" % (n_ref * n_qry))
    _check(fn(h, *_row_args(r), *_row_args(q), hv_d, ksize, path, int(lower), _ptr(out), ld))
    return out


def _ani_matrix_stats(ctx_handle):
    counts, ms = (C.c_uint64 * 4)(), (C.c_float * 4)()
    _check(load().hg_ani_matrix_stats(ctx_handle, counts, ms))
    return [int(x) for x in counts], [float(x) for x in ms]


def _order(order, n):
    """a priority order as the hg_derep_* entries take it: None, or n uint32 entries (kept alive by the caller)"""
    if order is None:
        return None
    order = np.ascontiguousarray(order, np.uint32)
    if order.shape != (n,):
        raise ValueError("order must have one entry per sketch (%d), got shape %s" % (n, order.shape))
    return order


class Context:
    """hg_ctx: one CUDA device + stream (replaces CudaDevice::new(0), sketch_cuda.rs:52)."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        _check(load().hg_init(device, C.byref(self._h)))
        self.device = device

    def close(self):
        if self._h:
            load().hg_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- plumbing --
    def sync(self):
        _check(load().hg_sync(self._h))

    @property
    def stream(self) -> int:
        return int(load().hg_stream_handle(self._h))

    @property
    def launches(self) -> int:
        return int(load().hg_launch_count(self._h))

    def set_profiling(self, enabled: bool):
        _check(load().hg_set_profiling(self._h, int(enabled)))

    def stage_ms(self):
        """device ms of the last call's stages: [staging, kmer_hash, encode, dist] (-1 = not run)"""
        out = (C.c_float * 4)()
        _check(load().hg_stage_ms(self._h, out))
        return [float(x) for x in out]

    def int_peak(self, which: int = 2) -> float:
        v = C.c_double(0)
        _check(load().hg_int_peak(self._h, which, C.byref(v)))
        return v.value

    def tensor_peak(self) -> float:
        v = C.c_double(0)
        _check(load().hg_tensor_peak(self._h, C.byref(v)))
        return v.value

    def dist_norm_flags(self, d_hv, n_rows, hv_d, path, d_flags):
        """hg_dist_norm_flags (device pointers as ints): per row 1 if tensor kernel `path` takes it as a row whose true
        norm reaches ceil(2^31 / 3)"""
        _check(load().hg_dist_norm_flags(self._h, d_hv, n_rows, hv_d, path, d_flags))

    # -- stage 1 --
    def kmer_hash(self, seq: np.ndarray, seg_off: np.ndarray, params: SketchParams):
        """hg_kmer_hash: per-genome sorted unique sampled hashes -> (hashes, hash_off)."""
        seq = np.ascontiguousarray(seq, np.uint8)
        off = np.ascontiguousarray(seg_off, np.uint64)
        n = off.size - 1
        hash_off = np.zeros(n + 1, np.uint64)
        total_len = int(off[-1] - off[0]) if n else 0
        cap = total_len // max(int(params.scaled), 1) * 2 + 4096 * max(n, 1)
        hashes = np.empty(cap, np.uint64)
        rc = load().hg_kmer_hash(self._h, _ptr(seq) if seq.size else None, _ptr(off), n, C.byref(params),
                                 _ptr(hashes), cap, _ptr(hash_off))
        if rc == HG_E_CAPACITY and int(hash_off[-1]) > cap:
            cap = int(hash_off[-1])
            hashes = np.empty(cap, np.uint64)
            rc = load().hg_kmer_hash(self._h, _ptr(seq), _ptr(off), n, C.byref(params), _ptr(hashes), cap,
                                     _ptr(hash_off))
        _check(rc)
        return hashes[: int(hash_off[-1])].copy(), hash_off

    def sketch_batch(self, seq: np.ndarray, seg_off: np.ndarray, params: SketchParams, want_hv: bool = True):
        """hg_sketch_batch with host buffers -> dict(hv, packed, quant_bits, norm2, n_hashes)."""
        seq = np.ascontiguousarray(seq, np.uint8)
        off = np.ascontiguousarray(seg_off, np.uint64)
        n = off.size - 1
        out = _sketch_out(n, int(params.hv_d), want_hv)
        _check(load().hg_sketch_batch(self._h, _ptr(seq) if seq.size else None, _ptr(off), n, C.byref(params),
                                      *map(_ptr, out.values())))
        return out

    def sketch_batch_dev(self, d_seq: int, seg_off: np.ndarray, params: SketchParams, d_hv, d_packed,
                         d_quant_bits: int, d_norm2: int, d_n_hashes: int):
        """hg_sketch_batch_dev: device pointers (ints), asynchronous on self.stream."""
        off = np.ascontiguousarray(seg_off, np.uint64)
        _check(load().hg_sketch_batch_dev(self._h, d_seq, _ptr(off), off.size - 1, C.byref(params), d_hv, d_packed,
                                          d_quant_bits, d_norm2, d_n_hashes))

    def encode_sets(self, sets, hv_d: int = 4096, want_hv: bool = True):
        """hg_encode_sets: list of unique-u64 arrays -> dict(hv, packed, quant_bits, norm2)."""
        n = len(sets)
        off = np.zeros(n + 1, np.uint64)
        off[1:] = np.cumsum([len(x) for x in sets])
        hashes = np.ascontiguousarray(np.concatenate(sets) if n and int(off[-1]) else np.zeros(0), np.uint64)
        out = _sketch_out(n, hv_d, want_hv, n_hashes=False)
        _check(load().hg_encode_sets(self._h, _ptr(hashes) if hashes.size else None, _ptr(off), n, hv_d,
                                     *map(_ptr, out.values())))
        return out

    def encode_sets_dev(self, d_hashes: int, hash_off: np.ndarray, hv_d: int, d_hv, d_packed, d_quant_bits, d_norm2):
        off = np.ascontiguousarray(hash_off, np.uint64)
        _check(load().hg_encode_sets_dev(self._h, d_hashes, _ptr(off), off.size - 1, hv_d, d_hv, d_packed,
                                         d_quant_bits, d_norm2))

    # -- raw FASTA in --
    @staticmethod
    def _concat_files(files):
        off = np.zeros(len(files) + 1, np.uint64)
        off[1:] = np.cumsum([len(f) for f in files])
        raw = np.frombuffer(b"".join(bytes(f) for f in files), dtype=np.uint8) if int(off[-1]) else np.zeros(0, np.uint8)
        return np.ascontiguousarray(raw), off

    def fasta_merge(self, files):
        """hg_fasta_merge: list of raw FASTA file contents (bytes) -> list of merged sequences (uint8 arrays)."""
        raw, off = self._concat_files(files)
        n = len(files)
        merged = np.empty(max(int(off[-1]), 1), np.uint8)
        moff = np.zeros(n + 1, np.uint64)
        _check(load().hg_fasta_merge(self._h, _ptr(raw) if raw.size else None, _ptr(off), n, _ptr(merged), merged.size,
                                     _ptr(moff)))
        return [merged[int(moff[f]):int(moff[f + 1])].copy() for f in range(n)]

    def sketch_fasta_batch(self, files, params: SketchParams, want_hv: bool = True):
        """hg_sketch_fasta_batch: raw FASTA file contents in, sketches out (as sketch_batch)."""
        raw, off = self._concat_files(files)
        n = len(files)
        out = _sketch_out(n, int(params.hv_d), want_hv)
        _check(load().hg_sketch_fasta_batch(self._h, _ptr(raw) if raw.size else None, _ptr(off), n, C.byref(params),
                                            *map(_ptr, out.values())))
        return out

    def sketch_fasta_records(self, files, params: SketchParams):
        """hg_sketch_fasta_records: raw FASTA file contents in, one sketch per record out ->
        dict(packed, quant_bits, norm2, n_hashes, records) with records a RECORD_DTYPE array."""
        return _sketch_records(load().hg_sketch_fasta_records, self._h, files, params)

    def fasta_records_stats(self):
        """hg_fasta_records_stats of the last records call -> ([chunks, records, table slots, 0],
        [ms of merge, record index, k-mer hash, encode], host gap ms) (ms -1: profiling off)"""
        counts, ms, gap = (C.c_uint64 * 4)(), (C.c_float * 4)(), C.c_float(0)
        _check(load().hg_fasta_records_stats(self._h, counts, ms, C.byref(gap)))
        return [int(x) for x in counts], [float(x) for x in ms], float(gap.value)

    def sketch_status(self):
        _check(load().hg_sketch_status(self._h))

    # -- format --
    def unpack(self, packed: np.ndarray, quant_bits: np.ndarray, hv_d: int) -> np.ndarray:
        packed = np.ascontiguousarray(packed, np.uint8)
        qb = np.ascontiguousarray(quant_bits, np.uint8)
        n = qb.size
        hv = np.empty((n, hv_d), np.int16)
        _check(load().hg_unpack(self._h, _ptr(packed), packed.shape[1], _ptr(qb), n, hv_d, _ptr(hv)))
        return hv

    def unpack_dev(self, d_packed: int, row_stride: int, d_quant_bits: int, n: int, hv_d: int, d_hv: int):
        _check(load().hg_unpack_dev(self._h, d_packed, row_stride, d_quant_bits, n, hv_d, d_hv))

    # -- stage 2 --
    def dist(self, ref_hv, ref_norm2, qry_hv, qry_norm2, ksize=21, ani_th=85.0, symmetric=False, path=0,
             cap=None, sorted_output=False, want_milli=False):
        """hg_dist with host buffers -> structured array of hits (i, j, dot, ani), unspecified order.
        sorted_output: hg_dist_sorted instead - the hits in the reference's output order (sorted on the
        GPU); with want_milli also the ANI in thousandths as `{:.3}` rounds it -> (hits, milli)."""
        r = np.ascontiguousarray(ref_hv, np.int16)
        rn = np.ascontiguousarray(ref_norm2, np.int32)
        same = qry_hv is ref_hv
        q = r if same else np.ascontiguousarray(qry_hv, np.int16)
        qn = rn if same and qry_norm2 is ref_norm2 else np.ascontiguousarray(qry_norm2, np.int32)
        R, D = r.shape
        Q = q.shape[0]
        if cap is None:
            cap = max(1024, R * Q // 64)
        while True:
            hits = np.empty(cap, HIT_DTYPE)
            n_hits = C.c_uint64(0)
            milli = np.empty(cap, np.uint32) if (sorted_output and want_milli) else None
            if sorted_output:
                rc = load().hg_dist_sorted(self._h, _ptr(r), _ptr(rn), R, _ptr(q), _ptr(qn), Q, D, ksize, ani_th,
                                           int(symmetric), path, _ptr(hits), _ptr(milli), cap, C.byref(n_hits))
            else:
                rc = load().hg_dist(self._h, _ptr(r), _ptr(rn), R, _ptr(q), _ptr(qn), Q, D, ksize, ani_th,
                                    int(symmetric), path, _ptr(hits), cap, C.byref(n_hits))
            if rc == HG_E_CAPACITY and n_hits.value > cap:
                cap = int(n_hits.value)
                continue
            _check(rc)
            if milli is not None:
                return hits[: n_hits.value].copy(), milli[: n_hits.value].copy()
            return hits[: n_hits.value].copy()

    def dist_dev(self, d_ref, d_ref_norm2, n_ref, i0, d_qry, d_qry_norm2, n_qry, j0, hv_d, ksize, ani_th,
                 symmetric, path, d_hits, cap, d_n_hits):
        _check(load().hg_dist_dev(self._h, d_ref, d_ref_norm2, n_ref, i0, d_qry, d_qry_norm2, n_qry, j0, hv_d, ksize,
                                  ani_th, int(symmetric), path, d_hits, cap, d_n_hits))

    def dist_status(self):
        """hg_dist_status: the verdict a dist_dev(path=3) did not wait for"""
        _check(load().hg_dist_status(self._h))

    def dist_packed(self, ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits, qry_norm2, hv_d, ksize=21, ani_th=85.0,
                    symmetric=False, path=0, sorted_output=True, cap=None):
        """hg_dist_packed: packed sketch rows (n x stride uint8) + quant bits + norms -> (hits, ani_milli)."""
        return _dist_packed(load().hg_dist_packed, self._h, ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits, qry_norm2, hv_d,
                            ksize, ani_th, (int(symmetric), path), sorted_output, cap)

    def search_dev(self, d_ref, d_ref_norm2, n_ref, d_qry, d_qry_norm2, n_qry, hv_d, ksize, top_k, ani_min, path, d_out,
                   d_n_found, d_ani_milli=None):
        """hg_search_dev: device pointers (ints); returns when the result is complete."""
        _check(load().hg_search_dev(self._h, d_ref, d_ref_norm2, n_ref, d_qry, d_qry_norm2, n_qry, hv_d, ksize, top_k, ani_min,
                                    path, d_out, d_n_found, d_ani_milli))

    def search_packed(self, ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits, qry_norm2, hv_d, ksize=21, top_k=10,
                      ani_min=0.0, path=0):
        """hg_search_packed: packed sketch rows (n x stride uint8) + quant bits + norms ->
        (hits[n_qry, top_k], n_found[n_qry], ani_milli[n_qry, top_k]); query j's results are hits[j, :n_found[j]]."""
        return _search_packed(load().hg_search_packed, self._h, ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits, qry_norm2,
                              hv_d, ksize, top_k, ani_min, path)

    def search_stats(self):
        """hg_search_stats of the last search -> ([s, floor-pass candidates, main-pass candidates, reruns],
        [ms of floor pass, its select, main pass, its select] (-1: not run or profiling off))"""
        return _search_stats(self._h)

    def search_merge_dev(self, n_lists, d_in, d_in_found, i0, n_qry, top_k, d_out, d_n_found, d_ani_milli=None):
        """hg_search_merge_dev: n_lists per-block results (device pointers as ints; list m's refs start at global index
        i0[m]) -> the result over all blocks; returns when it is complete."""
        off = np.ascontiguousarray(i0, np.uint32)
        assert off.size == n_lists
        _check(load().hg_search_merge_dev(self._h, n_lists, d_in, d_in_found, _ptr(off), n_qry, top_k, d_out, d_n_found,
                                          d_ani_milli))

    def cluster_dev(self, d_hv, d_norm2, n, hv_d, ksize, ani_th, path, d_rep) -> int:
        """hg_cluster_dev: device pointers (ints); d_rep receives rep[i] = the smallest index of i's cluster.
        Returns the number of clusters once the result is complete."""
        n_clusters = C.c_uint32(0)
        _check(load().hg_cluster_dev(self._h, d_hv, d_norm2, n, hv_d, ksize, ani_th, path, d_rep, C.byref(n_clusters)))
        return int(n_clusters.value)

    def cluster_packed(self, packed, bits, norm2, hv_d, ksize=21, ani_th=95.0, path=0):
        """hg_cluster_packed: packed sketch rows (n x stride uint8) + quant bits + norms -> (rep[n], n_clusters)"""
        return _cluster_packed(load().hg_cluster_packed, self._h, packed, bits, norm2, hv_d, ksize, ani_th, path)

    def cluster_union_dev(self, n, d_rep, d_edges, n_edges) -> int:
        """hg_cluster_union_dev: unite n_edges hg_hit records (device) into the forest d_rep[n] (device) and flatten it;
        returns the number of clusters"""
        n_clusters = C.c_uint32(0)
        _check(load().hg_cluster_union_dev(self._h, n, d_rep, d_edges, n_edges, C.byref(n_clusters)))
        return int(n_clusters.value)

    def cluster_stats(self):
        """hg_cluster_stats of the last cluster run -> ([windows, linked pairs, largest window's pairs, edge capacity],
        [ms of preparing the rows, dist windows, hooks, flatten + count] (-1: not run or profiling off))"""
        return _cluster_stats(self._h)

    def derep_dev(self, d_hv, d_norm2, n, hv_d, ksize, ani_th, path, d_rep, order=None) -> int:
        """hg_derep_dev: device pointers (ints); d_rep receives rep[i] = the index of i's representative; order (host
        array of n entries, or None for file order) is the priority.  Returns the number of representatives once the
        result is complete."""
        o = _order(order, n)
        n_reps = C.c_uint32(0)
        _check(load().hg_derep_dev(self._h, d_hv, d_norm2, n, hv_d, ksize, ani_th, path, _ptr(o), d_rep,
                                   C.byref(n_reps)))
        return int(n_reps.value)

    def derep_packed(self, packed, bits, norm2, hv_d, ksize=21, ani_th=95.0, path=0, order=None):
        """hg_derep_packed: packed sketch rows (n x stride uint8) + quant bits + norms -> (rep[n], n_reps)"""
        p, b, nm = _packed_rows(packed, bits, norm2, packed, bits, norm2)[0]
        o = _order(order, p.shape[0])
        rep = np.zeros(p.shape[0], np.uint32)
        n_reps = C.c_uint32(0)
        _check(load().hg_derep_packed(self._h, *_row_args((p, b, nm)), hv_d, ksize, ani_th, path, _ptr(o),
                                      _ptr(rep), C.byref(n_reps)))
        return rep, int(n_reps.value)

    def ani_matrix_dev(self, d_ref, d_ref_norm2, n_ref, d_qry, d_qry_norm2, n_qry, hv_d, ksize, path, lower, d_out, ld=0):
        """hg_ani_matrix_dev: device pointers (ints); d_out (float32) receives the strict lower triangle (lower) or the
        n_ref x n_qry rectangle with rows ld apart.  Returns when the result is complete."""
        _check(load().hg_ani_matrix_dev(self._h, d_ref, d_ref_norm2, n_ref, d_qry, d_qry_norm2, n_qry, hv_d, ksize, path, int(lower),
                                        d_out, ld))

    def ani_matrix_packed(self, ref_packed, ref_bits, ref_norm2, qry_packed=None, qry_bits=None, qry_norm2=None, hv_d=4096, ksize=21,
                          path=0, lower=True, out=None):
        """hg_ani_matrix_packed: packed sketch rows -> float32 ANI of every pair: the strict lower triangle of the ref rows
        (lower, n (n - 1) / 2 entries in PHYLIP order) or the ref x query rectangle (a square when qry_packed is None)."""
        if qry_packed is None:
            qry_packed, qry_bits, qry_norm2 = ref_packed, ref_bits, ref_norm2
        return _ani_matrix_packed(load().hg_ani_matrix_packed, self._h, ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits, qry_norm2,
                                  hv_d, ksize, path, lower, out)

    def ani_matrix_stats(self):
        """hg_ani_matrix_stats of the last matrix run -> ([bands, entries, bytes copied to the host, path], [ms of row
        preparation, band kernels, conversion, copies to the host])"""
        return _ani_matrix_stats(self._h)

    def derep_stats(self):
        """hg_derep_stats of the last derep run -> ([column chunks, windows, linked pairs, representatives], [ms of
        preparing the rows, dist windows, mark hooks + greedy steps, assignment] (-1: not run or profiling off))"""
        counts, ms = (C.c_uint64 * 4)(), (C.c_float * 4)()
        _check(load().hg_derep_stats(self._h, counts, ms))
        return [int(x) for x in counts], [float(x) for x in ms]

    def sort_hits_dev(self, d_hits, n, d_ani_milli=None):
        """hg_sort_hits_dev: device records to the reference's output order, in place."""
        _check(load().hg_sort_hits_dev(self._h, d_hits, n, d_ani_milli))

    @property
    def dist_last_path(self) -> int:
        return int(load().hg_dist_last_path(self._h))

    @property
    def dist_last_reason(self) -> str:
        return load().hg_dist_last_reason(self._h).decode()


class Peer:
    """hg_peer: this process's GPU as one member of a group of GPUs on the box (one process per GPU).

    `exchange(handle: bytes) -> list[bytes]` is the host's own all-gather of the 64-byte window handles
    (multigpu.PeerGroup passes one built on torch.distributed); world == 1 needs none."""

    def __init__(self, ctx: Context, rank: int, world: int, window_bytes: int, exchange=None):
        self.ctx, self.rank, self.world = ctx, rank, world
        self._h = C.c_void_p()
        handle = (C.c_uint8 * HG_IPC_HANDLE_BYTES)()
        _check(load().hg_peer_create(ctx._h, rank, world, window_bytes, handle, C.byref(self._h)))
        if world > 1:
            allh = exchange(bytes(handle))
            buf = (C.c_uint8 * (HG_IPC_HANDLE_BYTES * world)).from_buffer_copy(b"".join(allh))
            _check(load().hg_peer_connect(self._h, buf))

    def close(self):
        if self._h:
            load().hg_peer_destroy(self._h)
            self._h = C.c_void_p()

    def barrier(self):
        _check(load().hg_peer_barrier(self._h))

    def dist_sharded_dev(self, d_ref, d_ref_norm2, n_ref_local, ref_row0, d_qry, d_qry_norm2, qry_bounds, hv_d, ksize, ani_th,
                         symmetric, path, root, cap, mapped_hits=None):
        """hg_dist_sharded_dev (collective; device pointers as ints; qry_bounds: world + 1 row offsets)."""
        qb = np.ascontiguousarray(qry_bounds, np.uint32)
        assert qb.size == self.world + 1
        _check(load().hg_dist_sharded_dev(self._h, d_ref, d_ref_norm2, n_ref_local, ref_row0, d_qry, d_qry_norm2, _ptr(qb), hv_d,
                                          ksize, ani_th, int(symmetric), path, root, cap, mapped_hits))

    def dist_sharded_hits(self, cap: int, sorted_output: bool = False, hits=None, milli=None):
        """hg_dist_sharded_hits -> (hits, milli or None) on the root, (empty, None) elsewhere.  `hits` / `milli`
        may be preallocated (pinned) numpy arrays of at least `cap` records."""
        own = hits is None
        if own:
            hits = np.empty(cap, HIT_DTYPE)
        if sorted_output and milli is None:
            milli = np.empty(cap, np.uint32)
        n = C.c_uint64(0)
        _check(load().hg_dist_sharded_hits(self._h, int(sorted_output), _ptr(hits), _ptr(milli) if sorted_output else None, cap,
                                           C.byref(n)))
        h = hits[: n.value]
        return (h.copy() if own else h), (milli[: n.value] if sorted_output else None)

    def stage_ms(self):
        """device ms of the last sharded dist: [operands, chunked push, kernel incl. waits for the peers' chunks, final barrier]"""
        out = (C.c_float * 4)()
        _check(load().hg_peer_stage_ms(self._h, out))
        return [float(x) for x in out]

    def timeline(self):
        """globaltimer stamps (ns) of the last sharded dist (HG_PEER_TIMELINE=1); see hg_peer_timeline"""
        out = (C.c_uint64 * 32)()
        _check(load().hg_peer_timeline(self._h, out))
        return [int(x) for x in out]

    def hit_buffers(self, root: int = 0):
        dh, dc = C.c_void_p(), C.c_void_p()
        _check(load().hg_peer_hit_buffers(self._h, root, C.byref(dh), C.byref(dc)))
        return dh.value, dc.value


def host_register(arr: np.ndarray) -> int:
    """hg_host_register on a numpy array's memory -> the device pointer kernels of this process use for it"""
    dev = C.c_void_p()
    _check(load().hg_host_register(arr.ctypes.data, arr.nbytes, C.byref(dev)))
    return dev.value


def host_unregister(arr: np.ndarray) -> None:
    _check(load().hg_host_unregister(arr.ctypes.data))


def peer_plan_tiles(world: int, rank: int, symmetric: bool, path: int, n_ref_local: int, qry_bounds, hv_d: int = 4096):
    """hg_peer_plan_tiles -> (tile_row, tile_col, need_mask) arrays in walk order (host logic, no GPU)"""
    qb = np.ascontiguousarray(qry_bounds, np.uint32)
    n = C.c_uint64(0)
    load().hg_peer_plan_tiles(world, rank, int(symmetric), path, hv_d, n_ref_local, _ptr(qb), None, 0, C.byref(n))
    out = np.zeros((max(int(n.value), 1), 2), np.uint32)
    _check(load().hg_peer_plan_tiles(world, rank, int(symmetric), path, hv_d, n_ref_local, _ptr(qb), _ptr(out), out.shape[0], C.byref(n)))
    out = out[: n.value]
    return out[:, 0] & 0xFFFF, out[:, 0] >> 16, out[:, 1]


def peer_plan_push(world: int, rank: int, symmetric: bool, path: int, qry_bounds, hv_d: int = 4096):
    """hg_peer_plan_push -> (chunk row boundaries [5], [(set, destination mask)] in sending order, ring?)"""
    qb = np.ascontiguousarray(qry_bounds, np.uint32)
    rows = np.zeros(5, np.uint32)
    units = np.zeros((40, 2), np.uint32)
    n, ring = C.c_uint64(0), C.c_int(0)
    _check(load().hg_peer_plan_push(world, rank, int(symmetric), path, hv_d, _ptr(qb), _ptr(rows), _ptr(units), units.shape[0],
                                    C.byref(n), C.byref(ring)))
    return rows.tolist(), [(int(a), int(b)) for a, b in units[: n.value]], bool(ring.value)


def peer_window_need(gathered_rows: int, hv_d: int, hit_cap: int) -> int:
    return int(load().hg_peer_window_need(gathered_rows, hv_d, hit_cap))


class Group:
    """hg_group: one process driving several GPUs of the box (what the `hyper-gen` CLI uses)."""

    def __init__(self, n_devices: int = 0, ordinals=None):
        self._h = C.c_void_p()
        arr = None
        if ordinals is not None:
            arr = (C.c_int * len(ordinals))(*ordinals)
            n_devices = len(ordinals)
        _check(load().hg_group_create(n_devices, arr, C.byref(self._h)))

    def close(self):
        if self._h:
            load().hg_group_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def size(self) -> int:
        return int(load().hg_group_size(self._h))

    def dist_last_path(self, i: int = 0) -> int:
        return int(load().hg_dist_last_path(load().hg_group_ctx(self._h, i)))

    def sketch_fasta_batch(self, files, params: SketchParams, want_hv: bool = True):
        raw, off = Context._concat_files(files)
        n = len(files)
        out = _sketch_out(n, int(params.hv_d), want_hv)
        _check(load().hg_group_sketch_fasta_batch(self._h, _ptr(raw) if raw.size else None, _ptr(off), n, C.byref(params),
                                                  *map(_ptr, out.values())))
        return out

    def sketch_fasta_records(self, files, params: SketchParams):
        """hg_group_sketch_fasta_records: Context.sketch_fasta_records over the GPUs of the group; same bytes."""
        return _sketch_records(load().hg_group_sketch_fasta_records, self._h, files, params)

    def dist_packed(self, ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits, qry_norm2, hv_d, ksize=21, ani_th=85.0,
                    symmetric=False, sorted_output=True, cap=None):
        """hg_group_dist_packed: Context.dist_packed over the GPUs of the group (the group entry takes no path)."""
        return _dist_packed(load().hg_group_dist_packed, self._h, ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits, qry_norm2,
                            hv_d, ksize, ani_th, (int(symmetric),), sorted_output, cap)

    def search_packed(self, ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits, qry_norm2, hv_d, ksize=21, top_k=10,
                      ani_min=0.0, path=0):
        """hg_group_search_packed: Context.search_packed with the refs split into one block per GPU; same results."""
        return _search_packed(load().hg_group_search_packed, self._h, ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits,
                              qry_norm2, hv_d, ksize, top_k, ani_min, path)

    def search_stats(self, i: int = 0):
        """Context.search_stats of member i's part of the last group search"""
        return _search_stats(load().hg_group_ctx(self._h, i))

    def cluster_packed(self, packed, bits, norm2, hv_d, ksize=21, ani_th=95.0, path=0):
        """hg_group_cluster_packed: Context.cluster_packed over the GPUs of the group; same result."""
        return _cluster_packed(load().hg_group_cluster_packed, self._h, packed, bits, norm2, hv_d, ksize, ani_th, path)

    def cluster_stats(self, i: int = 0):
        """Context.cluster_stats of member i's part of the last group cluster run"""
        return _cluster_stats(load().hg_group_ctx(self._h, i))

    def ani_matrix_packed(self, ref_packed, ref_bits, ref_norm2, qry_packed=None, qry_bits=None, qry_norm2=None, hv_d=4096, ksize=21,
                          path=0, lower=True, out=None):
        """hg_group_ani_matrix_packed: Context.ani_matrix_packed with the ref rows split over the GPUs; same bytes."""
        if qry_packed is None:
            qry_packed, qry_bits, qry_norm2 = ref_packed, ref_bits, ref_norm2
        return _ani_matrix_packed(load().hg_group_ani_matrix_packed, self._h, ref_packed, ref_bits, ref_norm2, qry_packed, qry_bits,
                                  qry_norm2, hv_d, ksize, path, lower, out)

    def ani_matrix_stats(self, i: int = 0):
        """Context.ani_matrix_stats of member i's part of the last group matrix run"""
        return _ani_matrix_stats(load().hg_group_ctx(self._h, i))
