"""The packed-row entries (hg_dist_packed, hg_search_packed and their hg_group_* forms) check the rows they are given in
one way: every bad row or argument on either side is HG_E_INVALID, and the message names the entry that was called.
They go through the C ABI directly, so that any stride can be passed.  Also: the sharded dist's sorted output stage
returns what the single-GPU one does."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HV_D, BITS, N_REF, N_QRY, TOP_K = 256, 8, 2048, 64, 10
CAP = N_REF * N_QRY  # random rows: any number of pairs may pass the threshold
ALLOC = 1024  # bytes per row the buffers hold: every stride below stays inside them


def _rows(n, seed):
    rng = np.random.default_rng(seed)
    packed = rng.integers(0, 256, n * ALLOC, dtype=np.uint8)
    bits = np.full(n, BITS, np.uint8)
    norm = rng.integers(1, 1 << 20, n, dtype=np.int32)
    return packed, bits, norm


@pytest.fixture(scope="module")
def groups(hg):
    one, two = hg.Group(ordinals=[0]), hg.Group(ordinals=[0, 0])  # two members on GPU 0: the group search splits the refs
    yield one, two
    two.close()
    one.close()


def _call(hg, ctx, groups, entry, ref, ref_stride, qry, qry_stride, hv_d):
    lib = hg.ffi.load()
    rows = []
    for (packed, bits, norm), stride in ((ref, ref_stride), (qry, qry_stride)):
        rows += [packed.ctypes.data, stride, bits.ctypes.data, norm.ctypes.data, bits.size]
    hits = np.zeros(max(CAP, N_QRY * TOP_K), hg.ffi.HIT_DTYPE)
    milli = np.zeros(hits.size, np.uint32)
    n_found = np.zeros(N_QRY, np.uint32)
    n_hits = C.c_uint64(0)
    if entry == "hg_dist_packed":
        rc = lib.hg_dist_packed(ctx._h, *rows, hv_d, 21, 85.0, 0, 0, 1, hits.ctypes.data, milli.ctypes.data, CAP, C.byref(n_hits))
    elif entry == "hg_group_dist_packed":
        rc = lib.hg_group_dist_packed(groups[0]._h, *rows, hv_d, 21, 85.0, 0, 1, hits.ctypes.data, milli.ctypes.data, CAP,
                                      C.byref(n_hits))
    else:
        h = ctx._h if entry == "hg_search_packed" else groups[1]._h
        rc = getattr(lib, entry)(h, *rows, hv_d, 21, TOP_K, 0.0, 0, hits.ctypes.data, n_found.ctypes.data, milli.ctypes.data)
    return rc, lib.hg_last_error().decode()


BAD = ["ok", "bits_0", "bits_17", "stride_not_4", "stride_below_width"]


@pytest.mark.parametrize("entry", ["hg_dist_packed", "hg_search_packed", "hg_group_dist_packed", "hg_group_search_packed"])
@pytest.mark.parametrize("side", ["ref", "query"])
@pytest.mark.parametrize("bad", BAD)
def test_packed_entries_reject_bad_rows(hg, ctx, groups, entry, side, bad):
    ref, qry = _rows(N_REF, 1), _rows(N_QRY, 2)
    strides = {"ref": ALLOC, "query": ALLOC}
    bits = (ref if side == "ref" else qry)[1]
    if bad in ("bits_0", "bits_17"):
        bits[3] = 0 if bad == "bits_0" else 17
    elif bad == "stride_not_4":
        strides[side] = BITS * HV_D // 8 + 2
    elif bad == "stride_below_width":
        strides[side] = BITS * HV_D // 8 - 4
    rc, msg = _call(hg, ctx, groups, entry, ref, strides["ref"], qry, strides["query"], HV_D)
    if bad == "ok":
        assert rc == hg.ffi.HG_OK, msg
        return
    assert rc == hg.ffi.HG_E_INVALID
    assert msg.startswith(entry + ":"), msg
    if bad.startswith("bits"):
        assert "%s sketch 3 has hv_quant_bits %d" % (side, bits[3]) in msg, msg


@pytest.mark.parametrize("entry", ["hg_dist_packed", "hg_search_packed", "hg_group_dist_packed", "hg_group_search_packed"])
def test_packed_entries_reject_hv_d(hg, ctx, groups, entry):
    rc, msg = _call(hg, ctx, groups, entry, _rows(N_REF, 1), ALLOC, _rows(N_QRY, 2), ALLOC, HV_D + 128)
    assert rc == hg.ffi.HG_E_INVALID
    assert msg.startswith(entry + ":"), msg


@pytest.mark.parametrize("symmetric", [True, False])
def test_sharded_sorted_output_equals_single_gpu(hg, ctx, symmetric):
    """a world-1 Peer's sorted hits and ANI thousandths are the single-GPU hg_dist_sorted result on the same rows"""
    import torch
    from hypergen_b200 import synth
    n, hv_d, th = 700, 1024, 0.0  # every pair: ties of ANI are ordered by (i, j)
    hashes, off = synth.hash_sets_family_dev(n, n_per=800, scaled=1500)
    sets = [hashes.numpy().view(np.uint64)[int(off[g]):int(off[g + 1])] for g in range(n)]
    r = ctx.encode_sets(sets, hv_d=hv_d)
    hv, norm = r["hv"], r["norm2"]
    cap = n * n
    peer = hg.Peer(ctx, 0, 1, hg.ffi.peer_window_need(n, hv_d, cap))
    try:
        d_hv, d_n = torch.from_numpy(hv).cuda(), torch.from_numpy(norm).cuda()
        if symmetric:
            peer.dist_sharded_dev(None, None, 0, 0, d_hv.data_ptr(), d_n.data_ptr(), [0, n], hv_d, 21, th, True, 0, 0, cap)
        else:
            peer.dist_sharded_dev(d_hv[:300].data_ptr(), d_n[:300].data_ptr(), 300, 0, d_hv.data_ptr(), d_n.data_ptr(), [0, n], hv_d,
                                  21, th, False, 0, 0, cap)
        hits, milli = peer.dist_sharded_hits(cap, sorted_output=True)
    finally:
        peer.close()
    r = hv if symmetric else hv[:300]
    want, want_milli = ctx.dist(r, norm[:r.shape[0]], hv, norm, ani_th=th, symmetric=symmetric, cap=cap, sorted_output=True,
                                want_milli=True)
    assert want.size == (n * (n - 1) // 2 if symmetric else 300 * n)
    assert hits.tobytes() == want.tobytes()
    assert np.array_equal(milli, want_milli)
