"""GPU parity for the output stage: hg_sort_hits_dev / hg_dist_sorted put the hits in the order of
utils::dump_ani_file (reference src/utils.rs:262-285: stable ascending sort by ANI, reversed) and
round the `{:.3}` field like the reference's formatter.  Checked against the oracle's restatement
of that sort (oracle.ani_output_order) and against Python's exact decimal formatting."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _sort_on_gpu(ctx, hits, want_milli=True):
    d = torch.from_numpy(hits.view(np.uint8).reshape(-1).copy()).cuda()
    m = torch.zeros(max(hits.size, 1), dtype=torch.int32, device="cuda") if want_milli else None
    torch.cuda.synchronize()
    ctx.sort_hits_dev(d.data_ptr() if hits.size else None, hits.size, m.data_ptr() if want_milli else None)
    ctx.sync()
    out = d.cpu().numpy().view(hits.dtype)
    return out, (m.cpu().numpy().view(np.uint32)[:hits.size] if want_milli else None)


@pytest.mark.parametrize("n,R,Q,levels", [(0, 10, 10, 4), (1, 10, 10, 4), (2, 3, 3, 1), (37, 9, 9, 3), (5000, 300, 300, 50),
                                          (4096, 70000, 5, 7), (4097, 100, 70000, 4097), (300_000, 2000, 2000, 1000),
                                          (520_000, 1500, 1500, 77), (1_100_000, 1500, 1500, 3)])
@pytest.mark.parametrize("multi", [False, True])
def test_sort_matches_reference_order(ctx, hg, oracle, n, R, Q, levels, multi, monkeypatch):
    """multi=False: one cooperative kernel up to ~600 k records (4 or 16 rounds per warp), the multi-kernel
    path beyond; multi=True: the multi-kernel path at every size"""
    if multi:
        monkeypatch.setenv("HG_SORT_MULTI", "1")
    rng = np.random.default_rng(n + levels)
    # full R x Q enumeration; a few distinct ANI levels so that ties dominate
    pair = rng.choice(R * Q, size=n, replace=False) if n else np.zeros(0, np.int64)
    lv = np.float32(85.0) + rng.random(levels).astype(np.float32) * np.float32(15.0)
    lv[0] = np.float32(100.0)
    hits = np.zeros(n, hg.ffi.HIT_DTYPE)
    hits["i"], hits["j"] = pair // Q, pair % Q
    hits["ani"] = lv[rng.integers(0, levels, n)]
    hits["dot"] = rng.integers(-2**31, 2**31 - 1, n)
    got, milli = _sort_on_gpu(ctx, hits)
    # the oracle sorts the dense pair-indexed ANI vector: scatter the hits into it
    dense = np.zeros(R * Q, np.float32)
    dense[pair] = hits["ani"]
    want_pairs = oracle.ani_output_order(dense, 85.0)
    assert want_pairs.size == n
    assert np.array_equal(got["i"].astype(np.int64) * Q + got["j"], want_pairs)
    by_pair = {int(p): t for t, p in enumerate(pair)}
    src = np.array([by_pair[int(p)] for p in want_pairs[:2000]], np.int64)
    assert np.array_equal(got[:src.size], hits[src])                     # whole records travel with their keys
    want_milli = [int(("%.3f" % float(a)).replace(".", "")) for a in got["ani"][:5000]]
    assert milli[:5000].tolist() == want_milli


def test_milli_rounding_is_exact_half_even(ctx, hg):
    # f32 values that sit exactly on a .0005 boundary (representable: multiples of 2^-k) and neighbours
    vals = np.array([0.0, 100.0, 85.0, 99.9995, 87.0625, 87.1875, 90.4375, 96.5, 85.00049, 85.0005, 85.00051,
                     99.99949, 99.99951, 0.0004999, 12.3456789], np.float32)
    vals = np.concatenate([vals, np.nextafter(vals, np.float32(200)), np.nextafter(vals, np.float32(-1)).clip(0)])
    vals = np.concatenate([vals, (np.arange(0, 4000, dtype=np.float32) * np.float32(0.0078125) + np.float32(80.0))])  # k/128
    vals = np.unique(vals)
    hits = np.zeros(vals.size, hg.ffi.HIT_DTYPE)
    hits["ani"] = vals
    hits["i"] = np.arange(vals.size)
    got, milli = _sort_on_gpu(ctx, hits)
    assert np.array_equal(got["ani"], np.sort(vals)[::-1])
    assert milli.tolist() == [int(("%.3f" % float(a)).replace(".", "")) for a in got["ani"]]


def test_dist_sorted_is_dist_plus_reference_order(ctx, hg, oracle):
    from hypergen_b200 import synth, dist as hdist
    seq, off = synth.family_batch(96, 150_000, first=11)
    sk = oracle.sketch_batch(seq.numpy(), off, scaled=300, hv_d=1024)
    hv, norm = sk["hv"], sk["norm2"]
    for sym, q in ((True, slice(None)), (False, slice(5, 40))):
        qh, qn = (hv, norm) if sym else (hv[q].copy(), norm[q].copy())
        ani, dot = oracle.dist_all(hv, norm, qh, qn, symmetric=sym)
        for th in (0.0, 85.0, 97.0):
            hits, milli = ctx.dist(hv, norm, qh, qn, ani_th=th, symmetric=sym, sorted_output=True, want_milli=True)
            want = oracle.ani_output_order(ani, th)
            idx = hdist.pair_index(hits["i"].astype(np.int64), hits["j"].astype(np.int64), qh.shape[0], sym)
            assert np.array_equal(idx, want), (sym, th)
            assert np.array_equal(hits["ani"].view(np.uint32), ani[want].view(np.uint32))
            assert np.array_equal(hits["dot"], dot[want])
            assert milli.tolist() == [int(("%.3f" % float(a)).replace(".", "")) for a in hits["ani"]]


def _pack_bits(hv, b):
    """BitPacker8x at an explicit width b (hd.rs:139-153): lane l = idx % 8 carries the stream
    sum(u[8 r + l] << (b r)); its 32-bit word j sits at byte 32 j + 4 l of the block's 32 b bytes."""
    u = (hv.astype(np.int64) + (1 << (b - 1))).astype(np.uint64)
    out = np.zeros(b * hv.size // 8, np.uint8)
    for blk in range(hv.size // 256):
        ub = u[blk * 256:(blk + 1) * 256]
        o = out[blk * 32 * b:(blk + 1) * 32 * b].view(np.uint32).reshape(b, 8)
        for l in range(8):
            stream = 0
            for r in range(32):
                stream |= int(ub[8 * r + l]) << (b * r)
            for j in range(b):
                o[j, l] = (stream >> (32 * j)) & 0xFFFFFFFF
    return out


def test_dist_packed_equals_unpack_then_dist(ctx, hg, oracle):
    """hg_dist_packed (sketch-file payload in, sorted hits out) == oracle decompress + dist + order;
    mixed hv_quant_bits per row, different strides for ref and query, symmetric and not."""
    from hypergen_b200 import synth, dist as hdist
    D = 1024
    seq, off = synth.family_batch(140, 120_000, first=500)
    sk = oracle.sketch_batch(seq.numpy(), off, scaled=150, hv_d=D)
    hv, norm, bits, packed = sk["hv"].copy(), sk["norm2"].copy(), sk["quant_bits"].copy(), sk["packed"]
    # re-pack a few rows at a wider bit width than needed (legal in the file format) to mix widths
    for g in (3, 77, 139):
        bits[g] = min(int(bits[g]) + 2, 13)
    rows = [_pack_bits(hv[g], int(bits[g])) for g in range(140)]
    b0, p0 = oracle.compress_hd_sketch(hv[0])                   # pins the test's packer to the oracle's
    assert b0 == int(bits[0]) and np.array_equal(rows[0], p0)
    rp = np.zeros((140, 2 * D), np.uint8)
    for g, r in enumerate(rows):
        rp[g, :r.size] = r
    qsel = np.arange(20, 90)
    qp = np.zeros((qsel.size, 2 * D + 64), np.uint8)           # another stride
    qp[:, :2 * D] = rp[qsel]
    for sym in (True, False):
        if sym:
            args = (rp, bits, norm, rp, bits, norm)
            qh, qn = hv, norm
        else:
            args = (rp, bits, norm, qp, bits[qsel].copy(), norm[qsel].copy())
            qh, qn = hv[qsel], norm[qsel]
        ani, dot = oracle.dist_all(hv, norm, qh, qn, symmetric=sym)
        for th in (85.0, 0.0):
            hits, milli = ctx.dist_packed(*args, D, ani_th=th, symmetric=sym)
            want = oracle.ani_output_order(ani, th)
            idx = hdist.pair_index(hits["i"].astype(np.int64), hits["j"].astype(np.int64), qh.shape[0], sym)
            assert np.array_equal(idx, want), (sym, th)
            assert np.array_equal(hits["ani"].view(np.uint32), ani[want].view(np.uint32))
            assert np.array_equal(hits["dot"], dot[want])
            assert milli.tolist() == [int(("%.3f" % float(a)).replace(".", "")) for a in hits["ani"]]
        if sym:   # 140 x 140 fills a tensor tile and the rows are narrow: single-plane tensor path
            assert ctx.dist_last_path == 3 and "narrow" in ctx.dist_last_reason, ctx.dist_last_reason
        else:     # 140 x 70 pairs do not fill one 128 x 128 tile: exact SIMT path
            assert ctx.dist_last_path == 1


@pytest.mark.parametrize("sym", [True, False])
def test_dist_packed_streamed_in_chunks(ctx, hg, oracle, sym, monkeypatch):
    """hg_dist_packed with the packed rows arriving in several chunks (copy stream) while the earlier chunks are
    unpacked, pre-passed and compared: same sorted output as the oracle"""
    from hypergen_b200 import synth, dist as hdist
    monkeypatch.setenv("HG_DIST_CHUNK_ROWS", "256")
    D = 1024
    seq, off = synth.family_batch(600, 30_000, first=900)
    sk = oracle.sketch_batch(seq.numpy(), off, scaled=100, hv_d=D)
    hv, norm, bits, packed = sk["hv"], sk["norm2"], sk["quant_bits"], sk["packed"]
    if sym:
        args = (packed, bits, norm, packed, bits, norm)
        qh, qn = hv, norm
    else:
        q = np.arange(37, 337)
        args = (packed, bits, norm, packed[q].copy(), bits[q].copy(), norm[q].copy())
        qh, qn = hv[q], norm[q]
    ani, dot = oracle.dist_all(hv, norm, qh, qn, symmetric=sym)
    for th in (90.0, 0.0):
        hits, milli = ctx.dist_packed(*args, D, ani_th=th, symmetric=sym, cap=ani.size + 16)
        assert ctx.dist_last_path == 3 and "chunk" in ctx.dist_last_reason, ctx.dist_last_reason
        want = oracle.ani_output_order(ani, th)
        idx = hdist.pair_index(hits["i"].astype(np.int64), hits["j"].astype(np.int64), qh.shape[0], sym)
        assert np.array_equal(idx, want), (sym, th)
        assert np.array_equal(hits["ani"].view(np.uint32), ani[want].view(np.uint32))
        assert np.array_equal(hits["dot"], dot[want])


@pytest.mark.parametrize("sym", [True, False])
def test_dist_packed_wide_rows_streamed_two_limb(ctx, hg, oracle, sym, monkeypatch):
    """rows stored at 11 bits (wider than one s8 plane can hold): hg_dist_packed streams them through the two-limb
    tensor kernel, one partial launch per chunk"""
    from hypergen_b200 import synth, dist as hdist
    monkeypatch.setenv("HG_DIST_CHUNK_ROWS", "256")
    D = 1024
    seq, off = synth.family_batch(560, 30_000, first=1700)
    sk = oracle.sketch_batch(seq.numpy(), off, scaled=100, hv_d=D)
    hv, norm = sk["hv"], sk["norm2"]
    bits = np.full(560, 11, np.uint8)
    rp = np.zeros((560, 11 * D // 8), np.uint8)
    for g in range(560):
        rp[g] = _pack_bits(hv[g], 11)
    if sym:
        args = (rp, bits, norm, rp, bits, norm)
        qh, qn = hv, norm
    else:
        q = np.arange(11, 311)
        args = (rp, bits, norm, rp[q].copy(), bits[q].copy(), norm[q].copy())
        qh, qn = hv[q], norm[q]
    ani, dot = oracle.dist_all(hv, norm, qh, qn, symmetric=sym)
    hits, milli = ctx.dist_packed(*args, D, ani_th=0.0, symmetric=sym, cap=ani.size + 16)
    assert ctx.dist_last_path == 2 and "chunk" in ctx.dist_last_reason, ctx.dist_last_reason
    want = oracle.ani_output_order(ani, 0.0)
    idx = hdist.pair_index(hits["i"].astype(np.int64), hits["j"].astype(np.int64), qh.shape[0], sym)
    assert np.array_equal(idx, want), sym
    assert np.array_equal(hits["ani"].view(np.uint32), ani[want].view(np.uint32))
    assert np.array_equal(hits["dot"], dot[want])
