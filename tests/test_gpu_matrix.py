"""The all-vs-all ANI matrix (hg_ani_matrix_dev / hg_ani_matrix_packed / hg_group_ani_matrix_packed, matrix.py,
`hyper-gen triangle`) against the oracle, bit for bit.

The expected answer is oracle.dist_all's ANI of every (ref, query) pair: entry (i, j) of the rectangle, and of the
strict lower triangle for j < i.  Every comparison is of the float32 bits."""
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_dist_wrap import CASES as WRAP_CASES  # noqa: E402
from test_gpu_dist_wrap import _set as _wrap_set  # noqa: E402
from test_gpu_search import _correlated_rows, _family, _milli, _norms, _sketch_file  # noqa: E402

pytestmark = pytest.mark.gpu

AUTO, SIMT, TWO_LIMB, NARROW = 0, 1, 2, 3
PATHS = [SIMT, TWO_LIMB, NARROW, AUTO]


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _rect(oracle, r, rn, q, qn):
    return oracle.dist_all(r, rn, q, qn, want_dot=False)[0].reshape(r.shape[0], q.shape[0])


def _lower(square):
    return square[np.tril_indices(square.shape[0], -1)]


@pytest.fixture(scope="module")
def fam(ctx, oracle):
    """1500 family sketches at D 4096 (their square from the oracle) and a 1500 x 700 ref x query pair of sets"""
    hv, norm, packed, bits = _family(ctx, 2200, 4096)
    a, b = slice(0, 1500), slice(1500, 2200)
    sq = _rect(oracle, hv[a], norm[a], hv[a], norm[a])
    rxq = _rect(oracle, hv[a], norm[a], hv[b], norm[b])
    return (hv[a], norm[a], packed[a], bits[a]), (hv[b], norm[b], packed[b], bits[b]), sq, rxq


def _dev(ctx, r, rn, q=None, qn=None, lower=True, path=AUTO, ld=None, sentinel=None):
    """hg_ani_matrix_dev on torch copies of the rows; returns the float32 output (with its padding when ld is given)"""
    import torch
    d_r, d_rn = torch.from_numpy(np.ascontiguousarray(r)).cuda(), torch.from_numpy(np.ascontiguousarray(rn)).cuda()
    d_q, d_qn = (d_r, d_rn) if q is None else (torch.from_numpy(np.ascontiguousarray(q)).cuda(), torch.from_numpy(np.ascontiguousarray(qn)).cuda())
    R, Q = r.shape[0], d_q.shape[0]
    ld = ld or Q
    size = R * (R - 1) // 2 if lower else max(0, (R - 1) * ld + Q)
    out = torch.full((max(size, 1),), -1 if sentinel is None else sentinel, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.ani_matrix_dev(d_r.data_ptr(), d_rn.data_ptr(), R, d_q.data_ptr(), d_qn.data_ptr(), Q, r.shape[1], 21, path, lower, out.data_ptr(),
                       0 if lower else ld)
    return out.cpu().numpy()[:size].view(np.float32)


@pytest.mark.parametrize("path", PATHS, ids=["simt", "two_limb", "narrow", "auto"])
def test_family_lower_square_and_rectangle(ctx, oracle, fam, path):
    (r, rn, rp, rb), (q, qn, qp, qb), sq, rxq = fam
    tri = ctx.ani_matrix_packed(rp, rb, rn, hv_d=4096, path=path, lower=True)
    assert ctx.ani_matrix_stats()[0][3] == ctx.dist_last_path
    if path != AUTO:
        assert ctx.dist_last_path == path, ctx.dist_last_reason
    assert np.array_equal(_bits(tri), _bits(_lower(sq)))
    full = ctx.ani_matrix_packed(rp, rb, rn, hv_d=4096, path=path, lower=False)
    assert np.array_equal(_bits(full), _bits(sq))
    rect = ctx.ani_matrix_packed(rp, rb, rn, qp, qb, qn, hv_d=4096, path=path, lower=False)
    assert rect.shape == (1500, 700) and np.array_equal(_bits(rect), _bits(rxq))
    # the device entry writes the same bytes
    assert np.array_equal(_bits(_dev(ctx, r, rn, path=path)), _bits(tri))
    assert np.array_equal(_bits(_dev(ctx, r, rn, q, qn, lower=False, path=path)), _bits(rxq).ravel())


@pytest.mark.parametrize("n", [0, 1, 2, 255, 257])
def test_row_counts(ctx, oracle, fam, n):
    (r, rn, rp, rb), (q, qn, _, _), sq, rxq = fam
    tri = ctx.ani_matrix_packed(rp[:n], rb[:n], rn[:n], hv_d=4096, lower=True)
    assert tri.size == n * (n - 1) // 2
    assert np.array_equal(_bits(tri), _bits(_lower(sq[:n, :n])))
    if 2 <= n < 128:  # fewer pairs than one 128 x 128 tensor tile: auto runs SIMT
        assert ctx.dist_last_path == SIMT, ctx.dist_last_reason
    got = _dev(ctx, r[:n], rn[:n], q[:n // 2], qn[:n // 2], lower=False)
    assert np.array_equal(_bits(got), _bits(rxq[:n, :n // 2]).ravel())


def test_padding_cells_are_never_written(ctx, oracle, fam):
    (r, rn, _, _), (q, qn, _, _), _, rxq = fam
    R, Q, ld = 700, 300, 300 + 37
    got = _dev(ctx, r[:R], rn[:R], q[:Q], qn[:Q], lower=False, ld=ld).view(np.int32)
    full = np.full(R * ld, -1, np.int32)
    full[: got.size] = got
    full = full.reshape(R, ld)
    assert np.array_equal(full[:, :Q].view(np.uint32), _bits(rxq[:R, :Q]))
    assert (full[:, Q:] == -1).all()


@pytest.mark.parametrize("lower", [True, False], ids=["lower", "rect"])
def test_many_bands_equal_one(ctx, fam, monkeypatch, lower):
    (r, rn, rp, rb), (q, qn, qp, qb), sq, rxq = fam
    args = (rp, rb, rn) if lower else (rp, rb, rn, qp, qb, qn)
    want = _lower(sq) if lower else rxq
    one = ctx.ani_matrix_packed(*args, hv_d=4096, lower=lower)
    assert ctx.ani_matrix_stats()[0][0] == 1
    for rows in (256, 100):  # one tile row per band; a band edge that cuts a tile
        monkeypatch.setenv("HG_MATRIX_BAND_BYTES", str(rows * (1500 if lower else 700) * 4))
        for path in (SIMT, TWO_LIMB, NARROW):
            got = ctx.ani_matrix_packed(*args, hv_d=4096, lower=lower, path=path)
            counts = ctx.ani_matrix_stats()[0]
            assert counts[0] > 1 and counts[1] == want.size and counts[2] == 4 * want.size, counts
            assert np.array_equal(_bits(got), _bits(one)) and np.array_equal(_bits(got), _bits(want))


def test_declined_single_plane_reruns_two_limb_and_copies_once(ctx, oracle, monkeypatch):
    """10-bit packed rows whose values span far more than one s8 plane: auto tries the single plane, whose pre-pass
    declines them.  The verdict is read before the first band, so the two-limb run's bands are the only ones written and
    copied to the host."""
    hv = _correlated_rows(np.random.default_rng(32), 600, 1024, 8, 500, 20, 500)
    norm = _norms(oracle, hv)
    rows = [oracle.compress_hd_sketch(v) for v in hv]
    assert all(b == 10 for b, _ in rows)
    packed, bits = np.stack([p for _, p in rows]), np.full(600, 10, np.uint8)
    monkeypatch.setenv("HG_MATRIX_BAND_BYTES", str(100 * 600 * 4))
    got = ctx.ani_matrix_packed(packed, bits, norm, hv_d=1024, lower=True)
    assert ctx.dist_last_path == TWO_LIMB and "declined" in ctx.dist_last_reason, ctx.dist_last_reason
    auto = ctx.ani_matrix_stats()[0]
    forced = ctx.ani_matrix_packed(packed, bits, norm, hv_d=1024, lower=True, path=TWO_LIMB)
    assert ctx.ani_matrix_stats()[0] == auto and auto[0] > 1 and auto[1] == 600 * 599 // 2 and auto[2] == 4 * auto[1], auto
    assert np.array_equal(_bits(got), _bits(forced))
    assert np.array_equal(_bits(got), _bits(_lower(_rect(oracle, hv, norm, hv, norm))))
    # int16 rows on the device entry take the same route
    assert np.array_equal(_bits(_dev(ctx, hv, norm)), _bits(got))
    assert ctx.dist_last_path == TWO_LIMB and "declined" in ctx.dist_last_reason, ctx.dist_last_reason


@pytest.mark.parametrize("path", PATHS, ids=["simt", "two_limb", "narrow", "auto"])
def test_ref_rows_inside_the_query_buffer(ctx, fam, monkeypatch, path):
    """a rectangle whose ref rows are rows [k, k + m) of the query buffer itself (a row shard against the whole set), in
    one band and in many"""
    import torch
    (r, rn, _, _), _, sq, _ = fam
    d_hv, d_n = torch.from_numpy(r).cuda(), torch.from_numpy(rn).cuda()
    n, k, m = r.shape[0], 300, 700
    for band_rows in (None, 100):
        if band_rows:
            monkeypatch.setenv("HG_MATRIX_BAND_BYTES", str(band_rows * n * 4))
        out = torch.full((m * n,), -1, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        ctx.ani_matrix_dev(d_hv.data_ptr() + k * 4096 * 2, d_n.data_ptr() + k * 4, m, d_hv.data_ptr(), d_n.data_ptr(), n, 4096, 21, path,
                           False, out.data_ptr(), n)
        if path != AUTO:
            assert ctx.dist_last_path == path, ctx.dist_last_reason
        assert (ctx.ani_matrix_stats()[0][0] > 1) == bool(band_rows)
        assert np.array_equal(out.cpu().numpy().view(np.uint32).reshape(m, n), _bits(sq[k:k + m]))


@pytest.mark.parametrize("name,path", WRAP_CASES, ids=["%s-%d" % c for c in WRAP_CASES])
def test_wrapping_denominators_every_kernel(ctx, oracle, name, path):
    s = _wrap_set(name, oracle)
    n = s.hv.shape[0]
    sq = np.zeros((n, n), np.float32)
    sq[np.triu_indices(n, 1)] = s.sym[0]
    tri = _dev(ctx, s.hv, s.norm, path=path)
    assert np.array_equal(_bits(tri), _bits(sq.T[np.tril_indices(n, -1)]))
    rect = _dev(ctx, s.hv, s.norm, s.hv[: s.nq], s.norm[: s.nq], lower=False, path=path)
    assert np.array_equal(_bits(rect), _bits(s.rxq[0]))


def test_offsets_beyond_2_32(ctx, fam):
    """a rectangle whose last rows start past 2^32 floats (27 GB of HBM): every owned cell written, every gap untouched"""
    import torch
    (r, rn, _, _), _, sq, _ = fam
    n, ld = 200, (1 << 25) + 3
    assert (n - 1) * ld > 2**32
    d_r, d_rn = torch.from_numpy(r[:n]).cuda(), torch.from_numpy(rn[:n]).cuda()
    out = torch.full(((n - 1) * ld + n,), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.ani_matrix_dev(d_r.data_ptr(), d_rn.data_ptr(), n, d_r.data_ptr(), d_rn.data_ptr(), n, 4096, 21, AUTO, False, out.data_ptr(), ld)
    rows = torch.arange(n, device="cuda", dtype=torch.int64)[:, None] * ld + torch.arange(n, device="cuda")[None, :]
    got = out[rows.ravel()].cpu().numpy().view(np.uint32).reshape(n, n)
    assert np.array_equal(got, _bits(sq[:n, :n]))
    assert int((out != -1).sum().item()) == n * n
    del out
    torch.cuda.empty_cache()


@pytest.mark.parametrize("members", [2, 3])
def test_group_equals_one_context(hg, ctx, members):
    hv, norm, packed, bits = _family(ctx, 7400, 4096)
    g = hg.Group(ordinals=[0] * members)
    try:
        for lower, q in ((True, None), (False, slice(0, 3700))):
            qa = () if q is None else (packed[q], bits[q], norm[q])
            one = ctx.ani_matrix_packed(packed, bits, norm, *qa, hv_d=4096, lower=lower)
            got = g.ani_matrix_packed(packed, bits, norm, *qa, hv_d=4096, lower=lower)
            assert np.array_equal(_bits(got), _bits(one))
            assert all(g.ani_matrix_stats(m)[0][0] > 0 for m in range(members))  # every member had rows
    finally:
        g.close()


def test_cli_and_python_write_the_same_triangle(ctx, oracle, fam, tmp_path):
    from hypergen_b200 import _build, fileio, matrix
    exe = _build.build_host()
    (r, rn, rp, rb), _, sq, _ = fam
    n = 300
    names = ["set/g%04d.fna" % g for g in range(n)]
    f = str(tmp_path / "s.sketch")
    _sketch_file(fileio, f, rp[:n], rb[:n], rn[:n], names)
    py = matrix.triangle(f, str(tmp_path / "py.txt"), ctx=ctx)
    subprocess.check_call([exe, "triangle", "-r", f, "-o", str(tmp_path / "cc.txt")])
    assert open(tmp_path / "cc.txt", "rb").read() == py.encode()
    lines = py.split("\n")
    assert lines[0] == str(n) and lines[-1] == "" and len(lines) == n + 2
    want = _milli(sq[:n, :n])
    for i in (1, 2, 150, 299):
        cells = lines[i + 1].split("\t")
        assert cells[0] == names[i] and len(cells) == i + 1
        assert cells[1:] == ["%d.%03d" % (m // 1000, m % 1000) for m in want[i, :i]]


def test_argument_errors(ctx, hg):
    import torch
    d = torch.zeros(300 * 256, dtype=torch.int16, device="cuda")
    d2 = torch.zeros(300 * 256, dtype=torch.int16, device="cuda")
    n = torch.ones(300, dtype=torch.int32, device="cuda")
    out = torch.full((300 * 300,), -1, dtype=torch.int32, device="cuda")
    bad = [
        (d.data_ptr(), n.data_ptr(), 300, d2.data_ptr(), n.data_ptr(), 300, 256, 21, 0, True, out.data_ptr(), 0),  # lower, other rows
        (d.data_ptr(), n.data_ptr(), 300, d.data_ptr(), n.data_ptr(), 200, 256, 21, 0, True, out.data_ptr(), 0),  # lower, other n
        (d.data_ptr(), n.data_ptr(), 300, d2.data_ptr(), n.data_ptr(), 300, 256, 21, 0, False, out.data_ptr(), 299),  # ld < n_qry
        (None, n.data_ptr(), 300, d.data_ptr(), n.data_ptr(), 300, 256, 21, 0, True, out.data_ptr(), 0),
        (d.data_ptr(), n.data_ptr(), 300, d.data_ptr(), n.data_ptr(), 300, 256, 21, 0, True, None, 0),
        (d.data_ptr(), n.data_ptr(), 300, d.data_ptr(), n.data_ptr(), 300, 200, 21, 0, True, out.data_ptr(), 0),  # hv_d
        (d.data_ptr(), n.data_ptr(), 300, d.data_ptr(), n.data_ptr(), 300, 256, 21, 4, True, out.data_ptr(), 0),  # path
    ]
    for args in bad:
        with pytest.raises(hg.HyperGenError) as ei:
            ctx.ani_matrix_dev(*args)
        assert ei.value.code == hg.ffi.HG_E_INVALID
    assert (out == -1).all().item()  # nothing ran
    p = np.zeros((4, 512), np.uint8)
    b = np.full(4, 8, np.uint8)
    nm = np.ones(4, np.int32)
    with pytest.raises(hg.HyperGenError) as ei:
        ctx.ani_matrix_packed(p, b, nm, p.copy(), b, nm, hv_d=512, lower=True)  # lower, other rows
    assert ei.value.code == hg.ffi.HG_E_INVALID
