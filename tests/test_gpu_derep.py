"""Greedy ANI dereplication (hg_derep_dev / hg_derep_packed, derep.derep, `hyper-gen derep`) against a plain Python
greedy over the oracle's full n x n ANI matrix.

The expected answer: oracle.dist_all's ANI of every pair, mirrored into a symmetric matrix; the sketches walked in the
priority order, each a representative unless an earlier representative is within ani_th; every other sketch assigned to
the representative of the largest ANI at >= ani_th, ties to the first in the order.  Every case compares rep and n_reps
exactly: the result does not depend on the kernel, the window plan or the schedule."""
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_cluster import _expected as _single_linkage  # noqa: E402
from test_gpu_cluster import _linked_ani  # noqa: E402
from test_gpu_search import _correlated_rows, _family, _norms, _sketch_file  # noqa: E402

pytestmark = pytest.mark.gpu

AUTO, SIMT, TWO_LIMB, NARROW = 0, 1, 2, 3


def _full(n, ani):
    """the symmetric n x n matrix of the pair ANIs (np.triu_indices order); the diagonal is never read"""
    a = np.zeros((n, n), np.float32)
    i, j = np.triu_indices(n, 1)
    a[i, j] = ani
    a[j, i] = ani
    return a


def _greedy(a, ani_th, order=None):
    """(rep, n_reps) of greedy dereplication over the full ANI matrix a"""
    n = a.shape[0]
    th = np.float32(ani_th)
    order = np.arange(n) if order is None else np.asarray(order, np.int64)
    reps = []
    for g in order:
        if not reps or not (a[reps, g] >= th).any():
            reps.append(int(g))
    rep = np.arange(n, dtype=np.int64)
    is_rep = np.zeros(n, bool)
    is_rep[reps] = True
    r = np.asarray(reps)
    for g in np.flatnonzero(~is_rep):
        col = a[r, g]
        assert col.max() >= th
        rep[g] = r[int(np.argmax(col))]  # the first maximum: the first in the order among the best
    return rep.astype(np.uint32), len(reps)


def _derep_dev(ctx, hv, norm, ani_th, path=AUTO, order=None):
    import torch
    n, D = hv.shape
    d_hv, d_n = torch.from_numpy(np.ascontiguousarray(hv)).cuda(), torch.from_numpy(np.ascontiguousarray(norm)).cuda()
    d_rep = torch.full((max(n, 1),), -1, dtype=torch.int32, device="cuda")  # garbage: every slot must be written
    torch.cuda.synchronize()
    k = ctx.derep_dev(d_hv.data_ptr(), d_n.data_ptr(), n, D, 21, ani_th, path, d_rep.data_ptr(), order=order)
    return d_rep.cpu().numpy().view(np.uint32)[:n].copy(), k


def _check(got, want):
    rep, k = got
    assert k == want[1]
    assert np.array_equal(rep, want[0])


def _order(kind, norm, seed=5):
    if kind == "file":
        return None
    if kind == "random":
        return np.random.default_rng(seed).permutation(norm.size).astype(np.uint32)
    from hypergen_b200 import derep
    return derep.priority(norm, "size")


@pytest.fixture(scope="module")
def fam(ctx, oracle):
    """1500 family sketches at D 4096 and their full ANI matrix"""
    hv, norm, packed, bits = _family(ctx, 1500, 4096)
    ani = _linked_ani(oracle, hv, norm)
    return hv, norm, packed, bits, ani, _full(1500, ani)


@pytest.mark.parametrize("kind", ["file", "random", "size"])
@pytest.mark.parametrize("ani_th", [0.0, 85.0, 95.0, 99.5, 100.0])
def test_family_sketches_against_the_greedy(ctx, fam, ani_th, kind):
    hv, norm, _, _, ani, a = fam
    order = _order(kind, norm)
    want = _greedy(a, ani_th, order)
    if ani_th == 0.0:
        assert want[1] == 1
    if ani_th == 85.0:  # single linkage chains every family into one cluster; greedy keeps representatives apart
        assert _single_linkage(1500, ani, ani_th)[1] == 1 and want[1] > 100
    _check(_derep_dev(ctx, hv, norm, ani_th, order=order), want)


@pytest.mark.parametrize("path", [SIMT, TWO_LIMB, NARROW, AUTO])
def test_each_kernel_gives_the_same_rep(ctx, fam, path):
    hv, norm, _, _, _, a = fam
    order = _order("random", norm, seed=9)
    got = _derep_dev(ctx, hv, norm, 95.0, path, order)
    assert path == AUTO or ctx.dist_last_path == path, ctx.dist_last_reason
    _check(got, _greedy(a, 95.0, order))


def test_dist_last_path_reports_the_representative_phase(ctx, fam):
    """at ani_th 0 there is one representative: the assignment search is 1 x 1500 pairs, which auto runs on SIMT"""
    hv, norm = fam[0], fam[1]
    rep, k = _derep_dev(ctx, hv, norm, 0.0)
    assert k == 1 and not rep.any()
    assert ctx.dist_last_path == NARROW, ctx.dist_last_reason
    assert "tensor-narrow" in ctx.dist_last_reason


@pytest.fixture(scope="module")
def corr(oracle):
    """1400 rows of families of 8 whose packed form is 12 bits: past the single plane, within the limb split"""
    hv = _correlated_rows(np.random.default_rng(31), 1400, 1024, 8, 1500, 40, 2000)
    norm = _norms(oracle, hv)
    rows = [oracle.compress_hd_sketch(v) for v in hv]
    assert all(b == 12 for b, _ in rows)
    return hv, norm, np.stack([p for _, p in rows]), np.full(hv.shape[0], 12, np.uint8), _full(1400, _linked_ani(oracle, hv, norm))


def test_packed_12_bit_rows_run_two_limb(ctx, corr):
    hv, norm, packed, bits, a = corr
    order = _order("random", norm, seed=2)
    got = ctx.derep_packed(packed, bits, norm, 1024, ani_th=90.0, order=order)
    assert ctx.dist_last_path == TWO_LIMB and "fits two s8 limbs" in ctx.dist_last_reason, ctx.dist_last_reason
    _check(got, _greedy(a, 90.0, order))


def test_declined_single_plane_runs_no_greedy_step(ctx, corr, monkeypatch):
    """int16 rows give the kernel choice no bit width: auto tries the single plane, whose pre-pass declines these rows.
    The verdict is read before the first window, so no greedy step runs on the declined plane's empty edge lists (which
    would make every sketch of every chunk a representative) and the two-limb rerun starts from clean state."""
    hv, norm, _, _, a = corr
    monkeypatch.setenv("HG_CLUSTER_EDGE_CAP", str(1 << 17))
    got = _derep_dev(ctx, hv, norm, 90.0)
    assert ctx.dist_last_path == TWO_LIMB and "declined" in ctx.dist_last_reason, ctx.dist_last_reason
    assert ctx.derep_stats()[0][1] > 1
    want = _greedy(a, 90.0)
    assert want[1] < 1400
    _check(got, want)


# ---- a chain: only neighbours are linked ---------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def chain(ctx, oracle):
    """2500 sketches at D 1024, sketch t = hashes [400 t, 400 t + 2000) of one random universe: neighbours share 1600 of
    2000 hashes (ANI ~98.9), sketches two apart 1200 (~97.6)"""
    n, size, step = 2500, 2000, 400
    universe = np.random.default_rng(77).integers(1, 2**63, size + step * (n - 1), dtype=np.uint64)
    r = ctx.encode_sets([universe[step * t: step * t + size] for t in range(n)], hv_d=1024)
    hv, norm = r["hv"], r["norm2"]
    ani = _linked_ani(oracle, hv, norm)
    return hv, norm, ani, _full(n, ani)


def test_chain_single_linkage_is_one_cluster_and_greedy_takes_every_other(ctx, chain):
    hv, norm, ani, a = chain
    n, th = hv.shape[0], 98.3
    i, j = np.triu_indices(n, 1)
    linked = ani >= np.float32(th)
    assert np.array_equal(j[linked] - i[linked], np.ones(n - 1)), "the oracle's linked pairs are not exactly t, t + 1"
    assert _single_linkage(n, ani, th)[1] == 1
    want = _greedy(a, th)
    assert np.array_equal(np.flatnonzero(want[0] == np.arange(n)), np.arange(0, n, 2))
    got = _derep_dev(ctx, hv, norm, th)
    _check(got, want)
    counts = ctx.derep_stats()[0]
    assert counts[0] == 3 and counts[2] == n - 1 and counts[3] == n // 2  # the chain crosses two chunk boundaries
    rev = np.arange(n - 1, -1, -1, dtype=np.uint32)
    want_rev = _greedy(a, th, rev)
    assert np.array_equal(np.flatnonzero(want_rev[0] == np.arange(n)), np.arange(1, n, 2))
    _check(_derep_dev(ctx, hv, norm, th, order=rev), want_rev)


# ---- many windows ---------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def big(ctx, oracle):
    """3000 family sketches at D 1024: 4.5e6 pairs"""
    hv, norm, _, _ = _family(ctx, 3000, 1024, n_per=1000, first=20)
    return hv, norm, _full(3000, _linked_ani(oracle, hv, norm))


@pytest.mark.parametrize("path", [AUTO, SIMT, TWO_LIMB])
@pytest.mark.parametrize("ani_th", [0.0, 95.0])
def test_many_windows_with_ref_splits_equal_one_window_per_chunk(ctx, big, monkeypatch, path, ani_th):
    hv, norm, a = big
    n = hv.shape[0]
    order = _order("random", norm, seed=13)
    monkeypatch.delenv("HG_CLUSTER_EDGE_CAP", raising=False)
    one = _derep_dev(ctx, hv, norm, ani_th, path, order)
    counts = ctx.derep_stats()[0]
    assert counts[0] == 3 and counts[1] == 3 and counts[3] == one[1]  # chunks of 1024, 1024 and 952 columns
    monkeypatch.setenv("HG_CLUSTER_EDGE_CAP", "65536")  # 256 x 256 pairs: a new ref block every 256 rows
    many = _derep_dev(ctx, hv, norm, ani_th, path, order)
    chunks, windows, linked, reps = ctx.derep_stats()[0]
    assert chunks == (n + 255) // 256 and windows == 1 + sum(k + 1 for k in range(1, (n + 255) // 256))
    assert linked == counts[2] and reps == many[1]
    if ani_th == 0.0:
        assert linked == n * (n - 1) // 2
    _check(many, one)
    _check(many, _greedy(a, ani_th, order))


# ---- edge cases ---------------------------------------------------------------------------------------------------------

def test_no_rows_and_one_row(ctx, fam):
    hv, norm = fam[0], fam[1]
    assert ctx.derep_dev(None, None, 0, 4096, 21, 95.0, 0, None) == 0
    rep, k = ctx.derep_packed(np.zeros((0, 8192), np.uint8), np.zeros(0, np.uint8), np.zeros(0, np.int32), 4096)
    assert rep.size == 0 and k == 0
    for order in (None, np.zeros(1, np.uint32)):
        rep, k = _derep_dev(ctx, hv[:1], norm[:1], 95.0, order=order)
        assert k == 1 and rep.tolist() == [0]


def test_empty_sketch_is_its_own_representative(ctx, oracle, fam):
    hv, norm = fam[0][:600].copy(), fam[1][:600].copy()
    hv[37], norm[37] = 0, 0
    a = _full(600, _linked_ani(oracle, hv, norm))
    want = _greedy(a, 95.0)
    assert want[0][37] == 37 and np.count_nonzero(want[0] == 37) == 1
    _check(_derep_dev(ctx, hv, norm, 95.0), want)
    want = _greedy(a, 0.0, np.r_[37, np.delete(np.arange(600), 37)])
    assert want[1] == 1 and (want[0] == 37).all()
    _check(_derep_dev(ctx, hv, norm, 0.0, order=np.r_[37, np.delete(np.arange(600), 37)].astype(np.uint32)), want)


def test_threshold_above_100_makes_every_sketch_a_representative(ctx, fam):
    hv, norm = fam[0][:900], fam[1][:900]
    rep, k = _derep_dev(ctx, hv, norm, 100.5, order=_order("random", norm))
    assert k == 900 and np.array_equal(rep, np.arange(900))


@pytest.mark.parametrize("bad", ["repeat", "index_n", "nan"])
def test_bad_order_or_nan_is_rejected_with_nothing_written(ctx, hg, fam, bad):
    import torch
    hv, norm, packed, bits = fam[0][:500], fam[1][:500], fam[2][:500], fam[3][:500]
    order, th = np.arange(500, dtype=np.uint32)[::-1].copy(), 95.0
    if bad == "repeat":
        order[400] = order[3]
    elif bad == "index_n":
        order[250] = 500
    else:
        th = float("nan")
    d_hv, d_n = torch.from_numpy(hv).cuda(), torch.from_numpy(norm).cuda()
    d_rep = torch.full((500,), -7, dtype=torch.int32, device="cuda")
    with pytest.raises(hg.HyperGenError) as ei:
        ctx.derep_dev(d_hv.data_ptr(), d_n.data_ptr(), 500, 4096, 21, th, 0, d_rep.data_ptr(), order=order)
    assert ei.value.code == hg.ffi.HG_E_INVALID
    assert (d_rep.cpu().numpy() == -7).all()
    msg = {"repeat": "repeats an earlier entry", "index_n": "is not below n = 500", "nan": "NaN"}[bad]
    assert msg in str(ei.value)
    with pytest.raises(hg.HyperGenError, match=msg):
        ctx.derep_packed(packed, bits, norm, 4096, ani_th=th, order=order)


def test_dev_equals_packed(ctx, fam):
    hv, norm, packed, bits = fam[0], fam[1], fam[2], fam[3]
    order = _order("size", norm)
    dev = _derep_dev(ctx, hv, norm, 95.0, order=order)
    _check(ctx.derep_packed(packed, bits, norm, 4096, ani_th=95.0, order=order), dev)


# ---- CLI and Python ----------------------------------------------------------------------------------------------------

def _lines(names, rep):
    t = np.arange(rep.size)
    return "".join("%s\t%s\n" % (names[rep[k]], names[k]) for k in np.lexsort((t, t != rep, rep)))


def test_cli_and_python_write_the_expected_text(ctx, oracle, fam, tmp_path):
    from hypergen_b200 import _build, derep, fileio
    exe = _build.build_host()
    n = 700
    hv, norm, packed, bits = fam[0][:n], fam[1][:n], fam[2][:n], fam[3][:n]
    a = _full(n, _linked_ani(oracle, hv, norm))
    names = ["g/s%04d.fna" % g for g in range(n)]
    sk = str(tmp_path / "all.sketch")
    _sketch_file(fileio, sk, packed, bits, norm, names)
    assert derep.SketchDerep(sk).ani_th == 95.0 and derep.SketchDerep(sk).order == "file"
    for kind, th in (("file", 95.0), ("size", 95.0), ("size", 99.5)):
        order = None if kind == "file" else np.lexsort((np.arange(n), -norm.astype(np.int64)))
        rep, k = _greedy(a, th, order)
        want = _lines(names, rep)
        if kind == "size":  # members before their representative: the representative's line still comes first
            assert (rep < np.arange(n)).any()
        cmd = [exe, "derep", "-r", sk, "-o", str(tmp_path / "cc.tsv"), "-O", kind]
        sd = derep.SketchDerep(sk, str(tmp_path / "py.tsv"), order=kind)
        if th != 95.0:
            cmd += ["-a", str(th)]
            sd.ani_th = th
        py = derep.derep(sd, ctx=ctx)
        p = subprocess.run(cmd, capture_output=True, text=True, check=True)
        assert py == want
        assert open(tmp_path / "py.tsv", "rb").read() == want.encode()
        assert open(tmp_path / "cc.tsv", "rb").read() == want.encode()
        assert "Output %d sketches in %d clusters (greedy, ANI >= %.1f)" % (n, k, th) in p.stdout
    p = subprocess.run([exe, "derep", "-r", sk, "-o", str(tmp_path / "x.tsv"), "-O", "quality"], capture_output=True, text=True)
    assert p.returncode != 0 and "-O must be file or size" in p.stderr
    with pytest.raises(ValueError, match="unknown order"):
        derep.derep(derep.SketchDerep(sk, str(tmp_path / "x.tsv"), order="quality"), ctx=ctx)
    assert not os.path.exists(tmp_path / "x.tsv")
