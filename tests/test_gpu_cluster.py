"""ANI clustering (hg_cluster_dev / hg_cluster_packed / hg_group_cluster_packed / hg_cluster_union_dev, cluster.cluster,
`hyper-gen cluster`) against scipy's connected components of the oracle's linked pairs.

The expected answer: oracle.dist_all's ANI of every pair j > i, the pairs with ani >= ani_th as the edges of a graph,
scipy.sparse.csgraph.connected_components on it, and rep[i] = the smallest index of i's component.  Every case compares
rep and n_clusters exactly: the result does not depend on the kernel, the window plan, the schedule or the GPU count."""
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_search import _correlated_rows, _family, _norms, _sketch_file  # noqa: E402

pytestmark = pytest.mark.gpu

AUTO, SIMT, TWO_LIMB, NARROW = 0, 1, 2, 3


def _components(n, i, j):
    """(rep, n_clusters) of the graph on n nodes with edges (i[t], j[t]): rep = the smallest index of each component"""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    g = coo_matrix((np.ones(len(i), np.int8), (np.asarray(i, np.int64), np.asarray(j, np.int64))), shape=(n, n))
    k, lab = connected_components(g, directed=False)
    first = np.full(k, n, np.int64)
    np.minimum.at(first, lab, np.arange(n))
    return first[lab].astype(np.uint32), int(k)


def _linked_ani(oracle, hv, norm, k=21):
    """the ANI of every pair j > i, in np.triu_indices order"""
    return oracle.dist_all(hv, norm, hv, norm, k=k, symmetric=True, want_dot=False)[0]


def _expected(n, ani, ani_th):
    i, j = np.triu_indices(n, 1)
    m = ani >= np.float32(ani_th)
    return _components(n, i[m], j[m])


def _cluster_dev(ctx, hv, norm, ani_th, path=AUTO):
    import torch
    n, D = hv.shape
    d_hv, d_n = torch.from_numpy(np.ascontiguousarray(hv)).cuda(), torch.from_numpy(np.ascontiguousarray(norm)).cuda()
    d_rep = torch.full((max(n, 1),), -1, dtype=torch.int32, device="cuda")  # garbage: every slot must be written
    torch.cuda.synchronize()
    k = ctx.cluster_dev(d_hv.data_ptr(), d_n.data_ptr(), n, D, 21, ani_th, path, d_rep.data_ptr())
    return d_rep.cpu().numpy().view(np.uint32)[:n].copy(), k


def _check(got, want):
    rep, k = got
    assert k == want[1]
    assert np.array_equal(rep, want[0])


@pytest.fixture(scope="module")
def fam(ctx, oracle):
    """1500 family sketches at D 4096 (families of 10 with ANIs from ~80 to ~99.9 inside a family) and their pair ANIs"""
    hv, norm, packed, bits = _family(ctx, 1500, 4096)
    return hv, norm, packed, bits, _linked_ani(oracle, hv, norm)


@pytest.mark.parametrize("ani_th", [0.0, 85.0, 95.0, 99.5, 100.0])
def test_family_sketches_against_scipy(ctx, fam, ani_th):
    hv, norm, _, _, ani = fam
    want = _expected(1500, ani, ani_th)
    sizes = np.bincount(np.bincount(want[0])[np.unique(want[0])])
    if ani_th == 0.0:
        assert want[1] == 1
    if ani_th == 95.0:  # clusters of several sizes, and singletons
        assert sizes[1] > 0 and np.count_nonzero(sizes[2:]) >= 2, sizes
    _check(_cluster_dev(ctx, hv, norm, ani_th), want)


@pytest.mark.parametrize("path", [SIMT, TWO_LIMB, NARROW, AUTO])
def test_each_kernel_gives_the_same_rep(ctx, fam, path):
    hv, norm, _, _, ani = fam
    got = _cluster_dev(ctx, hv, norm, 95.0, path)
    assert path == AUTO or ctx.dist_last_path == path, ctx.dist_last_reason
    _check(got, _expected(1500, ani, 95.0))


@pytest.fixture(scope="module")
def corr(oracle):
    """1400 rows of families of 8 whose packed form is 12 bits: past the single plane, within the limb split"""
    hv = _correlated_rows(np.random.default_rng(31), 1400, 1024, 8, 1500, 40, 2000)
    norm = _norms(oracle, hv)
    rows = [oracle.compress_hd_sketch(v) for v in hv]
    assert all(b == 12 for b, _ in rows)
    return hv, norm, np.stack([p for _, p in rows]), np.full(hv.shape[0], 12, np.uint8), _linked_ani(oracle, hv, norm)


@pytest.mark.parametrize("ani_th", [90.0, 99.95])
def test_packed_12_bit_rows_run_two_limb(ctx, corr, ani_th):
    hv, norm, packed, bits, ani = corr
    got = ctx.cluster_packed(packed, bits, norm, 1024, ani_th=ani_th)
    assert ctx.dist_last_path == TWO_LIMB and "fits two s8 limbs" in ctx.dist_last_reason, ctx.dist_last_reason
    _check(got, _expected(1400, ani, ani_th))


def test_declined_single_plane_reruns_two_limb_through_every_window(ctx, corr, monkeypatch):
    """int16 rows give the kernel choice no bit width: auto tries the single plane, whose pre-pass declines these rows,
    and the two-limb rerun must unite every window's edges too"""
    hv, norm, _, _, ani = corr
    monkeypatch.setenv("HG_CLUSTER_EDGE_CAP", str(1 << 17))
    got = _cluster_dev(ctx, hv, norm, 90.0)
    assert ctx.dist_last_path == TWO_LIMB and "declined" in ctx.dist_last_reason, ctx.dist_last_reason
    assert ctx.cluster_stats()[0][0] > 1
    _check(got, _expected(1400, ani, 90.0))


@pytest.fixture(scope="module")
def big(ctx):
    """3000 family sketches at D 1024: 4.5e6 pairs"""
    hv, norm, _, _ = _family(ctx, 3000, 1024, n_per=1000, first=20)
    return hv, norm


@pytest.mark.parametrize("path", [AUTO, SIMT, TWO_LIMB])
@pytest.mark.parametrize("ani_th", [0.0, 95.0])
def test_many_windows_with_ref_splits_equal_one_window(ctx, big, monkeypatch, path, ani_th):
    hv, norm = big
    n = hv.shape[0]
    monkeypatch.delenv("HG_CLUSTER_EDGE_CAP", raising=False)
    one = _cluster_dev(ctx, hv, norm, ani_th, path)
    counts = ctx.cluster_stats()[0]
    assert counts[0] == 1 and counts[3] == 1 << 26 and counts[1] == counts[2]
    monkeypatch.setenv("HG_CLUSTER_EDGE_CAP", "65536")  # 256 x 256 pairs: a new ref block every 256 rows
    many = _cluster_dev(ctx, hv, norm, ani_th, path)
    windows, linked, largest, cap = ctx.cluster_stats()[0]
    assert cap == 65536 and largest <= cap and linked == counts[1]
    assert windows > (n + 255) // 256  # more windows than column chunks: the refs were split
    assert windows == 1 + sum(k + 1 for k in range(1, (n + 255) // 256))
    if ani_th == 0.0:  # every pair linked: 4.5e6 edges through 65536-record windows, one cluster
        assert linked == n * (n - 1) // 2 and many[1] == 1 and not many[0].any()
    assert many[1] == one[1] and np.array_equal(many[0], one[0])


# ---- hg_cluster_union_dev ---------------------------------------------------------------------------------------------

def _edges(i, j):
    """hg_hit records (i, j, 0, 0) on the device"""
    import torch
    e = np.zeros((len(i), 4), np.uint32)
    e[:, 0], e[:, 1] = i, j
    return torch.from_numpy(e.view(np.int32)).cuda()


def _union(ctx, rep, i, j):
    import torch
    d_rep = torch.from_numpy(np.ascontiguousarray(rep, np.uint32).view(np.int32)).cuda()
    d_e = _edges(i, j)
    k = ctx.cluster_union_dev(rep.size, d_rep.data_ptr(), d_e.data_ptr() if len(i) else None, len(i))
    return d_rep.cpu().numpy().view(np.uint32).copy(), k


@pytest.mark.parametrize("order", ["descending", "shuffled"])
def test_union_chain_of_a_million_nodes(ctx, order):
    n = 1_000_000
    i = np.arange(n - 1, dtype=np.uint32)
    i = i[::-1] if order == "descending" else np.random.default_rng(7).permutation(i)
    rep, k = _union(ctx, np.arange(n, dtype=np.uint32), i, i + 1)
    assert k == 1 and not rep.any()


def test_union_star_with_the_last_index_as_hub(ctx):
    n = 200_000
    leaves = np.random.default_rng(8).permutation(n - 1).astype(np.uint32)
    rep, k = _union(ctx, np.arange(n, dtype=np.uint32), np.full(n - 1, n - 1, np.uint32), leaves)
    assert k == 1 and not rep.any()


def _random_graph(n, m, seed):
    """random edges in both orientations, with duplicates and self-loops"""
    rng = np.random.default_rng(seed)
    i, j = rng.integers(0, n, m).astype(np.uint32), rng.integers(0, n, m).astype(np.uint32)
    dup = rng.integers(0, m, m // 10)
    loops = rng.integers(0, n, m // 20).astype(np.uint32)
    i = np.concatenate([i, j[dup], loops])
    j = np.concatenate([j, i[dup], loops])
    assert (i > j).any() and (i < j).any()
    return i, j


def test_union_random_graph_with_duplicates_self_loops_and_both_orientations(ctx):
    n = 300_000
    i, j = _random_graph(n, 250_000, 9)
    want = _components(n, i, j)
    assert 1 < want[1] < n
    _check(_union(ctx, np.arange(n, dtype=np.uint32), i, j), want)


def test_union_on_top_of_a_previous_result(ctx):
    n = 300_000
    i, j = _random_graph(n, 250_000, 10)
    h = i.size // 2
    first = _union(ctx, np.arange(n, dtype=np.uint32), i[:h], j[:h])
    _check(first, _components(n, i[:h], j[:h]))
    _check(_union(ctx, first[0], i[h:], j[h:]), _components(n, i, j))


def test_union_without_edges_flattens_the_forest(ctx):
    rep, k = _union(ctx, np.arange(1000, dtype=np.uint32), [], [])
    assert k == 1000 and np.array_equal(rep, np.arange(1000))
    forest = np.array([0, 0, 1, 2, 4, 4, 5, 0], np.uint32)  # two chains 0 <- 1 <- 2 <- 3, 7 -> 0 and 4 <- 5 <- 6
    rep, k = _union(ctx, forest, [], [])
    assert k == 2 and rep.tolist() == [0, 0, 0, 0, 4, 4, 4, 0]


@pytest.mark.parametrize("bad", ["edge_index", "rep_above_index"])
def test_union_rejects_bad_input_and_leaves_the_forest(ctx, hg, bad):
    import torch
    n = 5000
    rep = np.arange(n, dtype=np.uint32)
    rep[100:200] = 50
    i, j = np.arange(0, n - 1, dtype=np.uint32), np.arange(1, n, dtype=np.uint32)
    if bad == "edge_index":
        j[1234] = n
    else:
        rep[4000] = 4001
    d_rep = torch.from_numpy(rep.view(np.int32)).cuda()
    d_e = _edges(i, j)
    with pytest.raises(hg.HyperGenError) as ei:
        ctx.cluster_union_dev(n, d_rep.data_ptr(), d_e.data_ptr(), i.size)
    assert ei.value.code == hg.ffi.HG_E_INVALID
    assert np.array_equal(d_rep.cpu().numpy().view(np.uint32), rep)


# ---- edge cases ---------------------------------------------------------------------------------------------------------

def test_no_rows_and_one_row(ctx, fam):
    hv, norm = fam[0], fam[1]
    assert ctx.cluster_dev(None, None, 0, 4096, 21, 95.0, 0, None) == 0
    rep, k = ctx.cluster_packed(np.zeros((0, 8192), np.uint8), np.zeros(0, np.uint8), np.zeros(0, np.int32), 4096)
    assert rep.size == 0 and k == 0
    rep, k = _cluster_dev(ctx, hv[:1], norm[:1], 95.0)
    assert k == 1 and rep.tolist() == [0]


def test_empty_sketch_is_a_singleton(ctx, oracle, fam):
    hv, norm = fam[0][:600].copy(), fam[1][:600].copy()
    hv[37], norm[37] = 0, 0
    ani = _linked_ani(oracle, hv, norm)
    for th, joined in ((95.0, False), (0.0, True)):
        want = _expected(600, ani, th)
        assert (np.count_nonzero(want[0] == want[0][37]) > 1) == joined
        _check(_cluster_dev(ctx, hv, norm, th), want)


def test_identical_copies_are_linked_at_100(ctx, fam):
    hv, norm = fam[0][:400].copy(), fam[1][:400].copy()
    hv[333], norm[333] = hv[12], norm[12]
    rep, k = _cluster_dev(ctx, hv, norm, 100.0)
    assert rep[333] == 12 and k == 399
    assert np.array_equal(np.delete(rep, 333), np.delete(np.arange(400), 333))


@pytest.mark.parametrize("ani_th", [85.0, 95.0])
def test_dev_equals_packed(ctx, fam, ani_th):
    hv, norm, packed, bits, _ = fam
    dev = _cluster_dev(ctx, hv, norm, ani_th)
    rep, k = ctx.cluster_packed(packed, bits, norm, 4096, ani_th=ani_th)
    assert k == dev[1] and np.array_equal(rep, dev[0])


# ---- hg_group_cluster_packed ----------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def wide(ctx):
    """7200 family sketches at D 1024: 2.6e7 pairs, enough for three members of at least 2^23 pairs each"""
    hv, norm, packed, bits = _family(ctx, 7200, 1024, n_per=1000, first=40)
    return hv, norm, packed, bits


@pytest.mark.parametrize("ordinals,n,used", [([0, 0], 7200, 2), ([0, 0, 0], 7200, 3), ([0, 0, 0], 6000, 2), ([0, 0], 4000, 1)])
@pytest.mark.parametrize("ani_th", [85.0, 95.0])
def test_group_on_gpu0_equals_one_context(ctx, hg, wide, ordinals, n, used, ani_th):
    _, norm, packed, bits = wide
    args = (packed[:n], bits[:n], norm[:n], 1024)
    with hg.Group(ordinals=ordinals) as g:
        got = g.cluster_packed(*args, ani_th=ani_th)
        ran = [g.cluster_stats(m)[0][0] > 0 for m in range(len(ordinals))]
    assert ran == [m < used for m in range(len(ordinals))]
    want = ctx.cluster_packed(*args, ani_th=ani_th)
    assert got[1] == want[1] and np.array_equal(got[0], want[0])


def _n_gpus():
    import torch
    return torch.cuda.device_count()


def test_group_all_gpus_equals_one_gpu(ctx, hg, wide):
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    _, norm, packed, bits = wide
    with hg.Group() as g:
        got = g.cluster_packed(packed, bits, norm, 1024, ani_th=95.0)
        assert all(g.cluster_stats(m)[0][0] > 0 for m in range(min(g.size, 3)))
    want = ctx.cluster_packed(packed, bits, norm, 1024, ani_th=95.0)
    assert got[1] == want[1] and np.array_equal(got[0], want[0])


# ---- CLI and Python ----------------------------------------------------------------------------------------------------

def _lines(names, rep):
    order = np.lexsort((np.arange(rep.size), rep))
    return "".join("%s\t%s\n" % (names[rep[t]], names[t]) for t in order)


def test_cli_and_python_write_the_expected_text(ctx, oracle, fam, tmp_path):
    from hypergen_b200 import _build, cluster, fileio
    exe = _build.build_host()
    hv, norm, packed, bits = fam[0][:700], fam[1][:700], fam[2][:700], fam[3][:700]
    ani = _linked_ani(oracle, hv, norm)
    names = ["g/s%04d.fna" % g for g in range(700)]
    sk = str(tmp_path / "all.sketch")
    _sketch_file(fileio, sk, packed, bits, norm, names)
    for th in (95.0, 99.5):
        want = _lines(names, _expected(700, ani, th)[0])
        assert cluster.format_cluster_lines(names, _expected(700, ani, th)[0]) == want
        cmd = [exe, "cluster", "-r", sk, "-o", str(tmp_path / "cc.tsv")]
        sc = cluster.SketchCluster(sk, str(tmp_path / "py.tsv"))
        if th != 95.0:
            cmd += ["-a", str(th)]
            sc.ani_th = th
        assert cluster.SketchCluster(sk).ani_th == 95.0
        py = cluster.cluster(sc, ctx=ctx)
        p = subprocess.run(cmd, capture_output=True, text=True, check=True)
        assert py == want
        assert open(tmp_path / "py.tsv", "rb").read() == want.encode()
        assert open(tmp_path / "cc.tsv", "rb").read() == want.encode()
        assert "700 sketches in %d clusters (ANI >= %.1f)" % (_expected(700, ani, th)[1], th) in p.stdout


def test_cli_all_gpus_writes_the_same_bytes_as_one_gpu(hg, wide, tmp_path):
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    from hypergen_b200 import _build, cluster, fileio
    exe = _build.build_host()
    _, norm, packed, bits = wide
    sk = str(tmp_path / "all.sketch")
    _sketch_file(fileio, sk, packed, bits, norm, ["g/s%05d.fna" % g for g in range(norm.size)], hv_d=1024)
    outs = {}
    for name, env in (("one", dict(os.environ, HG_GPUS="1")), ("all", dict(os.environ))):
        tsv = str(tmp_path / (name + ".tsv"))
        p = subprocess.run([exe, "cluster", "-r", sk, "-o", tsv], env=env, capture_output=True, text=True, check=True)
        outs[name] = (open(tsv, "rb").read(), p.stdout.replace(tsv, "OUT"))
    assert outs["one"] == outs["all"] and outs["one"][0]
    with hg.Group() as g:
        assert cluster.cluster(cluster.SketchCluster(sk), group=g).encode() == outs["one"][0]


# ---- argument errors ----------------------------------------------------------------------------------------------------

def test_argument_errors(ctx, hg):
    import torch
    d = torch.zeros(300 * 256, dtype=torch.int16, device="cuda")
    nrm = torch.ones(300, dtype=torch.int32, device="cuda")
    rep = torch.zeros(300, dtype=torch.int32, device="cuda")
    ok = (d.data_ptr(), nrm.data_ptr(), 300, 256, 21, 95.0, 0, rep.data_ptr())
    assert ctx.cluster_dev(*ok) == 300  # zero rows with norm 1: every ANI is 0, nothing is linked at 95
    bad = [
        (None, nrm.data_ptr(), 300, 256, 21, 95.0, 0, rep.data_ptr()),
        (d.data_ptr(), None, 300, 256, 21, 95.0, 0, rep.data_ptr()),
        (d.data_ptr(), nrm.data_ptr(), 300, 256, 21, 95.0, 0, None),
        (d.data_ptr(), nrm.data_ptr(), 300, 320, 21, 95.0, 0, rep.data_ptr()),
        (d.data_ptr(), nrm.data_ptr(), 300, 256, 21, 95.0, 4, rep.data_ptr()),
        (d.data_ptr(), nrm.data_ptr(), 300, 256, 21, 95.0, -1, rep.data_ptr()),
        (d.data_ptr(), nrm.data_ptr(), 300, 256, 21, float("nan"), 0, rep.data_ptr()),
    ]
    for args in bad:
        with pytest.raises(hg.HyperGenError) as ei:
            ctx.cluster_dev(*args)
        assert ei.value.code == hg.ffi.HG_E_INVALID
    with pytest.raises(hg.HyperGenError, match="NaN"):
        ctx.cluster_dev(*bad[-1])
    e = torch.zeros(64, dtype=torch.int32, device="cuda")
    for args in ((10, None, e.data_ptr(), 4), (10, rep.data_ptr(), None, 4)):
        with pytest.raises(hg.HyperGenError) as ei:
            ctx.cluster_union_dev(*args)
        assert ei.value.code == hg.ffi.HG_E_INVALID


@pytest.mark.parametrize("entry", ["hg_cluster_packed", "hg_group_cluster_packed"])
@pytest.mark.parametrize("bad", ["ok", "bits_0", "bits_17", "stride_below_width", "null_rep", "nan"])
def test_packed_entries_reject_bad_rows(hg, ctx, entry, bad):
    import ctypes as C
    lib = hg.ffi.load()
    n, hv_d, bits_v, alloc = 600, 256, 8, 512
    rng = np.random.default_rng(3)
    packed = rng.integers(0, 256, n * alloc, dtype=np.uint8)
    bits = np.full(n, bits_v, np.uint8)
    norm = rng.integers(1, 1 << 20, n, dtype=np.int32)
    rep = np.zeros(n, np.uint32)
    stride, ani_th, rep_p = alloc, 95.0, rep.ctypes.data
    if bad in ("bits_0", "bits_17"):
        bits[3] = 0 if bad == "bits_0" else 17
    elif bad == "stride_below_width":
        stride = bits_v * hv_d // 8 - 4
    elif bad == "null_rep":
        rep_p = None
    elif bad == "nan":
        ani_th = float("nan")
    k = C.c_uint32(0)
    with hg.Group(ordinals=[0, 0]) as g:
        h = ctx._h if entry == "hg_cluster_packed" else g._h
        rc = getattr(lib, entry)(h, packed.ctypes.data, stride, bits.ctypes.data, norm.ctypes.data, n, hv_d, 21, ani_th, 0, rep_p,
                                 C.byref(k))
        msg = lib.hg_last_error().decode()
    if bad == "ok":
        assert rc == hg.ffi.HG_OK, msg
        return
    assert rc == hg.ffi.HG_E_INVALID
    assert msg.startswith(entry + ":"), msg
    if bad.startswith("bits"):
        assert "ref sketch 3 has hv_quant_bits %d" % bits[3] in msg, msg
