"""Top-k search (hg_search_dev / hg_search_packed, search.search, `hyper-gen search`) against the oracle.

The expected answer comes from oracle.dist_all: per query, the refs with ani >= ani_min ordered by (ANI desc, ref index
asc), the first top_k of them.  Every case compares n_found, every i, every dot, every ANI bit and ani_milli, and that
the unused slots are zero."""
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SIMT, TWO_LIMB, NARROW = 1, 2, 3


def _family(ctx, n, hv_d, n_per=3333, first=0):
    """family-structured sketches (synth.hash_sets_family_dev) encoded on the GPU -> (hv, norm, packed, bits)"""
    from hypergen_b200 import synth
    hashes, off = synth.hash_sets_family_dev(n, n_per=n_per, first=first)
    sets = [hashes.numpy().view(np.uint64)[int(off[g]):int(off[g + 1])] for g in range(n)]
    r = ctx.encode_sets(sets, hv_d=hv_d)
    return r["hv"], r["norm2"], r["packed"], r["quant_bits"]


def _norms(oracle, hv):
    return np.array([oracle.hv_l2_norm_sq(v) for v in hv], np.int32)


def _expected(oracle, r, rn, q, qn, top_k, ani_min, k=21):
    """(i, dot, ani, n_found) per query from the oracle's every-pair ANI"""
    ani, dot = oracle.dist_all(r, rn, q, qn, k=k)
    R, Q = r.shape[0], q.shape[0]
    ani, dot = ani.reshape(R, Q), dot.reshape(R, Q)
    ei = np.zeros((Q, top_k), np.uint32)
    ed = np.zeros((Q, top_k), np.int32)
    ea = np.zeros((Q, top_k), np.float32)
    nf = np.zeros(Q, np.uint32)
    for j in range(Q):
        cand = np.nonzero(ani[:, j] >= np.float32(ani_min))[0]
        order = cand[np.lexsort((cand, -ani[cand, j]))][:top_k]
        n = order.size
        nf[j] = n
        ei[j, :n], ed[j, :n], ea[j, :n] = order, dot[order, j], ani[order, j]
    return ei, ed, ea, nf


def _milli(a):
    return np.rint(a.astype(np.float64) * 1000.0).astype(np.uint32)


def _compare(got, want):
    hits, n_found, milli = got
    ei, ed, ea, nf = want
    Q, K = ei.shape
    assert np.array_equal(n_found, nf)
    live = np.arange(K)[None, :] < nf[:, None]
    assert np.array_equal(np.where(live, hits["i"], 0), ei)
    assert np.array_equal(np.where(live, hits["j"], 0), np.where(live, np.arange(Q, dtype=np.uint32)[:, None], 0))
    assert np.array_equal(hits["dot"], ed)
    assert np.array_equal(hits["ani"].view(np.uint32), ea.view(np.uint32))
    assert np.array_equal(milli, np.where(live, _milli(ea), 0))
    assert not hits["i"][~live].any() and not hits["j"][~live].any()  # unused slots are zero


def _search_dev(ctx, hg, r, rn, q, qn, top_k, ani_min=0.0, path=0, same=False):
    import torch
    R, D = r.shape
    Q = q.shape[0]
    d_r, d_rn = torch.from_numpy(np.ascontiguousarray(r)).cuda(), torch.from_numpy(np.ascontiguousarray(rn)).cuda()
    d_q, d_qn = (d_r, d_rn) if same else (torch.from_numpy(np.ascontiguousarray(q)).cuda(), torch.from_numpy(np.ascontiguousarray(qn)).cuda())
    d_out = torch.full((Q * top_k * 16,), 0xAB, dtype=torch.uint8, device="cuda")  # garbage: the unused slots must be zeroed
    d_nf = torch.zeros(Q, dtype=torch.int32, device="cuda")
    d_mi = torch.full((Q * top_k,), 7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.search_dev(d_r.data_ptr(), d_rn.data_ptr(), R, d_q.data_ptr(), d_qn.data_ptr(), Q, D, 21, top_k, ani_min, path,
                   d_out.data_ptr(), d_nf.data_ptr(), d_mi.data_ptr())
    hits = np.frombuffer(d_out.cpu().numpy().tobytes(), dtype=hg.ffi.HIT_DTYPE).reshape(Q, top_k).copy()
    return hits, d_nf.cpu().numpy().view(np.uint32).copy(), d_mi.cpu().numpy().view(np.uint32).reshape(Q, top_k).copy()


@pytest.fixture(scope="module")
def fam(ctx):
    """3000 refs and 300 queries at D 4096: queries are every 11th of 3300 family sketches, so most have their
    own sketch and its family among the refs, and the last 27 (families 300-329) are novel"""
    hv, norm, packed, bits = _family(ctx, 3300, 4096)
    sel = np.arange(0, 3300, 11)[:300]
    return (hv[:3000], norm[:3000], packed[:3000], bits[:3000]), (hv[sel], norm[sel], packed[sel], bits[sel])


@pytest.mark.parametrize("top_k", [1, 10, 64])
def test_family_sketches_both_passes(ctx, hg, oracle, fam, top_k):
    (r, rn, _, _), (q, qn, _, _) = fam
    got = _search_dev(ctx, hg, r, rn, q, qn, top_k)
    s, n_floor, n_main, _ = ctx.search_stats()[0]
    assert s < 3000 and n_floor > 0 and n_main > 0  # the floor pass ran
    _compare(got, _expected(oracle, r, rn, q, qn, top_k, 0.0))


def test_ani_min_above_some_queries_best(ctx, hg, oracle, fam):
    (r, rn, _, _), (q, qn, _, _) = fam
    want = _expected(oracle, r, rn, q, qn, 10, 97.0)
    assert (want[3] < 10).any() and (want[3] == 0).any()
    _compare(_search_dev(ctx, hg, r, rn, q, qn, 10, 97.0), want)


def test_dev_equals_packed(ctx, hg, oracle, fam):
    (r, rn, rp, rb), (q, qn, qp, qb) = fam
    dev = _search_dev(ctx, hg, r, rn, q, qn, 10)
    pk = ctx.search_packed(rp, rb, rn, qp, qb, qn, 4096, top_k=10)
    for a, b in zip(dev, pk):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("path", [SIMT, TWO_LIMB, NARROW])
def test_each_kernel_forced(ctx, hg, oracle, path):
    hv, norm, _, _ = _family(ctx, 1700, 1024, n_per=1000, first=50)
    r, rn, q, qn = hv[:1500], norm[:1500], hv[1500::2], norm[1500::2]
    q = np.concatenate([q, hv[:400:4]])  # and some queries with relatives among the refs
    qn = np.concatenate([qn, norm[:400:4]])
    got = _search_dev(ctx, hg, r, rn, q, qn, 16, path=path)
    assert ctx.dist_last_path == path, ctx.dist_last_reason
    _compare(got, _expected(oracle, r, rn, q, qn, 16, 0.0))


def _correlated_rows(rng, n, D, fam_size, lo, noise, peak):
    """rows of families: a shared base plus member noise, one element of magnitude `peak` per row"""
    base = rng.integers(-lo, lo + 1, (n // fam_size + 1, D))
    hv = base[np.arange(n) // fam_size] + rng.integers(-noise, noise + 1, (n, D)) * (np.arange(n) % fam_size)[:, None]
    hv = np.clip(hv, -lo, lo)
    hv[np.arange(n), rng.integers(0, D, n)] = np.where(rng.random(n) < 0.5, -peak, peak)
    return hv.astype(np.int16)


def test_packed_12_bit_rows_run_two_limb(ctx, hg, oracle):
    rng = np.random.default_rng(21)
    hv = _correlated_rows(rng, 1400, 1024, 8, 1500, 40, 2000)
    norm = _norms(oracle, hv)
    rows = [oracle.compress_hd_sketch(v) for v in hv]
    assert all(b == 12 for b, _ in rows)
    packed, bits = np.stack([p for _, p in rows]), np.full(hv.shape[0], 12, np.uint8)
    r, q = slice(0, 1200), slice(1150, 1400)
    got = ctx.search_packed(packed[r], bits[r], norm[r], packed[q], bits[q], norm[q], 1024, top_k=12)
    assert ctx.dist_last_path == TWO_LIMB, ctx.dist_last_reason
    _compare(got, _expected(oracle, hv[r], norm[r], hv[q], norm[q], 12, 0.0))


def test_shape_the_tensor_kernels_decline_runs_simt(ctx, hg, oracle):
    rng = np.random.default_rng(22)
    hv = _correlated_rows(rng, 1140, 33024, 6, 100, 10, 120)
    norm = _norms(oracle, hv)
    r, rn, q, qn = hv[:1100], norm[:1100], hv[1090:], norm[1090:]
    got = _search_dev(ctx, hg, r, rn, q, qn, 5)
    assert ctx.dist_last_path == SIMT and "declined this shape" in ctx.dist_last_reason
    _compare(got, _expected(oracle, r, rn, q, qn, 5, 0.0))


def test_fewer_pairs_than_one_tensor_tile(ctx, hg, oracle, fam):
    (r, rn, _, _), (q, qn, _, _) = fam
    r, rn, q, qn = r[:100], rn[:100], q[:50], qn[:50]
    got = _search_dev(ctx, hg, r, rn, q, qn, 7)
    assert ctx.dist_last_path == SIMT and ctx.search_stats()[0][0] == 100  # one pass over all refs
    _compare(got, _expected(oracle, r, rn, q, qn, 7, 0.0))


def test_top_k_at_least_n_ref(ctx, hg, oracle, fam):
    (r, rn, _, _), (q, qn, _, _) = fam
    r, rn, q, qn = r[:50], rn[:50], q[:20], qn[:20]
    for ani_min in (0.0, 90.0):
        want = _expected(oracle, r, rn, q, qn, 64, ani_min)
        assert ani_min or (want[3] == 50).all()
        _compare(_search_dev(ctx, hg, r, rn, q, qn, 64, ani_min), want)


@pytest.mark.parametrize("top_k", [8, 1024])
def test_duplicated_ref_ties_by_ascending_index(ctx, hg, oracle, top_k):
    """2100 copies of one sketch among 6000 refs.  top_k 8: the floor pass (every sample pair qualifies at ani_min 0)
    outgrows the initial candidate room of a fresh context, so the pass reruns.  top_k 1024: the sample has 2560 rows,
    so every floor-pass segment takes the select kernel's long-segment path (radix select), and 1024 of the 2100 tied
    copies are chosen by index."""
    hv, norm, _, _ = _family(ctx, 6016, 1024, n_per=1000, first=700)
    fresh = hg.Context(0)  # its scratch has never held candidates
    try:
        r, rn = hv[:6000].copy(), norm[:6000].copy()
        dup = np.sort(np.random.default_rng(5).choice(6000, 2100, replace=False))
        r[dup], rn[dup] = hv[6000], norm[6000]
        q, qn = hv[6000:], norm[6000:]  # the duplicated sketch, its family, and another family
        got = _search_dev(fresh, hg, r, rn, q, qn, top_k)
        counts = fresh.search_stats()[0]
        assert counts[3] >= 1 if top_k == 8 else counts[0] == 2560, counts
        want = _expected(oracle, r, rn, q, qn, top_k, 0.0)
        assert np.array_equal(want[0][0, :8], dup[:8])
        _compare(got, want)
    finally:
        fresh.close()


def test_empty_query_among_normal_ones(ctx, hg, oracle, fam):
    (r, rn, _, _), (q, qn, _, _) = fam
    q, qn = q[:40].copy(), qn[:40].copy()
    q[5], qn[5] = 0, 0
    got = _search_dev(ctx, hg, r, rn, q, qn, 10)
    want = _expected(oracle, r, rn, q, qn, 10, 0.0)
    assert np.array_equal(want[0][5], np.arange(10)) and not want[2][5].any()
    _compare(got, want)


def test_same_pointers_is_a_plain_self_search(ctx, hg, oracle, fam):
    (r, rn, _, _), _ = fam
    r, rn = r[:1500], rn[:1500]
    got = _search_dev(ctx, hg, r, rn, r, rn, 10, same=True)
    _compare(got, _expected(oracle, r, rn, r, rn, 10, 0.0))


def _sketch_file(fileio, path, packed, bits, norm, names, ksize=21, hv_d=4096):
    fileio.dump_sketch([fileio.FileSketch(ksize=ksize, hv_d=hv_d, hv_quant_bits=int(bits[g]), hv_norm_2=int(norm[g]), file_str=names[g],
                                          hv=packed[g, : int(bits[g]) * hv_d // 8].view(np.int16).copy())
                        for g in range(len(names))], path)


def test_cli_and_python_write_the_oracle_text(ctx, hg, oracle, fam, tmp_path):
    from hypergen_b200 import _build, fileio, search
    exe = _build.build_host()
    (r, rn, rp, rb), (q, qn, qp, qb) = fam
    R, Q = 1600, 60
    rnames = ["ref/g%04d.fna" % g for g in range(R)]
    qnames = ["qry/q%03d.fna" % g for g in range(Q)]
    ref_f, qry_f = str(tmp_path / "ref.sketch"), str(tmp_path / "qry.sketch")
    _sketch_file(fileio, ref_f, rp[:R], rb[:R], rn[:R], rnames)
    _sketch_file(fileio, qry_f, qp[:Q], qb[:Q], qn[:Q], qnames)
    ei, _, ea, nf = _expected(oracle, r[:R], rn[:R], q[:Q], qn[:Q], 5, 1.0)
    mi = _milli(ea)
    want = "".join("%s\t%s\t%d.%03d\n" % (rnames[ei[j, t]], qnames[j], mi[j, t] // 1000, mi[j, t] % 1000)
                   for j in range(Q) for t in range(nf[j]))
    py = search.search(search.SketchSearch(ref_f, qry_f, str(tmp_path / "py.tsv"), top_k=5, ani_min=1.0), ctx=ctx)
    subprocess.check_call([exe, "search", "-r", ref_f, "-q", qry_f, "-o", str(tmp_path / "cc.tsv"), "-n", "5", "-a", "1.0"])
    assert py == want and want
    assert open(tmp_path / "cc.tsv", "rb").read() == want.encode()
    bad = str(tmp_path / "k17.sketch")
    _sketch_file(fileio, bad, qp[:Q], qb[:Q], qn[:Q], qnames, ksize=17)
    with pytest.raises(ValueError, match="different kmer sizes"):
        search.search(search.SketchSearch(ref_f, bad, ""), ctx=ctx)
    p = subprocess.run([exe, "search", "-r", ref_f, "-q", bad, "-o", str(tmp_path / "x.tsv")], capture_output=True, text=True)
    assert p.returncode != 0 and "different kmer sizes" in p.stderr


def test_argument_errors(ctx, hg):
    import torch
    d = torch.zeros(300 * 256, dtype=torch.int16, device="cuda")
    n = torch.ones(300, dtype=torch.int32, device="cuda")
    out = torch.zeros(300 * 1025 * 16, dtype=torch.uint8, device="cuda")
    nf = torch.zeros(300, dtype=torch.int32, device="cuda")
    ok = (d.data_ptr(), n.data_ptr(), 300, d.data_ptr(), n.data_ptr(), 3, 256, 21)
    for top_k in (0, 1025):
        with pytest.raises(hg.HyperGenError) as ei:
            ctx.search_dev(*ok, top_k, 0.0, 0, out.data_ptr(), nf.data_ptr())
        assert ei.value.code == hg.ffi.HG_E_INVALID
    bad_args = [
        (None, n.data_ptr(), 300, d.data_ptr(), n.data_ptr(), 3, 256, 21, 4, 0.0, 0, out.data_ptr(), nf.data_ptr()),
        (d.data_ptr(), n.data_ptr(), 300, d.data_ptr(), None, 3, 256, 21, 4, 0.0, 0, out.data_ptr(), nf.data_ptr()),
        (*ok, 4, 0.0, 0, None, nf.data_ptr()),
        (*ok, 4, 0.0, 0, out.data_ptr(), None),
        (d.data_ptr(), n.data_ptr(), 300, d.data_ptr(), n.data_ptr(), 3, 320, 21, 4, 0.0, 0, out.data_ptr(), nf.data_ptr()),
    ]
    for args in bad_args:
        with pytest.raises(hg.HyperGenError) as ei:
            ctx.search_dev(*args)
        assert ei.value.code == hg.ffi.HG_E_INVALID
    # no refs: HG_OK, nothing found
    nf.fill_(9)
    ctx.search_dev(d.data_ptr(), n.data_ptr(), 0, d.data_ptr(), n.data_ptr(), 3, 256, 21, 4, 0.0, 0, out.data_ptr(), nf.data_ptr())
    assert not nf.cpu().numpy()[:3].any()
