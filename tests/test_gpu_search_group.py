"""Top-k search over ref blocks: hg_search_merge_dev over per-block hg_search_dev results, and hg_group_search_packed
(Group.search_packed, search.search(group=...), `hyper-gen search` over every GPU) against the oracle and against the
search over all refs on one context.

The group cases run on any box with two or three contexts on GPU 0 (Group(ordinals=[0, 0])): the same blocks, gather and
merge as on several GPUs.  The cases over every GPU of the box skip when fewer than two are visible."""
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_search import _compare, _correlated_rows, _expected, _family, _norms, _search_dev, _sketch_file  # noqa: E402

pytestmark = pytest.mark.gpu

TWO_LIMB = 2


def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.fixture(scope="module")
def fam(ctx):
    """as in test_gpu_search: 3000 refs, 300 queries (the last 27 novel), D 4096"""
    hv, norm, packed, bits = _family(ctx, 3300, 4096)
    sel = np.arange(0, 3300, 11)[:300]
    return (hv[:3000], norm[:3000], packed[:3000], bits[:3000]), (hv[sel], norm[sel], packed[sel], bits[sel])


def _blocks_then_merge(ctx, hg, r, rn, q, qn, bounds, top_k, ani_min=0.0):
    """hg_search_dev on every ref block [bounds[m], bounds[m + 1]) into one buffer of lists, then hg_search_merge_dev"""
    import torch
    R, D = r.shape
    Q, M = q.shape[0], len(bounds) - 1
    d_r, d_rn = torch.from_numpy(np.ascontiguousarray(r)).cuda(), torch.from_numpy(np.ascontiguousarray(rn)).cuda()
    d_q, d_qn = torch.from_numpy(np.ascontiguousarray(q)).cuda(), torch.from_numpy(np.ascontiguousarray(qn)).cuda()
    d_in = torch.full((M * Q * top_k * 16,), 0xCD, dtype=torch.uint8, device="cuda")
    d_found = torch.zeros(M * Q, dtype=torch.int32, device="cuda")
    for m in range(M):
        b0, b1 = bounds[m], bounds[m + 1]
        ctx.search_dev(d_r.data_ptr() + b0 * D * 2, d_rn.data_ptr() + b0 * 4, b1 - b0, d_q.data_ptr(), d_qn.data_ptr(), Q, D, 21,
                       top_k, ani_min, 0, d_in.data_ptr() + m * Q * top_k * 16, d_found.data_ptr() + m * Q * 4)
    d_out = torch.full((Q * top_k * 16,), 0xAB, dtype=torch.uint8, device="cuda")  # garbage: the unused slots must be zeroed
    d_nf = torch.full((Q,), 9, dtype=torch.int32, device="cuda")
    d_mi = torch.full((Q * top_k,), 7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.search_merge_dev(M, d_in.data_ptr(), d_found.data_ptr(), bounds[:-1], Q, top_k, d_out.data_ptr(), d_nf.data_ptr(),
                         d_mi.data_ptr())
    hits = np.frombuffer(d_out.cpu().numpy().tobytes(), dtype=hg.ffi.HIT_DTYPE).reshape(Q, top_k).copy()
    return hits, d_nf.cpu().numpy().view(np.uint32).copy(), d_mi.cpu().numpy().view(np.uint32).reshape(Q, top_k).copy()


def _same(a, b):
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


SPLITS = {
    "2": [0, 1234, 3000],
    "3": [0, 40, 1900, 3000],
    "8": [0, 0, 5, 6, 700, 1500, 2222, 2990, 3000],  # an empty block, blocks of 5, 1 and 10 refs
}


@pytest.mark.parametrize("top_k", [1, 10, 64])
@pytest.mark.parametrize("split", sorted(SPLITS))
def test_merge_of_family_blocks_equals_one_search(ctx, hg, oracle, fam, split, top_k):
    (r, rn, _, _), (q, qn, _, _) = fam
    got = _blocks_then_merge(ctx, hg, r, rn, q, qn, SPLITS[split], top_k)
    _compare(got, _expected(oracle, r, rn, q, qn, top_k, 0.0))
    _same(got, _search_dev(ctx, hg, r, rn, q, qn, top_k))


def test_top_k_1024_eight_lists_ani_0_ties_by_global_index(ctx, hg, oracle, fam):
    """1500 refs: a novel query has ANI > 0 with about half of them (positive dot), so of its 1024 results the last few
    hundred are ANI-0 ties, taken by lowest global index from several blocks"""
    (r, rn, _, _), (q, qn, _, _) = fam
    r, rn = r[:1500], rn[:1500]
    bounds = [0, 0, 5, 6, 100, 600, 1000, 1400, 1500]
    want = _expected(oracle, r, rn, q, qn, 1024, 0.0)
    ei, _, ea, nf = want
    novel = np.arange(273, 300)
    assert (nf[novel] == 1024).all()
    for j in novel:
        tail = ei[j][ea[j] == 0]
        assert tail.size and np.array_equal(tail, np.sort(tail))
        assert len(set(np.searchsorted(bounds, tail, side="right"))) >= 2  # the tied tail comes from several blocks
    got = _blocks_then_merge(ctx, hg, r, rn, q, qn, bounds, 1024)
    _compare(got, want)
    _same(got, _search_dev(ctx, hg, r, rn, q, qn, 1024))


@pytest.mark.parametrize("top_k", [8, 1024])
def test_tied_copies_over_blocks_decide_the_kth_place_by_index(ctx, hg, oracle, top_k):
    """2100 copies of one sketch among 6000 refs (as test_gpu_search), the blocks cut between the copies so that the
    copies a query takes, and the one at its top_k-th place, come from several blocks"""
    hv, norm, _, _ = _family(ctx, 6016, 1024, n_per=1000, first=700)
    r, rn = hv[:6000].copy(), norm[:6000].copy()
    dup = np.sort(np.random.default_rng(5).choice(6000, 2100, replace=False))
    r[dup], rn[dup] = hv[6000], norm[6000]
    q, qn = hv[6000:], norm[6000:]
    bounds = [0, int(dup[3]) + 1, int(dup[5]) + 1, 3000, 3001, 6000]
    want = _expected(oracle, r, rn, q, qn, top_k, 0.0)
    assert np.array_equal(want[0][0], dup[:top_k])
    assert len(set(np.searchsorted(bounds, dup[:top_k], side="right"))) >= 3
    got = _blocks_then_merge(ctx, hg, r, rn, q, qn, bounds, top_k)
    _compare(got, want)


def test_ani_min_above_some_queries_best_in_every_block(ctx, hg, oracle, fam):
    (r, rn, _, _), (q, qn, _, _) = fam
    want = _expected(oracle, r, rn, q, qn, 10, 97.0)
    assert (want[3] == 0).any() and (want[3] < 10).any()
    _compare(_blocks_then_merge(ctx, hg, r, rn, q, qn, SPLITS["3"], 10, 97.0), want)


def test_merge_argument_errors(ctx, hg):
    import torch
    Q, K = 4, 3
    d_in = torch.zeros(2 * Q * K * 4, dtype=torch.int32, device="cuda")
    d_found = torch.zeros(2 * Q, dtype=torch.int32, device="cuda")
    d_out = torch.zeros(Q * K * 4, dtype=torch.int32, device="cuda")
    d_nf = torch.zeros(Q, dtype=torch.int32, device="cuda")

    def merge(n_lists, top_k, i0):
        ctx.search_merge_dev(n_lists, d_in.data_ptr(), d_found.data_ptr(), i0, Q, top_k, d_out.data_ptr(), d_nf.data_ptr())

    for n_lists, top_k in ((0, K), (65, K), (2, 0), (2, 1025)):
        with pytest.raises(hg.HyperGenError) as ei:
            merge(n_lists, top_k, [0] * n_lists)
        assert ei.value.code == hg.ffi.HG_E_INVALID
    merge(2, K, [0, 100])  # nothing found anywhere: valid
    assert not d_nf.cpu().numpy().any()
    # list 1, query 0: one record with i = 1 in a block that starts at 2^32 - 1: i + i0 wraps
    d_in.view(Q * 2, K, 4)[Q, 0] = torch.tensor([1, 0, 5, 0], dtype=torch.int32)
    d_found[Q] = 1
    with pytest.raises(hg.HyperGenError, match="32 bits") as ei:
        merge(2, K, [0, 0xFFFFFFFF])
    assert ei.value.code == hg.ffi.HG_E_INVALID
    merge(2, K, [0, 0xFFFFFFFE])  # the largest index that fits
    assert d_nf.cpu().numpy()[0] == 1 and d_out.view(Q, K, 4)[0, 0, 0].item() == -1
    d_found[0] = K + 1  # more records than top_k
    with pytest.raises(hg.HyperGenError, match="exceeds top_k") as ei:
        merge(2, K, [0, 100])
    assert ei.value.code == hg.ffi.HG_E_INVALID


# ---- hg_group_search_packed ------------------------------------------------------------------------------------------

def test_group_of_two_contexts_on_gpu0_equals_one_context(ctx, hg, oracle, fam):
    (r, rn, rp, rb), (q, qn, qp, qb) = fam
    with hg.Group(ordinals=[0, 0]) as g:
        got = g.search_packed(rp, rb, rn, qp, qb, qn, 4096, top_k=10)
        assert g.search_stats(0)[0][0] > 0 and g.search_stats(1)[0][0] > 0  # both members searched a block
    _compare(got, _expected(oracle, r, rn, q, qn, 10, 0.0))
    _same(got, ctx.search_packed(rp, rb, rn, qp, qb, qn, 4096, top_k=10))


def test_group_12_bit_rows_run_two_limb(ctx, hg, oracle):
    rng = np.random.default_rng(23)
    hv = _correlated_rows(rng, 2600, 1024, 8, 1500, 40, 2000)
    norm = _norms(oracle, hv)
    rows = [oracle.compress_hd_sketch(v) for v in hv]
    assert all(b == 12 for b, _ in rows)
    packed, bits = np.stack([p for _, p in rows]), np.full(hv.shape[0], 12, np.uint8)
    r, q = slice(0, 2300), slice(2250, 2600)
    args = (packed[r], bits[r], norm[r], packed[q], bits[q], norm[q], 1024)
    with hg.Group(ordinals=[0, 0]) as g:
        got = g.search_packed(*args, top_k=12)
        assert g.dist_last_path(0) == TWO_LIMB and g.dist_last_path(1) == TWO_LIMB
    _compare(got, _expected(oracle, hv[r], norm[r], hv[q], norm[q], 12, 0.0))
    _same(got, ctx.search_packed(*args, top_k=12))


def test_group_self_search(ctx, hg, oracle, fam):
    (r, rn, rp, rb), _ = fam
    r, rn, rp, rb = r[:2100], rn[:2100], rp[:2100], rb[:2100]
    with hg.Group(ordinals=[0, 0]) as g:
        got = g.search_packed(rp, rb, rn, rp, rb, rn, 4096, top_k=10)
    _compare(got, _expected(oracle, r, rn, r, rn, 10, 0.0))


@pytest.mark.parametrize("n_ref,used", [(2500, 2), (1500, 1)])
def test_group_uses_only_members_with_1024_refs(ctx, hg, oracle, fam, n_ref, used):
    (r, rn, rp, rb), (q, qn, qp, qb) = fam
    r, rn, rp, rb = r[:n_ref], rn[:n_ref], rp[:n_ref], rb[:n_ref]
    with hg.Group(ordinals=[0, 0, 0]) as g:
        got = g.search_packed(rp, rb, rn, qp, qb, qn, 4096, top_k=10)
        ran = [g.search_stats(m)[0][0] > 0 for m in range(3)]
    assert ran == [m < used for m in range(3)]
    _compare(got, _expected(oracle, r, rn, q, qn, 10, 0.0))


# ---- every GPU of the box --------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def many(ctx):
    """8448 refs (a block of at least 1024 for each of up to 8 GPUs) and 150 queries, D 4096"""
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    hv, norm, packed, bits = _family(ctx, 8600, 4096)
    sel = np.arange(5, 8600, 57)[:150]
    return (hv[:8448], norm[:8448], packed[:8448], bits[:8448]), (hv[sel], norm[sel], packed[sel], bits[sel])


def test_group_all_gpus_equals_one_gpu(ctx, hg, oracle, many):
    (r, rn, rp, rb), (q, qn, qp, qb) = many
    with hg.Group() as g:
        assert g.size == min(_n_gpus(), 8)
        got = g.search_packed(rp, rb, rn, qp, qb, qn, 4096, top_k=10)
        assert all(g.search_stats(m)[0][0] > 0 for m in range(g.size))
    _compare(got, _expected(oracle, r, rn, q, qn, 10, 0.0))
    _same(got, ctx.search_packed(rp, rb, rn, qp, qb, qn, 4096, top_k=10))


def test_cli_and_python_all_gpus_write_the_same_bytes_as_one_gpu(ctx, hg, many, tmp_path):
    from hypergen_b200 import _build, fileio, search
    exe = _build.build_host()
    (r, rn, rp, rb), (q, qn, qp, qb) = many
    ref_f, qry_f = str(tmp_path / "ref.sketch"), str(tmp_path / "qry.sketch")
    _sketch_file(fileio, ref_f, rp, rb, rn, ["ref/g%05d.fna" % g for g in range(r.shape[0])])
    _sketch_file(fileio, qry_f, qp, qb, qn, ["qry/q%03d.fna" % g for g in range(q.shape[0])])
    outs = {}
    for name, env in (("one", dict(os.environ, HG_GPUS="1")), ("all", dict(os.environ))):
        tsv = str(tmp_path / (name + ".tsv"))
        p = subprocess.run([exe, "search", "-r", ref_f, "-q", qry_f, "-o", tsv, "-n", "10", "-a", "1.0"], env=env,
                           capture_output=True, text=True, check=True)
        outs[name] = (open(tsv, "rb").read(), p.stdout.replace(tsv, "OUT"))
    assert outs["one"] == outs["all"] and outs["one"][0]
    with hg.Group() as g:
        py = search.search(search.SketchSearch(ref_f, qry_f, str(tmp_path / "py.tsv"), top_k=10, ani_min=1.0), group=g)
    assert py.encode() == outs["one"][0] == open(tmp_path / "py.tsv", "rb").read()
