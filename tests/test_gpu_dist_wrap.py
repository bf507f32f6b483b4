"""Dist where the reference's i32 norms, dots and denominators wrap (dist.rs:147-160): rows whose true norms sum x^2 run
from 2^28 to 2^33, so pairs sit on both sides of ceil(2^31 / 3), 2^31 and 2^32.  There an anti-correlated pair (dot < 0)
can get a wrapped denominator den < 0 and a high ANI, and a pair with den > 0 can have J = dot / den <= -1, which the
reference scores 100.  Every dist entry and every kernel must report exactly the pairs the oracle scores >= ani_th, with
every dot and every ANI bit; search, cluster and derep must see the same pairs.

Each data set asserts its own coverage, so that the cases cannot drift back into the regime where nothing wraps."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_cluster import _expected as _components_of  # noqa: E402
from test_gpu_derep import _full, _greedy  # noqa: E402
from test_gpu_search import _compare, _expected as _search_expected, _search_dev  # noqa: E402

pytestmark = pytest.mark.gpu

AUTO, SIMT, TWO_LIMB, NARROW = 0, 1, 2, 3
CUT = 715827883  # ceil(2^31 / 3)


def _i32(x):
    return ((np.asarray(x, np.int64) + 2**31) % 2**32 - 2**31).astype(np.int64)


def _true_norms(hv):
    h = hv.astype(np.int64)
    return (h * h).sum(1)


def _pm1(rng, D):
    return rng.choice(np.array([-1, 1], np.int64), D)


def _exact_anti(rng, D, c):
    """r = c B and q = -c B: dot = -N exactly, both true norms N = D c^2"""
    r = c * _pm1(rng, D)
    return [r, -r]


def _fam_rows(seed, D=1024):
    """families sigma c B_f + noise (|x| <= 8127): norms 2^28 .. 2^33, co- and anti-correlated members, a few noise levels;
    plus exact anti pairs just below / above the cut and one with den > 0 and J <= -1"""
    rng = np.random.default_rng(seed)
    rows = []
    targets = [2**28, 4e8, 6.5e8, 7.3e8, 9e8, 1.1e9, 1.3e9, 1.6e9, 1.9e9, 2.1e9, 2.6e9, 3.5e9, 4.4e9, 6e9, 8.6e9]
    fracs = [0.03, 0.2, 0.45, 0.7, 1.2]
    for t, N in enumerate(targets):
        c = np.sqrt(N / D)
        B = _pm1(rng, D)
        for k in range(16):
            s = 1 if k % 2 == 0 else -1
            ck = c * (1 + rng.uniform(-0.01, 0.01))
            w = max(1, int(c * fracs[(t + k // 2) % len(fracs)]))
            rows.append(np.clip(np.rint(s * ck * B) + rng.integers(-w, w + 1, D), -8127, 8127))
    rows += _exact_anti(rng, D, 836)   # 1024 * 836^2 = 715 669 504: just below the cut, scores 0
    rows += _exact_anti(rng, D, 837)   # just above: den wraps negative, ANI ~96.7
    rows += _exact_anti(rng, D, 1300)  # N = 1.73e9: den = 3N - 2^32 > 0, J < -1, ANI 100
    hv = np.stack(rows).astype(np.int16)
    return hv[np.random.default_rng(seed + 1).permutation(hv.shape[0])]


def _narrow_rows(seed, D, cs, below, above):
    """sketch-like rows for the single s8 plane: one parity per row, every element within [s - 256, s + 254]"""
    rng = np.random.default_rng(seed)
    rows = []
    for c in cs:
        B = _pm1(rng, D)
        for k in range(40):
            s = 1 if k % 2 == 0 else -1
            rows.append(s * c * B + 2 * rng.integers(-3, 4, D))
    for c in (below, above):
        rows += _exact_anti(rng, D, c)
    hv = np.stack(rows).astype(np.int16)
    return hv[np.random.default_rng(seed + 1).permutation(hv.shape[0])]


def _outlier_rows(seed, D=4096):
    """|x| <= ~60 (one parity per row) plus 0, 1 or 2 far elements in shared dimensions that push the norm past the cut;
    the far elements stay within the single plane's outlier budget"""
    rng = np.random.default_rng(seed)
    rows = []
    for f in range(16):
        T = 2 * rng.integers(-29, 30, D)
        n_out = f % 3
        far = 2 * rng.integers(13000, 15000, 2)
        for k in range(14):
            s = 1 if k % 2 == 0 else -1
            p = k // 2 % 2
            r = s * T + 2 * rng.integers(-2, 3, D) + p
            for o in range(n_out):
                r[o] = s * far[o] + p
            rows.append(r)
    # an exact anti pair whose norms are just below the cut (one far element, odd parity)
    r = 2 * rng.integers(-29, 30, D) + 1
    base = int((r[1:] ** 2).sum())
    v = int(np.sqrt(CUT - 1 - base))
    v -= 1 - v % 2
    r[0] = v
    assert CUT - 200_000 < int((r ** 2).sum()) < CUT
    rows += [r, -r]
    hv = np.stack(rows).astype(np.int16)
    return hv[np.random.default_rng(seed + 1).permutation(hv.shape[0])]


def _wide_rows(seed):
    hv = _fam_rows(seed).copy()
    hv[::37, 5] = 9000  # above HG_LIMB_MAX_ABS: the limb split cannot take these rows
    return hv


SETS = {
    "fam1024": (lambda: _fam_rows(11), [SIMT, TWO_LIMB, AUTO], TWO_LIMB),
    "wide1024": (lambda: _wide_rows(12), [SIMT, AUTO], SIMT),
    "narrow16384": (lambda: _narrow_rows(13, 16384, [90, 150, 200, 212, 226, 240], 209, 210), [SIMT, TWO_LIMB, NARROW, AUTO], NARROW),
    "narrow32768": (lambda: _narrow_rows(14, 32768, [90, 140, 160, 200, 230, 240], 147, 148), [TWO_LIMB, NARROW, AUTO], NARROW),
    "outliers4096": (lambda: _outlier_rows(15), [SIMT, NARROW, AUTO], NARROW),
}
# J <= -1 with den > 0 needs true norms in (2^32 / 3, 2^31): rows of |x| <= 250 at D 16384 cannot get there
NO_J_LE_M1 = {"narrow16384"}


class _Set:
    def __init__(self, name, oracle):
        self.name = name
        self.hv = SETS[name][0]()
        self.norm = np.array([oracle.hv_l2_norm_sq(v) for v in self.hv], np.int32)
        self.sq = _true_norms(self.hv)
        n = self.hv.shape[0]
        self.nq = n // 3  # ref x query: every row against the first third
        self.sym = oracle.dist_all(self.hv, self.norm, self.hv, self.norm, symmetric=True)
        self.rxq = oracle.dist_all(self.hv, self.norm, self.hv[: self.nq], self.norm[: self.nq])

    def pairs(self, symmetric):
        n = self.hv.shape[0]
        if symmetric:
            i, j = np.triu_indices(n, 1)
        else:
            i, j = np.divmod(np.arange(n * self.nq), self.nq)
        return i, j


_cache = {}


def _set(name, oracle):
    if name not in _cache:
        _cache[name] = _Set(name, oracle)
        _check_coverage(_cache[name])
    return _cache[name]


def _check_coverage(s):
    ani, dot = s.sym
    i, j = s.pairs(True)
    dot = dot.astype(np.int64)
    den = _i32(s.norm[i].astype(np.int64) + s.norm[j] - dot)
    hit = ani >= np.float32(85.0)
    wrapped = hit & (dot < 0) & (den < 0)
    assert wrapped.any(), s.name
    le_m1 = hit & (den > 0) & (dot.astype(np.float32) <= -den.astype(np.float32))
    assert le_m1.any() == (s.name not in NO_J_LE_M1), s.name
    if le_m1.any():
        assert (ani[le_m1] == np.float32(100.0)).all()
    below = (s.sq[i] < CUT) & (s.sq[j] < CUT) & (s.sq[i] > CUT - 10_000_000) & (s.sq[j] > CUT - 10_000_000) & (dot < 0)
    assert below.any() and (ani[below] == 0).all(), s.name
    # the pairs on both sides of 2^31 and 2^32
    tot = s.sq[i] + s.sq[j]
    for lo, hi in ((CUT, 2**31), (2**31, 2**32), (2**32, 2**35)):
        if tot.max() >= hi or lo == CUT:
            assert (hit & (tot >= lo) & (tot < hi)).any(), (s.name, lo)


def _check(hits, s, symmetric, th, i0=0):
    ani, dot = s.sym if symmetric else s.rxq
    Q = s.hv.shape[0] if symmetric else s.nq
    i, j = hits["i"].astype(np.int64) - i0, hits["j"].astype(np.int64)
    idx = i * (Q - 1) - i * (i - 1) // 2 + (j - i - 1) if symmetric else i * Q + j
    want = np.nonzero(ani >= np.float32(th))[0]
    assert want.size > 0
    assert np.array_equal(np.sort(idx), want), (len(idx), len(want), np.setdiff1d(want, idx)[:8])
    assert np.array_equal(hits["dot"], dot[idx])
    assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))


def _dist_dev(ctx, hg, s, symmetric, th, path):
    import torch
    D = s.hv.shape[1]
    n = s.hv.shape[0]
    nq = n if symmetric else s.nq
    d_hv, d_n = torch.from_numpy(s.hv).cuda(), torch.from_numpy(s.norm).cuda()
    cap = n * nq
    d_hits = torch.empty(cap * 16, dtype=torch.uint8, device="cuda")
    d_cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    ctx.dist_dev(d_hv.data_ptr(), d_n.data_ptr(), n, 0, d_hv.data_ptr(), d_n.data_ptr(), nq, 0, D, 21, th, symmetric, path,
                 d_hits.data_ptr(), cap, d_cnt.data_ptr())
    ctx.sync()
    if path == NARROW:
        ctx.dist_status()  # the single plane took these rows
    cnt = int(d_cnt.item())
    return np.frombuffer(d_hits.cpu().numpy().tobytes(), dtype=hg.ffi.HIT_DTYPE)[:cnt].copy()


CASES = [(name, p) for name, (_, paths, _) in SETS.items() for p in paths]


@pytest.mark.parametrize("th", [85.0, 95.0, 99.5])
@pytest.mark.parametrize("symmetric", [True, False], ids=["sym", "rxq"])
@pytest.mark.parametrize("name,path", CASES, ids=["%s-%d" % c for c in CASES])
def test_dist_dev_every_kernel(ctx, hg, oracle, name, path, symmetric, th):
    s = _set(name, oracle)
    hits = _dist_dev(ctx, hg, s, symmetric, th, path)
    assert ctx.dist_last_path == (SETS[name][2] if path == AUTO else path), ctx.dist_last_reason
    _check(hits, s, symmetric, th)


def _packed(oracle, hv):
    rows = [oracle.compress_hd_sketch(v) for v in hv]
    w = max(p.size for _, p in rows)
    packed = np.zeros((hv.shape[0], w), np.uint8)
    for g, (_, p) in enumerate(rows):
        packed[g, : p.size] = p
    return packed, np.array([b for b, _ in rows], np.uint8)


@pytest.mark.parametrize("chunked", [False, True], ids=["whole", "chunks256"])
@pytest.mark.parametrize("name", ["fam1024", "narrow16384"])
def test_dist_packed(ctx, hg, oracle, monkeypatch, name, chunked):
    if chunked:
        monkeypatch.setenv("HG_DIST_CHUNK_ROWS", "256")
    s = _set(name, oracle)
    packed, bits = _packed(oracle, s.hv)
    assert bits.max() <= 15
    n, D = s.hv.shape
    hits, milli = ctx.dist_packed(packed, bits, s.norm, packed, bits, s.norm, D, ani_th=85.0, symmetric=True, cap=n * n)
    _check(hits, s, True, 85.0)
    # in the reference's output order
    ani = s.sym[0]
    order = oracle.ani_output_order(ani, 85.0)
    i, j = s.pairs(True)
    assert np.array_equal(hits["i"], i[order]) and np.array_equal(hits["j"], j[order])


@pytest.mark.parametrize("name,path", [("fam1024", TWO_LIMB), ("narrow16384", NARROW), ("outliers4096", NARROW)])
def test_dist_sorted_host_rows(ctx, hg, oracle, name, path):
    s = _set(name, oracle)
    n = s.hv.shape[0]
    hits, milli = ctx.dist(s.hv, s.norm, s.hv, s.norm, ani_th=95.0, symmetric=True, path=path, cap=n * n, sorted_output=True,
                           want_milli=True)
    assert ctx.dist_last_path == path
    _check(hits, s, True, 95.0)
    order = oracle.ani_output_order(s.sym[0], 95.0)
    i, j = s.pairs(True)
    assert np.array_equal(hits["i"], i[order]) and np.array_equal(hits["j"], j[order])


@pytest.mark.parametrize("top_k", [1, 16])
@pytest.mark.parametrize("name,path", [("fam1024", SIMT), ("fam1024", TWO_LIMB), ("narrow16384", NARROW), ("outliers4096", NARROW)])
def test_search(ctx, hg, oracle, name, path, top_k):
    s = _set(name, oracle)
    q = s.hv[: s.nq]
    qn = s.norm[: s.nq]
    got = _search_dev(ctx, hg, s.hv, s.norm, q, qn, top_k, ani_min=85.0, path=path)
    want = _search_expected(oracle, s.hv, s.norm, q, qn, top_k, 85.0)
    assert (want[3] > 0).any()
    _compare(got, want)


def _dev(t):
    import torch
    return torch.from_numpy(np.ascontiguousarray(t)).cuda()


@pytest.mark.parametrize("th", [85.0, 99.5])
@pytest.mark.parametrize("name,path", [("fam1024", SIMT), ("fam1024", TWO_LIMB), ("narrow16384", NARROW), ("outliers4096", NARROW)])
def test_cluster(ctx, hg, oracle, name, path, th):
    import torch
    s = _set(name, oracle)
    n, D = s.hv.shape
    want = _components_of(n, s.sym[0], th)
    d_hv, d_n = _dev(s.hv), _dev(s.norm)
    d_rep = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    k = ctx.cluster_dev(d_hv.data_ptr(), d_n.data_ptr(), n, D, 21, th, path, d_rep.data_ptr())
    assert k == want[1]
    assert np.array_equal(d_rep.cpu().numpy().view(np.uint32), want[0])


@pytest.mark.parametrize("th", [85.0, 99.5])
@pytest.mark.parametrize("name,path", [("fam1024", SIMT), ("fam1024", TWO_LIMB), ("narrow16384", NARROW), ("outliers4096", NARROW)])
def test_derep(ctx, hg, oracle, name, path, th):
    import torch
    s = _set(name, oracle)
    n, D = s.hv.shape
    want = _greedy(_full(n, s.sym[0]), th)
    d_hv, d_n = _dev(s.hv), _dev(s.norm)
    d_rep = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    k = ctx.derep_dev(d_hv.data_ptr(), d_n.data_ptr(), n, D, 21, th, path, d_rep.data_ptr())
    assert k == want[1]
    assert np.array_equal(d_rep.cpu().numpy().view(np.uint32), want[0])


@pytest.mark.parametrize("symmetric", [True, False], ids=["sym", "rxq"])
@pytest.mark.parametrize("name,path", [("fam1024", TWO_LIMB), ("narrow16384", NARROW), ("outliers4096", NARROW)])
def test_world1_sharded(ctx, hg, oracle, name, path, symmetric):
    s = _set(name, oracle)
    n, D = s.hv.shape
    cap = n * n
    peer = hg.Peer(ctx, 0, 1, hg.ffi.peer_window_need(n, D, cap))
    try:
        d_hv, d_n = _dev(s.hv), _dev(s.norm)
        if symmetric:
            peer.dist_sharded_dev(None, None, 0, 0, d_hv.data_ptr(), d_n.data_ptr(), [0, n], D, 21, 85.0, True, path, 0, cap)
            hits, _ = peer.dist_sharded_hits(cap)
            _check(hits, s, True, 85.0)
        else:
            # every row as a ref against the first third as the gathered query matrix
            dq, dqn = _dev(s.hv[: s.nq]), _dev(s.norm[: s.nq])
            peer.dist_sharded_dev(d_hv.data_ptr(), d_n.data_ptr(), n, 0, dq.data_ptr(), dqn.data_ptr(), [0, s.nq], D, 21, 85.0,
                                  False, path, 0, cap)
            hits, _ = peer.dist_sharded_hits(cap)
            _check(hits, s, False, 85.0)
        assert ctx.dist_last_path == path
    finally:
        peer.close()


def _sketch_like(seed, n, D, spread=110):
    """rows shaped like sketch HVs (one parity per row, centred near 0, half the elements negative): true norms of a
    few 1e7 to 1e8, far below the cut"""
    rng = np.random.default_rng(seed)
    par = rng.integers(0, 2, (n, 1))
    return (2 * np.clip(np.rint(rng.normal(0, spread / 3, (n, D))), -spread, spread).astype(np.int64) + par).astype(np.int16)


def _norm_flags(ctx, hv, path):
    import torch
    n, D = hv.shape
    d_hv = _dev(hv)
    d_f = torch.full((n,), 7, dtype=torch.int32, device="cuda")  # garbage: every row must be written
    torch.cuda.synchronize()
    ctx.dist_norm_flags(d_hv.data_ptr(), n, D, path, d_f.data_ptr())
    return d_f.cpu().numpy()


FLAG_CASES = [(name, p) for name in ["fam1024", "narrow16384", "narrow32768", "outliers4096"] for p in SETS[name][1] if p in (TWO_LIMB, NARROW)]
FLAG_CASES += [("sketch%d" % D, p) for D in (4096, 8192, 16384, 32768) for p in (TWO_LIMB, NARROW)]


@pytest.mark.parametrize("name,path", FLAG_CASES, ids=["%s-%d" % c for c in FLAG_CASES])
def test_norm_flags_are_exactly_the_rows_at_or_above_the_cut(ctx, hg, oracle, name, path):
    """the row preparation of each tensor kernel flags a row exactly when its true norm sum x^2 reaches the cut: never
    a sketch-sized row (the flag costs the kernel its candidate bound), always one whose i32 arithmetic may wrap"""
    hv = _sketch_like(20, 300, int(name[6:])) if name.startswith("sketch") else _set(name, oracle).hv
    sq = _true_norms(hv)
    flags = _norm_flags(ctx, hv, path)
    assert np.array_equal(flags, (sq >= CUT).astype(np.int32)), (np.flatnonzero(flags != (sq >= CUT))[:8], sq.min(), sq.max())
    if name.startswith("sketch"):
        assert sq.max() < CUT // 3 and not flags.any()
    else:
        assert flags.any() and not flags.all()
