"""The dist kernels' candidate pre-filters (csrc/dist_common.cuh, dist_tc.cu, dist_narrow.cu), restated in numpy f32 and
checked against the oracle's ani_from_dot (dist.rs:153-160): neither may reject a (dot, norm_r, norm_q) that the reference
scores >= ani_th, including where the i32 denominator norm_r + norm_q - dot wraps.  CPU only; the kernels themselves are
checked in tests/test_gpu_dist_wrap.py."""
import math

import numpy as np
import pytest

CUT = 715827883  # HG_NORM_WRAP_CUT = ceil(2^31 / 3)
I32_MIN = -(2**31)
THS = [0.5, 85.0, 95.0, 99.5]


def _w(v):
    return ((np.asarray(v, np.int64) + 2**31) % 2**32) - 2**31


def _jmin(ani_th, k=21):
    """dist_jmin"""
    a = ani_th / 100.0 - 1e-4
    if not a > 0.0:
        return np.float32(0.0)
    if a >= 1.0:
        return np.float32(1e30)
    E = math.exp(k * (a - 1.0))
    return np.float32(E / (2.0 - E) * (1.0 - 1e-3))


def _cfrac(jmin):
    return np.float32(float(jmin) / (1.0 + float(jmin))) if jmin > 0 else np.float32(0.0)


def exact_stage(dot, nr, nq, jmin):
    """dist_emit / dist_eval: den <= 0, or fl(dot) >= jmin fl(den), or fl(dot) <= -fl(den) (J <= -1)"""
    den = _w(np.asarray(nr, np.int64) + nq - dot)
    fd, fn = np.asarray(dot).astype(np.float32), den.astype(np.float32)
    return (den <= 0) | (fd >= jmin * fn) | (fd <= -fn)


def _rz(n):
    """__int2float_rz"""
    f = np.asarray(n).astype(np.float32)
    over = np.abs(f.astype(np.float64)) > np.abs(np.asarray(n, np.float64))
    return np.where(over, np.nextafter(f, np.float32(0)), f)


def _side_bound(n, cfrac, big, always):
    """tc_row_bound / tc_col_bound (and the narrow constants without outliers): always for a row at or above the cut"""
    b = np.floor((cfrac * _rz(n)).astype(np.float64)).astype(np.int64) - 1
    return np.where((cfrac > 0) & ~big & (np.asarray(n) > 0), b, always)


def tensor_bound(dot, nr, nq, sq_r, sq_q, cfrac):
    """tc_drain / n1_drain's per-element test: dot >= tr + tq (wrapping), or either side always a candidate"""
    tr = _side_bound(nr, cfrac, np.asarray(sq_r) >= CUT, I32_MIN // 2)
    tq = _side_bound(nq, cfrac, np.asarray(sq_q) >= CUT, I32_MIN)
    return (np.asarray(dot) >= _w(tr + tq)) | (tq == I32_MIN) | (tr == I32_MIN // 2)


def _accepted(oracle, dot, nr, nq, th):
    return np.array([oracle.ani_from_dot(int(d), int(a), int(b)) >= np.float32(th) for d, a, b in zip(dot, nr, nq)])


def _adversarial(rng, n):
    """i32 triples: uniform, den = 0, INT32_MIN anywhere, and fl(dot) = -fl(den) and its neighbours 1 ulp either side"""
    i32 = lambda size: rng.integers(I32_MIN, 2**31, size)
    out = [np.stack([i32(n), i32(n), i32(n)], 1)]
    nr, dot = i32(n), i32(n)
    out.append(np.stack([dot, nr, _w(dot - nr)], 1))  # den = 0
    t = np.stack([i32(n), i32(n), i32(n)], 1)
    t[np.arange(n), rng.integers(0, 3, n)] = I32_MIN
    out.append(t)
    den = rng.integers(2**24, 2**31, n)
    for step in (-1, 0, 1):
        fd = -den.astype(np.float32)
        if step:
            fd = np.nextafter(fd, np.float32(step * np.inf))
        d = fd.astype(np.int64)
        ok = (d >= I32_MIN) & (d < 2**31)
        d, dn = d[ok], den[ok]
        a = i32(d.size)
        b = _w(dn + d - a)  # nr + nq - dot = den (mod 2^32)
        assert (_w(a + b - d) == dn).all()
        out.append(np.stack([d, a, b], 1))
    return np.concatenate(out)


@pytest.mark.parametrize("th", THS)
def test_exact_stage_never_rejects_an_accepted_triple(oracle, th):
    rng = np.random.default_rng(int(th * 10))
    t = _adversarial(rng, 4000)
    dot, nr, nq = t[:, 0], t[:, 1], t[:, 2]
    acc = _accepted(oracle, dot, nr, nq, th)
    cand = exact_stage(dot, nr, nq, _jmin(th))
    assert not (acc & ~cand).any(), t[acc & ~cand][:5]
    assert acc.any() and (~cand).any()  # the filter does reject triples, and not only those


def test_j_le_minus_one_is_the_case_the_old_exact_stage_missed(oracle):
    """den > 0 and fl(dot) <= -fl(den): the reference says 100; without the third clause these were dropped"""
    den = np.array([1161220096, 1726152704, 2**24, 2**31 - 1], np.int64)
    dot = (-den.astype(np.float32)).astype(np.int64)
    dot = np.maximum(dot, I32_MIN)
    nr = np.array([1_000_000_000, 2_000_000_000, 5, 7], np.int64)
    nq = _w(den + dot - nr)
    jm = _jmin(85.0)
    for d, a, b in zip(dot, nr, nq):
        assert oracle.ani_from_dot(int(d), int(a), int(b)) == np.float32(100.0)
    old = (_w(nr + nq - dot) <= 0) | (dot.astype(np.float32) >= jm * _w(nr + nq - dot).astype(np.float32))
    assert not old.any()
    assert exact_stage(dot, nr, nq, jm).all()
    # one ulp short of -fl(den): |J| < 1 rounds below 1, the reference says 0
    short = np.nextafter(-den.astype(np.float32), np.float32(0)).astype(np.int64)
    nq2 = _w(den + short - nr)
    for d, a, b in zip(short, nr, nq2):
        assert oracle.ani_from_dot(int(d), int(a), int(b)) == np.float32(0.0)


@pytest.mark.parametrize("th", THS)
def test_tensor_bound_is_exact_below_the_cut(oracle, th):
    """both true norms below the cut: nothing wraps, |dot| <= sqrt(n_r n_q), the i32 norms are the true ones"""
    rng = np.random.default_rng(7 + int(th))
    n = 6000
    nr = np.concatenate([rng.integers(0, CUT, n), np.full(50, CUT - 1), rng.integers(CUT - 1000, CUT, 50)])
    nq = np.concatenate([rng.integers(0, CUT, n), np.full(50, CUT - 1), rng.integers(0, 1000, 50)])
    lim = np.floor(np.sqrt(nr.astype(np.float64) * nq)).astype(np.int64)
    u = rng.random(nr.size)
    dot = np.where(u < 0.3, lim, np.where(u < 0.5, -lim, np.rint((2 * rng.random(nr.size) - 1) * lim).astype(np.int64)))
    hi = rng.random(nr.size) < 0.5  # near-identical rows: dot just under the geometric mean
    dot = np.where(hi, lim - rng.integers(0, 1 + lim // 50 + 1, nr.size), dot)
    assert (np.abs(dot) <= lim).all() and (nr + nq - dot < 2**31).all()
    acc = _accepted(oracle, dot, nr, nq, th)
    cand = tensor_bound(dot, nr, nq, nr, nq, _cfrac(_jmin(th)))
    assert not (acc & ~cand).any(), np.stack([dot, nr, nq], 1)[acc & ~cand][:5]
    assert acc.any() and (~cand).any()
    # and the bound only ever passes what the exact stage would look at
    assert not (acc & ~exact_stage(dot, nr, nq, _jmin(th))).any()


@pytest.mark.parametrize("th", [85.0, 95.0, 99.5])
def test_tensor_bound_takes_every_pair_of_a_row_at_or_above_the_cut(oracle, th):
    """the issue's table: r = +-a, q = -r at D 4096 / 16384 / 32768; the true norms pass the cut, the i32 ones may wrap"""
    cfrac = _cfrac(_jmin(th))
    for D, a in [(4096, 480), (4096, 505), (16384, 250), (32768, 180), (4096, 700), (4096, 400)]:
        N = D * a * a
        nr = nq = int(_w(N))
        dot = int(_w(-N))
        big = N >= CUT
        flagged = tensor_bound(dot, nr, nq, N, N, cfrac)
        plain = tensor_bound(dot, nr, nq, 0, 0, cfrac)  # the bound without the flag
        acc = oracle.ani_from_dot(dot, nr, nq) >= np.float32(th)
        assert bool(flagged) == big or not acc
        if acc:
            assert flagged and big and not plain  # what the flag is for
