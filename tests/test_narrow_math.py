"""The arithmetic behind the single-plane dist kernel (csrc/dist_narrow.cu), restated in numpy and checked
against the plain i16 dot product of the reference (src/dist.rs:147-151).  CPU only: this pins the identities
the kernel relies on; the kernel itself is checked against the oracle in tests/test_gpu_dist.py."""
import numpy as np


def prep(m):
    """narrow_prep_kernel: per-row centre s, s8 plane a, residuals eps = x - (2a + s)"""
    lo, hi = m.min(1), m.max(1)
    d = m.shape[1]
    par = (2 * (m & 1).sum(1) > d).astype(np.int64)
    mid = (lo + hi + 2) >> 1
    tot = m.sum(1)
    mean = np.where(tot >= 0, (tot + d // 2) // d, -((-tot + d // 2) // d))
    mid = np.where(hi - lo > 510, mean, mid)
    s = mid - ((mid - par) & 1)
    t = m - s[:, None]
    a = np.clip(t >> 1, -128, 127)
    return s, a, t - 2 * a


def sketch_like(rng, n, d, sigma):
    par = rng.integers(0, 2, (n, 1))
    return 2 * np.rint(rng.normal(0, sigma / 2, (n, d))).astype(np.int64) + par


def test_rows_that_span_at_most_510_have_no_residuals():
    rng = np.random.default_rng(1)
    x = np.clip(sketch_like(rng, 50, 512, 60), -255, 255)
    x = x - ((x ^ x[:, :1]) & 1)  # one parity per row, as hv = 2 count - n
    assert (x.max(1) - x.min(1) <= 510).all()
    s, a, eps = prep(x)
    assert not eps.any() and a.min() >= -128 and a.max() <= 127


def test_single_plane_identity_with_outlier_corrections_and_bounds():
    rng = np.random.default_rng(2)
    d = 1024
    x, y = sketch_like(rng, 40, d, 58), sketch_like(rng, 60, d, 58)
    x[3, [5, 77]] = [901, -777]       # far outside the plane
    x[4, 9] += 1                      # wrong parity
    y[7, 100] = 8001
    y[8, [3, 5]] += np.array([1, -600])
    sx, ax, ex = prep(x)
    sy, ay, ey = prep(y)
    acc = ax @ ay.T                                            # the one s8 GEMM
    xt_sum = 2 * ax.sum(1) + d * sx                            # sum of x~ per ref row
    t_q = 2 * ay.sum(1)                                        # 2 sum(b) per query row
    dot_tilde = 4 * acc + sy[None, :] * xt_sum[:, None] + sx[:, None] * t_q[None, :]
    xt = 2 * ax + sx[:, None]
    c1, c2 = ex @ y.T, xt @ ey.T                               # sparse corrections
    assert np.array_equal(dot_tilde + c1 + c2, x @ y.T)
    # how far the candidate bound of a row / column has to be lowered
    assert (np.abs(c1) <= np.abs(ex).sum(1)[:, None] * np.abs(y).max()).all()
    assert (np.abs(c2) <= (np.abs(sx).max() + 256) * np.abs(ey).sum(1)[None, :]).all()
    assert (ex != 0).sum() <= 8 and (ey != 0).sum() <= 8       # the centre follows the bulk, not the outliers


def test_identity_holds_in_wrapping_i32():
    rng = np.random.default_rng(3)
    d = 256
    x = rng.integers(-32768, 32768, (6, d))
    y = rng.integers(-32768, 32768, (5, d))
    sx, ax, ex = prep(x)
    sy, ay, ey = prep(y)
    w = lambda v: ((v + 2**31) % 2**32) - 2**31                # i32 wrap-around, as the reference's i32 sum
    dot = w(4 * (ax @ ay.T) + sy[None, :] * (2 * ax.sum(1) + d * sx)[:, None] + sx[:, None] * (2 * ay.sum(1))[None, :]
            + ex @ y.T + (2 * ax + sx[:, None]) @ ey.T)
    assert np.array_equal(dot, w(x @ y.T))


def test_true_norm_from_the_plane_and_the_residuals():
    """narrow_prep_kernel's sum x^2 (HG_NORM_WRAP_CUT): 4 sum a^2 + 2 s sum 2a + D s^2 + sum eps (x - s + 2a + 2s)"""
    rng = np.random.default_rng(4)
    d = 2048
    x = sketch_like(rng, 30, d, 200)
    x[2, [1, 9, 700]] = [29001, -30999, 4001]
    x[5, 3] += 1
    x[7] = 255 - 2 * (np.arange(d) % 256)  # spans exactly 510
    s, a, eps = prep(x)
    t = x - s[:, None]
    xx = 4 * (a * a).sum(1) + 2 * s * (2 * a).sum(1) + d * s * s + (eps * (t + 2 * a + 2 * s[:, None])).sum(1)
    assert np.array_equal(xx, (x * x).sum(1))
