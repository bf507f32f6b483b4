"""Which dist kernel a single-GPU entry runs, for the inputs no other test pins: the requested path, too few pairs
for a tensor tile, a shape the tensor kernels do not tile, packed rows whose hv_quant_bits settle the choice, rows the
single-plane pre-pass declines, and a ref block that is a row window of the query matrix.  Every row checks the
return code, hg_dist_last_path and a reason substring, and that the hits equal the oracle (every dot, every ANI bit)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SIMT, TWO_LIMB, NARROW = 1, 2, 3
WIDE_D = 33024  # a multiple of 256 above the tensor kernels' hv_d limit of 32768


def _norms(oracle, hv):
    return np.array([oracle.hv_l2_norm_sq(v) for v in hv], np.int32)


def _narrow_rows(rng, n, D, spread=110):
    """rows shaped like sketch HVs: one parity per row, centred near 0, within one s8 plane"""
    par = rng.integers(0, 2, (n, 1))
    return (2 * np.clip(np.rint(rng.normal(0, spread / 3, (n, D))), -spread, spread).astype(np.int64) + par).astype(np.int16)


def _rows(rng, n, D, lo, peak, bits=None):
    """uniform rows in [-lo, lo] with one element of magnitude `peak` per row: the rows need max |hv| = peak (and,
    packed, exactly `bits` bits); small enough that no norm or dot wraps i32"""
    hv = rng.integers(-lo, lo + 1, (n, D)).astype(np.int16)
    hv[np.arange(n), rng.integers(0, D, n)] = np.where(rng.random(n) < 0.5, -peak, peak).astype(np.int16)
    return hv


def _pack(oracle, hv, bits):
    rows = [oracle.compress_hd_sketch(v) for v in hv]
    assert all(b == bits for b, _ in rows)
    return np.stack([p for _, p in rows]), np.full(hv.shape[0], bits, np.uint8)


def _check_hits(oracle, hits, r, rn, q, qn, symmetric):
    ani, dot = oracle.dist_all(r, rn, q, qn, symmetric=symmetric)
    i, j = hits["i"].astype(np.int64), hits["j"].astype(np.int64)
    Q = q.shape[0]
    idx = i * (Q - 1) - i * (i - 1) // 2 + (j - i - 1) if symmetric else i * Q + j
    assert np.array_equal(np.sort(idx), np.arange(ani.size))
    assert np.array_equal(hits["dot"], dot[idx])
    assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))


def _expect(ctx, path, reason):
    assert ctx.dist_last_path == path and reason in ctx.dist_last_reason, (ctx.dist_last_path, ctx.dist_last_reason)


def test_host_auto_too_few_pairs_runs_simt(ctx, hg, oracle):
    rng = np.random.default_rng(1)
    hv = _narrow_rows(rng, 230, 1024)
    r, q = hv[:130], hv[130:]
    rn, qn = _norms(oracle, r), _norms(oracle, q)
    hits = ctx.dist(r, rn, q, qn, ani_th=0.0, path=0, cap=130 * 100)
    _expect(ctx, SIMT, "SIMT")
    _check_hits(oracle, hits, r, rn, q, qn, False)


def test_host_auto_shape_declined_runs_simt(ctx, hg, oracle):
    rng = np.random.default_rng(2)
    hv = _narrow_rows(rng, 130, WIDE_D)
    norm = _norms(oracle, hv)
    hits = ctx.dist(hv, norm, hv, norm, ani_th=0.0, symmetric=True, path=0, cap=130 * 130)
    _expect(ctx, SIMT, "declined this shape")
    _check_hits(oracle, hits, hv, norm, hv, norm, True)


@pytest.mark.parametrize("path", [TWO_LIMB, NARROW])
def test_host_forced_tensor_path_refuses_the_shape(ctx, hg, oracle, path):
    rng = np.random.default_rng(3)
    hv = _narrow_rows(rng, 130, WIDE_D)
    norm = _norms(oracle, hv)
    with pytest.raises(hg.HyperGenError) as ei:
        ctx.dist(hv, norm, hv, norm, ani_th=0.0, symmetric=True, path=path, cap=130 * 130)
    assert ei.value.code == hg.ffi.HG_E_UNSUPPORTED


def _packed_case(ctx, oracle, hv, bits):
    norm = _norms(oracle, hv)
    packed, qb = _pack(oracle, hv, bits)
    hits, _ = ctx.dist_packed(packed, qb, norm, packed, qb, norm, hv.shape[1], ani_th=0.0, symmetric=True,
                              cap=hv.shape[0] ** 2)
    _check_hits(oracle, hits, hv, norm, hv, norm, True)


def test_packed_12_bit_rows_of_a_shape_the_tensor_kernels_decline_run_simt(ctx, hg, oracle):
    rng = np.random.default_rng(4)
    _packed_case(ctx, oracle, _rows(rng, 130, WIDE_D, 200, 1500), 12)
    _expect(ctx, SIMT, "SIMT")


def test_packed_14_bit_rows_within_the_limb_budget_run_two_limb(ctx, hg, oracle):
    rng = np.random.default_rng(5)
    _packed_case(ctx, oracle, _rows(rng, 130, 1024, 1200, 5000), 14)
    _expect(ctx, TWO_LIMB, "declined")


def test_packed_14_bit_rows_beyond_the_limb_budget_run_simt(ctx, hg, oracle):
    rng = np.random.default_rng(6)
    _packed_case(ctx, oracle, _rows(rng, 130, 1024, 1200, 8150), 14)
    _expect(ctx, SIMT, "SIMT")


def test_packed_12_bit_rows_run_two_limb_at_hv_d_768(ctx, hg, oracle):
    rng = np.random.default_rng(7)
    _packed_case(ctx, oracle, _rows(rng, 130, 768, 1500, 2000), 12)
    _expect(ctx, TWO_LIMB, "two s8 limbs")


def _dev(ctx, hg, hv, norm, ref_row0, n_ref, path, symmetric=True):
    """hg_dist_dev of rows [ref_row0, ref_row0 + n_ref) of hv against all of hv; returns the hits"""
    import torch
    n, D = hv.shape
    d_hv, d_n = torch.from_numpy(hv).cuda(), torch.from_numpy(norm).cuda()
    cap = n_ref * n
    d_hits = torch.empty(cap * 16, dtype=torch.uint8, device="cuda")
    d_cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    ctx.dist_dev(d_hv.data_ptr() + ref_row0 * D * 2, d_n.data_ptr() + ref_row0 * 4, n_ref, ref_row0, d_hv.data_ptr(),
                 d_n.data_ptr(), n, 0, D, 21, 0.0, symmetric, path, d_hits.data_ptr(), cap, d_cnt.data_ptr())
    ctx.sync()
    cnt = int(d_cnt.item())
    return np.frombuffer(d_hits.cpu().numpy().tobytes(), dtype=hg.ffi.HIT_DTYPE)[:cnt].copy()


def test_dev_forced_narrow_on_wide_rows_defers_the_refusal(ctx, hg, oracle):
    rng = np.random.default_rng(8)
    wide = (2 * rng.binomial(40000, 0.5, (140, 1024)) - 40000).astype(np.int16)
    _dev(ctx, hg, wide, _norms(oracle, wide), 0, 140, NARROW)
    _expect(ctx, NARROW, "narrow")
    with pytest.raises(hg.HyperGenError) as ei:
        ctx.dist_status()
    assert ei.value.code == hg.ffi.HG_E_UNSUPPORTED


def test_dev_auto_beyond_the_limb_budget_runs_simt(ctx, hg, oracle):
    rng = np.random.default_rng(9)
    hv = _rows(rng, 130, 1024, 1200, 9000)
    norm = _norms(oracle, hv)
    hits = _dev(ctx, hg, hv, norm, 0, 130, 0)
    _expect(ctx, SIMT, "SIMT")
    _check_hits(oracle, hits, hv, norm, hv, norm, True)


def test_dev_two_limb_on_a_row_window_of_the_query_matrix(ctx, hg, oracle):
    rng = np.random.default_rng(10)
    n, D, i0, rows = 600, 1024, 256 + 17, 300
    hv = _narrow_rows(rng, n, D, spread=1000)
    norm = _norms(oracle, hv)
    ani, dot = oracle.dist_all(hv, norm, hv, norm, symmetric=True)
    hits = _dev(ctx, hg, hv, norm, i0, rows, TWO_LIMB)
    _expect(ctx, TWO_LIMB, "tensor")
    i, j = hits["i"].astype(np.int64), hits["j"].astype(np.int64)
    idx = i * (n - 1) - i * (i - 1) // 2 + (j - i - 1)
    ii, jj = np.meshgrid(np.arange(i0, i0 + rows), np.arange(n), indexing="ij")
    keep = jj > ii
    assert np.array_equal(np.sort(idx), np.sort(ii[keep] * (n - 1) - ii[keep] * (ii[keep] - 1) // 2 + (jj[keep] - ii[keep] - 1)))
    assert np.array_equal(hits["dot"], dot[idx])
    assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))
