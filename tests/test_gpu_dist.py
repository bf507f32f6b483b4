"""GPU parity: dist (exact i32 dots, f32 ANI bit-for-bit, threshold filter) vs the oracle.

Reference behaviour under test: src/dist.rs:139-161 (compute_pairwise_ani), :231-294 (pair
enumeration), src/utils.rs:260-286 (sort + `ani >= ani_th` filter)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PATHS = [1, 2, 3]  # 1 = SIMT, 2 = tcgen05 two-limb tensor path, 3 = tcgen05 single-plane (narrow) tensor path


def _sketches(oracle, n, length=150_000, hv_d=4096, scaled=1500, first=0):
    from hypergen_b200 import synth
    seq, off = synth.family_batch(n, length, first=first)
    sk = oracle.sketch_batch(seq.numpy(), off, scaled=scaled, hv_d=hv_d)
    return sk["hv"], sk["norm2"]


def _as_pairs(hits, R, Q, symmetric):
    """hits -> dict keyed by the reference's pair index (dist.rs:251-265)"""
    i, j = hits["i"].astype(np.int64), hits["j"].astype(np.int64)
    if symmetric:
        idx = i * (Q - 1) - i * (i - 1) // 2 + (j - i - 1)
    else:
        idx = i * Q + j
    return idx


def _try_path(ctx, hg, path, fn):
    try:
        return fn()
    except hg.HyperGenError as e:
        if path == 2 and e.code == hg.ffi.HG_E_UNSUPPORTED:
            pytest.skip("tensor path not built")
        raise


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("symmetric", [False, True])
def test_all_pairs_dot_and_ani_bit_exact(ctx, hg, oracle, path, symmetric):
    hv, norm = _sketches(oracle, 150, length=60_000, hv_d=1024, scaled=300)
    if symmetric:
        r, rn, q, qn = hv, norm, hv, norm
    else:
        r, rn, q, qn = hv[:70], norm[:70], hv[40:], norm[40:]
    ani, dot = oracle.dist_all(r, rn, q, qn, symmetric=symmetric)
    hits = _try_path(ctx, hg, path, lambda: ctx.dist(r, rn, q, qn, ani_th=0.0, symmetric=symmetric, path=path,
                                                      cap=ani.size + 16))
    assert hits.size == ani.size  # ani >= 0 always: every enumerated pair is reported
    idx = _as_pairs(hits, r.shape[0], q.shape[0], symmetric)
    assert np.array_equal(np.sort(idx), np.arange(ani.size))
    assert np.array_equal(hits["dot"], dot[idx])                      # exact integers
    assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))  # every f32 bit
    assert float(np.max(np.abs(hits["ani"] - ani[idx]))) <= 1e-6


@pytest.mark.parametrize("path", PATHS)
def test_threshold_filter_and_output_order(ctx, hg, oracle, path):
    hv, norm = _sketches(oracle, 64, length=200_000)
    ani, dot = oracle.dist_all(hv, norm, hv, norm, symmetric=True)
    for th in (85.0, 95.0, 99.9, 100.0):
        hits = _try_path(ctx, hg, path, lambda: ctx.dist(hv, norm, hv, norm, ani_th=th, symmetric=True, path=path))
        idx = _as_pairs(hits, 64, 64, True)
        want = np.nonzero(ani >= np.float32(th))[0]
        assert np.array_equal(np.sort(idx), want), th
        # the reference's emission order (utils.rs:262-269) rebuilt from the hits
        from hypergen_b200 import dist as hdist
        order = hdist.reference_output_order(hits, 64, 64, True)
        assert np.array_equal(idx[order], oracle.ani_output_order(ani, th)), th


@pytest.mark.parametrize("path", PATHS)
def test_headline_shape_D4096_and_D8192(ctx, hg, oracle, path):
    for hv_d, scaled in ((4096, 1500), (8192, 500)):
        hv, norm = _sketches(oracle, 40, length=400_000, hv_d=hv_d, scaled=scaled, first=3)
        ani, dot = oracle.dist_all(hv[:17], norm[:17], hv, norm, symmetric=False)
        hits = _try_path(ctx, hg, path, lambda: ctx.dist(hv[:17], norm[:17], hv, norm, ani_th=0.0, path=path,
                                                          cap=ani.size))
        idx = _as_pairs(hits, 17, 40, False)
        assert np.array_equal(hits["dot"], dot[idx])
        assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))


@pytest.mark.parametrize("path", PATHS)
def test_degenerate_inputs(ctx, hg, oracle, path, monkeypatch):
    """zero vectors (0/0 -> NaN -> 0), negative dots (ln of a negative -> NaN -> 0), identical HVs (100)."""
    # random parity and a 600-wide range: for the single-plane path every other element is an outlier;
    # with the budget lifted it must still be exact (all of it through the sparse corrections)
    monkeypatch.setenv("HG_NARROW_BUDGET", "2048")
    rng = np.random.default_rng(5)
    D = 1024
    hv = rng.integers(-300, 300, (130, D)).astype(np.int16)
    hv[0] = 0
    hv[1] = hv[2]
    hv[3] = -hv[4]
    norm = np.array([oracle.hv_l2_norm_sq(v) for v in hv], np.int32)
    ani, dot = oracle.dist_all(hv, norm, hv, norm, symmetric=False)
    hits = _try_path(ctx, hg, path, lambda: ctx.dist(hv, norm, hv, norm, ani_th=0.0, path=path, cap=ani.size))
    idx = _as_pairs(hits, 130, 130, False)
    assert np.array_equal(hits["dot"], dot[idx])
    assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))
    assert hits["ani"][(hits["i"] == 1) & (hits["j"] == 2)][0] == np.float32(100.0)
    assert hits["ani"][(hits["i"] == 0) & (hits["j"] == 0)][0] == np.float32(0.0)


def test_auto_path_reports_reason_and_wide_values_fall_back(ctx, hg, oracle):
    rng = np.random.default_rng(9)
    hv = rng.integers(-20000, 20000, (130, 512)).astype(np.int16)  # needs 16 bits: no int8 limb split
    norm = np.array([oracle.hv_l2_norm_sq(v) for v in hv], np.int32)
    ani, dot = oracle.dist_all(hv, norm, hv, norm, symmetric=True)
    hits = ctx.dist(hv, norm, hv, norm, ani_th=0.0, symmetric=True, path=0, cap=ani.size)
    assert ctx.dist_last_path == 1 and "SIMT" in ctx.dist_last_reason
    idx = _as_pairs(hits, 130, 130, True)
    assert np.array_equal(hits["dot"], dot[idx])  # wrapping i32, like the reference
    assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))


def test_golden_small_pipeline(ctx, hg):
    """Committed fixture (tests/golden/small_pipeline.npz): sketch -> dist end to end on the GPU."""
    from hypergen_b200 import synth, dist as hdist
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "small_pipeline.npz"))
    k, scaled, seed, canonical, hv_d, n, length, first = [int(x) for x in z["params"]]
    seq, off = synth.family_batch(n, length, first=first)
    sk = ctx.sketch_batch(seq.numpy(), off, hg.make_params(k=k, scaled=scaled, seed=seed, canonical=canonical, hv_d=hv_d))
    assert np.array_equal(sk["hv"], z["hv"]) and np.array_equal(sk["norm2"], z["norm2"])
    assert np.array_equal(sk["quant_bits"], z["quant_bits"]) and np.array_equal(sk["n_hashes"], z["n_hashes"])
    for g in range(n):
        nb = int(z["quant_bits"][g]) * hv_d // 8
        assert np.array_equal(sk["packed"][g, :nb], z["packed"][g, :nb])
    hits = ctx.dist(sk["hv"], sk["norm2"], sk["hv"], sk["norm2"], ksize=k, ani_th=85.0, symmetric=True)
    idx = _as_pairs(hits, n, n, True)
    order = hdist.reference_output_order(hits, n, n, True)
    assert np.array_equal(idx[order], z["order"])
    assert np.array_equal(hits["ani"][order].view(np.uint32), z["ani"][z["order"]].view(np.uint32))
    assert np.array_equal(hits["dot"][order], z["dot"][z["order"]])


# ---- single-plane (narrow) tensor path: x = 2a + s in one s8 plane + sparse outlier corrections ----

def _narrow_rows(rng, n, D, spread=110):
    """rows shaped like sketch HVs (hv = 2 count - n: one parity per row, centred near 0)"""
    par = rng.integers(0, 2, (n, 1))
    return (2 * np.clip(np.rint(rng.normal(0, spread / 3, (n, D))), -spread, spread).astype(np.int64) + par).astype(np.int16)


def _norms(oracle, hv):
    return np.array([oracle.hv_l2_norm_sq(v) for v in hv], np.int32)


@pytest.mark.parametrize("chunks", [1, 2])
@pytest.mark.parametrize("symmetric", [False, True])
def test_narrow_many_tiles_exact(ctx, hg, oracle, symmetric, chunks, monkeypatch):
    """several 256 x 256 tiles per CTA pair (stage ring across tiles, TMEM accumulator double buffered, ragged edges).
    chunks = 2: the host entry streams the ref rows in two chunks, i.e. two launches into one hit list, the second
    with a tile walk that starts at a row offset (symmetric: j0 > i0, so the walk skips the tiles below the diagonal)"""
    rng = np.random.default_rng(31)
    D = 512
    hv = _narrow_rows(rng, 700, D)
    hv[5] = hv[400]          # a 100 % pair far from the diagonal
    hv[650] = hv[12]
    norm = _norms(oracle, hv)
    if symmetric:
        r, rn, q, qn = hv, norm, hv, norm
    else:
        r, rn, q, qn = hv[:300], norm[:300], hv[100:], norm[100:]
    if chunks == 2:  # chunk size: half of the ref rows, rounded up to a multiple of 256 as the library does
        half = (r.shape[0] + 1) // 2
        monkeypatch.setenv("HG_DIST_CHUNK_ROWS", str((half + 255) // 256 * 256))
    ani, dot = oracle.dist_all(r, rn, q, qn, symmetric=symmetric)
    hits = ctx.dist(r, rn, q, qn, ani_th=0.0, symmetric=symmetric, path=3, cap=ani.size + 16)
    assert ctx.dist_last_path == 3
    assert "%d row chunk" % chunks in ctx.dist_last_reason, ctx.dist_last_reason
    idx = _as_pairs(hits, r.shape[0], q.shape[0], symmetric)
    assert np.array_equal(np.sort(idx), np.arange(ani.size))
    assert np.array_equal(hits["dot"], dot[idx])
    assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))


@pytest.mark.parametrize("chunks", [1, 2])
@pytest.mark.parametrize("ani_th", [0.0, 85.0])
def test_narrow_outlier_corrections(ctx, hg, oracle, ani_th, chunks, monkeypatch):
    """rows with a few elements outside the s8 plane (range and parity outliers, both sides): the kernel
    loosens their bound and corrects each candidate exactly.  chunks = 2: the host entry streams the symmetric run's
    300 rows in two chunks of 256 rows, so the outlier entries of the second chunk's pre-pass follow those of the
    first and a launch reads both (the ref x query run has 130 ref rows: one chunk either way)"""
    if chunks == 2:
        monkeypatch.setenv("HG_DIST_CHUNK_ROWS", "256")
    hv, norm = _sketches(oracle, 300, length=120_000, hv_d=1024, scaled=300)
    hv = hv.copy()
    rng = np.random.default_rng(7)
    rows = rng.choice(300, 40, replace=False)
    for t, r in enumerate(rows):
        d = rng.choice(1024, 1 + t % 5, replace=False)
        if t % 3 == 0:
            hv[r, d] += np.int16(1)                                   # wrong parity
        elif t % 3 == 1:
            hv[r, d] = (hv[r, d] + rng.choice([-700, 600, 1400], d.size)).astype(np.int16)   # far outside the plane
        else:
            hv[r, d] = np.int16(8001)                                # odd and far
    norm = _norms(oracle, hv)
    for symmetric in (True, False):
        if symmetric:
            r_, rn, q_, qn = hv, norm, hv, norm
        else:
            r_, rn, q_, qn = hv[:130], norm[:130], hv[90:], norm[90:]
        ani, dot = oracle.dist_all(r_, rn, q_, qn, symmetric=symmetric)
        hits = ctx.dist(r_, rn, q_, qn, ani_th=ani_th, symmetric=symmetric, path=0, cap=ani.size + 16)
        assert ctx.dist_last_path == 3 and "narrow" in ctx.dist_last_reason, ctx.dist_last_reason
        assert "%d row chunk" % (chunks if symmetric else 1) in ctx.dist_last_reason, ctx.dist_last_reason
        idx = _as_pairs(hits, r_.shape[0], q_.shape[0], symmetric)
        want = np.nonzero(ani >= np.float32(ani_th))[0]
        assert np.array_equal(np.sort(idx), want)
        assert np.array_equal(hits["dot"], dot[idx])
        assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))


def test_auto_path_narrow_for_sketches_and_two_limb_for_wide_rows(ctx, hg, oracle):
    hv, norm = _sketches(oracle, 140, length=200_000)
    ani, dot = oracle.dist_all(hv, norm, hv, norm, symmetric=True)
    hits = ctx.dist(hv, norm, hv, norm, ani_th=85.0, symmetric=True, path=0)
    assert ctx.dist_last_path == 3, ctx.dist_last_reason
    assert np.array_equal(np.sort(_as_pairs(hits, 140, 140, True)), np.nonzero(ani >= np.float32(85.0))[0])
    # rows twice as wide as scaled=500 / D=8192 sketches (sigma 200): a fifth of the elements lie outside one s8 plane
    rng = np.random.default_rng(3)
    wide = (2 * rng.binomial(40000, 0.5, (140, 1024)) - 40000).astype(np.int16)
    wn = _norms(oracle, wide)
    ani, dot = oracle.dist_all(wide, wn, wide, wn, symmetric=True)
    hits = ctx.dist(wide, wn, wide, wn, ani_th=0.0, symmetric=True, path=0, cap=ani.size)
    assert ctx.dist_last_path == 2 and "declined" in ctx.dist_last_reason, ctx.dist_last_reason
    idx = _as_pairs(hits, 140, 140, True)
    assert np.array_equal(hits["dot"], dot[idx])
    assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))
    with pytest.raises(hg.HyperGenError) as ei:
        ctx.dist(wide, wn, wide, wn, ani_th=0.0, symmetric=True, path=3, cap=ani.size)
    assert ei.value.code == hg.ffi.HG_E_UNSUPPORTED


@pytest.mark.parametrize("shards", [1, 2])
def test_narrow_row_shard_offsets(ctx, hg, oracle, shards):
    """hg_dist_dev on a row shard of the query matrix (i0 > 0, symmetric filter on global indices) - the
    multi-GPU dist step - through the single-plane path.  shards = 2: the same rows as two calls at row offsets
    273 and 423, as two members of a GPU group would compute them"""
    import torch
    rng = np.random.default_rng(11)
    D, n = 2048, 600
    hv = _narrow_rows(rng, n, D)
    hv[37, [3, 99]] = [901, -777]  # one outlier row inside the shard
    norm = _norms(oracle, hv)
    ani, dot = oracle.dist_all(hv, norm, hv, norm, symmetric=True)
    d_hv = torch.from_numpy(hv).cuda()
    d_n = torch.from_numpy(norm).cuda()
    i0, rows = 256 + 17, 300
    cap = rows * n
    d_hits = torch.empty(cap * 16, dtype=torch.uint8, device="cuda")
    d_cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    parts = []
    bounds = [i0 + rows * s // shards for s in range(shards + 1)]
    for a, b in zip(bounds[:-1], bounds[1:]):  # every call resets the hit counter: read its hits before the next one
        ctx.dist_dev(d_hv.data_ptr() + a * D * 2, d_n.data_ptr() + a * 4, b - a, a, d_hv.data_ptr(), d_n.data_ptr(), n, 0, D, 21,
                     0.0, True, 3, d_hits.data_ptr(), cap, d_cnt.data_ptr())
        ctx.sync()
        cnt = int(d_cnt.item())
        parts.append(np.frombuffer(d_hits.cpu().numpy().tobytes(), dtype=hg.ffi.HIT_DTYPE)[:cnt])
    hits = np.concatenate(parts)
    idx = _as_pairs(hits, n, n, True)
    ii, jj = np.meshgrid(np.arange(i0, i0 + rows), np.arange(n), indexing="ij")
    keep = jj > ii
    want = np.sort(ii[keep] * (n - 1) - ii[keep] * (ii[keep] - 1) // 2 + (jj[keep] - ii[keep] - 1))
    assert np.array_equal(np.sort(idx), want)
    assert np.array_equal(hits["dot"], dot[idx])
    assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))


@pytest.mark.parametrize("hv_d", [256, 2048])
def test_narrow_short_and_mid_k(ctx, hg, oracle, hv_d):
    """hv_d = 256 is two K blocks, fewer than the 6-stage ring; 2048 is sixteen"""
    rng = np.random.default_rng(hv_d)
    hv = _narrow_rows(rng, 330, hv_d)
    hv[7] = hv[300]
    norm = _norms(oracle, hv)
    ani, dot = oracle.dist_all(hv, norm, hv, norm, symmetric=True)
    hits = ctx.dist(hv, norm, hv, norm, ani_th=0.0, symmetric=True, path=3, cap=ani.size + 16)
    idx = _as_pairs(hits, 330, 330, True)
    assert np.array_equal(np.sort(idx), np.arange(ani.size))
    assert np.array_equal(hits["dot"], dot[idx])
    assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))


@pytest.mark.parametrize("hv_d", [256, 768, 1280])
@pytest.mark.parametrize("symmetric", [False, True])
def test_two_limb_k_not_a_multiple_of_512(ctx, hg, oracle, hv_d, symmetric):
    """two-limb kernel at hv_d % 512 != 0: its K loop runs whole trips of the 4-stage ring (512 columns) and the
    tensor maps fill the columns past hv_d with zeros; several 256 x 128 tiles with ragged edges, both limbs in use"""
    rng = np.random.default_rng(hv_d + symmetric)
    hv = _narrow_rows(rng, 420, hv_d, spread=1000)  # |hv| <= 2001: the high limb is not zero
    hv[9] = hv[333]
    hv[200] = hv[201]
    norm = _norms(oracle, hv)
    if symmetric:
        r, rn, q, qn = hv, norm, hv, norm
    else:
        r, rn, q, qn = hv[:300], norm[:300], hv[90:], norm[90:]
    ani, dot = oracle.dist_all(r, rn, q, qn, symmetric=symmetric)
    hits = ctx.dist(r, rn, q, qn, ani_th=0.0, symmetric=symmetric, path=2, cap=ani.size + 16)
    assert ctx.dist_last_path == 2, ctx.dist_last_reason
    idx = _as_pairs(hits, r.shape[0], q.shape[0], symmetric)
    assert np.array_equal(np.sort(idx), np.arange(ani.size))
    assert np.array_equal(hits["dot"], dot[idx])
    assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))


@pytest.mark.parametrize("chunk_rows", [0, 256])
def test_narrow_random_sweep(ctx, hg, oracle, chunk_rows, monkeypatch):
    """random shapes, thresholds, symmetric or not, outliers sprinkled on both sides: auto path == oracle.
    chunk_rows = 256: the host entry streams the rows in 256-row chunks (H2D of one chunk under the kernels of the
    previous one), i.e. several partial launches appending to one hit list; 0: its default chunking"""
    if chunk_rows:
        monkeypatch.setenv("HG_DIST_CHUNK_ROWS", str(chunk_rows))
    rng = np.random.default_rng(2026)
    for trial in range(8):
        D = int(rng.choice([256, 512, 1024, 2048]))
        R, Q = int(rng.integers(130, 700)), int(rng.integers(130, 700))
        sym = bool(trial % 2)
        th = float(rng.choice([0.0, 80.0, 95.0]))
        q = _narrow_rows(rng, Q, D, spread=int(rng.integers(40, 125)))
        for _ in range(int(rng.integers(0, 6))):            # a few near-duplicates so that thresholds > 0 keep something
            a, b = rng.integers(0, Q, 2)
            q[a] = q[b]
            q[a, rng.integers(0, D, 8)] += np.int16(2)
        for _ in range(int(rng.integers(0, 12))):           # outliers: far values and parity flips
            q[rng.integers(0, Q), rng.integers(0, D)] += np.int16(rng.choice([1, -1, 700, -900, 3001]))
        if sym:
            r, R = q, Q
        else:
            r = np.concatenate([q[: min(R, Q) // 2], _narrow_rows(rng, R - min(R, Q) // 2, D)])
            r[rng.integers(0, R), rng.integers(0, D)] = np.int16(-2500)
        rn = _norms(oracle, r)
        qn = rn if sym else _norms(oracle, q)
        ani, dot = oracle.dist_all(r, rn, q, qn, symmetric=sym)
        hits = ctx.dist(r, rn, q, qn, ani_th=th, symmetric=sym, path=0, cap=ani.size + 16)
        assert ctx.dist_last_path == 3, (trial, ctx.dist_last_reason)
        idx = _as_pairs(hits, R, Q, sym)
        want = np.nonzero(ani >= np.float32(th))[0]
        assert np.array_equal(np.sort(idx), want), (trial, D, R, Q, sym, th)
        assert np.array_equal(hits["dot"], dot[idx]), trial
        assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32)), trial


def test_streamed_dist_declines_midway_and_falls_back(ctx, hg, oracle, monkeypatch):
    """narrow rows first, wide rows in the last chunk: the chunks already computed are discarded and the two-limb
    kernel runs on the matrices that are complete in HBM by then"""
    monkeypatch.setenv("HG_DIST_CHUNK_ROWS", "256")
    rng = np.random.default_rng(77)
    D = 512
    hv = _narrow_rows(rng, 700, D)
    hv[600:] = (2 * rng.binomial(40000, 0.5, (100, D)) - 40000).astype(np.int16)
    norm = _norms(oracle, hv)
    ani, dot = oracle.dist_all(hv, norm, hv, norm, symmetric=True)
    hits = ctx.dist(hv, norm, hv, norm, ani_th=0.0, symmetric=True, path=0, cap=ani.size + 16)
    assert ctx.dist_last_path == 2, ctx.dist_last_reason
    idx = _as_pairs(hits, 700, 700, True)
    assert np.array_equal(np.sort(idx), np.arange(ani.size))
    assert np.array_equal(hits["dot"], dot[idx])
    assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))


def test_full_size_config3_against_the_oracle_cross_kernel_and_symmetry_properties(ctx, hg, oracle):
    """BASELINE config 3 at full size (10,000 sketches, D=4096, ani_th=85): the hit list must be the oracle's over all
    49,995,000 pairs (src/dist.rs:139-161,231-294 + the filter of src/utils.rs:274-285: same set, i32 dots, f32 ANI
    bits - about two seconds of the C restatement on the box's cores); the three kernels must report the same hits bit
    for bit; the symmetric run must equal the j > i half of the full ref x query run, whose other half must mirror it
    (dot and ANI are symmetric in the pair); and every sketch against itself must come out at exactly 100."""
    import torch
    from hypergen_b200 import synth
    n, D = 10_000, 4096
    dev = torch.device("cuda", 0)
    sets = synth.hash_sets_family(n)
    off = np.zeros(n + 1, np.uint64)
    off[1:] = np.cumsum([len(x) for x in sets])
    hashes = torch.from_numpy(np.concatenate(sets).view(np.int64)).to(dev)
    hv = torch.empty((n, D), dtype=torch.int16, device=dev)
    bits = torch.empty(n, dtype=torch.uint8, device=dev)
    norm = torch.empty(n, dtype=torch.int32, device=dev)
    ctx.encode_sets_dev(hashes.data_ptr(), off, D, hv.data_ptr(), None, bits.data_ptr(), norm.data_ptr())
    ctx.sync()
    cap = 1_000_000
    d_hits = torch.empty(cap * 16, dtype=torch.uint8, device=dev)
    d_cnt = torch.zeros(1, dtype=torch.int64, device=dev)

    def run(path, sym):
        ctx.dist_dev(hv.data_ptr(), norm.data_ptr(), n, 0, hv.data_ptr(), norm.data_ptr(), n, 0, D, 21, 85.0, sym, path,
                     d_hits.data_ptr(), cap, d_cnt.data_ptr())
        ctx.sync()
        c = int(d_cnt.item())
        assert c <= cap
        h = np.frombuffer(d_hits[: c * 16].cpu().numpy().tobytes(), dtype=hg.ffi.HIT_DTYPE)
        return np.sort(h, order=["i", "j"])

    narrow = run(3, True)
    assert ctx.dist_last_path == 3
    oracle.set_threads(os.cpu_count() or 1)
    hv_np, norm_np = hv.cpu().numpy(), norm.cpu().numpy()
    ani, dot = oracle.dist_all(hv_np, norm_np, hv_np, norm_np, symmetric=True)
    want = np.nonzero(ani >= np.float32(85.0))[0]
    hi, hj = narrow["i"].astype(np.int64), narrow["j"].astype(np.int64)
    idx = hi * (n - 1) - hi * (hi - 1) // 2 + (hj - hi - 1)  # (i, j)-sorted hits are in pair-index order
    assert np.array_equal(idx, want)
    assert np.array_equal(narrow["dot"], dot[want])
    assert np.array_equal(narrow["ani"].view(np.uint32), ani[want].view(np.uint32))
    del ani, dot
    assert np.array_equal(narrow, run(2, True))      # two-limb tensor kernel
    assert np.array_equal(narrow, run(1, True))      # CUDA-core kernel
    assert narrow.size > 100_000 and (narrow["i"] < narrow["j"]).all()
    full = run(3, False)
    upper = full[full["j"] > full["i"]]
    lower = full[full["j"] < full["i"]]
    diag = full[full["j"] == full["i"]]
    assert np.array_equal(upper, narrow)
    mirrored = np.sort(np.rec.fromarrays([lower["j"], lower["i"], lower["dot"], lower["ani"]], dtype=hg.ffi.HIT_DTYPE), order=["i", "j"])
    assert np.array_equal(mirrored, narrow)
    assert diag.size == n and (diag["ani"] == np.float32(100.0)).all() and np.array_equal(diag["dot"], norm.cpu().numpy())
    # family members 0 and ... keep probability 1.0 means member 0 IS the pool; members with the same kept set are rare,
    # but every hit must respect the threshold and the ANI bound
    assert (narrow["ani"] >= np.float32(85.0)).all() and (narrow["ani"] <= np.float32(100.0)).all()
