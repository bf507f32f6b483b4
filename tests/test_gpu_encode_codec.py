"""The HV encoder (encode_kernel: hash set -> hv, norm2, width b, BitPacker8x bytes) and the packed-row codec
(unpack_kernel) against the oracle, bit for bit, where the natural sets of test_gpu_sketch never go: every width from 6
to 16, i16 and i32 wrapping, every work split of the encoder up to its shared-memory limit, empty sets, u64::MAX as an
element of a dense set, and unpacking at every width, stride and alignment.

Exact hv values: dimension 64 i + p counts bit q = (p % 4) 16 + p / 4 of WyRng word i of each hash (hd.rs:61-87).  So c
hashes that set that bit and n - c that clear it give hv = 2 c - n there exactly, while every other dimension stays
near +-sqrt(n).  With n = |v| no other dimension can leave [-n, n], so the width is the one v asks for; every set still
asserts the oracle's width before the GPU is asked anything."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

M64 = (1 << 64) - 1
WY_P0, WY_P1 = 0xA0761D6478BD642F, 0xE7037ED1A0B428DB
HG_EMPTY = np.uint64(M64)
AUTO = 0


def _wyrng_word(h, i):
    """word i (from 0) of the WyRng seeded with each element of h (the state advances by P0 before every word)"""
    s = h + np.uint64(WY_P0 * (i + 1) & M64)
    a = s ^ np.uint64(WY_P1)
    m, t = np.uint64(0xFFFFFFFF), np.uint64(32)
    a0, a1, s0, s1 = a & m, a >> t, s & m, s >> t
    p00, p01, p10, p11 = a0 * s0, a0 * s1, a1 * s0, a1 * s1
    mid = (p00 >> t) + (p01 & m) + (p10 & m)
    lo = (p00 & m) | (mid << t)
    hi = p11 + (p01 >> t) + (p10 >> t) + (mid >> t)
    return lo ^ hi


def _dim(chunk, q):
    """the dimension that bit q of word `chunk` counts"""
    return 64 * chunk + 4 * (q % 16) + q // 16


def _random_hashes(rng, n):
    h = np.unique(rng.integers(0, M64, int(n * 1.01) + 64, dtype=np.uint64, endpoint=True))
    h = h[h != HG_EMPTY]
    assert h.size >= n
    return rng.permutation(h)[:n]


def _with_value(rng, dim, v):
    """|v| distinct hashes, all setting (v > 0) or all clearing (v < 0) the bit that dimension `dim` counts: hv[dim] = v"""
    n = abs(v)
    cand = _random_hashes(rng, 2 * n + 4096)
    chunk, p = divmod(dim, 64)
    q = (p % 4) * 16 + p // 4
    bit = (_wyrng_word(cand, chunk) >> np.uint64(q)) & np.uint64(1)
    side = cand[bit == np.uint64(1 if v > 0 else 0)]
    assert side.size >= n
    return side[:n]


def _width(oracle, hv):
    return oracle.compress_hd_sketch(hv)[0]


class _Want:
    """the oracle's sketches of a list of hash sets"""

    def __init__(self, oracle, sets, hv_d):
        self.hv_d = hv_d
        self.hv = np.stack([oracle.encode_hd(s, hv_d) for s in sets])
        self.norm2 = np.array([oracle.hv_l2_norm_sq(v) for v in self.hv], np.int32)
        packed = [oracle.compress_hd_sketch(v) for v in self.hv]
        self.bits = np.array([b for b, _ in packed], np.uint8)
        self.packed = [p for _, p in packed]


def _check_sketches(got, want, rows=None):
    rows = range(want.hv.shape[0]) if rows is None else rows
    for g in rows:
        assert np.array_equal(got["hv"][g], want.hv[g]), g
        assert got["norm2"][g] == want.norm2[g], g
        assert got["quant_bits"][g] == want.bits[g], g
        nb = int(want.bits[g]) * want.hv_d // 8
        assert nb == want.packed[g].size
        assert np.array_equal(got["packed"][g, :nb], want.packed[g]), g
        assert not got["packed"][g, nb:].any(), g


def test_wyrng_word_matches_oracle(oracle):
    rng = np.random.default_rng(1)
    h = np.concatenate([np.array([0, 1, M64], np.uint64), rng.integers(0, M64, 61, dtype=np.uint64, endpoint=True)])
    for x in h:
        words = oracle.wyrng_words(int(x), 40)
        assert [int(_wyrng_word(np.array([x]), i)[0]) for i in range(40)] == words


# ---- 1. width boundaries: max = 2^(b-1) - 1 | 2^(b-1), min = -2^(b-1) | -2^(b-1) - 1, for every b in 6..15 ----

BOUNDARY_D = 2304  # 36 chunks: chunk 0 and the last chunk sit in different chunk-blocks of 32


@pytest.fixture(scope="module")
def boundary(ctx, oracle):
    rng = np.random.default_rng(0xB0)
    C = BOUNDARY_D // 64
    sets, cases = [], []
    for b in range(6, 16):
        h = 1 << (b - 1)
        for v, wb in ((h - 1, b), (h, b + 1), (-h, b), (-h - 1, b + 1)):
            if wb == 16:
                continue  # refused: test_b16_is_refused
            for chunk in (0, C - 1):
                for q in (b, 48 + b):  # q < 16 and q >= 48: both ends of the spill's inverse permutation
                    sets.append(_with_value(rng, _dim(chunk, q), v))
                    cases.append((b, v, wb, _dim(chunk, q)))
    want = _Want(oracle, sets, BOUNDARY_D)
    for g, (b, v, wb, dim) in enumerate(cases):
        assert want.hv[g, dim] == v and want.bits[g] == wb, (b, v, wb, dim, want.hv[g, dim], want.bits[g])
    assert sorted(set(want.bits.tolist())) == list(range(6, 16))
    got = ctx.encode_sets(sets, hv_d=BOUNDARY_D)
    return got, want


def test_width_boundaries_encode(boundary):
    got, want = boundary
    _check_sketches(got, want)


def test_width_boundaries_unpack(ctx, boundary):
    got, want = boundary
    assert np.array_equal(ctx.unpack(got["packed"], got["quant_bits"], BOUNDARY_D), want.hv)


def test_width_boundaries_dist_packed(ctx, oracle, boundary):
    """one hg_dist_packed over every row (|hv| up to 16383: beyond the two-limb bound) with the automatic kernel choice"""
    got, want = boundary
    n = want.hv.shape[0]
    decoded = np.stack([oracle.decompress_hd_sketch(p, BOUNDARY_D, int(b)) for p, b in zip(want.packed, want.bits)])
    assert np.array_equal(decoded, want.hv)
    ani, dot = oracle.dist_all(decoded, want.norm2, decoded, want.norm2, symmetric=True)
    hits, _ = ctx.dist_packed(got["packed"], got["quant_bits"], got["norm2"], got["packed"], got["quant_bits"], got["norm2"],
                              BOUNDARY_D, ani_th=0.0, symmetric=True, path=AUTO, sorted_output=False, cap=n * n)
    i, j = hits["i"].astype(np.int64), hits["j"].astype(np.int64)
    idx = i * (n - 1) - i * (i - 1) // 2 + (j - i - 1)
    assert np.array_equal(np.sort(idx), np.arange(n * (n - 1) // 2))
    assert np.array_equal(hits["dot"], dot[idx])
    assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))


# ---- 2. b = 16: the reference's own arithmetic breaks there (hd.rs:140), so the GPU refuses the batch ----

@pytest.mark.parametrize("v", [16384, -16385])
def test_b16_is_refused(ctx, hg, oracle, v):
    import torch
    hv_d, dim = 1024, _dim(5, 60)
    rng = np.random.default_rng(v & 0xFFFF)
    sets = [_random_hashes(rng, 3000), _with_value(rng, dim, v)]
    want = _Want(oracle, sets, hv_d)
    assert want.hv[1, dim] == v and want.bits[1] == 16 and want.bits[0] < 16
    with pytest.raises(hg.HyperGenError) as e:
        ctx.encode_sets(sets, hv_d=hv_d)
    assert e.value.code == hg.ffi.HG_E_RANGE
    assert "hv_quant_bits = 16" in str(e.value)

    off = np.array([0, sets[0].size, sets[0].size + sets[1].size], np.uint64)
    d_h = torch.from_numpy(np.concatenate(sets).view(np.int64)).cuda()
    d_hv = torch.empty((2, hv_d), dtype=torch.int16, device="cuda")
    d_packed = torch.empty((2, 2 * hv_d), dtype=torch.uint8, device="cuda")
    d_bits = torch.empty(2, dtype=torch.uint8, device="cuda")
    d_norm = torch.empty(2, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.encode_sets_dev(d_h.data_ptr(), off, hv_d, d_hv.data_ptr(), d_packed.data_ptr(), d_bits.data_ptr(), d_norm.data_ptr())
    with pytest.raises(hg.HyperGenError) as e:
        ctx.sketch_status()
    assert e.value.code == hg.ffi.HG_E_RANGE
    assert np.array_equal(d_bits.cpu().numpy(), want.bits)
    assert np.array_equal(d_hv.cpu().numpy(), want.hv)
    assert np.array_equal(d_norm.cpu().numpy(), want.norm2)


# ---- 3. wrapping: hv in i16 (hd.rs:29), norm2 in i32 (dist.rs:133-136) ----

def test_hv_wraps_i16(ctx, oracle):
    hv_d, dim = 1024, _dim(9, 33)
    rng = np.random.default_rng(3)
    sets = [_with_value(rng, dim, 50_000)]
    want = _Want(oracle, sets, hv_d)
    assert want.hv[0, dim] == -15536 and want.bits[0] == 15
    _check_sketches(ctx.encode_sets(sets, hv_d=hv_d), want)


def test_norm2_wraps_i32(ctx, oracle):
    hv_d = 32000
    sets = [_random_hashes(np.random.default_rng(4), 70_000)]
    want = _Want(oracle, sets, hv_d)
    true = int((want.hv[0].astype(np.int64) ** 2).sum())
    assert true > 2**31
    assert want.norm2[0] == (true + 2**31) % 2**32 - 2**31
    _check_sketches(ctx.encode_sets(sets, hv_d=hv_d), want)


# ---- 4. encoder shapes: C = hv_d / 64 chunks in nCB = ceil(C / 32) chunk-blocks, S = 16 / nCB hash strides ----

SIZES = [0, 1, 4095, 4096, 4097, 8193]  # across the 4096-hash staging batch


@pytest.mark.parametrize("hv_d", [256, 2304, 6144, 10240, 20480, 31744, 32000])
def test_encoder_shapes(ctx, oracle, hv_d):
    rng = np.random.default_rng(hv_d)
    sets = [_random_hashes(rng, n) for n in SIZES]
    if hv_d == 20480:  # S = 1: one lane counts all 4096 hashes of the batch, up to the top counter plane
        dim = _dim(hv_d // 64 - 3, 47)
        sets.append(_with_value(rng, dim, 4096))
    want = _Want(oracle, sets, hv_d)
    if hv_d == 20480:
        assert want.hv[-1, dim] == 4096 and want.bits[-1] == 14
    _check_sketches(ctx.encode_sets(sets, hv_d=hv_d), want)


def test_encoder_refuses_hv_d_past_its_shared_memory(ctx, hg):
    with pytest.raises(hg.HyperGenError) as e:
        ctx.encode_sets([np.arange(1, 100, dtype=np.uint64)], hv_d=32256)
    assert e.value.code == hg.ffi.HG_E_UNSUPPORTED
    assert "max 32000" in str(e.value)


@pytest.mark.parametrize("hv_d", [16384, 32000])
def test_sketch_batch_wide(ctx, hg, oracle, hv_d):
    """the k-mer path (table slots and counts) at widths past the ones test_gpu_sketch covers"""
    from hypergen_b200 import synth
    seqs = [synth.family_member(g, 400_000).numpy() for g in (2, 5)]
    off = np.array([0, seqs[0].size, seqs[0].size + seqs[1].size], np.uint64)
    seq = np.concatenate(seqs)
    got = ctx.sketch_batch(seq, off, hg.make_params(scaled=200, hv_d=hv_d))
    want = oracle.sketch_batch(seq, off, scaled=200, hv_d=hv_d)
    assert (want["n_hashes"] > 1000).all()
    assert np.array_equal(got["n_hashes"], want["n_hashes"])
    assert np.array_equal(got["hv"], want["hv"])
    assert np.array_equal(got["norm2"], want["norm2"]) and np.array_equal(got["quant_bits"], want["quant_bits"])
    for g in range(2):
        nb = int(want["quant_bits"][g]) * hv_d // 8
        assert np.array_equal(got["packed"][g, :nb], want["packed"][g, :nb]), g
        assert not got["packed"][g, nb:].any(), g


# ---- 5. empty sets between large ones: an empty set's CTA reads counters the batch loop never touched ----

@pytest.mark.parametrize("waves,size", [(2, 20_000), (1, 2_000)], ids=["two_waves", "one_wave"])
def test_empty_sets_among_large_ones(ctx, oracle, waves, size):
    """At hv_d 31744 one CTA fits an SM.  Each wave is one large set per SM followed by one empty set per SM, so the
    empty sets start as the large ones finish, on SMs whose shared memory still holds a large set's counters.  An empty
    set is all-zero hv, norm2 0, b 6 and every 6-bit field holding the offset 32.  Whether a missing barrier after the
    counter clear shows in these values depends on warp timing (profiles/r4_encode_empty_set_race.md); `one_wave` is
    sized for a run under a shared-memory race checker."""
    import torch
    hv_d = 31744
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rng = np.random.default_rng(5)
    big = [_random_hashes(rng, size) for _ in range(3)]
    want = _Want(oracle, big + [np.zeros(0, np.uint64)], hv_d)
    assert want.bits[3] == 6 and want.norm2[3] == 0 and not want.hv[3].any()
    kind = np.tile(np.repeat([0, 3], sms), waves)  # 0..2: a large set, 3: the empty set
    kind[kind == 0] = np.arange(waves * sms) % 3
    sets = [big[k] if k < 3 else np.zeros(0, np.uint64) for k in kind]
    got = ctx.encode_sets(sets, hv_d=hv_d)
    empty = np.flatnonzero(kind == 3)
    assert not got["hv"][empty].any()
    assert not got["norm2"][empty].any()
    assert (got["quant_bits"][empty] == 6).all()
    nb = 6 * hv_d // 8
    assert (got["packed"][empty, :nb] == want.packed[3]).all()
    assert not got["packed"][empty, nb:].any()
    for g in np.flatnonzero(kind < 3):
        k = kind[g]
        assert np.array_equal(got["hv"][g], want.hv[k]), g
        assert got["norm2"][g] == want.norm2[k] and got["quant_bits"][g] == want.bits[k], g
        nb = int(want.bits[k]) * hv_d // 8
        assert np.array_equal(got["packed"][g, :nb], want.packed[k]) and not got["packed"][g, nb:].any(), g


# ---- 6. dense sets (hg_encode_sets): every element is a hash, 0 and u64::MAX included ----

def test_dense_sets_with_zero_and_u64_max(ctx, oracle):
    hv_d = 1024
    rng = np.random.default_rng(6)
    zero, top = np.array([0], np.uint64), np.array([M64], np.uint64)

    def at(x, pos, extra):
        return np.insert(x, pos, extra)

    sets = [top, zero, np.array([0, M64], np.uint64), np.array([M64, 0], np.uint64),
            at(_random_hashes(rng, 999), 0, top),
            at(_random_hashes(rng, 4096), 4096, top),           # the only hash of the second staging batch
            at(_random_hashes(rng, 777), 300, [M64, 0]),
            at(_random_hashes(rng, 5000), 2500, zero),
            at(_random_hashes(rng, 31), 31, top)]               # the last slot of a 32-slot warp pass
    want = _Want(oracle, sets, hv_d)
    _check_sketches(ctx.encode_sets(sets, hv_d=hv_d), want)


# ---- 7. unpack (decompress_hd_sketch, hd.rs:184-212) on random bytes ----

UNPACK_D = 768


@pytest.mark.parametrize("b", range(1, 17))
def test_unpack_every_width_and_stride(ctx, oracle, b):
    """every width, also those the encoder never emits, on rows b * hv_d / 8 bytes apart and 4 and 12 more.  The row
    width 32 b (hv_d / 256) is always a multiple of 32, so only the +4 and +12 strides take the unaligned loads."""
    rng = np.random.default_rng(70 + b)
    width = b * UNPACK_D // 8
    for stride in (width, width + 4, width + 12):
        packed = rng.integers(0, 256, (7, stride), dtype=np.uint8)
        got = ctx.unpack(packed, np.full(7, b, np.uint8), UNPACK_D)
        for g in range(7):
            assert np.array_equal(got[g], oracle.decompress_hd_sketch(packed[g, :width], UNPACK_D, b)), (stride, g)


def test_unpack_dev_unaligned_source_and_destination(ctx, oracle):
    """rows 16 * hv_d / 8 + 4 bytes apart from 4 bytes past an aligned address, into hv 2 bytes past one, with
    sentinels on both sides"""
    import torch
    rng = np.random.default_rng(8)
    n = 37
    stride = 16 * UNPACK_D // 8 + 4
    bits = rng.integers(1, 17, n).astype(np.uint8)
    packed = rng.integers(0, 256, n * stride + 4, dtype=np.uint8)
    d_packed = torch.from_numpy(packed).cuda()
    d_bits = torch.from_numpy(bits).cuda()
    sentinel = -12345
    d_out = torch.full((n * UNPACK_D + 16,), sentinel, dtype=torch.int16, device="cuda")
    assert d_out.data_ptr() % 16 == 0 and d_packed.data_ptr() % 16 == 0
    torch.cuda.synchronize()
    ctx.unpack_dev(d_packed.data_ptr() + 4, stride, d_bits.data_ptr(), n, UNPACK_D, d_out.data_ptr() + 2)
    ctx.sync()
    out = d_out.cpu().numpy()
    assert out[0] == sentinel and (out[1 + n * UNPACK_D:] == sentinel).all()
    got = out[1:1 + n * UNPACK_D].reshape(n, UNPACK_D)
    for g in range(n):
        row = packed[4 + g * stride:4 + g * stride + int(bits[g]) * UNPACK_D // 8]
        assert np.array_equal(got[g], oracle.decompress_hd_sketch(row, UNPACK_D, int(bits[g]))), g


def test_unpack_more_rows_than_one_grid(ctx, oracle):
    """65 539 rows of mixed widths: past the 65 535 rows one launch's gridDim.y holds"""
    hv_d, n = 256, 65_539
    rng = np.random.default_rng(9)
    bits = rng.integers(1, 17, n).astype(np.uint8)
    bits[65_535:] = [3, 16, 7, 11]
    packed = rng.integers(0, 256, (n, 16 * hv_d // 8), dtype=np.uint8)
    got = ctx.unpack(packed, bits, hv_d)
    for g in range(n):
        b = int(bits[g])
        assert np.array_equal(got[g], oracle.decompress_hd_sketch(packed[g, :b * hv_d // 8], hv_d, b)), g


@pytest.mark.parametrize("bad", ["bits_0", "bits_17", "stride_below_width", "stride_not_4"])
def test_unpack_rejects_bad_rows(ctx, hg, bad):
    bits = np.full(4, 9, np.uint8)
    stride = 9 * UNPACK_D // 8
    if bad == "bits_0":
        bits[2] = 0
    elif bad == "bits_17":
        bits[2] = 17
    elif bad == "stride_below_width":
        stride -= 4
    else:
        stride += 2
    with pytest.raises(hg.HyperGenError) as e:
        ctx.unpack(np.zeros((4, stride), np.uint8), bits, UNPACK_D)
    assert e.value.code == hg.ffi.HG_E_INVALID
