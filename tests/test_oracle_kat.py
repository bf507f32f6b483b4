"""The oracle pinned against every known answer available for this path (no GPU needed):
upstream t1ha2 self-check constants, the reference's own kernel source compiled as host code
(committed vectors), wyhash-rs README vectors, real AVX2
execution of the encode routine, the SURVEY §8c fixtures and the host libm's logf."""
import hashlib
import json
import os

import numpy as np

G = os.path.join(os.path.dirname(__file__), "golden")


def _load(name):
    with open(os.path.join(G, name)) as f:
        return json.load(f)


def test_t1ha2_upstream_and_reference_vectors(oracle):
    v = _load("t1ha2_vectors.json")
    for hexdata, seed, want in v["upstream"] + v["reference"]:
        assert oracle.t1ha2_atonce(bytes.fromhex(hexdata), seed) == want
    assert oracle.t1ha2_atonce(b"ACGTACGTACGTACGTACGTA", 123) == 0xA5823556992034CF


def test_t1ha2_matches_reference_source_live(oracle):
    """The reference's own t1ha2_atonce (src/cuda_kernel.cu:196-246 compiled as host code) on random bytes of every
    length a k-mer can have, odd and even seeds: its answers are stored in golden/t1ha2_vectors.json."""
    v = _load("t1ha2_vectors.json")["reference"]
    by_len = {}
    for hexdata, seed, want in v:
        by_len.setdefault(len(hexdata) // 2, []).append((bytes.fromhex(hexdata), seed, want))
    assert set(range(33)) <= set(by_len)
    assert {s & 1 for _, s, _ in v} == {0, 1}
    for L, cases in sorted(by_len.items()):
        for d, s, want in cases:
            assert oracle.t1ha2_atonce(d, s) == want, (L, d.hex(), s)


def test_kmer_sets_match_reference_kernel_vectors(oracle):
    from hypergen_b200 import synth
    g = synth.genome(0xB200 + 77, 60_000).numpy().copy()
    g[5000:5030] = ord("N")
    g[20000:26000] |= 0x20
    for name, c in _load("kmer_ref_sets.json")["sets"].items():
        # the reference CPU path is always canonical; its GPU path honours the flag
        hs = oracle.kmer_hash_set(g, k=c["k"], scaled=c["scaled"], canonical=c["canonical"])
        assert hs.size == c["n"], name
        assert hashlib.sha256(hs.tobytes()).hexdigest() == c["sha256"], name


def test_wyrng_vectors(oracle):
    for state, outs in _load("wyrng_vectors.json")["vectors"]:
        assert oracle.wyrng_words(state, len(outs)) == outs


def test_encode_layout_is_the_avx2_permutation(oracle):
    rng = np.random.default_rng(11)
    for n in (0, 1, 2, 3, 4, 5, 63, 257):
        for hv_d in (64, 256, 4096):
            hs = np.unique(rng.integers(0, 1 << 62, n, dtype=np.uint64))
            a = oracle.encode_hd(hs, hv_d)
            b = oracle.encode_hd_avx2_intrinsics(hs, hv_d)     # real AVX2 on this host
            assert np.array_equal(a, b)
            s = oracle.encode_hd(hs, hv_d, layout="scalar")    # hd.rs:94-112
            p = np.arange(64)
            pi = (p % 4) * 16 + p // 4
            assert np.array_equal(a.reshape(-1, 64), s.reshape(-1, 64)[:, pi])


def test_encode_wraps_like_i16(oracle):
    # hv is initialised to -(n as i16) and accumulated in i16 (hd.rs:29,84-87)
    hs = np.arange(1, 40001, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
    a = oracle.encode_hd(hs, 64)
    st = [int(h) for h in hs]
    words = np.array([oracle.wyrng_words(s, 1)[0] for s in st[:200]], dtype=np.uint64)
    assert a.dtype == np.int16 and words.size == 200  # smoke: wrapping path executes
    b = oracle.encode_hd_avx2_intrinsics(hs, 64)
    assert np.array_equal(a, b)


def test_bitpack_roundtrip_and_layout(oracle):
    rng = np.random.default_rng(5)
    for b in range(6, 16):
        lo, hi = -(1 << (b - 1)), (1 << (b - 1)) - 1
        hv = rng.integers(lo, hi + 1, 512).astype(np.int16)
        hv[0], hv[1] = lo, hi
        bb, packed = oracle.compress_hd_sketch(hv)
        assert bb == b and packed.size == b * 512 // 8
        assert np.array_equal(oracle.decompress_hd_sketch(packed, 512, b), hv)
        # published BitPacker8x layout: lane l = idx % 8, row r = idx / 8; word j of the lane
        # stream at byte 32 j + 4 l of the block
        u = (hv[:256].astype(np.int64) + (1 << (b - 1)))
        for l in (0, 3, 7):
            stream = 0
            for r in range(32):
                stream |= int(u[8 * r + l]) << (b * r)
            for j in range(b):
                w = int.from_bytes(packed[32 * j + 4 * l:32 * j + 4 * l + 4].tobytes(), "little")
                assert w == (stream >> (32 * j)) & 0xFFFFFFFF
    assert oracle.compress_hd_sketch(np.zeros(256, np.int16))[0] == 6


def test_synthetic_probe_golden(oracle):
    from hypergen_b200 import synth
    g = synth.genome(0xB200, 5_000_000).numpy()
    assert bytes(g[:20]) == b"TACGTTCTTTCAACGAGCAT"
    case = _load("synthetic_probe.json")["cases"][0]
    hs = oracle.kmer_hash_set(g, scaled=case["scaled"])
    assert hs.size == case["n_hashes"] == 3428
    assert [int(x) for x in hs[:3]] == case["smallest_hashes"] == [0x47B6159ADB3, 0x72335081133, 0xB60DD5A31F1]
    hv = oracle.encode_hd(hs, case["hv_d"])
    assert [int(x) for x in hv[:4]] == [-44, -8, -90, -58]
    assert (int(hv.min()), int(hv.max())) == (-238, 234)
    assert oracle.hv_l2_norm_sq(hv) == case["norm2"] == 14209484
    b, packed = oracle.compress_hd_sketch(hv)
    assert b == 9 and hashlib.sha256(packed.tobytes()).hexdigest() == case["packed_sha256"]


def test_config1_fixture(oracle):
    fna = b">test\nAGCTCTTANNAGCCCNTTacgttacagccctgaaaacttt"
    seq = oracle.read_merge_seq(fna)
    assert bytes(seq) == b"NAGCTCTTANNAGCCCNTTacgttacagccctgaaaacttt"
    assert oracle.kmer_hash_set(seq).size == 0
    assert [int(x) for x in oracle.kmer_hash_set(seq, scaled=1)] == [
        0x908794018D1F0246, 0x967BDE3C7BCDBCBA, 0xC0BD0CEE44A5F3E0, 0xE003C78B7D4BACE3]
    sk = oracle.sketch_batch(seq, np.array([0, seq.size], np.uint64))
    assert sk["quant_bits"][0] == 6 and sk["norm2"][0] == 0 and not sk["hv"].any()
    ani, _ = oracle.dist_all(sk["hv"], sk["norm2"], sk["hv"], sk["norm2"], symmetric=True)
    assert ani.size == 0  # 1 * (1 - 1) / 2 pairs: empty output file


def test_logf_restatement_matches_host_libm(oracle):
    # exhaustive over all positive floats was run once (0 mismatches, see DESIGN.md); here a stride
    assert oracle.logf_selfcheck(0, 0x7F800001, 4099) == 0
    assert oracle.logf_selfcheck(0x3F000000, 0x3F900000, 1) == 0   # the whole ANI-relevant band
    assert oracle.logf_selfcheck(0x80000000, 0xFFFFFFFF, 65537) == 0


def test_ani_formula_edges(oracle):
    f = oracle.ani_from_dot
    assert f(0, 0, 0) == 0.0                      # 0/0 -> NaN -> 0
    assert f(100, 100, 100) == np.float32(100.0)  # J = 1
    assert f(-5, 100, 100) == 0.0                 # ln(negative) -> NaN -> 0
    assert f(0, 100, 100) == 0.0                  # ln(0) = -inf -> clamp
    j = np.float32(50) / np.float32(150)
    want = np.float32(1) + np.float32(np.log(np.float32(2) / (np.float32(1) / j + np.float32(1)))) / np.float32(21)
    assert abs(float(f(50, 100, 100)) - float(want) * 100) < 1e-4


def test_output_order_and_format(oracle):
    ani = np.array([90.0, 85.0, 99.5, 85.0, 10.0, 99.5], np.float32)
    order = oracle.ani_output_order(ani, 85.0)
    assert list(order) == [5, 2, 0, 3, 1]  # descending ANI, ties by descending pair index
    pairs = oracle.pair_indices(4, 4, True)
    assert [tuple(p) for p in pairs] == [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]
    txt = oracle.format_ani_tsv(list("abcd"), list("abcd"), pairs, ani, order)
    assert txt.splitlines()[0] == "c\td\t99.500"
