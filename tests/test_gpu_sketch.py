"""GPU parity: the CUDA sketch path (through the C ABI) vs the CPU oracle, bit for bit.

Reference behaviour under test: src/sketch.rs:71-98 (hash set), src/hd.rs:15-92 (AVX2 HV
layout), src/dist.rs:132-137 (norm), src/hd.rs:116-157 (quantise + BitPacker8x bytes)."""
import numpy as np
import pytest

from conftest import random_dna

pytestmark = pytest.mark.gpu


def _batch(seqs, lead=0):
    """concatenate with `lead` junk bytes in front so genome starts are unaligned"""
    parts, off, pos = [], [lead], lead
    if lead:
        parts.append(np.full(lead, ord("A"), np.uint8))
    for s in seqs:
        parts.append(s)
        pos += s.size
        off.append(pos)
    seq = np.concatenate(parts) if parts else np.zeros(0, np.uint8)
    return seq, np.array(off, np.uint64)


def _oracle_sets(O, seq, off, **kw):
    return [O.kmer_hash_set(seq[int(off[g]):int(off[g + 1])], **kw) for g in range(off.size - 1)]


@pytest.mark.parametrize("k", [1, 2, 5, 8, 9, 15, 16, 17, 21, 24, 25, 31, 32])
@pytest.mark.parametrize("canonical", [True, False])
def test_kmer_hash_set_matches_oracle_all_k(ctx, hg, oracle, k, canonical):
    rng = np.random.default_rng(100 + k)
    seqs = [random_dna(rng, 30011, p_n=0.002, p_lower=0.05), random_dna(rng, 9000), random_dna(rng, 64)]
    seq, off = _batch(seqs, lead=3)
    scaled = 20 if k > 6 else 1
    p = hg.make_params(k=k, scaled=scaled, canonical=canonical)
    hashes, hoff = ctx.kmer_hash(seq, off, p)
    want = _oracle_sets(oracle, seq, off, k=k, scaled=scaled, canonical=canonical)
    for g, w in enumerate(want):
        got = hashes[int(hoff[g]):int(hoff[g + 1])]
        assert got.size == w.size, (k, canonical, g)
        assert np.array_equal(got, w), (k, canonical, g)


def test_kmer_hash_edge_cases(ctx, hg, oracle):
    """empty / shorter-than-k / all-N / every byte value / tile-boundary lengths / duplicates"""
    rng = np.random.default_rng(7)
    tile = 8192
    junk = random_dna(rng, 50000, p_junk=0.01)
    junk[:256] = np.arange(256, dtype=np.uint8)  # every byte value at least once
    rep = np.tile(random_dna(rng, 137), 300)      # heavy duplication: the set must collapse it
    seqs = [np.zeros(0, np.uint8), random_dna(rng, 20), random_dna(rng, 21), np.full(5000, ord("N"), np.uint8), junk,
            rep, random_dna(rng, tile), random_dna(rng, tile + 20), random_dna(rng, tile + 21),
            random_dna(rng, 2 * tile + 19), random_dna(rng, 1)]
    for lead in (0, 1, 15):
        seq, off = _batch(seqs, lead=lead)
        p = hg.make_params(k=21, scaled=7)
        hashes, hoff = ctx.kmer_hash(seq, off, p)
        want = _oracle_sets(oracle, seq, off, k=21, scaled=7)
        for g, w in enumerate(want):
            assert np.array_equal(hashes[int(hoff[g]):int(hoff[g + 1])], w), (lead, g)


def test_u_and_iupac_bytes_break_kmers_like_the_reference_gpu_path(ctx, hg, oracle):
    """Which reference semantics are reproduced: those of the reference's GPU path (src/cuda_kernel.cu:272-296) - only
    ACGT / acgt are bases; U, IUPAC codes and anything else end the k-mer run.  needletail's normalize() on the CPU path
    (src/sketch.rs:84) would map U/u to T instead: a sequence with U therefore sketches differently there (documented
    deviation, DESIGN.md 2) - here it must equal the same sequence with every U replaced by N, not by T."""
    rng = np.random.default_rng(21)
    s = random_dna(rng, 60_000)
    pos = rng.choice(s.size, 400, replace=False)
    s_u = s.copy()
    s_u[pos] = np.frombuffer(b"UuRYKMSWBDHVryn-*", np.uint8)[rng.integers(0, 17, pos.size)]
    s_n, s_t = s_u.copy(), s_u.copy()
    s_n[pos] = ord("N")
    s_t[pos] = ord("T")
    p = hg.make_params(k=21, scaled=5)
    off = np.array([0, s.size], np.uint64)
    got, _ = ctx.kmer_hash(s_u, off, p)
    as_n, _ = ctx.kmer_hash(s_n, off, p)
    as_t, _ = ctx.kmer_hash(s_t, off, p)
    assert np.array_equal(got, as_n) and not np.array_equal(got, as_t)
    assert np.array_equal(got, _oracle_sets(oracle, s_u, off, k=21, scaled=5)[0])
    if oracle.ref() is not None:  # the reference kernel itself (host build) agrees, capacity drops aside
        ref = oracle.ref_kmer_hash_set(s_u, k=21, scaled=5)
        assert np.isin(ref, got).all()


def test_kmer_hash_matches_reference_kernel_compiled_for_host(ctx, hg):
    """The reference's own cuda_kmer_t1ha2 (compiled as host code) agrees too: its hash sets of one genome with an N run
    and a lower-case stretch, at three (k, scaled) and both strand modes, are stored in golden/kmer_ref_sets.json."""
    import hashlib
    import json
    import os
    from hypergen_b200 import synth
    with open(os.path.join(os.path.dirname(__file__), "golden", "kmer_ref_sets.json")) as f:
        sets = json.load(f)["sets"]
    g = synth.genome(0xB200 + 77, 60_000).numpy().copy()
    g[5000:5030] = ord("N")
    g[20000:26000] |= 0x20
    off = np.array([0, g.size], np.uint64)
    assert len(sets) == 6
    for name, c in sets.items():
        hashes, _ = ctx.kmer_hash(g, off, hg.make_params(k=c["k"], scaled=c["scaled"], canonical=c["canonical"]))
        assert hashes.size == c["n"], name
        assert [int(x) for x in hashes[:4]] == c["head"], name
        assert hashlib.sha256(hashes.tobytes()).hexdigest() == c["sha256"], name


@pytest.mark.parametrize("hv_d,scaled", [(256, 200), (1024, 1500), (4096, 1500), (8192, 500), (4096, 60)])
def test_sketch_batch_bit_exact(ctx, hg, oracle, hv_d, scaled):
    from hypergen_b200 import synth
    rng = np.random.default_rng(hv_d + scaled)
    seqs = [synth.family_member(g, 300_000).numpy() for g in (0, 1, 7, 13)]
    seqs += [random_dna(rng, 70_001, p_n=0.001, p_lower=0.3), np.zeros(0, np.uint8), random_dna(rng, 20)]
    seq, off = _batch(seqs, lead=5)
    p = hg.make_params(scaled=scaled, hv_d=hv_d)
    got = ctx.sketch_batch(seq, off, p)
    want = oracle.sketch_batch(seq, off, scaled=scaled, hv_d=hv_d)
    assert np.array_equal(got["n_hashes"], want["n_hashes"])
    assert np.array_equal(got["hv"], want["hv"])            # AVX2 layout, wrapping i16
    assert np.array_equal(got["norm2"], want["norm2"])
    assert np.array_equal(got["quant_bits"], want["quant_bits"])
    for g in range(len(seqs)):
        nb = int(want["quant_bits"][g]) * hv_d // 8
        assert np.array_equal(got["packed"][g, :nb], want["packed"][g, :nb]), g
        assert not got["packed"][g, nb:].any()
    # decompress_hd_sketch on the GPU is the inverse
    back = ctx.unpack(got["packed"], got["quant_bits"], hv_d)
    assert np.array_equal(back, want["hv"])


def test_config1_test_fna_fixture(ctx, hg, oracle):
    """BASELINE config 1: test/test.fna -> empty set, all-zero HV, b = 6, norm 0 (SURVEY 8c)."""
    fna = b">test\nAGCTCTTANNAGCCCNTTacgttacagccctgaaaacttt"
    seq = oracle.read_merge_seq(fna)
    got = ctx.sketch_batch(seq, np.array([0, seq.size], np.uint64), hg.make_params())
    assert got["n_hashes"][0] == 0 and got["quant_bits"][0] == 6 and got["norm2"][0] == 0
    assert not got["hv"].any()
    # every 6-bit field holds the offset 32
    assert np.array_equal(oracle.decompress_hd_sketch(got["packed"][0, :6 * 4096 // 8], 4096, 6), np.zeros(4096, np.int16))
    # with scaled = 1 the four canonical 21-mers hash to the survey's values
    h, _ = ctx.kmer_hash(seq, np.array([0, seq.size], np.uint64), hg.make_params(scaled=1))
    assert [int(x) for x in h] == [0x908794018D1F0246, 0x967BDE3C7BCDBCBA, 0xC0BD0CEE44A5F3E0, 0xE003C78B7D4BACE3]


def test_full_size_genome_golden(ctx, hg):
    """One 5 Mbp synthetic genome at the headline parameters against the committed golden values."""
    import json, os
    from hypergen_b200 import synth
    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "synthetic_probe.json")))
    g = synth.genome(0xB200, 5_000_000).numpy()
    off = np.array([0, g.size], np.uint64)
    for case in gold["cases"]:
        p = hg.make_params(scaled=case["scaled"], hv_d=case["hv_d"])
        got = ctx.sketch_batch(g, off, p)
        assert int(got["n_hashes"][0]) == case["n_hashes"]
        assert int(got["quant_bits"][0]) == case["quant_bits"]
        assert int(got["norm2"][0]) == case["norm2"]
        assert [int(x) for x in got["hv"][0, :8]] == case["hv_head"]
        import hashlib
        assert hashlib.sha256(got["hv"][0].tobytes()).hexdigest() == case["hv_sha256"]
        nb = case["quant_bits"] * case["hv_d"] // 8
        assert hashlib.sha256(got["packed"][0, :nb].tobytes()).hexdigest() == case["packed_sha256"]


def test_invalid_arguments_return_status(ctx, hg):
    seq = np.frombuffer(b"ACGT" * 100, np.uint8)
    off = np.array([0, 400], np.uint64)
    for bad in (hg.make_params(k=0), hg.make_params(k=33), hg.make_params(hv_d=100), hg.make_params(scaled=0)):
        with pytest.raises(hg.HyperGenError) as e:
            ctx.sketch_batch(seq, off, bad)
        assert e.value.code == hg.ffi.HG_E_INVALID


def test_large_genome_and_many_small_ones(ctx, hg, oracle):
    """One 60 Mbp genome (long N runs, lower-case islands) next to 300 tiny ones in a single batch:
    exercises many tiles per genome, tables of different sizes and zero-tile genomes."""
    from hypergen_b200 import synth
    rng = np.random.default_rng(21)
    big = synth.genome(0xB200 + 99, 60_000_000).numpy().copy()
    for s in rng.integers(0, big.size - 200_000, 40):
        big[s:s + int(rng.integers(1, 150_000))] = ord("N")
    for s in rng.integers(0, big.size - 50_000, 60):
        big[s:s + 40_000] |= 0x20
    small = [random_dna(rng, int(rng.integers(0, 3000)), p_n=0.01) for _ in range(300)]
    seq, off = _batch([big] + small + [big[:1_000_003]], lead=7)
    p = hg.make_params()
    got = ctx.sketch_batch(seq, off, p)
    want = oracle.sketch_batch(seq, off)
    assert np.array_equal(got["n_hashes"], want["n_hashes"]) and got["n_hashes"][0] > 30000
    assert np.array_equal(got["hv"], want["hv"])
    assert np.array_equal(got["norm2"], want["norm2"]) and np.array_equal(got["quant_bits"], want["quant_bits"])
    h, hoff = ctx.kmer_hash(seq, off, p)
    assert np.array_equal(h[: int(hoff[1])], oracle.kmer_hash_set(big))
