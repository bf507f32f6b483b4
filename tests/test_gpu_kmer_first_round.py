"""GPU parity of t1ha2's first round, which the k-mer kernel takes from product tables for K >= 8.

Word 0 of such a k-mer is the ASCII of its first 8 bases, so a de Bruijn sequence B(4, 8) hashes every one of the
4^8 possible words 0.  The seeds cover the carries the table formulation has to get right: Y + w0 wrapping past 2^64
(for about half of all words 0, for all of them, for none), a carry from the low into the high 32 bits of Y + w0
without a wrap, and a seed in the X role with both halves set."""
import numpy as np
import pytest

from conftest import random_dna

pytestmark = pytest.mark.gpu

M64 = (1 << 64) - 1
SEEDS = [0, 123, (1 << 32) - 1, 1 << 32, M64,
         (1 << 64) - 0x4747474747474747,  # Y + w0 wraps for about half of all words 0
         (1 << 32) - 0x47474747,          # carry from the low word into the high word, no wrap
         0x9E3779B97F4A7C15, 0xF1357AEA2E62A9C5]
WRAP_SEED, PLAIN_SEED = (1 << 64) - 0x4747474747474747, 0x9E3779B97F4A7C15


def _de_bruijn_acgt(n):
    """cyclic B(4, n) over ACGT (every n-base word exactly once), as a list of base values 0..3"""
    a, out = [0] * (n + 1), []

    def db(t, p):
        if t > n:
            if n % p == 0:
                out.extend(a[1:p + 1])
        else:
            a[t] = a[t - p]
            db(t + 1, p)
            for j in range(a[t - p] + 1, 4):
                a[t] = j
                db(t + 1, t)

    db(1, 1)
    return out


def test_de_bruijn_covers_every_first_word():
    b = np.array(_de_bruijn_acgt(8), np.int64)
    assert b.size == 4 ** 8
    ext = np.concatenate([b, b[:7]])
    words = sum(ext[i:i + b.size] << (2 * i) for i in range(8))
    assert np.unique(words).size == 4 ** 8


@pytest.mark.parametrize("canonical", [False, True])
@pytest.mark.parametrize("k", [8, 9, 16, 17, 21, 24, 25, 32])
def test_every_first_word_every_seed(ctx, hg, oracle, k, canonical):
    """scaled = 1 keeps every hash: the GPU set equals the oracle's for all 4^8 words 0 (as forward k-mers; the
    canonical run hashes whichever strand is smaller)"""
    b = _de_bruijn_acgt(8)
    seq = np.frombuffer(b"ACGT", np.uint8)[np.array(b + b[:k - 1])]
    off = np.array([0, seq.size], np.uint64)
    for seed in SEEDS:
        p = hg.make_params(k=k, scaled=1, seed=seed, canonical=canonical)
        got, _ = ctx.kmer_hash(seq, off, p)
        want = oracle.kmer_hash_set(seq, k=k, scaled=1, seed=seed, canonical=canonical)
        assert got.size == want.size and np.array_equal(got, want), (k, canonical, hex(seed))


@pytest.mark.parametrize("seed", [WRAP_SEED, PLAIN_SEED])
@pytest.mark.parametrize("k", [8, 16, 21, 32])
def test_random_genomes_sketch_bit_exact(ctx, hg, oracle, k, seed):
    """N runs, lower case, unaligned starts: the hash sets and the full sketch outputs equal the oracle's"""
    rng = np.random.default_rng(7000 + k)
    seqs = [random_dna(rng, 30011, p_n=0.002, p_lower=0.05), random_dna(rng, 9000), random_dna(rng, 64),
            random_dna(rng, 200_003, p_n=0.001, p_lower=0.2)]
    lead = 5
    seq = np.concatenate([np.full(lead, ord("A"), np.uint8)] + seqs)
    off = np.cumsum([lead] + [s.size for s in seqs]).astype(np.uint64)
    scaled = 20
    p = hg.make_params(k=k, scaled=scaled, seed=seed, canonical=True, hv_d=4096)
    hashes, hoff = ctx.kmer_hash(seq, off, p)
    for g in range(len(seqs)):
        want = oracle.kmer_hash_set(seq[int(off[g]):int(off[g + 1])], k=k, scaled=scaled, seed=seed)
        assert np.array_equal(hashes[int(hoff[g]):int(hoff[g + 1])], want), (k, hex(seed), g)
    got = ctx.sketch_batch(seq, off, p)
    want = oracle.sketch_batch(seq, off, k=k, scaled=scaled, seed=seed, hv_d=4096)
    assert np.array_equal(got["hv"], want["hv"])
    assert np.array_equal(got["norm2"], want["norm2"]) and np.array_equal(got["quant_bits"], want["quant_bits"])
    assert np.array_equal(got["n_hashes"], want["n_hashes"])
    for g in range(len(seqs)):
        nb = int(want["quant_bits"][g]) * 4096 // 8
        assert np.array_equal(got["packed"][g, :nb], want["packed"][g, :nb]), (k, hex(seed), g)
