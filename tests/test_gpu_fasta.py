"""GPU parity for the FASTA-bytes entry points: hg_fasta_merge == fastx_reader::read_merge_seq
(reference src/fastx_reader.rs:6-29, restated in the oracle), and sketches from raw files equal
sketches from the merged sequences."""
import numpy as np
import pytest

from conftest import random_dna

pytestmark = pytest.mark.gpu


def _fasta(seq, name=b"g", width=80, eol=b"\n", records=1, final_eol=True):
    out = bytearray()
    per = max(len(seq) // records, 1)
    for r in range(records):
        part = bytes(seq[r * per:(r + 1) * per if r < records - 1 else len(seq)])
        out += b">" + name + b"_%d some text" % r + eol
        for i in range(0, len(part), width):
            out += part[i:i + width] + eol
    if not final_eol and out.endswith(eol):
        out = out[:-len(eol)]
    return bytes(out)


def _assert_sketches_equal(got, want, hv_d):
    assert np.array_equal(got["n_hashes"], want["n_hashes"])
    assert np.array_equal(got["hv"], want["hv"]) and np.array_equal(got["norm2"], want["norm2"])
    assert np.array_equal(got["quant_bits"], want["quant_bits"])
    for g in range(want["quant_bits"].size):  # the live bytes of each packed row
        nb = int(want["quant_bits"][g]) * hv_d // 8
        assert np.array_equal(got["packed"][g, :nb], want["packed"][g, :nb]), g


def test_fasta_merge_matches_reference_reader(ctx, hg, oracle):
    rng = np.random.default_rng(8)
    s = random_dna(rng, 30_000, p_n=0.01, p_lower=0.1)
    files = [
        _fasta(s), _fasta(s, eol=b"\r\n"), _fasta(s, width=7, records=5), _fasta(s, final_eol=False),
        _fasta(s, eol=b"\r\n", final_eol=False), _fasta(s, width=60_000),           # one 30 kB line (> 7 blocks)
        b"", b">only header", b">only header\n", b"ACGT", b"ACGT\r", b"\n\n\nAC\n\nGT\n", b"AC>GT\nA\rC\r\nGG\r",
        b">" + b"x" * 10_000 + b"\nACGTACGT\n",                                     # header longer than a block
        b">h1\n>h2\n>h3\nAAAA\n", b"\r\n\r\n>h\r\nCC\r\n",
        _fasta(random_dna(rng, 4096 * 3 - 5), width=4095),                           # line ends around block edges
        _fasta(random_dna(rng, 4096 * 2), width=4096), bytes(random_dna(rng, 4096)) + b"\n>x\n" + bytes(random_dna(rng, 5000)),
    ]
    got = ctx.fasta_merge(files)
    for f, g in zip(files, got):
        want = oracle.read_merge_seq(f)
        assert bytes(g) == bytes(want), f[:60]


def test_sketch_from_raw_fasta_equals_sketch_from_merged(ctx, hg, oracle):
    from hypergen_b200 import synth
    files = []
    for g in range(6):
        seq = synth.family_member(g + 30, 200_000 + 1111 * g).numpy()
        files.append(_fasta(seq, width=80 if g % 2 else 61, eol=b"\r\n" if g == 3 else b"\n", records=1 + g % 3))
    files.append(b"")
    p = hg.make_params(scaled=300, hv_d=1024)
    got = ctx.sketch_fasta_batch(files, p)
    seqs = [oracle.read_merge_seq(f) for f in files]
    off = np.cumsum([0] + [s.size for s in seqs]).astype(np.uint64)
    want = oracle.sketch_batch(np.concatenate(seqs), off, scaled=300, hv_d=1024)
    _assert_sketches_equal(got, want, 1024)


def test_raw_fasta_chunk_pipeline(ctx, hg, oracle, monkeypatch):
    """Several 1 MB chunks through the double-buffered copy/merge/hash/encode pipeline, with files
    whose merged length is far below the raw size the tiles were planned from (long headers, a file
    that is all header, a merged length below k); then the merged sequences of the same files through
    the sequence entry's chunks, which start at several alignments modulo 16."""
    from hypergen_b200 import synth
    monkeypatch.setenv("HG_CHUNK_MB", "1")
    rng = np.random.default_rng(77)
    files = []
    for g in range(14):
        seq = synth.family_member(g + 90, 150_000 + 40_001 * (g % 5)).numpy()
        files.append(_fasta(seq, width=70 + g, records=1 + g % 4))
    files.insert(3, b">" + b"h" * 300_000 + b"\n" + bytes(random_dna(rng, 5000)) + b"\n")
    files.insert(7, b">" + b"h" * 100_000)
    files.insert(9, b">x\nACGTACGTAC\n")
    files.insert(11, _fasta(random_dna(rng, 1_500_000, p_n=0.001)))       # a file larger than the chunk size
    p = hg.make_params(scaled=200, hv_d=2048)
    got = ctx.sketch_fasta_batch(files, p)
    seqs = [oracle.read_merge_seq(f) for f in files]
    off = np.cumsum([0] + [s.size for s in seqs]).astype(np.uint64)
    want = oracle.sketch_batch(np.concatenate(seqs), off, scaled=200, hv_d=2048)
    _assert_sketches_equal(got, want, 2048)
    again = ctx.sketch_fasta_batch(files, p)                                # scratch reuse across calls
    assert np.array_equal(again["hv"], want["hv"])

    lead = 5                                                                # bytes before the first genome
    buf = np.concatenate([np.full(lead, ord("N"), np.uint8)] + seqs)
    seq_off = off + np.uint64(lead)
    starts, g = [], 0                                                       # chunk starts: genome boundaries, <= 1 MB a chunk
    while g < len(seqs):
        starts.append(int(seq_off[g]))
        g += 1
        while g < len(seqs) and int(seq_off[g + 1]) - starts[-1] <= 1 << 20:
            g += 1
    assert len(starts) > 2 and len({(buf.ctypes.data + s) % 16 for s in starts}) > 1
    _assert_sketches_equal(ctx.sketch_batch(buf, seq_off, p), want, 2048)
