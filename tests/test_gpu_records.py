"""One sketch per FASTA record (hg_sketch_fasta_records): every record's row equals the per-file entry's row for a file
holding that record alone, and the oracle's; the record table equals a host parse; the chunked pipeline, the contract
edges, the group entry and `hyper-gen sketch -i true`."""
import ctypes as C
import os
import subprocess

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


def _merge(data):
    from hypergen_b200 import fileio
    return fileio.merge_seq_bytes(data)


def split_records(data):
    """The contract's records of one file by a host parse: [(one-record file bytes, has_header, name_off, name_len,
    seq_len)], name_off relative to the file."""
    starts = [0] + [i + 1 for i in range(len(data)) if data[i] == 0x0A and i + 1 < len(data)]
    hdr = [s for s in starts if data[s:s + 1] == b">"]
    out = []
    lead = data[:hdr[0]] if hdr else data
    if _merge(lead).size:
        out.append((lead, 0, 0, 0, _merge(lead).size))
    for t, s in enumerate(hdr):
        body = data[s:hdr[t + 1] if t + 1 < len(hdr) else len(data)]
        nl = data.find(b"\n", s)
        end = len(data) if nl < 0 else nl
        name_len = end - s - 1 - (1 if nl >= 0 and end > s + 1 and data[end - 1:end] == b"\r" else 0)
        out.append((body, 1, s + 1, name_len, _merge(body).size - 1))
    return out


def _expect(files):
    """(one-record files, expected table) of the records of `files`, in file order"""
    one, table, base = [], [], 0
    for f, data in enumerate(files):
        for body, has, noff, nlen, slen in split_records(data):
            one.append(body)
            table.append((base + noff if has else base, nlen, slen, f, has))
        base += len(data)
    return one, table


def _rows_equal(got, want, hv_d, rows=None):
    rows = range(want["quant_bits"].size) if rows is None else rows
    for key in ("n_hashes", "norm2", "quant_bits"):
        if key in got and key in want:
            assert np.array_equal(got[key], want[key]), key
    for g in rows:
        nb = int(want["quant_bits"][g]) * hv_d // 8
        assert np.array_equal(got["packed"][g, :nb], want["packed"][g, :nb]), g


def _check_records(ctx, oracle, files, p, oracle_too=True):
    got = ctx.sketch_fasta_records(files, p)
    one, table = _expect(files)
    rec = got["records"]
    assert rec.size == len(table)
    assert [tuple(int(x) for x in r) for r in rec.tolist()] == table
    if not one:
        return got
    want = ctx.sketch_fasta_batch(one, p, want_hv=False)
    _rows_equal(got, want, int(p.hv_d))
    if oracle_too:
        seqs = [oracle.read_merge_seq(f) for f in one]
        off = np.cumsum([0] + [s.size for s in seqs]).astype(np.uint64)
        ref = oracle.sketch_batch(np.concatenate(seqs) if off[-1] else np.zeros(0, np.uint8), off, k=int(p.ksize),
                                  scaled=int(p.scaled), seed=int(p.seed), canonical=bool(p.canonical), hv_d=int(p.hv_d),
                                  want_hv=False)
        _rows_equal(got, ref, int(p.hv_d))
    return got


def _corpus(rng):
    s = random_dna(rng, 30_000, p_n=0.01, p_lower=0.1)
    return [
        _fasta(s), _fasta(s, eol=b"\r\n"), _fasta(s, width=7, records=5), _fasta(s, final_eol=False),
        _fasta(s, eol=b"\r\n", final_eol=False), _fasta(s, width=60_000),
        b"", b">only header", b">only header\n", b"ACGT", b"ACGT\r", b"\n\n\nAC\n\nGT\n", b"AC>GT\nA\rC\r\nGG\r",
        b">" + b"x" * 10_000 + b"\nACGTACGT\n",
        b">h1\n>h2\n>h3\nAAAA\n", b"\r\n\r\n>h\r\nCC\r\n",
        _fasta(random_dna(rng, 4096 * 3 - 5), width=4095),
        _fasta(random_dna(rng, 4096 * 2), width=4096), bytes(random_dna(rng, 4096)) + b"\n>x\n" + bytes(random_dna(rng, 5000)),
        _fasta(random_dna(rng, 50_000), width=61, records=17, eol=b"\r\n"),
        bytes(random_dna(rng, 300)) + b"\n" + _fasta(random_dna(rng, 9000), width=50, records=9),
        b">\n" + bytes(random_dna(rng, 200)) + b"\n>\r\n>  desc\nACGTAC\n>\r",
        b">" + b"h" * 300_000 + b"\n" + bytes(random_dna(rng, 5000)) + b"\n>y\nACGTTGCA\n",
    ]


def test_records_equal_split_files(ctx, hg, oracle):
    rng = np.random.default_rng(11)
    _check_records(ctx, oracle, _corpus(rng), hg.make_params(scaled=100, hv_d=1024))


def test_records_chunked_pipeline(ctx, hg, oracle, monkeypatch):
    """1 MB chunks: many files of many records, a file larger than a chunk with thousands of records, one file of more
    than 65 535 records; scratch reuse, and the per-file entry before and after a records call."""
    from hypergen_b200 import synth
    monkeypatch.setenv("HG_CHUNK_MB", "1")
    rng = np.random.default_rng(12)
    files = []
    for g in range(30):
        seq = synth.family_member(g + 200, 60_000 + 3_001 * g).numpy()
        files.append(_fasta(seq, name=b"f%d" % g, width=60 + g, records=10 + 3 * g))
    files.insert(5, _fasta(random_dna(rng, 1_500_000, p_n=0.001), width=70, records=3000))
    p = hg.make_params(scaled=200, hv_d=2048)
    seqs = [oracle.read_merge_seq(f) for f in files]
    off = np.cumsum([0] + [s.size for s in seqs]).astype(np.uint64)
    per_file = oracle.sketch_batch(np.concatenate(seqs), off, scaled=200, hv_d=2048, want_hv=False)
    _rows_equal(ctx.sketch_fasta_batch(files, p, want_hv=False), per_file, 2048)   # per-file, then records
    first = _check_records(ctx, oracle, files, p)
    again = ctx.sketch_fasta_records(files, p)                                     # scratch reuse
    for k in first:
        assert np.array_equal(first[k], again[k]), k
    _rows_equal(ctx.sketch_fasta_batch(files, p, want_hv=False), per_file, 2048)   # records, then per-file

    many = b"".join(b">r%d\n" % i + bytes(random_dna(rng, 24)) + b"\n" for i in range(70_000))
    assert len(many) > (1 << 20)
    got = _check_records(ctx, oracle, [b">a\nACGT\n", many, b"ACGTACGTACGT\n"], hg.make_params(k=9, scaled=1, hv_d=256))
    assert got["records"].size == 1 + 70_000 + 1  # the last file is one leading record
    assert np.count_nonzero(got["n_hashes"]) > 69_000


def test_records_contract_edges(ctx, hg, oracle):
    L = hg.ffi.load()
    rng = np.random.default_rng(13)
    files = [_fasta(random_dna(rng, 3000), records=4), b"ACGT\n>x\nAC\n", b"", b">only"]
    raw, off = hg.Context._concat_files(files)
    p = hg.make_params(scaled=10, hv_d=256)
    need = 4 + 2 + 1
    n_rec = C.c_uint32(0)
    rec = np.zeros(need + 2, hg.ffi.RECORD_DTYPE)
    rec["seq_len"] = 12345
    packed = np.full((need + 2, 512), 7, np.uint8)
    bits = np.full(need + 2, 7, np.uint8)
    norm2 = np.full(need + 2, 7, np.int32)
    nh = np.full(need + 2, 7, np.uint32)
    args = lambda cap: (ctx._h, raw.ctypes.data, off.ctypes.data, len(files), C.byref(p), cap, rec.ctypes.data,
                        packed.ctypes.data, bits.ctypes.data, norm2.ctypes.data, nh.ctypes.data, C.byref(n_rec))
    assert L.hg_sketch_fasta_records(*args(need - 1)) == hg.ffi.HG_E_CAPACITY
    assert n_rec.value == need
    assert (rec["seq_len"] == 12345).all() and (packed == 7).all() and (bits == 7).all() and (norm2 == 7).all() and (nh == 7).all()
    assert L.hg_sketch_fasta_records(*args(need)) == hg.ffi.HG_OK and n_rec.value == need
    assert rec["seq_len"][need] == 12345 and (packed[need:] == 7).all()
    g = hg.Group(ordinals=[0, 0])
    assert L.hg_group_sketch_fasta_records(g._h, *args(need - 1)[1:]) == hg.ffi.HG_E_CAPACITY and n_rec.value == need
    g.close()

    n_rec.value = 99
    assert L.hg_sketch_fasta_records(ctx._h, None, off.ctypes.data, 0, C.byref(p), 0, None, None, None, None, None,
                                     C.byref(n_rec)) == hg.ffi.HG_OK and n_rec.value == 0
    assert L.hg_sketch_fasta_records(ctx._h, None, off.ctypes.data, len(files), C.byref(p), need, None, None, None, None,
                                     None, C.byref(n_rec)) == hg.ffi.HG_E_INVALID
    bad = off.copy()
    bad[2] = bad[1] - 1
    assert L.hg_sketch_fasta_records(ctx._h, raw.ctypes.data, bad.ctypes.data, len(files), C.byref(p), need, None, None,
                                     None, None, None, C.byref(n_rec)) == hg.ffi.HG_E_INVALID
    assert L.hg_sketch_fasta_records(ctx._h, raw.ctypes.data, off.ctypes.data, len(files), C.byref(p), need, None, None,
                                     None, None, None, None) == hg.ffi.HG_E_INVALID

    short = [b">a\nACG\n>b\nACGTACGTACG\n>c\n" + bytes(random_dna(rng, 5000)) + b"\n>d\nA\n", b"AC\n>e\n" + bytes(random_dna(rng, 40))]
    for k, canon in ((1, True), (32, True), (21, False), (32, False)):
        _check_records(ctx, oracle, short + _corpus(rng)[:8], hg.make_params(k=k, scaled=20, hv_d=512, canonical=canon))


def test_records_group_matches_one_context(ctx, hg, oracle):
    rng = np.random.default_rng(14)
    files = _corpus(rng) + [_fasta(random_dna(rng, 20_000), records=40, name=b"q%d" % i) for i in range(6)]
    p = hg.make_params(scaled=100, hv_d=1024)
    one = ctx.sketch_fasta_records(files, p)
    lopsided = [_fasta(random_dna(rng, 400_000), records=3), b">a\nACGTACGTAC\n", b">b\nACGTACGTAC\n"]
    one_l = ctx.sketch_fasta_records(lopsided, p)
    for ordinals in ([0, 0], [0, 0, 0]):
        with hg.Group(ordinals=ordinals) as g:
            for fs, want in ((files, one), (lopsided, one_l)):   # lopsided: with 3 members the first gets no file
                got = g.sketch_fasta_records(fs, p)
                for k in want:
                    assert np.array_equal(got[k], want[k]), (ordinals, k)


def _write(d, name, data):
    with open(os.path.join(d, name), "wb") as f:
        f.write(data)


def test_cli_individual(ctx, hg, oracle, tmp_path):
    from hypergen_b200 import _build, fileio, sketch, synth
    exe = _build.build_host()
    rng = np.random.default_rng(15)
    d = tmp_path / "multi"
    d.mkdir()
    recs = {}  # record name -> its one-record file
    for g in range(5):
        data = _fasta(synth.family_member(g + 40, 90_000).numpy(), name=b"m%d" % g, records=1 + 2 * g)
        _write(d, "m%d.fna" % g, data)
        for t, (body, *_rest) in enumerate(split_records(data)):
            recs["m%d_%d" % (g, t)] = body
    lead = bytes(random_dna(rng, 700)) + b"\n>\tdesc only\n" + bytes(random_dna(rng, 900)) + b"\n>z9 x\n" + bytes(random_dna(rng, 800)) + b"\n"
    _write(d, "x.fa", lead)
    for t, (body, *_rest) in enumerate(split_records(lead)):
        recs[["%s#0" % (d / "x.fa"), "%s#1" % (d / "x.fa"), "z9"][t]] = body
    args = ["-s", "300", "-d", "1024", "-t", "4", "-i", "true"]
    out_cc, out_py, out_1 = str(tmp_path / "cc.sketch"), str(tmp_path / "py.sketch"), str(tmp_path / "one.sketch")
    subprocess.check_call([exe, "sketch", "-p", str(d), "-o", out_cc, *args])
    sketch.sketch(sketch.SketchParams(path=str(d), out_file=out_py, scaled=300, hv_d=1024, individual=True), ctx=ctx)
    subprocess.check_call([exe, "sketch", "-p", str(d), "-o", out_1, *args], env=dict(os.environ, HG_GPUS="1"))
    assert open(out_cc, "rb").read() == open(out_py, "rb").read() == open(out_1, "rb").read()
    sk = fileio.load_sketch(out_cc)
    assert [s.file_str for s in sk] == list(recs)  # IDs cut at a space or tab; `<file>#<index>` for lead / empty IDs

    # the split files: one record each, named so that their file order is the record order
    s = tmp_path / "split"
    s.mkdir()
    split_names = {}
    for t, (name, body) in enumerate(recs.items()):
        _write(s, "r%03d.fna" % t, body)
        split_names[str(s / ("r%03d.fna" % t))] = name
    out_s, out_si = str(tmp_path / "split.sketch"), str(tmp_path / "split_i.sketch")
    subprocess.check_call([exe, "sketch", "-p", str(s), "-o", out_s, *args[:-2]])
    subprocess.check_call([exe, "sketch", "-p", str(s), "-o", out_si, *args])
    per_file, per_rec = fileio.load_sketch(out_s), fileio.load_sketch(out_si)
    assert len(per_file) == len(sk) == len(per_rec)
    for a, b, c in zip(per_file, sk, per_rec):  # one-record files: every field but the name equals the per-file row
        assert split_names[a.file_str] == b.file_str
        assert (a.hv_quant_bits, a.hv_norm_2, a.hv.tobytes()) == (b.hv_quant_bits, b.hv_norm_2, b.hv.tobytes())
        assert (c.hv_quant_bits, c.hv_norm_2, c.hv.tobytes()) == (b.hv_quant_bits, b.hv_norm_2, b.hv.tobytes())
    tsv_i, tsv_s = str(tmp_path / "i.tsv"), str(tmp_path / "s.tsv")
    subprocess.check_call([exe, "dist", "-r", out_cc, "-q", out_cc, "-o", tsv_i, "-a", "0.0"])
    subprocess.check_call([exe, "dist", "-r", out_s, "-q", out_s, "-o", tsv_s, "-a", "0.0"])
    mapped = []
    for line in open(tsv_s).read().splitlines():
        a, b, ani = line.split("\t")
        mapped.append("\t".join((split_names[a], split_names[b], ani)))
    assert open(tsv_i).read().splitlines() == mapped and mapped

    r = subprocess.run([exe, "sketch", "-p", str(d), "-o", str(tmp_path / "hp.sketch"), *args], capture_output=True, text=True,
                       env=dict(os.environ, HG_HOST_PARSE="1"))
    assert r.returncode != 0 and "HG_HOST_PARSE" in r.stderr
