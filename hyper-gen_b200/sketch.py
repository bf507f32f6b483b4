"""Host mirror of sketch_cuda::sketch_cuda (reference src/sketch_cuda.rs:43-117): discover
FASTA files, read them, sketch the whole batch through one C-ABI call, write the sketch file."""
from __future__ import annotations

import os
import re
from dataclasses import dataclass

import numpy as np

from . import fileio
from .ffi import Context, make_params


@dataclass
class SketchParams:
    """types.rs:83-113 (defaults included)"""
    path: str = ""
    out_file: str = ""
    canonical: bool = True
    ksize: int = 21
    seed: int = 123
    scaled: int = 1500
    hv_d: int = 4096
    individual: bool = False  # one sketch per FASTA record (`hyper-gen sketch -i true`) instead of one per file


def sketch_sequences(ctx: Context, seqs: list[np.ndarray], names: list[str], p: SketchParams,
                     batch_bytes: int = 1 << 30) -> list[fileio.FileSketch]:
    """Sketch in-memory sequences in batches of at most `batch_bytes` of sequence."""
    out: list[fileio.FileSketch] = []
    params = make_params(k=p.ksize, scaled=p.scaled, seed=p.seed, canonical=p.canonical, hv_d=p.hv_d)
    start = 0
    while start < len(seqs):
        end, tot = start, 0
        while end < len(seqs) and (end == start or tot + seqs[end].size <= batch_bytes):
            tot += seqs[end].size
            end += 1
        sizes = np.array([0] + [s.size for s in seqs[start:end]], np.uint64)
        seg_off = np.cumsum(sizes).astype(np.uint64)
        seq = np.concatenate(seqs[start:end]) if tot else np.zeros(0, np.uint8)
        r = ctx.sketch_batch(seq, seg_off, params, want_hv=False)
        for t in range(end - start):
            b = int(r["quant_bits"][t])
            nbytes = b * p.hv_d // 8
            out.append(fileio.FileSketch(p.ksize, p.scaled, p.canonical, p.seed, p.hv_d, b, int(r["norm2"][t]),
                                         names[start + t], r["packed"][t, :nbytes].copy().view("<i2")))
        start = end
    return out


def record_id(path: str, header: bytes, has_header: bool, index: int) -> str:
    """The name of a record's sketch: its header text up to the first space or tab; `<file path>#<index of the record
    in its file, from 0>` for a leading record (sequence before the first header) or an empty ID."""
    rid = re.split(rb"[ \t]", header, maxsplit=1)[0] if has_header else b""
    return rid.decode("utf-8", "replace") if rid else "%s#%d" % (path, index)


def sketch_records(ctx: Context, files: list[str], p: SketchParams, batch_bytes: int = 1 << 30) -> list[fileio.FileSketch]:
    """One sketch per record of every file, from the raw file bytes (hg_sketch_fasta_records), in batches of at most
    `batch_bytes` of file bytes."""
    out: list[fileio.FileSketch] = []
    params = make_params(k=p.ksize, scaled=p.scaled, seed=p.seed, canonical=p.canonical, hv_d=p.hv_d)
    start = 0
    while start < len(files):
        datas, tot = [], 0
        while start + len(datas) < len(files) and (not datas or tot + os.path.getsize(files[start + len(datas)]) <= batch_bytes):
            with open(files[start + len(datas)], "rb") as f:
                datas.append(f.read())
            tot += len(datas[-1])
        base = np.cumsum([0] + [len(d) for d in datas])
        r = ctx.sketch_fasta_records(datas, params)
        prev, index = -1, 0
        for t, rec in enumerate(r["records"]):
            f = int(rec["file"])
            index = index + 1 if f == prev else 0
            prev = f
            a = int(rec["name_off"]) - int(base[f])
            name = record_id(files[start + f], datas[f][a:a + int(rec["name_len"])], bool(rec["has_header"]), index)
            b = int(r["quant_bits"][t])
            out.append(fileio.FileSketch(p.ksize, p.scaled, p.canonical, p.seed, p.hv_d, b, int(r["norm2"][t]), name,
                                         r["packed"][t, :b * p.hv_d // 8].copy().view("<i2")))
        start += len(datas)
    return out


def sketch(p: SketchParams, ctx: Context | None = None) -> list[fileio.FileSketch]:
    own = ctx is None
    ctx = ctx or Context(0)
    try:
        files = fileio.get_fasta_files(p.path)
        if p.individual:
            sk = sketch_records(ctx, files, p)
        else:
            seqs = [fileio.read_merge_seq(f) for f in files]
            sk = sketch_sequences(ctx, seqs, files, p)
        if p.out_file:
            fileio.dump_sketch(sk, p.out_file)
        return sk
    finally:
        if own:
            ctx.close()
