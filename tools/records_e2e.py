"""Time the per-record FASTA entry (hg_sketch_fasta_records) end to end from pinned host memory, on the same 5 GB of
sequence bytes in three layouts of 1000 files each (the bases of one 5 Mbp genome, 80-column lines):
  1. 1 record of 5 Mbp per file: hg_sketch_fasta_batch and hg_sketch_fasta_records alternating;
  2. 100 records of 50 kb per file;
  3. 5000 records of 1 kb per file.
The files go through in calls of --files-per-call files (the outputs of a call are pinned too: layout 3 returns 8 KB of
packed row per 1 KB record).  Prints one JSON line per measurement (and writes them all to --json if given):
records/s and GB/s of file bytes (best of --reps passes), then a separate profiled pass with the device ms of merge,
record index, k-mer hash and encode and the host gap, summed over its calls, and per chunk.  The card's name, power
limit and max SM clock are read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hypergen_b200 as hg  # noqa: E402
from hypergen_b200 import synth  # noqa: E402


def layout(seq, records):
    """one FASTA file: `records` records of equal length cut from seq, 80-column lines"""
    per = seq.size // records
    out = []
    for r in range(records):
        part = seq[r * per:(r + 1) * per]
        lines = part.reshape(-1, 80) if part.size % 80 == 0 else None
        out.append(np.frombuffer(b">rec%d sample\n" % r, np.uint8))
        if lines is not None:
            out.append(np.concatenate([lines, np.full((lines.shape[0], 1), 10, np.uint8)], axis=1).reshape(-1))
        else:
            for i in range(0, part.size, 80):
                out.append(part[i:i + 80])
                out.append(np.array([10], np.uint8))
    return np.concatenate(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=1000)
    ap.add_argument("--files-per-call", type=int, default=100)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--json", help="also write the measurements to this file")
    a = ap.parse_args()
    results = []

    def emit(d):
        print(json.dumps(d), flush=True)
        results.append(d)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    emit({"card": q[0] if q else torch.cuda.get_device_name(0)})
    ctx = hg.Context(0)
    lib = hg.ffi.load()
    p = hg.make_params()
    D = 4096
    seq = synth.genome(0xB200, 5_000_000).numpy()
    n, per_call = a.files, a.files_per_call
    files = {1: layout(seq, 1), 100: layout(seq, 100), 5000: layout(seq, 5000)}
    size = max(f.size for f in files.values())
    raw = torch.empty(size * per_call, dtype=torch.uint8).pin_memory()
    rn = raw.numpy()
    max_rec = 5000 * per_call
    packed = torch.empty((max_rec, 2 * D), dtype=torch.uint8).pin_memory()
    bits = torch.empty(max_rec, dtype=torch.uint8).pin_memory()
    norm = torch.empty(max_rec, dtype=torch.int32).pin_memory()
    nh = torch.empty(max_rec, dtype=torch.int32).pin_memory()
    rec = torch.empty(max_rec * 32, dtype=torch.uint8).pin_memory()
    n_rec = C.c_uint32(0)
    ptr = lambda t: C.c_void_p(t.data_ptr())

    def calls(one, records):
        """one pass over the n files (n / per_call calls on the same pinned buffer of per_call copies of `one`)"""
        off = (np.arange(per_call + 1, dtype=np.uint64) * one.size)
        for _ in range(n // per_call):
            if records:
                rc = lib.hg_sketch_fasta_records(ctx._h, ptr(raw), C.c_void_p(off.ctypes.data), per_call, C.byref(p), max_rec,
                                                 ptr(rec), ptr(packed), ptr(bits), ptr(norm), ptr(nh), C.byref(n_rec))
            else:
                rc = lib.hg_sketch_fasta_batch(ctx._h, ptr(raw), C.c_void_p(off.ctypes.data), per_call, C.byref(p), None,
                                               ptr(packed), ptr(bits), ptr(norm), ptr(nh))
            assert rc == 0, lib.hg_last_error()

    for r_per_file, one in files.items():
        for i in range(per_call):
            rn[i * one.size:(i + 1) * one.size] = one
        modes = [False, True] if r_per_file == 1 else [True]
        for m in modes:
            calls(one, m)  # warm-up
        best = {m: 1e30 for m in modes}
        for _ in range(a.reps):
            for m in modes:
                t = time.perf_counter()
                calls(one, m)
                best[m] = min(best[m], time.perf_counter() - t)
        n_rec_file = int(n_rec.value) // per_call
        for m in modes:
            t = best[m]
            emit({"layout": "%d files x %d records" % (n, r_per_file), "entry": "records" if m else "per-file",
                  "s": round(t, 4), "records_per_s": round(n * (n_rec_file if m else 1) / t),
                  "file_GB_per_s": round(n * one.size / t / 1e9, 2), "file_bytes": n * one.size,
                  "row_bytes_to_host": n * (n_rec_file if m else 1) * 2 * D})
        # profiled pass (a run of its own: the events and the reads of them cost host time)
        ctx.set_profiling(True)
        tot, gap, chunks = np.zeros(4), 0.0, 0
        off = (np.arange(per_call + 1, dtype=np.uint64) * one.size)
        for _ in range(n // per_call):
            rc = lib.hg_sketch_fasta_records(ctx._h, ptr(raw), C.c_void_p(off.ctypes.data), per_call, C.byref(p), max_rec,
                                             ptr(rec), ptr(packed), ptr(bits), ptr(norm), ptr(nh), C.byref(n_rec))
            assert rc == 0, lib.hg_last_error()
            counts, ms, g = ctx.fasta_records_stats()
            tot += ms
            gap += g
            chunks += counts[0]
        ctx.set_profiling(False)
        emit({"layout": "%d files x %d records" % (n, r_per_file), "profiled": True, "chunks": chunks,
              "device_ms": dict(zip(["merge", "index", "hash", "encode"], [round(x, 2) for x in tot])), "host_gap_ms": round(gap, 2),
              "per_chunk_ms": dict(zip(["merge", "index", "hash", "encode", "host_gap"], [round(x / chunks, 3) for x in list(tot) + [gap]]))})
    if a.json:
        with open(a.json, "w") as f:
            json.dump(results, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
