"""The all-vs-all ANI matrix (hg_ani_matrix_*) next to what it replaces and what bounds it.

Cases:
  dev     config 3 (10,000 family sketches, D 4096): hg_ani_matrix_dev, lower and square, against hg_dist_dev (symmetric) at
          ani_th 95 and 0, timed alternately with CUDA events on the library's stream; a 256 MB buffer is overwritten before
          every timed call.  One profiled call per layout splits the time into band kernels and conversion.
  packed  hg_ani_matrix_packed, lower, at config 3 (200 MB) and 50,000 sketches (5 GB): host clock around the call (it
          returns complete), into a page-locked buffer and into a pageable one (registered for the call); next to one
          cudaMemcpyAsync of the same bytes device to host into the same kind of buffer, and the pinned run plus a host
          copy into the pageable buffer (what a staging pair would at best reach), and the pinned run with the packed rows
          in page-locked memory too.  Its profiled stages: row upload + unpack + preparation, band kernels, conversion,
          copies.
  route   the existing way at config 3: hg_dist_packed at ani_th 0 (unsorted, room for every pair) and a numpy scatter.
  cli     `hyper-gen triangle` at config 3: its own split into load, GPU, formatting and file write.
  big     93,000 sketches drawn from 8 distinct rows, lower (4.3e9 entries, 17 GB of pinned host memory), run once and
          checked cell by cell against the oracle's 8 x 8 class table.
Prints one JSON line per case, with the GPU's name, power limit and max SM clock read in the same run.

    python tools/matrix_bench.py [--cases dev,packed,route,cli,big] [--steps 5] [--warmup 2] [--packed-n 10000,50000]

HG_MATRIX_BAND_BYTES applies as in the library (the band budget of every matrix call).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True

from cluster_bench import timed  # noqa: E402
from search_bench import encode_family, gpu_info  # noqa: E402

K, D = 21, 4096


def host_rows(ctx, synth, n):
    """n family sketches: device (hv, norm) and host (packed, bits, norm)"""
    import torch
    packed = torch.empty((n, 2 * D), dtype=torch.uint8, device="cuda")
    hv, norm, bits = encode_family(ctx, synth, n, D, packed=packed)
    return hv, norm, packed.cpu().numpy(), bits.cpu().numpy(), norm.cpu().numpy()


def wall(fn, steps):
    out = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        out.append((time.perf_counter() - t0) * 1e3)
    return out


def case_dev(ctx, hg, synth, card, steps, warmup):
    import torch
    n = 10000
    hv, norm = encode_family(ctx, synth, n, D)
    tri = torch.empty(n * (n - 1) // 2, dtype=torch.float32, device="cuda")
    sq = torch.empty(n * n, dtype=torch.float32, device="cuda")
    cap = n * (n - 1) // 2
    hits = torch.empty(cap * 16, dtype=torch.uint8, device="cuda")
    cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
    a = (hv.data_ptr(), norm.data_ptr(), n, hv.data_ptr(), norm.data_ptr(), n, D, K, 0)
    calls = {
        "matrix_lower": lambda: ctx.ani_matrix_dev(*a, True, tri.data_ptr(), 0),
        "matrix_square": lambda: ctx.ani_matrix_dev(*a, False, sq.data_ptr(), n),
        "dist_95": lambda: ctx.dist_dev(hv.data_ptr(), norm.data_ptr(), n, 0, hv.data_ptr(), norm.data_ptr(), n, 0, D, K, 95.0, True, 0,
                                        hits.data_ptr(), cap, cnt.data_ptr()),
        "dist_0": lambda: ctx.dist_dev(hv.data_ptr(), norm.data_ptr(), n, 0, hv.data_ptr(), norm.data_ptr(), n, 0, D, K, 0.0, True, 0,
                                       hits.data_ptr(), cap, cnt.data_ptr()),
    }
    t = timed(ctx, calls, steps, warmup)
    split = {}
    for name in ("matrix_lower", "matrix_square"):
        ctx.set_profiling(True)
        calls[name]()
        ctx.set_profiling(False)
        counts, ms = ctx.ani_matrix_stats()
        split[name] = dict(bands=counts[0], entries=counts[1], prepare_ms=ms[0], band_kernels_ms=ms[1], convert_ms=ms[2])
    return dict(case="dev", n=n, ms={k: statistics.median(v) for k, v in t.items()}, ms_all=t, split=split,
                dist_path=ctx.dist_last_path, gpu=card)


def case_packed(ctx, hg, synth, card, steps, warmup, sizes=(10000, 50000)):
    import torch
    out = []
    for n in sizes:
        hv, norm, packed, bits, hnorm = host_rows(ctx, synth, n)
        del hv, norm
        m = n * (n - 1) // 2
        pinned = torch.empty(m, dtype=torch.float32).pin_memory()
        pageable = np.empty(m, np.float32)
        pageable.fill(0)  # the pages exist before the first call
        dev = torch.empty(m, dtype=torch.float32, device="cuda")
        pin_np = pinned.numpy()
        p_packed = hg.ffi.pinned_empty(packed.shape, np.uint8)  # the rows too in page-locked memory: their upload at link rate
        p_packed[:] = packed
        calls = {
            "matrix_pinned": lambda: ctx.ani_matrix_packed(packed, bits, hnorm, hv_d=D, lower=True, out=pin_np),
            "matrix_pinned_rows_pinned": lambda: ctx.ani_matrix_packed(p_packed, bits, hnorm, hv_d=D, lower=True, out=pin_np),
            "matrix_pageable": lambda: ctx.ani_matrix_packed(packed, bits, hnorm, hv_d=D, lower=True, out=pageable),
            "matrix_pinned_then_host_copy": lambda: (ctx.ani_matrix_packed(packed, bits, hnorm, hv_d=D, lower=True, out=pin_np),
                                                     np.copyto(pageable, pin_np)),
            "bare_d2h_pinned": lambda: (pinned.copy_(dev, non_blocking=True), torch.cuda.synchronize()),
            "bare_d2h_pageable": lambda: (torch.from_numpy(pageable).copy_(dev), torch.cuda.synchronize()),
        }
        for fn in calls.values():
            for _ in range(warmup):
                fn()
        t = {k: [] for k in calls}
        for _ in range(steps):
            for k, fn in calls.items():
                t[k] += wall(fn, 1)
        ok = bool(np.array_equal(pageable.view(np.uint32), pin_np.view(np.uint32)))
        ctx.set_profiling(True)
        calls["matrix_pinned"]()
        ctx.set_profiling(False)
        counts, ms = ctx.ani_matrix_stats()
        out.append(dict(case="packed", n=n, bytes=4 * m, band_bytes=os.environ.get("HG_MATRIX_BAND_BYTES", "default"), ms={k: statistics.median(v) for k, v in t.items()}, ms_all=t,
                        pageable_equals_pinned=ok, bands=counts[0], stage_ms=dict(prepare=ms[0], band_kernels=ms[1], convert=ms[2],
                                                                               copies=ms[3]), dist_path=ctx.dist_last_path, gpu=card))
        del pinned, pageable, dev
    return out


def case_route(ctx, hg, synth, card, steps, warmup):
    n = 10000
    _, _, packed, bits, hnorm = host_rows(ctx, synth, n)
    m = n * (n - 1) // 2
    tri = np.empty(m, np.float32)

    def route():
        hits, _ = ctx.dist_packed(packed, bits, hnorm, packed, bits, hnorm, D, ani_th=0.0, symmetric=True, sorted_output=False, cap=m)
        i, j = hits["i"].astype(np.int64), hits["j"].astype(np.int64)
        tri[j * (j - 1) // 2 + i] = hits["ani"]  # pair (i < j) is cell (j, i) of the lower triangle

    for _ in range(warmup):
        route()
    t = wall(route, steps)
    want = ctx.ani_matrix_packed(packed, bits, hnorm, hv_d=D, lower=True)
    return dict(case="route", n=n, ms=statistics.median(t), ms_all=t, equals_matrix=bool(np.array_equal(tri.view(np.uint32), want.view(np.uint32))),
                gpu=card)


def case_cli(ctx, hg, synth, card, steps, warmup):
    from hypergen_b200 import _build, fileio
    exe = _build.build_host()
    n = 10000
    _, _, packed, bits, hnorm = host_rows(ctx, synth, n)
    with tempfile.TemporaryDirectory() as d:
        f = os.path.join(d, "s.sketch")
        fileio.dump_sketch([fileio.FileSketch(ksize=K, hv_d=D, hv_quant_bits=int(bits[g]), hv_norm_2=int(hnorm[g]), file_str="g/%05d.fna" % g,
                                              hv=packed[g, : int(bits[g]) * D // 8].view(np.int16).copy()) for g in range(n)], f)
        lines = []
        for _ in range(warmup + steps):
            t0 = time.perf_counter()
            p = subprocess.run([exe, "triangle", "-r", f, "-o", os.path.join(d, "t.txt")], capture_output=True, text=True, check=True)
            lines.append((time.perf_counter() - t0) * 1e3)
        size = os.path.getsize(os.path.join(d, "t.txt"))
    return dict(case="cli", n=n, wall_ms=lines[warmup:], last_report=p.stdout.strip(), bytes=size, gpu=card)


def case_big(ctx, hg, synth, card, steps, warmup):
    import torch
    import oracle
    oracle.build()
    n, c = 93000, 8
    hv, norm, packed, bits, hnorm = host_rows(ctx, synth, c)
    cls = np.random.default_rng(5).integers(0, c, n)
    hv = hv.cpu().numpy()
    table = oracle.dist_all(hv, hnorm, hv, hnorm, want_dot=False)[0].reshape(c, c)
    m = n * (n - 1) // 2
    assert m > 2**32
    out = torch.empty(m, dtype=torch.float32).pin_memory().numpy()
    t0 = time.perf_counter()
    got = ctx.ani_matrix_packed(packed[cls], bits[cls], hnorm[cls], hv_d=D, lower=True, out=out)
    ms = (time.perf_counter() - t0) * 1e3
    counts = ctx.ani_matrix_stats()[0]
    tb = table.view(np.uint32)
    bad = 0
    step = 2000
    for i0 in range(1, n, step):
        i1 = min(n, i0 + step)
        for i in range(i0, i1):
            row = got[i * (i - 1) // 2: i * (i - 1) // 2 + i].view(np.uint32)
            bad += int((row != tb[cls[i], cls[:i]]).sum())
    return dict(case="big", n=n, entries=m, ms=ms, bands=counts[0], mismatches=bad, dist_path=ctx.dist_last_path, gpu=card)


CASES = {"dev": case_dev, "packed": case_packed, "route": case_route, "cli": case_cli, "big": case_big}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="dev,packed,route,cli")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--packed-n", default="10000,50000", help="sketch counts of the packed case")
    a = ap.parse_args()
    import hypergen_b200 as hg
    from hypergen_b200 import synth
    card = gpu_info()
    ctx = hg.Context(0)
    try:
        for name in a.cases.split(","):
            extra = dict(sizes=[int(x) for x in a.packed_n.split(",")]) if name == "packed" else {}
            r = CASES[name](ctx, hg, synth, card, a.steps, a.warmup, **extra)
            for rec in (r if isinstance(r, list) else [r]):
                print(json.dumps(rec), flush=True)
    finally:
        ctx.close()


if __name__ == "__main__":
    main()
