"""Top-k search (hg_search_dev) next to the threshold dist (hg_dist_dev, ani_th = 85) on the same device rows.

Shapes: config 4 (100,000 refs x 1,000 queries, D 4096, family hash sets; the queries are ref rows with relatives among
the refs, as bench.py takes them) and 10,000 x 10,000 non-symmetric (refs = sketches 0..9,999, queries = sketches
5,000..14,999: half of them have their family among the refs).  For every top_k, both calls are warmed up, then timed
alternately with CUDA events on the library's stream.  One extra profiled search per case reports the sample size s,
the candidates of each pass and the device time of each step.  64 sampled queries per case are checked against the
oracle (every i, dot, ANI bit, n_found).  Prints one JSON line per case, with the GPU's name and power limit.

With --gpus N the tool times the host entries instead, end to end from packed host rows as a sketch file holds them
(the H2D copies, the unpack, the search and the copy of the result back): hg_search_packed on one GPU next to
hg_group_search_packed on groups of 1..N GPUs (--same-gpu: groups of 1..N contexts on GPU 0, which measures what the
block split, gather and merge add and nothing of the scaling).  Host clock around each call (the call returns with the
result on the host), calls alternated; every group result is compared with the single-GPU result, slot for slot.

    python tools/search_bench.py [--shapes cfg4,10k] [--top-k 1,10,100] [--steps 5] [--warmup 2] [--out FILE]
                                 [--gpus N [--same-gpu]]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

K = 21


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def encode_family(ctx, synth, n, D, n_per=3333, scaled=1500, seed=0xD157, first=0, packed=None):
    """-> device (hv, norm); with `packed` (a device uint8 tensor of n x 2D) also the packed rows there, and the bits"""
    import torch
    hv = torch.empty((n, D), dtype=torch.int16, device="cuda")
    norm = torch.empty(n, dtype=torch.int32, device="cuda")
    bits = torch.empty(n, dtype=torch.uint8, device="cuda")
    chunk = max(256, min(n, (1 << 28) // (8 * n_per)))
    for c0 in range(0, n, chunk):
        m = min(chunk, n - c0)
        hashes, off = synth.hash_sets_family_dev(m, n_per=n_per, scaled=scaled, seed=seed, device="cuda", first=first + c0)
        torch.cuda.current_stream().synchronize()  # the encoder runs on the library's stream
        ctx.encode_sets_dev(hashes.data_ptr(), off, D, hv[c0:].data_ptr(), None if packed is None else packed[c0:].data_ptr(),
                            bits[c0:].data_ptr(), norm[c0:].data_ptr())
        ctx.sync()
        del hashes
    if packed is not None:
        return hv, norm, bits
    return hv, norm


def shapes(names):
    import torch
    from hypergen_b200 import synth
    for name in names:
        ctx = CTX
        if name == "cfg4":
            ref, rn = encode_family(ctx, synth, 100000, 4096)
            q_idx = torch.arange(5, 100000, 100, device="cuda")[:1000]
            yield "config 4: 100000 refs x 1000 queries, D 4096", ref, rn, ref[q_idx].contiguous(), rn[q_idx].contiguous()
        elif name == "10k":
            hv, norm = encode_family(ctx, synth, 15000, 4096)
            yield "10000 refs x 10000 queries (non-symmetric), D 4096", hv[:10000], norm[:10000], hv[5000:].contiguous(), norm[5000:].contiguous()
        else:
            raise SystemExit("unknown shape " + name)


def packed_shapes(names):
    """the shapes above as host (packed, bits, norm) of refs and queries: rows of 2 D bytes, as the CLI stacks a sketch file"""
    import torch
    from hypergen_b200 import synth
    D = 4096
    for name in names:
        n, label = {"cfg4": (100000, "config 4: 100000 refs x 1000 queries, D 4096"),
                    "10k": (15000, "10000 refs x 10000 queries (non-symmetric), D 4096")}.get(name, (0, ""))
        if not n:
            raise SystemExit("unknown shape " + name)
        d_packed = torch.empty((n, 2 * D), dtype=torch.uint8, device="cuda")
        hv, norm, bits = encode_family(CTX, synth, n, D, packed=d_packed)
        del hv
        packed, norm, bits = d_packed.cpu().numpy(), norm.cpu().numpy(), bits.cpu().numpy()
        del d_packed
        torch.cuda.empty_cache()
        if name == "cfg4":
            r, q = slice(0, 100000), np.arange(5, 100000, 100)[:1000]
        else:
            r, q = slice(0, 10000), slice(5000, 15000)
        yield label, (packed[r], bits[r], norm[r]), (np.ascontiguousarray(packed[q]), bits[q].copy(), norm[q].copy())


def group_bench(args, hg):
    """hg_search_packed next to hg_group_search_packed at 1..N GPUs (or N contexts on GPU 0), end to end from host rows"""
    ctx = CTX
    sizes = list(range(1, args.gpus + 1))
    groups = {n: hg.Group(ordinals=[0] * n if args.same_gpu else list(range(n))) for n in sizes}
    card = gpu_info()
    lines = []
    for label, (rp, rb, rn), (qp, qb, qn) in packed_shapes(args.shapes.split(",")):
        for top_k in [int(x) for x in args.top_k.split(",")]:
            calls = {"single": lambda: ctx.search_packed(rp, rb, rn, qp, qb, qn, 4096, ksize=K, top_k=top_k)}
            for n in sizes:
                calls["group%d" % n] = (lambda g: lambda: g.search_packed(rp, rb, rn, qp, qb, qn, 4096, ksize=K, top_k=top_k))(groups[n])
            results = {}
            for _ in range(args.warmup):
                for name, fn in calls.items():
                    results[name] = fn()
            times = {name: [] for name in calls}
            for _ in range(args.steps):
                for name, fn in calls.items():
                    t0 = time.perf_counter()
                    fn()
                    times[name].append((time.perf_counter() - t0) * 1e3)
            identical = all(all(np.array_equal(a, b) for a, b in zip(results[name], results["single"])) for name in calls)
            rec = dict(shape=label, top_k=top_k, ani_min=0.0, same_gpu=bool(args.same_gpu),
                       ms={name: statistics.median(t) for name, t in times.items()},
                       ms_all=times, identical_to_single=identical,
                       members_used={n: sum(groups[n].search_stats(m)[0][0] > 0 for m in range(n)) for n in sizes},
                       ref_bytes_h2d=int(rb.astype(np.int64).sum() * 4096 // 8), gpu=card)
            print(json.dumps(rec), flush=True)
            lines.append(rec)
    for g in groups.values():
        g.close()
    return lines


def oracle_check(ref, rn, qry, qn, hits, n_found, top_k, rng):
    import oracle as O
    O.build()
    O.set_threads(os.cpu_count() or 1)
    Q = qry.shape[0]
    sel = np.sort(rng.choice(Q, min(64, Q), replace=False))
    r, rnn = ref.cpu().numpy(), rn.cpu().numpy()
    q, qnn = qry[sel].cpu().numpy(), qn[sel].cpu().numpy()
    ani, dot = O.dist_all(r, rnn, q, qnn, k=K)
    ani, dot = ani.reshape(r.shape[0], len(sel)), dot.reshape(r.shape[0], len(sel))
    bad = 0
    for t, j in enumerate(sel):
        order = np.lexsort((np.arange(r.shape[0]), -ani[:, t]))[:top_k]
        n = int(n_found[j])
        ok = (n == order.size and np.array_equal(hits["i"][j, :n], order) and np.array_equal(hits["dot"][j, :n], dot[order, t])
              and np.array_equal(hits["ani"][j, :n].view(np.uint32), ani[order, t].view(np.uint32)))
        bad += not ok
    return len(sel), bad


def main():
    global CTX
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="cfg4,10k")
    ap.add_argument("--top-k", default="1,10,100")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--out", default="")
    ap.add_argument("--gpus", type=int, default=0)
    ap.add_argument("--same-gpu", action="store_true")
    args = ap.parse_args()
    import torch
    import hypergen_b200 as hg
    CTX = hg.Context(0)
    ctx = CTX
    if args.gpus:
        if not args.same_gpu and torch.cuda.device_count() < args.gpus:
            raise SystemExit("--gpus %d: %d GPUs visible" % (args.gpus, torch.cuda.device_count()))
        write_lines(args.out, group_bench(args, hg))
        ctx.close()
        return
    stream = torch.cuda.ExternalStream(ctx.stream)
    card = gpu_info()
    rng = np.random.default_rng(1)
    lines = []
    cap = 4_000_000
    d_hits = torch.empty(cap * 16, dtype=torch.uint8, device="cuda")
    d_cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
    for label, ref, rn, qry, qn in shapes(args.shapes.split(",")):
        R, D = ref.shape
        Q = qry.shape[0]

        def dist_call():
            ctx.dist_dev(ref.data_ptr(), rn.data_ptr(), R, 0, qry.data_ptr(), qn.data_ptr(), Q, 0, D, K, 85.0, False, 0,
                         d_hits.data_ptr(), cap, d_cnt.data_ptr())
            ctx.sync()

        for top_k in [int(x) for x in args.top_k.split(",")]:
            d_out = torch.empty(Q * top_k * 16, dtype=torch.uint8, device="cuda")
            d_nf = torch.empty(Q, dtype=torch.int32, device="cuda")
            d_mi = torch.empty(Q * top_k, dtype=torch.int32, device="cuda")

            def search_call():
                ctx.search_dev(ref.data_ptr(), rn.data_ptr(), R, qry.data_ptr(), qn.data_ptr(), Q, D, K, top_k, 0.0, 0,
                               d_out.data_ptr(), d_nf.data_ptr(), d_mi.data_ptr())

            def timed(fn):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                fn()
                e1.record(stream)
                e1.synchronize()
                return e0.elapsed_time(e1)

            for _ in range(args.warmup):
                search_call()
                dist_call()
            t_search, t_dist = [], []
            for _ in range(args.steps):
                t_search.append(timed(search_call))
                t_dist.append(timed(dist_call))
            ctx.set_profiling(True)
            search_call()
            counts, ms = ctx.search_stats()
            ctx.set_profiling(False)
            path, reason = ctx.dist_last_path, ctx.dist_last_reason
            rec = dict(shape=label, top_k=top_k, search_ms=statistics.median(t_search), dist85_ms=statistics.median(t_dist),
                       search_ms_all=t_search, dist85_ms_all=t_dist, sample_rows=counts[0], floor_candidates=counts[1],
                       main_candidates=counts[2], reruns=counts[3],
                       step_ms=dict(floor_pass=ms[0], floor_select=ms[1], main_pass=ms[2], main_select=ms[3]),
                       main_path=path, main_reason=reason, ani_min=0.0, gpu=card)
            if not args.no_check:
                hits = np.frombuffer(d_out.cpu().numpy().tobytes(), dtype=hg.ffi.HIT_DTYPE).reshape(Q, top_k)
                n, bad = oracle_check(ref, rn, qry, qn, hits, d_nf.cpu().numpy(), top_k, rng)
                rec["oracle_checked_queries"], rec["oracle_mismatches"] = n, bad
            print(json.dumps(rec), flush=True)
            lines.append(rec)
        del ref, rn, qry, qn
        torch.cuda.empty_cache()
    write_lines(args.out, lines)
    ctx.close()


def write_lines(path, lines):
    if path:
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


CTX = None

if __name__ == "__main__":
    main()
