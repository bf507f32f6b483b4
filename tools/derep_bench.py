"""Greedy ANI dereplication (hg_derep_dev) next to the single-linkage clustering (hg_cluster_dev) and the threshold dist
(hg_dist_dev, symmetric) it is built on: same device rows, same ani_th.

Cases:
  cfg3   config 3 (10,000 family sketches, D 4096, all-vs-all) at -a 95 and 85: derep in file order, cluster and dist.  The
         dist gets a hit buffer of every pair, so it never reruns; its hits also give the expected answer (a Python greedy
         over the linked pairs and their ANIs).
  heavy  20,000 family sketches (D 4096) at ani_th 0: every one of the 2.0e8 pairs is linked, one representative.
  big    100,000 family sketches (D 4096) at ani_th 95, in size order: 5.0e9 pairs through 117 column chunks (1024
         columns wide until the edge capacity narrows them).
Each call is warmed up, then the calls of a case are timed alternately with CUDA events on the library's stream; a
256 MB buffer is overwritten before every timed call so that no operand is read from L2.  One extra profiled derep call
per case reports the device time of its phases (hg_derep_stats).  Prints one JSON line per case, with the GPU's name,
power limit and max SM clock read in the same run.

    python tools/derep_bench.py [--cases cfg3,heavy,big] [--steps 5] [--warmup 2]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True

from cluster_bench import timed  # noqa: E402
from search_bench import encode_family, gpu_info  # noqa: E402

K = 21


def greedy_from_pairs(n, i, j, ani, ani_th, order=None):
    """(rep, n_reps) of greedy dereplication from every linked pair (i, j, ani) with ani >= ani_th (the rest is below)"""
    pos = np.arange(n) if order is None else np.argsort(order)
    m = ani >= np.float32(ani_th)
    i, j, ani = i[m], j[m], ani[m]
    a, b, w = np.r_[i, j], np.r_[j, i], np.r_[ani, ani]  # both directions: a -> b
    srt = np.argsort(b, kind="stable")
    a, b, w = a[srt], b[srt], w[srt]
    start = np.searchsorted(b, np.arange(n + 1))
    is_rep = np.zeros(n, bool)
    for g in (np.arange(n) if order is None else order):
        nb = a[start[g]:start[g + 1]]
        if not is_rep[nb].any():
            is_rep[g] = True
    rep = np.arange(n, dtype=np.int64)
    keep = is_rep[a] & ~is_rep[b]  # representative a, member b
    a, b, w = a[keep], b[keep], w[keep]
    best = np.lexsort((pos[a], -w, b))  # per member: largest ANI, then first in the order
    b_s = b[best]
    first = np.ones(b_s.size, bool)
    first[1:] = b_s[1:] != b_s[:-1]
    rep[b_s[first]] = a[best][first]
    return rep.astype(np.uint32), int(is_rep.sum())


def profiled(ctx, fn):
    ctx.set_profiling(True)
    fn()
    ctx.set_profiling(False)
    return ctx.derep_stats()


def consistent(rep, k):
    """every label a representative of itself, and k of them"""
    return bool(np.array_equal(rep[rep], rep) and int((rep == np.arange(rep.size)).sum()) == k)


def record(case, ani_th, t, counts, ms, ctx, card, **extra):
    return dict(case=case, ani_th=ani_th, ms={k: statistics.median(v) for k, v in t.items()}, ms_all=t,
                dist_path=ctx.dist_last_path, chunks=counts[0], windows=counts[1], linked_pairs=counts[2], n_reps=counts[3],
                phase_ms=dict(prepare=ms[0], dist_windows=ms[1], marks_and_greedy=ms[2], assignment=ms[3]), gpu=card, **extra)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="cfg3,heavy,big")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import torch
    import hypergen_b200 as hg
    from hypergen_b200 import derep, synth
    ctx = hg.Context(0)
    card = gpu_info()
    D = 4096
    os.environ.pop("HG_CLUSTER_EDGE_CAP", None)
    for case in args.cases.split(","):
        if case == "cfg3":
            n = 10000
            hv, norm = encode_family(ctx, synth, n, D)
            pairs = n * (n - 1) // 2
            d_hits = torch.empty((pairs, 4), dtype=torch.int32, device="cuda")
            d_cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
            d_rep = torch.empty(n, dtype=torch.int32, device="cuda")
            d_cl = torch.empty(n, dtype=torch.int32, device="cuda")
            for ani_th in (95.0, 85.0):
                res = {}

                def dist():
                    ctx.dist_dev(hv.data_ptr(), norm.data_ptr(), n, 0, hv.data_ptr(), norm.data_ptr(), n, 0, D, K, ani_th, True, 0,
                                 d_hits.data_ptr(), pairs, d_cnt.data_ptr())

                def cluster():
                    res["clusters"] = ctx.cluster_dev(hv.data_ptr(), norm.data_ptr(), n, D, K, ani_th, 0, d_cl.data_ptr())

                def dr():
                    res["k"] = ctx.derep_dev(hv.data_ptr(), norm.data_ptr(), n, D, K, ani_th, 0, d_rep.data_ptr())

                t = timed(ctx, {"dist": dist, "cluster": cluster, "derep": dr}, args.steps, args.warmup)
                counts, ms = profiled(ctx, dr)
                path = ctx.dist_last_path
                dist()
                ctx.sync()
                h = d_hits[: int(d_cnt.item())].cpu().numpy()
                want = greedy_from_pairs(n, h[:, 0].view(np.uint32).astype(np.int64), h[:, 1].view(np.uint32).astype(np.int64),
                                         h[:, 3].view(np.float32), ani_th)
                ok = res["k"] == want[1] and np.array_equal(d_rep.cpu().numpy().view(np.uint32), want[0])
                rec = record("config 3: 10000 family sketches, D 4096", ani_th, t, counts, ms, ctx, card,
                             n_clusters_single_linkage=res["clusters"], equals_greedy_of_dist_hits=bool(ok))
                rec["dist_path"] = path
                print(json.dumps(rec), flush=True)
            del d_hits, hv, norm
            torch.cuda.empty_cache()
        elif case in ("heavy", "big"):
            n, ani_th, first, kind = (20000, 0.0, 10000, "file") if case == "heavy" else (100000, 95.0, 0, "size")
            hv, norm = encode_family(ctx, synth, n, D, first=first)
            order = derep.priority(norm.cpu().numpy(), kind)
            d_rep = torch.empty(n, dtype=torch.int32, device="cuda")
            d_cl = torch.empty(n, dtype=torch.int32, device="cuda")
            res = {}

            def cluster():
                res["clusters"] = ctx.cluster_dev(hv.data_ptr(), norm.data_ptr(), n, D, K, ani_th, 0, d_cl.data_ptr())

            def dr():
                res["k"] = ctx.derep_dev(hv.data_ptr(), norm.data_ptr(), n, D, K, ani_th, 0, d_rep.data_ptr(), order=order)

            t = timed(ctx, {"cluster": cluster, "derep": dr}, args.steps, args.warmup)
            d_rep.fill_(-1)
            torch.cuda.synchronize()
            counts, ms = profiled(ctx, dr)
            rep = d_rep.cpu().numpy().view(np.uint32)
            ok = consistent(rep, res["k"]) and (case != "heavy" or (res["k"] == 1 and not rep.any()))
            desc = ("20000 family sketches at ani_th 0 (every pair linked), D 4096" if case == "heavy"
                    else "100000 family sketches, D 4096, size order")
            print(json.dumps(record(desc, ani_th, t, counts, ms, ctx, card, n_clusters_single_linkage=res["clusters"],
                                    labels_consistent=bool(ok))), flush=True)
            del hv, norm
            torch.cuda.empty_cache()
        else:
            raise SystemExit("unknown case " + case)
    ctx.close()


if __name__ == "__main__":
    main()
