"""ANI clustering (hg_cluster_dev) next to the threshold dist it is built on (hg_dist_dev, symmetric, same rows, same ani_th).

Cases:
  cfg3   config 3 (10,000 family sketches, D 4096, all-vs-all) at -a 95 and 85: hg_cluster_dev against hg_dist_dev on the same
         device rows.  The dist gets a hit buffer of every pair, so neither call ever reruns.
  heavy  20,000 family sketches (D 4096) at ani_th 0: every one of the 2.0e8 pairs is linked.  hg_cluster_dev at several
         edge capacities (HG_CLUSTER_EDGE_CAP), which is what the default was chosen from.
Each call is warmed up, then the calls of a case are timed alternately with CUDA events on the library's stream; a
256 MB buffer is overwritten before every timed call so that no operand is read from L2.  One extra profiled call per
cluster case reports the device time of its steps (hg_cluster_stats).  Every result is checked: at cfg3 against
scipy's connected components of the dist call's own hits, at ani_th 0 against the single cluster.  Prints one JSON line
per case, with the GPU's name, power limit and max SM clock read in the same run.

    python tools/cluster_bench.py [--cases cfg3,heavy] [--caps 4194304,16777216,67108864,134217728] [--steps 5] [--warmup 2]
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

from search_bench import encode_family, gpu_info  # noqa: E402

K = 21


def timed(ctx, calls, steps, warmup):
    """{name: [device ms]} of calls run alternately, each between two events on the library's stream"""
    import torch
    stream = torch.cuda.ExternalStream(ctx.stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    out = {name: [] for name in calls}
    for _ in range(warmup):
        for fn in calls.values():
            fn()
    for _ in range(steps):
        for name, fn in calls.items():
            flush.fill_(1)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            out[name].append(e0.elapsed_time(e1))
    return out


def components(n, i, j):
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    k, lab = connected_components(coo_matrix((np.ones(len(i), np.int8), (i, j)), shape=(n, n)), directed=False)
    first = np.full(k, n, np.int64)
    np.minimum.at(first, lab, np.arange(n))
    return first[lab].astype(np.uint32), int(k)


def profiled(ctx, fn):
    ctx.set_profiling(True)
    fn()
    ctx.set_profiling(False)
    return ctx.cluster_stats()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="cfg3,heavy")
    ap.add_argument("--caps", default="4194304,16777216,67108864,134217728")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import torch
    import hypergen_b200 as hg
    from hypergen_b200 import synth
    ctx = hg.Context(0)
    card = gpu_info()
    D = 4096
    for case in args.cases.split(","):
        if case == "cfg3":
            n = 10000
            hv, norm = encode_family(ctx, synth, n, D)
            pairs = n * (n - 1) // 2
            d_hits = torch.empty((pairs, 4), dtype=torch.int32, device="cuda")
            d_cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
            d_rep = torch.empty(n, dtype=torch.int32, device="cuda")
            os.environ.pop("HG_CLUSTER_EDGE_CAP", None)
            for ani_th in (95.0, 85.0):
                res = {}

                def dist():
                    ctx.dist_dev(hv.data_ptr(), norm.data_ptr(), n, 0, hv.data_ptr(), norm.data_ptr(), n, 0, D, K, ani_th, True, 0,
                                 d_hits.data_ptr(), pairs, d_cnt.data_ptr())

                def cluster():
                    res["k"] = ctx.cluster_dev(hv.data_ptr(), norm.data_ptr(), n, D, K, ani_th, 0, d_rep.data_ptr())

                t = timed(ctx, {"dist": dist, "cluster": cluster}, args.steps, args.warmup)
                counts, ms = profiled(ctx, cluster)
                dist()
                ctx.sync()
                h = d_hits[: int(d_cnt.item())].cpu().numpy().view(np.uint32)
                want_rep, want_k = components(n, h[:, 0].astype(np.int64), h[:, 1].astype(np.int64))
                ok = res["k"] == want_k and np.array_equal(d_rep.cpu().numpy().view(np.uint32), want_rep)
                rec = dict(case="config 3: 10000 family sketches all-vs-all, D 4096", ani_th=ani_th,
                           ms={k: statistics.median(v) for k, v in t.items()}, ms_all=t, dist_path=ctx.dist_last_path,
                           windows=counts[0], linked_pairs=counts[1], largest_window=counts[2], edge_cap=counts[3],
                           step_ms=dict(prepare=ms[0], dist_windows=ms[1], hooks=ms[2], flatten=ms[3]),
                           n_clusters=res["k"], equals_scipy_of_dist_hits=bool(ok), gpu=card)
                print(json.dumps(rec), flush=True)
            del d_hits, hv, norm
            torch.cuda.empty_cache()
        elif case == "heavy":
            n = 20000
            hv, norm = encode_family(ctx, synth, n, D, first=10000)
            d_rep = torch.empty(n, dtype=torch.int32, device="cuda")
            res = {}
            calls = {}
            for cap in [int(c) for c in args.caps.split(",")]:
                def cluster(cap=cap):
                    os.environ["HG_CLUSTER_EDGE_CAP"] = str(cap)
                    res[cap] = ctx.cluster_dev(hv.data_ptr(), norm.data_ptr(), n, D, K, 0.0, 0, d_rep.data_ptr())
                calls["cap%d" % cap] = cluster
            t = timed(ctx, calls, args.steps, args.warmup)
            for name, fn in calls.items():
                d_rep.fill_(-1)
                torch.cuda.synchronize()
                counts, ms = profiled(ctx, fn)
                cap = counts[3]
                all_zero = not d_rep.any().item()
                rec = dict(case="20000 family sketches all-vs-all at ani_th 0 (every pair linked), D 4096", edge_cap=cap,
                           ms=statistics.median(t[name]), ms_all=t[name], dist_path=ctx.dist_last_path, windows=counts[0],
                           linked_pairs=counts[1], largest_window=counts[2],
                           step_ms=dict(prepare=ms[0], dist_windows=ms[1], hooks=ms[2], flatten=ms[3]),
                           one_cluster=bool(res[cap] == 1 and all_zero), gpu=card)
                print(json.dumps(rec), flush=True)
            os.environ.pop("HG_CLUSTER_EDGE_CAP", None)
            del hv, norm
            torch.cuda.empty_cache()
        else:
            raise SystemExit("unknown case " + case)
    ctx.close()


if __name__ == "__main__":
    main()
