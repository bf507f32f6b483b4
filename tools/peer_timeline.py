"""Per-member timeline of the sharded dist (run under torchrun with HG_PEER_TIMELINE=1): the kernels' %globaltimer stamps
(hg_peer_timeline), every member's shifted so that the barrier exit of the step before is t = 0.
    HG_PEER_TIMELINE=1 torchrun ... tools/peer_timeline.py [cfg3|cfg4|cfg5]"""
import os, sys
os.environ.setdefault("HG_PEER_TIMELINE", "1")
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, torch.distributed as dist
rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
torch.cuda.set_device(rank); dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
host_pg = dist.new_group(backend="gloo")
import hypergen_b200 as hg
from hypergen_b200 import multigpu, synth
import bench as B
which = sys.argv[1] if len(sys.argv) > 1 else "cfg3"
cfg = {"cfg3": B.DIST_CONFIGS[0], "cfg4": B.DIST_CONFIGS[1], "cfg5": B.DIST_CONFIGS[2]}[which]
ctx = hg.Context(rank)
ext = torch.cuda.ExternalStream(ctx.stream, device=dev)
D, sym = cfg["hv_d"], cfg["symmetric"]
if sym:
    n_ref = n_qry = cfg["n"]
    hv, norm, bits, _ = B.encode_family(ctx, synth, dev, n_ref, D, cfg["n_per"], cfg["scaled"], cfg["seed"])
    ref_hv, ref_norm, qry_hv, qry_norm = hv, norm, hv, norm
else:
    n_ref, n_qry = cfg["n_ref"], cfg["n_qry"]
    ref_hv, ref_norm, bits, _ = B.encode_family(ctx, synth, dev, n_ref, D, cfg["n_per"], cfg["scaled"], cfg["seed"])
    q_idx = torch.arange(5, n_ref, n_ref // n_qry, device=dev)[:n_qry]
    qry_hv, qry_norm = ref_hv[q_idx].contiguous(), ref_norm[q_idx].contiguous()
cap = 4_000_000
pg = multigpu.PeerGroup(ctx, hg.ffi.peer_window_need(n_qry, D, cap), dev)
qb = multigpu.block_rows(n_qry, world); rb = multigpu.block_rows(n_ref, world)
a, b = qb[rank], qb[rank + 1]; ra, rbb = rb[rank], rb[rank + 1]
from multiprocessing import shared_memory
name = "hg_tl_hits_%s" % os.environ.get("MASTER_PORT", "0")
shm = shared_memory.SharedMemory(name=name, create=True, size=cap * 16) if rank == 0 else None
dist.barrier(group=host_pg)
if rank != 0:
    shm = shared_memory.SharedMemory(name=name)
hits_np = np.ndarray((cap,), dtype=hg.ffi.HIT_DTYPE, buffer=shm.buf)
mapped = hg.ffi.host_register(hits_np)


def step(path):
    if sym:
        pg.peer.dist_sharded_dev(None, None, 0, 0, qry_hv[a:b].data_ptr(), qry_norm[a:b].data_ptr(), qb, D, 21, 85.0, True, path, 0, cap, mapped)
    else:
        pg.peer.dist_sharded_dev(ref_hv[ra:rbb].data_ptr(), ref_norm[ra:rbb].data_ptr(), rbb - ra, ra, qry_hv[a:b].data_ptr(),
                                 qry_norm[a:b].data_ptr(), qb, D, 21, 85.0, False, path, 0, cap, mapped)
    return pg.peer.dist_sharded_hits(cap, hits=hits_np)[0]


with torch.cuda.stream(ext):
    step(0)
path = ctx.dist_last_path
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
NAMES = {0: "first node", 1: "kernel in", 2: "start flags", 4: "last CTA out", 8: "start set out", 9: "1st chunk out", 10: "1st dest done", 11: "all rows out",
         12: "flush", 13: "barrier in", 14: "barrier out"}
rows, ms = [], []
for it in range(8):
    flush.fill_(1); torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(ext):
        pg.peer.barrier()
        e0.record()
        h = step(path)
        e1.record()
    e1.synchronize()
    ms.append(e0.elapsed_time(e1))
    rows.append(pg.peer.timeline())
t = rows[-1]
rel = {i: (t[i] - t[16]) / 1e3 if t[i] else None for i in NAMES}
mine = dict(rank=rank, ms=float(np.mean(ms[3:])), rel=rel, wait0=t[3] / 1e3, waitmax=t[5] / 1e3, hits=int(h.size))
allr = [None] * world
dist.all_gather_object(allr, mine, group=host_pg)
if rank == 0:
    print("== %s world %d path %d: step %.3f ms (max over ranks %.3f), hits %d" % (
        which, world, path, allr[0]["ms"], max(x["ms"] for x in allr), allr[0]["hits"]))
    print("   us after the previous step's barrier exit; rank: " + " ".join("%9d" % x["rank"] for x in allr))
    for i in sorted(NAMES):
        print("   %-14s " % NAMES[i] + "      " + " ".join("%9.1f" % x["rel"][i] if x["rel"][i] is not None else "        -" for x in allr))
    print("   %-14s " % "CTA0 row wait" + "      " + " ".join("%9.1f" % x["wait0"] for x in allr))
    print("   %-14s " % "max row wait" + "      " + " ".join("%9.1f" % x["waitmax"] for x in allr))
    k = [x["rel"][4] - x["rel"][1] for x in allr]
    print("   kernel in->out      " + " ".join("%9.1f" % v for v in k), flush=True)
dist.barrier(group=host_pg)
hg.ffi.host_unregister(hits_np); del hits_np, h; shm.close()
if rank == 0: shm.unlink()
pg.close(); ctx.close()
dist.destroy_process_group()
