"""GPU parity of the multi-GPU dist (csrc/peer.cu): NVLink-window exchange + sharded tensor kernels vs the oracle.

Reference behaviour under test: src/dist.rs:139-161,231-294 (every enumerated pair, exact i32 dot, f32 ANI bits),
src/utils.rs:262-285 (output order) - whichever GPU computed the pair.  The world-size-1 cases run on any box; the
2-GPU cases (one process driving two GPUs, and one process per GPU over cudaIpc) skip when fewer GPUs are visible."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _n_gpus():
    import torch
    return torch.cuda.device_count()


def _sketch_sets(ctx, n, hv_d, n_per, scaled, first=0):
    """encode hash sets on the GPU -> host (hv, norm, packed, bits)"""
    import torch
    from hypergen_b200 import synth
    hashes, off = synth.hash_sets_family_dev(n, n_per=n_per, scaled=scaled, first=first)
    sets = [hashes.numpy().view(np.uint64)[int(off[g]):int(off[g + 1])] for g in range(n)]
    r = ctx.encode_sets(sets, hv_d=hv_d)
    return r["hv"], r["norm2"], r["packed"], r["quant_bits"]


def _check_hits(oracle, hits, r, rn, q, qn, symmetric, th, i0=0):
    ani, dot = oracle.dist_all(r, rn, q, qn, symmetric=symmetric)
    R, Q = r.shape[0], q.shape[0]
    i, j = hits["i"].astype(np.int64) - i0, hits["j"].astype(np.int64)
    idx = i * (Q - 1) - i * (i - 1) // 2 + (j - i - 1) if symmetric else i * Q + j
    want = np.nonzero(ani >= np.float32(th))[0]
    assert np.array_equal(np.sort(idx), want)
    assert np.array_equal(hits["dot"], dot[idx])
    assert np.array_equal(hits["ani"].view(np.uint32), ani[idx].view(np.uint32))


def _dev(t):
    import torch
    return torch.from_numpy(np.ascontiguousarray(t)).cuda()


@pytest.mark.parametrize("path,hv_d", [(0, 1024), (2, 1024), (3, 1024), (2, 768)], ids=["0", "2", "3", "2-768"])
@pytest.mark.parametrize("symmetric", [True, False])
def test_world1_sharded_equals_oracle(ctx, hg, oracle, path, hv_d, symmetric):
    """One member: the window path (operands prepared inside the window, tile walk 0/1) must equal the plain path.
    hv_d = 768: the two-limb kernel's K loop runs past hv_d into the tensor maps' zero fill."""
    hv, norm, _, _ = _sketch_sets(ctx, 700, hv_d, 800, 1500)
    cap = 700 * 700
    peer = hg.Peer(ctx, 0, 1, hg.ffi.peer_window_need(700, hv_d, cap))
    try:
        d_hv, d_n = _dev(hv), _dev(norm)
        if symmetric:
            peer.dist_sharded_dev(None, None, 0, 0, d_hv.data_ptr(), d_n.data_ptr(), [0, 700], hv_d, 21, 80.0, True, path, 0, cap)
            hits, _ = peer.dist_sharded_hits(cap)
            _check_hits(oracle, hits, hv, norm, hv, norm, True, 80.0)
        else:
            peer.dist_sharded_dev(d_hv[:300].data_ptr(), d_n[:300].data_ptr(), 300, 1000, d_hv.data_ptr(), d_n.data_ptr(), [0, 700],
                                  hv_d, 21, 0.0, False, path, 0, cap)
            hits, _ = peer.dist_sharded_hits(cap)
            _check_hits(oracle, hits, hv[:300], norm[:300], hv, norm, False, 0.0, i0=1000)
        assert ctx.dist_last_path == (path or 3)
    finally:
        peer.close()


def test_world1_outlier_corrections_from_planes(ctx, hg, oracle, monkeypatch):
    """rows with elements outside the s8 plane: the exact correction is rebuilt from planes + outlier lists alone"""
    monkeypatch.setenv("HG_NARROW_BUDGET", "64")
    hv, norm, _, _ = _sketch_sets(ctx, 400, 1024, 800, 1500)
    rng = np.random.default_rng(3)
    hv = hv.copy()
    for r in rng.choice(400, 60, replace=False):   # a few far elements (same parity) in some rows, shared dimensions too
        d = rng.choice(64, 5, replace=False)
        hv[r, d] += np.int16(2) * rng.integers(200, 900, 5).astype(np.int16) * rng.choice([-1, 1], 5).astype(np.int16)
    norm = np.array([oracle.hv_l2_norm_sq(v) for v in hv], np.int32)
    cap = 400 * 400
    peer = hg.Peer(ctx, 0, 1, hg.ffi.peer_window_need(400, 1024, cap))
    try:
        d_hv, d_n = _dev(hv), _dev(norm)
        peer.dist_sharded_dev(None, None, 0, 0, d_hv.data_ptr(), d_n.data_ptr(), [0, 400], 1024, 21, 0.0, True, 3, 0, cap)
        hits, _ = peer.dist_sharded_hits(cap)
        _check_hits(oracle, hits, hv, norm, hv, norm, True, 0.0)
        # the plain single-GPU narrow path shares the rewritten correction
        hits2 = ctx.dist(hv, norm, hv, norm, ani_th=0.0, symmetric=True, path=3, cap=cap)
        _check_hits(oracle, hits2, hv, norm, hv, norm, True, 0.0)
    finally:
        peer.close()


@pytest.mark.parametrize("case", ["narrow_sym", "narrow_refq", "wide_sym", "wide_refq"])
def test_group_dist_packed_two_gpus(hg, oracle, case):
    """one process, two GPUs (hg_group): identical hits, in the reference's output order, to the single-GPU entry"""
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    wide = case.startswith("wide")
    # wide_sym: 10-bit rows with ~1 % of the elements outside one s8 plane (the members' verdict declines, two-limb kernel
    # on the rows already in HBM); wide_refq: 11-bit rows (two-limb kernel chosen from hv_quant_bits alone)
    D, n_per, scaled = {"narrow_sym": (2048, 1700, 1500), "narrow_refq": (2048, 1700, 1500), "wide_sym": (2048, 9000, 500),
                        "wide_refq": (2048, 20000, 200)}[case]
    with hg.Context(0) as c0:
        hv, norm, packed, bits = _sketch_sets(c0, 2300, D, n_per, scaled)
        assert (int(bits.max()) > 10) == (case == "wide_refq")
        sym = case.endswith("sym")
        if sym:
            args = (packed, bits, norm, packed, bits, norm)
        else:
            args = (packed[:1500], bits[:1500], norm[:1500], packed[1100:], bits[1100:], norm[1100:])
        want, want_m = c0.dist_packed(*args, D, ksize=21, ani_th=70.0, symmetric=sym, sorted_output=True)
    with hg.Group(2) as g:
        assert g.size == 2
        got, got_m = g.dist_packed(*args, D, ksize=21, ani_th=70.0, symmetric=sym, sorted_output=True)
        assert g.dist_last_path(0) == (2 if wide else 3) and g.dist_last_path(1) == (2 if wide else 3)
        # a second call reuses the windows (epochs, counters and statistics are reset correctly)
        got2, _ = g.dist_packed(*args, D, ksize=21, ani_th=70.0, symmetric=sym, sorted_output=True)
    assert want.size > 100
    assert np.array_equal(got, want) and np.array_equal(got_m, want_m) and np.array_equal(got2, want)
    r, rn = (hv, norm) if sym else (hv[:1500], norm[:1500])
    q, qn = (hv, norm) if sym else (hv[1100:], norm[1100:])
    _check_hits(oracle, got, r, rn, q, qn, sym, 70.0)


def test_group_sketch_two_gpus_same_bytes(hg, oracle):
    """files split over two GPUs: the same packed sketches, file for file, as one GPU"""
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    from hypergen_b200 import synth
    files = []
    for g in range(9):
        body = synth.family_member(g, 90_000 + 7000 * g).numpy()
        files.append(b">g%d\n" % g + b"".join(bytes(body[t:t + 60]) + b"\n" for t in range(0, body.size, 60)))
    p = hg.make_params(k=21, scaled=1500, seed=123, canonical=True, hv_d=4096)
    with hg.Context(0) as c0:
        want = c0.sketch_fasta_batch(files, p)
    with hg.Group(2) as g:
        got = g.sketch_fasta_batch(files, p)
    for k in ("hv", "quant_bits", "norm2", "n_hashes"):
        assert np.array_equal(got[k], want[k]), k
    for f in range(9):
        nb = int(want["quant_bits"][f]) * 4096 // 8
        assert np.array_equal(got["packed"][f, :nb], want["packed"][f, :nb])


_RANK_SCRIPT = r"""
import os, sys
sys.path.insert(0, %(root)r)
import numpy as np, torch, torch.distributed as dist
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("gloo")
import hypergen_b200 as hg
from hypergen_b200 import multigpu
d = np.load(%(npz)r)
hv, norm = d["hv"], d["norm"]
n, D = hv.shape
ctx = hg.Context(rank)
cap = 1 << 22
pg = multigpu.PeerGroup(ctx, hg.ffi.peer_window_need(n, D, cap))
b = multigpu.block_rows(n, world)
a0, a1 = b[rank], b[rank + 1]
dev = torch.device("cuda", rank)
d_hv = torch.from_numpy(hv[a0:a1].copy()).to(dev); d_n = torch.from_numpy(norm[a0:a1].copy()).to(dev)
out = {}
hv_o, norm_o = d["hv_o"], d["norm_o"]  # the same rows with a few far-off elements: outlier entries travel in the start set
d_hv_o = torch.from_numpy(hv_o[a0:a1].copy()).to(dev); d_n_o = torch.from_numpy(norm_o[a0:a1].copy()).to(dev)
for name, sym, path in (("sym", True, 0), ("sym3", True, 3), ("refq", False, 0), ("sym2", True, 2), ("mapped", True, 3), ("outl", True, 3)):
    mapped = None
    if name == "mapped":  # hits straight into a host buffer both ranks have mapped (POSIX shared memory)
        from multiprocessing import shared_memory
        if rank == 0:
            try:
                shm = shared_memory.SharedMemory(name="hg_test_hits", create=True, size=cap * 16)
            except FileExistsError:  # left behind by a run that died
                old = shared_memory.SharedMemory(name="hg_test_hits"); old.close(); old.unlink()
                shm = shared_memory.SharedMemory(name="hg_test_hits", create=True, size=cap * 16)
        dist.barrier()
        if rank != 0:
            shm = shared_memory.SharedMemory(name="hg_test_hits")
        host_hits = np.ndarray((cap,), dtype=hg.ffi.HIT_DTYPE, buffer=shm.buf)
        mapped = hg.ffi.host_register(host_hits)
    if name == "outl":
        pg.peer.dist_sharded_dev(None, None, 0, 0, d_hv_o.data_ptr(), d_n_o.data_ptr(), b, D, 21, 75.0, True, path, 0, cap, mapped)
    elif sym:
        pg.peer.dist_sharded_dev(None, None, 0, 0, d_hv.data_ptr(), d_n.data_ptr(), b, D, 21, 75.0, True, path, 0, cap, mapped)
    else:  # refs: this rank's block; queries: all on rank 1 (a "broadcast" from a non-root member)
        q_hv = torch.from_numpy(hv.copy()).to(dev) if rank == 1 else None
        q_n = torch.from_numpy(norm.copy()).to(dev) if rank == 1 else None
        pg.peer.dist_sharded_dev(d_hv.data_ptr(), d_n.data_ptr(), a1 - a0, a0, q_hv.data_ptr() if rank == 1 else None,
                                 q_n.data_ptr() if rank == 1 else None, [0, 0, n], D, 21, 75.0, False, path, 0, cap)
    hits, _ = pg.peer.dist_sharded_hits(cap, sorted_output=(mapped is None), hits=host_hits if mapped else None)
    if mapped:
        hits = np.sort(hits.copy(), order=["i", "j"])
        dist.barrier()
        hg.ffi.host_unregister(host_hits)
        del host_hits
        shm.close()
        if rank == 0:
            shm.unlink()
    out[name] = hits
if rank == 0:
    np.savez(%(out)r, **out)
pg.close()
ctx.close()
dist.destroy_process_group()
"""


def test_one_process_per_gpu_ipc_windows(hg, oracle, ctx, tmp_path):
    """two ranks under torchrun (gloo carries the window handles): the hits gathered on rank 0 equal the oracle's"""
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    hv, norm, _, _ = _sketch_sets(ctx, 1900, 2048, 1700, 1500)
    rng = np.random.default_rng(5)
    hv_o = hv.copy()
    for r in rng.choice(1900, 200, replace=False):  # far elements of the row's parity, in both members' blocks
        dd = rng.choice(2048, 4, replace=False)
        hv_o[r, dd] += np.int16(2) * rng.integers(200, 900, 4).astype(np.int16) * rng.choice([-1, 1], 4).astype(np.int16)
    norm_o = np.array([oracle.hv_l2_norm_sq(v) for v in hv_o], np.int32)
    npz, outp, script = str(tmp_path / "in.npz"), str(tmp_path / "out.npz"), str(tmp_path / "rank.py")
    np.savez(npz, hv=hv, norm=norm, hv_o=hv_o, norm_o=norm_o)
    with open(script, "w") as f:
        f.write(_RANK_SCRIPT % dict(root=ROOT, npz=npz, out=outp))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29533", script], capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, HG_NARROW_BUDGET="64"))  # room for the outlier entries of the "outl" case
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    got = np.load(outp)
    from hypergen_b200.ffi import HIT_DTYPE
    _check_hits(oracle, got["sym"].view(HIT_DTYPE), hv, norm, hv, norm, True, 75.0)
    def same(a, b, what):
        if np.array_equal(a, b):
            return
        ka = a["i"].astype(np.int64) * 100000 + a["j"]
        kb = b["i"].astype(np.int64) * 100000 + b["j"]
        ea, eb = a[~np.isin(ka, kb)], b[~np.isin(kb, ka)]
        raise AssertionError("%s: %d vs %d hits; %d only in first (e.g. %s), %d only in second (e.g. %s)"
                             % (what, a.size, b.size, ea.size, ea[:4], eb.size, eb[:4]))
    same(got["sym3"], got["sym"], "forced single-plane vs auto")
    same(got["sym2"], got["sym"], "forced two-limb vs auto")
    same(got["mapped"], np.sort(got["sym"], order=["i", "j"]), "hits in mapped host memory vs window")
    _check_hits(oracle, got["refq"].view(HIT_DTYPE), hv, norm, hv, norm, False, 75.0)
    _check_hits(oracle, got["outl"].view(HIT_DTYPE), hv_o, norm_o, hv_o, norm_o, True, 75.0)


def test_cli_all_gpus_writes_the_same_bytes_as_one_gpu(hg, tmp_path):
    """`hyper-gen sketch` / `hyper-gen dist` over every GPU of the box (hg_group) vs HG_GPUS=1: byte-identical sketch
    file and TSV (src/main.rs:14-21 drives one GPU; the C++ host mirrors its drivers above the C ABI)"""
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    from hypergen_b200 import synth, _build
    exe = _build.build_host()
    d = tmp_path / "genomes"
    d.mkdir()
    for g in range(1200):
        body = synth.family_member(g, 30_000).numpy()
        with open(d / ("g%04d.fna" % g), "wb") as f:
            f.write(b">g%d\n" % g + b"".join(bytes(body[t:t + 80]) + b"\n" for t in range(0, body.size, 80)))
    outs = {}
    for name, env in (("one", dict(os.environ, HG_GPUS="1")), ("all", dict(os.environ))):
        sk, tsv = str(tmp_path / (name + ".sketch")), str(tmp_path / (name + ".tsv"))
        subprocess.check_call([exe, "sketch", "-p", str(d), "-o", sk, "-s", "200", "-d", "1024", "-t", "8"], env=env)
        subprocess.check_call([exe, "dist", "-r", sk, "-q", sk, "-o", tsv, "-a", "80.0"], env=env)
        outs[name] = (open(sk, "rb").read(), open(tsv, "rb").read())
    assert outs["one"][0] == outs["all"][0]
    assert outs["one"][1] == outs["all"][1] and len(outs["all"][1]) > 1000
