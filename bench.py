#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on BASELINE.json's configs, on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Headline (`metric`/`value`): genomes sketched per second, config[1] of BASELINE.json —
1,000 synthetic 5 Mbp genomes, k=21 scaled=1500 D=4096 per GPU (weak scaling: every rank
sketches its own 1,000 genomes, no collective on the data path).  A "step" is one pass of
the sketch hot path (k-mer hash -> set -> HV encode -> norm -> quantise -> bit-pack) over the
whole batch with the sequence bytes already resident in HBM.  `e2e` is the same pass through
the host-pointer C-ABI call (pinned host buffers, H2D of the FASTA bytes and D2H of the
sketches inside the timed region).  The `dist`, `dist_cfg4` and `dist_cfg5` objects carry the
second half of the metric, ANI pairs/s, on configs[2] (10,000 all-vs-all), configs[3]
(100,000 refs x 1,000 queries) and configs[4] (20,000 all-vs-all at scaled=500, D=8192), each
with its own roofline, oracle parity check and CPU baseline; at N > 1 the rows are sharded over
the ranks and exchanged through the library's NVLink windows (csrc/peer.cu).
`reference_gpu_kernel` times the reference's own CUDA kernel (oracle/_ref) on the same GPU.

`--impl reference` times the reference's CPU path restated in C (oracle/hg_oracle.c — the
Rust crate cannot be built here: no cargo/rustc) on the host cores.

`--steps K` is the number of timed steps of every leg.  `--dump-outputs DIR` writes what the sketch
call returned in the last timed step as DIR/<name>.npy (see dump_outputs); the inputs are generated
from fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: leave no __pycache__ in it

K, SCALED, SEED, HV_D = 21, 1500, 123, 4096
GENOME_LEN = 5_000_000
# algorithmic bytes of the k-mer hash kernel per genome: 1 B per base read + 8 B per sampled
# hash written (SURVEY.md §8d) — n ~= L / scaled
ALG_BYTES_PER_GENOME = GENOME_LEN + 8 * (GENOME_LEN // SCALED)
# integer instructions the k-mer kernel executes per k-mer (ncu smsp__inst_executed /
# k-mers, profiles/): used only for the auxiliary INT32 roofline
def _kmer_inst_per_kmer():
    """warp-level instructions per 32 k-mers (= lane instructions per k-mer) of kmer_hash_kernel<21,true>, from the committed
    ncu capture's smsp__inst_executed.sum (profiles/kmer_traffic.json); HG_KMER_INST_PER_KMER overrides"""
    if os.environ.get("HG_KMER_INST_PER_KMER"):
        return float(os.environ["HG_KMER_INST_PER_KMER"])
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "kmer_traffic.json")) as f:
            tj = json.load(f)
        return tj["smsp_inst_executed"] / (tj["genomes_per_launch"] * (5_000_000 - 20) / 32.0)
    except (OSError, KeyError, ValueError):
        return 127.0


KMER_INST_PER_KMER = _kmer_inst_per_kmer()


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=float(d["hbm_gbs"]), bf16_tflops=float(d["bf16_tflops"]),
                    bf16_tflops_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(out_dir: str, outputs: dict):
    """--dump-outputs: one DIR/<name>.npy per array the sketch call returned (one row per genome), converted
    exactly to float32 (8- and 16-bit integers) or float64 (32-bit integers), and DIR/genome.npy, the batch index of
    every row.  A batch whose rows would exceed DUMP_LIMIT_BYTES in all is cut to a sample of rows drawn with a fixed
    seed, the same in every run."""
    wide = {k: np.float64 if v.dtype.itemsize >= 4 else np.float32 for k, v in outputs.items()}
    n = len(next(iter(outputs.values())))
    row_bytes = 8 + sum(np.dtype(wide[k]).itemsize * v[0].size for k, v in outputs.items())
    rows = np.arange(n)
    if n * row_bytes > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT_BYTES // row_bytes, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "genome.npy"), rows.astype(np.float64))
    for k, v in outputs.items():
        np.save(os.path.join(out_dir, k + ".npy"), v[rows].astype(wide[k]))


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (NVML, 50 ms period)."""

    def __init__(self, index: int):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._t = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None
            return self
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def _run(self):
        nv = self._nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                 "hw_power_brake_slowdown": 0x80, "sync_boost": 0x10, "applications_clocks_setting": 0x2}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.05)

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        med = statistics.median(self.samples) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def cpu_sketch_baseline(seq_host: np.ndarray, n_avail: int, seconds_hint: float = 10.0):
    """The restated reference CPU path (oracle, `kind: port`) on a bounded sample, all cores."""
    import oracle as O  # the checker / baseline: never on the product path
    cores = os.cpu_count() or 1
    O.set_threads(cores)
    # ~0.15 s per 5 Mbp genome per core: size the sample for roughly seconds_hint of wall time
    n = int(min(n_avail, max(cores, cores * seconds_hint / 0.15)))
    off = np.arange(n + 1, dtype=np.uint64) * np.uint64(GENOME_LEN)
    t0 = time.perf_counter()
    O.sketch_batch(seq_host[: n * GENOME_LEN], off, k=K, scaled=SCALED, seed=SEED, hv_d=HV_D, want_hv=False)
    dt = time.perf_counter() - t0
    O.set_threads(1)
    t1 = time.perf_counter()
    O.sketch_batch(seq_host[: 4 * GENOME_LEN], off[:5], k=K, scaled=SCALED, seed=SEED, hv_d=HV_D, want_hv=False)
    per_core = 4 / (time.perf_counter() - t1)
    O.set_threads(cores)
    return dict(value=n / dt, unit="genomes/s", cores=cores, kind="port", value_1_thread=per_core,
                sample="%d of the step's 5 Mbp genomes, oracle/hg_oracle.c (C restatement of src/sketch.rs:35-52), %d threads, %.1f s"
                % (n, cores, dt))


def parity_sample(seq_host, packed, bits, norm, n):
    """Checker leg: the e2e results of a few genomes of the timed batch against the oracle."""
    import oracle as O
    pick = sorted(set(list(range(0, n, 50)) + [1, n - 1]))  # every 50th genome of the batch + the ends
    O.set_threads(os.cpu_count() or 1)
    sub = np.concatenate([seq_host[g * GENOME_LEN:(g + 1) * GENOME_LEN] for g in pick])
    off = np.arange(len(pick) + 1, dtype=np.uint64) * np.uint64(GENOME_LEN)
    w = O.sketch_batch(sub, off, k=K, scaled=SCALED, seed=SEED, hv_d=HV_D, want_hv=False)
    bad = 0
    for t, g in enumerate(pick):
        nb = int(w["quant_bits"][t]) * HV_D // 8
        ok = (int(w["quant_bits"][t]) == int(bits[g]) and int(w["norm2"][t]) == int(norm[g])
              and np.array_equal(w["packed"][t, :nb], packed[g, :nb]))
        bad += 0 if ok else 1
    if bad:
        raise RuntimeError("parity check failed on %d of %d sampled genomes" % (bad, len(pick)))
    return "ok: %d genomes of the timed batch (every 50th) bit-identical to the oracle (packed HV, bits, norm)" % len(pick)


def reference_gpu_leg(ctx, params, seq_dev, seq_host, n, our_resident_per_gpu, our_e2e_per_gpu, n_ref_genomes=32):
    """The reference's own GPU kernel (cuda_kmer_t1ha2, /root/reference/src/cuda_kernel.cu:250-321, built by
    oracle/Makefile into oracle/_ref) with its launch geometry (src/sketch_cuda.rs:130-154) on genomes of the timed batch."""
    try:
        from oracle import ref_gpu
        if not ref_gpu.available():
            return {"unavailable": "oracle/_ref holds no GPU image of the reference kernel (built where /root/reference is mounted)"}
        m = min(n, n_ref_genomes)
        out = {}
        sets = None
        for image in ("cubin", "ptx"):
            try:
                r, sets_i = ref_gpu.time_reference_kernel(seq_dev, seq_host, GENOME_LEN, m, K, SCALED, SEED, image=image)
                out[image] = r
                sets = sets or sets_i
            except Exception as ex:  # noqa: BLE001
                out[image] = {"error": str(ex)[:200]}
        best = min((v for v in out.values() if "kernel_ms_per_genome" in v), key=lambda v: v["kernel_ms_per_genome"], default=None)
        if best is None:
            return out
        # its hash sets against ours (set semantics; the reference drops samples beyond 8 per 512-k-mer chunk and h == 0)
        sh = seq_host.numpy()
        missing = extra = 0
        for g, rs in enumerate(sets):
            ours, _ = ctx.kmer_hash(sh[g * GENOME_LEN:(g + 1) * GENOME_LEN], np.array([0, GENOME_LEN], np.uint64), params)
            missing += int((~np.isin(rs, ours)).sum())
            extra += int((~np.isin(ours, rs)).sum())
        out.update({
            "kernel": "cuda_kmer_t1ha2 (reference, unmodified, compiled from /root/reference/src/cuda_kernel.cu where it lies)",
            "genomes_s": best["kernel_genomes_per_s"], "ms": best["kernel_ms_per_genome"], "e2e_genomes_s": best["e2e_genomes_per_s"],
            "scope": "k-mer hashing only (the reference encodes, norms and packs on the CPU afterwards, src/sketch_cuda.rs:85-100)",
            "ours_over_reference_kernel": our_resident_per_gpu / best["kernel_genomes_per_s"],
            "ours_over_reference_e2e": our_e2e_per_gpu / best["e2e_genomes_per_s"],
            "set_check": {"genomes": len(sets), "reference_hashes_missing_from_ours": missing, "ours_not_in_reference": extra,
                          "note": "ours_not_in_reference are the samples the reference kernel drops (more than 8 per 512-k-mer "
                                  "chunk, src/cuda_kernel.cu:316) or h == 0 (src/sketch_cuda.rs:159)"}})
        return out
    except Exception as ex:  # noqa: BLE001
        return {"error": str(ex)[:300]}


def run_reference(args, rank):
    """--impl reference: the reference's CPU algorithm on the host cores (rank 0 only)."""
    if rank != 0:
        return
    import torch
    from hypergen_b200 import synth
    cores = os.cpu_count() or 1
    import oracle as O
    O.set_threads(cores)
    n = int(min(args.genomes, 4 * cores))  # a bounded sample: ~0.3 s of work per step on the box's cores, several genomes per thread
    seq, off = synth.family_batch(n, GENOME_LEN, device="cpu")
    seq = seq.numpy()
    times = []
    for step in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        r = O.sketch_batch(seq, off, k=K, scaled=SCALED, seed=SEED, hv_d=HV_D, want_hv=False)
        if step >= args.warmup:
            times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: v for k, v in r.items() if v is not None})
    total = sum(times)
    value = n * len(times) / total
    line = {
        "impl": "reference", "metric": "genomes sketched/sec (5 Mbp, k=21, D=4096)", "value": value, "unit": "genomes/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "sketch %d synthetic 5 Mbp genomes per step (bounded sample of config[1]), k=21 scaled=1500 D=4096, CPU" % n},
        "cpu_baseline": {"value": value, "unit": "genomes/s", "cores": cores, "kind": "port",
                         "sample": "%d genomes per step; oracle/hg_oracle.c restates src/sketch.rs:35-52 (Rust crate not buildable here: no cargo)" % n},
        "e2e": {"value": value, "unit": "genomes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)


_JSON_OUT = None


def _claim_stdout():
    """Keep stdout for the one JSON line: everything else that writes to fd 1 from here on (NCCL's
    version banner, library chatter) goes to stderr."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def _emit(line: dict):
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--genomes", type=int, default=1000, help="genomes per GPU per step (config[1]: 1000)")
    ap.add_argument("--dist-configs", default="dist,dist_cfg4,dist_cfg5",
                    help="which dist workloads to run: dist (configs[2]), dist_cfg4 (configs[3]), dist_cfg5 (configs[4])")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip timing the reference's own GPU kernel (oracle/_ref)")
    ap.add_argument("--no-dist", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fasta", action="store_true", help="skip the raw-FASTA end-to-end leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the sketch outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world == 1 and "RANK" not in os.environ:
        # convenience: relaunch under torchrun exactly as the driver does
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29577", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))

    _claim_stdout()
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    import hypergen_b200 as hg
    from hypergen_b200 import multigpu, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = multigpu.bind_to_gpu_numa(local_rank) if os.environ.get("HG_NUMA_BIND", "1") != "0" else {"bound": False}
    host_pg = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        host_pg = dist.new_group(backend="gloo")  # host-only waits (an NCCL barrier would park a kernel on the waiting GPUs)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    peaks = load_peaks()
    ctx = hg.Context(local_rank)
    ext = torch.cuda.ExternalStream(ctx.stream, device=dev)
    params = hg.make_params(k=K, scaled=SCALED, seed=SEED, canonical=True, hv_d=HV_D)
    n = args.genomes

    # ---------------- workload: this rank's genomes, generated on the GPU ----------------
    seq_dev, seg_off = synth.family_batch(n, GENOME_LEN, device=dev, first=rank * n)
    d_packed = torch.empty((n, 2 * HV_D), dtype=torch.uint8, device=dev)
    d_bits = torch.empty(n, dtype=torch.uint8, device=dev)
    d_norm = torch.empty(n, dtype=torch.int32, device=dev)
    d_nh = torch.empty(n, dtype=torch.int32, device=dev)
    d_hv = torch.empty((n, HV_D), dtype=torch.int16, device=dev)
    torch.cuda.synchronize()

    def sketch_step():
        ctx.sketch_batch_dev(seq_dev.data_ptr(), seg_off, params, d_hv.data_ptr(), d_packed.data_ptr(),
                             d_bits.data_ptr(), d_norm.data_ptr(), d_nh.data_ptr())

    # ---------------- device-resident timing (`value`) ----------------
    ctx.set_profiling(True)
    for _ in range(args.warmup):
        sketch_step()
    ctx.sync()
    ctx.sketch_status()
    sampler = ClockSampler(local_rank).start()
    barrier()
    l0 = ctx.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stage = []
    with torch.cuda.stream(ext):
        e0.record()
        for _ in range(args.steps):
            sketch_step()
            stage.append(ctx.stage_ms())  # syncs the stream: < 20 us against a ~30 ms step
        e1.record()
    e1.synchronize()
    barrier()
    clocks = sampler.stop()
    launches = ctx.launches - l0
    dev_ms = max_over_ranks(e0.elapsed_time(e1))
    ctx.sketch_status()
    if args.dump_outputs and rank == 0:  # rank 0's genomes (every rank sketches its own)
        dump_outputs(args.dump_outputs, {"hv": d_hv.cpu().numpy(), "packed": d_packed.cpu().numpy(),
                                         "quant_bits": d_bits.cpu().numpy(), "norm2": d_norm.cpu().numpy(),
                                         "n_hashes": d_nh.cpu().numpy()})
    value = world * n * args.steps / (dev_ms * 1e-3)
    kmer_ms = statistics.mean(s[1] for s in stage)
    enc_ms = statistics.mean(s[2] for s in stage)
    stg_ms = statistics.mean(s[0] for s in stage)
    achieved_gbs = n * ALG_BYTES_PER_GENOME / (kmer_ms * 1e-3) / 1e9
    kmers_per_s = n * (GENOME_LEN - K + 1) / (kmer_ms * 1e-3)

    # ---------------- end to end through the host-pointer C ABI ----------------
    seq_host = torch.empty(n * GENOME_LEN, dtype=torch.uint8, pin_memory=True)
    seq_host.copy_(seq_dev)
    h_packed = torch.empty((n, 2 * HV_D), dtype=torch.uint8, pin_memory=True)
    h_bits = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    h_norm = torch.empty(n, dtype=torch.int32, pin_memory=True)
    h_nh = torch.empty(n, dtype=torch.int32, pin_memory=True)
    torch.cuda.synchronize()
    lib = hg.ffi.load()
    import ctypes as C

    def e2e_step():
        rc = lib.hg_sketch_batch(ctx._h, seq_host.data_ptr(), seg_off.ctypes.data, n, C.byref(params), None,
                                 h_packed.data_ptr(), h_bits.data_ptr(), h_norm.data_ptr(), h_nh.data_ptr())
        if rc != 0:
            raise RuntimeError(lib.hg_last_error().decode())

    # H2D of the FASTA bytes alone (north star: reported separately)
    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    scratch_dev = torch.empty_like(seq_dev)
    scratch_dev.copy_(seq_host, non_blocking=True)
    torch.cuda.synchronize()
    h0.record()
    for _ in range(3):
        scratch_dev.copy_(seq_host, non_blocking=True)
    h1.record()
    h1.synchronize()
    h2d_only_gbs = 3 * n * GENOME_LEN / (h0.elapsed_time(h1) * 1e-3) / 1e9
    del scratch_dev

    e2e_steps = args.steps
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()  # synchronous: returns after the D2H of the sketches
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    e2e_value = world * n * e2e_steps / e2e_s
    h2d = int(n * GENOME_LEN + (n + 1) * 8 + n * 40)
    d2h = int(n * 2 * HV_D + n * 9)
    # sanity: the e2e results equal the device-resident ones
    assert torch.equal(h_norm, d_norm.cpu()) and torch.equal(h_bits, d_bits.cpu())

    # ---------------- the same, from raw FASTA file bytes (hg_sketch_fasta_batch) ----------------
    # files = ">g\n" + 80-column lines; the library merges the records on the GPU (fastx_reader::read_merge_seq)
    fasta = None
    if not args.no_fasta:
        hdr = torch.tensor(list(b">g\n"), dtype=torch.uint8, device=dev).expand(n, 3)
        body = torch.cat([seq_dev.view(n, GENOME_LEN // 80, 80),
                          torch.full((n, GENOME_LEN // 80, 1), 10, dtype=torch.uint8, device=dev)], dim=2).view(n, -1)
        raw_dev = torch.cat([hdr, body], dim=1).contiguous()
        file_len = raw_dev.shape[1]
        raw_host = torch.empty(n * file_len, dtype=torch.uint8, pin_memory=True)
        raw_host.copy_(raw_dev.view(-1))
        del raw_dev, body, hdr
        file_off = (np.arange(n + 1, dtype=np.uint64) * np.uint64(file_len))

        def fasta_step():
            rc = lib.hg_sketch_fasta_batch(ctx._h, raw_host.data_ptr(), file_off.ctypes.data, n, C.byref(params), None,
                                           h_packed.data_ptr(), h_bits.data_ptr(), h_norm.data_ptr(), h_nh.data_ptr())
            if rc != 0:
                raise RuntimeError(lib.hg_last_error().decode())

        for _ in range(2):
            fasta_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            fasta_step()
        torch.cuda.synchronize()
        fa_s = max_over_ranks(time.perf_counter() - t0)
        barrier()
        assert torch.equal(h_norm, d_norm.cpu()) and torch.equal(h_bits, d_bits.cpu())
        fasta = {"value": world * n * e2e_steps / fa_s, "unit": "genomes/s", "ms_per_step": 1e3 * fa_s / e2e_steps,
                 "h2d_bytes_per_step": int(n * file_len + (n + 1) * 8 + n * 40), "d2h_bytes_per_step": d2h,
                 "h2d_gbs": world * n * file_len * e2e_steps / fa_s / 1e9,
                 "input": "%d FASTA files of %d bytes (one record, 80-column lines) in pinned host memory; "
                          "records merged on the GPU" % (n, file_len)}
        del raw_host

    # DRAM bytes of one kmer_hash launch, from the committed `ncu --set full` capture (bytes, per launch like `achieved`)
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "kmer_traffic.json")) as f:
            tj = json.load(f)
        traffic = tj["dram_bytes_per_launch"] * (n / tj["genomes_per_launch"])
        traffic_src = tj["source"] + ("" if n == tj["genomes_per_launch"] else " (scaled per genome)")
    except (OSError, KeyError, ValueError):
        pass

    line = {
        "metric": "genomes sketched/sec (5 Mbp, k=21, D=4096)", "value": value, "unit": "genomes/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "sketch %d synthetic 5 Mbp genomes per GPU per step (BASELINE configs[1]), k=21 scaled=1500 D=4096"
                               % n, "genomes_per_gpu": n, "genome_bp": GENOME_LEN, "k": K, "scaled": SCALED, "hv_d": HV_D,
                   "l2": "inputs (%.1f GB per step) larger than L2" % (n * GENOME_LEN / 1e9), "parallelism": "genomes sharded, no collective"},
        "e2e": {"value": e2e_value, "unit": "genomes/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "ms_per_step": 1e3 * e2e_s / e2e_steps,
                "h2d_gbs": world * h2d * e2e_steps / e2e_s / 1e9, "h2d_only_gbs_per_gpu": h2d_only_gbs,
                "h2d_only_genomes_per_s_per_gpu": h2d_only_gbs * 1e9 / GENOME_LEN, "from_fasta_files": fasta},
        "numa": numa,
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "kmer_hash_kernel<21,true>", "achieved": achieved_gbs, "peak": peaks["hbm_gbs"],
                     "unit": "GB/s", "frac": achieved_gbs / peaks["hbm_gbs"], "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": peaks["source"],
                     "alg_bytes_per_launch": n * ALG_BYTES_PER_GENOME, "ms_per_launch": kmer_ms,
                     "note": "bit-exact t1ha2 makes this kernel INT32-issue bound, not HBM bound (SURVEY.md 8d): see roofline_int32"},
        "stages_ms": {"staging_memset": stg_ms, "kmer_hash": kmer_ms, "encode_pack": enc_ms},
    }

    # auxiliary INT32 roofline (denominator measured live with the library's probe kernels)
    int_peak = float("nan")
    try:
        int_peak = ctx.int_peak(2)
        line["roofline_int32"] = {"bound": "int32_issue", "achieved": kmers_per_s * KMER_INST_PER_KMER * 1.0,
                                  "peak": int_peak, "unit": "lane-instr/s", "frac": kmers_per_s * KMER_INST_PER_KMER / int_peak,
                                  "kmers_per_s": kmers_per_s, "inst_per_kmer": KMER_INST_PER_KMER,
                                  "peak_imad_only": ctx.int_peak(0), "peak_alu_only": ctx.int_peak(1),
                                  "peak_source": "measured live by this build's own probe (hg_int_peak, csrc/probe.cu), not a published figure"}
    except Exception as ex:  # pragma: no cover
        line["roofline_int32"] = {"error": str(ex)}

    # ---------------- encode: INT32 roofline (north star: "INT32 ALU for encode") ----------------
    try:
        nh_sum = float(d_nh.sum().item())
        enc_updates = nh_sum * HV_D * (1.0 + 1.0 / 64.0)  # n*D counter updates + n*D/64 wyrng words per genome (SURVEY.md 8d)
        line["roofline_encode"] = {"bound": "int32_alu", "kernel": "encode_kernel", "achieved": enc_updates / (enc_ms * 1e-3),
                                   "peak": int_peak, "unit": "counter updates/s vs lane-instr/s", "frac": enc_updates / (enc_ms * 1e-3) / int_peak,
                                   "ms_per_launch": enc_ms, "alg_updates_per_launch": enc_updates,
                                   "note": "algorithmic work n*D counter updates + n*D/64 wyrng words over the measured dual-pipe INT32 "
                                           "lane-instruction rate; the kernel counts bit-sliced (carry-save adders retire 32 one-bit "
                                           "updates per LOP3), so this is a work-rate ratio, not a pipe utilisation (ncu: profiles/r1_encode_full.md)"}
    except Exception as ex:  # pragma: no cover
        line["roofline_encode"] = {"error": str(ex)}

    # ---------------- the reference's own GPU kernel on this GPU (rank 0) ----------------
    if rank == 0 and not args.no_ref_gpu:
        line["reference_gpu_kernel"] = reference_gpu_leg(ctx, params, seq_dev, seq_host, n, value / world, e2e_value / world)
    barrier()

    # ---------------- dist: configs[2], [3], [4] ----------------
    if not args.no_dist:
        try:
            i8_peak = {"tops": ctx.tensor_peak() / 1e12,
                       "source": "measured live: hg_tensor_peak (tcgen05 kind::i8 256x256x32 MMAs back to back on every TPC)"}
        except Exception as ex:  # pragma: no cover
            i8_peak = {"tops": 2.0 * peaks["bf16_tflops"], "source": "2 x measured bf16 (probe failed: %s)" % ex}
        if world > 1:  # every rank reports its own; the denominators use the slowest
            t = torch.tensor([i8_peak["tops"]], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            i8_peak["tops"] = float(t.item())
        line["int8_tensor_peak"] = dict(i8_peak, unit="TOP/s per GPU", vs_2x_bf16=i8_peak["tops"] / (2.0 * peaks["bf16_tflops"]))
        wanted = [c for c in DIST_CONFIGS if c["key"] in args.dist_configs.split(",")]
        pg = None
        if world > 1 and wanted:
            need = max(hg.ffi.peer_window_need(c.get("n", c.get("n_qry")), c["hv_d"], 4_000_000) for c in wanted)
            pg = multigpu.PeerGroup(ctx, need, dev)
        for cfg in wanted:
            line[cfg["key"]] = bench_dist_config(cfg, args, ctx, ext, hg, multigpu, synth, dev, rank, world, barrier, max_over_ranks,
                                                 i8_peak, pg, host_pg)
            torch.cuda.empty_cache()
        if pg is not None:
            pg.close()

    if rank == 0 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_sketch_baseline(seq_host.numpy(), n) if world == 1 else None
        line["parity_check"] = parity_sample(seq_host.numpy(), h_packed.numpy(), h_bits.numpy(), h_norm.numpy(), n)
        line["config"]["reference_arm"] = ("same_config: false by construction - the CPU reference arm sketches a bounded sample "
                                           "(4 x cores genomes per step) of the same 5 Mbp / k=21 / D=4096 genomes; both report genomes/s; "
                                           "ratios against it scale with the host's %d cores" % (os.cpu_count() or 1))

    if rank == 0:
        _emit(line)
    torch.cuda.synchronize()
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DIST_CONFIGS = [
    dict(key="dist", label="BASELINE configs[2]", n=10000, hv_d=4096, n_per=3333, scaled=1500, symmetric=True, seed=0xD157,
         metric="ANI pairs/sec (all-vs-all, D=4096, ani_th=85)"),
    dict(key="dist_cfg4", label="BASELINE configs[3]", n_ref=100000, n_qry=1000, hv_d=4096, n_per=3333, scaled=1500, symmetric=False,
         seed=0xD157, metric="ANI pairs/sec (database search 100,000 refs x 1,000 queries, D=4096, ani_th=85)"),
    dict(key="dist_cfg5", label="BASELINE configs[4]", n=20000, hv_d=8192, n_per=10000, scaled=500, symmetric=True, seed=0xD158,
         metric="ANI pairs/sec (all-vs-all, scaled=500 D=8192, ani_th=85)"),
]


def encode_family(ctx, synth, dev, n, D, n_per, scaled, seed, want_packed=False):
    """n family-structured sketches encoded on this GPU from device-generated hash sets (never random i16: quant bits and
    norms stay realistic, SURVEY.md 8d).  Deterministic: every rank builds the same matrix."""
    import torch
    hv = torch.empty((n, D), dtype=torch.int16, device=dev)
    norm = torch.empty(n, dtype=torch.int32, device=dev)
    bits = torch.empty(n, dtype=torch.uint8, device=dev)
    packed = torch.empty((n, 2 * D), dtype=torch.uint8, device=dev) if want_packed else None
    chunk = max(256, min(n, (1 << 28) // (8 * n_per)))
    for c0 in range(0, n, chunk):
        m = min(chunk, n - c0)
        hashes, off = synth.hash_sets_family_dev(m, n_per=n_per, scaled=scaled, seed=seed, device=dev, first=c0)
        # the generator's last copies run on torch's stream, the encoder on the library's: without this the encoder can
        # read the tail of `hashes` before it is written (seen once: one rank's row 13332 of config 5 differed from rank 0's)
        torch.cuda.current_stream().synchronize()
        ctx.encode_sets_dev(hashes.data_ptr(), off, D, hv[c0:].data_ptr(), packed[c0:].data_ptr() if want_packed else None,
                            bits[c0:].data_ptr(), norm[c0:].data_ptr())
        ctx.sync()
        del hashes
    return hv, norm, bits, packed


def dist_parity(cfg, hits, ref_hv, ref_norm, qry_hv, qry_norm, th=85.0, sample_rows=64):
    """Checker leg (rank 0): the hit list of the last timed step against the oracle - the hit set, the exact i32 dots and
    the f32 ANI bits.  Config 3 in full (every one of the 49,995,000 pairs); configs 4 / 5 on `sample_rows` ref rows."""
    import oracle as O
    O.set_threads(os.cpu_count() or 1)
    R, Q = ref_hv.shape[0], qry_hv.shape[0]
    sym = cfg["symmetric"]
    t0 = time.perf_counter()
    hi, hj = hits["i"].astype(np.int64), hits["j"].astype(np.int64)
    if sym and R <= 10000:
        r, rn = ref_hv.cpu().numpy(), ref_norm.cpu().numpy()
        ani, dot = O.dist_all(r, rn, r, rn, k=K, symmetric=True)
        dt = time.perf_counter() - t0
        idx = hi * (Q - 1) - hi * (hi - 1) // 2 + (hj - hi - 1)
        want = np.nonzero(ani >= np.float32(th))[0]
        order = np.argsort(idx, kind="stable")
        ok = (idx.size == want.size and np.array_equal(idx[order], want) and np.array_equal(hits["dot"][order], dot[want])
              and np.array_equal(hits["ani"][order].view(np.uint32), ani[want].view(np.uint32)))
        if not ok:
            raise RuntimeError("dist parity failed (%s): GPU hits differ from the oracle" % cfg["key"])
        return ("ok: all %d pairs against the oracle - %d hits, same set, i32 dots equal, f32 ANI bit-identical"
                % (ani.size, want.size)), dict(pairs=int(ani.size), seconds=dt)
    rows = np.unique(np.linspace(0, R - 1, sample_rows).astype(np.int64))
    q, qn = qry_hv.cpu().numpy(), qry_norm.cpu().numpy()
    r, rn = ref_hv[torch_index(rows, ref_hv)].cpu().numpy(), ref_norm[torch_index(rows, ref_norm)].cpu().numpy()
    ani, dot = O.dist_all(r, rn, q, qn, k=K, symmetric=False)
    dt = time.perf_counter() - t0
    ani, dot = ani.reshape(rows.size, Q), dot.reshape(rows.size, Q)
    n_checked = 0
    for t, i in enumerate(rows):
        keep = ani[t] >= np.float32(th)
        if sym:
            keep &= np.arange(Q) > i
        wj = np.nonzero(keep)[0]
        sel = np.nonzero(hi == i)[0]
        sel = sel[np.argsort(hj[sel], kind="stable")]
        ok = (sel.size == wj.size and np.array_equal(hj[sel], wj) and np.array_equal(hits["dot"][sel], dot[t, wj])
              and np.array_equal(hits["ani"][sel].view(np.uint32), ani[t, wj].view(np.uint32)))
        if not ok:
            raise RuntimeError("dist parity failed (%s): ref row %d differs from the oracle: GPU has %d hits (j = %s ...), the oracle %d "
                               "(j = %s ...)" % (cfg["key"], i, sel.size, hj[sel][:6].tolist(), wj.size, wj[:6].tolist()))
        n_checked += wj.size
    return ("ok: %d sampled ref rows x all %d queries against the oracle - %d hits, same set, i32 dots equal, f32 ANI bit-identical"
            % (rows.size, Q, n_checked)), dict(pairs=int(rows.size * Q), seconds=dt)


def torch_index(rows, like):
    import torch
    return torch.from_numpy(rows).to(like.device)


def bench_dist_config(cfg, args, ctx, ext, hg, multigpu, synth, dev, rank, world, barrier, max_over_ranks, i8_peak, pg, host_pg):
    """One dist configuration at this world size.  N = 1: hg_dist_dev, hits written by the kernel straight into pinned
    host memory.  N > 1: hg_dist_sharded_dev over the NVLink windows (every rank holds a block of the rows, turns it
    into operand planes, pushes them to the ranks that compute with them; block pairs owned along the ring; every rank's hits
    moved into one host buffer all GPUs have mapped, which rank 0 reads in place)."""
    import torch
    import torch.distributed as dist
    D, sym = cfg["hv_d"], cfg["symmetric"]
    want_packed = rank == 0 and (cfg["key"] == "dist" or (cfg["key"] == "dist_cfg4" and world > 1))  # the e2e legs' input
    if sym:
        n_ref = n_qry = cfg["n"]
        hv, norm, bits, packed = encode_family(ctx, synth, dev, n_ref, D, cfg["n_per"], cfg["scaled"], cfg["seed"], want_packed)
        ref_hv, ref_norm, qry_hv, qry_norm = hv, norm, hv, norm
        n_pairs = n_ref * (n_ref - 1) // 2
    else:
        n_ref, n_qry = cfg["n_ref"], cfg["n_qry"]
        ref_hv, ref_norm, bits, packed = encode_family(ctx, synth, dev, n_ref, D, cfg["n_per"], cfg["scaled"], cfg["seed"], want_packed)
        q_idx = torch.arange(5, n_ref, n_ref // n_qry, device=dev)[:n_qry]  # queries with relatives among the refs
        qry_hv, qry_norm = ref_hv[q_idx].contiguous(), ref_norm[q_idx].contiguous()
        n_pairs = n_ref * n_qry
    if world > 1:  # every rank generated the matrices itself: they must be the same bytes everywhere
        sums = [None] * world
        dist.all_gather_object(sums, (int(ref_hv.view(torch.int64).sum().item()), int(ref_norm.to(torch.int64).sum().item())), group=host_pg)
        if any(x != sums[0] for x in sums):
            raise RuntimeError("%s: the ranks' synthetic matrices differ: %s" % (cfg["key"], sums))
    cap = 4_000_000
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    hits_pin = torch.empty(cap * 16, dtype=torch.uint8, pin_memory=True)
    hits_np = hits_pin.numpy().view(hg.ffi.HIT_DTYPE)
    qb = multigpu.block_rows(n_qry, world)
    rb = multigpu.block_rows(n_ref, world)
    if world == 1:
        d_cnt = torch.zeros(1, dtype=torch.int64, device=dev)
        cnt_pin = torch.zeros(1, dtype=torch.int64, pin_memory=True)

        def step(path, done=None):
            ctx.dist_dev(ref_hv.data_ptr(), ref_norm.data_ptr(), n_ref, 0, qry_hv.data_ptr(), qry_norm.data_ptr(), n_qry, 0, D, K,
                         85.0, sym, path, hits_pin.data_ptr(), cap, d_cnt.data_ptr())  # hits land in host memory as they are found
            cnt_pin.copy_(d_cnt, non_blocking=True)
            if done is not None:
                done.record()  # everything of the step, the count's D2H included, is in the stream ahead of this event
            torch.cuda.current_stream().synchronize()
            c = int(cnt_pin.item())
            if c > cap:
                raise RuntimeError("hit buffer too small: %d > %d" % (c, cap))
            return hits_np[:c]
    else:
        a, b = qb[rank], qb[rank + 1]
        ra, rbb = rb[rank], rb[rank + 1]
        # the hit list lives in host memory that every rank's GPU has mapped (POSIX shared memory): records cross each
        # GPU's own PCIe link while the kernels run, and rank 0 reads them in place
        from multiprocessing import shared_memory
        shm_name = "hg_bench_hits_%s_%s" % (os.environ.get("MASTER_PORT", "0"), cfg["key"])
        shm = None
        if rank == 0:
            try:
                shm = shared_memory.SharedMemory(name=shm_name, create=True, size=cap * 16)
            except FileExistsError:  # left behind by a run that died: take it over
                old = shared_memory.SharedMemory(name=shm_name)
                old.close()
                old.unlink()
                shm = shared_memory.SharedMemory(name=shm_name, create=True, size=cap * 16)
        dist.barrier(group=host_pg)
        if rank != 0:
            shm = shared_memory.SharedMemory(name=shm_name)
        hits_np = np.ndarray((cap,), dtype=hg.ffi.HIT_DTYPE, buffer=shm.buf)
        mapped = hg.ffi.host_register(hits_np)

        def step(path, done=None):
            if sym:
                pg.peer.dist_sharded_dev(None, None, 0, 0, qry_hv[a:b].data_ptr(), qry_norm[a:b].data_ptr(), qb, D, K, 85.0, True, path,
                                         0, cap, mapped)
            else:  # refs: this rank's resident block; queries: every rank holds 1/N of them (as hg_group_dist_packed deals them)
                pg.peer.dist_sharded_dev(ref_hv[ra:rbb].data_ptr(), ref_norm[ra:rbb].data_ptr(), rbb - ra, ra, qry_hv[a:b].data_ptr(),
                                         qry_norm[a:b].data_ptr(), qb, D, K, 85.0, False, path, 0, cap, mapped)
            if done is not None:
                done.record()  # the call's last node (status + hit counters to host memory) is in the stream ahead of this event
            h, _ = pg.peer.dist_sharded_hits(cap, hits=hits_np)
            return h

    ctx.set_profiling(True)
    with torch.cuda.stream(ext):
        step(0)  # auto: single-plane tensor kernel if the rows are narrow, else two-limb; records why
    path, path_reason = ctx.dist_last_path, ctx.dist_last_reason
    steps = args.steps
    tot_ms, kern_ms, hits, stages = 0.0, [], None, []

    def one_step(timed):
        flush.fill_(1)  # the operands of config 3 fit in L2: flush it between timed iterations
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(ext):
            if world > 1:
                # the GPUs meet at a device-side barrier first: the step is timed from a common start, as in back-to-back
                # calls, not from whenever each rank's host happened to get its launch out after the host barrier
                pg.peer.barrier()
            e0.record()
            h = step(path, e1)
        e1.synchronize()
        return h, max_over_ranks(e0.elapsed_time(e1))

    if world == 1:
        for _ in range(3):
            one_step(False)
        for _ in range(steps):
            hits, ms = one_step(True)
            tot_ms += ms
            kern_ms.append(ctx.stage_ms()[3])
    else:
        # stage times from profiled steps (the library launches node by node when it profiles) ...
        for _ in range(4):
            one_step(False)
            kern_ms.append(max_over_ranks(ctx.stage_ms()[3]))
            stages.append(pg.peer.stage_ms())
        kern_ms, stages = kern_ms[1:], stages[1:]
        # ... the timed steps replay the member's launch sequence as a CUDA graph (captured on the second identical call)
        ctx.set_profiling(False)
        for _ in range(3):
            one_step(False)
        for _ in range(steps):
            hits, ms = one_step(True)
            tot_ms += ms
    if world == 1 and path == 3:
        ctx.dist_status()  # the verdict the forced single-plane calls did not wait for
    kms = statistics.mean(kern_ms)
    del flush
    out = {
        "metric": cfg["metric"], "unit": "pairs/s", "value": n_pairs * steps / (tot_ms * 1e-3), "kernel_value": n_pairs / (kms * 1e-3),
        "ms_per_step": tot_ms / steps, "kernel_ms": kms, "steps": steps, "hits": int(hits.size) if rank == 0 else None, "pairs": n_pairs,
        "n_gpus": world, "path": path, "path_reason": path_reason,
        "rank0_stages_ms": (dict(zip(("operand_form_of_my_rows", "(unused)", "dist_kernel_with_pusher_warps_and_waits_for_peer_chunks",
                                      "hit_flush_to_root_and_final_barrier"),
                                     [statistics.mean(x[i] for x in stages) for i in range(4)])) if stages else None),
        "timing": ("ms_per_step: CUDA events on the library's stream around everything the step enqueues (operand form, kernels, hit "
                   "records and their count into host memory), max over ranks; the host's wake-up after the stream drains is not in it" +
                   ("; every rank's stream passes a device-side barrier before the first event (common start, host launch skew excluded)"
                    if world > 1 else "") +
                   ("; kernel_ms / stages from separate profiled steps (direct launches), the timed steps replay a CUDA graph"
                    if world > 1 else "; kernel_ms from the same steps")),
        "config": {"workload": ("all-vs-all dist over %d synthetic sketches (%s), D=%d, ani_th=85" % (n_ref, cfg["label"], D)) if sym else
                   ("%d ref sketches x %d queries (%s), D=%d, ani_th=85" % (n_ref, n_qry, cfg["label"], D)),
                   "rows_per_rank": ([qb[r + 1] - qb[r] for r in range(world)] if sym else [rb[r + 1] - rb[r] for r in range(world)]),
                   "sharding": ("single GPU; hits written by the kernel into pinned host memory" if world == 1 else
                                ("rows sharded in blocks of 256-row tile rows; operand planes pushed over NVLink windows in chunks with "
                                 "arrival flags the kernels' TMA producers wait on; " +
                                 "block pairs owned along the ring: a rank's rows go to the N/2 ranks that compute with them" +
                                 "; hits appended into one host buffer every GPU has mapped" if sym else
                                 "ref rows sharded and resident; every rank holds 1/N of the queries and pushes their operand plane to "
                                 "every GPU (chunks + arrival flags); hits appended into one host buffer every GPU has mapped")),
                   "step": "i16 rows resident in HBM -> operand form -> dist kernel -> hit list in rank 0's host memory",
                   "l2": "flushed between iterations"},
    }
    alg_ops = 2.0 * D * n_pairs
    mac_mult = 1.0 if path == 3 else 4.0
    peak = i8_peak["tops"] * world
    out["roofline"] = {"bound": "tensor", "achieved": alg_ops / (kms * 1e-3) / 1e12, "peak": peak, "unit": "TOP/s",
                       "frac": alg_ops / (kms * 1e-3) / 1e12 / peak, "executed_frac": mac_mult * alg_ops / (kms * 1e-3) / 1e12 / peak,
                       "frac_of_step": alg_ops / (tot_ms / steps * 1e-3) / 1e12 / peak, "peak_source": i8_peak["source"],
                       "note": "algorithmic 2*D integer ops per pair over kernel_ms (operand pre-pass" +
                               (", NVLink push and barrier" if world > 1 else "") + " + dist kernel, max over ranks); peak = n_gpus x " +
                               "tcgen05 kind::i8 rate; " + ("single s8 plane: executed MACs = algorithmic MACs" if path == 3 else
                                                            "two s8 limbs: 4 MMAs per algorithmic MAC, frac tops out at 0.25"),
                       "traffic": (165.0e6 if (path == 3 and cfg["key"] == "dist" and world == 1) else None)}
    # ---- parity of the timed step's result + CPU baseline (rank 0) ----
    if rank == 0 and not args.no_cpu_baseline:
        msg, cost = dist_parity(cfg, hits.copy(), ref_hv, ref_norm, qry_hv, qry_norm)
        out["parity_check"] = msg
        cores = os.cpu_count() or 1
        out["cpu_baseline"] = {"value": cost["pairs"] / cost["seconds"], "unit": "pairs/s", "cores": cores, "kind": "port",
                               "sample": "%d pairs of this workload, oracle/hg_oracle.c (dist.rs:139-161,231-294 restated), %d threads, %.1f s"
                               % (cost["pairs"], cores, cost["seconds"])}
    # ---- end to end through the host-pointer C ABI ----
    import ctypes as C
    lib = hg.ffi.load()
    if world == 1 and cfg["key"] == "dist":
        out.update(dist_e2e_single(ctx, hg, lib, ref_hv, ref_norm, bits, packed, n_ref, D, cap, path, n_pairs, hits, args.steps))
    if cfg["key"] in ("dist", "dist_cfg4") and world > 1:
        # `hyper-gen dist` with all GPUs behind one process (hg_group_dist_packed): rank 0 drives the N GPUs from packed
        # sketch rows in pinned host memory while the other ranks wait on the host
        if rank == 0:
            width = int(bits.max().item()) * D // 8
            rp = torch.empty((n_ref, width), dtype=torch.uint8, pin_memory=True); rp.copy_(packed[:, :width])
            rbt = torch.empty(n_ref, dtype=torch.uint8, pin_memory=True); rbt.copy_(bits)
            rn = torch.empty(n_ref, dtype=torch.int32, pin_memory=True); rn.copy_(ref_norm)
            if sym:
                qp, qbt, qn, nq = rp, rbt, rn, n_ref
            else:
                qi = q_idx.cpu()
                qp = torch.empty((n_qry, width), dtype=torch.uint8, pin_memory=True); qp.copy_(rp[qi])
                qbt = torch.empty(n_qry, dtype=torch.uint8, pin_memory=True); qbt.copy_(rbt[qi])
                qn = torch.empty(n_qry, dtype=torch.int32, pin_memory=True); qn.copy_(rn[qi])
                nq = n_qry
            milli = torch.empty(cap, dtype=torch.int32, pin_memory=True)
            nh = C.c_uint64(0)
            torch.cuda.synchronize()
            grp = hg.Group(world)

            def gcall():
                rc = lib.hg_group_dist_packed(grp._h, rp.data_ptr(), width, rbt.data_ptr(), rn.data_ptr(), n_ref, qp.data_ptr(), width,
                                              qbt.data_ptr(), qn.data_ptr(), nq, D, K, 85.0, int(sym), 1, hits_pin.data_ptr(),
                                              milli.data_ptr(), cap, C.byref(nh))
                if rc != 0:
                    raise RuntimeError(lib.hg_last_error().decode())

            gcall(); gcall()
            t0 = time.perf_counter()
            reps = args.steps
            for _ in range(reps):
                gcall()
            dtg = (time.perf_counter() - t0) / reps
            out["e2e"] = {"value": n_pairs / dtg, "unit": "pairs/s", "ms_per_step": dtg * 1e3,
                          "h2d_bytes_per_step": int(rp.numel() + (0 if sym else qp.numel()) + (n_ref + (0 if sym else nq)) * 5),
                          "d2h_bytes_per_step": int(nh.value * 20 + 8), "hits": int(nh.value),
                          "same_hit_count_as_resident_step": bool(nh.value == hits.size),
                          "call": "hg_group_dist_packed: one process, %d GPUs, packed sketch rows in pinned host memory -> sorted hits" % world}
            grp.close()
        dist.barrier(group=host_pg)
    if world > 1:
        hits = None
        dist.barrier(group=host_pg)
        hg.ffi.host_unregister(hits_np)
        del hits_np
        shm.close()
        if rank == 0:
            shm.unlink()
    return out


def dist_e2e_single(ctx, hg, lib, hv, norm, bits, packed_d, nq, D, cap, path, n_pairs, hits_ref, reps):
    """config 3 through the single-GPU host-pointer entries (hg_dist, hg_dist_sorted, hg_dist_packed)"""
    import ctypes as C
    import torch
    out = {}
    hv_h = torch.empty((nq, D), dtype=torch.int16, pin_memory=True)
    norm_h = torch.empty(nq, dtype=torch.int32, pin_memory=True)
    hv_h.copy_(hv)
    norm_h.copy_(norm)
    hits_h = torch.empty(cap * 16, dtype=torch.uint8, pin_memory=True)
    torch.cuda.synchronize()
    n_hits_c = C.c_uint64(0)

    def e2e():
        rc = lib.hg_dist(ctx._h, hv_h.data_ptr(), norm_h.data_ptr(), nq, hv_h.data_ptr(), norm_h.data_ptr(), nq, D, K,
                         85.0, 1, path, hits_h.data_ptr(), cap, C.byref(n_hits_c))
        if rc != 0:
            raise RuntimeError(lib.hg_last_error().decode())

    e2e()
    t0 = time.perf_counter()
    for _ in range(reps):
        e2e()
    dt = (time.perf_counter() - t0) / reps
    assert n_hits_c.value == hits_ref.size
    out["e2e"] = {"value": n_pairs / dt, "unit": "pairs/s", "h2d_bytes_per_step": int(hv_h.numel() * 2 + norm_h.numel() * 4),
                  "d2h_bytes_per_step": int(n_hits_c.value * 16 + 8), "ms_per_step": dt * 1e3,
                  "call": "hg_dist: pinned host i16 matrices -> hits"}
    milli_h = torch.empty(cap, dtype=torch.int32, pin_memory=True)

    def e2e_sorted():
        rc = lib.hg_dist_sorted(ctx._h, hv_h.data_ptr(), norm_h.data_ptr(), nq, hv_h.data_ptr(), norm_h.data_ptr(), nq, D,
                                K, 85.0, 1, path, hits_h.data_ptr(), milli_h.data_ptr(), cap, C.byref(n_hits_c))
        if rc != 0:
            raise RuntimeError(lib.hg_last_error().decode())

    e2e_sorted()
    t0 = time.perf_counter()
    for _ in range(reps):
        e2e_sorted()
    dts = (time.perf_counter() - t0) / reps
    hs = hits_h[: n_hits_c.value * 16].numpy().view(hg.ffi.HIT_DTYPE).copy()
    ok = bool(np.all((hs["ani"][:-1] > hs["ani"][1:]) | ((hs["ani"][:-1] == hs["ani"][1:]) & (
        (hs["i"][:-1] > hs["i"][1:]) | ((hs["i"][:-1] == hs["i"][1:]) & (hs["j"][:-1] > hs["j"][1:]))))))
    same = bool(np.array_equal(np.sort(hs, order=["i", "j"]), np.sort(hits_ref, order=["i", "j"])))
    out["e2e_sorted"] = {"value": n_pairs / dts, "unit": "pairs/s", "ms_per_step": dts * 1e3, "sort_ms": (dts - dt) * 1e3,
                         "d2h_bytes_per_step": int(n_hits_c.value * 20 + 8), "order_verified": ok, "same_hits_as_resident_step": same,
                         "note": "hg_dist_sorted: hits radix-sorted on the GPU into dump_ani_file's order (utils.rs:262-285)"}
    bits_np = bits.cpu().numpy()
    width = int(bits_np.max()) * D // 8
    packed_h = torch.empty((nq, 2 * D), dtype=torch.uint8, pin_memory=True)
    packed_h.copy_(packed_d)
    bits_h = torch.empty(nq, dtype=torch.uint8, pin_memory=True)
    bits_h.copy_(bits)
    torch.cuda.synchronize()

    def e2e_packed():
        rc = lib.hg_dist_packed(ctx._h, packed_h.data_ptr(), 2 * D, bits_h.data_ptr(), norm_h.data_ptr(), nq,
                                packed_h.data_ptr(), 2 * D, bits_h.data_ptr(), norm_h.data_ptr(), nq, D, K, 85.0, 1, 0, 1,
                                hits_h.data_ptr(), milli_h.data_ptr(), cap, C.byref(n_hits_c))
        if rc != 0:
            raise RuntimeError(lib.hg_last_error().decode())

    e2e_packed()
    t0 = time.perf_counter()
    for _ in range(reps):
        e2e_packed()
    dtp = (time.perf_counter() - t0) / reps
    hp = hits_h[: n_hits_c.value * 16].numpy().view(hg.ffi.HIT_DTYPE)
    out["e2e_packed_sorted"] = {"value": n_pairs / dtp, "unit": "pairs/s", "ms_per_step": dtp * 1e3,
                                "h2d_bytes_per_step": int(nq * width + nq * 5), "d2h_bytes_per_step": int(n_hits_c.value * 20 + 8),
                                "same_hits_as_sorted": bool(n_hits_c.value == hs.size and np.array_equal(hp, hs)),
                                "note": "hg_dist_packed: %d-bit packed sketch rows over PCIe, decompress + dist + sort on the GPU" % int(bits_np.max())}
    return out


if __name__ == "__main__":
    main()
