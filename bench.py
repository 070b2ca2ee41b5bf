#!/usr/bin/env python
"""bench.py -- batch-fetch throughput of the get() hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU; torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU MPI_Get path on host cores

Headline workload (BASELINE.json configs[1]): 10,000,000 samples x 1024 float32 (4096 B rows, 40.96 GB) sharded by
contiguous blocks over the N GPUs; one "step" = every rank fetches one batch of B=65536 uniform-random samples
(268 MB) into a packed device buffer. Payload is synthetic (splitmix64 of the element index, generated on device);
indices are seeded per rank and per step.

Printed JSON (one line, rank 0):
  value      aggregate GB/s over all ranks, indices and output resident in HBM: one block of exactly K back-to-back
             async launches between two CUDA events on the launching stream, barrier + synchronize on both sides, max
             over ranks
  verified_rows  rows of the LAST timed batch of every rank regenerated and compared on the device (all of them, at
             every N), with the number of requests every owner served
  e2e        same metric through the host-facing call: pinned HOST index arrays in, pinned HOST buffer out,
             H2D + kernel + D2H all inside the timed region; next to it the same call into a PAGEABLE buffer (the
             reference's np.zeros contract) and a plain pinned D2H copy of the same size (the PCIe ceiling of this box)
  roofline   dominant kernel (dds_gather_kernel): algorithmic bytes = 2 x payload (one HBM read + one HBM write per byte
             at N=1; payload x (N-1)/N over NVLink at N>1), per-launch duration from CUDA events on the launching stream
  cpu_baseline  oracle/_ref (the unmodified reference compiled against the MPI thread-rank shim) doing the same
             per-sample get() loop on the host cores, on a bounded sample of the workload
  configs    the other BASELINE.json configs, each with value / ms_per_step / roofline / verified_rows and (N=1) the
             reference's get() loop on the same shape: cfg3 variable-length (explicit and by sample id, B=4096/16384),
             cfg4 multi-array in one launch, cfg5 size sweep 1 KiB..16 MiB (mode A: all ranks; mode B: one requester),
             the config-1 row shape, the legacy per-sample loop, streaming ingest and prefetch overlap
"""
import argparse
import ctypes
import glob
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

TOTAL_SAMPLES = 10_000_000
DISP = 1024
ROW_BYTES = DISP * 4
SEED = 0xDD5
METRIC = "batch_fetch_GBps"
UNIT = "GB/s"
NVLINK_PEAK = 770.0  # GB/s per direction, peer-copy figure of /opt/skills/guides/B200_PROFILING.md (not in MEASURED_PEAKS.json)
CFG5_SIZES = (1 << 10, 4 << 10, 16 << 10, 64 << 10, 256 << 10, 1 << 20, 4 << 20, 16 << 20)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed launches of the headline, in one block")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=10,
                    help="how many times the timed block of each extra config is repeated (the headline times --steps steps)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=65536, help="samples per rank per step")
    ap.add_argument("--samples", type=int, default=TOTAL_SAMPLES, help="total samples (default: the full config)")
    ap.add_argument("--cpu-samples", type=int, default=1_000_000, help="rows in the CPU baseline's bounded sample")
    ap.add_argument("--cpu-batch", type=int, default=32768, help="get() calls per rank-thread per CPU step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="headline workload only")
    ap.add_argument("--push", action="store_true",
                    help="N > 1: also measure the collective owner-push fetch (slower than the pull at every N measured, "
                         "profiles/r2_configs.md; a rank that dies inside it makes the others trap after 30 s, so it is not part "
                         "of the default run)")
    ap.add_argument("--configs", default="cfg3,cfg4,cfg5,cfg1,persample,ingest,prefetch")
    ap.add_argument("--config-scale", type=float, default=1.0, help="shrink the stores of the extra configs (tests)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed seeded sample of the rows the headline's last timed step "
                         "fetched to DIR/batch_rows_rank<r>.npy (the rows' 32-bit words as float64; 4096 rows, 32 MiB, "
                         "over all ranks together), to compare two builds output for output")
    return ap.parse_args()


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def np_synth_rows(seed, first_global_row, nrows, disp, dtype):
    """host recomputation of the device payload generator (SURVEY.md 8d): low bytes of splitmix64(seed ^ index)"""
    dtype = np.dtype(dtype)
    g = (np.arange(nrows, dtype=np.uint64)[:, None] + np.uint64(first_global_row)) * np.uint64(disp) \
        + np.arange(disp, dtype=np.uint64)[None, :]
    x = (g ^ np.uint64(seed)) + np.uint64(0x9E3779B97F4A7C15)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    x = x ^ (x >> np.uint64(31))
    raw = x.view(np.uint8).reshape(nrows, disp, 8)[:, :, :dtype.itemsize]
    return np.ascontiguousarray(raw).view(dtype).reshape(nrows, disp)


def bind_to_gpu_numa(gpu_index):
    """pin this rank to the CPUs next to its GPU (NVML's ideal affinity) so pinned host buffers and the PCIe
    copies of the e2e path stay on the GPU's NUMA node"""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
    except Exception:  # noqa: BLE001 -- best effort
        pass


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------- index tables of configs 3 / 4
def cfg3_tables(nsamp):
    """config 3: sample lengths U{100..10000} float32 elements (disp=1), default_rng(42)"""
    L = np.random.default_rng(42).integers(100, 10001, size=nsamp)
    return np.concatenate([[0], np.cumsum(L)]), L


def cfg4_tables(nsamp):
    """config 4: node_feat f32 [n, 16], n ~ U{8..512}; edge_index i64 [8n, 2]"""
    n = np.random.default_rng(43).integers(8, 513, size=nsamp)
    e = 8 * n
    return np.concatenate([[0], np.cumsum(n)]), n, np.concatenate([[0], np.cumsum(e)]), e


def workload_config(N, total, B):
    """the `config` object BOTH arms print: it names the workload (BASELINE.json configs[1]); how an arm runs it -- the
    GPU arm's queue and kernel geometry, the CPU arm's bounded sample -- is said elsewhere in its line"""
    per = total // N
    return {"workload": "configs[1]: 10M fixed-length 1024-float32 samples, uniform-random batch fetch",
            "total_samples": total, "row_bytes": ROW_BYTES, "batch_per_gpu": B, "bytes_per_step_per_gpu": B * ROW_BYTES,
            "store_bytes": total * ROW_BYTES,
            "l2": "inputs larger than L2 (random rows of a %.1f GB shard per GPU; 268 MB output)" % (per * ROW_BYTES / 1e9),
            "parallelism": f"store sharded over {N} GPU(s) by contiguous blocks of rows (the reference's lenlist partition), no collective"}


# --------------------------------------------------------------------------------------------- reference arm
def host_cpu_info():
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    return cores


def calibrate_threads(cpu_samples, cpu_batch):
    """'all the host threads it can use': more rank-threads than the memory system can feed only adds contention, and
    threads spread over both sockets pay for remote memory, so time a short run for every candidate (cpu set, thread
    count) and keep the fastest. Returns (threads, cpu-set tag); the process affinity is left on the winning set."""
    cores = host_cpu_info()
    base = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    cpu_sets = [("all", base)]
    for nd in sorted(glob.glob("/sys/devices/system/node/node[0-9]*")):
        try:
            cpus = set()
            for part in open(os.path.join(nd, "cpulist")).read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus |= set(range(int(lo), int(hi or lo) + 1))
            if base is not None and cpus & base and (cpus & base) != base:
                cpu_sets.append((os.path.basename(nd), cpus & base))
        except Exception:  # noqa: BLE001
            pass
    best = None
    for tag, cset in cpu_sets:
        if cset is not None:
            os.sched_setaffinity(0, cset)
        ncs = len(cset) if cset is not None else cores
        for cand in sorted({c for c in (8, 16, 32, 64, 128, ncs) if c <= ncs} | {min(ncs, 8)}):
            g, _ = cpu_reference_run(min(cpu_samples, 250_000), cpu_batch // 4, 2, 1, nthreads=cand)
            if best is None or g > best[0]:
                best = (g, cand, cset, tag)
    if best[2] is not None:
        os.sched_setaffinity(0, best[2])
    return best[1], best[3]


_CAL = {}


def reference_world():
    """-> (kind, world class): the compiled reference when oracle/_ref is built, else the oracle's C port"""
    from oracle import oracle as O
    return ("reference", O.RefWorld) if O.have_ref() else ("port", O.PortWorld)


def cpu_reference_run(cpu_samples, cpu_batch, steps, warmup, nthreads=None):
    """The reference's own get() path on the host cores: the UNMODIFIED DDStore (method 0) compiled against the
    MPI thread-rank shim when oracle/_ref is built, else the oracle's C port. One rank-thread per core,
    each doing `cpu_batch` blocking single-row get() calls per step into a packed host buffer -- the loader loop
    of examples/vae/distdataset.py:79-89. Returns (GB/s aggregate, info dict)."""
    from oracle import oracle as O
    cores = host_cpu_info()
    if nthreads is None:
        if "threads" not in _CAL:
            _CAL["threads"], _CAL["cpu_set"] = calibrate_threads(cpu_samples, cpu_batch)
        nthreads = _CAL["threads"]
    P = max(1, min(256, nthreads))
    per = cpu_samples // P
    co = O.COracle()
    shards = [co.synth_rows(SEED, r * per, per, DISP, np.float32) for r in range(P)]
    total = per * P
    rngs = [np.random.default_rng(1234 + r) for r in range(P)]
    outs = [np.empty(cpu_batch * ROW_BYTES, np.uint8) for _ in range(P)]
    counts = [np.ones(cpu_batch, np.int64) for _ in range(P)]
    times = []
    kind, World = reference_world()
    w = World(P)
    w.add("x", shards)
    for it in range(warmup + steps):
        starts = [rng.integers(0, total, size=cpu_batch) for rng in rngs]
        ns = w.get_loop_all("x", starts, counts, outs)
        if ns < 0:
            raise RuntimeError("reference get() failed: " + w.err())
        if it >= warmup:
            times.append(ns * 1e-9)
    # parity spot check of the timed path against the generator
    exp = co.synth_rows(SEED, int(starts[0][-1]), 1, DISP, np.float32)
    assert outs[0][-ROW_BYTES:].tobytes() == exp.tobytes()
    w.close()
    step_bytes = P * cpu_batch * ROW_BYTES
    t = float(np.sum(times))
    gbs = step_bytes * len(times) / t / 1e9
    info = {"value": gbs, "unit": UNIT, "cores": P, "kind": kind,
            "sample": f"{P} rank-threads (fastest of the calibrated thread counts / cpu sets) x {cpu_batch} single-row "
                      f"get() per step x {len(times)} steps on a {total}-row ({total * ROW_BYTES / 1e9:.2f} GB) slice "
                      f"of the workload, host buffers",
            "samples_per_s": P * cpu_batch * len(times) / t, "host_cpus": cores,
            "cpu_set": _CAL.get("cpu_set", "inherited"),
            "ms_per_step": 1e3 * t / len(times)}
    return gbs, info


def cpu_reference_configs(names, nthreads, steps=3, warmup=1):
    """The reference's get() loop (count > 1: ONE MPI_Get of count rows per request, ddstore.hpp:229-236) on the shapes of
    configs 3 / 4 / 5 / 1, bounded samples, `nthreads` rank-threads. -> {config name: {value, samples_per_s, ...}}"""
    from oracle import oracle as O
    kind, World = reference_world()
    co = O.COracle()
    P = max(1, nthreads)
    out = {}

    def loop(world, var_runs, nbytes_per_step, nsamples_per_step, label):
        """var_runs: list of (name, starts_per_rank, counts_per_rank, outs) timed back to back (multi-array samples)"""
        ts = []
        for it in range(warmup + steps):
            t = 0.0
            for (nm, st, ct, ob) in var_runs:
                ns = world.get_loop_all(nm, st, ct, ob)
                if ns < 0:
                    raise RuntimeError("reference get() failed: " + world.err())
                t += ns * 1e-9
            if it >= warmup:
                ts.append(t)
        tt = float(np.mean(ts))
        return {"value": nbytes_per_step / tt / 1e9, "unit": UNIT, "samples_per_s": nsamples_per_step / tt,
                "ms_per_step": 1e3 * tt, "cores": P, "kind": kind, "sample": label}

    if "cfg3" in names:
        nsamp = 2048 * P  # ~20 KB each: ~40 MB per rank-thread
        sstart, L = cfg3_tables(nsamp)
        per = nsamp // P
        shards = [co.synth_rows(SEED, int(sstart[r * per]), int(sstart[(r + 1) * per] - sstart[r * per]), 1, np.float32)
                  for r in range(P)]
        w = World(P)
        w.add("x", shards)
        del shards
        for B in (4096, 16384):
            b = min(B, 1024)  # requests per rank-thread per step (bounded; the loop's cost per request is what matters)
            ids = [np.random.default_rng(1234 + r).integers(0, nsamp, size=b) for r in range(P)]
            st, ct = [sstart[i] for i in ids], [L[i] for i in ids]
            outs = [np.empty(int(c.sum()) * 4, np.uint8) for c in ct]
            nb = sum(int(c.sum()) * 4 for c in ct)
            out[f"cfg3_B{B}"] = loop(w, [("x", st, ct, outs)], nb, b * P,
                                     f"{P} rank-threads x {b} get(count=L_i) per step on a {nsamp}-sample "
                                     f"({int(sstart[-1]) * 4 / 1e9:.2f} GB) store")
            exp = co.synth_rows(SEED, int(st[0][-1]), int(ct[0][-1]), 1, np.float32)
            assert outs[0][-exp.nbytes:].tobytes() == exp.tobytes()
        w.close()
    if "cfg4" in names:
        nsamp = 1024 * P
        ns_, n, es_, e = cfg4_tables(nsamp)
        per = nsamp // P
        nf = [co.synth_rows(SEED, int(ns_[r * per]), int(ns_[(r + 1) * per] - ns_[r * per]), 16, np.float32) for r in range(P)]
        ei = [co.synth_rows(SEED + 1, int(es_[r * per]), int(es_[(r + 1) * per] - es_[r * per]), 2, np.int64) for r in range(P)]
        w = World(P)
        w.add("node_feat", nf)
        w.add("edge_index", ei)
        del nf, ei
        b = 512
        ids = [np.random.default_rng(1234 + r).integers(0, nsamp, size=b) for r in range(P)]
        s1, c1, s2, c2 = [ns_[i] for i in ids], [n[i] for i in ids], [es_[i] for i in ids], [e[i] for i in ids]
        o1 = [np.empty(int(c.sum()) * 64, np.uint8) for c in c1]
        o2 = [np.empty(int(c.sum()) * 16, np.uint8) for c in c2]
        nb = sum(int(c.sum()) * 64 for c in c1) + sum(int(c.sum()) * 16 for c in c2)
        out["cfg4_B4096"] = loop(w, [("node_feat", s1, c1, o1), ("edge_index", s2, c2, o2)], nb, b * P,
                                 f"{P} rank-threads x {b} samples x 2 get() per step (node_feat then edge_index) on a "
                                 f"{nsamp}-sample store")
        w.close()
    if "cfg5" in names or "cfg1" in names:
        sizes = list(CFG5_SIZES) if "cfg5" in names else []
        for R in sizes + ([512] if "cfg1" in names else []):
            rows_per = max(64, (32 << 20) // R)  # >= 32 MiB (or 64 rows) per rank-thread
            if R * rows_per * P > (8 << 30):  # bound the host memory (twice this: add() copies) and the set-up time
                rows_per = max(4, (8 << 30) // (R * P))
            shards = [co.synth_rows(SEED, r * rows_per, rows_per, R // 4, np.float32) for r in range(P)]
            w = World(P)
            w.add("s", shards)
            del shards
            b = max(2, min(4096, (16 << 20) // R))
            st = [np.random.default_rng(1234 + r).integers(0, rows_per * P, size=b) for r in range(P)]
            ct = [np.ones(b, np.int64) for _ in range(P)]
            outs = [np.empty(b * R, np.uint8) for _ in range(P)]
            key = f"cfg5_R{R}" if R != 512 else "cfg1_rows512_B4096"
            out[key] = loop(w, [("s", st, ct, outs)], P * b * R, P * b,
                            f"{P} rank-threads x {b} get() of {R} B per step, {rows_per} rows per rank")
            w.close()
    if "persample" in names:
        # the legacy loop itself (distdataset.py:79-92): one 4 KiB row + one 4 B label per sample, ONE rank-thread
        rows = 262144
        data = [co.synth_rows(SEED, 0, rows, DISP, np.float32)]
        lab = [co.synth_rows(SEED + 2, 0, rows, 1, np.int32)]
        w = World(1)
        w.add("d", data)
        w.add("l", lab)
        b = 65536
        st = [np.random.default_rng(1234).integers(0, rows, size=b)]
        ct = [np.ones(b, np.int64)]
        o1, o2 = [np.empty(b * ROW_BYTES, np.uint8)], [np.empty(b * 4, np.uint8)]
        out["per_sample_loop"] = loop(w, [("d", st, ct, o1), ("l", st, ct, o2)], b * (ROW_BYTES + 4), b,
                                      "1 rank-thread, C++ loop of 65536 x (get(data row 4 KiB) + get(label)) -- without the "
                                      "Python / torch.tensor overhead of distdataset.py:84-88")
        w.close()
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, args.warmup
    # keep the whole run within a few minutes whatever K is asked for
    gbs, info = cpu_reference_run(args.cpu_samples, args.cpu_batch, min(steps, 20), min(warmup, 3))
    cfgs = {}
    if not args.no_configs:
        try:
            cfgs = cpu_reference_configs(set(args.configs.split(",")), info["cores"])
        except Exception as e:  # noqa: BLE001
            cfgs = {"error": repr(e)}
    line = {"impl": "reference", "metric": METRIC, "value": gbs, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": info["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args.gpus, args.samples, args.batch),
            "cpu_baseline": {k: info[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "host_cpus": info["host_cpus"], "cpu_set": info["cpu_set"],
            "samples_per_s": info["samples_per_s"],
            "e2e": {"value": gbs, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "configs": [dict(name=k, **v) for k, v in cfgs.items()] if "error" not in cfgs else cfgs}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- our arm
class Ctx:
    """per-process bench context: device, communicator, timing helpers"""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from ddstore_b200 import SelfComm, TorchDistComm
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.N = args.gpus
        if self.world != self.N:
            raise SystemExit(f"--gpus {self.N} but WORLD_SIZE={self.world}: launch with torchrun --nproc-per-node {self.N}")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        bind_to_gpu_numa(self.local)
        if self.N > 1:
            dist.init_process_group("nccl", init_method="env://", device_id=self.dev)
            self.comm = TorchDistComm()
        else:
            self.comm = SelfComm()
        self.side = torch.cuda.Stream(device=self.dev)  # the launching stream: kernels AND the timing events live on it
        torch.cuda.set_stream(self.side)
        self.stream = self.side.cuda_stream
        self.peaks, self.peak_src = measured_peaks()

    def barrier(self):
        if self.N > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def allmax(self, vals):
        if self.N == 1:
            return list(vals)
        t = self.torch.tensor(list(vals), device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def allsum(self, vals):
        if self.N == 1:
            return list(vals)
        t = self.torch.tensor(list(vals), device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(x) for x in t]

    def share(self, total):
        per = total // self.N
        return per if self.rank < self.N - 1 else total - per * (self.N - 1)

    def timed_blocks(self, store, launch, K, W, R, active=True):
        """W warm-up launches, then R blocks of EXACTLY K launches, each block between two CUDA events on the launching
        stream with barrier + synchronize on both sides; per block the max over ranks. `launch(i)` enqueues step i.
        Ranks with active=False (mode B bystanders) launch nothing but take part in the barriers.
        -> list of R ms_per_step values"""
        torch = self.torch
        if active:
            for i in range(W):
                launch(i)
            store.wait()
        out = []
        for r in range(R):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            self.barrier()
            e0.record()
            if active:
                for i in range(K):
                    launch(W + r * K + i)
            e1.record()
            if active:
                store.wait()
            self.barrier()
            out.append(e0.elapsed_time(e1) / K)
        return self.allmax(out)

    def roofline(self, payload_bytes_per_gpu, ms, requesters=None):
        """HBM roofline at N=1 (2 x payload per launch); NVLink-in at N>1 (payload x (N-1)/N per launch)"""
        N = self.N
        if N == 1:
            alg, peak, bound, src = 2 * payload_bytes_per_gpu, float(self.peaks["hbm_gbs"]), "hbm", self.peak_src
        else:
            alg, peak, bound = payload_bytes_per_gpu * (N - 1) / N, NVLINK_PEAK, "nvlink"
            src = "guide constant (B200_PROFILING.md peer copy 770 GB/s per direction; not in MEASURED_PEAKS.json)"
        ach = alg / (ms * 1e-3) / 1e9
        return {"bound": bound, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "algorithmic_bytes_per_launch": alg, "peak_source": src}


def pct(vals):
    return [float(np.percentile(vals, q)) for q in (10, 50, 90)]


def verify_entry(ctx, store, name, packed, starts, counts, count, offsets, seed, expect_rows):
    """whole-batch on-device check of one packed result; -> (rows verified over all ranks, mismatches over all ranks,
    owners hit (min over ranks of the number of owners that served >= 1 request))"""
    bad, rows, owners = store.synth_verify(name, packed, starts, counts=counts, count=count, offsets=offsets, seed=seed,
                                           stream=ctx.stream)
    assert bad == 0 and rows == expect_rows, f"bench: batch of {name} differs from the generator ({bad} elements, {rows}/{expect_rows} rows)"
    tot = ctx.allsum([rows, bad])
    hit = -ctx.allmax([-sum(1 for o in owners if o > 0)])[0]
    return int(tot[0]), int(tot[1]), int(hit)


def run_configs(ctx, args, names, ref):
    """the other BASELINE.json configs -> list of entries for the `configs` array"""
    import torch
    from ddstore_b200 import PyDDStore
    N, rank, dev, st = ctx.N, ctx.rank, ctx.dev, ctx.stream
    K, W, R = max(5, min(args.steps, 20)), 3, max(3, min(args.repeats, 5))
    sc = args.config_scale
    rng = np.random.default_rng(1234 + rank)
    entries = []

    def entry(name, workload, ms_list, nbytes, nsamples, verified, extra=None, requesters=None):
        ms = float(np.median(ms_list))
        nreq_gpus = N if requesters is None else requesters
        e = {"name": name, "workload": workload, "value": nreq_gpus * nbytes / ms / 1e6, "unit": UNIT, "ms_per_step": ms,
             "ms_per_step_p10_p50_p90": pct(ms_list), "samples_per_s": nreq_gpus * nsamples / (ms * 1e-3),
             "bytes_per_step_per_gpu": int(nbytes), "steps": K, "repeats": len(ms_list),
             "roofline": ctx.roofline(nbytes, ms), "verified_rows": verified[0], "mismatches": verified[1],
             "owners_hit": verified[2]}
        if extra:
            e.update(extra)
        if ref and name in ref:
            e["reference"] = ref[name]
        entries.append(e)

    # ---- config 3: variable-length float32 samples, 100..10000 elements, disp = 1
    if "cfg3" in names:
        nsamp = max(N * 64, int(500_000 * sc) * N)
        sstart, L = cfg3_tables(nsamp)
        per = nsamp // N
        lo, hi = rank * per, ((rank + 1) * per if rank < N - 1 else nsamp)
        store = PyDDStore(ctx.comm, device=ctx.local)
        store.init("x", int(sstart[hi] - sstart[lo]), 1, 4)
        store.synth_fill("x", SEED)
        d_start, d_len = torch.from_numpy(sstart[:-1].copy()).to(dev), torch.from_numpy(L).to(dev)
        store.set_sample_index("x", d_start, d_len)
        for B in (4096, 16384):
            # FOUR different id sets, rotated step by step (a loader never asks for the same samples twice in a row)
            NS = 4
            ids = [torch.from_numpy(rng.integers(0, nsamp, size=B)).to(dev) for _ in range(NS)]
            s_ = [d_start[i].contiguous() for i in ids]
            c_ = [d_len[i].contiguous() for i in ids]
            rows = [int(c.sum().item()) for c in c_]
            nbytes = float(np.mean(rows)) * 4
            outs = [torch.empty(max(rows) * 4, dtype=torch.uint8, device=dev) for _ in range(2)]
            offs = [torch.empty(B + 1, dtype=torch.int64, device=dev) for _ in range(2)]
            wl = f"configs[2]: variable-length 100..10000 float32 samples, {nsamp} samples ({int(sstart[-1]) * 4 / 1e9:.1f} GB) over {N} GPU(s), B={B} per GPU"
            for mode, fn in (("", lambda i: store.get_batch("x", s_[i % NS], c_[i % NS], out=outs[i & 1], offsets=offs[i & 1], stream=st,
                                                           wait=False, overlap=True)),
                             ("_by_sample_id", lambda i: store.get_samples("x", ids[i % NS], outs[i & 1], offsets=offs[i & 1],
                                                                          stream=st, wait=False, overlap=True))):
                ms = ctx.timed_blocks(store, fn, K, W, R)
                li = W + R * K - 1  # the last step: which ids, which buffer
                ver = verify_entry(ctx, store, "x", outs[li & 1], s_[li % NS], c_[li % NS], 1, offs[li & 1], SEED, rows[li % NS])
                # the same queue with every launch waiting for the previous one (no DDS_OVERLAP)
                ser = ctx.timed_blocks(store, (lambda i, m=mode: store.get_batch("x", s_[i % NS], c_[i % NS], out=outs[0], offsets=offs[0], stream=st, wait=False)
                                               if not m else store.get_samples("x", ids[i % NS], outs[0], offsets=offs[0], stream=st, wait=False)),
                                       K, W, 3)
                entry(f"cfg3{mode}_B{B}", wl + (", explicit (start, count) arrays" if not mode else ", by sample id (device-resident index)"),
                      ms, nbytes, B, ver, {"serialized_ms_per_step": float(np.median(ser)), "queue": "DDS_OVERLAP double-buffered, 4 id sets rotated"})
        store.free()
        store.close()

    # ---- config 4: node_feat f32 [n,16] + edge_index i64 [8n,2], both arrays of a sample in ONE launch
    if "cfg4" in names:
        nsamp = max(N * 64, int(250_000 * sc) * N)
        ns_, n, es_, e = cfg4_tables(nsamp)
        per = nsamp // N
        lo, hi = rank * per, ((rank + 1) * per if rank < N - 1 else nsamp)
        store = PyDDStore(ctx.comm, device=ctx.local)
        store.init("node_feat", int(ns_[hi] - ns_[lo]), 16, 4)
        store.init("edge_index", int(es_[hi] - es_[lo]), 2, 8)
        store.synth_fill("node_feat", SEED)
        store.synth_fill("edge_index", SEED + 1)
        dns, dn = torch.from_numpy(ns_[:-1].copy()).to(dev), torch.from_numpy(n).to(dev)
        des, de = torch.from_numpy(es_[:-1].copy()).to(dev), torch.from_numpy(e).to(dev)
        store.set_sample_index("node_feat", dns, dn)
        store.set_sample_index("edge_index", des, de)
        B = 4096
        ids = torch.from_numpy(rng.integers(0, nsamp, size=B)).to(dev)
        s1, c1, s2, c2 = dns[ids].contiguous(), dn[ids].contiguous(), des[ids].contiguous(), de[ids].contiguous()
        r1, r2 = int(c1.sum().item()), int(c2.sum().item())
        b1, b2 = r1 * 64, r2 * 16
        o1 = [torch.empty(b1, dtype=torch.uint8, device=dev) for _ in range(2)]
        o2 = [torch.empty(b2, dtype=torch.uint8, device=dev) for _ in range(2)]
        f1 = [torch.empty(B + 1, dtype=torch.int64, device=dev) for _ in range(2)]
        f2 = [torch.empty(B + 1, dtype=torch.int64, device=dev) for _ in range(2)]
        names2 = ["node_feat", "edge_index"]
        ms = ctx.timed_blocks(store, lambda i: store.get_samples_multi(names2, ids, [o1[i & 1], o2[i & 1]], offsets=[f1[i & 1], f2[i & 1]],
                                                                        stream=st, wait=False, overlap=True), K, W, R)
        last = (W + R * K - 1) & 1
        v1 = verify_entry(ctx, store, "node_feat", o1[last], s1, c1, 1, f1[last], SEED, r1)
        v2 = verify_entry(ctx, store, "edge_index", o2[last], s2, c2, 1, f2[last], SEED + 1, r2)
        ser = ctx.timed_blocks(store, lambda i: store.get_samples_multi(names2, ids, [o1[0], o2[0]], offsets=[f1[0], f2[0]], stream=st,
                                                                         wait=False), K, W, 3)
        entry("cfg4_B4096", f"configs[3]: node_feat f32[n,16] + edge_index i64[8n,2] of the same {B} samples per GPU in ONE launch, "
                            f"{nsamp} samples over {N} GPU(s)", ms, b1 + b2, B,
              (v1[0] + v2[0], v1[1] + v2[1], min(v1[2], v2[2])),
              {"serialized_ms_per_step": float(np.median(ser)), "queue": "DDS_OVERLAP double-buffered"})
        store.free()
        store.close()

    # ---- config 5: size sweep (mode A: every rank fetches; mode B: one requester) and the config-1 row shape
    sweep = []
    if "cfg5" in names:
        sweep += [(R_, f"cfg5_R{R_}", max(1, (256 << 20) // R_)) for R_ in CFG5_SIZES]
    if "cfg1" in names:
        # (the last one = 16 loader batches of 4096 served by ONE launch: PrefetchLoader(group=16))
        sweep += [(512, "cfg1_rows512_B4096", 4096), (512, "cfg1_rows512_B4096_group16", 65536), (512, "cfg1_rows512_B262144", 262144)]
    for R_, key, B in sweep:
        shard = max(int((1 << 30) * sc), 64 * R_)
        rows = shard // R_
        store = PyDDStore(ctx.comm, device=ctx.local)
        store.init("s", rows, R_ // 4, 4)
        store.synth_fill("s", SEED)
        idx = torch.from_numpy(rng.integers(0, rows * N, size=B)).to(dev)
        outs = [torch.empty(B * R_, dtype=torch.uint8, device=dev) for _ in range(2)]
        fn = lambda i: store.get_batch("s", idx, out=outs[i & 1], count=1, stream=st, wait=False, overlap=True)  # noqa: E731
        ms = ctx.timed_blocks(store, fn, K, W, R)
        ver = verify_entry(ctx, store, "s", outs[(W + R * K - 1) & 1], idx, None, 1, None, SEED, B)
        cfgname = "configs[4]: fetch-bandwidth sweep" if key.startswith("cfg5") else "configs[0] row shape (64 float64 = 512 B)"
        entry(key, f"{cfgname}, rows of {R_} B, B={B} per GPU, {shard / 2**30:.2f} GiB shard per GPU, mode A (all ranks fetch)",
              ms, B * R_, B, ver, {"queue": "DDS_OVERLAP double-buffered"})
        if N > 1 and key in ("cfg5_R4096", "cfg5_R1048576"):
            msb = ctx.timed_blocks(store, fn, K, W, 3, active=(rank == 0))
            e = {"name": key + "_modeB", "workload": f"same store, mode B: rank 0 alone fetches (one origin), B={B}",
                 "value": B * R_ / float(np.median(msb)) / 1e6, "unit": UNIT, "ms_per_step": float(np.median(msb)),
                 "ms_per_step_p10_p50_p90": pct(msb), "samples_per_s": B / (float(np.median(msb)) * 1e-3),
                 "bytes_per_step_per_gpu": B * R_, "roofline": ctx.roofline(B * R_, float(np.median(msb)))}
            entries.append(e)
        store.free()
        store.close()

    # ---- N = 1 extras: legacy per-sample loop, streaming ingest, prefetch overlap
    if N == 1 and "persample" in names:
        entries.append(bench_per_sample(ctx, ref))
    if N == 1 and "ingest" in names:
        entries.append(bench_ingest(ctx, sc))
    if N == 1 and "prefetch" in names:
        entries.append(bench_prefetch(ctx, sc))
    return entries


def bench_per_sample(ctx, ref):
    """the reference's loader contract, unmodified: one get() per variable per sample (distdataset.py:79-92)"""
    import torch
    from ddstore_b200 import PyDDStore
    store = PyDDStore(ctx.comm, device=ctx.local)
    rows = 262144
    store.init("d", rows, DISP, 4)
    store.init("l", rows, 1, 4)
    store.synth_fill("d", SEED)
    store.synth_fill("l", SEED + 2)
    idx = np.random.default_rng(1234).integers(0, rows, size=4096)
    val, lab = np.zeros((1, DISP), np.float32), np.zeros((1, 1), np.int32)
    dval = torch.zeros((1, DISP), dtype=torch.float32, device=ctx.dev)

    def loop(n, host=True):
        t0 = time.perf_counter()
        for i in range(n):
            j = int(idx[i & 4095])
            store.get("d", val if host else dval, j)
            store.get("l", lab, j)
        return (time.perf_counter() - t0) / n

    loop(200)
    t_host = loop(3000)
    exp = np_synth_rows(SEED, int(idx[2999 & 4095]), 1, DISP, np.float32)
    assert val.tobytes() == exp.tobytes(), "per-sample loop: last row differs from the generator"
    loop(200, host=False)
    t_dev = loop(3000, host=False)
    # the raw C-ABI call without the Python wrapper's argument handling
    from ddstore_b200 import _capi
    L, h = _capi.lib(), store._h
    t0 = time.perf_counter()
    for i in range(3000):
        L.dds_get(h, b"d", int(idx[i & 4095]), 1, 4, val.ctypes.data, 0)
    t_c = (time.perf_counter() - t0) / 3000
    store.free()
    store.close()
    e = {"name": "per_sample_loop", "workload": "legacy loader contract: per sample get(data row 4 KiB -> pageable ndarray) + "
         "get(label), one after the other, through PyDDStore.get (1-CTA kernel, completion spun on in pinned memory)",
         "value": (ROW_BYTES + 4) / t_host / 1e9, "unit": UNIT, "samples_per_s": 1.0 / t_host,
         "us_per_sample_host_dst": t_host * 1e6, "us_per_sample_device_dst": t_dev * 1e6,
         "us_per_get_c_abi": t_c * 1e6, "n_gpus": 1}
    if ref and "per_sample_loop" in ref:
        e["reference"] = ref["per_sample_loop"]
    return e


def bench_ingest(ctx, sc):
    """(f3) streaming ingest: dataset.ingest_chunks (pinned double buffer, bounds-checked async updates) vs one plain
    pinned H2D copy of the same bytes"""
    import torch
    from ddstore_b200 import PyDDStore
    from ddstore_b200.dataset import ingest_chunks
    store = PyDDStore(ctx.comm, device=ctx.local)
    rows, chunk = int(262144 * max(sc, 0.05)), 16384  # 1 GiB of 4 KiB rows in 64 MiB chunks
    rows = (rows // chunk) * chunk or chunk
    store.init("ing", rows, DISP, 4)
    src = np.random.default_rng(3).integers(0, 2**32, size=(chunk, DISP), dtype=np.uint32).view(np.float32)
    chunks = lambda: (src for _ in range(rows // chunk))  # noqa: E731
    ingest_chunks(store, "ing", chunks())
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n = ingest_chunks(store, "ing", chunks())
    torch.cuda.synchronize()
    t_ing = time.perf_counter() - t0
    assert n == rows
    got = torch.empty((2, DISP), dtype=torch.float32, device=ctx.dev)
    store.get_batch("ing", [chunk - 1, rows - 1], out=got, count=1)
    assert got[0].cpu().numpy().tobytes() == src[-1].tobytes() and got[1].cpu().numpy().tobytes() == src[-1].tobytes()
    pin = torch.empty(rows * ROW_BYTES, dtype=torch.uint8).pin_memory()
    dst = torch.empty(rows * ROW_BYTES, dtype=torch.uint8, device=ctx.dev)
    dst.copy_(pin, non_blocking=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dst.copy_(pin, non_blocking=True)
    torch.cuda.synchronize()
    t_copy = time.perf_counter() - t0
    store.free()
    store.close()
    nb = rows * ROW_BYTES
    return {"name": "ingest", "workload": f"(f3) init + update in {chunk}-row chunks: {nb / 2**30:.2f} GiB from pageable host "
            f"arrays through the pinned double buffer (CPU staging copy + async H2D overlapped)",
            "value": nb / t_ing / 1e9, "unit": UNIT, "plain_pinned_h2d_GBps": nb / t_copy / 1e9,
            "frac_of_plain_h2d": t_copy / t_ing, "n_gpus": 1}


def bench_prefetch(ctx, sc):
    """(f4) does the double-buffered prefetch hide the fetch under a training step? A dummy 5 ms 'training kernel'
    per batch; compare (a) PrefetchLoader, (b) the reference's bracket: epoch_begin; blocking fetch; epoch_end; train
    (examples/vae/vae-ddp.py:240-265), (c) the training kernel alone. Two stand-ins: one CTA per SM that leaves the SMs'
    shared memory free, one that holds 200 KB of it per SM (nothing of the gather fits beside it), and the latter cut
    into 50 back-to-back kernels of 100 us (a step made of many layers: the fetch slips into the gaps between them)."""
    import torch
    from ddstore_b200 import _capi
    from ddstore_b200.dataset import DeviceBatchSampler, DistDataset, PrefetchLoader
    L = _capi.lib()
    nsamp, B, steps = int(200_000 * max(sc, 0.05)), 8192, 24
    data = np.random.default_rng(5).integers(0, 2**32, size=(nsamp, DISP), dtype=np.uint32).view(np.float32)

    class _DS:
        def __len__(self):
            return nsamp

        def __getitem__(self, i):
            return data[i], int(i & 7)

    ds = DistDataset(_DS(), "pf", comm=ctx.comm, device=ctx.local)
    cur = torch.cuda.current_stream(ctx.dev)
    train_ns = 5_000_000
    out = {}
    cpu_side = [0.0]
    for tag, smem, pieces in (("smem_free", 0, 1), ("smem_64k", 64 * 1024, 1), ("smem_200k", 200 * 1024, 1),
                              ("smem_200k_50_kernels", 200 * 1024, 50)):
        def train():  # one 5 ms kernel, or the same 5 ms as `pieces` back-to-back kernels (a step of many layers)
            for _ in range(pieces):
                _capi.raise_for(L.dds_test_occupy(ctx.local, 148, smem, train_ns // pieces, ctypes.c_void_p(cur.cuda_stream)))

        def run_prefetch():
            sampler = DeviceBatchSampler(nsamp, B, 0, 1, seed=0, drop_last=True, device=ctx.dev)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            k = 0
            for vals, labs in PrefetchLoader(ds, sampler, B, drop_last=True):
                train()
                k += 1
                if k == steps:
                    break
            cpu_side[0] = (time.perf_counter() - t0) / k  # how long the host needed to QUEUE a step
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) / k

        def run_bracket():
            sampler = DeviceBatchSampler(nsamp, B, 0, 1, seed=0, drop_last=True, device=ctx.dev)
            vals = torch.empty((B, DISP), dtype=torch.float32, device=ctx.dev)
            labs = torch.empty((B, 1), dtype=torch.int32, device=ctx.dev)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            k = 0
            for ids in sampler:
                ds.epoch_begin()
                ds.ddstore.get_batch("pfdata", ids, out=vals, count=1)
                ds.ddstore.get_batch("pflabels", ids, out=labs, count=1)
                ds.epoch_end()
                train()
                k += 1
                if k == steps:
                    break
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) / k

        def run_train_only():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                train()
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) / steps

        run_prefetch()
        t_only, t_br = run_train_only(), run_bracket()
        t_pf = min(run_prefetch(), run_prefetch())
        fetch = max(t_br - t_only, 1e-9)
        out[tag] = {"ms_train_only": t_only * 1e3, "ms_step_bracketed_fetch": t_br * 1e3, "ms_step_prefetch": t_pf * 1e3,
                    "fetch_ms_exposed_bracketed": (t_br - t_only) * 1e3, "fetch_ms_exposed_prefetch": (t_pf - t_only) * 1e3,
                    "hidden_fraction": 1.0 - max(t_pf - t_only, 0.0) / fetch, "host_ms_to_queue_a_prefetch_step": cpu_side[0] * 1e3}
    ds.free()
    ds.ddstore.close()
    e = {"name": "prefetch_overlap", "workload": f"(f4) {steps} steps of a {train_ns / 1e6:.0f} ms dummy training kernel on batches of "
         f"{B} x 4 KiB rows + labels: PrefetchLoader (fetch of batch k+1 on a side stream) vs the reference's "
         "epoch_begin / blocking fetch / epoch_end bracket; training stand-in without / with 200 KB of shared memory per SM",
         "value": B * (ROW_BYTES + 4) / (out["smem_free"]["ms_step_prefetch"] * 1e-3) / 1e9, "unit": UNIT, "n_gpus": 1}
    e.update({f"{k}_{tag}": v for tag, d in out.items() for k, v in d.items()})
    # (the gather needs an SM's whole shared memory: it overlaps with training on the SMs the training kernel leaves free --
    # the 64 KB stand-in is packed three CTAs per SM and leaves two thirds of them -- and otherwise runs in the gaps)
    e["hidden_fraction"] = out["smem_64k"]["hidden_fraction"]
    return e


DUMP_ROWS = 4096  # rows dumped over all ranks together: 4096 rows x 1024 words x 8 B = 32 MiB as float64


def sample_batch(packed, B, N):
    """DUMP_ROWS // N of the B packed rows one rank received, at positions drawn from a fixed seed, copied to the host
    as uint32 [rows, DISP]"""
    import torch
    sel = np.sort(np.random.default_rng(SEED).choice(B, size=min(B, max(1, DUMP_ROWS // N)), replace=False))
    return packed.view(torch.int32).view(B, DISP)[torch.from_numpy(sel).to(packed.device)].cpu().numpy().view(np.uint32)


def dump_batch(dirname, rank, rows):
    """DIR/batch_rows_rank<r>.npy: float64 [rows, DISP], each row's 32-bit words as unsigned integers. The payload is raw
    bit patterns (NaN, Inf among them as float32); every uint32 is exact and finite in float64, so the file carries the
    bytes bit for bit"""
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, f"batch_rows_rank{rank}.npy"), rows.astype(np.float64))


def run_ours(args):
    import torch
    from ddstore_b200 import PyDDStore, _capi

    ctx = Ctx(args)
    N, rank, local, dev, stream = ctx.N, ctx.rank, ctx.local, ctx.dev, ctx.stream
    K, W, B = args.steps, max(args.warmup, 3), args.batch
    total = args.samples
    nrows = ctx.share(total)

    store = PyDDStore(ctx.comm, device=local)
    store.init("x", nrows, DISP, 4)
    store.synth_fill("x", SEED)
    lenlist = store.query("x")["lenlist"]
    assert lenlist[-1] == total

    rng = np.random.default_rng(1234 + rank)
    nsets = min(K + W, 16)
    idx_host = [torch.from_numpy(rng.integers(0, total, size=B)).pin_memory() for _ in range(nsets)]
    idx_dev = [t.to(dev) for t in idx_host]
    out_dev = torch.empty(B * ROW_BYTES, dtype=torch.uint8, device=dev)
    step_bytes = B * ROW_BYTES
    torch.cuda.synchronize()

    # ---- value: device-resident indices and output, K back-to-back async launches per block. The batches are
    # independent (static device-resident index sets, two alternating output buffers -- a double-buffered prefetch
    # queue), so they are queued with overlap=True: the head of batch k+1 fills the SMs the tail of batch k vacates,
    # under the kernel-enforced contract (batch k+2 writes nothing before batch k has retired).
    out_dev2 = torch.empty_like(out_dev)
    outs = (out_dev, out_dev2)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    launches0 = _capi.lib().dds_kernel_launches()
    ms_step = ctx.timed_blocks(store, lambda i: store.get_batch("x", idx_dev[i % nsets], out=outs[i & 1], count=1, stream=stream,
                                                                wait=False, overlap=True), K, W, 1)[0]
    launches = (_capi.lib().dds_kernel_launches() - launches0) * K // (W + K)  # kernels per K-step block
    clocks = sampler.stop() if rank == 0 else None
    # every row of the last two timed batches of every rank, regenerated and compared on the device
    last = W + K - 1
    ver = [verify_entry(ctx, store, "x", outs[i & 1], idx_dev[i % nsets], None, 1, None, SEED, B) for i in (last - 1, last)]
    dumped = sample_batch(outs[last & 1], B, N) if args.dump_outputs else None  # (the buffer is reused below)
    owners_hit = min(v[2] for v in ver)
    if B >= 64 * N:
        assert owners_hit == N, f"bench: only {owners_hit} of {N} owners served requests"
    value = N * step_bytes / (ms_step * 1e-3) / 1e9

    # second pass, K steps, one CUDA-event pair around every launch: the kernel's own duration serialised
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for i in range(K):
        ev[i][0].record()
        store.get_batch("x", idx_dev[(W + i) % nsets], out=out_dev, count=1, stream=stream, wait=False)
        ev[i][1].record()
    store.wait()
    ctx.barrier()
    pair_list = [a.elapsed_time(b) for a, b in ev]
    pair_ms = ctx.allmax([float(np.mean(pair_list))])[0]
    pair_pcts = pct(pair_list)
    # and the same queue without DDS_OVERLAP (every launch waits for the previous one)
    ser_blocks = ctx.timed_blocks(store, lambda i: store.get_batch("x", idx_dev[i % nsets], out=out_dev, count=1, stream=stream,
                                                                   wait=False), K, 1, 3)

    # ---- N > 1: the same steps as a COLLECTIVE owner-push fetch (every rank fetches in every step anyway): posted NVLink
    # writes instead of pull reads. Same rows, same packed layout, in the rank's window of the store.
    push = None
    if N > 1 and args.push:
        store.push_setup(B, step_bytes)
        last_view = [None, None]

        def push_step(i):
            last_view[i & 1] = store.get_batch_push("x", idx_dev[i % nsets], count=1, stream=stream)

        ms_p = ctx.timed_blocks(store, push_step, K, W, 1)[0]
        # (the window's buffers alternate with the store's own step counter; verify what the last two steps returned)
        lastp = W + K - 1
        pver = [verify_entry(ctx, store, "x", last_view[i & 1], idx_dev[i % nsets], None, 1, None, SEED, B) for i in (lastp - 1, lastp)]
        dumped_push = sample_batch(last_view[lastp & 1], B, N) if args.dump_outputs else None
        push = {"value": N * step_bytes / (ms_p * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": ms_p,
                "roofline": ctx.roofline(step_bytes, ms_p),
                "verified_rows": sum(v[0] for v in pver), "mismatches": sum(v[1] for v in pver),
                "path": "dds_get_batch_push: every rank publishes its start rows, every owner TMA-stores the rows it owns into "
                        "the requesters' peer-mapped windows, arrival signalled with system-scope words; one launch per rank "
                        "per step, no NCCL"}

    # ---- e2e: pinned host indices in, host buffer out, through the same call
    e2e = None
    if not args.no_e2e:
        out_host = torch.empty(B * ROW_BYTES, dtype=torch.uint8).pin_memory()
        out_np = out_host.numpy()
        idx_np = [t.numpy() for t in idx_host]
        Ke = max(3, min(K, 10))

        def e2e_loop(buf):
            for i in range(2):
                store.get_batch("x", idx_np[i % nsets], out=buf, count=1)
            ctx.barrier()
            t0 = time.perf_counter()
            for i in range(Ke):
                store.get_batch("x", idx_np[(W + i) % nsets], out=buf, count=1)
            torch.cuda.synchronize()
            t_e = time.perf_counter() - t0
            exp = np_synth_rows(SEED, int(idx_np[(W + Ke - 1) % nsets][B - 1]), 1, DISP, np.float32)
            assert buf[-ROW_BYTES:].tobytes() == exp.tobytes(), "bench e2e: last row differs from the generator"
            return ctx.allmax([t_e])[0]

        t_pin = e2e_loop(out_np)
        pageable = np.zeros(B * ROW_BYTES, np.uint8)  # the reference's destination contract (distdataset.py:80-85)
        t_page = e2e_loop(pageable)
        # the PCIe ceiling of THIS box under the same concurrency: a plain pinned D2H copy of the packed batch
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(Ke):
            out_host.copy_(out_dev, non_blocking=True)
        torch.cuda.synchronize()
        t_raw = ctx.allmax([time.perf_counter() - t0])[0]
        e2e = {"value": N * Ke * step_bytes / t_pin / 1e9, "unit": UNIT, "h2d_bytes_per_step": B * 8,
               "d2h_bytes_per_step": step_bytes, "steps": Ke, "ms_per_step": 1e3 * t_pin / Ke,
               "pageable_dst_value": N * Ke * step_bytes / t_page / 1e9,
               "plain_pinned_d2h_copy_value": N * Ke * step_bytes / t_raw / 1e9,
               "path": "dds_get_batch(host int64 starts -> host buffer): H2D idx + gather kernel + D2H payload; `value` = "
                       "pinned destination, `pageable_dst_value` = np.zeros destination, `plain_pinned_d2h_copy_value` = "
                       "cudaMemcpy of the same bytes on all ranks at once (what the PCIe links of this box deliver)"}

    # ---- roofline of the dominant kernel
    geom = [ctypes.c_int() for _ in range(5)]
    _capi.lib().dds_gather_geometry(*[ctypes.byref(g) for g in geom])
    roofline = ctx.roofline(step_bytes, ms_step)
    traffic = None
    tp = os.path.join(ROOT, "profiles", "gather_fixed_traffic.json" if N == 1 else "r2_nvlink_traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        if N == 1:
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
        else:
            # NVLink bytes INTO this GPU per launch: measured at N=2 with ncu on rank 0 (payload x 1.125 response bytes +
            # the peers' read requests, 0.1875 per payload byte served), scaled to this N's remote fraction
            r = tj.get("per_payload_byte", {"response_header": 0.125, "read_request_packet": 0.1875})
            traffic = step_bytes * (N - 1) / N * (1.0 + r["response_header"] + r["read_request_packet"])
    roofline.update({"traffic": traffic, "kernel": "dds_gather_kernel<FIXED,12,4,4096>", "per_launch_ms": ms_step,
                     "per_launch_event_pair_ms": pair_ms, "per_launch_event_pair_ms_p10_p50_p90": pair_pcts,
                     "note": "per_launch_ms = median K-step block / K with the launches overlapping head-to-tail (DDS_OVERLAP); "
                             "per_launch_event_pair_ms = the same kernel serialised, one CUDA-event pair per launch"})

    # ---- the other configs, and the reference beside them at N = 1
    ref_cfg, cpu = {}, None
    names = set() if args.no_configs else set(args.configs.split(","))
    if rank == 0 and N == 1 and not args.no_cpu_baseline:
        try:
            _, info = cpu_reference_run(args.cpu_samples, args.cpu_batch, 8, 2)
            cpu = {k: info[k] for k in ("value", "unit", "cores", "kind", "sample", "host_cpus", "cpu_set")}
            cpu["samples_per_s"] = info["samples_per_s"]
            if names:
                ref_cfg = cpu_reference_configs(names, info["cores"])
        except Exception as e:  # noqa: BLE001
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {e!r}"}
        if hasattr(os, "sched_setaffinity"):
            bind_to_gpu_numa(local)
    store.free()
    store.close()
    configs = run_configs(ctx, args, names, ref_cfg) if names else []

    fetch_mode = "one-sided pull (dds_get_batch)"
    pull = None
    if push and push["value"] > value:
        # the headline is the faster of the two ways a DDP loader can fetch its batch; the other one is kept beside it
        pull = {"value": value, "ms_per_step": ms_step, "roofline": dict(roofline)}
        value, ms_step, dumped = push["value"], push["ms_per_step"], dumped_push
        roofline.update(push["roofline"])
        roofline["per_launch_ms"] = ms_step
        fetch_mode = "collective owner-push (dds_get_batch_push)"
    if args.dump_outputs:  # the rows of the last timed step of the path the headline reports
        dump_batch(args.dump_outputs, rank, dumped)
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": N, "steps": K, "warmup": W,
                "ms_per_step": ms_step,
                "fetch_mode": fetch_mode, "pull": pull, "push": push,
                "serialized_ms_per_step": float(np.median(ser_blocks)),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic",
                "config": workload_config(N, total, B),
                "method": {"queue": "K independent batches in one timed block queued asynchronously on one stream with DDS_OVERLAP "
                                    "into two alternating output buffers (double-buffered prefetch; the kernel enforces that "
                                    "batch k+2 writes nothing before batch k retired)",
                           "mapping": "VMM peer mappings (fd passing), no NCCL in the data path",
                           "gather_geometry": {"ctas": geom[0].value, "warps_per_cta": geom[1].value,
                                               "stages": geom[2].value, "chunk_bytes": geom[3].value,
                                               "smem_bytes": geom[4].value}},
                "samples_per_s": N * B / (ms_step * 1e-3), "clocks": clocks, "e2e": e2e,
                "verified_rows": sum(v[0] for v in ver), "verified_batches": 2, "mismatches": sum(v[1] for v in ver),
                "owners_hit": owners_hit,
                "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "configs": configs}
        print(json.dumps(line), flush=True)
    ctx.barrier()
    if N > 1:
        ctx.dist.destroy_process_group()


def main():
    args = parse()
    if not os.path.exists(os.path.join(ROOT, "ddstore_b200", "libddstore_b200.so")):
        import __graft_entry__  # fresh checkout: build the native pieces in-tree first
        __graft_entry__.build()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
