#!/usr/bin/env python
"""bench.py — rate-limit decisions/s of the B200 evaluation path on BASELINE.json's headline workloads.

  python bench.py --gpus 1 --steps K --warmup W            # this repo's CUDA path (default)
  python bench.py --impl reference --steps K --warmup W    # the reference's CPU worker-pool path (oracle port) on the host cores
  torchrun --nproc-per-node N bench.py --gpus N ...        # N GPUs: key space sharded by the replicated-hash ring
  python bench.py --workload global ...                    # BASELINE config 5: GLOBAL hot keys + sync ticks (any N)
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's responses as DIR/<field>.npy

A "step" is one 65 536-request batch per GPU through the whole hot path (group -> probe -> bucket update -> response):
ONE launch of the persistent batch kernel k_batch.  Workload at N = 1: BASELINE config 3 — 100 M resident keys, Zipf s = 1.1,
TOKEN/LEAKY 50/50 by key.  At N > 1: config 4 — the same key space sharded over the N GPUs by the 512-replica FNV-1 ring; the
routing kernel stores every request into its owner's NVLink mailbox, the owner's batch kernel evaluates out of the mailboxes
and stores the responses back (weak scaling: 65 536 requests ingested per GPU per step).

Prints ONE JSON line (rank 0).
  value     decisions/s with the request batches already resident in HBM (a pool of pre-generated batches larger than L2 is
            cycled; the 12.8 GB table is far larger than L2).
  e2e       the same from KEY STRINGS in pinned host memory through the public host API (gub_submit_keys_async): H2D of key
            bytes + 16-byte request records, hashing (XXH64 + FNV-1) on the device, evaluation, D2H of the responses, all inside
            the timed region; every batch of the pool cycles through the pinned ring.
  roofline  k_batch: algorithmic bytes per launch (SURVEY 8d: 224 B x decisions) / its CUDA-event time, vs MEASURED_PEAKS.json;
            traffic = DRAM bytes per launch measured by ncu in this very run (a sub-process on the same workload).
  cpu_baseline / --impl reference: the oracle's worker-pool port on this host's cores, from key strings too.
"""
import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

BATCH = 65536
T0 = 1_700_000_000_000
ALGO_BYTES_PER_DECISION = 224  # SURVEY.md §8d: 64 slot read + 64 slot write-back + 64 request + 32 response


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="zipf", choices=["zipf", "global"],
                    help="zipf: BASELINE config 3 (N = 1) / 4 (N > 1); global: config 5 (10 M keys, 1 %% GLOBAL hot keys, sync tick every 500 ms)")
    ap.add_argument("--keys", type=int, default=int(os.environ.get("GUB_BENCH_KEYS", 0)), help="resident keys (default: 100 M, config 5: 10 M)")
    ap.add_argument("--zipf", type=float, default=1.1)
    ap.add_argument("--pool", type=int, default=32, help="distinct pre-generated batches cycled through (32 x 6 MiB > L2)")
    ap.add_argument("--cpu-keys", type=int, default=int(os.environ.get("GUB_BENCH_CPU_KEYS", 0)),
                    help="resident keys of the CPU arm (default: as many of --keys as host memory allows)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-traffic", action="store_true", help="skip the ncu sub-process that measures k_batch's DRAM bytes")
    ap.add_argument("--variants", action="store_true", help="also time the heterogeneous-hits and refill variants of the workload (informational)")
    ap.add_argument("--tick-ms", type=float, default=500.0, help="config 5: wall-clock period of the GLOBAL sync tick")
    ap.add_argument("--no-route-overlap", action="store_true", help="N > 1: routing and evaluation on one stream")
    ap.add_argument("--traffic-probe", action="store_true", help=argparse.SUPPRESS)  # the ncu sub-process runs this
    ap.add_argument("--ncu-window", type=int, default=0,
                    help="profile this many extra steps between cudaProfilerStart/Stop (run under `ncu --profile-from-start off`)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the responses of the last timed step as DIR/<field>.npy (float64; with N > 1 "
                         "every rank writes DIR/<field>_rank<r>.npy).  The inputs depend on the arguments alone; with --workload global "
                         "the tick period is calibrated from wall-clock time, so the table state there depends on it too")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if not a.keys:
        a.keys = 10_000_000 if a.workload == "global" else 100_000_000
    return a


# ---- helpers ---------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.rows, self.proc, self.dev = [], None, device_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.dev}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        if not self.rows:  # the timed region was shorter than one sampling period: take one reading now
            try:
                self.rows = subprocess.run(["nvidia-smi", f"--id={self.dev}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                           capture_output=True, text=True, timeout=10).stdout.strip().splitlines()
            except Exception:
                pass
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def zipf_rank_ids(rng, n, n_keys, s, hot):
    """Zipf(s) ranks -> ids with the `hot` top ranks mapped to ids 0..hot-1 in rank order (config 5: the GLOBAL hot set is 'drawn
    first in Zipf rank') and the others spread over [hot, n_keys) by the fixed multiplicative permutation."""
    from workloads import spread_ranks, zipf_ranks
    rank = zipf_ranks(rng, n, n_keys, s)
    out = rank.copy()
    cold = rank >= hot
    out[cold] = hot + spread_ranks(rank[cold] - hot, n_keys - hot)
    return out


def gen_batch(rng, n, n_keys, created_at, zipf_s, dtype, global_hot=0, hits_mix=0.0, duration=60000):
    """One ingest batch of the synthetic workload (SURVEY 8d).  global_hot: ids < global_hot carry Behavior_GLOBAL (config 5).
    hits_mix: fraction of requests with hits = 2 (the heterogeneous-hits variant); duration: the refill variant shortens it."""
    from workloads import bench_requests, zipf_ids
    import oracle_py as O
    ids = zipf_rank_ids(rng, n, n_keys, zipf_s, global_hot) if global_hot else zipf_ids(rng, n, n_keys, zipf_s)
    reqs = bench_requests(ids, created_at, mixed=True, dtype=dtype)
    if duration != 60000:
        reqs["duration"] = duration
    if hits_mix > 0:
        reqs["hits"] = np.where(rng.random(n) < hits_mix, 2, 1)
    if global_hot:
        reqs["behavior"] = np.where(ids < global_hot, O.GLOBAL | O.REQ_IS_OWNER, O.REQ_IS_OWNER).astype(np.uint32)
    return reqs, ids


def dump_outputs(out_dir, resp, suffix=""):
    """The response records of one step as one float64 array per field (every value is an integer below 2^53: exact)."""
    os.makedirs(out_dir, exist_ok=True)
    for f in resp.dtype.names:
        np.save(os.path.join(out_dir, f"{f}{suffix}.npy"), resp[f].astype(np.float64))


def batch_stats(ids):
    _, counts = np.unique(ids, return_counts=True)
    return dict(distinct=int(len(counts)), singles=int((counts == 1).sum()), repeated_keys=int((counts > 1).sum()),
                repeated_requests=int(counts[counts > 1].sum()), top=int(counts.max()))


def key_blob(ids):
    """(uint8 key bytes, uint64 offsets) of "bench_k%09d" for the ids: what a front end holds before hashing."""
    from workloads import bench_key_bytes
    b = bench_key_bytes(ids)
    offs = (np.arange(len(ids) + 1, dtype=np.uint64) * np.uint64(16))
    return np.ascontiguousarray(b).reshape(-1), offs


# ---- reference arm: the reference's CPU path (oracle port; the Go reference cannot be built in this image) ----------
def cpu_keys_that_fit(want):
    """The oracle keeps ~250 B per key (LRU node + hash map + item); leave half of the host memory alone."""
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 32 << 30
    return int(max(1_000_000, min(want, (avail // 2) // 250)))


def cpu_leg(n_keys, zipf_s, seconds, seed, steps=None, warmup=0, step_size=BATCH, from_keys=True):
    """The oracle's worker-pool port (W = cores shard threads) over the same synthetic traffic.  from_keys: every step starts
    from the key strings (XXH64 + FNV-1 inside the timed call), like the reference's own path (client.go:39, workers.go:153)."""
    import oracle_py as O
    from workloads import bench_requests
    cores = os.cpu_count() or 1
    pool = O.Pool(workers=cores, cache_size=max(4 * n_keys, 1 << 20), now_ms=T0)
    rng = np.random.default_rng(seed)
    t_fill = time.perf_counter()
    chunk = 1 << 20
    for lo in range(0, n_keys, chunk):  # warm pass: make every key resident (BASELINE.md), through the same worker-pool path
        ids = np.arange(lo, min(n_keys, lo + chunk), dtype=np.int64)
        pool.submit_hashed(bench_requests(ids, T0), threads=cores)
    t_fill = time.perf_counter() - t_fill
    batches = []
    for b in range(16):
        reqs, ids = gen_batch(rng, step_size, n_keys, T0 + 1 + b, zipf_s, O.HREQ_DTYPE)
        blob, offs = key_blob(ids)
        batches.append((reqs, blob, offs))

    last = [None]

    def one(b):
        reqs, blob, offs = batches[b % len(batches)]
        pool.set_now(T0 + 1 + b)
        if from_keys:
            last[0] = pool.submit_keys(blob, offs, reqs, threads=cores)
        else:
            last[0] = pool.submit_hashed(reqs, threads=cores)
        return pool.last_mt_seconds
    for w in range(max(warmup, 1)):
        one(w)
    done, t_used, b = 0, 0.0, 0
    while True:
        if steps is None:
            if t_used >= seconds:
                break
        elif b >= steps:
            break
        t_used += one(b)
        done += step_size
        b += 1
    return dict(value=done / t_used, seconds=t_used, steps=b, cores=cores, fill_seconds=t_fill, keys=n_keys, step_size=step_size,
                last_responses=last[0])


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    keys = args.cpu_keys or cpu_keys_that_fit(args.keys)
    # exactly --steps timed steps; beyond 20 000 steps the batch is shrunk so that the whole run stays within about a minute
    step_size = BATCH if args.steps <= 20000 else max(2048, int(BATCH * 20000 / args.steps) // 256 * 256)
    r = cpu_leg(keys, args.zipf, args.cpu_seconds, 0xB200 + 3, steps=args.steps, warmup=min(args.warmup, 20), step_size=step_size)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r["last_responses"])
    sample = (f"{r['steps']} x {step_size}-request Zipf({args.zipf}) batches over {r['keys']:,} resident keys"
              + ("" if r["keys"] == args.keys else f" (the GPU arm holds {args.keys:,}: host memory bounds the CPU table)")
              + f", TOKEN/LEAKY 50/50, from key strings (XXH64 + FNV-1 inside the timed call), {r['cores']} worker threads, {r['seconds']:.1f} s timed")
    line = {
        "impl": "reference", "metric": "rate-limit decisions/sec", "value": r["value"], "unit": "decisions/s", "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": args.warmup, "ms_per_step": 1e3 * r["seconds"] / max(r["steps"], 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int64+f64", "data": "synthetic",
        "config": {"workload": f"BASELINE config 3 shape on CPU: {sample}", "batch": step_size, "keys": r["keys"], "gpu_arm_keys": args.keys, "zipf_s": args.zipf},
        "cpu_baseline": {"value": r["value"], "unit": "decisions/s", "cores": r["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": r["value"], "unit": "decisions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def parse_traffic_csv(path):
    """{kernel: DRAM read / write bytes per launch} from an `ncu --csv --metrics dram__bytes_read.sum,dram__bytes_write.sum` log."""
    import csv
    with open(path) as f:
        rows = [r for r in csv.reader(f) if len(r) > 5]
    hdr = next((r for r in rows if "Metric Name" in r), None)
    if hdr is None:
        return {"error": "ncu produced no metric rows"}
    ik, im, iv, iu = hdr.index("Kernel Name"), hdr.index("Metric Name"), hdr.index("Metric Value"), hdr.index("Metric Unit")
    per = {}
    for r in rows:
        if r is hdr or len(r) <= max(ik, im, iv, iu) or r[im] not in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            continue
        m = re.search(r"k_(group|rank|eval|finish|batch)", r[ik])  # "void gub::k_rank<0>(gub::BatchArgs)" -> k_rank
        name = m.group(0) if m else r[ik].split("(")[0].split("::")[-1]
        v = float(r[iv].replace(",", "")) * {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(r[iu], 1.0)
        e = per.setdefault(name, {"read": 0.0, "write": 0.0, "launches": 0})
        if r[im] == "dram__bytes_read.sum":
            e["read"] += v; e["launches"] += 1
        else:
            e["write"] += v
    if not per:
        return {"error": "ncu reported no batch kernel launch"}
    return {k: {"dram_read_bytes_per_launch": e["read"] / e["launches"], "dram_write_bytes_per_launch": e["write"] / e["launches"], "launches": e["launches"]}
            for k, e in per.items()}


# ---- DRAM traffic of k_batch, measured by ncu on this very workload (a sub-process of the default run) ------------------
def measure_traffic(args):
    """{kernel: DRAM bytes per launch} for the batch kernels of this workload, by running this script's --traffic-probe under ncu."""
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu) or os.environ.get("GUB_BENCH_NO_NCU"):
        return None
    with tempfile.TemporaryDirectory() as d:
        log = os.path.join(d, "traffic.csv")
        cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "--cache-control", "none",
               "--profile-from-start", "off", "-k", "regex:k_(group|rank|eval|finish|batch)", "--csv", "--log-file", log,
               sys.executable, os.path.abspath(__file__), "--traffic-probe", "--keys", str(args.keys), "--zipf", str(args.zipf), "--pool", str(args.pool)]
        try:
            res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=300, check=False, text=True)
            out = parse_traffic_csv(log)
            if "error" in out:
                out["error"] += ": " + (res.stdout or "")[-300:]
                return out
            out["how"] = "ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum --cache-control none over warm steps of this workload (a sub-process of this run)"
            return out
        except Exception as ex:
            return {"error": repr(ex)}


# ---- this repo's arm --------------------------------------------------------------------------------------------
def run_b200(args):
    # A stalled collective run must end by itself: after GUB_BENCH_WATCHDOG seconds (default 20 minutes when several ranks run, off on one
    # GPU) every thread's Python stack goes to stderr and the process exits.
    wd = os.environ.get("GUB_BENCH_WATCHDOG") or ("1200" if int(os.environ.get("WORLD_SIZE", "1")) > 1 else "")
    if wd and float(wd) > 0:
        import faulthandler
        faulthandler.dump_traceback_later(float(wd), exit=True)
    import torch
    import gubernator_b200 as g
    import oracle_py as O
    from workloads import bench_requests

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    N = world
    t_start = time.perf_counter()

    def progress(what):  # stderr, every rank: where a multi-GPU run is when something stalls
        if os.environ.get("GUB_BENCH_PROGRESS"):
            sys.stderr.write(f"[bench rank {rank} +{time.perf_counter() - t_start:7.1f}s] {what}\n")
            sys.stderr.flush()
    n_keys = args.keys
    is_global = args.workload == "global"
    global_hot = n_keys // 100 if is_global else 0  # config 5: 1 % of the keys carry Behavior_GLOBAL, the top of the Zipf ranking
    seed = 0xB200 + (5 if is_global else (3 if N == 1 else 4))
    rng = np.random.default_rng(seed + 1000 * rank)

    # table sized at load factor <= 0.5 for this shard's share of the key space (+25 % for ring imbalance; GLOBAL keys are replicated everywhere)
    shard_keys = n_keys if N == 1 else int(n_keys / N * 1.25) + global_hot
    capacity = max(2 * shard_keys, 1 << 16)
    tab = g.Table(capacity, device=local)
    stream = torch.cuda.current_stream().cuda_stream

    # ---- the ring of GPUs (N > 1, or the GLOBAL workload at any N): fused routing over NVLink mailboxes
    p2p = None
    if N > 1 or is_global:
        from gubernator_b200.sharded import shard_addresses
        ring = g.Ring(0, 512)
        for a in shard_addresses(N):
            ring.add(a)
        p2p = g.native.P2P(tab, ring, rank, BATCH)
        if N > 1:
            handles = [None] * N
            dist.all_gather_object(handles, p2p.export())
            p2p.connect(handles)
        else:
            p2p.connect_local([p2p])
        if is_global:
            p2p.enable_global(1 << 18)
            if N > 1:
                uid = [g.native.nccl_unique_id() if rank == 0 else None]
                dist.broadcast_object_list(uid, src=0)
                p2p.nccl_init(uid[0])
        if dist is not None:
            dist.barrier()

    ingest = None
    if p2p is not None and N > 1 and not args.no_route_overlap:
        ingest = torch.cuda.Stream(device=dev)  # the routing kernel runs on its own stream: step e+1 is routed while step e is evaluated

    def ring_step(d_reqs, n, clk, d_out):
        p2p.step(d_reqs.data_ptr(), n, clk, d_out.data_ptr(), stream, ingest.cuda_stream if ingest is not None else None)

    # ---- warm pass: make every key resident through the real path
    t_fill = time.perf_counter()
    clk0 = g.clock_fill(T0)
    chunk = BATCH if p2p is not None else 1 << 20
    d_chunk = torch.empty((chunk, 64), dtype=torch.uint8, device=dev)
    d_chunk_out = torch.empty((chunk, 32), dtype=torch.uint8, device=dev)
    my_lo = (n_keys * rank) // N
    my_hi = (n_keys * (rank + 1)) // N
    n_fill_steps = (n_keys // N + chunk - 1) // chunk  # identical on every rank (collective steps)
    for s in range(n_fill_steps):
        lo = my_lo + s * chunk
        hi = min(my_hi, lo + chunk)
        ids = np.arange(lo, max(hi, lo), dtype=np.int64)
        reqs = bench_requests(ids, T0, dtype=g.REQ_DTYPE)
        if global_hot:
            reqs["behavior"] = np.where(ids < global_hot, O.GLOBAL | O.REQ_IS_OWNER, O.REQ_IS_OWNER).astype(np.uint32)
        n = len(reqs)
        if n:
            # (the routing kernel reads d_chunk on the ingest stream: the copy of the next chunk must queue behind it)
            with torch.cuda.stream(ingest if ingest is not None else torch.cuda.current_stream()):
                d_chunk[:n].copy_(torch.from_numpy(reqs.view(np.uint8).reshape(n, 64)), non_blocking=False)
        if p2p is None:
            tab.submit_device(d_chunk.data_ptr(), n, clk0, d_chunk_out.data_ptr(), stream)
        else:
            ring_step(d_chunk, n, clk0, d_chunk_out)
    progress(f"fill enqueued ({n_fill_steps} steps)")
    torch.cuda.synchronize()
    t_fill = time.perf_counter() - t_fill
    c0 = tab.counters()
    progress("fill done")

    # ---- pre-generated batch pool, resident in HBM
    pool_n = max(2, args.pool)
    host_batches, host_ids, stats = [], [], []
    for b in range(pool_n):
        reqs, ids = gen_batch(rng, BATCH, n_keys, T0 + 1 + b, args.zipf, g.REQ_DTYPE, global_hot=global_hot)
        host_batches.append(reqs); host_ids.append(ids)
        stats.append(batch_stats(ids))
    d_batches = [torch.from_numpy(r.view(np.uint8).reshape(BATCH, 64)).to(dev) for r in host_batches]
    d_outs = [torch.empty((BATCH, 32), dtype=torch.uint8, device=dev) for _ in range(pool_n)]
    clocks = [g.clock_fill(T0 + 1 + b) for b in range(args.steps + args.warmup + 64)]

    def clk_of(b):
        return clocks[min(b, len(clocks) - 1)]

    def one_step(b):
        k = b % pool_n
        if p2p is None:
            tab.submit_device(d_batches[k].data_ptr(), BATCH, clk_of(b), d_outs[k].data_ptr(), stream)
        else:
            ring_step(d_batches[k], BATCH, clk_of(b), d_outs[k])

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    if args.traffic_probe:  # the ncu sub-process: 8 warm steps, then 8 profiled ones, nothing else
        for b in range(8):
            one_step(b)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        for b in range(8, 16):
            one_step(b)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return

    # ---- config 5: GLOBAL sync tick every --tick-ms of wall clock.  Collective, so every rank ticks at the same step: the period
    # in steps is calibrated during warm-up (max over ranks).
    tick_every = None
    tick_log = []

    def do_tick(b):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        # (the receivers' "now" — UpdatedAt / CreatedAt of the installed replicas — in the clock domain of the requests' created_at,
        # which cycles with the batch pool; the kernels' expiry clock clk_of(b) keeps advancing)
        st = p2p.tick(clk_of(b), T0 + 1 + (b % pool_n), stream)
        e1.record()
        torch.cuda.synchronize()
        st["ms"] = e0.elapsed_time(e1)
        tick_log.append(st)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    tw = time.perf_counter()
    for b in range(args.warmup):
        one_step(b)
    progress("warm-up enqueued")
    barrier()
    progress("warm-up done")
    if is_global:
        per_step = (time.perf_counter() - tw) / max(args.warmup, 1)
        t_ps = torch.tensor([per_step], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t_ps, op=dist.ReduceOp.MAX)
        tick_every = max(1, int(args.tick_ms * 1e-3 / float(t_ps.item())))
        do_tick(args.warmup)  # first tick: replicas of the hot set are installed everywhere
        tick_log.clear()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for b in range(args.steps):
        one_step(args.warmup + b)
        if tick_every and (b + 1) % tick_every == 0:
            do_tick(args.warmup + b)
    ev1.record()
    progress("timed steps enqueued")
    barrier()
    progress("timed steps done")
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs:  # before the legs below reuse the output buffers
        last = d_outs[(args.warmup + args.steps - 1) % pool_n].cpu().numpy().view(g.RESP_DTYPE).reshape(BATCH)
        dump_outputs(args.dump_outputs, last, f"_rank{rank}" if N > 1 else "")
    clocks_info = sampler.stop() if rank == 0 else None
    if dist is not None:
        tms = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms.item())
    value = N * BATCH * args.steps / (ms * 1e-3)

    # ---- config 5: convergence after a quiesced tick (functional_test.go:1816-1821): every shard answers a Hits = 0 query on
    # every hot key exactly like shard 0 does
    convergence = None
    if is_global:
        do_tick(args.warmup + args.steps)
        do_tick(args.warmup + args.steps)
        hot = min(global_hot, BATCH)
        # created_at of the query = the installed replicas' "now" (same clock domain as the traffic: a query stamped seconds ahead of
        # every request's created_at would credit the owners' leaky buckets tokens their freshly installed replicas do not see)
        q = bench_requests(np.arange(hot, dtype=np.int64), T0 + 1 + ((args.warmup + args.steps) % pool_n), dtype=g.REQ_DTYPE)
        q["hits"] = 0
        q["behavior"] = np.uint32(O.GLOBAL | O.REQ_IS_OWNER)
        d_q = torch.from_numpy(q.view(np.uint8).reshape(hot, 64)).to(dev)
        d_qo = torch.zeros((hot, 32), dtype=torch.uint8, device=dev)
        ring_step(d_q, hot, clk_of(args.warmup + args.steps), d_qo)
        torch.cuda.synchronize()
        mine = d_qo.view(torch.int64).reshape(hot, 4).clone()  # per key: status | err << 32, limit, remaining, reset_time
        token = torch.from_numpy((q["algorithm"] == 0)).to(dev)
        conv = {"hot_keys_checked": hot, "token_keys": int(token.sum().item())}
        if dist is not None:
            ref = mine.clone()
            dist.broadcast(ref, src=0)
            # TestGlobalBehavior's check (functional_test.go:1816-1821, TOKEN_BUCKET): every peer reports the same status and remaining
            tok_bad = ((ref[:, 0] != mine[:, 0]) | (ref[:, 2] != mine[:, 2])) & token
            # leaky replicas are installed from an int64 Remaining (UpdatePeerGlobals, gubernator.go:443: float64(g.Status.Remaining)) with
            # UpdatedAt = the receiver's now, so a replica may trail its owner by the fraction of a token the owner has leaked since
            lk_diff = (ref[:, 2] - mine[:, 2]).abs() * (~token)
            cst = torch.stack([tok_bad.sum(), lk_diff.max(), (lk_diff > 0).sum(), (ref != mine).any(dim=1).sum()]).to(torch.int64)
            dist.all_reduce(cst, op=dist.ReduceOp.MAX)
            conv.update({"token_keys_differing_max_over_shards": int(cst[0].item()), "leaky_remaining_max_abs_diff": int(cst[1].item()),
                         "leaky_keys_differing_max_over_shards": int(cst[2].item()), "keys_with_any_field_differing": int(cst[3].item()),
                         # the reference's own consistency check is on TOKEN_BUCKET (functional_test.go:1690-1821): that is the criterion;
                         # the leaky replicas' distance from their owners is reported beside it
                         "all_shards_agree": bool(cst[0].item() == 0)})
        else:
            conv["all_shards_agree"] = True
        convergence = conv

    # ---- informational: one C-ABI call with 4 x 65 536 requests (one launch, four rounds inside the kernel)
    big = None
    if N == 1 and p2p is None and pool_n >= 4:
        d_big = torch.cat(d_batches[:4], dim=0).contiguous()
        d_big_out = torch.empty((4 * BATCH, 32), dtype=torch.uint8, device=dev)
        big_steps = max(10, args.steps // 8)
        for b in range(3):
            tab.submit_device(d_big.data_ptr(), 4 * BATCH, clocks[0], d_big_out.data_ptr(), stream)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for b in range(big_steps):
            tab.submit_device(d_big.data_ptr(), 4 * BATCH, clk_of(b), d_big_out.data_ptr(), stream)
        e1.record()
        torch.cuda.synchronize()
        big = {"requests_per_call": 4 * BATCH, "value": 4 * BATCH * big_steps / (e0.elapsed_time(e1) * 1e-3), "unit": "decisions/s",
               "note": "four pool batches with four different created_at in one call: every repeated key is a non-uniform group (segment path); informational"}

    # ---- informational variants of the workload (VERDICT r1): heterogeneous hits on the hot keys; a refill-rate workload whose
    # buckets keep being written back (60 ms duration instead of 60 s)
    variants = None
    if args.variants and N == 1 and p2p is None:
        variants = {}
        for name, kw in (("hetero_hits_5pct", dict(hits_mix=0.05)), ("refill_60ms", dict(duration=60))):
            vb = []
            for b in range(8):
                reqs, _ = gen_batch(rng, BATCH, n_keys, T0 + 1 + b, args.zipf, g.REQ_DTYPE, **kw)
                vb.append(torch.from_numpy(reqs.view(np.uint8).reshape(BATCH, 64)).to(dev))
            for b in range(8):
                tab.submit_device(vb[b % 8].data_ptr(), BATCH, clk_of(b), d_outs[0].data_ptr(), stream)
            torch.cuda.synchronize()
            cb = tab.counters()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            vs = max(50, args.steps // 10)
            e0.record()
            for b in range(vs):
                tab.submit_device(vb[b % 8].data_ptr(), BATCH, clk_of(8 + b), d_outs[0].data_ptr(), stream)
            e1.record()
            torch.cuda.synchronize()
            ca = tab.counters()
            variants[name] = {"value": BATCH * vs / (e0.elapsed_time(e1) * 1e-3), "unit": "decisions/s", "us_per_step": 1e3 * e0.elapsed_time(e1) / vs,
                              "mixed_groups_per_batch": (ca["mixed_groups"] - cb["mixed_groups"]) / vs,
                              "over_limit_fraction": (ca["over_limit"] - cb["over_limit"]) / max(1, ca["requests"] - cb["requests"])}

    # ---- per-kernel timing leg (separate from the number above: the events perturb the pipeline)
    progress("profiling leg")
    tab.set_profiling(True)
    prof_steps = min(args.steps, 200)
    for b in range(prof_steps):
        one_step(args.warmup + args.steps + b)
    barrier()
    prof = tab.get_profile()
    tab.set_profiling(False)

    if args.ncu_window > 0:  # the only launches an `ncu --profile-from-start off` run sees
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        for b in range(args.ncu_window):
            one_step(args.warmup + args.steps + prof_steps + b)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()

    # ---- phase trace of the batch kernel (diagnostic): per-CTA %globaltimer stamps of one launch
    progress("trace legs")
    phase_trace = None
    try:
        tab.set_trace(True)
        for b in range(3):
            one_step(args.warmup + args.steps + prof_steps + 64 + b)
        barrier()
        phase_trace = tab.get_trace()
        raw = tab.get_trace_raw()
        live = raw[:, 0] > 0
        t0 = raw[live, 0].min()
        rel = (raw[live].astype(np.int64) - np.int64(t0)) / 1e3
        slow = int(np.argmax(rel[:, 10]))
        phase_trace["slowest_cta"] = {"cta": int(np.nonzero(live)[0][slow]), "us": [round(float(v), 2) for v in rel[slow]]}
        phase_trace["median_cta_us"] = [round(float(v), 2) for v in np.median(rel, axis=0)]
        tab.set_trace(False)
    except Exception as ex:
        phase_trace = {"error": str(ex)}

    # ---- time stamps of the four pipeline kernels (diagnostic): one isolated batch, then the last of six back to back
    if os.environ.get("GUB_PATH") != "fused":
        try:
            tab.set_trace(True)
            base_b = args.warmup + args.steps + prof_steps + 80
            names = ["k_group", "k_rank", "k_eval", "k_finish"]

            def summarise(raw):
                live = raw[:, :, 0] > 0
                t0 = int(raw[0][live[0], 0].min())
                out = {}
                for k in range(4):
                    r = raw[k][live[k]].astype(np.int64)
                    if not len(r):
                        continue
                    rel = np.where(r > 0, (r - t0) / 1e3, np.nan)
                    out[names[k]] = {"blocks": int(len(r)), "first_entry_us": round(float(np.nanmin(rel[:, 0])), 2),
                                     "median_us": [None if np.all(np.isnan(rel[:, m])) else round(float(np.nanmedian(rel[:, m])), 2) for m in range(8)],
                                     "max_us": [None if np.all(np.isnan(rel[:, m])) else round(float(np.nanmax(rel[:, m])), 2) for m in range(8)]}
                return out
            for b in range(3):
                one_step(base_b + b)
            torch.cuda.synchronize()
            tab.get_ktrace(reset=True)
            one_step(base_b + 3)
            torch.cuda.synchronize()
            iso = summarise(tab.get_ktrace(reset=True))
            for b in range(6):
                one_step(base_b + 4 + b)
            torch.cuda.synchronize()
            piped = summarise(tab.get_ktrace(reset=True))
            phase_trace = {"marks": "0 entry, 1 after griddepcontrol.wait, 2..5 kernel-specific (k_group: keys in table / local ranks / - / fragment joined; "
                                    "k_rank: entry read / base rank / snapshot stored / single answered; k_eval: entry read / member answered), 6 work done, 7 exit; "
                                    "us since the first k_group block entered; latest stamp per block",
                           "isolated_batch": iso, "six_back_to_back_latest": piped}
            tab.set_trace(False)
        except Exception as ex:
            phase_trace = {"error": str(ex)}

    # ---- end-to-end leg from key strings in pinned host memory (N == 1: the public host API; N > 1: pinned H2D + ring step + D2H)
    e2e = None
    progress("end-to-end leg")
    if not args.no_e2e:
        depth = 4
        e2e_steps = args.steps
        if N == 1 and p2p is None:
            native = g.native
            C = native.C
            params = np.zeros(2, dtype=native.PARAMS_DTYPE)  # the workload's two limit configurations: TOKEN and LEAKY, same numbers
            params["limit"] = 100; params["duration"] = 60000; params["algorithm"] = [0, 1]; params["behavior"] = O.REQ_IS_OWNER
            ppin = native.PinnedArray(2, native.PARAMS_DTYPE); ppin.array[:] = params
            packed = []
            for k in range(pool_n):  # every pool batch has its own pinned buffer: the ring cycles all of them
                ids = host_ids[k]
                keys_u8 = key_blob(ids)[0]
                o_at, b_at, tot = C.c_size_t(), C.c_size_t(), C.c_size_t()
                native.lib().gub_keys_layout(BATCH, len(keys_u8), C.byref(o_at), C.byref(b_at), C.byref(tot))
                pin = native.PinnedArray(tot.value, np.uint8)
                kr = pin.array[:BATCH * 16].view(native.KREQ_DTYPE)
                kr["hits"] = host_batches[k]["hits"]; kr["params"] = (ids & 1).astype(np.uint32); kr["created_delta"] = 0
                pin.array[o_at.value:o_at.value + 4 * (BATCH + 1)].view(np.uint32)[:] = np.arange(BATCH + 1, dtype=np.uint32) * 16
                pin.array[b_at.value:b_at.value + len(keys_u8)] = keys_u8
                packed.append((pin, tot.value))
            outs = [native.PinnedArray(BATCH, g.RESP_DTYPE) for _ in range(depth)]
            cpin = []
            for k in range(pool_n):
                c, prm, base = native.compact_batch(host_batches[k])
                ca = native.PinnedArray(BATCH, native.CREQ_DTYPE); ca.array[:] = c
                pa = native.PinnedArray(max(len(prm), 1), native.PARAMS_DTYPE); pa.array[:len(prm)] = prm
                cpin.append((ca, pa, len(prm), base))

            def e2e_run(submit):
                tickets = [None] * depth
                for b in range(min(args.warmup, 8)):
                    tab.wait(submit(b % pool_n, b % depth, b))
                torch.cuda.synchronize()
                t_sub = t_wait = 0.0
                t0_ = time.perf_counter()
                for b in range(e2e_steps):
                    k = b % depth
                    a = time.perf_counter()
                    if tickets[k] is not None:
                        tab.wait(tickets[k])  # the response buffer of this slot has been read back
                    c = time.perf_counter()
                    tickets[k] = submit(b % pool_n, k, b)
                    t_wait += c - a
                    t_sub += time.perf_counter() - c
                for k in range(depth):
                    if tickets[k] is not None:
                        tab.wait(tickets[k])
                torch.cuda.synchronize()
                dt_ = time.perf_counter() - t0_
                return dt_, {"cpu_us_in_submit": 1e6 * t_sub / e2e_steps, "cpu_us_in_wait": 1e6 * t_wait / e2e_steps, "us_per_step": 1e6 * dt_ / e2e_steps}
            dt, split = e2e_run(lambda pb, k, b: tab.submit_keys_async(packed[pb][0].ptr, packed[pb][1], BATCH, ppin.ptr, 2, T0 + 1 + pb, clk_of(b), outs[k].ptr))
            dt_c, split_c = e2e_run(lambda pb, k, b: tab.submit_compact_async(cpin[pb][0].ptr, BATCH, cpin[pb][1].ptr, cpin[pb][2], cpin[pb][3], clk_of(b), outs[k].ptr))
            e2e = {"value": BATCH * e2e_steps / dt, "unit": "decisions/s", "h2d_bytes_per_step": packed[0][1] + 64, "d2h_bytes_per_step": BATCH * 32,
                   "api": "gub_submit_keys_async: key strings (16 B each) + 16-byte request records in pinned host memory, hashing on the device, depth 4; "
                          f"all {pool_n} pool batches cycle through the pinned ring",
                   "host_time": split,
                   "prehashed_compact": {"value": BATCH * e2e_steps / dt_c, "unit": "decisions/s", "h2d_bytes_per_step": BATCH * 32 + 64, "d2h_bytes_per_step": BATCH * 32,
                                         "api": "gub_submit_compact_async (32-byte pre-hashed records)", "host_time": split_c}}
            for pin, _ in packed:
                pin.free()
            for a in outs + [ppin] + [x for c in cpin for x in c[:2]]:
                a.free()
        else:
            # the ring: per step copy the batch from pinned host memory, run the routed step, read the responses back
            h_in = [torch.from_numpy(host_batches[k].view(np.uint8).reshape(BATCH, 64)).pin_memory() for k in range(pool_n)]
            h_out = [torch.empty((BATCH, 32), dtype=torch.uint8).pin_memory() for _ in range(depth)]
            d_ins = [torch.empty((BATCH, 64), dtype=torch.uint8, device=dev) for _ in range(2)]
            d_o = [torch.empty((BATCH, 32), dtype=torch.uint8, device=dev) for _ in range(2)]
            barrier()
            t0_ = time.perf_counter()
            for b in range(e2e_steps):
                if ingest is not None:  # ingest copy + routing on the ingest stream, evaluation + read-back on the current one
                    with torch.cuda.stream(ingest):
                        d_ins[b & 1].copy_(h_in[b % pool_n], non_blocking=True)
                else:
                    d_ins[b & 1].copy_(h_in[b % pool_n], non_blocking=True)
                ring_step(d_ins[b & 1], BATCH, clk_of(b), d_o[b & 1])
                h_out[b % depth].copy_(d_o[b & 1], non_blocking=True)
            barrier()
            dt = time.perf_counter() - t0_
            if dist is not None:
                tdt = torch.tensor([dt], device=dev, dtype=torch.float64)
                dist.all_reduce(tdt, op=dist.ReduceOp.MAX)
                dt = float(tdt.item())
            e2e = {"value": N * BATCH * e2e_steps / dt, "unit": "decisions/s", "h2d_bytes_per_step": N * BATCH * 64, "d2h_bytes_per_step": N * BATCH * 32,
                   "api": "pinned H2D of 64-byte pre-hashed records + gub_p2p_step (route / evaluate out of the mailboxes / collect) + D2H per step"}

    progress("legs done")
    c1 = tab.counters()
    ring_error = None
    if p2p is not None:
        try:
            p2p.status()
        except Exception as ex:
            ring_error = str(ex)
    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel of the evaluation path
    peak, peak_src = load_peaks()
    launches = max(prof["launches"], 1)
    st = {k: float(np.mean([s[k] for s in stats])) for k in stats[0]}
    multi_req, multi_keys = st["repeated_requests"], st["repeated_keys"]
    fused_path = os.environ.get("GUB_PATH") == "fused"
    if fused_path:
        kms = {"k_batch": prof["k_group_ms"] / launches}  # the first timing slot brackets the whole launch of k_batch
        alg = {"k_batch": float(ALGO_BYTES_PER_DECISION * BATCH)}
    else:
        kms = {k: prof[k + "_ms"] / launches for k in ("k_group", "k_rank", "k_eval", "k_finish")}
        # SURVEY 8d's 224 B per decision (64 slot read + 64 slot write-back + 64 request + 32 response), split by where the pipeline
        # moves them (DESIGN.md): a key seen once is done entirely in k_rank; a member of a repeated key has its request read in
        # k_rank (uniformity) and again, with its response written, in k_eval; a repeated key's slot is read once (k_rank, into the
        # snapshot) and written back once (k_eval); k_group reads every request's 8-byte key hash.
        alg = {"k_group": 8.0 * BATCH,
               "k_rank": ALGO_BYTES_PER_DECISION * st["singles"] + 64.0 * multi_req + 64.0 * multi_keys,
               "k_eval": (64.0 + 32.0) * multi_req + 64.0 * multi_keys,
               "k_finish": 0.0}
    dom = max(kms, key=kms.get)
    k_ms = kms[dom]
    path_ms = sum(kms.values())
    achieved = alg[dom] / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
    traffic = None
    if N == 1 and p2p is None and not args.no_traffic:
        traffic = measure_traffic(args)
    dram = None
    if traffic and "error" not in traffic and dom in traffic:
        dram = traffic[dom]["dram_read_bytes_per_launch"] + traffic[dom]["dram_write_bytes_per_launch"]
    dram_path = sum(v["dram_read_bytes_per_launch"] + v["dram_write_bytes_per_launch"] for k, v in traffic.items() if isinstance(v, dict)) \
        if traffic and "error" not in traffic else None
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": dram, "traffic_detail": traffic, "peak_source": peak_src, "kernel_ms": kms, "algorithmic_bytes_per_launch": alg,
                "bytes_per_decision": ALGO_BYTES_PER_DECISION,
                "fractions": {
                    # (1) SURVEY 8d: 224 B x decisions / step time (kernels of consecutive batches overlap; launch gaps included)
                    "survey_8d_over_step_time": ALGO_BYTES_PER_DECISION * BATCH / (ms / args.steps * 1e-3) / 1e9 / peak,
                    # ... and over the sum of the kernels' own times (no overlap credited)
                    "survey_8d_over_kernel_time_sum": ALGO_BYTES_PER_DECISION * BATCH / (path_ms * 1e-3) / 1e9 / peak if path_ms > 0 else None,
                    # (2) what the dominant kernel really moved through DRAM / its time; and the whole path's DRAM bytes / step time
                    "measured_dram_over_kernel_time": (dram / (k_ms * 1e-3) / 1e9 / peak) if dram and k_ms > 0 else None,
                    "measured_dram_path_over_step_time": (dram_path / (ms / args.steps * 1e-3) / 1e9 / peak) if dram_path else None,
                }}
    # (3) north_star's "HBM-random-access roofline": the measured random 64-byte read-modify-write rate of this device over this very
    # table; the batch's distinct-slot traffic (128 B x distinct keys per batch) as a fraction of it
    try:
        ra_gbs = tab.probe_random_access(1 << 26)
        slot_gbs = st["distinct"] * 128.0 / (ms / args.steps * 1e-3) / 1e9
        roofline["random_access"] = {"measured_gbs": ra_gbs, "accesses": 1 << 26, "bytes_per_access": 128, "distinct_keys_per_batch": st["distinct"],
                                     "distinct_slot_gbs": slot_gbs, "frac": slot_gbs / ra_gbs if ra_gbs > 0 else None}
        roofline["fractions"]["distinct_slot_traffic_over_random_access_probe"] = roofline["random_access"]["frac"]
    except Exception as ex:  # diagnostic only
        roofline["random_access"] = {"error": str(ex)}

    cpu = None
    if not args.no_cpu_baseline and N == 1 and not is_global:
        keys = args.cpu_keys or cpu_keys_that_fit(n_keys)
        r = cpu_leg(keys, args.zipf, args.cpu_seconds, seed)
        cpu = {"value": r["value"], "unit": "decisions/s", "cores": r["cores"], "kind": "port", "keys": r["keys"],
               "sample": f"{r['steps']} x {BATCH}-request Zipf({args.zipf}) batches over {r['keys']:,} resident keys"
                         + ("" if r["keys"] == n_keys else f" (of {n_keys:,}: host memory bounds the CPU table)")
                         + f", from key strings (XXH64 + FNV-1 inside the timed call), oracle worker-pool port on {r['cores']} threads, {r['seconds']:.1f} s timed"}

    # single table: k_group, k_rank, k_eval, k_finish (or k_batch alone with GUB_PATH=fused); ring: k_p2p_route, k_seg_wait, the four batch
    # kernels per pass (one pass covers min(N x 65 536, 262 144) requests), k_seg_publish, k_p2p_collect (+ two queue kernels on either side with GLOBAL)
    ring_passes = -(-N * BATCH // min(N * BATCH, 262144))
    per_step_launches = (1 if fused_path else 4) if p2p is None else ((3 if fused_path else 4 + 4 * ring_passes) + (4 if is_global else 0))
    if is_global:
        workload = (f"BASELINE config 5: {n_keys:,} keys, {global_hot:,} GLOBAL hot keys (the top of the Zipf ranking), Zipf s={args.zipf}, {N}xB200, GLOBAL sync tick "
                    f"every {tick_every} steps (~{args.tick_ms:.0f} ms of wall clock): hits to owners over the NVLink mailboxes, UpdatePeerGlobal items by NCCL all-gather")
    elif N == 1:
        workload = "BASELINE config 3: 100M keys, Zipf s=1.1, TOKEN/LEAKY 50/50, 1xB200"
    else:
        workload = (f"BASELINE config 4: 100M keys sharded over {N}xB200 by replicated_hash (fnv1, 512 replicas), Zipf s=1.1; routing kernel stores the records into the owners' "
                    "NVLink mailboxes, the batch kernels evaluate out of them and store the responses into the sources' mailboxes"
                    + ("" if args.no_route_overlap else "; routing, evaluation and collect of consecutive steps overlap (ingest stream + the ring's own evaluation and collect streams)"))
    line = {
        "metric": "rate-limit decisions/sec", "value": value, "unit": "decisions/s", "n_gpus": N, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int64+f64", "data": "synthetic",
        "config": {"workload": workload, "keys": n_keys, "batch_per_gpu": BATCH, "zipf_s": args.zipf, "table_slots_per_gpu": capacity,
                   "cache": f"inputs cycle through {pool_n} resident batches ({pool_n * 6} MiB > L2); table {capacity * 64 / 1e9:.1f} GB >> L2",
                   "batch_profile": st, "fill_seconds": t_fill, "resident_keys_after_fill": c0["inserts"]},
        "clocks": clocks_info, "e2e": e2e, "gpu_launches": per_step_launches * args.steps + (len(tick_log) * 12 if tick_log else 0),
        "roofline": roofline, "cpu_baseline": cpu, "larger_calls": big, "variants": variants, "phase_trace": phase_trace,
        "counters": {k: c1[k] - c0[k] for k in c1},
    }
    if is_global:
        tl = tick_log[:-2] if len(tick_log) > 2 else tick_log
        line["global"] = {"ticks": len(tl), "tick_every_steps": tick_every, "tick_ms_mean": float(np.mean([t["ms"] for t in tl])) if tl else None,
                          "hit_records_per_tick": float(np.mean([t["hits_sent"] for t in tl])) if tl else None,
                          "update_items_per_tick": float(np.mean([t["updates_made"] for t in tl])) if tl else None,
                          "installed_per_tick": float(np.mean([t["installed"] for t in tl])) if tl else None,
                          "gathered_bytes_per_tick": float(np.mean([t["gathered_bytes"] for t in tl])) if tl else None,
                          "convergence": convergence}
    if ring_error:
        line["ring_error"] = ring_error
    print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
