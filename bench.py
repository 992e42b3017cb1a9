#!/usr/bin/env python
"""bench.py — top-k queries/sec of the brute-force scan on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config c2|c4]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Default workload (BASELINE.json configs[1], "c2"): vector_quantize_scan, int8 quantized from a synthetic N(0,1) f32
10M x 384 corpus with the reference's S8 rule, L2 (the default metric), k=20, batch=1.  A "step" is one query scanned against
the whole resident corpus (3.84 GB >> 126 MB L2, so every step streams from HBM).  Exactly K steps are timed, on queries
that depend only on the arguments.  `--dump-outputs DIR` writes the top-k the last timed step returned (rowids and distances,
float64 .npy) so that two builds can be compared output for output.

Our arm prints `value` (queries already in HBM; launch -> candidates -> exact top-k on the host, per query), `e2e` (HOST query
in, host top-k out through the C ABI call the SQLite plugin makes, vsb_scan_topk, one at a time; the pipelined
submit/collect figure beside it; sharded runs: the peer-memory exchange fed with host queries), the batch=1024 half of the
metric (`batched`, tensor-core path, with its own roofline and parity sample), a f32 single-query roofline, the same
statements through SQL for both extensions (`sql_e2e`) and the reference's CPU scan beside it (`cpu_baseline`).
`--config c4` runs BASELINE configs[3] (uint8 cosine dim 1536 n=50M k=100 batch=256, row-sharded over the ranks).
`--impl reference` times the reference's own CPU scan (oracle/_ref built from the unmodified sources with -mavx2 -mfma;
falls back to the oracle port) on all host cores.  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import glob
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC_NAME = "top-k queries/sec, 10M x 384 f32 corpus (int8-quantized scan), k=20, batch=1"
SEED_CORPUS, SEED_QUERY = 1234, 4321
BLOCK = 1 << 19  # rows per generation block (block b is seeded with SEED_CORPUS + b, so shards are N-independent)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------ synthetic data (torch on the GPU: plumbing only)
def gen_block_f32(torch, b: int, rows: int, dim: int, device):
    g = torch.Generator(device=device).manual_seed(SEED_CORPUS + b)
    return torch.randn((rows, dim), generator=g, device=device, dtype=torch.float32)


def quantize_s8(torch, x, scale: float):
    """the reference's S8 rule: q = clamp(trunc(v*scale +- 0.5)) (src/sqlite-vector.c:626-656), offset 0"""
    s = x * scale
    r = torch.where(s < 0, s - 0.5, s + 0.5).trunc()
    return r.clamp_(-128, 127).to(torch.int8)


def corpus_blocks(n: int, lo: int, hi: int):
    """(block index, first row, rows) of the generation blocks overlapping rows [lo, hi)"""
    out = []
    for b in range(lo // BLOCK, (hi + BLOCK - 1) // BLOCK):
        a0, a1 = b * BLOCK, min(n, (b + 1) * BLOCK)
        out.append((b, a0, a1 - a0))
    return out


def corpus_absmax(torch, n, dim, lo, hi, device):
    m = 0.0
    for b, a0, rows in corpus_blocks(n, lo, hi):
        x = gen_block_f32(torch, b, rows, dim, device)
        s, e = max(lo, a0) - a0, min(hi, a0 + rows) - a0
        m = max(m, float(x[s:e].abs().max()))
    return m


def make_queries(torch, count, dim, scale, device):
    g = torch.Generator(device=device).manual_seed(SEED_QUERY)
    qf = torch.randn((count, dim), generator=g, device=device, dtype=torch.float32)
    return quantize_s8(torch, qf, scale)


# ------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None
        self.first = 0

    def mark(self):
        """the timed legs start here; keep one earlier sample (taken under the warm-up load) in case the legs are short"""
        self.first = max(len(self.lines) - 1, 0)

    def wait_first(self, timeout_s: float):
        t0 = time.perf_counter()
        while self.proc and not self.lines and time.perf_counter() - t0 < timeout_s:
            time.sleep(0.01)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines[self.first:]:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "window": "nvidia-smi -lms 20 over the timed value leg and the timed e2e leg (plus the last sample before them)"}


# ------------------------------------------------------------------ CPU reference arm
def host_quant_buffer(parts, dim: int, threads: int = 16) -> np.ndarray:
    """the vector_quantize_preload layout n x [int64 LE rowid | dim bytes] (src/sqlite-vector.c:1295-1311).  Filled by a
    thread pool, block by block, so that the pages are first touched by many threads (spread over the NUMA nodes instead of
    all landing next to one core: round 1 saw the many-thread reference arm move 6.6x between boxes)."""
    n = sum(p.shape[0] for p in parts)
    buf = np.empty((n, 8 + dim), dtype=np.uint8)
    offs = np.cumsum([0] + [p.shape[0] for p in parts])

    def fill(i):
        a, b = int(offs[i]), int(offs[i + 1])
        buf[a:b, :8] = np.arange(a + 1, b + 1, dtype=np.int64).view(np.uint8).reshape(b - a, 8)
        buf[a:b, 8:] = parts[i].view(np.uint8)
    with ThreadPoolExecutor(max(1, threads)) as ex:
        list(ex.map(fill, range(len(parts))))
    return buf.reshape(-1)


def numa_info():
    nodes = glob.glob("/sys/devices/system/node/node[0-9]*")
    model = ""
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                model = ln.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"numa_nodes": len(nodes) or None, "cpu_model": model, "logical_cpus": os.cpu_count(),
            "placement": "unpinned pthreads (OS scheduler), one query per thread over one shared read-only buffer; buffer pages first-touched by a 16-thread pool"}


def cpu_reference_run(buf, n, dim, k, queries_i8: np.ndarray, threads: int, reps: int):
    """times threads*reps queries of the reference's own vQuantRunMemory + vFullScanSortSlots; returns (seconds, kind)"""
    from oracle import pyoracle as po
    need = threads * reps
    q = np.ascontiguousarray(np.resize(queries_i8, (need, dim)))
    try:
        ref = po.RefHarness("avx2")
        assert ref.backend == "AVX2"
        sec = ref.time_queries(buf, n, dim, 8 + dim, 8, po.L2, po.I8, True, po.Q_S8, k, q, threads, reps)
        return sec, "reference"
    except (FileNotFoundError, OSError, AssertionError):
        orc = po.Oracle()

        def work(t):
            for r in range(reps):
                orc.scan_quant_buffer(po.L2, po.Q_S8, q[t * reps + r], buf, n, dim, k)
        ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
        t0 = time.perf_counter()
        [t.start() for t in ths]
        [t.join() for t in ths]
        return time.perf_counter() - t0, "port"


def reference_topk_quant(buf, n, dim, k, q_i8):
    """the UNMODIFIED reference's scalar path (distance-cpu.c) on one query; falls back to the oracle port"""
    from oracle import pyoracle as po
    try:
        return po.RefHarness("cpu").scan_quant_buffer(po.L2, po.Q_S8, q_i8, buf, n, dim, k), "reference(cpu)"
    except (FileNotFoundError, OSError):
        return po.Oracle().scan_quant_buffer(po.L2, po.Q_S8, q_i8, buf, n, dim, k), "oracle"


# ------------------------------------------------------------------ output plumbing
_REAL_STDOUT = None


def claim_stdout():
    """stdout must carry exactly one JSON line: route everything else (NCCL banners, library prints) to stderr"""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm": float(d["hbm_gbs"]), "bf16": float(d["bf16_tflops"]), "bf16_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm": 6650.0, "bf16": 1590.0, "bf16_sustained": 1590.0, "source": "fallback (B200_PROFILING.md)"}


def measure_int8_peak(torch, device):
    """dense int8 tensor throughput of this GPU through the library GEMM (torch._int_mm -> cuBLASLt), 8192^3, best of 5:
    the denominator of the int8 batched roofline (MEASURED_PEAKS.json has no int8 figure)"""
    try:
        n = 8192
        a = torch.randint(-8, 8, (n, n), device=device, dtype=torch.int8)
        b = torch.randint(-8, 8, (n, n), device=device, dtype=torch.int8)
        torch._int_mm(a, b)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch._int_mm(a, b)
            e1.record()
            e1.synchronize()
            best = min(best, e0.elapsed_time(e1))
        del a, b
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12, "measured in this run: torch._int_mm (cuBLASLt int8 -> int32) 8192^3, best of 5"
    except Exception as ex:  # noqa: BLE001
        return None, f"unavailable ({ex})"


def ncu_fact(pattern: str, key: str):
    """a figure from the newest committed ncu summary that has it (profiles/*<pattern>*.json)"""
    for p in sorted(glob.glob(os.path.join(ROOT, "profiles", f"*{pattern}*.json")), reverse=True):
        try:
            d = json.load(open(p))
        except (OSError, ValueError):
            continue
        if isinstance(d, dict) and d.get(key) is not None:
            return d[key], os.path.relpath(p, ROOT)
    return None, None


def dump_outputs(dirname: str, arrays: dict):
    """--dump-outputs: every result array as DIR/<name>.npy in float64 (which holds the int64 rowids exactly)"""
    os.makedirs(dirname, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(dirname, f"{name}.npy"), np.asarray(arr, dtype=np.float64))


# ------------------------------------------------------------------ main
def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c4"], help="c2: BASELINE configs[1] (the metric's config); c4: configs[3]")
    ap.add_argument("--n", "--rows", dest="n", type=int, default=0, help="corpus rows (--rows: torchrun's own parser rejects a bare --n as ambiguous)")
    ap.add_argument("--dim", type=int, default=0)
    ap.add_argument("--k", type=int, default=0)
    ap.add_argument("--cpu-threads", type=int, default=0, help="threads of the CPU reference leg (0 = all cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-batched", action="store_true", help="skip the batch=1024 tensor-core legs")
    ap.add_argument("--no-extras", action="store_true", help="skip the f32 roofline and the SQL end-to-end legs")
    ap.add_argument("--group", type=int, default=8, help="sharded runs: queries per exchange group")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"], help="sharded single queries: NVLink peer-memory push (engine) or NCCL all-gather (round 1)")
    ap.add_argument("--engine-opt", action="append", default=[], help="name=value passed to vsb_set_option (experiments)")
    ap.add_argument("--batch-depth", type=int, default=2, choices=[1, 2], help="sharded batches over the peer exchange: batches in flight")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step to DIR/<name>.npy")
    a = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != a.gpus and world > 1:
        log(f"warning: WORLD_SIZE={world} but --gpus {a.gpus}; using WORLD_SIZE")
    cores = a.cpu_threads or (os.cpu_count() or 1)

    import torch

    if a.config == "c4":
        if a.impl == "reference":
            if rank == 0:
                emit({"impl": "reference", "unavailable": "config c4 has no CPU arm: one batch is ~1.7 h of the reference's AVX2 scan (BASELINE.md section 2)"})
            return 0
        return run_c4(torch, a, rank, local_rank, world)

    n, dim, k = a.n or 10_000_000, a.dim or 384, a.k or 20
    K, W = max(a.steps, 1), max(a.warmup, 0)
    workload = f"vector_quantize_scan int8 dim={dim} n={n} k={k} batch=1 L2"
    if a.impl == "reference":
        if rank != 0:
            return 0
        reference_arm(torch, a, n, dim, k, K, W, workload, cores)
        return 0

    import torch.distributed as dist

    import sqlite_vector_b200 as vs
    from sqlite_vector_b200 import api, shard

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    eng = vs.load_engine()
    for kv in a.engine_opt:
        name, val = kv.split("=")
        eng.set_option(name, int(val))

    # ---- resident corpus shard (preload is outside the timed region, like the reference's preloaded buffer)
    bounds = shard.shard_bounds(n, world)
    lo, hi = bounds[rank], bounds[rank + 1]
    t0 = time.perf_counter()
    amax = corpus_absmax(torch, n, dim, lo, hi, device)
    if world > 1:
        t = torch.tensor([amax], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        amax = float(t.item())
    scale = float(np.float32(127.0) / np.float32(amax))  # S8: 127/max(|min|,|max|), offset 0 (:1265-1268)
    ix = vs.Index(api.I8, dim, hi - lo, device=local_rank, first_seq=lo)
    want_host = (rank == 0 and not a.no_cpu_baseline)      # rank 0 keeps the WHOLE corpus on the host for the reference checks
    host_parts = []
    for b, a0, rows in corpus_blocks(n, lo, hi):
        x = quantize_s8(torch, gen_block_f32(torch, b, rows, dim, device), scale)
        s, e = max(lo, a0) - a0, min(hi, a0 + rows) - a0
        xs = x[s:e].contiguous()
        torch.cuda.synchronize()
        ix.append_device(xs.data_ptr(), e - s)
        if want_host and world == 1:
            host_parts.append(xs.cpu().numpy())
    ix.finalize()
    if want_host and world > 1:                             # the other shards' rows, generated here only for the check
        for b, a0, rows in corpus_blocks(n, 0, n):
            host_parts.append(quantize_s8(torch, gen_block_f32(torch, b, rows, dim, device), scale).cpu().numpy())
    NQ = max(K + W + 8, 1024)
    q_all = make_queries(torch, NQ, dim, scale, device)                  # int8 [NQ, dim]
    pitch = ix.query_pitch
    q_dev = torch.zeros((NQ, pitch), dtype=torch.uint8, device=device)
    q_dev[:, :dim] = q_all.view(torch.uint8)
    q_host = q_all.cpu().numpy()
    torch.cuda.synchronize()
    log(f"[rank {rank}] shard rows [{lo},{hi}) resident in {time.perf_counter() - t0:.1f}s; scale={scale:.4f}")

    st = torch.cuda.ExternalStream(ix.stream, device=device)

    def step_device(i):
        ix.scan_device_query(api.L2, q_dev[i].data_ptr(), k)
        return ix.collect_last(k)

    exch = None
    if world > 1:
        exch = (shard.PeerExchange(ix, eng, world, rank, bounds, group=a.group) if a.exchange == "peer"
                else shard.DeviceExchange(ix, eng, world, bounds, device, group=a.group))
    G = exch.group if exch else 1
    depth = getattr(exch, "max_in_flight", 2) if exch else 2

    def run_sharded(first, count, on_device):
        """`count` independent queries through the grouped exchange, `depth` groups in flight: the exchange + merge of group g
        overlaps the scans of the following groups.  on_device=False: host queries (pinned H2D inside the call)."""
        pending, last_res = [], None
        for g0 in range(0, count, G):
            i0, m = (first + g0) % (NQ - G), min(G, count - g0)
            if on_device:
                t = exch.submit_strided(api.L2, q_dev[i0].data_ptr(), pitch, m, k, True)
            else:
                t = exch.submit_strided(api.L2, q_host[i0:i0 + m], q_host.strides[0], m, k, False)
            pending.append((t, i0 + m - 1))
            if len(pending) == depth:
                t0_, last_i = pending.pop(0)
                last_res = (exch.finish(t0_)[-1], last_i)
        while pending:
            t0_, last_i = pending.pop(0)
            last_res = (exch.finish(t0_)[-1], last_i)
        return last_res

    def run_single(first, count):
        """independent single queries, two in flight: query i+1 is scanning while the host finishes query i"""
        pending, last = None, None
        for i in range(count):
            qi = (first + i) % NQ
            slot = ix.scan_device_query(api.L2, q_dev[qi].data_ptr(), k)
            if pending is not None:
                last = (ix.collect(pending[0], k), pending[1])
            pending = (slot, qi)
        last = (ix.collect(pending[0], k), pending[1])
        return last

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: queries resident in HBM
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()         # nvidia-smi needs a moment before its first line: start it ahead of the warm-up
    if world == 1:
        run_single(0, max(W, 1))
    else:
        run_sharded(0, max(W, 1), True)
    if sampler:
        sampler.wait_first(2.0)
    barrier()
    if sampler:
        sampler.mark()          # samples from here on (value leg and e2e leg, both under the same load) are the ones reported
    l0 = eng.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    e0.record(st)
    last, last_qi = run_single(W, K) if world == 1 else run_sharded(W, K, True)
    e1.record(st)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    ms_dev = e0.elapsed_time(e1)
    launches = eng.kernel_launches() - l0
    # the step time is the slower of the device-event span and the wall clock around the same region
    ms_total = max(ms_dev, t_wall * 1e3) if world > 1 else ms_dev
    if world > 1:
        t = torch.tensor([ms_total], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())

    # the scan kernel alone (one launch at a time on one stream, events around it): what ncu's serialised list shows
    alone_ms = None
    try:
        old_streams = eng.set_option("scan_streams", 1)
        eng.set_option("time_kernels", 1)
        ix.profile_read()
        for i in range(12):
            step_device(W + i)
        prof = ix.profile_read()
        eng.set_option("time_kernels", 0)
        eng.set_option("scan_streams", old_streams)
        alone_ms = prof["scan_ms"] / max(prof["scan_launches"], 1)
        filter_ms = prof["filter_ms"] / max(prof["filter_launches"], 1)
    except Exception as ex:  # noqa: BLE001
        log("kernel-alone timing failed:", ex)
        filter_ms = None
    # sequential single-query latency (launch -> complete exact top-k), for information
    lat_ms, lat_pct = None, None
    if world == 1:
        torch.cuda.synchronize()
        lats = []
        for i in range(min(K, 100)):
            t0l = time.perf_counter()
            step_device(W + i)
            lats.append((time.perf_counter() - t0l) * 1e3)
        lat_ms = float(np.mean(lats))
        lat_pct = {"p50": float(np.percentile(lats, 50)), "p95": float(np.percentile(lats, 95)), "n": len(lats)}

    # ---- e2e: host query in, host top-k out, through the public C-ABI call
    pipelined_qps = None
    if world == 1:
        for i in range(max(W, 1)):
            ix.scan_topk(api.L2, q_host[i], k)
        barrier()
        surv0, q0 = ix.stat("survivors"), ix.stat("queries")
        # (a) THE call the SQLite plugin makes from xFilter (vsb_scan_topk), one query at a time: pinned H2D of the query + scan +
        #     filter + D2H of the candidate head + host slot replay, nothing overlapped across queries.  This is e2e.value.
        t0 = time.perf_counter()
        for i in range(K):
            last_e2e = ix.scan_topk(api.L2, q_host[W + (i % (NQ - W - 1))], k)[0]
        e2e_s = time.perf_counter() - t0
        e2e_qi = W + ((K - 1) % (NQ - W - 1))
        # (b) the asynchronous pair vsb_scan_submit(host query) / vsb_collect, two queries in flight (what a batching caller gets)
        t0 = time.perf_counter()
        pending = None
        for i in range(K):
            slot = ix.scan_submit(api.L2, q_host[W + (i % (NQ - W - 1))], k, on_device=False, fetch=True)
            if pending is not None:
                ix.collect(pending, k)
            pending = slot
        ix.collect(pending, k)
        pipelined_qps = K / (time.perf_counter() - t0)
        avg_surv = (ix.stat("survivors") - surv0) / max(ix.stat("queries") - q0, 1)
    else:
        run_sharded(0, max(W, 1), False)
        barrier()
        t0 = time.perf_counter()
        last_e2e, e2e_qi = run_sharded(W, K, False)
        barrier()
        e2e_s = time.perf_counter() - t0
        t = torch.tensor([e2e_s], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
        avg_surv = None
    clocks = sampler.stop() if sampler else None
    d2h_bytes = int(ix.stat("fetch_bytes")) if world == 1 else int(exch.d2h_bytes_per_query)

    # ---- sharded runs: the batch=1024 half of the metric through the row-sharded tensor-core path (every rank takes part)
    batched_sharded = None
    if world > 1 and not a.no_batched:
        try:
            B = 1024
            use_peer = a.exchange == "peer"
            if use_peer:
                # entry logs pushed over NVLink peer memory by the engine, device-side wait, GPU merge; two batches in flight
                rb = exch.batch_finish(exch.batch_submit(api.L2, q_host[:B], k), as_arrays=True)   # warm-up: row norms, tensor maps
                barrier()
                nb, t0b, pending = 10, time.perf_counter(), None
                for _ in range(nb):
                    t = exch.batch_submit(api.L2, q_host[:B], k)
                    if a.batch_depth == 1:
                        rb = exch.batch_finish(t, as_arrays=True)
                        continue
                    if pending is not None:
                        rb = exch.batch_finish(pending, as_arrays=True)
                    pending = t
                if pending is not None:
                    rb = exch.batch_finish(pending, as_arrays=True)
            else:
                shard.sharded_batch_topk(ix, api.L2, q_host[:B], k, bounds, device, as_arrays=True)   # warm-up
                barrier()
                nb, t0b = 5, time.perf_counter()
                for _ in range(nb):
                    rb = shard.sharded_batch_topk(ix, api.L2, q_host[:B], k, bounds, device, as_arrays=True)
            barrier()
            dtb = (time.perf_counter() - t0b) / nb
            t = torch.tensor([dtb], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dtb = float(t.item())
            if rb is None:
                batched_sharded = {"error": "the batch path refused on some shard"}
            else:
                batched_sharded = {"workload": f"vector_quantize_scan int8 dim={dim} n={n} k={k} batch={B} L2, {world} row shards",
                                   "queries_per_s": B / dtb, "ms_per_batch": dtb * 1e3, "batch": B,
                                   "end_to_end_tflops": 2.0 * dim * B * n / dtb / 1e12,
                                   "path": ("per shard: tcgen05 scoring + exact refine + slot replay with entry logs; the log blocks are pushed into every peer's log area over NVLink "
                                            "(push_logs_kernel), device-side flag wait, GPU merge replay; two batches in flight, one host wait per batch" if use_peer else
                                            "per shard: tcgen05 scoring + exact refine + slot replay with entry logs; NCCL all-gather of the logs; GPU merge replay"),
                                   "_result": rb}
        except Exception as ex:  # never lose the headline line
            batched_sharded = {"error": str(ex)}
    # ---- and through REPLICAS: the column fits one GPU (n * dim bytes), so every rank holds all of it and the global batch of
    # world x 1024 queries is split by query (shard.query_sharded_batch_topk): no exchange on the data path
    batched_replicas = None
    if world > 1 and not a.no_batched and n * dim <= 40e9:
        try:
            B = 1024
            ixr = vs.Index(api.I8, dim, n, device=local_rank)
            for b, a0, rows in corpus_blocks(n, 0, n):
                x = quantize_s8(torch, gen_block_f32(torch, b, rows, dim, device), scale)
                torch.cuda.synchronize()
                ixr.append_device(x.data_ptr(), rows)
                del x
            ixr.finalize()
            q_glob = np.concatenate([np.roll(q_host[:B], 37 * r, axis=0) for r in range(world)])      # the global batch; rank r answers [r*B, (r+1)*B)
            shard.query_sharded_batch_topk(ixr, api.L2, q_glob, k, gather=False)                        # warm-up: row norms, tensor maps
            barrier()
            nb, t0b = 10, time.perf_counter()
            for _ in range(nb):
                (rid, rdd, rcn), (qlo, qhi) = shard.query_sharded_batch_topk(ixr, api.L2, q_glob, k, gather=False)
            barrier()
            dtb = (time.perf_counter() - t0b) / nb
            t = torch.tensor([dtb], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dtb = float(t.item())
            # once more with the results all-gathered to every rank (what sharded_batch_topk / the peer exchange deliver)
            barrier()
            t0g = time.perf_counter()
            for _ in range(3):
                shard.query_sharded_batch_topk(ixr, api.L2, q_glob, k, device=device, gather=True)
            barrier()
            dtg = (time.perf_counter() - t0g) / 3
            t = torch.tensor([dtg], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dtg = float(t.item())
            ixr.close()
            batched_replicas = {"workload": f"vector_quantize_scan int8 dim={dim} n={n} k={k} L2, global batch {world} x {B} queries, column replicated on {world} GPUs",
                                "queries_per_s": world * B / dtb, "ms_per_global_batch": dtb * 1e3, "batch_per_gpu": B, "global_batch": world * B,
                                "queries_per_s_results_on_every_rank": world * B / dtg,
                                "scaling": "weak in queries (each GPU answers its own 1024 of the global batch over the whole column)",
                                "path": "shard.query_sharded_batch_topk: vsb_scan_topk (tcgen05 batch path) on this rank's query slice, host queries in, host top-k out; "
                                        "no exchange on the data path; queries_per_s_results_on_every_rank adds one NCCL all-gather of the results",
                                "_result": (rid, rdd, rcn, q_glob[qlo:qhi])}
        except Exception as ex:  # never lose the headline line
            batched_replicas = {"error": str(ex)}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"topk_ids": last[0], "topk_distances": last[1],
                                      "e2e_topk_ids": last_e2e[0], "e2e_topk_distances": last_e2e[1]})

    # ---- roofline of the dominant kernel (scan_kernel): algorithmic bytes = rows * dim * 1 B per launch
    pk = peaks()
    shard_bytes = (hi - lo) * dim
    step_ms = ms_total / K
    achieved = shard_bytes / (step_ms * 1e-3) / 1e9
    traffic, traffic_src = (ncu_fact("scan_kernel_traffic", "dram_bytes_per_launch") if (world == 1 and n == 10_000_000 and dim == 384) else (None, None))

    out = {
        "metric": METRIC_NAME, "value": K / (ms_total * 1e-3), "unit": "queries/s", "n_gpus": world, "steps": K, "warmup": W,
        "steps_timed": K, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int8",
        "data": "synthetic N(0,1) f32 (seed 1234) quantized to int8 with the reference S8 rule; queries seed 4321",
        "config": {"workload": workload, "metric": "L2", "k": k, "batch": 1, "rows": n, "dim": dim, "shards": world,
                   "l2_flush": "none needed: each step streams the whole shard (%.2f GB) which exceeds the 126 MB L2" % (shard_bytes / 1e9),
                   "result_mode": "exact reference slot replay (bit-exact rowids/order/distances vs distance-cpu.c)",
                   "timed_region": f"the {K} steps back to back",
                   "in_flight": 2 if world == 1 else depth * G,
                   "exchange": None if world == 1 else (
                       f"groups of {G} independent queries, {depth} groups in flight; every filter kernel stores its result head into every peer's gather buffer over NVLink "
                       "(cudaIpc peer memory) and raises a flag; the receiver waits on the flags on its own stream, one D2H per group, host slot replay (no collective library on the data path)"
                       if a.exchange == "peer" else f"groups of {G} queries: one NCCL all-gather of the shards' result heads + one D2H per group")},
        "e2e": {"value": K / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": int(pitch),
                "d2h_bytes_per_step": d2h_bytes, "avg_candidates_per_query": avg_surv, "pipelined_value": pipelined_qps,
                "note": ("value = the synchronous vsb_scan_topk call the SQLite plugin makes from xFilter, one query at a time (pinned H2D of the query, scan + filter kernels, "
                         "one D2H of the candidate head, host slot replay); pipelined_value = vsb_scan_submit(host query)/vsb_collect with two queries in flight"
                         if world == 1 else
                         "vsb_exchange_submit with HOST queries (pinned H2D per query) + scan/filter kernels on every rank + peer-memory push of the heads + D2H + host slot replay, same grouping as value")},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": pk["hbm"], "unit": "GB/s", "frac": achieved / pk["hbm"], "traffic": traffic,
                     "traffic_source": traffic_src, "kernel": "vsb::scan_kernel<int8,L2>", "avg_launch_ms": step_ms, "launches_timed": K,
                     "kernel_alone_ms": alone_ms, "kernel_alone_gbs": (shard_bytes / (alone_ms * 1e-3) / 1e9) if alone_ms else None,
                     "filter_kernel_alone_ms": filter_ms, "peak_source": pk["source"] + " hbm_gbs",
                     "algorithmic_bytes_per_launch": int(shard_bytes),
                     "note": "consecutive scan launches alternate between two streams and overlap at CTA granularity (an SM starts the next query's CTA when its CTA of the "
                             "current one exits), so per-launch events would double count: avg_launch_ms is the device-timed span of the timed region / launches, i.e. achieved is "
                             "the WHOLE-STEP rate (filter, copies and host replay included); kernel_alone_* is one launch at a time on one stream. peak is the measured COPY bandwidth "
                             "(reads + writes); this kernel only reads, so frac can exceed 1.0"},
        "clocks": clocks,
        "wall_s_timed_region": t_wall,
        "single_query_latency_ms": lat_ms,
        "single_query_latency_percentiles_ms": lat_pct,
        "top1": {"rowid": int(last[0][0]), "distance": float(last[1][0])},
    }

    # ---- parity of the timed results against the UNMODIFIED reference on the same data (rank 0, every N)
    buf = None
    if want_host:
        try:
            buf = host_quant_buffer(host_parts, dim)
            del host_parts
            par = {}
            for name, (res, qi) in (("value_leg_last_query", (last, last_qi)), ("e2e_leg_last_query", (last_e2e, e2e_qi))):
                (ids_ref, d_ref), how = reference_topk_quant(buf, n, dim, k, q_host[qi])
                par[name] = bool(np.array_equal(ids_ref, res[0]) and np.array_equal(d_ref, res[1]))
                par["checked_against"] = how
            par["gpu_result_matches_reference"] = all(v for kk, v in par.items() if kk.endswith("_query"))
            out["parity"] = par
        except MemoryError as ex:
            out["parity"] = {"error": str(ex)}

    # ---- batched queries on the tensor cores (BASELINE metric "batch=1024"; configs[2])
    if world == 1 and not a.no_batched:
        try:
            out["batched"] = batched_legs(torch, vs, api, eng, ix, q_host, buf, n, dim, k, device, pk)
        except Exception as ex:  # never lose the headline line
            out["batched"] = {"error": str(ex)}
    if batched_sharded is not None:
        rb = batched_sharded.pop("_result", None)
        if rb is not None and buf is not None:
            chk = []
            for b in (0, 511, 1023):
                (ids_ref, d_ref), how = reference_topk_quant(buf, n, dim, k, q_host[b])
                chk.append(bool(np.array_equal(ids_ref, rb[0][b, :rb[2][b]]) and np.array_equal(d_ref, rb[1][b, :rb[2][b]])))
            batched_sharded["parity"] = {"queries_checked": [0, 511, 1023], "gpu_result_matches_reference": all(chk), "checked_against": how}
        out["batched"] = {"int8_L2_dim%d_n%d_b1024_sharded" % (dim, n): batched_sharded}
    if batched_replicas is not None:
        rr = batched_replicas.pop("_result", None)
        if rr is not None and buf is not None:
            chk = []
            for b in (0, 511, 1023):
                (ids_ref, d_ref), how = reference_topk_quant(buf, n, dim, k, rr[3][b])
                chk.append(bool(np.array_equal(ids_ref, rr[0][b, :rr[2][b]]) and np.array_equal(d_ref, rr[1][b, :rr[2][b]])))
            batched_replicas["parity"] = {"queries_checked": [0, 511, 1023], "gpu_result_matches_reference": all(chk), "checked_against": how}
        out.setdefault("batched", {})["int8_L2_dim%d_n%d_b1024_replicas" % (dim, n)] = batched_replicas

    # ---- extras (N = 1): f32 single-query roofline, SQL end to end
    if world == 1 and not a.no_extras:
        try:
            out["fp_single_query"] = fp_single_query_leg(torch, vs, api, ix, device, pk, n, dim, k)
        except Exception as ex:  # noqa: BLE001
            out["fp_single_query"] = {"error": str(ex)}
        try:
            out["sql_e2e"] = sql_e2e_leg()
        except Exception as ex:  # noqa: BLE001
            out["sql_e2e"] = {"error": str(ex)}

    # ---- CPU baseline beside it (rank 0, N=1): the reference's AVX2 scan on a bounded sample
    if want_host and world == 1 and buf is not None:
        qs = q_host[W:W + 8]
        sec1, kind = cpu_reference_run(buf, n, dim, k, qs, 1, 1)
        secN, kind = cpu_reference_run(buf, n, dim, k, qs, cores, 1)
        out["cpu_baseline"] = {"value": cores / secN, "unit": "queries/s", "cores": cores, "kind": kind,
                               "sample": f"{cores} independent queries (one per thread) over the same {n}x{dim} int8 preload buffer, "
                                         f"reference vQuantRunMemory+vFullScanSortSlots built -O3 -mavx2 -mfma; wall {secN:.2f}s",
                               "achieved_gbs": cores * n * dim / secN / 1e9, "host": numa_info(),
                               "single_thread_value": 1.0 / sec1, "single_thread_s_per_query": sec1,
                               "gpu_result_matches_reference": (out.get("parity") or {}).get("gpu_result_matches_reference")}
    emit(out)
    if world > 1:
        dist.destroy_process_group()
    return 0


def batched_legs(torch, vs, api, eng, ix, q_host, buf, n, dim, k, device, pk):
    """batch=1024 through vsb_scan_topk (host queries in, host top-k out): tcgen05 scoring + exact refinement.  First-class
    half of the BASELINE metric: each leg carries its own tensor roofline (tc_scan_kernel device time from the engine's CUDA
    events, peak measured) and a parity sample against the reference / oracle on the same data."""
    from oracle import pyoracle as po
    res = {}
    int8_peak, int8_note = measure_int8_peak(torch, device)
    pct_i8, src_i8 = ncu_fact("ncu_summary", "tc_int8_tensor_pipe_pct")
    pct_bf, src_bf = ncu_fact("ncu_summary", "tc_bf16_tensor_pipe_pct")

    def run(name, index, queries, metric, flop_per_pair, peak, peak_note, parity):
        B = queries.shape[0]
        index.scan_topk(metric, queries, k)                      # warm-up (row norms, tensor maps, workspaces)
        us0, rows0, bus0 = index.stat("tc_us"), index.stat("tc_rows"), index.stat("batch_us")
        reps = 10
        for _ in range(reps):
            r = index.scan_topk(metric, queries, k)
        dt = (index.stat("batch_us") - bus0) / reps * 1e-6       # wall time inside the C-ABI call (host queries in, host top-k out)
        tc_s = (index.stat("tc_us") - us0) / reps * 1e-6
        tc_rows = (index.stat("tc_rows") - rows0) / reps
        tc_tflops = flop_per_pair * B * tc_rows / tc_s / 1e12 if tc_s > 0 else None
        res[name] = {"queries_per_s": B / dt, "ms_per_batch": dt * 1e3, "batch": B,
                     "end_to_end_tflops": flop_per_pair * B * index.rows / dt / 1e12,
                     "h2d_bytes_per_batch": int(queries.nbytes), "d2h_bytes_per_batch": int(B * ((k + 31) // 32 * 32) * 8),
                     "roofline": {"bound": "tensor", "kernel": "vsb::tc_scan_kernel", "achieved": tc_tflops, "peak": peak, "unit": "TFLOP/s",
                                  "frac": (tc_tflops / peak) if (tc_tflops and peak) else None, "peak_note": peak_note,
                                  "tc_kernel_ms_per_batch": tc_s * 1e3, "rows_scored_on_tensor_cores": tc_rows,
                                  "hbm_gbs": index.rows * index.dim * api.ELEM_SIZE[index.vtype] / tc_s / 1e9 if tc_s > 0 else None},
                     "parity": parity(r) if parity else None}

    def parity_int8(r):
        if buf is None:
            return None
        ok, how = [], None
        for b in (0, 257, 1023):
            (ids_ref, d_ref), how = reference_topk_quant(buf, n, dim, k, q_host[b])
            ok.append(bool(np.array_equal(ids_ref, r[b][0]) and np.array_equal(d_ref, r[b][1])))
        return {"queries_checked": [0, 257, 1023], "gpu_result_matches_reference": all(ok), "checked_against": how, "rule": "bit-exact rowids, order, distances"}

    run("int8_L2_dim%d_n%d_b1024" % (dim, n), ix, q_host[:1024], api.L2, 2.0 * dim, int8_peak, int8_note, parity_int8)
    res["int8_L2_dim%d_n%d_b1024" % (dim, n)]["roofline"]["tensor_pipe_pct_ncu"] = pct_i8
    res["int8_L2_dim%d_n%d_b1024" % (dim, n)]["roofline"]["tensor_pipe_pct_source"] = src_i8

    # BASELINE configs[2]: vector_full_scan dot bf16 dim=768 n=10M k=20 batch=1024
    n3, d3 = 10_000_000, 768
    ix3 = vs.Index(api.BF16, d3, n3, device=device.index or 0)
    host3 = np.empty((n3, d3), dtype=np.uint16) if buf is not None else None      # 15.4 GB: the oracle's copy (only with the CPU legs on)
    for b, a0, rows in corpus_blocks(n3, 0, n3):
        x = gen_block_f32(torch, 7000 + b, rows, d3, device).to(torch.bfloat16)
        torch.cuda.synchronize()
        ix3.append_device(x.data_ptr(), rows)
        if host3 is not None:
            host3[a0:a0 + rows] = x.view(torch.int16).cpu().numpy().view(np.uint16)
    ix3.finalize()
    g = torch.Generator(device=device).manual_seed(SEED_QUERY + 1)
    q3 = torch.randn((1024, d3), generator=g, device=device).to(torch.bfloat16).view(torch.int16).cpu().numpy().view(np.uint16)

    def parity_bf16(r):
        if host3 is None:
            return None
        from tests.fpcheck import assert_fp_topk
        orc = po.Oracle()
        rowids = np.arange(1, n3 + 1, dtype=np.int64)
        sample = [0, 300, 777, 1023]
        with ThreadPoolExecutor(len(sample)) as ex:
            wants = list(ex.map(lambda b: orc.scan_dense(po.DOT, po.BF16, q3[b], host3, rowids, k), sample))
        ok, worst = True, 0.0
        for b, (wi, wd) in zip(sample, wants):
            try:
                assert_fp_topk(r[b][0], r[b][1], wi, wd, po.DOT, lambda rr, b=b: orc.distance(po.DOT, po.BF16, q3[b], host3[rr - 1]), ("c3", b))
            except AssertionError as ex:
                ok = False
                log("bf16 parity:", ex)
            worst = max(worst, float(np.max(np.abs(r[b][1] - wd) / np.maximum(np.abs(wd).max(), 1e-30))))
        # and every query against the single-query CUDA-core path (same kernel the -m gpu tests pin to the oracle)
        eng.set_option("no_batch", 1)
        try:
            same = 0
            for b in range(0, 1024, 16):
                (one,) = ix3.scan_topk(api.DOT, q3[b], k)
                same += int(np.array_equal(one[0], r[b][0]) and np.allclose(one[1], r[b][1], rtol=1e-5, atol=0))
        finally:
            eng.set_option("no_batch", 0)
        return {"queries_checked_vs_oracle": sample, "gpu_result_matches_reference": ok, "checked_against": "oracle (distance-cpu.c restatement, pinned to the reference)",
                "rule": "distances within 1e-5 relative, rowids equal except oracle near-ties (tests/fpcheck.py)", "max_rel_err": worst,
                "queries_equal_to_single_query_path": f"{same}/64"}

    run("bf16_DOT_dim768_n10M_b1024", ix3, q3, api.DOT, 2.0 * d3, pk["bf16"], "measured cuBLAS bf16 burst peak (MEASURED_PEAKS.json bf16_tflops)", parity_bf16)
    res["bf16_DOT_dim768_n10M_b1024"]["roofline"]["frac_of_sustained_peak"] = (
        res["bf16_DOT_dim768_n10M_b1024"]["roofline"]["achieved"] / pk["bf16_sustained"] if res["bf16_DOT_dim768_n10M_b1024"]["roofline"]["achieved"] else None)
    res["bf16_DOT_dim768_n10M_b1024"]["roofline"]["tensor_pipe_pct_ncu"] = pct_bf
    res["bf16_DOT_dim768_n10M_b1024"]["roofline"]["tensor_pipe_pct_source"] = src_bf
    ix3.close()
    return res


def fp_single_query_leg(torch, vs, api, ix_i8, device, pk, n, dim, k):
    """vector_full_scan on the raw f32 column (15.36 GB per query at 10M x 384): the CUDA-core FFMA path against HBM"""
    ixf = vs.Index(api.F32, dim, n, device=device.index or 0)
    for b, a0, rows in corpus_blocks(n, 0, n):
        x = gen_block_f32(torch, b, rows, dim, device)
        torch.cuda.synchronize()
        ixf.append_device(x.data_ptr(), rows)
    ixf.finalize()
    g = torch.Generator(device=device).manual_seed(SEED_QUERY)
    qf = torch.randn((64, dim), generator=g, device=device, dtype=torch.float32)
    pitch = ixf.query_pitch
    qd = torch.zeros((64, pitch), dtype=torch.uint8, device=device)
    qd[:, :dim * 4] = qf.view(torch.uint8).reshape(64, dim * 4)
    torch.cuda.synchronize()
    st = torch.cuda.ExternalStream(ixf.stream, device=device)
    for i in range(3):
        ixf.scan_device_query(api.L2, qd[i].data_ptr(), k)
        ixf.collect_last(k)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters, pending = 40, None
    e0.record(st)
    for i in range(iters):
        slot = ixf.scan_device_query(api.L2, qd[i % 64].data_ptr(), k)
        if pending is not None:
            ixf.collect(pending, k)
        pending = slot
    res = ixf.collect(pending, k)
    e1.record(st)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    nbytes = n * dim * 4
    out = {"workload": f"vector_full_scan L2 f32 dim={dim} n={n} k={k} batch=1", "queries_per_s": 1e3 / ms, "ms_per_query": ms,
           "roofline": {"bound": "hbm", "kernel": "vsb::scan_kernel<f32,L2>", "achieved": nbytes / (ms * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                        "frac": nbytes / (ms * 1e-3) / 1e9 / pk["hbm"], "algorithmic_bytes_per_launch": nbytes},
           "top1": [int(res[0][0]), float(res[1][0])]}
    ixf.close()
    return out


def sql_e2e_leg(n=200_000, queries=30):
    """the same SQL statements through stock SQLite for both extensions, each in its own process (tools/sql_bench.py)"""
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sql_bench.py"), "--n", str(n), "--dim", "384", "--queries", str(queries), "--which", "both"],
                       capture_output=True, text=True, timeout=600)
    rows = [json.loads(ln) for ln in p.stdout.splitlines() if ln.startswith("{")]
    out = {"n": n, "dim": 384, "k": 20, "queries": queries}
    for r in rows:
        tag = "ours" if "sqlite_vector_b200" in r.get("lib", "") else "reference_avx2"
        out[tag] = {kk: r.get(kk) for kk in ("backend", "first_use_s", "quantize_s", "preload_s", "quantize_scan_ms", "full_scan_ms", "quantize_scan_ids_crc", "error") if r.get(kk) is not None}
    if "ours" in out and "reference_avx2" in out and "quantize_scan_ms" in out["ours"] and "quantize_scan_ms" in out["reference_avx2"]:
        out["same_quantize_scan_ids"] = out["ours"].get("quantize_scan_ids_crc") == out["reference_avx2"].get("quantize_scan_ids_crc")
    return out


# ------------------------------------------------------------------ BASELINE configs[3]
def run_c4(torch, a, rank, local_rank, world):
    """vector_quantize_scan cosine uint8 dim=1536 n=50M k=100 batch=256, row-sharded over the ranks (8 x B200 in BASELINE.json;
    the whole column also fits ONE B200).  A step is one batch of 256 queries; value = queries/s."""
    import torch.distributed as dist

    import sqlite_vector_b200 as vs
    from sqlite_vector_b200 import api, shard
    n, dim, k, B = a.n or 50_000_000, a.dim or 1536, a.k or 100, 256
    K, W = max(a.steps, 1), max(a.warmup, 1)
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    eng = vs.load_engine()
    for kv in a.engine_opt:
        name, val = kv.split("=")
        eng.set_option(name, int(val))
    bounds = shard.shard_bounds(n, world)
    lo, hi = bounds[rank], bounds[rank + 1]
    ix = vs.Index(api.U8, dim, hi - lo, device=local_rank, first_seq=lo)
    t0 = time.perf_counter()
    blk = 1 << 18
    for a0 in range((lo // blk) * blk, hi, blk):
        g = torch.Generator(device=device).manual_seed(SEED_CORPUS + a0 // blk)
        x = (torch.randn((blk, dim), generator=g, device=device).abs_() * 48.0).round_().clamp_(0, 255).to(torch.uint8)
        s, e = max(lo, a0) - a0, min(hi, a0 + blk) - a0
        xs = x[s:e].contiguous()
        torch.cuda.synchronize()
        ix.append_device(xs.data_ptr(), e - s)
    ix.finalize()
    g = torch.Generator(device=device).manual_seed(SEED_QUERY)
    q = (torch.randn((B, dim), generator=g, device=device).abs_() * 48.0).round_().clamp_(0, 255).to(torch.uint8).cpu().numpy()
    log(f"[rank {rank}] c4 shard rows [{lo},{hi}) resident in {time.perf_counter() - t0:.1f}s")

    exch = shard.PeerExchange(ix, eng, world, rank, bounds) if (world > 1 and a.exchange == "peer") else None

    def batch():
        if world == 1:
            r = ix.scan_topk(api.COSINE, q, k)
            return (np.stack([np.pad(x[0], (0, k - len(x[0]))) for x in r]), np.stack([np.pad(x[1], (0, k - len(x[1]))) for x in r]), np.array([len(x[0]) for x in r]))
        if exch is not None:
            return exch.batch_finish(exch.batch_submit(api.COSINE, q, k), as_arrays=True)
        return shard.sharded_batch_topk(ix, api.COSINE, q, k, bounds, device, as_arrays=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    for _ in range(W):
        rb = batch()
    if rb is None:
        raise SystemExit("the batch path refused this shard")
    barrier()
    if sampler:
        sampler.wait_first(2.0)
        sampler.mark()
    us0, rows0 = ix.stat("tc_us"), ix.stat("tc_rows")
    l0 = eng.kernel_launches()
    t0 = time.perf_counter()
    if exch is not None and a.batch_depth == 2:   # two batches in flight
        pending = None
        for _ in range(K):
            t = exch.batch_submit(api.COSINE, q, k)
            if pending is not None:
                rb = exch.batch_finish(pending, as_arrays=True)
            pending = t
        rb = exch.batch_finish(pending, as_arrays=True)
    else:
        for _ in range(K):
            rb = batch()
    barrier()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    launches = eng.kernel_launches() - l0
    tc_s = (ix.stat("tc_us") - us0) / K * 1e-6
    tc_rows = (ix.stat("tc_rows") - rows0) / K
    clocks = sampler.stop() if sampler else None
    # parity: the exact single-query CUDA-core path (the kernel the -m gpu tests pin bit-exact to the oracle) on a sample
    same = None
    if world == 1:
        eng.set_option("no_batch", 1)
        try:
            same = all(np.array_equal(ix.scan_topk(api.COSINE, q[b], k)[0][0], rb[0][b]) and np.array_equal(ix.scan_topk(api.COSINE, q[b], k)[0][1], rb[1][b]) for b in (0, 100, 255))
        finally:
            eng.set_option("no_batch", 0)
    elif exch is not None:                    # every rank takes part: the per-query exchange (k = 100: the generic filter path)
        same = True
        for b in (0, 100, 255):
            one = exch.query(api.COSINE, q[b], k, on_device=False)
            same = same and bool(np.array_equal(one[0], rb[0][b][:rb[2][b]]) and np.array_equal(one[1], rb[1][b][:rb[2][b]]))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"topk_ids": rb[0], "topk_distances": rb[1], "topk_counts": rb[2]})
    pk = peaks()
    int8_peak, int8_note = measure_int8_peak(torch, device)
    ops = 2.0 * B * tc_rows * dim
    out = {"metric": "top-k queries/sec, vector_quantize_scan cosine uint8 dim=1536 n=50M k=100 batch=256 (BASELINE configs[3])",
           "value": B * K / dt, "unit": "queries/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": dt / K * 1e3,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic |N(0,1)|*48 rounded to uint8 (seed 1234); queries seed 4321",
           "config": {"workload": f"vector_quantize_scan cosine uint8 dim={dim} n={n} k={k} batch={B}", "shards": world, "rows_per_shard": hi - lo,
                      "l2_flush": "none needed: every batch streams the whole shard (%.1f GB)" % ((hi - lo) * dim / 1e9),
                      "path": "per shard: tcgen05 (kind::i8) scoring + exact refine + slot replay" + ("" if world == 1 else (" with entry logs; logs pushed over NVLink peer memory, device-side wait, GPU merge replay; two batches in flight" if exch is not None else " with entry logs; NCCL all-gather of the logs; GPU merge replay"))},
           "e2e": {"value": B * K / dt, "unit": "queries/s", "h2d_bytes_per_step": int(q.nbytes), "d2h_bytes_per_step": int(B * 128 * 8),
                   "note": "host queries in, host top-k out: the timed call IS the public C-ABI call (vsb_scan_topk / vsb_batch_shard_scan + vsb_batch_merge)"},
           "gpu_launches": int(launches),
           "roofline": {"bound": "tensor", "kernel": "vsb::tc_scan_kernel<u8,COSINE>", "achieved": ops / tc_s / 1e12 if tc_s > 0 else None, "peak": int8_peak, "unit": "TOP/s",
                        "frac": (ops / tc_s / 1e12 / int8_peak) if (tc_s > 0 and int8_peak) else None, "peak_note": int8_note, "traffic": None,
                        "tc_kernel_ms_per_batch": tc_s * 1e3,
                        "hbm": {"achieved": tc_rows * dim / tc_s / 1e9 if tc_s > 0 else None, "peak": pk["hbm"], "unit": "GB/s",
                                "frac": (tc_rows * dim / tc_s / 1e9 / pk["hbm"]) if tc_s > 0 else None,
                                "note": "this config sits at the ridge (AI = 2B = 512 OP/B): both fractions are per GPU, rank 0's shard"}},
           "clocks": clocks, "parity": {"matches_single_query_path": same, "queries_checked": [0, 100, 255] if same is not None else None,
                                        "note": "at this size the oracle would need the 77 GB corpus on the host; tests/test_gpu_at_size.py checks the same shape bit-exact against the oracle at n = 1M"},
           "top1": [int(rb[0][0, 0]), float(rb[1][0, 0])]}
    emit(out)
    if world > 1:
        dist.destroy_process_group()
    return 0


def reference_arm(torch, a, n, dim, k, K, W, workload, cores):
    """the reference's own CPU scan on this box's host cores; each step = `cores` queries in parallel"""
    device = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    amax = corpus_absmax(torch, n, dim, 0, n, device)
    scale = float(np.float32(127.0) / np.float32(amax))
    parts = []
    for b, a0, rows in corpus_blocks(n, 0, n):
        parts.append(quantize_s8(torch, gen_block_f32(torch, b, rows, dim, device), scale).cpu().numpy())
    buf = host_quant_buffer(parts, dim)
    del parts
    q = make_queries(torch, max(8, cores), dim, scale, device).cpu().numpy()
    # bounded sample: a step is `cores` independent queries (one per host thread) over the full corpus; the run stops early
    # when the time budget is spent (stated below), it never silently changes the step
    budget_s = 150.0
    kind = "reference"
    w_done = 0
    t_w0 = time.perf_counter()
    for _ in range(W):
        _, kind = cpu_reference_run(buf, n, dim, k, q, cores, 1)
        w_done += 1
        if time.perf_counter() - t_w0 > 30.0:
            break
    t, done = 0.0, 0
    for _ in range(K):
        s, kind = cpu_reference_run(buf, n, dim, k, q, cores, 1)
        t += s
        done += 1
        if t > budget_s:
            break
    val = done * cores / t
    out = {"impl": "reference", "metric": METRIC_NAME, "value": val, "unit": "queries/s", "n_gpus": a.gpus, "steps": done, "warmup": w_done,
           "steps_requested": K, "warmup_requested": W,
           "clamp": None if done == K else f"stopped after {done} of {K} steps: the {budget_s:.0f} s budget of the CPU arm was spent (a step is {cores} full-corpus queries)",
           "ms_per_step": t / done * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int8",
           "data": "synthetic N(0,1) f32 (seed 1234) quantized to int8 with the reference S8 rule; queries seed 4321",
           "config": {"workload": workload, "metric": "L2", "k": k, "batch": 1, "rows": n, "dim": dim,
                      "step": f"{cores} independent queries, one per host thread (bounded sample of the same workload)"},
           "cpu_baseline": {"value": val, "unit": "queries/s", "cores": cores, "kind": kind, "achieved_gbs": val * n * dim / 1e9, "host": numa_info(),
                            "sample": f"{done} steps x {cores} queries over the {n}x{dim} preload buffer"},
           "e2e": {"value": val, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    emit(out)


if __name__ == "__main__":
    sys.exit(main())
