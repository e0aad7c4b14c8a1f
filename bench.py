#!/usr/bin/env python
"""Benchmark of the float_vector brute-force KNN hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W          our arm (CUDA, through the C ABI)
  python bench.py --impl reference --gpus N ...          the reference's own CPU implementation on this box's host cores

Workload at N=1 = BASELINE.json configs[1]: brute-force KNN, 10M x 768 fp32, inner product, k=10, batch of 1024 queries on one
B200.  A "step" is one batch of 1024 queries against the resident index.  For N>1 the namespace is sharded by row range, 10M rows
per GPU (weak scaling, configs[4] at N=8); every rank scans its shard for all 1024 queries and ONE C-ABI call per rank
(rxgpu_sharded_search_knn: scan, ncclAllGather, device merge) yields the global top-k; `value` counts the (query x 10M-row-shard)
scans all ranks complete per second.
Synthetic data: rows and queries from the counter-based generator in reindexer_b200/csrc/common.cuh (sigma 0.25, like the
reference's own test generator), produced directly in HBM.  Inputs are far larger than L2 (30.7 GB vs 126 MB), so no flush.

At N=1 the line also carries `sub`: driver-visible records of the other BASELINE configs -- Q=1 / Q=4 latency on the same 10M x 768
index (the >= 70 % HBM-roofline headline), config 0 (100k x 128, L2-resident), config 3 (ft_fast BM25, 50M docs) and config 2 (HNSW,
at the largest N whose reference graph build fits the time budget, labelled) -- each with its own e2e, roofline and cpu_baseline.
The reference arm (`--impl reference`, and `cpu_baseline` in our line) runs hnswlib::BruteforceSearch::SearchKnn from oracle/_ref over
the FULL 10M rows when the host has the RAM, with as many threads as the process may actually use (affinity and cgroup quota).
"""
import argparse
import concurrent.futures
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "KNN QPS @ recall@10 (10Mx768, k=10) + HBM GB/s vs roofline"
UNIT = "queries/s"
DIM, K, NQ = 768, 10, 1024
ROWS_FULL = 10_000_000
SEED = 0x5EED0001


def workload_config(world, rows):
    """identical in both arms (the driver compares them)"""
    return {"workload": "brute-force KNN, 10M x 768 fp32, inner-product, k=10, batch=1024 queries (BASELINE configs[1])"
            if world == 1 else f"brute-force KNN, {world} x 10M x 768 fp32 sharded by row range, inner-product, k=10, batch=1024, "
                               f"NCCL all-gather top-k merge (BASELINE configs[4] at N=8)",
            "rows_per_gpu": rows, "total_rows": rows * world, "dim": DIM, "k": K, "batch": NQ}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    return json.load(open(path)) if os.path.exists(path) else {}


def hbm_peak():
    p = load_peaks()
    if p.get("hbm_gbs"):
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def host_threads():
    """threads this process may really run: the affinity mask, bounded by the cgroup CPU quota (os.cpu_count() ignores both)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    why = f"affinity {n}"
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    q = max(1, int(float(txt[0]) / float(txt[1]) + 0.5))
                    if q < n:
                        n, why = q, f"cgroup quota {q}"
            else:
                quota = int(txt[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0 and max(1, quota // period) < n:
                    n, why = max(1, quota // period), f"cgroup quota {max(1, quota // period)}"
            break
        except (OSError, ValueError, IndexError):
            continue
    return max(1, n), why


def host_mem_available_gb():
    avail = None
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable:"):
                avail = int(ln.split()[1]) / 1e6
    except OSError:
        pass
    for path in ("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory/memory.limit_in_bytes"):
        try:
            txt = open(path).read().strip()
            if txt != "max":
                lim = int(txt) / 1e9
                cur = 0.0
                for cp in ("/sys/fs/cgroup/memory.current", "/sys/fs/cgroup/memory/memory.usage_in_bytes"):
                    try:
                        cur = int(open(cp).read()) / 1e9
                        break
                    except OSError:
                        continue
                avail = min(avail, lim - cur) if avail is not None else lim - cur
            break
        except (OSError, ValueError):
            continue
    return avail if avail is not None else 16.0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,"
             "enforced.power.limit")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50", "-i",
                                          str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin=None, t_end=None):
        """samples taken inside [t_begin, t_end] (the timed region); nvidia-smi is started before the warm-up so that it is
        already reporting when the region begins"""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons, watts, limit = [], [], set(), [], None
        inside = [ln for (ts, ln) in self.lines if t_begin is None or (t_begin <= ts <= t_end + 0.2)]
        window = "timed region"
        if not inside:  # region shorter than one sampling period: report the samples under the same load (warm-up + region)
            inside, window = [ln for (_, ln) in self.lines], "warm-up + timed region"
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
            try:  # board power next to its enforced limit: the filter kernel runs AT the limit (DESIGN 9), which is what bounds it
                watts.append(float(f[3]))
                limit = float(f[9]) if len(f) > 9 else limit
            except ValueError:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window,
                "power_w": float(np.median(watts)) if watts else None, "power_limit_w": limit}


# ----------------------------------------------------------------------------------------------------------------- CPU arm
class CpuReference:
    """The reference's own hnswlib::BruteforceSearch::SearchKnn (oracle/_ref, runtime ISA dispatch -> AVX-512 here) -- or the C port
    when the reference build is absent -- over `rows` rows of the workload's generator, `threads` host threads each issuing independent
    single-threaded queries against one shared index (exactly the concurrency the reference permits).  `rows` is the full 10M when the
    host has the RAM (no extrapolation); otherwise the largest row count that fits, and the QPS is scaled linearly and labelled."""

    def __init__(self, threads, rows=None, first_row=0):
        from oracle import oracle as O

        self.O = O
        self.kind = "reference" if O.ref_knn_available() else "port"
        self.threads = threads if self.kind == "reference" else 1
        need_gb = lambda r: r * (DIM * 4 + 8) / 1e9 + 4.0
        avail = host_mem_available_gb()
        if rows is None:
            rows = ROWS_FULL
            while need_gb(rows) > avail * 0.9 and rows > 250_000:
                rows //= 2
        self.rows = rows
        self.first_row = first_row
        self.isa = "scalar-c"
        t0 = time.perf_counter()
        if self.kind == "reference":
            self.bf = O.RefBF(O.IP, DIM, rows)
            self.isa = {3: "avx512", 2: "avx2", 1: "avx", 0: "sse"}[O.ref_knn_lib().ref_isa_level()]
        else:
            self.bf = O.PortBF(O.IP, DIM, rows)
        # fill in slices: the generator runs on all threads (ctypes releases the GIL), the index copies each slice in
        slice_rows = 250_000
        buf = np.empty((slice_rows, DIM), np.float32)
        fill = O.port_lib().port_synth_fill
        nthr = max(1, threads)

        def gen(lo, hi, base):
            fill(SEED, (first_row + base + lo) * DIM, (hi - lo) * DIM, buf[lo:hi].ctypes.data_as(O._f32p))

        with concurrent.futures.ThreadPoolExecutor(nthr) as pool:
            for base in range(0, rows, slice_rows):
                m = min(slice_rows, rows - base)
                step = (m + nthr - 1) // nthr
                list(pool.map(lambda lo: gen(lo, min(m, lo + step), base), range(0, m, step)))
                assert self.bf.add_batch(O.row_labels(m, first_row=first_row + base), buf[:m]) == 0
        self.fill_s = time.perf_counter() - t0

    def round(self, queries):
        t0 = time.perf_counter()
        if self.kind == "reference":
            d, l, c = self.bf.search_knn_batch(queries, K, self.threads)
        else:
            res = [self.bf.search_knn(q, K) for q in queries]
            d, l = np.stack([r[0] for r in res]), np.stack([r[1] for r in res])
        return time.perf_counter() - t0, d, l

    def describe(self, nq, rounds, secs):
        scaled = self.rows != ROWS_FULL
        qps = nq * rounds / secs * (self.rows / ROWS_FULL)
        sample = (f"{nq} queries x {rounds} round(s) over {self.rows} rows x {DIM} (the workload's generator), {self.threads} threads"
                  + ("; full row count, no extrapolation" if not scaled else
                     f"; host RAM holds only {self.rows} rows: QPS scaled linearly to {ROWS_FULL} rows (extrapolated)"))
        return {"value": qps, "unit": UNIT, "cores": self.threads, "kind": self.kind, "isa": self.isa, "sample": sample,
                "rows": self.rows, "extrapolated": scaled, "index_fill_s": round(self.fill_s, 1)}


def bench_queries(n):
    from oracle import oracle as O

    return O.synth_matrix(SEED + 1, n, DIM)


def dump_outputs(out_dir, arrays):
    """--dump-outputs: the last timed step's results as DIR/<name>.npy, so that two builds can be compared output for output.
    Integer outputs are written as float64, which holds them exactly (a label is row << 32: its significant bits are the row id's)."""
    arrays = {name: np.asarray(a).astype(np.float32 if np.asarray(a).dtype == np.float32 else np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, f"--dump-outputs: {total} bytes of outputs (limit 64 MB)"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads, why = host_threads()
    ref = CpuReference(threads)
    queries = bench_queries(NQ)
    # one step = a bounded sample of the batch: `per_step` queries (a multiple of the thread count), sized so that
    # (steps + warmup) steps stay within ~3 minutes; with --dump-outputs a fixed 64, so that the dumped queries do not depend on timing
    t_probe, _, _ = ref.round(queries[:threads])
    budget = 170.0 / max(1, args.steps + args.warmup)
    per_step = int(max(1, min(8, budget // max(t_probe, 1e-3))) * threads)
    per_step = min(per_step, NQ) if not args.dump_outputs else 64
    for w in range(args.warmup):
        ref.round(queries[(w * per_step) % NQ:][:per_step] if (w * per_step) % NQ + per_step <= NQ else queries[:per_step])
    secs = []
    for s in range(args.steps):
        lo = (s * per_step) % max(1, NQ - per_step + 1)
        dt, d, l = ref.round(queries[lo:lo + per_step])
        secs.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"distances": d, "labels": l, "query_index": np.arange(lo, lo + per_step), "rows": ref.rows})
    total = float(np.sum(secs))
    desc = ref.describe(per_step, len(secs), total)
    value = desc["value"]
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(secs),
            "warmup": args.warmup, "ms_per_step": 1000.0 * total / len(secs), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(1, ROWS_FULL),
            "step_definition": f"{per_step} queries of the 1024-query batch per step (bounded sample), every query a full scan of {ref.rows} rows",
            "cpu_baseline": {k: desc[k] for k in ("value", "unit", "cores", "kind", "sample", "isa", "rows", "extrapolated", "index_fill_s")},
            "threads_source": why,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------- GPU arm
def roofline_record(stats_sum, ms_total, rows, tc_used, qt, nlaunch_timed, scan_ms, alg_bytes, passes):
    peak, peak_src = hbm_peak()
    peaks_all = load_peaks()
    if tc_used:  # dominant kernel = the tensor-core filter: bf16 shadow rows + row norms + the resident query block, per launch
        per_launch_bytes = rows * DIM * 2 + rows * 8 + qt * DIM * 2
        kernel = {5: "knn_tc_filter_p"}.get(stats_sum.get("tc_kernel"), "knn_tc_filter_q")
    else:
        per_launch_bytes = alg_bytes / max(passes, 1)
        kernel = "knn_scan_warp"
    avg_launch_ms = scan_ms / max(nlaunch_timed, 1)
    achieved = per_launch_bytes / (avg_launch_ms * 1e-3) / 1e9 if avg_launch_ms > 0 else 0.0
    # Which roofline binds the dominant kernel: the larger of its HBM time (algorithmic bytes / measured copy peak) and its tensor
    # time (algorithmic bf16 MMA flops / measured cuBLAS rate).  The timed region is a fraction of a second, so the BURST cuBLAS
    # figure is the honest denominator (VERDICT r1); the sustained one is reported beside it.
    tensor_burst, tensor_sust = peaks_all.get("bf16_tflops"), peaks_all.get("bf16_tflops_sustained")
    tensor_src = "measured (MEASURED_PEAKS.json bf16_tflops, burst: the timed region is < 1 s)"
    if not tensor_burst:
        tensor_burst, tensor_sust, tensor_src = 1590.0, 1590.0, "fallback (B200_PROFILING.md 1.59 PFLOP/s)"
    flops_per_launch = 2.0 * rows * DIM * qt if tc_used else 0.0
    tensor_tflops = flops_per_launch / (avg_launch_ms * 1e-3) / 1e12 if tc_used and avg_launch_ms > 0 else None
    t_hbm = per_launch_bytes / (peak * 1e9)
    t_tensor = flops_per_launch / (tensor_burst * 1e12) if tc_used else 0.0
    common = {
        # dram__bytes_read.sum + dram__bytes_write.sum per launch from the ncu --set full captures under profiles/, full-size workload only
        "traffic": (None if rows != ROWS_FULL else 15.4224e9 if tc_used else 30.7201e9),
        "kernel": kernel, "bytes_per_launch": per_launch_bytes, "flops_per_launch": flops_per_launch, "avg_launch_ms": avg_launch_ms,
        "launches_timed": nlaunch_timed, "kernel_share_of_step": scan_ms / ms_total if ms_total else None,
        "hbm": {"achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src},
        "tensor": {"achieved": tensor_tflops, "peak": tensor_burst, "peak_sustained": tensor_sust, "unit": "TFLOP/s",
                   "frac": (tensor_tflops / tensor_burst) if tensor_tflops else None,
                   "frac_of_sustained": (tensor_tflops / tensor_sust) if tensor_tflops and tensor_sust else None, "peak_source": tensor_src},
    }
    if t_tensor > t_hbm:
        return {"bound": "tensor", "achieved": tensor_tflops, "peak": tensor_burst, "unit": "TFLOP/s", "frac": tensor_tflops / tensor_burst,
                "peak_source": tensor_src, **common}
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src, **common}


def sub_small_batches(idx, rx, hq, cpu, threads):
    """Q = 1 and Q = 4 on the 10M x 768 index through rxgpu_search_knn (host buffers): the reference's real API shape (one query per
    call) and the small tile the >= 70 % HBM-roofline target is defined on (SURVEY.md 8d)."""
    from reindexer_b200 import binding as B

    out = []
    peak, peak_src = hbm_peak()
    rows = idx.size()
    for q in (1, 4):
        for _ in range(3):
            idx.search_knn(hq[:q], K)
        B.lib().rxgpu_set_profile(1)
        reps, ms, nl, alg = 20, 0.0, 0, 0
        t0 = time.perf_counter()
        for r in range(reps):
            idx.search_knn(hq[r * q:(r + 1) * q], K)
            st = rx.last_search_stats()
            ms += st["scan_kernel_ms"]
            nl += st["scan_launches"]
            alg += st["algorithmic_bytes"]
        wall = (time.perf_counter() - t0) / reps
        B.lib().rxgpu_set_profile(0)
        per_launch = alg / max(nl, 1)
        ach = per_launch / (ms / max(nl, 1) * 1e-3) / 1e9
        rec = {"workload": f"brute-force KNN, 10M x 768 fp32, inner-product, k=10, {q} quer{'y' if q == 1 else 'ies'} per call "
                           f"(BASELINE configs[1] index, the reference's one-query API shape)", "metric": "latency per call", "value": wall * 1e3,
               "unit": "ms", "higher_is_better": False, "queries_per_s": q / wall,
               "e2e": {"value": q / wall, "unit": UNIT, "h2d_bytes_per_step": q * DIM * 4, "d2h_bytes_per_step": q * (K + 1) * 16 + q * 4,
                       "ms_per_call": wall * 1e3},
               "roofline": {"bound": "hbm", "kernel": "knn_scan_warp", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                            "peak_source": peak_src + " -- a copy (read + write) figure; a read-only stream can exceed it",
                            "bytes_per_launch": per_launch, "avg_launch_ms": ms / max(nl, 1), "launches_timed": nl,
                            "traffic": 30.7201e9 if rows == ROWS_FULL else None}}
        if cpu is not None:
            dt, _, _ = cpu.round(hq[:1] if cpu.kind == "reference" else hq[:1])  # ONE query on ONE thread: the reference's latency
            if cpu.kind == "reference":
                t1 = time.perf_counter()
                cpu.bf.search_knn_batch(hq[:1], K, 1)
                dt = time.perf_counter() - t1
            scale = ROWS_FULL / cpu.rows
            rec["cpu_baseline"] = {"value": dt * scale * 1e3 * 1.0, "unit": "ms per query (1 thread)", "cores": 1, "kind": cpu.kind,
                                   "sample": f"1 query over {cpu.rows} rows" + ("" if cpu.rows == ROWS_FULL else " (scaled linearly)"),
                                   "batch_qps_all_threads": None}
        out.append(rec)
    return out


def sub_config0(rx):
    """BASELINE configs[0]: 100k x 128 fp32, L2 metric, k=10, one query per call (float_vector_index_test.go shape).  The set (51 MB)
    lives in the GPU's L2: latency-bound, reported as latency next to the algorithmic bandwidth."""
    from oracle import oracle as O
    from reindexer_b200 import binding as B

    n, dim = 100_000, 128
    gpu = rx.GpuBruteforceSearch(rx.L2, dim, n)
    gpu.append_synth(0x5EED0000, 0, n)
    queries = O.synth_matrix(0x5EED0100, 256, dim)
    for i in range(5):
        gpu.search_knn(queries[i:i + 1], K)
    B.lib().rxgpu_set_profile(1)
    reps, ms, nl = 200, 0.0, 0
    t0 = time.perf_counter()
    for r in range(reps):
        d, l, c = gpu.search_knn(queries[r:r + 1], K)
        st = rx.last_search_stats()
        ms += st["scan_kernel_ms"]
        nl += st["scan_launches"]
    wall = (time.perf_counter() - t0) / reps
    B.lib().rxgpu_set_profile(0)
    peak, peak_src = hbm_peak()
    bytes_q = n * dim * 4
    rec = {"workload": "float_vector brute-force, 100k x 128 fp32, L2, k=10, 1 query per call (BASELINE configs[0])", "metric": "latency per query",
           "value": wall * 1e3, "unit": "ms", "higher_is_better": False, "queries_per_s": 1.0 / wall,
           "e2e": {"value": 1.0 / wall, "unit": UNIT, "h2d_bytes_per_step": dim * 4, "d2h_bytes_per_step": (K + 1) * 16 + 4, "ms_per_call": wall * 1e3},
           "roofline": {"bound": "latency (51 MB set is L2-resident; launch + copies dominate)", "kernel": "knn_scan_warp",
                        "achieved": bytes_q / (ms / max(nl, 1) * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": bytes_q / (ms / max(nl, 1) * 1e-3) / 1e9 / peak, "peak_source": peak_src + " (HBM figure; the data comes from L2)",
                        "avg_launch_ms": ms / max(nl, 1), "bytes_per_launch": bytes_q, "traffic": None}}
    kind = "reference" if O.ref_knn_available() else "port"
    vecs = O.synth_matrix(0x5EED0000, n, dim)
    cpu = (O.RefBF if kind == "reference" else O.PortBF)(O.L2, dim, n)
    cpu.add_batch(O.row_labels(n), vecs)
    t0 = time.perf_counter()
    same = 0
    nref = 20
    for r in range(nref):
        dr, lr = cpu.search_knn(queries[r], K)
        if r < 8:
            dg, lg, _ = gpu.search_knn(queries[r:r + 1], K)
            same += int((lg[0] == lr).all())
    cpu_s = (time.perf_counter() - t0) / nref
    rec["cpu_baseline"] = {"value": cpu_s * 1e3, "unit": "ms per query (1 thread)", "cores": 1, "kind": kind,
                           "sample": f"{nref} queries, single thread, same 100k x 128 rows"}
    rec["parity"] = f"{same}/8 queries: labels identical to the CPU reference"
    gpu.close()
    return rec


def run_ours(args):
    import torch
    import torch.distributed as dist

    import reindexer_b200 as rx
    from reindexer_b200 import binding as B
    from reindexer_b200.sharded import ShardedBruteforceSearch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if rx.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device -- librxgpu has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # the contract is ONE JSON line on stdout: NCCL announces its version on stdout when the first communicator is created, so
        # stdout points at stderr while the process group comes up
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    rows = args.rows or ROWS_FULL
    free_b, _ = torch.cuda.mem_get_info()
    if rows * DIM * 4 * 1.05 > free_b:
        raise SystemExit(f"bench.py: {rows} x {DIM} fp32 does not fit in {free_b / 1e9:.0f} GB of free HBM")

    t_fill = time.perf_counter()
    idx = rx.GpuBruteforceSearch(rx.IP, DIM, rows, device=local_rank)
    idx.append_synth(SEED, rank * rows, rows)  # shard `rank` = global rows [rank*rows, (rank+1)*rows)
    if args.query_tile:
        idx.set_query_tile(args.query_tile)
    if args.tc:
        idx.set_tensor_core_filter(args.tc)
    fill_s = time.perf_counter() - t_fill
    sharded = None
    if world > 1:
        saved_stdout = os.dup(1)  # the library's own NCCL communicator may print too
        os.dup2(2, 1)
        try:
            sharded = ShardedBruteforceSearch(idx, rows)
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    stream = torch.cuda.current_stream()
    dq = torch.empty((NQ, DIM), dtype=torch.float32, device="cuda")
    B._check(B.lib().rxgpu_synth_fill_device(dq.data_ptr(), SEED + 1, 0, NQ * DIM, local_rank, stream.cuda_stream))
    hq = dq.cpu().numpy()
    hq_pinned = torch.from_numpy(hq).pin_memory()
    k1 = K + 1
    od = torch.zeros((NQ, k1), dtype=torch.float32, device="cuda")
    oi = torch.zeros((NQ, k1), dtype=torch.int32, device="cuda")
    ol = torch.zeros((NQ, k1), dtype=torch.int64, device="cuda")
    oc = torch.zeros((NQ,), dtype=torch.int32, device="cuda")

    def step_resident():
        if sharded is not None:
            return sharded.search_knn(dq, K)
        idx.search_knn_device(NQ, dq.data_ptr(), k1, od.data_ptr(), oi.data_ptr(), ol.data_ptr(), oc.data_ptr(), stream.cuda_stream)
        return None

    def step_e2e():
        if sharded is not None:
            return sharded.search_knn(hq_pinned.numpy(), K)
        return idx.search_knn(hq, K)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident leg: CUDA events on the launching stream, max over ranks
    B.lib().rxgpu_set_profile(1)
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        step_resident()
    barrier()
    t_begin = time.perf_counter()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = passes = 0
    scan_ms = 0.0
    scan_launches = 0
    alg_bytes = 0
    tie_replays = tie_from_lists = 0
    main_stats = {}
    ev0.record(stream)
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        last = step_resident()
        st = rx.last_search_stats()
        launches += st["launches"]
        passes += st["passes"]
        scan_ms += st["scan_kernel_ms"]
        scan_launches += st["scan_launches"]
        alg_bytes += st["algorithmic_bytes"]
        tie_replays += st["tie_replays"]
        tie_from_lists += st["tie_from_lists"]
        main_stats = st  # the C call reports the shard scan's figures (kernel, tile), not the rare tie pass
    ev1.record(stream)
    barrier()
    wall_ms = (time.perf_counter() - t_wall0) * 1e3
    clocks = sampler.stop(t_begin, time.perf_counter())
    # sharded steps run on the library's stream inside one blocking C call each: the events on torch's stream bracket them through the
    # host-side ordering, so take the larger of the event time and the host clock around the same region
    ms_total = max(ev0.elapsed_time(ev1), wall_ms if sharded is not None else 0.0)
    B.lib().rxgpu_set_profile(0)
    if args.dump_outputs and rank == 0:
        if sharded is not None:
            d_out, l_out, c_out = last
        else:  # the device call fills k + 1 columns per query
            d_out, l_out, c_out = od.cpu().numpy(), ol.cpu().numpy().view(np.uint64), oc.cpu().numpy()
        dump_outputs(args.dump_outputs, {"distances": d_out, "labels": l_out, "counts": c_out})
    qt, tc_used = main_stats["query_tile"], main_stats["tc_used"]
    # ---- end-to-end leg: host buffers through the reference-facing C ABI call, copies inside the timed region
    for _ in range(min(args.warmup, 1)):
        res = step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = step_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_stats = rx.last_search_stats()
    if world > 1:
        t = torch.tensor([ms_total, e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, e2e_s = float(t[0]), float(t[1])
        tot = torch.tensor([launches], dtype=torch.int64, device="cuda")
        dist.all_reduce(tot)
        launches_all = int(tot[0])
    else:
        launches_all = launches

    # sanity on the timed work: every query of the last batch got k results, sorted
    d_chk, l_chk, c_chk = res
    assert (np.asarray(c_chk) == K).all() and (np.diff(d_chk[:, :K], axis=1) >= 0).all()
    # the timed path against the exact fp32 scan of the same index / shards (outside the timed regions): identical labels and bits
    nchk = 8
    if world == 1:
        idx.set_tensor_core_filter(2)
        d_ex, l_ex, _ = idx.search_knn(hq[:nchk], K)
    else:
        idx.set_tensor_core_filter(2)
        d_ex, l_ex, _ = sharded.search_knn(hq[:nchk], K)
    idx.set_tensor_core_filter(args.tc or 0)
    assert (np.asarray(l_ex) == np.asarray(l_chk)[:nchk, :K]).all() and \
        (np.asarray(d_ex).view(np.uint32) == np.asarray(d_chk)[:nchk, :K].view(np.uint32)).all(), "timed path differs from the exact scan"

    if rank == 0:
        ms_per_step = ms_total / args.steps
        value = world * NQ / (ms_per_step / 1000.0)
        e2e_value = world * NQ / (e2e_s / args.steps)
        roofline = roofline_record(main_stats, ms_total, rows, tc_used, qt, scan_launches, scan_ms, alg_bytes, passes)
        kernel_name = {5: "knn_tc_filter_p (tcgen05 cta_group::2 bf16 filter: CTA pairs, queries in TMEM, half a row tile per SM, certified bound) + knn_rerank (exact fp32)",
                       2: "knn_tc_filter_q (tcgen05 bf16 filter, queries in TMEM, certified bound) + knn_rerank (exact fp32)",
                       1: "knn_tc_filter (tcgen05 bf16 filter, queries in shared memory) + knn_rerank (exact fp32)"}.get(
            main_stats.get("tc_kernel") if tc_used else 0, "knn_scan_warp (fp32 FMA, fused top-k)")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": workload_config(world, rows),
            "details": {"query_tile": qt, "kernel": kernel_name, "tc_candidates_per_step": main_stats["tc_candidates"],
                        "tc_fallbacks": main_stats["tc_fallbacks"], "tc_cluster": main_stats["tc_cluster"],
                        "tail_grid": "clusters of 4 fit 33 times (132 of 148 SMs); 2-CTA clusters of the same kernel scan the last ~10 % of the "
                                     "row tiles on the other 16 SMs beside every main launch (second stream); roofline.avg_launch_ms is the main "
                                     "launch, whose window covers all rows for its 512 queries",
                        "l2_policy": "inputs (30.7 GB/GPU) larger than L2, no flush",
                        "global_queries_per_s": NQ / (ms_per_step / 1000.0), "index_fill_s": round(fill_s, 2),
                        "value_definition": "(query x 10M-row shard) scans per second over all ranks",
                        "tie_replays_timed": tie_replays, "tie_replays_from_candidate_lists": tie_from_lists,
                        "self_check": f"{nchk} queries of the timed batch re-run on the fp32 exact-scan path"
                                      f"{' of all shards' if world > 1 else ''}: identical labels and distance bits"},
            "roofline": roofline,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": NQ * DIM * 4,
                    "d2h_bytes_per_step": NQ * K * 12 + NQ * 4 if world == 1 else NQ * K * 20 + NQ * 5, "ms_per_step": 1000.0 * e2e_s / args.steps,
                    "tie_replays": e2e_stats["tie_replays"]},
            "gpu_launches": launches_all,
            "clocks": clocks,
        }
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            threads, why = host_threads()
            cpu = CpuReference(threads)
            nq_cpu = min(NQ, max(threads, 8))
            secs, d_ref, l_ref = cpu.round(hq[:nq_cpu])
            cb = cpu.describe(nq_cpu, 1, secs)
            cb["threads_source"] = why
            line["cpu_baseline"] = cb
            # recall@10 of what was timed, against the reference's own brute force on the same rows and queries
            if cpu.rows == rows:
                hits = sum(len(set(l_ref[i].tolist()) & set(np.asarray(l_chk)[i, :K].tolist())) for i in range(nq_cpu))
                line["details"]["recall_at_10"] = hits / (nq_cpu * K)
                line["details"]["recall_basis"] = f"{nq_cpu} queries of the timed batch vs oracle/_ref BruteforceSearch over the same {rows} rows"
            else:
                line["details"]["recall_at_10"] = None
                line["details"]["recall_basis"] = "host RAM too small for the full row set: only the exact-scan self-check above"
        else:
            line["details"]["recall_at_10"] = None
            line["details"]["recall_basis"] = "exact search by construction; see self_check (no CPU arm in this run)"
        if world == 1 and not args.no_sub and rows == ROWS_FULL:
            sub = []
            t_sub = time.perf_counter()
            try:
                sub += sub_small_batches(idx, rx, hq, cpu, 1)
                sub.append(sub_config0(rx))
                del cpu
                idx.close()  # the BM25 / HNSW records need their own HBM and host RAM
                import bench_extra as X

                threads, _ = host_threads()
                sub.append(X.ft_record(50_000_000 if not args.quick_sub else 2_000_000))
                hn = int(min(150_000, max(20_000, threads * 9000))) if not args.quick_sub else 20_000  # ~40 s of reference graph build
                sub.append(X.hnsw_record(hn, 4096, threads))
            except Exception as e:  # a sub-record must never take the headline down with it
                sub.append({"error": f"{type(e).__name__}: {e}"})
            line["sub"] = sub
            line["sub_seconds"] = round(time.perf_counter() - t_sub, 1)
    if world > 1 and not args.no_sub and rows == ROWS_FULL:
        # config 3 over docid-range shards: a collective, so every rank takes part; rank 0 reports it
        rec = None
        try:
            idx.close()
            import bench_extra as X

            rec = X.ft_sharded_record(sharded.comm, rank, world, 50_000_000 if not args.quick_sub else 2_000_000, local_rank)
        except Exception as e:  # a sub-record must never take the headline down with it
            rec = {"error": f"{type(e).__name__}: {e}"}
        if rank == 0:
            line["sub"] = [rec]
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=0, help="rows per GPU (default 10M = BASELINE config)")
    ap.add_argument("--query-tile", type=int, default=0)
    ap.add_argument("--tc", type=int, default=0, help="tensor-core filter: 0 auto, 1 on, 2 off (exact fp32 scan only), 3..6, 9, 14..16 kernel variants")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the sub-records of the other BASELINE configs")
    ap.add_argument("--quick-sub", action="store_true", help="small sub-record sizes (smoke)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step as DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
