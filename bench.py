#!/usr/bin/env python
"""bench.py — filtered-scan throughput of the HBM-resident liquid cache (BASELINE.json metric).

Workload (BASELINE.json configs[1], SURVEY.md §8d row 2): ClickBench `hits` URL column, 100 M rows as 12 208
entries of 8192 rows (FSST + u16 dictionary + fingerprints), predicate `URL LIKE '%google%'` over ALL entries,
then `get().with_selection(mask)` of the matching rows. One "step" = one such pass over every entry.

  value   device-resident pass: the liquid columns and the running selection stay in HBM (lc_scan_* pipeline),
          timed with CUDA events on the launching stream; Mrows/s over all ranks
  e2e     the same pass through the reference-facing C ABI with HOST buffers: lc_eval_predicate_many writes the
          masks into host memory, the harness picks the entries with hits (as LiquidCacheReader does) and
          lc_to_arrow_many returns the filtered Arrow array on the host; H2D/D2H copies inside the timed region
  roofline  k_str_scan (the dominant kernel): algorithmic bytes per launch / CUDA-event time of that launch
  cpu_baseline  the C port of the reference's CPU path (oracle/c) on a bounded sample, all host cores

`--impl reference` times the CPU port as the measured arm (the reference itself is Rust and cannot be built here).
Launch: python bench.py --gpus N --steps K --warmup W   (N>1: torchrun, one rank per GPU, entries sharded by EntryID).
"""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ROWS_PER_ENTRY = 8192
PATTERN = "%google%"
METRIC = "filtered-scan Mrows/s (URL LIKE '%google%' + get-with-selection, hot cache)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)  # a step is ~0.5 ms: 100 keep one host hiccup from deciding the mean
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--rows", type=int, default=100_000_000, help="rows PER GPU (weak scaling)")
    ap.add_argument("--cpu-sample-entries", type=int, default=0,
                    help="entries per CPU-arm pass; 0 = max(8192, 64 per host thread), bounded by the workload")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--url-source", choices=["synthetic", "sample"], default="synthetic",
                    help="url_like: the synthetic URL generator, or URLs resampled from the reference's ClickBench sample")
    ap.add_argument("--no-secondary", action="store_true", help="url_like at one GPU: skip the configs[2] / configs[3] runs that are "
                                                               "reported under config.secondary")
    ap.add_argument("--workload", choices=["url_like", "int_filter", "shipdate", "clickbench_sweep", "squeeze", "insert"], default="url_like",
                    help="url_like = BASELINE configs[1] (the bench line the driver records); int_filter = configs[2]; "
                         "shipdate = configs[3] (TPC-H SF100 l_shipdate range, one GPU's shard of the 8-way split per rank); "
                         "clickbench_sweep = configs[4] (scan stage of the 43 ClickBench queries, bench_sweep.py)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="url_like: after the timed steps, write the filtered URLs the last step returned as DIR/url_*.npy, so that "
                         "two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "url_like" or args.impl != "ours"):
        ap.error("--dump-outputs is written by --workload url_like --impl ours")
    return args


DUMP_BYTES = 64 << 20


def dump_strings(out_dir: str, name: str, arr):
    """The Utf8 array `arr` as <name>_offsets.npy (float64, from 0) and <name>_bytes.npy (float32, the UTF-8 bytes), both exact,
    with <name>_rows.npy (float64) the positions of the rows written: all of them, or when that would take more than
    DUMP_BYTES, a sample of rows fixed by seed 0 and the row lengths, in row order."""
    import numpy as np
    import pyarrow as pa

    def offsets(a):
        return np.frombuffer(a.buffers()[1], dtype=np.int32)[a.offset:a.offset + len(a) + 1].astype(np.int64)

    lens = np.diff(offsets(arr))
    order = np.random.default_rng(0).permutation(len(arr))
    # 8 + 8 + 4 * len bytes per row; the last offset and the three .npy headers fit in 1 KB
    fits = int(np.searchsorted(np.cumsum(16 + 4 * lens[order]), DUMP_BYTES - 1024, side="right"))
    rows = np.arange(len(arr)) if fits == len(arr) else np.sort(order[:fits])
    if fits < len(arr):
        arr = arr.take(pa.array(rows))
    offs = offsets(arr)
    data = np.frombuffer(arr.buffers()[2] or b"", dtype=np.uint8)[offs[0]:offs[-1]]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"{name}_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, f"{name}_offsets.npy"), (offs - offs[0]).astype(np.float64))
    np.save(os.path.join(out_dir, f"{name}_bytes.npy"), data.astype(np.float32))


def recorded_traffic(rows: int, entries: int):
    """DRAM bytes (read + write) of one k_str_like launch, REPLAYED from the committed `ncu --set full` capture of this
    exact seeded workload (profiles/r02_k_str_like_traffic.json) — not measured in this run; None when the shape differs
    or the file is absent. A number taken under the profiler is only ever used for this field, never for a timing."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_k_str_like_traffic.json")) as f:
            t = json.load(f)
        if t["workload"]["rows"] == rows and t["workload"]["entries"] == entries:
            return int(t["dram__bytes_read.sum"]) + int(t["dram__bytes_write.sum"])
    except (OSError, KeyError, ValueError):
        pass
    return None


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md; MEASURED_PEAKS.json absent)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        if os.environ.get("LC_BENCH_NO_CLOCKS") == "1":  # diagnosis only: is the sampler perturbing the steps?
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            # the sampler must be up and running BEFORE the clock starts: nvidia-smi's start-up (NVML initialisation, its
            # first device queries) takes driver locks that CUDA calls wait behind — with 20 steps of 0.16 ms in the timed
            # region, one such stall (9.5 ms was measured) is three times the region
            t_end = time.perf_counter() + 3.0
            while not self.rows and time.perf_counter() < t_end and self.proc.poll() is None:
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for i, nm in enumerate(names):
                if len(r) > 3 + i and r[3 + i].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def pin_to_gpu_numa(local_rank: int):
    """Run this rank (and the library's host threads it spawns) on the CPUs of its GPU's NUMA node: the readbacks of a
    step land in that node's memory (VERDICT r1: 8 unpinned ranks, GPU4-7 on node 1). Returns what was done for the record."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        n_words = ((os.cpu_count() or 1) + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {i for i in range(os.cpu_count() or 1) if (int(mask[i // 64]) >> (i % 64)) & 1}
        allowed = os.sched_getaffinity(0)
        want = cpus & allowed
        if want:
            os.sched_setaffinity(0, want)
            return {"pinned_cpus": len(want), "first": min(want), "last": max(want)}
    except Exception as e:  # no NVML / not permitted: run unpinned
        return {"pinned_cpus": 0, "why": str(e)[:80]}
    return {"pinned_cpus": 0}


def generate_entries(first: int, count: int, workers: int, source: str = "synthetic"):
    """Yield (entry_index, pyarrow URL batch) in order, generated by a thread pool (the C generator drops the GIL)."""
    import synth

    if source == "sample":
        from synth.hits import HitsSample

        sample = HitsSample()
        for g0 in range(first, first + count, 256):
            nb = min(256, first + count - g0)
            for k, arr in enumerate(sample.batches(["URL"], g0, nb)["URL"]):
                yield g0 + k, arr
        return

    synth.lib().lcs_init(synth.URL_POOL)
    with cf.ThreadPoolExecutor(max_workers=workers) as ex:
        window = workers * 4
        futs = {}
        nxt = first
        end = first + count
        for i in range(first, min(end, first + window)):
            futs[i] = ex.submit(synth.url_entry, i)
            nxt = i + 1
        for i in range(first, end):
            arr = futs.pop(i).result()
            if nxt < end:
                futs[nxt] = ex.submit(synth.url_entry, nxt)
                nxt += 1
            yield i, arr


def cpu_sample_entries(args, threads: int, cap: int) -> int:
    import bench_cpu

    return min(cap, args.cpu_sample_entries) if args.cpu_sample_entries > 0 else bench_cpu.default_sample_entries(threads, cap)


def cpu_baseline(sample_entries: int, threads: int, target_s: float = 8.0):
    """C port of the reference's CPU path (oracle/c) on a persistent thread pool: LIKE over every sampled entry + get of
    the hits (bench_cpu.py says how the arm is driven and why)."""
    import bench_cpu

    return bench_cpu.cpu_baseline_line("url_like", sample_entries, threads, target_s=target_s)


def shipdate_params():
    import datetime as dt

    d0 = dt.date(1970, 1, 1)
    return {"lo_days": (dt.date(1994, 1, 1) - d0).days, "hi_days": (dt.date(1995, 1, 1) - d0).days}


def int_filter_params(first_entry: int = 0):
    import synth

    return {"lo": 1373832014 + 20000, "hi": 1373832014 + 28640,  # 10 % of the 86 400 s window
            "uid": int(synth.int_entry("UserID", first_entry)[17].as_py())}


REFERENCE_WORKLOADS = {
    "url_like": ("clickbench-hits URL LIKE '%google%' + get-with-selection (configs[1])", "u8", METRIC, 100_000_000),
    "shipdate": ("TPC-H SF100 lineitem l_shipdate range + get of the survivors (configs[3])", "int32",
                 METRIC.replace("URL LIKE '%google%'", "l_shipdate range"), 600_037_902 // 8),
    "int_filter": ("clickbench-hits EventTime>=lo AND EventTime<hi AND UserID=k, then get(UserID, EventTime) (configs[2])", "int64",
                   METRIC.replace("URL LIKE '%google%'", "EventTime range AND UserID ="), 100_000_000),
}


def run_reference(args, rank: int, world: int):
    """--impl reference: the reference's CPU implementation of the path (its C port; no Rust toolchain here) on the host
    cores — one step = one pass over a bounded sample of the workload on a persistent pool of all host threads."""
    if rank != 0:
        return
    import bench_cpu

    if args.workload not in REFERENCE_WORKLOADS:
        print(json.dumps({"impl": "reference", "unavailable": f"no CPU arm for workload {args.workload}"}))
        return
    name, dtype, metric, rows_cap = REFERENCE_WORKLOADS[args.workload]
    threads, _host = bench_cpu.usable_cpus()
    steps = max(1, args.steps)
    n = cpu_sample_entries(args, threads, max(1, min(args.rows, rows_cap) // ROWS_PER_ENTRY))
    params = {"url_like": lambda: None, "shipdate": shipdate_params, "int_filter": int_filter_params}[args.workload]()
    arm = bench_cpu.CpuArm(args.workload, n, threads, params=params)
    try:
        single = arm.single_thread_mrows()
        for _ in range(max(3, args.warmup)):
            arm.one_pass()
        t0 = time.perf_counter()
        rows = 0
        matched = 0
        for _ in range(steps):
            matched, r = arm.one_pass()
            rows += r
        dt = time.perf_counter() - t0
        val = rows / dt / 1e6
        sample = (f"{n} entries x {ROWS_PER_ENTRY} rows per step (bounded sample of one GPU's shard of the workload), {matched} rows "
                  f"matched per step; C port of the reference's CPU path (oracle/c/lc_oracle.c), persistent pool of {threads} threads")
        base = {"value": val, "unit": "Mrows/s", "cores": threads, "kind": "port", "sample": sample}
        base.update(arm.describe(single, val))
    finally:
        arm.close()
    print(json.dumps({
        "impl": "reference", "metric": metric, "value": val, "unit": "Mrows/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": max(3, args.warmup), "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": dtype, "data": "synthetic",
        "config": {"workload": name, "rows_per_step": rows // steps, "rows_per_entry": ROWS_PER_ENTRY,
                   "same_config": "same generator, seeds, predicate and per-batch reader loop as the GPU arm; a bounded sample of its rows"},
        "cpu_baseline": base,
        "e2e": {"value": val, "unit": "Mrows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def run_int_filter(args, rank, world, local_rank, emit=True):
    """BASELINE configs[2]: EventTime range (two conjuncts) AND UserID equality on bit-packed Int64 columns, then
    get-with-selection of both columns. Secondary workload: its own JSON line when run by itself, an object under
    `config.secondary` of the driver's bench line otherwise."""
    import numpy as np
    import pyarrow as pa
    import torch

    import synth
    from liquid_cache_b200 import BinaryExpr, Column, LiquidCacheBuilder, LiquidExpr, Literal, parquet_array_id

    torch.cuda.set_device(local_rank)
    cache = LiquidCacheBuilder.new().with_device(local_rank).build()
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    cache.set_stream(stream.cuda_stream)
    n_entries = max(1, args.rows // ROWS_PER_ENTRY)
    ids_t, ids_u = [], []
    for i in range(n_entries):
        et = parquet_array_id(0, i // 32, 4, i % 32)
        ui = parquet_array_id(0, i // 32, 9, i % 32)
        cache.insert(et, synth.int_entry("EventTime", rank * n_entries + i)).run()
        cache.insert(ui, synth.int_entry("UserID", rank * n_entries + i)).run()
        ids_t.append(int(et))
        ids_u.append(int(ui))
    h_t, h_u = cache.handles(ids_t), cache.handles(ids_u)
    rows_local = n_entries * ROWS_PER_ENTRY
    lo, hi = 1373832014 + 20000, 1373832014 + 28640  # 10 % of the 86 400 s window
    uid = int(synth.int_entry("UserID", rank * n_entries)[17].as_py())

    def native(op, v):
        return LiquidExpr.new_unchecked(BinaryExpr(Column("c", 0), op, Literal(v))).to_native(pa.int64())

    p_ge, p_lt, p_eq = native(">=", lo), native("<", hi), native("=", uid)
    scan = cache.scan(np.full(n_entries, ROWS_PER_ENTRY, dtype=np.uint64))
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    k_ms = [[], [], []]

    cache.kernel_timing(True)

    def step(timed):
        scan.reset()
        scan.filter_native(h_t, p_ge)
        if timed:
            k_ms[0].append(cache.last_kernel_ms())
        scan.filter_native(h_t, p_lt)
        if timed:
            k_ms[1].append(cache.last_kernel_ms())
        scan.filter_native(h_u, p_eq)
        if timed:
            k_ms[2].append(cache.last_kernel_ms())
        a = scan.read(h_u)
        b = scan.read(h_t)
        return len(a), a, b

    for _ in range(max(3, args.warmup)):
        step(False)
    torch.cuda.synchronize()
    st_a = cache.stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        total, a, b = step(True)
    e1.record(stream)
    torch.cuda.synchronize()
    st_b = cache.stats()
    ms = e0.elapsed_time(e1)
    peak, peak_src = measured_peak_gbs()
    # algorithmic bytes per launch: packed words + selection in (dense first conjunct: none) + selection out
    w_t, w_u = 17, 64
    b_ge = rows_local * w_t // 8 + rows_local // 8
    b_lt = rows_local * w_t // 8 + 2 * (rows_local // 8)
    b_eq = rows_local * w_u // 8 + 2 * (rows_local // 8)
    med = lambda x: float(np.median(x))  # noqa: E731
    line = {
        "metric": METRIC.replace("URL LIKE '%google%'", "EventTime range AND UserID ="), "value": rows_local * args.steps / (ms / 1e3) / 1e6,
        "unit": "Mrows/s", "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": "clickbench-hits EventTime>=lo AND EventTime<hi AND UserID=k, then get(UserID, EventTime) (BASELINE configs[2])",
                   "rows_per_gpu": rows_local, "entries_per_gpu": n_entries, "matching_rows": int(total),
                   "liquid_bytes_per_gpu": int(cache.stats().hbm_bytes_used)},
        "gpu_launches": int(st_b.kernel_launches - st_a.kernel_launches),
        "roofline": [
            {"kernel": "k_int_bits<REFINE> EventTime>=lo (W=17, dense selection in)", "bound": "hbm", "achieved": b_ge / (med(k_ms[0]) / 1e3) / 1e9, "peak": peak,
             "unit": "GB/s", "frac": b_ge / (med(k_ms[0]) / 1e3) / 1e9 / peak, "kernel_ms": med(k_ms[0]), "algorithmic_bytes_per_launch": b_ge},
            {"kernel": "k_int_bits<REFINE> EventTime<hi (W=17, selection in+out)", "bound": "hbm", "achieved": b_lt / (med(k_ms[1]) / 1e3) / 1e9, "peak": peak,
             "unit": "GB/s", "frac": b_lt / (med(k_ms[1]) / 1e3) / 1e9 / peak, "kernel_ms": med(k_ms[1]), "algorithmic_bytes_per_launch": b_lt},
            {"kernel": "k_int_scan<REFINE> UserID=k (W=64)", "bound": "hbm", "achieved": b_eq / (med(k_ms[2]) / 1e3) / 1e9, "peak": peak,
             "unit": "GB/s", "frac": b_eq / (med(k_ms[2]) / 1e3) / 1e9 / peak, "kernel_ms": med(k_ms[2]), "algorithmic_bytes_per_launch": b_eq},
        ],
        "peak_source": peak_src,
    }
    # e2e: the same step through the public scan API by the host's clock (predicate literals go up, the two filtered Arrow
    # arrays come down every step); the device-timed `value` above uses CUDA events around the same calls
    torch.cuda.synchronize()
    st_c = cache.stats()
    t0 = time.perf_counter()
    e2e_steps = max(3, args.steps // 2)
    for _ in range(e2e_steps):
        total, a, b = step(False)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    st_d = cache.stats()
    line["e2e"] = {"value": rows_local / (e2e_ms / 1e3) / 1e6, "unit": "Mrows/s", "ms_per_step": e2e_ms,
                   "h2d_bytes_per_step": int((st_d.h2d_bytes - st_c.h2d_bytes) / e2e_steps),
                   "d2h_bytes_per_step": int((st_d.d2h_bytes - st_c.d2h_bytes) / e2e_steps),
                   "note": "lc_scan_filter x3 + lc_scan_read x2 (host Arrow results), wall clock"}
    if not args.no_cpu_baseline:
        import bench_cpu

        cpu_threads, _h = bench_cpu.usable_cpus()
        line["cpu_baseline"] = bench_cpu.cpu_baseline_line("int_filter", cpu_sample_entries(args, cpu_threads, n_entries), cpu_threads,
                                                           params=int_filter_params(), target_s=6.0)
    if emit:
        print(json.dumps(line))
    scan.close()
    cache.close()
    return line


def run_squeeze(args, rank, world, local_rank):
    """SURVEY §8f-4: `UserID = k` over the UserID column (Int64, W = 64) with every entry SQUEEZED to half-width codes
    (IntegerSqueezePolicy::Quantize, the reference's default: 32-bit bucket indices, full LQDA images in host memory behind
    the read callback), through lc_eval_predicate_many — against the same call over the full entries. Reports rows/s of
    both, HBM bytes of both, and how many entries had to read their backing. Secondary workload: prints its own JSON line."""
    import numpy as np
    import pyarrow as pa
    import torch

    import synth
    from liquid_cache_b200 import BinaryExpr, CacheExpression, Column, EntryID, LiquidCacheBuilder, LiquidExpr, Literal, parquet_array_id

    torch.cuda.set_device(local_rank)
    cache = LiquidCacheBuilder.new().with_device(local_rank).build()
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    cache.set_stream(stream.cuda_stream)
    n_entries = max(1, args.rows // ROWS_PER_ENTRY)
    ids = [parquet_array_id(0, i // 32, 9, i % 32) for i in range(n_entries)]
    for g0 in range(0, n_entries, 1024):
        part = range(g0, min(n_entries, g0 + 1024))
        cache.insert_many([EntryID(int(ids[i])) for i in part], [synth.int_entry("UserID", rank * n_entries + i) for i in part])
    hbm_full = int(cache.stats().hbm_bytes_used)

    class Store:  # the "disk": one image per entry in host memory
        def __init__(self):
            self.image, self.reads = b"", 0

        def read(self, rng):
            self.reads += 1
            return self.image[rng[0]:rng[1]]

    policy = os.environ.get("LC_SQUEEZE_POLICY", "quantize")
    t0 = time.perf_counter()
    full, squeezed, stores = [], [], []
    for i in range(n_entries):
        la = cache.try_read_liquid(EntryID(int(ids[i])))
        st = Store()
        sq, st.image = la.squeeze(st, CacheExpression.PredicateColumn, policy)
        full.append(la)
        squeezed.append(sq)
        stores.append(st)
    squeeze_s = time.perf_counter() - t0
    hbm_both = int(cache.stats().hbm_bytes_used)
    h_full = np.array([a.handle for a in full], dtype=np.uint64)
    h_sq = np.array([a.handle for a in squeezed], dtype=np.uint64)
    rows = np.full(n_entries, ROWS_PER_ENTRY, dtype=np.uint64)
    rows_local = n_entries * ROWS_PER_ENTRY
    uid = int(synth.int_entry("UserID", rank * n_entries)[17].as_py())
    pred = LiquidExpr.new_unchecked(BinaryExpr(Column("c", 0), "=", Literal(uid))).to_native(pa.int64())
    out = None

    def step(handles):
        nonlocal out
        out = cache._eval_many_native(handles, rows, pred, None, out)
        return int(out[5].sum())

    def timed(handles):
        for _ in range(max(3, args.warmup)):
            step(handles)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            hits = step(handles)
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps, hits

    ms_full, hits_full = timed(h_full)
    for st in stores:
        st.reads = 0
    ms_sq, hits_sq = timed(h_sq)
    reads = sum(st.reads for st in stores) / (args.steps + max(3, args.warmup))
    # the device-resident pipeline (selection stays in HBM, only the survivor counts come back): lc_scan_filter
    scan = cache.scan(rows)

    def scan_step(handles):
        scan.reset()
        scan.filter_native(handles, pred)
        return int(scan.counts()[1])

    def scan_timed(handles):
        for _ in range(max(3, args.warmup)):
            scan_step(handles)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            hits = scan_step(handles)
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps, hits

    scan_ms_full, scan_hits_full = scan_timed(h_full)
    scan_ms_sq, scan_hits_sq = scan_timed(h_sq)
    scan.close()
    peak, peak_src = measured_peak_gbs()
    width = squeezed[0].bit_width()
    line = {
        "metric": METRIC.replace("URL LIKE '%google%'", "UserID = k on squeezed entries"), "value": rows_local / (scan_ms_sq / 1e3) / 1e6, "unit": "Mrows/s",
        "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": scan_ms_sq, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": f"clickbench-hits UserID = k through lc_eval_predicate_many, entries squeezed ({policy}) to {width}-bit codes (SURVEY 8f-4)",
                   "rows_per_gpu": rows_local, "entries_per_gpu": n_entries, "matching_rows": hits_sq, "matches_full_entries": hits_sq == hits_full,
                   "matches_full_entries_scan": scan_hits_sq == scan_hits_full == hits_full,
                   "full_entries": {"scan_Mrows_per_s": rows_local / (scan_ms_full / 1e3) / 1e6, "scan_ms_per_step": scan_ms_full,
                                    "eval_many_Mrows_per_s": rows_local / (ms_full / 1e3) / 1e6, "eval_many_ms_per_step": ms_full, "hbm_bytes": hbm_full},
                   "squeezed_hbm_bytes": hbm_both - hbm_full, "backing_reads_per_step": reads, "backing_bytes_host": sum(len(st.image) for st in stores),
                   "squeeze_seconds": squeeze_s,
                   "note": "value: lc_scan_filter (selection stays in HBM, counts come back); e2e: lc_eval_predicate_many (masks to host buffers)"},
        "e2e": {"value": rows_local / (ms_sq / 1e3) / 1e6, "unit": "Mrows/s", "ms_per_step": ms_sq},
        "roofline": {"bound": "hbm", "kernel": "lc_scan_filter over squeezed entries (whole call)", "achieved": rows_local * width / 8 / (scan_ms_sq / 1e3) / 1e9,
                     "peak": peak, "unit": "GB/s", "frac": rows_local * width / 8 / (scan_ms_sq / 1e3) / 1e9 / peak, "peak_source": peak_src},
    }
    print(json.dumps(line))
    cache.close()


def run_shipdate(args, rank, world, local_rank, emit=True):
    """BASELINE configs[3]: TPC-H SF100 lineitem `l_shipdate >= 1994-01-01 AND l_shipdate < 1995-01-01` (q6's date
    range; Date32, W = 12), entries sharded across 8 B200: every rank holds one eighth of the 600 037 902 rows
    (weak scaling: at --gpus 8 the job is the whole table). Step = both conjuncts over every entry + get-with-selection
    of the survivors (~14 %). value: device-resident (result left in HBM); e2e: the same pipeline with the filtered
    Arrow array copied to the host every step. Secondary workload: prints its own JSON line."""
    import datetime as dt

    import numpy as np
    import pyarrow as pa
    import torch
    import torch.distributed as dist

    import synth
    from liquid_cache_b200 import BinaryExpr, Column, LiquidCacheBuilder, LiquidExpr, Literal, parquet_array_id

    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    cache = LiquidCacheBuilder.new().with_device(local_rank).build()
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    cache.set_stream(stream.cuda_stream)
    rows_shard = 600_037_902 // 8 if args.rows == 100_000_000 else args.rows
    n_entries = max(1, rows_shard // ROWS_PER_ENTRY)
    ids = []
    t_setup = time.perf_counter()
    insert_s, group = 0.0, 1024  # row-group sized lists: one lc_cache_insert_many call per 1024 batches
    for g0 in range(0, n_entries, group):
        idx = range(g0, min(n_entries, g0 + group))
        eids = [parquet_array_id(1, i // 32, 10, i % 32) for i in idx]  # l_shipdate is column 10 of lineitem
        batches = [synth.int_entry("l_shipdate", rank * n_entries + i, seed=synth.SEED_TPCH) for i in idx]
        t_i = time.perf_counter()
        cache.insert_many(eids, batches)
        insert_s += time.perf_counter() - t_i
        ids.extend(int(e) for e in eids)
    setup_s = time.perf_counter() - t_setup
    handles = cache.handles(ids)
    rows_local = n_entries * ROWS_PER_ENTRY
    lo, hi = dt.date(1994, 1, 1), dt.date(1995, 1, 1)

    def native(op, v):
        return LiquidExpr.new_unchecked(BinaryExpr(Column("l_shipdate", 0), op, Literal(v))).to_native(pa.date32())

    p_ge, p_lt = native(">=", lo), native("<", hi)
    scan = cache.scan(np.full(n_entries, ROWS_PER_ENTRY, dtype=np.uint64))
    dev = torch.device("cuda", local_rank)
    k_ms = [[], []]
    cache.kernel_timing(True)

    from liquid_cache_b200.dist import DeviceGather

    pin = pin_to_gpu_numa(local_rank)
    gather = DeviceGather(pa.date32(), rank, world, dev, rows_cap=rows_local // 4)

    def filters(timed):
        scan.reset()
        scan.filter_native(handles, p_ge)
        if timed:
            k_ms[0].append(cache.last_kernel_ms())
        scan.filter_native(handles, p_lt)
        if timed:
            k_ms[1].append(cache.last_kernel_ms())

    def step(timed):
        """Both conjuncts over every entry of this rank, then get-with-selection of the survivors as Arrow-layout buffers in
        HBM (lc_scan_read_async writes straight into this rank's gather slot); at N > 1 ONE NCCL all_gather — the one exchange
        of the path — delivers every rank's batch into rank 0's HBM. One host synchronisation per step (the 64-byte headers)."""
        for _ in range(16):
            filters(timed)
            if not scan.read_async(handles, *gather.addresses()):
                raise RuntimeError("l_shipdate must be readable by the device-planned path")
            hdrs = gather.exchange()
            if not gather.overflowed():
                return hdrs
            gather.grow()
        raise RuntimeError("gather slot capacities did not settle")

    def e2e_step():
        """The same filters, the result as a HOST Arrow array on every rank (lc_scan_read: one synchronisation, the download
        inside it) — what a reference-side caller holding host buffers gets."""
        filters(False)
        return scan.read(handles)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        hdrs = step(False)
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    for _ in range(3):  # back to the steady state after the sampler's start-up
        hdrs = step(False)
    barrier()
    st_a = cache.stats()
    grows_before = gather.grows
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        hdrs = step(True)
    e1.record(stream)
    barrier()
    st_b = cache.stats()
    ms = e0.elapsed_time(e1)
    grows_in_timed = gather.grows - grows_before
    total = hdrs[rank][0]
    gathered_rows = sum(h[0] for h in hdrs)
    device_res = gather.to_arrow([rank])  # this rank's batch as it sits in the gathered slots, downloaded for the checks
    # e2e: the same filters by the host's clock, the filtered Arrow array delivered to every rank's host memory each step
    e2e_steps = max(3, args.steps // 2)
    host_res = None
    for _ in range(3):
        host_res = e2e_step()  # the previous result stays alive like in the timed loop: both result blocks exist
    barrier()
    st_c = cache.stats()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        host_res = e2e_step()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    st_d = cache.stats()
    # parity inside the bench: the device-resident and the host results agree, and match pyarrow on regenerated entries
    import pyarrow.compute as pc
    chk = pa.concat_arrays([synth.int_entry("l_shipdate", rank * n_entries + i, seed=synth.SEED_TPCH) for i in range(min(4, n_entries))])
    want = chk.filter(pc.and_(pc.greater_equal(chk, pa.scalar(lo)), pc.less(chk, pa.scalar(hi))))
    ok = host_res.slice(0, len(want)).equals(want) and device_res.equals(host_res) and len(host_res) == total
    ok_t = torch.tensor([1.0 if ok else 0.0], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ok_t, op=dist.ReduceOp.MIN)
    ok = bool(ok_t.item() == 1.0)
    t = torch.tensor([ms, e2e_ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms = [float(x) for x in t.tolist()]
    clk = clocks.stop() if rank == 0 else None
    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        w = 12
        med = lambda x: float(np.median(x))  # noqa: E731
        b_ge = rows_local * w // 8 + rows_local // 8          # packed words + selection out (dense in: none)
        b_lt = rows_local * w // 8 + 2 * (rows_local // 8)    # packed words + selection in + out
        total_rows = rows_local * world
        line = {
            "metric": METRIC.replace("URL LIKE '%google%'", "l_shipdate range"), "value": total_rows * args.steps / (ms / 1e3) / 1e6,
            "unit": "Mrows/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": "TPC-H SF100 lineitem l_shipdate >= 1994-01-01 AND < 1995-01-01 (Date32, W=12), then get-with-selection "
                                   "(BASELINE configs[3]); each rank holds 1/8 of the 600 037 902 rows",
                       "rows_per_gpu": rows_local, "entries_per_gpu": n_entries, "matching_rows_per_gpu": int(total),
                       "selectivity": int(total) / rows_local, "liquid_bytes_per_gpu": int(cache.stats().hbm_bytes_used),
                       "parallelism": f"entries sharded by EntryID over {world} GPU(s), no collective in the scan; every step ends with ONE "
                                      "NCCL all_gather of the filtered batches (HBM to HBM) inside the clock" if world > 1 else "one GPU",
                       "result": "Arrow-layout buffers in HBM (lc_scan_read_async): value; host Arrow arrays (lc_scan_read): e2e",
                       "gathered_rows": int(gathered_rows), "host_syncs_per_step": 1, "gather_slot_bytes": gather.slot,
                       "slot_regrown_in_timed_steps": grows_in_timed, "numa": pin,
                       "l2": "packed column (113 MB) + selections do not fit the L2 together with the 44 MB result; no flush",
                       "setup_seconds": setup_s, "result_matches_arrow": bool(ok),
                       "insert": {"Mrows_per_s": rows_local / insert_s / 1e6, "arrow_GB_per_s": rows_local * 4 / insert_s / 1e9,
                                  "note": "lc_cache_insert_many, 1024 batches of 8192 rows per call, host Arrow in (pageable), device transcode"}},
            "e2e": {"value": total_rows * e2e_steps / (e2e_ms / 1e3) / 1e6, "unit": "Mrows/s", "ms_per_step": e2e_ms / e2e_steps,
                    "h2d_bytes_per_step": int((st_d.h2d_bytes - st_c.h2d_bytes) / e2e_steps),
                    "d2h_bytes_per_step": int((st_d.d2h_bytes - st_c.d2h_bytes) / e2e_steps)},
            "gpu_launches": int(st_b.kernel_launches - st_a.kernel_launches),
            "roofline": [
                {"kernel": "k_int_bits<REFINE> l_shipdate>=lo (W=12, dense selection in)", "bound": "hbm", "achieved": b_ge / (med(k_ms[0]) / 1e3) / 1e9,
                 "peak": peak, "unit": "GB/s", "frac": b_ge / (med(k_ms[0]) / 1e3) / 1e9 / peak, "kernel_ms": med(k_ms[0]),
                 "algorithmic_bytes_per_launch": b_ge, "traffic": None},
                {"kernel": "k_int_bits<REFINE> l_shipdate<hi (W=12, selection in+out)", "bound": "hbm", "achieved": b_lt / (med(k_ms[1]) / 1e3) / 1e9,
                 "peak": peak, "unit": "GB/s", "frac": b_lt / (med(k_ms[1]) / 1e3) / 1e9 / peak, "kernel_ms": med(k_ms[1]),
                 "algorithmic_bytes_per_launch": b_lt, "traffic": None},
            ],
            "peak_source": peak_src, "clocks": clk,
        }
        if not args.no_cpu_baseline and world == 1:
            import bench_cpu

            cpu_threads, _h = bench_cpu.usable_cpus()
            line["cpu_baseline"] = cpu_baseline_shipdate(cpu_sample_entries(args, cpu_threads, n_entries), cpu_threads)
        if emit:
            print(json.dumps(line))
    scan.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    cache.close()
    return line if rank == 0 else None


def cpu_baseline_shipdate(sample_entries: int, threads: int, target_s: float = 6.0):
    """C port of the reference's CPU path on the same column: two conjuncts (decode, filter, compare) joined by
    boolean_buffer_and_then per entry, then the get of the survivors; persistent pool of all host threads."""
    import bench_cpu

    return bench_cpu.cpu_baseline_line("shipdate", sample_entries, threads, params=shipdate_params(), target_s=target_s)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1 and "LC_HOST_THREADS" not in os.environ:
        # the library's host pool (selection staging, mask zero-fill of the host-buffer calls) defaults to 8 threads per
        # process; N ranks share one container's CPU quota (16 CPUs on the round-2 box), and threads beyond it are throttled
        import bench_cpu

        cpus, _ = bench_cpu.usable_cpus()
        os.environ["LC_HOST_THREADS"] = str(max(1, min(8, cpus // world - 1)))  # one CPU per rank is the Python thread's
    if args.workload == "int_filter":
        run_int_filter(args, rank, world, local_rank)
        return
    if args.workload == "shipdate":
        run_shipdate(args, rank, world, local_rank)
        return
    if args.workload == "squeeze":
        run_squeeze(args, rank, world, local_rank)
        return
    if args.workload == "insert":
        import bench_insert

        bench_insert.main(args, rank, world, local_rank)
        return
    if args.workload == "clickbench_sweep":
        import bench_sweep

        bench_sweep.main(args, rank, world, local_rank)
        return
    run_url_like(args, rank, world, local_rank, dump_dir=args.dump_outputs)


def run_url_like(args, rank, world, local_rank, emit=True, source=None, rows=None, secondary=True, dump_dir=None):
    """BASELINE configs[1] — the headline bench line. `source`: "synthetic" (synth/lc_synth.c: the 100 M-row column the
    metric is quoted on) or "sample" (URLs resampled from the reference's 24 586-row ClickBench sample, synth/hits.py: the
    real column's dictionary sizes, lengths and compressibility; reported beside it under config.secondary). `dump_dir`:
    rank 0 writes there the filtered URLs of every rank that the last timed step gathered (dump_strings)."""
    source = source or args.url_source
    import numpy as np
    import pyarrow as pa
    import torch
    import torch.distributed as dist

    from liquid_cache_b200 import (CacheExpression, Column, LikeExpr, LiquidCacheBuilder, LiquidExpr, Literal,
                                   parquet_array_id)

    torch.cuda.set_device(local_rank)
    numa_pin = pin_to_gpu_numa(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    cache = LiquidCacheBuilder.new().with_device(local_rank).build()
    # an explicit (non-default) stream shared by torch's events and every kernel / copy of the library
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    cache.set_stream(stream.cuda_stream)

    # ---- setup (untimed): this rank's shard of the column, transcoded into HBM ----
    n_entries = max(1, (rows or args.rows) // ROWS_PER_ENTRY)
    first = rank * n_entries  # entries shard by EntryID (file, row group, batch): rank r owns [r*E, (r+1)*E)
    t_setup = time.perf_counter()
    ids = []
    insert_s, arrow_bytes = 0.0, 0
    workers = max(2, min(32, (os.cpu_count() or 8) // max(1, world)))
    pend_ids, pend_arrs = [], []

    def flush():
        nonlocal insert_s
        if pend_ids:
            t_i = time.perf_counter()
            cache.insert_many(pend_ids, pend_arrs, hint=CacheExpression.SubstringSearch)
            insert_s += time.perf_counter() - t_i  # transcode on the device, 256 batches (8 row groups) per call (untimed setup)
            pend_ids.clear()
            pend_arrs.clear()

    for i, arr in generate_entries(first, n_entries, workers, source):
        # 32 batches per row group, column id 13 (= URL in hits); the FSST table is per (file, row group, column)
        eid = parquet_array_id(0, i // 32, 13, i % 32)
        pend_ids.append(eid)
        pend_arrs.append(arr)
        arrow_bytes += arr.nbytes
        ids.append(int(eid))
        if len(pend_ids) == 256:
            flush()
    flush()
    handles = cache.handles(ids)
    rows_local = n_entries * ROWS_PER_ENTRY
    setup_s = time.perf_counter() - t_setup
    st0 = cache.stats()
    hbm_bytes = int(st0.hbm_bytes_used)

    expr = LiquidExpr.try_new(LikeExpr(False, False, Column("URL", 0), Literal(PATTERN)), pa.string(),
                              CacheExpression.SubstringSearch)
    assert expr is not None
    pred = expr.to_native(pa.string())
    rows_arr = np.full(n_entries, ROWS_PER_ENTRY, dtype=np.uint64)
    scan = cache.scan(rows_arr)

    # ---- algorithmic bytes of one predicate launch (measurement aid, outside any timed region) ----
    cache.profile_counters(True)
    scan.reset()
    scan.filter_native(handles, pred)
    cache.synchronize()
    prof = cache.profile_counters(False)
    uniques, cand, cand_bytes = int(prof[0]), int(prof[1]), int(prof[2])
    if int(prof[11]) and rank == 0:  # library built with -DLC_PHASE_PROF: per-phase cycle split of k_str_scan
        names = ["staging wait", "plan", "symbol tables", "candidate gate", "code walk", "row-section wait", "rows"]
        tot = float(prof[11])
        print("[phase cycles per CTA] " + ", ".join(f"{nm} {float(prof[4 + i]) / n_entries:.0f} ({100 * float(prof[4 + i]) / tot:.1f}%)"
                                                      for i, nm in enumerate(names)) + f", total {tot / n_entries:.0f}", file=sys.stderr)
    # Algorithmic bytes of one predicate launch, SURVEY.md §8d "string predicate, fingerprint path", counted by the kernel's
    # own counters in the untimed launch above:  R = keys 2n + staged head (header, shared prefix, fingerprints 4U, ALL offset
    # residuals (U+1)*res_bytes) + compressed bytes of the walked candidates;  W = selection words n/8.
    # That is the reference's data for this predicate; roofline.achieved is quoted on it. `kernel_reads` says what THIS build
    # moves instead: the header, the needle's planes of the private trigram filter (entry_layout.h: k * ceil(U/32) words per
    # entry; fingerprints and residuals of values that are not walked are never read), the walked values, the keys of
    # the batches whose dictionary had a match (the others are answered without their keys: k_str.cu, k_str_like), and
    # the selection words.
    ref_pass, meta_bytes, rows_phase_entries, gate_bytes = int(prof[12]), int(prof[13]), int(prof[3]), int(prof[14])
    if meta_bytes == 0:  # the launch did not take the streaming LIKE kernel
        meta_bytes = 4 * uniques + 2 * uniques
        ref_pass = uniques
        rows_phase_entries = n_entries
        gate_bytes = 4 * uniques
    algo_bytes = 2 * rows_local + meta_bytes + cand_bytes + rows_local // 8
    kernel_reads = 128 * n_entries + gate_bytes + cand_bytes + rows_phase_entries * 2 * ROWS_PER_ENTRY + rows_local // 8

    k_start = torch.cuda.Event(enable_timing=True)
    k_stop = torch.cuda.Event(enable_timing=True)
    kernel_ms = []
    result_rows = [0]

    trace = os.environ.get("LC_BENCH_TRACE") == "1"

    from liquid_cache_b200.dist import DeviceGather

    dev = torch.device("cuda", local_rank)
    gather = DeviceGather(pa.string(), rank, world, dev)

    def step(time_kernel: bool):
        """LIKE over every entry of this rank, then get-with-selection of the survivors, delivered as Arrow-layout buffers in
        HBM: lc_scan_read_async plans rows / bytes on the device and decodes straight into this rank's gather slot; at N > 1
        ONE all_gather over NVLink — the one exchange of the path — puts every rank's batch into rank 0's HBM. The only host
        synchronisation of the step is the download of the 64-byte headers (DeviceGather.exchange)."""
        t0 = time.perf_counter()
        for _ in range(16):
            scan.reset()
            scan.filter_native(handles, pred)
            if not scan.read_async(handles, *gather.addresses()):
                raise RuntimeError("the URL column must be readable by the device-planned path")
            hdrs = gather.exchange()
            if not gather.overflowed():
                break
            gather.grow()  # warm-up only: capacities settle on the first steps
        else:
            raise RuntimeError("gather slot capacities did not settle")
        t3 = time.perf_counter()
        result_rows[0] = hdrs[rank][0]
        if time_kernel:
            kernel_ms.append(cache.last_kernel_ms())  # events recorded by the library right around the launch
        if trace and rank == 0:
            print(f"[trace] step (filter + read + exchange) {1e3*(t3-t0):.3f} ms", file=sys.stderr)
        return hdrs

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = None
    for _ in range(max(3, args.warmup)):
        last = step(False)
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    for _ in range(3):  # the sampler's start-up left the GPU idle for a moment: back to the steady state before the clock
        last = step(False)
    cache.kernel_timing(True)
    barrier()
    st_a = cache.stats()
    grows_before = gather.grows
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    import gc

    gc.disable()  # a collection inside a 0.5 ms step is a visible spike; re-enabled after the timed loops
    ev0.record(stream)
    step_wall = []
    for _ in range(args.steps):
        w0 = time.perf_counter()
        last = step(True)
        step_wall.append((time.perf_counter() - w0) * 1e3)  # every step ends synchronised: host wall == device time
    ev1.record(stream)
    barrier()
    gc.enable()
    st_b = cache.stats()
    ms_total = ev0.elapsed_time(ev1)
    launches = int(st_b.kernel_launches - st_a.kernel_launches)
    gathered_rows = sum(h[0] for h in last)
    grows_in_timed = gather.grows - grows_before
    # what the e2e arm below is compared with: THIS rank's own filtered batch, downloaded from the gathered slots
    local_last = gather.to_arrow([rank])
    if dump_dir and rank == 0:
        dump_strings(dump_dir, "url", gather.to_arrow())

    # where a step's time goes (untimed, after the measurement): device events between the three calls of a step
    ph = [[], [], [], []]
    for _ in range(5):
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        w0 = time.perf_counter()
        evs[0].record(stream)
        scan.reset()
        scan.filter_native(handles, pred)
        evs[1].record(stream)
        scan.read_async(handles, *gather.addresses())
        evs[2].record(stream)
        gather.exchange()
        evs[3].record(stream)
        stream.synchronize()
        ph[3].append((time.perf_counter() - w0) * 1e3)
        for i in range(3):
            ph[i].append(evs[i].elapsed_time(evs[i + 1]))
    step_phases = {k: float(np.median(v)) for k, v in zip(("filter_ms", "read_async_ms", "exchange_ms", "host_wall_ms"), ph)}

    # ---- e2e: the same pass through the host-buffer C ABI (H2D + D2H inside the timed region) ----
    # host result buffers, allocated once and page-locked (the reference-side caller would own these)
    sizes = (((rows_arr + 7) // 8 + 15) // 16) * 16
    offs = np.zeros(n_entries, dtype=np.uint64)
    np.cumsum(sizes[:-1], out=offs[1:])
    total_mask_bytes = int(sizes.sum())
    pin = lambda nbytes: torch.empty(nbytes, dtype=torch.uint8, pin_memory=True).numpy()  # noqa: E731
    # no validity buffer: `hits.URL` is declared NOT NULL, a BooleanArray over it carries no null bitmap (lc_gpu.h: out_validity
    # may be NULL; the null counts still come back and are checked to be zero below)
    out_bufs = (pin(total_mask_bytes), None, offs, np.zeros(n_entries, dtype=np.uint64),
                np.zeros(n_entries, dtype=np.uint64), np.zeros(n_entries, dtype=np.uint64))

    vals_addr = np.uint64(out_bufs[0].ctypes.data)

    def e2e_step():
        t0 = time.perf_counter()
        vals, valid, offs, out_len, out_nulls, true_counts = cache._eval_many_native(handles, rows_arr, pred, None, out_bufs)
        t1 = time.perf_counter()
        assert not out_nulls.any()
        # like LiquidCacheReader::read_from_cache: only batches with surviving rows are read
        hit = np.flatnonzero(true_counts)
        if len(hit) == 0:
            return None
        sel_ptrs = vals_addr + offs[hit]  # each surviving batch's mask is its selection for the read
        t2 = time.perf_counter()
        out = cache.to_arrow_many_ptrs(handles[hit], sel_ptrs)
        t3 = time.perf_counter()
        if trace and rank == 0:
            print(f"[trace] e2e: eval_many {1e3*(t1-t0):.3f} ms, pick {1e3*(t2-t1):.3f} ms, to_arrow_many {1e3*(t3-t2):.3f} ms",
                  file=sys.stderr)
        return out

    for _ in range(3):
        e2e_out = e2e_step()
    barrier()
    st_c = cache.stats()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    e2e_steps = max(3, args.steps // 2)
    for _ in range(e2e_steps):
        e2e_out = e2e_step()
    e1.record(stream)
    barrier()
    e2e_wall = time.perf_counter() - t0
    st_d = cache.stats()
    e2e_ok = (e2e_out is None and result_rows[0] == 0) or (e2e_out is not None and len(e2e_out) == result_rows[0] and e2e_out.equals(local_last))

    # max over ranks
    t = torch.tensor([ms_total, e2e_wall * 1e3, float(sum(kernel_ms) / max(1, len(kernel_ms)))], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms, kern_ms = [float(x) for x in t.tolist()]
    clk = clocks.stop() if rank == 0 else None

    if rank == 0:
        total_rows = rows_local * world
        value = total_rows * args.steps / (ms_total / 1e3) / 1e6
        e2e_val = total_rows * e2e_steps / (e2e_ms / 1e3) / 1e6
        peak, peak_src = measured_peak_gbs()
        achieved = algo_bytes / (kern_ms / 1e3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": "Mrows/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {
                "workload": "clickbench-hits URL column (FSST+dict+fingerprints) LIKE '%google%' then get-with-selection (BASELINE configs[1])"
                            + ("" if source == "synthetic" else "; URLs resampled from the reference's ClickBench sample (synth/hits.py)"),
                "url_source": source,
                "rows_per_gpu": rows_local, "entries_per_gpu": n_entries, "rows_per_entry": ROWS_PER_ENTRY,
                "liquid_bytes_per_gpu": hbm_bytes, "liquid_bytes_per_row": hbm_bytes / rows_local,
                "unique_values_per_entry": uniques / n_entries, "walked_candidates_frac": cand / max(1, uniques),
                "matching_rows": int(gathered_rows),
                "parallelism": f"entries sharded by EntryID over {world} GPU(s), no collective in the scan; every step ends with ONE NCCL all_gather of the filtered batches (HBM to HBM) inside the clock" if world > 1 else "one GPU",
                "result": "Arrow-layout buffers in HBM (lc_scan_read_async): value; host Arrow arrays through the host-buffer ABI: e2e",
                "host_syncs_per_step": 1, "gather_slot_bytes": gather.slot, "slot_regrown_in_timed_steps": grows_in_timed,
                "untimed_steps_before_the_clock": max(3, args.warmup) + 3,  # --warmup, then 3 more once the clock sampler is up
                "step_phases": step_phases,
                "step_ms_rank0": {"min": min(step_wall), "median": float(np.median(step_wall)), "max": max(step_wall)}, "numa": numa_pin,
                "l2": "inputs (liquid column) larger than the 126 MB L2, no flush needed",
                "setup_seconds": setup_s,
                "insert": {"Mrows_per_s": rows_local / insert_s / 1e6, "arrow_GB_per_s": arrow_bytes / insert_s / 1e9,
                           "note": "lc_cache_insert_many, 256 batches of 8192 rows per call, host Arrow in, device transcode (k_str_encode.cu *_many), single stream"},
            },
            "e2e": {"value": e2e_val, "unit": "Mrows/s", "h2d_bytes_per_step": int((st_d.h2d_bytes - st_c.h2d_bytes) / e2e_steps),
                    "d2h_bytes_per_step": int((st_d.d2h_bytes - st_c.d2h_bytes) / e2e_steps), "ms_per_step": e2e_ms / e2e_steps,
                    "matches_device_path": bool(e2e_ok)},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "k_str_like<MODE_REFINE>", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": recorded_traffic(rows_local, n_entries) if source == "synthetic" else None,
                         "traffic_source": "replayed from profiles/r02_k_str_like_traffic.json (ncu --set full of this seeded workload), not measured in this run",
                         "algorithmic_bytes_per_launch": algo_bytes,
                         "gate_bytes_read": gate_bytes,
                         "bytes_this_kernel_must_move": kernel_reads,
                         "achieved_on_bytes_moved": kernel_reads / (kern_ms / 1e3) / 1e9,
                         "reference_gate_pass_frac": ref_pass / max(1, uniques),
                         "batches_with_a_match_frac": rows_phase_entries / n_entries,
                         "kernel_ms": kern_ms, "peak_source": peak_src,
                         "kernel_share_of_step": kern_ms / (ms_total / args.steps)},
            "clocks": clk,
        }
        if not args.no_cpu_baseline and world == 1 and source == "synthetic":
            import bench_cpu

            cpu_threads, _h = bench_cpu.usable_cpus()
            line["cpu_baseline"] = cpu_baseline(cpu_sample_entries(args, cpu_threads, n_entries), cpu_threads)
    scan.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    cache.close()
    if rank == 0:
        if world == 1 and not args.no_secondary and secondary:
            # BASELINE configs[2] and [3] measured in the SAME run, so that their rooflines sit in the driver's bench line
            # (VERDICT r1 item 4) — each is also a workload of its own (--workload int_filter / shipdate)
            sec = {}
            if source == "synthetic":
                # the same step on URLs resampled from the real table's sample (16.8 M rows): what the synthetic column's
                # higher compressibility hides (VERDICT r1 weak 8)
                try:
                    sub = run_url_like(args, 0, 1, local_rank, emit=False, source="sample", rows=16_777_216, secondary=False)
                    sec["url_like_clickbench_sample"] = {k: sub[k] for k in ("value", "unit", "ms_per_step", "e2e", "roofline", "gpu_launches")}
                    sec["url_like_clickbench_sample"].update({k: sub["config"][k] for k in (
                        "rows_per_gpu", "liquid_bytes_per_row", "unique_values_per_entry", "walked_candidates_frac", "matching_rows", "insert")})
                except Exception as e:
                    sec["url_like_clickbench_sample"] = {"error": f"{type(e).__name__}: {e}"[:300]}
            for name, fn in (("int_filter", run_int_filter), ("shipdate", run_shipdate)):
                try:
                    sub = fn(args, 0, 1, local_rank, emit=False)
                    sec[name] = {k: sub[k] for k in ("metric", "value", "unit", "ms_per_step", "e2e", "roofline", "cpu_baseline", "gpu_launches")
                                 if k in sub}
                    sec[name]["workload"] = sub["config"]["workload"]
                    sec[name]["rows_per_gpu"] = sub["config"]["rows_per_gpu"]
                except Exception as e:  # a secondary workload must not take the headline line down with it
                    sec[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
            line["config"]["secondary"] = sec
        if emit:
            print(json.dumps(line))
        return line
    return None


if __name__ == "__main__":
    main()
