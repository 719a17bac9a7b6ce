#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native FiloDB chunk-scan + range-vector-aggregation path.

Workload (BASELINE.json configs[1], "C2"): per GPU 10M series x 2h@15s (480 rows, chunks 400+80), const-DDV timestamps,
XOR-NibblePack ("Gorilla-compressed") gauge values 15+sin(n+1)+N(0,1) with 0.1% NaN stale markers at chunk ends,
query rate()[5m] step 15s over the 2 h (T = 481 windows), gauge schema => RateOverDeltaChunkedFunctionD
(sum_over_time / window * 1000), no across-series aggregate: output is [series x T] f64.

  python bench.py [--gpus N] [--steps K] [--warmup W]            # product arm, one JSON line on rank 0
  python bench.py --impl reference ...                           # reference CPU path (oracle port) on host cores
  python bench.py ... --dump-outputs DIR                         # also write the last timed step's result arrays as DIR/<name>.npy

A step = one pass of the hot path over the whole resident table (1 kernel launch).  `value` = samples scanned per second
(Σ numRows of the chunks scanned, the quantity FiloDB counts in samplesScannedCtr) with inputs resident in HBM;
`e2e` = the same through the C-ABI with HOST buffers: filo_load_series (gather + H2D) + filo_query (+ D2H) every step.
Multi-GPU: series are sharded by id across ranks (FiloDB shard -> GPU), no data-path collective for this query
(`--workload c5` runs sum(rate) by(cluster) with one NCCL all-reduce of the [G x T] partials).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T0_MS = 1_700_000_000_000
INTERVAL = 15000
ROWS = 480
ROWS_PER_CHUNK = 400
WINDOW = 300000
STEP = 15000


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="filo", choices=["filo", "reference"])
    ap.add_argument("--series", type=int, default=10_000_000, help="series per GPU")
    ap.add_argument("--workload", default="c2", choices=["c1", "c2", "c2-raw", "c2-counter", "c3", "c3-const", "c4", "c5"])
    ap.add_argument("--e2e-series", type=int, default=-1, help="series in the end-to-end leg (-1 = all)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-series", type=int, default=2_000_000, help="bounded sample for the CPU baseline legs")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-staged", action="store_true", help="e2e leg: stage inputs through pinned slabs on the host instead of the registered-memory gather")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the kernel-only sub-records of the other BASELINE configs (C1, C3, C3-const, C4) of the default single-GPU C2 run")
    ap.add_argument("--no-c5", action="store_true", help="skip the C5 sub-record (sum(rate) by(cluster) with the NCCL all-reduce) of the default C2 run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float64; a fixed, seeded sample of the rows "
                         "when the result is larger than %d MB), so that two builds can be compared output for output" % (DUMP_LIMIT_BYTES // 1_000_000))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 60_000_000
DUMP_SEED = 20231114
NPY_HEADER_BYTES = 4096          # generous bound on the header np.save writes in front of the data


def dump_row_sample(n_rows, row_bytes):
    """Rows of an [n_rows x ...] result that fit the dump limit: all of them, or a sorted sample drawn with a fixed seed (the same rows
    for the same arguments, whichever build runs).  Each sampled row also costs 8 bytes in the `<name>_rows` index array."""
    fit = (DUMP_LIMIT_BYTES - 2 * NPY_HEADER_BYTES) // (row_bytes + 8)
    if n_rows <= fit:
        return None
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n_rows, size=fit, replace=False))


def dump_outputs(d, arrays):
    """Writes each named result array as d/<name>.npy in float64.  `arrays` maps a name to (array, rows), where rows is None (the whole
    array) or the sorted indices of the first axis the array holds; those go beside it as d/<name>_rows.npy (float64, exact)."""
    os.makedirs(d, exist_ok=True)
    total = 0
    for name, (a, rows) in arrays.items():
        files = [(name, a)] + ([(name + "_rows", rows)] if rows is not None else [])
        for fname, x in files:
            path = os.path.join(d, fname + ".npy")
            np.save(path, np.ascontiguousarray(x, dtype=np.float64))
            total += os.path.getsize(path)
    assert total <= DUMP_LIMIT_BYTES, total


def host_rows(a, rows):
    """The given rows of the first axis of a device tensor or host array (all of them when rows is None), as a host numpy array."""
    if rows is not None:
        if hasattr(a, "index_select"):
            import torch
            a = a.index_select(0, torch.from_numpy(rows).to(a.device))
        else:
            a = a[rows]
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


WORKLOADS = {
    # name: (synth kwargs, fn, aggr, n_groups, description)
    "c1": (dict(value_kind=0, value_enc=1, nan_per_million=1000), "FN_SUM_OVER_TIME", "AGG_NONE", 0,
           "C1: {S} series x 1h@15s (240 rows, one chunk), const-DDV ts, XOR-NibblePack doubles, sum_over_time[5m] step 15s (BASELINE configs[0]: the reference's own CPU-runnable case)"),
    "c2": (dict(value_kind=0, value_enc=1, nan_per_million=1000), "FN_RATE", "AGG_NONE", 0,
           "C2: {S} series x 2h@15s (480 rows, chunks 400+80), const-DDV ts, XOR-NibblePack gauge, rate()[5m] step 15s, T=481, no aggregate"),
    "c2-raw": (dict(value_kind=0, value_enc=0, nan_per_million=1000), "FN_RATE", "AGG_NONE", 0,
               "C2 variant: raw f64 gauge values (the reference's native DoubleVector encoding)"),
    "c2-counter": (dict(value_kind=1, value_enc=1, nan_per_million=1000, reset_period=1000, schema_flags=1), "FN_RATE", "AGG_NONE", 0,
                   "C2 variant: prom-counter schema (extrapolated Prometheus rate with counter correction)"),
    "c3": (dict(value_kind=1, value_enc=1, reset_period=1000, schema_flags=1, ts_jitter_ms=2000), "FN_INCREASE", "AGG_SUM", 1000,
           "C3: counters, DDV ts + XOR values, increase()[1m] then sum by(job), 1000 jobs"),
    "c3-const": (dict(value_kind=1, value_enc=1, reset_period=1000, schema_flags=1), "FN_INCREASE", "AGG_SUM", 1000,
                 "C3 variant: regular scrapes (const-DDV ts, what the reference's +-250 ms rule produces for <=100 ms jitter), XOR counters, increase()[1m] then sum by(job), 1000 jobs"),
    "c5": (dict(value_kind=1, value_enc=1, reset_period=1000, schema_flags=1), "FN_RATE", "AGG_SUM", 100,
           "C5: counters, sum(rate()[5m]) by(cluster), 100 clusters, NCCL all-reduce of the [G x T] partials"),
}


def query_range(workload):
    window = 60000 if workload.startswith("c3") else WINDOW
    return T0_MS, STEP, T0_MS + (ROWS * INTERVAL), window


def host_cores():
    """Threads this process may actually run on: scheduler affinity capped by the cgroup CPU quota (os.cpu_count() ignores both, and a
    128-thread run inside an 8-CPU lease is how the round-1 CPU baseline moved 5x between boxes)."""
    visible = os.cpu_count() or 1
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = visible
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                      # cgroup v2: "<quota|max> <period>"
            q, per = f.read().split()[:2]
            if q != "max":
                quota = float(q) / float(per)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f: q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f: per = float(f.read())
            if q > 0:
                quota = q / per
        except Exception:
            quota = None
    usable = aff if quota is None else max(1, min(aff, int(quota + 0.999)))
    return {"cores_visible": visible, "cores_affinity": aff, "cpu_quota": quota, "cores_usable": usable}


class ClockSampler:
    """SM clocks / throttle reasons DURING the timed region (B200_PROFILING.md).  NVML polled from a thread of this process (the
    library is initialised before the warm-up, so nothing starts up inside the timed region -- an `nvidia-smi` child launched right
    before it was seen to delay the first steps on some boxes); `nvidia-smi -lms` is the fallback when pynvml is missing.  Only the
    samples taken between mark_start() and stop() count."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.samples = []          # (t, sm_mhz, reasons bitmask or set)
        self.mx = None
        self.t0 = None
        self._stop = False
        self.nvml = None

    def start(self):
        """Call before the warm-up."""
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES remaps ordinals: go through the PCI bus id of the torch device
            import torch
            h = None
            try:
                bus = torch.cuda.get_device_properties(self.idx).pci_bus_id
                for i in range(pynvml.nvmlDeviceGetCount()):
                    hh = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if pynvml.nvmlDeviceGetPciInfo(hh).bus == bus:
                        h = hh
                        break
            except Exception:
                h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            self.nvml, self.h = pynvml, h
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv, h = self.nvml, self.h
        names = (("hw_slowdown", getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8)), ("hw_thermal_slowdown", getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40)),
                 ("sw_thermal_slowdown", getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20)), ("sw_power_cap", getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)))
        while not self._stop:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((time.perf_counter(), sm, {n for n, bit in names if r & bit}))
            except Exception:
                pass
            time.sleep(0.01)

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            if len(f) < 8:
                continue
            try:
                sm = float(f[1]); self.mx = float(f[2])
            except ValueError:
                continue
            rs = {name for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]) if v.lower().startswith("active")}
            self.samples.append((time.perf_counter(), sm, rs))

    def mark_start(self):
        self.t0 = time.perf_counter()

    def stop(self):
        t1 = time.perf_counter()
        if self.nvml is None and not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml / nvidia-smi unavailable"]}
        if self.nvml is None:
            time.sleep(0.1)
        self._stop = True
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        t0 = self.t0 if self.t0 is not None else 0.0
        inside = [x for x in self.samples if t0 <= x[0] <= t1 + 0.2]
        sm = [x[1] for x in inside]
        reasons = set()
        for x in inside:
            reasons |= x[2]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.mx, "reasons": sorted(reasons), "samples": len(sm),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}



def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def host_chunk_infos(arena, rec_off, n_series):
    """Host mirror of a shard's chunk metadata over a host copy of the arena: builds ChunkSetInfo blocks
    (core/src/main/scala/filodb.core/store/ChunkSetInfo.scala:133-154) whose vector pointers point into `arena`.
    Returns (n_chunks int32[S], info_addrs uint64[Σ], keepalive)."""
    base = arena.ctypes.data
    nch = arena[(rec_off[:n_series, None] + np.arange(4, 8)[None, :])].copy().view(np.uint32).reshape(-1).astype(np.int32)
    total = int(nch.sum())
    infos = np.zeros((total, 44), np.uint8)
    cb = np.concatenate([[0], np.cumsum(nch)]).astype(np.int64)
    maxc = int(nch.max()) if n_series else 0
    for c in range(maxc):
        sel = np.nonzero(nch > c)[0]
        eoff = rec_off[sel] + 16 + 32 * c
        ent = arena[(eoff[:, None] + np.arange(32)[None, :])].copy()
        start = ent[:, 0:8].copy().view(np.int64).reshape(-1)
        end = ent[:, 8:16].copy().view(np.int64).reshape(-1)
        nrows = ent[:, 16:20].copy().view(np.int32).reshape(-1)
        tso = ent[:, 20:24].copy().view(np.uint32).reshape(-1).astype(np.uint64)
        vlo = ent[:, 24:28].copy().view(np.uint32).reshape(-1).astype(np.uint64)
        row = cb[sel] + c
        ing = end + 1000
        chunk_id = ((np.uint64(1) << np.uint64(63)) ^ (start.astype(np.uint64) << np.uint64(22))) | ((ing // 1000) % (48 * 24 * 3600)).astype(np.uint64)
        infos[row, 0:8] = chunk_id.view(np.uint8).reshape(-1, 8)
        infos[row, 8:12] = nrows.view(np.uint8).reshape(-1, 4)
        infos[row, 12:20] = ing.view(np.uint8).reshape(-1, 8)
        infos[row, 20:28] = end.view(np.uint8).reshape(-1, 8)
        recb = np.uint64(base) + rec_off[sel].astype(np.uint64)
        infos[row, 28:36] = (recb + tso).view(np.uint8).reshape(-1, 8)
        infos[row, 36:44] = (recb + vlo).view(np.uint8).reshape(-1, 8)
    addrs = np.uint64(infos.ctypes.data) + np.arange(total, dtype=np.uint64) * np.uint64(44)
    return nch, addrs, infos


def _splitmix64_np(x):
    with np.errstate(over="ignore"):
        x = x + np.uint64(0x9E3779B97F4A7C15)
        z = x
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def synth_group_ids(seed, base, n, n_groups):
    """group id of series base..base+n of a synthetic table (same hash as filodb_b200/csrc/synth_kernels.cu)."""
    with np.errstate(over="ignore"):
        gid = np.arange(base, base + n, dtype=np.uint64)
        h = _splitmix64_np(np.uint64(seed) ^ np.uint64(0xA5A5A5A5) ^ (gid * np.uint64(0x9E3779B97F4A7C15)))
    return (h % np.uint64(n_groups)).astype(np.int32)


def measured_traffic(workload, S):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed ncu capture of this same
    command (profiles/traffic.json: bytes per launch at the recorded series count); None when not captured."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            rec = json.load(f).get(workload)
        if rec and int(rec["series"]) == int(S):
            return float(rec["dram_bytes_per_launch"])
        if rec and "dram_bytes_per_series" in rec:      # captured at another series count: every series is read and written once, traffic scales with S
            return float(rec["dram_bytes_per_series"]) * int(S)
    except (OSError, ValueError, KeyError):
        pass
    return None


def run_reference(args, rank, world):
    """Reference arm: the reference's own CPU path for this query — the C++ restatement under oracle/ (the JVM cannot run
    in this image) — on all host threads, on a bounded sample of the same workload."""
    if rank != 0:
        return
    from oracle import oracle as o
    if args.workload == "c4" and rank == 0:
        from oracle import hist as H, oracle as o
        nb, K = 20, min(args.cpu_series, 1024)
        b = H.Buckets.custom([2.0 * 3 ** i for i in range(nb - 1)] + [float("inf")])
        rng = np.random.default_rng(42)
        st = H.HistStore(b)
        ts = T0_MS + np.arange(ROWS, dtype=np.int64) * INTERVAL
        for s_ in range(K):
            obs = np.zeros((ROWS, nb), np.int64)
            obs[np.arange(ROWS), (np.arange(ROWS) + s_) % nb] = 1 + rng.integers(0, 3, ROWS)
            st.add_series(ts, np.cumsum(np.cumsum(obs, axis=1), axis=0), [ROWS_PER_CHUNK, ROWS - ROWS_PER_CHUNK])
        start, step, end, window = T0_MS, STEP, T0_MS + 7200000, WINDOW
        def one_h():
            return st.query(o.FN_RATE, start, step, end, window, aggr=True, group_ids=np.zeros(K, np.int32), n_groups=1, q=0.99)
        for _ in range(args.warmup): one_h()
        t0 = time.perf_counter()
        for _ in range(args.steps): res = one_h()
        dt = (time.perf_counter() - t0) / args.steps
        if args.dump_outputs:
            hv, hempty, hq = res
            dump_outputs(args.dump_outputs, {"values": (hv, None), "empty": (hempty, None), "quantile": (hq, None)})
        val = K * ROWS / dt
        print(json.dumps({"impl": "reference", "metric": "samples/s scanned+aggregated (rate over 10M series); % HBM roofline", "value": val, "unit": "samples/s",
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "i64 bucket counts -> f64 rates", "data": "synthetic",
                          "config": {"workload": "C4: histogram_quantile(0.99, sum(rate(h[5m]))) over SectDelta histogram series, 20 custom buckets", "sample": "%d series per step" % K},
                          "cpu_baseline": {"value": val, "unit": "samples/s", "cores": 1, "kind": "port", "sample": "%d series per step, 1 thread, oracle restatement of ChunkedWindowIteratorH + HistRateFunction" % K},
                          "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)
        return
    if args.workload == "c4":
        return
    synth, fn_name, aggr_name, n_groups, desc = WORKLOADS[args.workload]
    S = min(args.series, args.cpu_series)
    hc = host_cores()
    cores = hc["cores_usable"]
    st = o.Store()
    st.add_synth(S, ROWS, ROWS_PER_CHUNK, T0_MS, INTERVAL, seed=42, threads=cores, **synth)   # same rows/bytes as the GPU generator
    start, step, end, window = query_range(args.workload)
    cumulative = bool(synth.get("schema_flags", 0) & 1)
    groups = o.synth_group_ids(42, 0, S, n_groups) if n_groups else None

    def one():
        return st.query(getattr(o, fn_name), start, step, end, window, cumulative=cumulative, aggr=getattr(o, aggr_name),
                        group_ids=groups, n_groups=max(n_groups, 1), threads=cores, reuse_out=True)
    for _ in range(args.warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = one()
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:      # [series x T] for the sample of S series, or [groups x T]
        rows = dump_row_sample(res.shape[0], res.shape[1] * 8)
        dump_outputs(args.dump_outputs, {"values": (host_rows(res, rows), rows)})
    samples = S * ROWS
    val = samples / dt
    line = {"impl": "reference", "metric": "samples/s scanned+aggregated (rate over 10M series); % HBM roofline", "value": val, "unit": "samples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": desc.format(S=args.series) + " (per GPU; series sharded by id across GPUs)", "series_per_gpu": args.series, "rows": ROWS,
                       "windows": int(o.num_windows(start, step, end)), "window_ms": window, "step_ms": step,
                       "sample": "%d of %d series per step" % (S, args.series)},
            "cpu_baseline": dict({"value": val, "unit": "samples/s", "cores": cores, "kind": "port",
                             "sample": "%d series (%.1f%% of the workload) per step, %d host threads (= usable cores), oracle C++ restatement of ChunkedWindowIteratorD" % (S, 100.0 * S / args.series, cores)}, **hc),
            "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)



def run_c5_sub(args, ctx, rank, world, dist, stream, peak):
    """BASELINE C5 beside the headline workload: sum(rate(counter[5m])) by (cluster), 100 clusters, 128 shards over the GPUs of the box,
    every rank folds its shards into [G x T] partials (FILO_Q_PARTIAL), ONE NCCL all-reduce merges them (the plan's only fan-in,
    ReduceAggregateExec), filo_present_partials finishes.  The collective is inside the timed region.  Shards -> GPUs by
    shard.shards_of_rank (ShardMapper.scala:93-102,122-130); a shard is a block of S * N / 128 consecutive series ids."""
    import torch
    import filodb_b200.capi as capi
    from filodb_b200 import shard
    synth, fn_name, aggr_name, G, desc = WORKLOADS["c5"]
    fn, aggr = getattr(capi, fn_name), getattr(capi, aggr_name)
    S = args.series
    NSH = 128
    my_shards = shard.shards_of_rank(NSH, rank, world)
    tab = ctx.synth_table(S, ROWS, ROWS_PER_CHUNK, T0_MS, INTERVAL, n_groups=G, seed=42, series_id_base=rank * S, **synth)
    torch.cuda.synchronize()
    ti = tab.info()
    start, step, end, window = query_range("c5")
    T = capi.num_windows(start, step, end)
    out = torch.empty(G * T, dtype=torch.float64, device="cuda")
    aux = torch.empty(G * T, dtype=torch.int64, device="cuda")
    final = torch.empty(G * T, dtype=torch.float64, device="cuda")
    flags = capi.Q_PARTIAL if world > 1 else 0

    def step_fn():
        ctx.query_device(tab, fn, start, step, end, window, out.data_ptr(), aux.data_ptr(), aggr=aggr, flags=flags, stream=stream, want_stats=False)
        if world > 1:
            shard.merge_partials(out, aux, aggr, dist)
            ctx.present_partials(aggr, G * T, out.data_ptr(), aux.data_ptr(), final.data_ptr(), stream=stream)
    st = ctx.query_device(tab, fn, start, step, end, window, out.data_ptr(), aux.data_ptr(), aggr=aggr, flags=flags, stream=stream, want_stats=True)
    assert st["samples_scanned"] == ti.n_samples, (st, ti.n_samples)
    for _ in range(max(3, args.warmup)):
        step_fn()
    torch.cuda.synchronize()
    kern_ns = [ctx.query_device(tab, fn, start, step, end, window, out.data_ptr(), aux.data_ptr(), aggr=aggr, flags=flags, stream=stream, want_stats=True)["kernel_ns"]
               for _ in range(3)]
    if dist: dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_fn()
    e1.record()
    torch.cuda.synchronize()
    if dist: dist.barrier()
    ms = e0.elapsed_time(e1) / args.steps
    ms_per_rank = [ms]
    if dist:
        tl = [torch.zeros(1, device="cuda") for _ in range(world)]
        dist.all_gather(tl, torch.tensor([ms], device="cuda", dtype=torch.float32))
        ms_per_rank = [float(x.item()) for x in tl]
        ms = max(ms_per_rank)
    kern_ms = float(np.median(kern_ns)) / 1e6
    alg_bytes = ti.algorithmic_bytes + S * 4 + G * T * 8
    achieved = alg_bytes / (kern_ms / 1e3) / 1e9
    rec = {"workload": desc + "; %d series per GPU, %d series in all; 128 shards, GPU g owns shards {s : s mod N == g} (shard.shards_of_rank)" % (S, S * world),
           "value": ti.n_samples * world / (ms / 1e3), "unit": "samples/s", "n_gpus": world, "ms_per_step": ms, "ms_per_rank": [round(x, 3) for x in ms_per_rank],
           "steps": args.steps, "scaling": "weak", "collective": "NCCL all-reduce of [G x T] sums and counts + filo_present_partials, inside the timed region" if world > 1 else "none (one GPU)",
           "shards_of_rank0": my_shards if rank == 0 else None, "groups": G, "windows": T,
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "kernel_ms": kern_ms, "algorithmic_bytes": alg_bytes,
                        "kernel": "scan_wp_ctr_kernel<rate, fused> + v2 fallback over declined items + merge_partials"}}
    del out, aux, final
    tab.free()
    torch.cuda.empty_cache()
    # ---- parity at bench scale (outside the timed region, one GPU): the fused device result for the first Sc series against the oracle's
    # fold of its own per-series rates, every (cluster, window) cell within 1e-9 relative
    if world == 1 and rank == 0 and not args.no_cpu:
        try:
            from oracle import oracle as o
            Sc = min(S, args.cpu_series)
            tab2 = ctx.synth_table(Sc, ROWS, ROWS_PER_CHUNK, T0_MS, INTERVAL, n_groups=G, seed=42, series_id_base=0, **synth)
            got = np.asarray(ctx.query(tab2, fn, start, step, end, window, aggr=aggr)).reshape(-1)
            arena, rec_off = tab2.read_arena(0, Sc)
            ost = o.Store(); ost.add_from_arena(arena, rec_off, Sc)
            gids = synth_group_ids(42, 0, Sc, G)
            exp = ost.query(getattr(o, fn_name), start, step, end, window, cumulative=True, aggr=getattr(o, aggr_name), group_ids=gids, n_groups=G,
                            threads=host_cores()["cores_usable"])
            if isinstance(exp, tuple): exp = exp[0]
            expf = np.asarray(exp).reshape(-1)
            m = ~np.isnan(expf) & ~np.isnan(got)
            rel = float(np.max(np.abs(got[m] - expf[m]) / np.maximum(np.abs(expf[m]), 1e-300))) if m.any() else 0.0
            nanmis = int((np.isnan(got) != np.isnan(expf)).sum())
            rec["parity_check"] = {"series": int(Sc), "groups": int(G), "windows": int(T), "max_rel_err": rel, "tolerance": 1e-9,
                                   "within_tolerance": bool(rel <= 1e-9 and nanmis == 0), "nan_mismatches": nanmis,
                                   "against": "oracle (C++ restatement of ChunkedRateFunction + SumRowAggregator) on the same chunk bytes"}
            tab2.free(); del arena
        except Exception as e:
            rec["parity_check"] = {"error": repr(e)}
    return rec


def gen_hist_series_np(seed, gid, rows, nb, reset_period):
    """numpy model of the device histogram generator (hist_row in filodb_b200/csrc/synth_kernels.cu): cumulative bucket counts [rows, nb]."""
    with np.errstate(over="ignore"):
        key = _splitmix64_np(np.uint64(seed) ^ (np.uint64(gid) * np.uint64(0xD1342543DE82EF95)))
        r = np.arange(rows, dtype=np.uint64)
        h = _splitmix64_np(key + (r << np.uint64(3)) + np.uint64(7))
    inc = 1 + (h % np.uint64(3)).astype(np.int64)
    obs = np.zeros((rows, nb), np.int64)
    obs[np.arange(rows), (np.arange(rows) + gid) % nb] = inc
    cnt = np.cumsum(obs, axis=0)
    if reset_period > 0 and gid % reset_period == 0:
        r0 = (rows * 5) // 8
        cnt[r0:] = np.cumsum(obs[r0:], axis=0)
    return np.cumsum(cnt, axis=1)


def run_c4(args, rank, world, local_rank):
    """C4: histogram_quantile(0.99, sum(rate(h[5m]))) over SectDelta histogram series, 20 custom buckets 2 * 3^i, +Inf
    (gateway/.../TestTimeseriesProducer.scala:229-235).  The table is generated AND encoded on the device (filo_synth_hist_table: the same
    SectDelta encoder an ingest batch goes through); the query path is filo_query_hist.  The oracle only appears in the cpu_baseline /
    parity_check leg."""
    import torch
    import filodb_b200.capi as capi
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    S = min(args.series, 1_000_000)
    K = min(S, 2048)
    nb = 20
    bdef, bfmt = capi.custom_bucket_def([2.0 * 3 ** i for i in range(nb - 1)] + [float("inf")])      # TestTimeseriesProducer.scala:229-235
    ctx = capi.Context(local_rank)
    t_gen = time.perf_counter()
    tab = ctx.synth_hist_table(S, ROWS, bdef, bfmt, nb, rows_per_chunk=ROWS_PER_CHUNK, t0_ms=T0_MS, interval_ms=INTERVAL, reset_period=97, seed=42, series_id_base=rank * S)
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t_gen
    ti = tab.info()
    start, step, end, window = T0_MS, STEP, T0_MS + 7200000, WINDOW
    T = capi.num_windows(start, step, end)

    last = {}

    def one():
        last["quantile"] = ctx.query_hist(tab, capi.FN_RATE, start, step, end, window, aggr=capi.AGG_SUM, quantile=0.99, want_values=False)
        return ctx.last_stats
    st0 = one()
    assert st0["samples_scanned"] == ti.n_samples, (st0, ti.n_samples)
    sampler = ClockSampler(local_rank); sampler.start()
    for _ in range(args.warmup): one()
    if dist: dist.barrier()
    torch.cuda.synchronize(); sampler.mark_start()
    kns = [one()["kernel_ns"] for _ in range(args.steps)]          # device time of the step's kernels (CUDA events on the launching stream)
    torch.cuda.synchronize()
    if dist: dist.barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"quantile": (last["quantile"], None)})      # [groups x T], histogram_quantile(0.99, ...)
    ms = float(np.sum(kns)) / 1e6 / args.steps
    if dist:
        t = torch.tensor([ms], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
    peak, peak_src = measured_peak()
    alg_bytes = ti.algorithmic_bytes + T * 8
    kern_ms = float(np.median(kns)) / 1e6
    line = {"metric": "samples/s scanned+aggregated (rate over 10M series); % HBM roofline", "value": ti.n_samples * world / (ms / 1e3), "unit": "samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "i64 bucket counts -> f64 rates", "data": "synthetic",
            "config": {"workload": "C4: %d histogram series x 2h@15s (480 rows, chunks 400+80), SectDelta vectors encoded on the device, 20 custom buckets 2*3^i .. +Inf, "
                                   "histogram_quantile(0.99, sum(rate(h[5m]))) step 15s, T=%d (per GPU; shards are independent, no cross-GPU merge)" % (S, T),
                       "series_per_gpu": S, "rows": ROWS, "windows": T, "buckets": nb, "window_ms": window, "step_ms": step,
                       "l2": "inputs (%.1f GB arena) larger than the 126 MB L2" % (ti.arena_bytes / 1e9), "table_gen_s": round(t_gen, 2)},
            "gpu_launches": int(st0["kernel_launches"]) * args.steps, "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": alg_bytes / (kern_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg_bytes / (kern_ms / 1e3) / 1e9 / peak,
                         "traffic": None, "kernel": "hist_scan_kernel (+ hist_merge_kernel)", "kernel_ms": kern_ms, "algorithmic_bytes": alg_bytes, "peak_source": peak_src}}
    # end to end: load (host gather + H2D) + query + quantile read-back per step, bounded number of series
    if not args.no_e2e:
        Se = min(S, 200_000 if args.e2e_series < 0 else args.e2e_series)
        harena, hrec_off = tab.read_arena(0, Se)                      # host mirror of the chunk memory a shard would hold off-heap
        nche, addrse, hkeep = host_chunk_infos(harena, hrec_off, Se)
        def e2e_step():
            tb = ctx.load_series(nche, addrse, schema_flags=capi.SCHEMA_CUMULATIVE)
            ctx.query_hist(tb, capi.FN_RATE, start, step, end, window, aggr=capi.AGG_SUM, quantile=0.99, want_values=False)
            tb.free()
        e2e_step()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps): e2e_step()
        dt = (time.perf_counter() - t0) / args.e2e_steps
        line["e2e"] = {"value": Se * ROWS * world / dt, "unit": "samples/s", "h2d_bytes_per_step": int(ti.arena_bytes * Se / S), "d2h_bytes_per_step": T * 8,
                       "s_per_step": dt, "series_per_gpu": Se, "what": "filo_load_series + filo_query_hist + filo_table_free per step"}
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import hist as H, oracle as o
        b = H.Buckets.custom([2.0 * 3 ** i for i in range(nb - 1)] + [float("inf")])
        st = H.HistStore(b)
        ts = T0_MS + np.arange(ROWS, dtype=np.int64) * INTERVAL
        for s_ in range(K):                                           # the first K series of the device table, rebuilt from the generator's model
            st.add_series(ts, gen_hist_series_np(42, s_, ROWS, nb, 97), [ROWS_PER_CHUNK, ROWS - ROWS_PER_CHUNK])
        t0 = time.perf_counter()
        st.query(o.FN_RATE, start, step, end, window, aggr=True, group_ids=np.zeros(K, np.int32), n_groups=1, q=0.99)
        dtc = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": K * ROWS / dtc, "unit": "samples/s", "cores": 1, "kind": "port",
                                "sample": "%d of %d series (%.1f s on 1 thread); C++ restatement of ChunkedWindowIteratorH + HistRateFunction + HistSum + quantile" % (K, S, dtc)}
        # ---- parity at bench scale (outside the timed region): the K distinct series as one group, fused sum + quantile against the oracle
        try:
            avals, aempty, aq = st.query(o.FN_RATE, start, step, end, window, aggr=True, group_ids=np.zeros(K, np.int32), n_groups=1, q=0.99)
            tabk = ctx.synth_hist_table(K, ROWS, bdef, bfmt, nb, rows_per_chunk=ROWS_PER_CHUNK, t0_ms=T0_MS, interval_ms=INTERVAL, reset_period=97, seed=42, series_id_base=0)
            gv, gq = ctx.query_hist(tabk, capi.FN_RATE, start, step, end, window, aggr=capi.AGG_SUM, quantile=0.99)
            tabk.free()
            live = ~aempty.reshape(-1)
            gv2 = np.asarray(gv).reshape(-1, nb)[live]; av2 = avals.reshape(-1, nb)[live]
            rel = np.abs(gv2 - av2) / np.maximum(np.abs(av2), 1e-300)
            qrel = np.abs(np.asarray(gq).reshape(-1)[live] - aq.reshape(-1)[live]) / np.maximum(np.abs(aq.reshape(-1)[live]), 1e-300)
            line["parity_check"] = {"series": int(K), "windows": int(T), "buckets": nb, "cells": int(rel.size), "max_rel_err_sum": float(rel.max()) if rel.size else 0.0,
                                    "max_rel_err_quantile": float(qrel.max()) if qrel.size else 0.0, "tolerance": 1e-9,
                                    "within_tolerance": bool((rel.max() if rel.size else 0.0) <= 1e-9 and (qrel.max() if qrel.size else 0.0) <= 1e-9),
                                    "nan_mismatches": int((np.isnan(np.asarray(gq).reshape(-1)) != np.isnan(aq.reshape(-1))).sum()),
                                    "against": "oracle: HistSumRowAggregator fold (copy + MutableHistogram.add per series) + Histogram.quantile; the device folds the same way inside work items and across them"}
        except Exception as e:
            line["parity_check"] = {"error": repr(e)}
    if rank == 0:
        print(json.dumps(line), flush=True)
    tab.free()
    if dist: dist.destroy_process_group()


def main():
    global ROWS
    args = parse_args()
    if args.workload == "c1":                       # BASELINE configs[0]: 1k series x 1h@15s
        ROWS = 240
        args.series = min(args.series, 1000)
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.workload == "c4":
        run_c4(args, rank, world, local_rank)
        return
    import torch
    import filodb_b200.capi as capi
    from filodb_b200 import shard
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    synth, fn_name, aggr_name, n_groups, desc = WORKLOADS[args.workload]
    fn, aggr = getattr(capi, fn_name), getattr(capi, aggr_name)
    S = args.series
    ctx = capi.Context(local_rank)
    t_gen = time.perf_counter()
    tab = ctx.synth_table(S, ROWS, ROWS_PER_CHUNK, T0_MS, INTERVAL, n_groups=n_groups, seed=42, series_id_base=rank * S, **synth)
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t_gen
    ti = tab.info()
    start, step, end, window = query_range(args.workload)
    T = capi.num_windows(start, step, end)
    # a non-default torch stream made current: the kernels are launched on it (its handle goes through the C-ABI), the
    # timing events are recorded on it, and NCCL collectives issued by torch.distributed are ordered on it as well
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0
    if aggr == capi.AGG_NONE:
        out = torch.empty(S * T, dtype=torch.float64, device="cuda"); aux = None
        out_bytes = S * T * 8
        flags = 0
    else:
        out = torch.empty(n_groups * T, dtype=torch.float64, device="cuda")
        aux = torch.empty(n_groups * T, dtype=torch.int64, device="cuda")
        final = torch.empty(n_groups * T, dtype=torch.float64, device="cuda")
        out_bytes = n_groups * T * 8
        flags = capi.Q_PARTIAL if world > 1 else 0

    def step_fn():
        ctx.query_device(tab, fn, start, step, end, window, out.data_ptr(), aux.data_ptr() if aux is not None else 0,
                         aggr=aggr, flags=flags, stream=stream, want_stats=False)
        if aggr != capi.AGG_NONE and world > 1:      # the one cross-shard exchange of the plan (ReduceAggregateExec)
            shard.merge_partials(out, aux, aggr, dist)
            ctx.present_partials(aggr, n_groups * T, out.data_ptr(), aux.data_ptr(), final.data_ptr(), stream=stream)

    # kernel-only duration of the dominant kernel (for the roofline) via the library's own CUDA events
    st = ctx.query_device(tab, fn, start, step, end, window, out.data_ptr(), aux.data_ptr() if aux is not None else 0,
                          aggr=aggr, flags=flags, stream=stream, want_stats=True)
    assert st["samples_scanned"] == ti.n_samples, (st, ti.n_samples)
    sampler = ClockSampler(local_rank); sampler.start()      # started before the warm-up: nothing spins up inside the timed region
    for _ in range(args.warmup):
        step_fn()
    torch.cuda.synchronize()
    kern_ns = []
    for _ in range(3):
        kern_ns.append(ctx.query_device(tab, fn, start, step, end, window, out.data_ptr(), aux.data_ptr() if aux is not None else 0,
                                        aggr=aggr, flags=flags, stream=stream, want_stats=True)["kernel_ns"])
    if dist: dist.barrier()
    torch.cuda.synchronize()
    sampler.mark_start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_fn()
    e1.record()
    torch.cuda.synchronize()
    if dist: dist.barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        # what a caller of the step receives: the [series x T] rates of this rank's series, or the presented [groups x T] aggregate
        res = out.view(S, T) if aggr == capi.AGG_NONE else (final if world > 1 else out).view(n_groups, T)
        rows = dump_row_sample(res.shape[0], T * 8)
        dump_outputs(args.dump_outputs, {"values": (host_rows(res, rows), rows)})
    ms = e0.elapsed_time(e1) / args.steps
    ms_per_rank = [ms]
    if dist:
        tl = [torch.zeros(1, device="cuda") for _ in range(world)]
        dist.all_gather(tl, torch.tensor([ms], device="cuda", dtype=torch.float32))
        ms_per_rank = [float(x.item()) for x in tl]
        ms = max(ms_per_rank)
    samples_step = ti.n_samples * world
    value = samples_step / (ms / 1e3)
    peak, peak_src = measured_peak()
    alg_bytes = ti.algorithmic_bytes + (S * 4 if aggr != capi.AGG_NONE else 0) + out_bytes
    kern_ms = float(np.median(kern_ns)) / 1e6
    achieved = alg_bytes / (kern_ms / 1e3) / 1e9
    launches_per_step = int(st["kernel_launches"])
    traffic = measured_traffic(args.workload, S)

    line = {"metric": "samples/s scanned+aggregated (rate over 10M series); % HBM roofline", "value": value, "unit": "samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": desc.format(S=S) + " (per GPU; series sharded by id across GPUs)", "series_per_gpu": S, "rows": ROWS, "windows": T,
                       "window_ms": window, "step_ms": step, "l2": "inputs (%.1f GB arena) far larger than the 126 MB L2; no flush needed" % (ti.arena_bytes / 1e9),
                       "table_gen_s": round(t_gen, 2), "arena_bytes": ti.arena_bytes},
            "gpu_launches": launches_per_step * args.steps,
            "ms_per_rank": [round(x, 3) for x in ms_per_rank],
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "kernel": "scan_wp_*_kernel (warp-pipeline scan, scan_wp.cuh / scan_wp_ctr.cuh; + v2 fallback pass over declined series" + ("" if aggr == capi.AGG_NONE else " + merge_partials") + ")",
                         "kernel_ms": kern_ms, "algorithmic_bytes": alg_bytes, "peak_source": peak_src}}

    # ---- end-to-end through the C-ABI with host buffers (load + query + result read-back every step)
    del out
    torch.cuda.empty_cache()
    if args.workload == "c2" and not args.no_c5:
        try:
            line["c5"] = run_c5_sub(args, ctx, rank, world, dist, stream, peak)
        except Exception as e:
            line["c5"] = {"error": repr(e)}
    if not args.no_e2e:
        # default: all series on one GPU; with several ranks on one host each rank takes a 1/world share (the host gather, the pinned
        # result buffers and PCIe are shared by the ranks of a box)
        Se = (S if world == 1 else max(1_000_000, S // world)) if args.e2e_series < 0 else min(S, args.e2e_series)
        os.environ.setdefault("FILO_HOST_THREADS", str(max(4, min(64, host_cores()["cores_usable"] // world))))   # host gather threads per rank
        arena, rec_off = tab.read_arena(0, Se)
        nch, addrs, keep = host_chunk_infos(arena, rec_off, Se)
        n_out = Se * T if aggr == capi.AGG_NONE else n_groups * T
        hout = torch.empty(n_out, dtype=torch.float64).pin_memory()
        hout_np = hout.numpy()
        gids = None
        if n_groups:
            gids = synth_group_ids(42, rank * S, Se, n_groups)
        import ctypes as C
        L = capi.lib()

        def e2e_step():
            st_ = capi.Stats()
            if aggr == capi.AGG_NONE:      # per-series result: one pipelined call (gather / H2D / kernels / D2H of consecutive batches overlap)
                ctx._check(L.filo_scan_series(ctx.h, Se, nch.ctypes.data_as(C.c_void_p), addrs.ctypes.data_as(C.c_void_p), 0, 1, synth.get("schema_flags", 0),
                                              fn, start, step, end, window, hout_np.ctypes.data_as(C.c_void_p), C.byref(st_)))
                return
            h = C.c_void_p()
            ctx._check(L.filo_load_series(ctx.h, Se, nch.ctypes.data_as(C.c_void_p), addrs.ctypes.data_as(C.c_void_p), 0, 1,
                                          gids.ctypes.data_as(C.c_void_p) if gids is not None else None, n_groups, synth.get("schema_flags", 0), C.byref(h)))
            ctx._check(L.filo_query(ctx.h, h, fn, start, step, end, window, aggr, 0, 0, hout_np.ctypes.data_as(C.c_void_p), None, C.byref(st_)))
            L.filo_table_free(ctx.h, h)
        # one-time set-up, like FiloDB mapping its off-heap block memory at start-up: the region that holds the chunk vectors is
        # registered (pinned + mapped), so the per-step host->device transfer of the inputs is a device-side gather over PCIe
        registered = False
        if aggr == capi.AGG_NONE and not args.e2e_staged:
            ctx.host_register(arena); registered = True
        e2e_step()
        if dist: dist.barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            e2e_step()
        dt = (time.perf_counter() - t0) / args.e2e_steps
        if dist:
            t = torch.tensor([dt], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); dt = float(t.item())
        line["e2e"] = {"value": Se * ROWS * world / dt, "unit": "samples/s", "h2d_bytes_per_step": int(arena.size), "d2h_bytes_per_step": int(n_out * 8),
                       "s_per_step": dt, "steps": args.e2e_steps, "series_per_gpu": Se,
                       "what": (("filo_scan_series over registered (pinned, mapped) chunk memory: walk ChunkSetInfo blocks on the host, device-side gather of the vectors over PCIe, kernels, D2H into a pinned host buffer, pipelined in batches" if registered else "filo_scan_series: walk ChunkSetInfo blocks in host memory, gather into pinned slabs, H2D, kernels, D2H into a pinned host buffer, pipelined in batches")
                                if aggr == capi.AGG_NONE else
                                "filo_load_series (walk ChunkSetInfo blocks in host memory, gather into pinned slabs, H2D) + filo_query (kernels + D2H) + filo_table_free, per step")}
        if registered: ctx.host_unregister(arena)
        # ---- the same query against the RESIDENT table (an incremental arena keeps a shard's chunks on the device, filo_table_append):
        # no input crosses PCIe, the result is read back into the pinned host buffer every step
        if aggr == capi.AGG_NONE and Se == S:
            try:
                def res_step():
                    st_ = capi.Stats()
                    ctx._check(L.filo_query(ctx.h, tab.h, fn, start, step, end, window, aggr, 0, 0, hout_np.ctypes.data_as(C.c_void_p), None, C.byref(st_)))
                res_step()
                if dist: dist.barrier()
                t0 = time.perf_counter()
                for _ in range(args.e2e_steps): res_step()
                dtr = (time.perf_counter() - t0) / args.e2e_steps
                if dist:
                    t = torch.tensor([dtr], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); dtr = float(t.item())
                line["e2e_resident"] = {"value": Se * ROWS * world / dtr, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": int(n_out * 8), "s_per_step": dtr,
                                        "what": "filo_query over the resident table (chunks already in the device arena, as after filo_table_append): kernels + D2H of the [series x T] result into pinned host memory"}
            except Exception as e_:
                line["e2e_resident"] = {"error": repr(e_)}
        del arena, keep, hout
    # ---- CPU baseline beside it (rank 0, N=1 only): the oracle port on a bounded sample, all host threads
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import oracle as o
        Sc = min(S, args.cpu_series)
        arena, rec_off = tab.read_arena(0, Sc)
        ost = o.Store(); ost.add_from_arena(arena, rec_off, Sc)
        hc = host_cores()
        cores = hc["cores_usable"]
        cumulative = bool(synth.get("schema_flags", 0) & 1)
        gids = None
        if n_groups:
            gids = synth_group_ids(42, 0, Sc, n_groups)
        dts = []
        for _ in range(3):        # first run also pays page faults / allocator warm-up; report the best
            t0 = time.perf_counter()
            exp = ost.query(getattr(o, fn_name), start, step, end, window, cumulative=cumulative, aggr=getattr(o, aggr_name), group_ids=gids,
                            n_groups=max(n_groups, 1), threads=cores, reuse_out=True)
            dts.append(time.perf_counter() - t0)
        dt = min(dts)
        line["cpu_baseline"] = dict({"value": Sc * ROWS / dt, "unit": "samples/s", "cores": cores, "kind": "port",
                                     "sample": "%d of %d series (%.1f s wall on %d threads = usable cores); C++ restatement of ChunkedWindowIteratorD + range functions, not a JVM number" % (Sc, S, dt, cores)}, **hc)
        # ---- parity at bench scale (outside every timed region): the oracle's answer for these Sc series against the CUDA path on a table
        # of the same Sc series (same generator, same seed): bit-exact per series, 1e-9 relative for across-series aggregates
        try:
            tab2 = ctx.synth_table(Sc, ROWS, ROWS_PER_CHUNK, T0_MS, INTERVAL, n_groups=n_groups, seed=42, series_id_base=0, **synth)
            got = ctx.query(tab2, fn, start, step, end, window, aggr=aggr)
            if isinstance(got, tuple): got = got[0]
            if isinstance(exp, tuple): exp = exp[0]
            got = np.asarray(got).reshape(-1); expf = np.asarray(exp).reshape(-1)
            if aggr == capi.AGG_NONE:
                bad = 0
                CH = 1 << 26
                for i0 in range(0, got.size, CH):
                    a = got[i0:i0 + CH]; b = expf[i0:i0 + CH]
                    if not np.array_equal(a.view(np.uint64), b.view(np.uint64)):
                        bad += int((~((a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b)))).sum())
                line["parity_check"] = {"series": int(Sc), "windows": int(T), "values": int(got.size), "bit_exact": bad == 0, "mismatches": bad,
                                        "against": "oracle (C++ restatement of the reference path) on the same chunk bytes"}
            else:
                nanmis = int((np.isnan(got) != np.isnan(expf)).sum())
                m = ~np.isnan(expf) & ~np.isnan(got)
                rel = float(np.max(np.abs(got[m] - expf[m]) / np.maximum(np.abs(expf[m]), 1e-300))) if m.any() else 0.0
                line["parity_check"] = {"series": int(Sc), "groups": int(n_groups), "windows": int(T), "max_rel_err": rel, "tolerance": 1e-9,
                                        "within_tolerance": bool(rel <= 1e-9 and nanmis == 0), "nan_mismatches": nanmis,
                                        "against": "oracle (C++ restatement of the reference path) on the same chunk bytes"}
            tab2.free()
        except Exception as e:      # the check must not take the measurement down; its failure is reported
            line["parity_check"] = {"error": repr(e)}
    tab.free(); ctx.close()
    # ---- the other BASELINE configs beside the headline one (single GPU, default workload only): each runs kernel-only in a child
    # process of this script after this process has released the device memory; their lines are attached as sub-records
    if rank == 0 and world == 1 and args.workload == "c2" and not args.no_extra:
        torch.cuda.empty_cache()
        extra = {}
        for wl, steps in (("c1", 20), ("c3-const", 6), ("c3", 3), ("c4", 4)):
            try:
                cmd = [sys.executable, os.path.abspath(__file__), "--workload", wl, "--steps", str(steps), "--warmup", "3", "--no-e2e", "--no-c5", "--no-extra", "--no-cpu"]
                r = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
                d = json.loads(r.stdout.strip().splitlines()[-1])
                extra[wl] = {"workload": d["config"]["workload"], "value": d["value"], "unit": d["unit"], "ms_per_step": d["ms_per_step"], "steps": d["steps"],
                             "roofline": {k: d["roofline"].get(k) for k in ("achieved", "peak", "frac", "kernel_ms", "algorithmic_bytes", "kernel")},
                             "parity_check": d.get("parity_check")}
            except Exception as e_:
                extra[wl] = {"error": repr(e_)}
        line["other_configs"] = extra
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist: dist.destroy_process_group()


if __name__ == "__main__":
    main()
