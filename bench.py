#!/usr/bin/env python3
"""bench.py -- the hot path of BASELINE.json on N B200s of one node.

Workload (BASELINE.json configs[1], the configuration `metric` is quoted on for one GPU):
  decode 100 000 blocks (8192 samples each; timestamps delta-const, values ZSTD nearest-delta2 counters at scale -2,
  rare resets) + rate(m[5m]) at step 15 s  ->  [100 000 x 8172] float64.
The blocks are marshaled by the REFERENCE encoder (oracle restatement of marshalInt64Array + the reference's own libzstd
1.5.7 at getCompressLevel): the bytes a vmstorage part holds.  `--encoder library` marshals the same values with the
library's own encoder instead (reported beside the default as `alt_encoder`).
One "step" = one pass of the hot path over that batch.  N > 1: every rank owns its own 100 000 blocks (series shard by
TSID, no data-path collective; SURVEY.md 8e) -> weak scaling.

  value : samples/s with the compressed blocks already resident in HBM (device-timed, CUDA events, max over ranks)
  e2e   : the same through the public host-buffer call (vmb_eval_rollup_host): H2D of descriptors+payload from pinned
          host memory, decode, rollup, D2H of the result, all inside the timed region
  roofline : the dominant kernel stage, algorithmic bytes / measured stage time vs MEASURED_PEAKS.json
  cpu_baseline : the oracle (C++ restatement of the Go path, zstd through the reference's own libzstd when
          oracle/_ref is present) on a persistent pool of host threads over the SAME blocks  (rank 0, N = 1)
  aggr  : sum(rate(m[5m])) by (label) into 8 and 1024 groups; N > 1: the per-GPU partial states are merged by the
          library's own NCCL all-reduce (vmb_comm_*), no Python in the data path
  configs2 : (N = 1) BASELINE.json configs[2] and the north-star size: 1 M series x 8192 samples on one GPU --
          rate() over counters, avg/max/quantile_over_time(0.99) over gauges

  --impl reference : times the reference's CPU implementation of the path (see cpu_baseline) on the same config.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T0 = 1_700_000_000_000
SCRAPE_MS = 15000
SCALE = -2
KIND_ID = {"counter": 0, "gauge": 1, "mixed": 2}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--blocks", type=int, default=100_000, help="blocks (= series) per GPU")
    ap.add_argument("--rows", type=int, default=8192)
    ap.add_argument("--func", default="rate")
    ap.add_argument("--ts", default="regular", choices=["regular", "jitter"],
                    help="timestamps: regular = t0 + 15 s * i (one shared MarshalTypeDeltaConst payload, configs[1]); jitter = "
                         "every series has its own +-50 ms scrape jitter (zstd nearest-delta2 timestamp columns)")
    ap.add_argument("--kind", default="counter", choices=["counter", "gauge", "mixed"],
                    help="synthetic values: counter = configs[1] (default), gauge = configs[2]-style round(N(5000,300)) at "
                         "scale -2, mixed = configs[4]-style 40%% counters / 30%% gauges / 20%% const / 10%% delta-const")
    ap.add_argument("--encoder", default="reference", choices=["reference", "library"],
                    help="who marshals the synthetic blocks: reference = oracle marshalInt64Array + the reference's libzstd 1.5.7 "
                         "(what a vmstorage part holds); library = the product's own encoder (Huffman-only zstd frames)")
    ap.add_argument("--window-ms", type=int, default=300_000)
    ap.add_argument("--step-ms", type=int, default=15_000)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-aggr", action="store_true", help="skip the sum(rate) by (label) sub-record")
    ap.add_argument("--no-alt-encoder", action="store_true", help="skip the library-encoded run reported beside the default")
    ap.add_argument("--configs2-series", type=int, default=-1,
                    help="series of the configs[2] sub-record (1 M x 8192 on one GPU); -1 = 1 000 000 at N = 1 with the default "
                         "workload, 0 = off")
    ap.add_argument("--parity-series", type=int, default=1000, help="series of the timed batch compared with the oracle (rank 0)")
    ap.add_argument("--aggr", default="", help="run ONLY aggr(func(m[d])) by (label) as the main record, e.g. --aggr sum")
    ap.add_argument("--groups", type=int, default=1000, help="label groups for --aggr")
    ap.add_argument("--cpu-seconds", type=float, default=2.0, help="minimum wall time of the cpu_baseline measurement (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the result of the last one (rank 0) to DIR as float64 .npy files: "
                         "result.npy (rows of the [series or groups x points] result, a fixed seeded sample when it exceeds "
                         "%d MB), result_rows.npy (their row indices) and samples_scanned.npy" % (DUMP_BYTES // 1_000_000))
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


DUMP_BYTES = 60_000_000  # result.npy stays below this; the three files of --dump-outputs stay below 64 MB


def dump_outputs(dirname, rows_of, nrows, ncols, scanned):
    """--dump-outputs: writes rows of a [nrows x ncols] result (rows_of(idx) -> float array) to DIR/result.npy.  The row
    sample depends only on the shape, so two builds run with the same arguments write files that compare row for row."""
    k = min(nrows, max(1, DUMP_BYTES // (8 * ncols)))
    idx = np.arange(nrows) if k == nrows else np.sort(np.random.default_rng(0).choice(nrows, size=k, replace=False))
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "result.npy"), np.asarray(rows_of(idx), dtype=np.float64))
    np.save(os.path.join(dirname, "result_rows.npy"), idx.astype(np.float64))
    np.save(os.path.join(dirname, "samples_scanned.npy"), np.array([scanned], dtype=np.float64))


# ------------------------------------------------------------------------------------------------ oracle side (input + CPU arm)
def oracle():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    L = O.lib()
    if not getattr(L, "_bench_sigs", False):
        vp, sz = C.c_void_p, C.c_size_t
        L.vmo_pool_create.restype = vp
        L.vmo_pool_create.argtypes = [C.c_int]
        L.vmo_pool_destroy.restype = None
        L.vmo_pool_destroy.argtypes = [vp]
        L.vmo_pool_threads.argtypes = [vp]
        L.vmo_pool_eval_rollup.restype = C.c_int
        L.vmo_pool_eval_rollup.argtypes = [vp, vp, sz, O.u8p, C.c_int64, C.c_int64, C.POINTER(O.RollupCfg), C.c_int, C.c_int, O.f64p,
                                           C.POINTER(C.c_uint64), C.c_int]
        L.vmo_pool_gen_blocks.restype = C.c_int64
        L.vmo_pool_gen_blocks.argtypes = [vp, C.c_int, C.c_int, sz, sz, C.c_uint64, C.c_int64, C.c_int64, C.c_int16, vp, O.u8p, sz,
                                          C.POINTER(C.c_uint64)]
        L.vmo_pool_gen_values.restype = C.c_int
        L.vmo_pool_gen_values.argtypes = [vp, C.c_int, sz, sz, sz, C.c_uint64, O.i64p]
        L._bench_sigs = True
    return O, L


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def numa_layout():
    out = []
    try:
        base = "/sys/devices/system/node"
        for n in sorted(d for d in os.listdir(base) if d.startswith("node") and d[4:].isdigit()):
            with open(os.path.join(base, n, "cpulist")) as f:
                out.append("%s: cpus %s" % (n, f.read().strip()))
    except Exception:
        pass
    return "; ".join(out) or "unknown"


_POOLS = {}
try:
    _AFFINITY0 = os.sched_getaffinity(0)
except Exception:
    _AFFINITY0 = None


def get_pool(nthreads):
    """persistent worker pool of the oracle (created once, outside every timed region)"""
    O, L = oracle()
    if nthreads not in _POOLS:
        # worker threads inherit the creating thread's CPU mask: create them under the process' original mask, not under the
        # GPU-local one the main thread wears while it allocates pinned buffers (a 64-thread pool born there would sit on 32 cores)
        cur = None
        try:
            cur = os.sched_getaffinity(0)
            if _AFFINITY0 and cur != _AFFINITY0:
                os.sched_setaffinity(0, _AFFINITY0)
        except Exception:
            cur = None
        try:
            _POOLS[nthreads] = C.c_void_p(L.vmo_pool_create(nthreads))
        finally:
            if cur is not None and _AFFINITY0 and cur != _AFFINITY0:
                try:
                    os.sched_setaffinity(0, cur)
                except Exception:
                    pass
    return _POOLS[nthreads]


# ------------------------------------------------------------------------------------------------ synthetic input
def gen_blocks(nblocks, rows, seed, kind="counter", ts_kind="regular", encoder="reference"):
    """node_cpu_seconds_total-like counters (SURVEY.md 8d config 2) / gauges / the configs[4] mix, generated and marshaled
    series by series on host threads (oracle/cpu_pipeline.cpp vmo_pool_gen_blocks).
    -> (descs structured array, payload np.uint8, stats dict)"""
    from victoriametrics_b200 import encoding, storage
    O, L = oracle()
    pool = get_pool(host_threads())
    stats = (C.c_uint64 * 4)()
    if encoder == "reference":
        if not L.vmo_zstd_ref_available():
            raise RuntimeError("oracle/_ref/libzstd_ref.so is missing: build it in the container that holds /root/reference "
                               "(python -c 'import __graft_entry__ as g; g.build()'), or run with --encoder library")
        descs = np.zeros(nblocks, dtype=storage.DESC_DTYPE)
        per_row = 3 * (2 if ts_kind == "jitter" else 1)
        while True:
            cap = nblocks * rows * per_row + (1 << 20)
            payload = np.empty(cap, dtype=np.uint8)
            n = L.vmo_pool_gen_blocks(pool, KIND_ID[kind], 1 if ts_kind == "jitter" else 0, nblocks, rows, seed, T0, SCRAPE_MS, SCALE,
                                      descs.ctypes.data, payload.ctypes.data_as(O.u8p), cap, stats)
            if n == -101 and per_row < 40:  # VMO_ERR_CAP
                per_row *= 2
                continue
            if n < 0:
                raise RuntimeError("vmo_pool_gen_blocks failed: %d" % n)
            break
        payload = payload[:n]
    else:
        # the same values (same per-series RNG streams), marshaled by the product's own encoder through its C ABI
        ts = T0 + SCRAPE_MS * np.arange(rows, dtype=np.int64)
        tdata, tmt, tfirst = encoding.marshal_timestamps(ts)
        pieces, pos = [tdata], tdata.size
        cols = {k: [] for k in ("first_value", "val_off", "val_size", "val_mt", "ts_off", "ts_size", "ts_mt", "min_ts", "max_ts")}
        rng = np.random.default_rng(seed)
        chunk = 4000
        for c0 in range(0, nblocks, chunk):
            n = min(chunk, nblocks - c0)
            v = np.empty((n, rows), dtype=np.int64)
            rc = L.vmo_pool_gen_values(pool, KIND_ID[kind], c0, n, rows, seed, v.ctypes.data_as(O.i64p))
            assert rc == 0, rc
            if ts_kind == "jitter":
                tj = ts[None, :] + rng.integers(-50, 51, (n, rows))
                tp_, toffs, tmts, tfirsts = encoding.marshal_columns(tj)
                pieces.append(tp_)
                cols["ts_off"].append(toffs[:-1] + pos)
                cols["ts_size"].append(np.diff(toffs).astype(np.uint32))
                cols["ts_mt"].append(tmts)
                cols["min_ts"].append(tfirsts)
                cols["max_ts"].append(tj[:, -1].copy())
                pos += tp_.size
            p_, offs, mts, firsts = encoding.marshal_columns(v)
            pieces.append(p_)
            cols["first_value"].append(firsts)
            cols["val_off"].append(offs[:-1] + pos)
            cols["val_size"].append(np.diff(offs).astype(np.uint32))
            cols["val_mt"].append(mts)
            pos += p_.size
            dropped = np.diff(v, axis=1) < 0
            has = dropped.any(axis=1)
            stats[1] += int(np.count_nonzero(has))
            stats[3] += int((rows - ((np.argmax(dropped, axis=1)[has] + 1) & ~127)).sum())
        stats[0], stats[2] = nblocks, nblocks * rows
        tcols = dict(min_ts=tfirst, max_ts=int(ts[-1]), ts_off=0, ts_size=tdata.size, ts_mt=tmt)
        if ts_kind == "jitter":
            tcols = {k: np.concatenate(cols[k]) for k in ("min_ts", "max_ts", "ts_off", "ts_size", "ts_mt")}
        descs = storage.descs_from_arrays(
            first_value=np.concatenate(cols["first_value"]), val_off=np.concatenate(cols["val_off"]),
            val_size=np.concatenate(cols["val_size"]), rows=np.full(nblocks, rows, dtype=np.uint32),
            series_idx=np.arange(nblocks, dtype=np.uint32), scale=SCALE, val_mt=np.concatenate(cols["val_mt"]), precision_bits=64,
            **tcols)
        payload = np.concatenate(pieces)
    st = {"series": int(stats[0]), "series_with_drop": int(stats[1]), "rows": int(stats[2]), "rows_from_first_drop": int(stats[3])}
    return descs, payload, st


def compressed_bytes(descs, ts_kind):
    return int(descs["val_size"].sum()) + (int(descs["ts_size"].sum()) if ts_kind == "jitter" else int(descs["ts_size"][0]))


def query_range(rows, window_ms, step_ms):
    start = T0 + window_ms
    end = T0 + SCRAPE_MS * (rows - 1)
    return start, end, step_ms


RCR_FUNCS = ("rate", "increase", "irate", "increase_pure", "increase_prometheus", "rate_prometheus", "rollup_rate", "rollup_increase")

# ------------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    """SM clock / throttle reasons / power sampled DURING the timed region: NVML in-process every ~2 ms (the timed region of
    the device-resident arm is < 100 ms), `nvidia-smi -lms` as the fallback"""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index, pci_bus_id=None):
        self.gpu = gpu_index
        self.pci = pci_bus_id
        self.rows = []   # (time, sm_mhz, max_mhz, power_w, [reasons])
        self.proc = None
        self.nvml = None
        self.stop_flag = False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if self.pci:
                try:
                    h = pynvml.nvmlDeviceGetHandleByPciBusId(self.pci.encode() if isinstance(self.pci, str) else self.pci)
                except Exception:
                    h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.nvml = (pynvml, h)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        pynvml, h = self.nvml
        R = (("hw_slowdown", getattr(pynvml, "nvmlClocksEventReasonHwSlowdown", 0x8)),
             ("hw_thermal_slowdown", getattr(pynvml, "nvmlClocksEventReasonHwThermalSlowdown", 0x40)),
             ("sw_thermal_slowdown", getattr(pynvml, "nvmlClocksEventReasonSwThermalSlowdown", 0x20)),
             ("sw_power_cap", getattr(pynvml, "nvmlClocksEventReasonSwPowerCap", 0x4)))
        get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            try:
                sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                mask = int(get_reasons(h))
                try:
                    pw = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
                except Exception:
                    pw = 0.0
                self.rows.append((time.time(), sm, self.max_mhz, pw, [n for n, bit in R if mask & bit]))
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            r = [x.strip() for x in line.split(",")]
            if len(r) >= 9:
                try:
                    reasons = [n for n, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9])
                               if v.lower().startswith("active")]
                    self.rows.append((time.time(), float(r[1]), float(r[2]), float(r[3]), reasons))
                except ValueError:
                    pass

    def window(self, t_begin, t_end):
        rows = [r for r in self.rows if t_begin <= r[0] <= t_end]
        src = "inside the timed region"
        if not rows:
            rows = [r for r in self.rows if t_begin - 0.2 <= r[0] <= t_end + 0.2]
            src = "within 0.2 s of the timed region"
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(r[1] for r in rows)
        reasons = sorted({n for r in rows for n in r[4]})
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": rows[0][2], "reasons": reasons, "samples": len(rows),
                "power_w_max": round(max(r[3] for r in rows), 1), "sampled": src,
                "via": "nvml" if self.nvml else "nvidia-smi"}

    def stop(self, t_begin=None, t_end=None):
        self.stop_flag = True
        if self.proc:
            time.sleep(0.05)
            self.proc.terminate()
        if t_begin is None:
            return None
        return self.window(t_begin, t_end)


# ------------------------------------------------------------------------------------------------ CPU reference arm
class CpuArm:
    """the oracle's per-series loop (oracle/cpu_pipeline.cpp) over ALL blocks of the batch on a persistent pool of host
    threads: Results.RunParallel + the closure of evalRollupNoIncrementalAggregate (netstorage.go:221, eval.go:1855)"""

    def __init__(self, descs, payload, func, start, end, step, window):
        from rollup_names import RF
        from victoriametrics_b200 import promql
        self.O, self.L = oracle()
        O = self.O
        self.descs, self.payload = descs, payload
        self.rc = promql.get_rollup_configs(func, start, end, step, window)
        self.phis = np.full(self.rc.points, 0.99) if func == "quantile_over_time" else None
        self.cfg = O.RollupCfg(RF[func], start, end, step, window, 0, 0, int(self.rc.MayAdjustWindow), int(self.rc.isDefaultRollup),
                               self.rc.samplesScannedPerCall, self.phis.ctypes.data_as(O.f64p) if self.phis is not None else None, None)
        self.P = self.rc.points
        self.rows = int(descs["rows"][0])
        self.kind = "reference" if self.L.vmo_zstd_ref_available() else "port"
        self.out = None

    def alloc_out(self, nb):
        if self.out is None or self.out.shape[0] < nb:
            self.out = np.empty((nb, self.P), dtype=np.float64)
            self.out.fill(0.0)  # touch the pages outside the timed region (the Go code reuses pooled buffers)
        return self.out

    def run(self, nthreads, nb=None, descs=None, out=None):
        """one pass over the first nb blocks on the pool of `nthreads` threads -> seconds"""
        d = self.descs if descs is None else descs
        nb = len(d) if nb is None else nb
        out = self.alloc_out(nb) if out is None else out
        pool = get_pool(nthreads)
        scanned = C.c_uint64(0)
        t = time.perf_counter()
        r = self.L.vmo_pool_eval_rollup(pool, d.ctypes.data, nb, self.payload.ctypes.data_as(self.O.u8p), -(1 << 63), (1 << 63) - 1,
                                        C.byref(self.cfg), int(self.rc.removeCounterResets), int(self.rc.dropStaleNaNs),
                                        out.ctypes.data_as(self.O.f64p), C.byref(scanned), 1)
        dt = time.perf_counter() - t
        assert r == 0, r
        self.scanned = scanned.value
        return dt

    def thread_candidates(self):
        """one software thread per hardware thread is not always the fastest on a hyper-threaded host: one per two is tried as well"""
        cores = host_threads()
        return [cores, cores // 2] if cores >= 16 else [cores]

    def measure(self, steps=None, min_wall=2.0, warmup=1):
        """-> dict.  EVERY candidate thread count gets `warmup` untimed passes and then `steps` whole passes (or as many as fill min_wall
        seconds, at least 2) timed back to back; the faster count is the one reported -- the baseline gets the benefit of the doubt,
        and both of this file's CPU measurements (cpu_baseline of the library arm, the --impl reference arm) choose the same way"""
        nb = len(self.descs)
        runs = {}
        for nt in self.thread_candidates():
            for _ in range(max(1, warmup)):
                self.run(nt)
            times = []
            t_all = time.perf_counter()
            while True:
                times.append(self.run(nt))
                if steps is not None and len(times) >= steps:
                    break
                if steps is None and len(times) >= 2 and time.perf_counter() - t_all >= min_wall:
                    break
            runs[nt] = (time.perf_counter() - t_all, times)
        nthreads = min(runs, key=lambda k: runs[k][0] / len(runs[k][1]))
        wall, times = runs[nthreads]
        per = wall / len(times)
        return {"value": nb * self.rows / per, "unit": "samples/s", "cores": nthreads, "kind": self.kind,
                "sample": "all %d blocks x %d rows, %d passes back to back in %.2f s wall (%.3f s per pass; min %.3f, max %.3f) on a "
                          "persistent pool of %d threads (C++ restatement of the Go path%s); every thread count tried was timed the "
                          "same way, the fastest is reported" %
                          (nb, self.rows, len(times), wall, per, min(times), max(times), nthreads,
                           "; zstd via the reference's libzstd 1.5.7" if self.kind == "reference" else ""),
                "seconds": wall, "passes": len(times), "ms_per_pass": per * 1e3, "blocks": nb,
                "host_threads_available": host_threads(),
                "thread_counts_tried_s_per_pass": {str(k): round(v[0] / len(v[1]), 4) for k, v in sorted(runs.items())},
                "numa": numa_layout()}


def parity_check(arm, out_rows_fn, nseries, seed=7):
    """full-size parity: `nseries` random series of the timed batch through the oracle (CPU) against the GPU result rows.
    out_rows_fn(idx) -> np.float64[len(idx), P] (rows of the GPU result).  1e-12 relative like tests/ (north_star: 1e-9)."""
    nb = len(arm.descs)
    idx = np.sort(np.random.default_rng(seed).choice(nb, size=min(nseries, nb), replace=False))
    sub = np.ascontiguousarray(arm.descs[idx])
    exp = np.empty((len(idx), arm.P), dtype=np.float64)
    arm.run(min(host_threads(), 32), descs=sub, out=exp)
    got = out_rows_fn(idx)
    both_nan = np.isnan(got) & np.isnan(exp)
    with np.errstate(invalid="ignore", divide="ignore"):
        rel = np.abs(got - exp) / np.maximum(np.abs(exp), 1e-300)
    rel[both_nan] = 0.0
    rel[(got == exp)] = 0.0
    rel[np.isnan(rel)] = np.inf  # NaN on one side only
    worst = float(rel.max()) if rel.size else 0.0
    return {"series": int(len(idx)), "points": int(arm.P), "max_rel_err": worst, "tolerance": 1e-12, "ok": bool(worst <= 1e-12),
            "nan_points": int(both_nan.sum())}

# ------------------------------------------------------------------------------------------------ main
def main():
    a = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    start, end, step = query_range(a.rows, a.window_ms, a.step_ms)
    points = 1 + (end - start) // step
    what = {"counter": "configs[1]: decode %d blocks x %d samples (ts delta-const, values zstd nearest-delta2 counters, scale %d)",
            "gauge": "configs[2]-style: decode %d blocks x %d samples (ts delta-const, values zstd nearest-delta gauges, scale %d)",
            "mixed": "configs[4]-style: decode %d blocks x %d samples (40%% counters, 30%% gauges, 20%% const, 10%% delta-const, scale %d)"}[a.kind]
    if a.ts == "jitter":
        what = what.replace("ts delta-const", "ts zstd nearest-delta2 with +-50 ms jitter")
    workload = (what + " + %s()[%ds] step=%ds per GPU") % (a.blocks, a.rows, SCALE, a.func, a.window_ms // 1000, a.step_ms // 1000)
    enc_note = {"reference": "reference encoder: marshalInt64Array restated by the oracle + the reference's own libzstd 1.5.7 at "
                             "getCompressLevel (what a vmstorage part holds)",
                "library": "the library's own encoder (vmb_marshal_columns: Huffman-only zstd frames)"}[a.encoder]
    base = {"metric": "rollup samples/sec (block decode + %s, raw samples decoded and scanned per second)" % a.func,
            "unit": "samples/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int64 codec -> f64 rollup", "data": "synthetic",
            "config": {"workload": workload, "blocks_per_gpu": a.blocks, "rows_per_block": a.rows, "points_per_series": int(points),
                       "encoder": enc_note,
                       "parallelism": "series sharded by TSID across %d GPU(s), no data-path collective" % a.gpus,
                       "l2": "inputs (>=1.3 GB compressed, 6.5 GB result) exceed the 126 MB L2; no flush needed"}}

    if a.impl == "reference":
        if rank != 0:
            return 0
        t_all = time.perf_counter()
        descs, payload, _ = gen_blocks(a.blocks, a.rows, seed=1234, kind=a.kind, ts_kind=a.ts, encoder=a.encoder)
        arm = CpuArm(descs, payload, a.func, start, end, step, a.window_ms)
        m = arm.measure(steps=a.steps, warmup=a.warmup)  # per thread count: `warmup` untimed passes, then `steps` timed ones
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, lambda idx: arm.out[idx], a.blocks, arm.P, arm.scanned)
        out = dict(base)
        out.update({"impl": "reference", "value": m["value"], "ms_per_step": m["ms_per_pass"],
                    "cpu_baseline": m, "gpu_launches": 0,
                    "e2e": {"value": m["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                    "wall_s": time.perf_counter() - t_all})
        out["config"]["note"] = ("CPU reference arm: every step is one whole pass over the same %d blocks on a persistent thread pool; "
                                 "ms_per_step is measured (wall of the %d timed passes / %d, at the faster of the thread counts tried)" % (a.blocks, a.steps, a.steps))
        print(json.dumps(out))
        return 0

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import victoriametrics_b200 as vm
    from victoriametrics_b200 import _lib, promql, storage
    ctx = vm.Context(local_rank)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)

    t_gen = time.perf_counter()
    descs, payload, gstats = gen_blocks(a.blocks, a.rows, seed=1234 + rank, kind=a.kind, ts_kind=a.ts, encoder=a.encoder)
    gen_s = time.perf_counter() - t_gen
    rows_total = int(a.blocks) * int(a.rows)
    compressed = compressed_bytes(descs, a.ts)

    blocks = storage.Blocks(descs, payload, ctx)
    out_dev = torch.empty((a.blocks, points), dtype=torch.float64, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def time_steps(fn, warmup, steps):
        """W untimed + K timed calls of fn bracketed by barrier + synchronize; CUDA events on the launching stream -> ms per step
        (this rank), launches, wall-clock window"""
        for _ in range(warmup):
            fn()
        barrier()
        l0 = ctx.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tb = time.time()
        e0.record(stream)
        r = None
        for _ in range(steps):
            r = fn()
        e1.record(stream)
        barrier()
        return e0.elapsed_time(e1) / steps, ctx.launch_count - l0, (tb, time.time()), r

    def max_over_ranks(*xs):
        t = torch.tensor([float(x) for x in xs], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    func_args = np.full(points, 0.99) if a.func == "quantile_over_time" else None  # quantile_over_time(0.99, m[d])

    def dev_step():
        return promql.eval_rollup_func(a.func, blocks, start, end, step, a.window_ms, args=func_args, out_dev_ptr=out_dev.data_ptr())

    # aggr(rollup) by (label): every rank folds its own series into [groups x points] partial states; N > 1: merged by an
    # NCCL all-reduce of values and counts (SURVEY.md 8e); every rank finalizes; the [groups x points] result goes to the host
    rc_aggr = promql.get_rollup_configs(a.func, start, end, step, a.window_ms)

    class Buf:
        def __init__(self, nbytes):
            self.t = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
            self.ptr = self.t.data_ptr()

    # N > 1: the library's own NCCL communicator (csrc/comm.inc); torch.distributed only carries the 128-byte unique id
    if world > 1:
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(vm.Context.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        ctx.comm_init(bytes(uid.cpu().numpy().tobytes()), world, rank)

    def make_aggr(aggr, groups):
        group_ids = ((np.arange(a.blocks, dtype=np.int64) * world + rank) % groups).astype(np.uint32)
        h = _lib.lib().vmb_host_alloc(groups * points * 8)
        assert h, "pinned host allocation failed"
        res = np.ctypeslib.as_array(C.cast(h, C.POINTER(C.c_double)), shape=(groups, points))

        def aggr_step():
            # one library call: fold this rank's series on the GPU, all-reduce {values, counts} over NCCL, finalize, D2H of the result
            _, scanned_ = promql.eval_rollup_aggr_dist(aggr, a.func, blocks, group_ids, groups, start, end, step, a.window_ms,
                                                       args=func_args, out=res)
            return None, scanned_
        ia = promql.IncrementalAggr(aggr, groups, points, Buf) if not a.no_e2e and a.aggr else None
        reduce_cb = (lambda v, c, op: check_rc(_lib.lib().vmb_aggr_allreduce(ctx.h, promql.AGGR_FUNCS[aggr], C.c_void_p(v.ptr), C.c_void_p(c.ptr),
                                                                            groups * points))) if world > 1 else None
        return aggr_step, ia, reduce_cb, group_ids, res

    def check_rc(rc_):
        _lib.check(rc_)

    main_step = dev_step
    if a.aggr:
        main_step, ia, reduce_cb, group_ids, aggr_host = make_aggr(a.aggr, a.groups)
        base["metric"] = "rollup samples/sec (block decode + %s(%s) by label, raw samples decoded and scanned per second)" % (a.aggr, a.func)
        base["config"]["workload"] = workload.replace("configs[1]", "configs[4]-style") + "; %s by %d groups" % (a.aggr, a.groups)
        base["config"]["parallelism"] = ("series sharded by TSID across %d GPU(s); per-GPU partial [groups x points] states merged by "
                                         "NCCL all-reduce (values: %s, counts: sum)" % (a.gpus, promql.ALLREDUCE_OP[a.aggr]))

    # ---- kernel-only: compressed blocks resident in HBM
    pci = None
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        pci = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
    except Exception:
        pass
    # NUMA placement: run this rank (and first-touch its pinned buffers) on the CPUs next to its GPU's PCIe root, like any
    # multi-GPU host process would be deployed; restored before the CPU baseline, which uses every core
    affinity0 = None
    numa_cpus = None
    try:
        affinity0 = os.sched_getaffinity(0)
        with open("/sys/bus/pci/devices/%s/local_cpulist" % pci[4:]) as f:  # sysfs uses a 4-digit PCI domain
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= affinity0
        if cpus:
            os.sched_setaffinity(0, cpus)
            numa_cpus = len(cpus)
    except Exception:
        pass
    sampler = ClockSampler(local_rank, pci)
    sampler.start()
    dev_ms_step, launches, (tb, te), last = time_steps(main_step, a.warmup, a.steps)
    scanned = last[1]
    clocks = sampler.window(tb, te)
    if a.dump_outputs and rank == 0:  # before any later call reuses out_dev / the aggregate's host buffer
        if a.aggr:
            dump_outputs(a.dump_outputs, lambda idx: aggr_host[idx], a.groups, points, scanned)
        else:
            dump_outputs(a.dump_outputs, lambda idx: out_dev[torch.from_numpy(idx).cuda()].cpu().numpy(), a.blocks, points, scanned)
    # per-stage device times of one extra step (CUDA events inside the library, same stream)
    ctx.enable_stage_timing(True)
    main_step()
    stage_ms = ctx.stage_ms()
    ctx.enable_stage_timing(False)

    # ---- full-size parity: sampled series of the timed batch against the oracle (rank 0)
    parity = None
    arm = None
    if rank == 0 and a.parity_series > 0 and not a.aggr:
        arm = CpuArm(descs, payload, a.func, start, end, step, a.window_ms)
        dev_step()
        parity = parity_check(arm, lambda idx: out_dev[torch.from_numpy(idx).cuda()].cpu().numpy(), a.parity_series)
        assert parity["ok"], parity

    # ---- e2e: host buffers in, host result out
    e2e = None
    if not a.no_e2e:
        nbytes_out = (a.groups if a.aggr else a.blocks) * points * 8
        hp = _lib.lib().vmb_host_alloc(payload.size + 64)
        ho = _lib.lib().vmb_host_alloc(nbytes_out)
        hd = _lib.lib().vmb_host_alloc(descs.nbytes)
        assert hp and ho and hd, "pinned host allocation failed"
        h_payload = np.ctypeslib.as_array(C.cast(hp, C.POINTER(C.c_uint8)), shape=(payload.size,))
        h_payload[:] = payload
        h_descs = np.ctypeslib.as_array(C.cast(hd, C.POINTER(C.c_uint8)), shape=(descs.nbytes,)).view(descs.dtype)
        h_descs[:] = descs
        h_out = np.ctypeslib.as_array(C.cast(ho, C.POINTER(C.c_double)), shape=((a.groups if a.aggr else a.blocks), points))

        def host_step():
            if a.aggr and world > 1:  # per-rank partial from host buffers, NCCL all-reduce, finalize + D2H of the result
                sc_ = ia.update_host(h_descs, h_payload, rc_aggr, group_ids, ctx)
                ia.finalize(ctx, all_reduce=reduce_cb, out=h_out)
                return h_out, sc_
            if a.aggr:
                return promql.eval_rollup_aggr_host(a.aggr, a.func, h_descs, h_payload, group_ids, a.groups, start, end, step,
                                                    a.window_ms, args=func_args, out=h_out, ctx=ctx)
            return promql.eval_rollup_func_host(a.func, h_descs, h_payload, start, end, step, a.window_ms, args=func_args,
                                                out=h_out, nseries=a.blocks, ctx=ctx)
        tw = time.perf_counter()
        e2e_ms_step, _, (tb2, te2), _ = time_steps(host_step, max(1, min(a.warmup, 2)), a.steps)
        e2e_clocks = sampler.window(tb2, te2)
        e2e = {"ms": e2e_ms_step, "h2d": int(descs.nbytes + payload.size), "d2h": int(nbytes_out)}
        if a.aggr:  # same query result as the device-resident arm (chunk-wise folding only reorders float additions)
            assert np.allclose(h_out, aggr_host, rtol=1e-9, atol=0, equal_nan=True)
        else:
            check = float(np.nansum(h_out[: min(a.blocks, 64)]))
            dcheck = float(torch.nansum(out_dev[: min(a.blocks, 64)]).item())
            assert abs(check - dcheck) <= 1e-9 * max(1.0, abs(dcheck)), (check, dcheck)
        for p_ in (hp, ho, hd):
            _lib.lib().vmb_host_free(p_)

    # ---- sub-record: sum(rate(m[5m])) by (label), 8 and 1024 groups (configs[3] shape at this batch size)
    aggr_rec = None
    if not a.no_aggr and not a.aggr:
        aggr_rec = {}
        for groups in (8, 1024):
            fn, _ia, _cb, _g, res = make_aggr("sum", groups)
            ms_, launches_, _, _ = time_steps(fn, 2, max(3, min(a.steps, 5)))
            ms_, = max_over_ranks(ms_)
            aggr_rec["sum_by_%d_groups" % groups] = {
                "value": world * rows_total / (ms_ / 1e3), "unit": "samples/s", "ms_per_step": ms_, "gpu_launches_per_step": launches_ / max(3, min(a.steps, 5)),
                "result": "[%d x %d] f64 finalized on every rank, copied to pinned host memory inside the timed region" % (groups, points),
                "api": "vmb_eval_rollup_aggr_dist (fold inside the fused kernel; NCCL inside the library)",
                "collective": ("ncclAllReduce of {values, counts}[%d x %d] f64 across %d ranks, issued by libvmb200 on its stream" % (groups, points, world)) if world > 1 else "none (one GPU)"}
            del fn, _ia, res

    sampler.stop()
    dev_ms_step, e2e_ms_step = max_over_ranks(dev_ms_step, e2e["ms"] if e2e else 0.0)

    # ---- sub-record: the library-encoded input beside the default (same values, other zstd frames)
    alt = None
    if rank == 0 and world == 1 and not a.no_alt_encoder and not a.aggr:
        other = "library" if a.encoder == "reference" else "reference"
        try:
            nalt = min(a.blocks, 20000)
            d2, p2, _ = gen_blocks(nalt, a.rows, seed=1234 + rank, kind=a.kind, ts_kind=a.ts, encoder=other)
            d1 = np.ascontiguousarray(descs[:nalt])
            b1 = storage.Blocks(d1, payload, ctx)
            b2 = storage.Blocks(d2, p2, ctx)
            res = {}
            for name, bl in ((a.encoder, b1), (other, b2)):
                fn = lambda bl=bl: promql.eval_rollup_func(a.func, bl, start, end, step, a.window_ms, args=func_args, out_dev_ptr=out_dev.data_ptr())
                ms_, _, _, _ = time_steps(fn, 2, 5)
                ctx.enable_stage_timing(True)
                fn()
                st_ = ctx.stage_ms()
                ctx.enable_stage_timing(False)
                res[name] = {"ms_per_step": ms_, "value": nalt * a.rows / (ms_ / 1e3), "zstd_stage_ms": round(st_[0], 4)}
            res["blocks"] = nalt
            res["bytes_per_sample"] = {a.encoder: round(compressed_bytes(d1, a.ts) / (nalt * a.rows), 3),
                                       other: round(compressed_bytes(d2, a.ts) / (nalt * a.rows), 3)}
            alt = res
            b1.close()
            b2.close()
        except Exception as e:
            alt = {"failed": repr(e)}

    # ---- sub-record: configs[2] / north-star size, 1 M series x 8192 on one GPU, chunked by 100 000 blocks
    c2 = None
    n2 = a.configs2_series
    if n2 < 0:
        n2 = 1_000_000 if (world == 1 and a.kind == "counter" and a.func == "rate" and a.blocks == 100_000 and a.ts == "regular") else 0
    if rank == 0 and world == 1 and n2 > 0 and not a.aggr:
        c2 = run_configs2(a, ctx, n2, out_dev, time_steps, start, end, step, points)

    if rank == 0:
        ms_per_step = dev_ms_step
        value = world * rows_total / (ms_per_step / 1e3)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)"
        varint_bytes = int(2 * rows_total) * (2 if a.ts == "jitter" else 1)  # ~2 B/sample zig-zag varints per zstd column
        drop_frac = (gstats["rows_from_first_drop"] / max(gstats["rows"], 1)) if a.func in RCR_FUNCS else 0.0
        stage_names = ["zstd", "column_decode", "series_preamble", "rollup", "aggregate", "fused_decode_rollup"]
        fused_on = len(stage_ms) > 5 and stage_ms[5] > 0
        stage_bytes = [compressed + varint_bytes,                          # zstd: read frames, write varint bytes
                       varint_bytes + 64 * a.blocks + rows_total * 16,     # decode: read varints + descs, write ts+val
                       int(rows_total * 16 * drop_frac),                   # preamble: read+write values from the first value drop
                                                                           # of a series on (removeCounterResets); the rest is skipped
                       rows_total * 8 * (2 if a.ts == "jitter" else 1) + a.blocks * points * 8, 0,  # rollup: read val (+ts), write result
                       varint_bytes + 64 * a.blocks + a.blocks * points * 8]  # fused kernel: read varint bytes + descs, write the result
        if fused_on:  # with the fused kernel on, stage 1 is the un-fused sub-batch of the series it did not take (none here)
            stage_bytes[1] = stage_bytes[2] = stage_bytes[3] = 0
        stages = {}
        for n_, ms_, b_ in zip(stage_names, stage_ms, stage_bytes):
            if ms_ > 0 and b_ > 0:
                stages[n_] = {"ms": round(ms_, 4), "algorithmic_GB": round(b_ / 1e9, 3), "GBps": round(b_ / 1e9 / (ms_ / 1e3), 1)}
        dom = max(stages, key=lambda k: stages[k]["ms"]) if stages else None

        def traffic_of(stage):
            """dram__bytes_read.sum + dram__bytes_write.sum of the stage's kernel from the committed `ncu --set full`
            capture (profiles/*/traffic.json: bytes per launch at 20 000 blocks, rate workload), scaled to this launch"""
            for rnd in ("r02", "r01"):
                try:
                    t = json.load(open(os.path.join(ROOT, "profiles", rnd, "traffic.json")))
                    if a.func != t["func"] or a.rows != t["rows"] or stage not in t["bytes_per_launch"]:
                        continue
                    return int(t["bytes_per_launch"][stage] * (a.blocks / t["blocks"])), "profiles/%s/traffic.json (ncu --set full capture of a %d-block run, scaled; not measured by this run)" % (rnd, t["blocks"])
                except Exception:
                    continue
            return None, None
        def issue_of(stage):
            """what actually bounds the stage: issue-slot utilisation of its kernel from the same committed ncu capture"""
            try:
                t = json.load(open(os.path.join(ROOT, "profiles", "r02", "traffic.json")))
                if a.func == t["func"] and stage in t.get("issue", {}):
                    return dict(t["issue"][stage], source=t["issue"]["source"] + " (committed capture, not measured by this run)")
            except Exception:
                pass
            return None
        fused_bytes = compressed + a.blocks * points * 8
        out = dict(base)
        out.update({"value": value, "ms_per_step": ms_per_step, "gpu_launches": int(launches), "clocks": clocks,
                    "samples_scanned_per_step": int(scanned)})
        if dom:
            ach = stages[dom]["GBps"]
            tr, tr_src = traffic_of(dom)
            out["roofline"] = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                               "traffic": tr, "traffic_source": tr_src, "peak_source": peak_src, "stages": stages,
                               "whole_step": {"fused_algorithmic_GB": round(fused_bytes / 1e9, 3),
                                              "GBps": round(fused_bytes / 1e9 / (ms_per_step / 1e3), 1),
                                              "frac": round(fused_bytes / 1e9 / (ms_per_step / 1e3) / peak, 4)},
                               "note": "the path is entropy + varint decoding: every stage is instruction-issue bound, not HBM bound "
                                       "(see `issue`); the HBM fraction is reported because the contract asks for it",
                               "issue": issue_of(dom)}
        # "block decode GB/s" of BASELINE.json's metric on the decoded-output basis (rows x 16 B): zstd + column decode stages of the
        # kernel-per-stage pipeline; with the fused kernel the decoded columns never exist, the whole step stands in for the stage
        dec_ms = (stage_ms[0] + stage_ms[1]) if not fused_on else ms_per_step
        out["decode_GBps_decoded_basis"] = round(rows_total * 16 / 1e9 / (dec_ms / 1e3), 1) if dec_ms > 0 else None
        out["decode_basis_note"] = "zstd + column decode stages" if not fused_on else "whole fused step (decode and rollup are one kernel)"
        if e2e:
            per = e2e_ms_step
            out["e2e"] = {"value": world * rows_total / (per / 1e3), "unit": "samples/s", "ms_per_step": per,
                          "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"],
                          "api": (("vmb_eval_rollup_aggr_host_partial + NCCL all-reduce + vmb_aggr_finalize" if world > 1 else
                                   "vmb_eval_rollup_aggr_host") + " (pinned host descriptors+payload in, [groups x points] result out)"
                                  if a.aggr else "vmb_eval_rollup_host (pinned host descriptors+payload in, pinned host result out)"),
                          "clocks": e2e_clocks}
        if parity:
            out["parity_check"] = parity
        if aggr_rec:
            out["aggr"] = aggr_rec
        if alt:
            out["alt_encoder"] = alt
        if c2:
            out["configs2"] = c2
        out["config"]["compressed_bytes_per_gpu"] = compressed
        out["config"]["bytes_per_sample_compressed"] = round(compressed / rows_total, 3)
        out["config"]["input_generation_s"] = round(gen_s, 1)
        out["config"]["series_with_a_counter_reset"] = round(gstats["series_with_drop"] / max(gstats["series"], 1), 3)
        out["config"]["host_affinity"] = ("GPU-local NUMA node, %d CPUs" % numa_cpus) if numa_cpus else "unchanged"
        if affinity0:
            try:
                os.sched_setaffinity(0, affinity0)
            except Exception:
                pass
        if world == 1 and a.cpu_seconds > 0:
            try:
                arm = arm or CpuArm(descs, payload, a.func, start, end, step, a.window_ms)
                out["cpu_baseline"] = arm.measure(min_wall=a.cpu_seconds)
            except Exception as e:  # the oracle is optional for the product; report instead of failing the bench
                out["cpu_baseline"] = {"value": None, "unit": "samples/s", "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_configs2(a, ctx, nseries, out_dev, time_steps, start, end, step, points):
    """BASELINE.json configs[2] + the north-star size on ONE GPU: nseries x rows samples resident in HBM as compressed blocks
    (chunks of a.blocks series, the [chunk x points] result buffer is reused: the result of 1 M series is 65 GB), rate() over
    counters and avg/max/quantile_over_time(0.99) over gauges.  One step = one pass over all chunks."""
    import torch
    from victoriametrics_b200 import promql, storage
    rec = {"series": nseries, "rows_per_series": a.rows, "chunk_series": a.blocks, "window_s": a.window_ms // 1000, "step_s": a.step_ms // 1000,
           "note": "compressed blocks of all series resident in HBM; result written chunk by chunk into one reused [chunk x points] buffer"}
    phis = np.full(points, 0.99)
    for kind, funcs in (("counter", ["rate"]), ("gauge", ["avg_over_time", "max_over_time", "quantile_over_time"])):
        t0 = time.perf_counter()
        chunks, comp = [], 0
        first = None
        for c0 in range(0, nseries, a.blocks):
            n = min(a.blocks, nseries - c0)
            d, p, _ = gen_blocks(n, a.rows, seed=777 + c0, kind=kind, ts_kind="regular", encoder=a.encoder)
            comp += compressed_bytes(d, "regular")
            chunks.append(storage.Blocks(d, p, ctx))
            if first is None:
                first = (d, p)
            del d, p
        gen_s = time.perf_counter() - t0
        for func in funcs:
            args = phis if func == "quantile_over_time" else None

            def fn():
                r = None
                for bl in chunks:
                    r = promql.eval_rollup_func(func, bl, start, end, step, a.window_ms, args=args,
                                                out_dev_ptr=out_dev.data_ptr())
                return r
            ms_, launches_, _, _ = time_steps(fn, 1, 2)
            r = {"value": nseries * a.rows / (ms_ / 1e3), "unit": "samples/s", "ms_per_step": ms_, "gpu_launches_per_step": launches_ / 2,
                 "values": kind, "compressed_GB": round(comp / 1e9, 2), "input_generation_and_upload_s": round(gen_s, 1)}
            # parity of the first chunk (its result is recomputed last)
            promql.eval_rollup_func(func, chunks[0], start, end, step, a.window_ms, args=args, out_dev_ptr=out_dev.data_ptr())
            arm = CpuArm(first[0], first[1], func, start, end, step, a.window_ms)
            r["parity_check"] = parity_check(arm, lambda idx: out_dev[torch.from_numpy(idx).cuda()].cpu().numpy(), 200)
            assert r["parity_check"]["ok"], (func, r["parity_check"])
            rec[func] = r
        if kind == "counter":
            # configs[3] per GPU: sum(rate(m[5m])) by (label) over the same nseries series, 1024 groups.  Every chunk is folded inside
            # the fused kernel into a partial {values, counts}[G x P] and merged into the running state (updateTimeseries +
            # the merge of aggr_incremental.go:141); then the library's all-reduce (a no-op on one GPU), finalize, result to the host
            import ctypes as C
            from victoriametrics_b200 import _lib
            G = 1024
            rcfg = promql.get_rollup_configs("rate", start, end, step, a.window_ms)
            cfg = rcfg._cfg()
            cells = G * points
            tot = torch.empty(2 * cells, dtype=torch.float64, device="cuda")
            part = torch.empty(2 * cells, dtype=torch.float64, device="cuda")
            gids = [((np.arange(bl.count, dtype=np.int64) + 131 * k) % G).astype(np.uint32) for k, bl in enumerate(chunks)]
            res = np.empty((G, points), dtype=np.float64)
            L = _lib.lib()
            SUM = promql.AGGR_FUNCS["sum"]

            def fn_aggr():
                sc = C.c_uint64(0)
                for k, bl in enumerate(chunks):
                    dst = tot if k == 0 else part
                    _lib.check(L.vmb_eval_rollup_aggr_device(ctx.h, bl.h, storage.INT64_MIN, storage.INT64_MAX, C.byref(cfg), SUM,
                                                             gids[k].ctypes.data_as(_lib.u32p), G, C.c_void_p(dst.data_ptr()),
                                                             C.c_void_p(dst.data_ptr() + cells * 8), C.byref(sc)))
                    if k:
                        _lib.check(L.vmb_aggr_merge(ctx.h, SUM, C.c_void_p(tot.data_ptr()), C.c_void_p(tot.data_ptr() + cells * 8),
                                                    C.c_void_p(part.data_ptr()), C.c_void_p(part.data_ptr() + cells * 8), cells))
                _lib.check(L.vmb_aggr_allreduce(ctx.h, SUM, C.c_void_p(tot.data_ptr()), C.c_void_p(tot.data_ptr() + cells * 8), cells))
                _lib.check(L.vmb_aggr_finalize(ctx.h, SUM, C.c_void_p(tot.data_ptr()), C.c_void_p(tot.data_ptr() + cells * 8), cells,
                                               res.ctypes.data_as(_lib.f64p)))
                return res
            ms_, launches_, _, _ = time_steps(fn_aggr, 1, 2)
            # check against the (parity-checked) per-series result: chunk 0's rows summed by group, then the same path on chunk 0 alone
            promql.eval_rollup_func("rate", chunks[0], start, end, step, a.window_ms, out_dev_ptr=out_dev.data_ptr())
            rows0 = out_dev[: chunks[0].count]
            want = torch.zeros((G, points), dtype=torch.float64, device="cuda")
            want.index_add_(0, torch.from_numpy(gids[0].astype(np.int64)).cuda(), torch.nan_to_num(rows0, nan=0.0))
            got0, _ = promql.eval_rollup_aggr_dist("sum", "rate", chunks[0], gids[0], G, start, end, step, a.window_ms)
            w = want.cpu().numpy()
            ok = bool(np.allclose(np.nan_to_num(got0, nan=0.0), w, rtol=1e-9, atol=1e-9))
            assert ok, "sum(rate) by over chunk 0 differs from the per-series result summed by group"
            rec["sum_rate_by_1024_groups"] = {
                "value": nseries * a.rows / (ms_ / 1e3), "unit": "samples/s", "ms_per_step": ms_, "gpu_launches_per_step": launches_ / 2,
                "groups": G, "result": "[1024 x %d] f64 finalized and copied to the host inside the timed region" % points,
                "api": "per chunk vmb_eval_rollup_aggr_device (fold inside the fused kernel) + vmb_aggr_merge; then vmb_aggr_allreduce "
                       "(NCCL inside the library; a no-op on one GPU) + vmb_aggr_finalize",
                "note": "BASELINE.json configs[3] is this on 8 GPUs x 1 M series each; the N = 8 `aggr` record of this bench shows the "
                        "all-reduce of [1024 x %d] adds 0.7 ms" % points,
                "check": {"chunk0_vs_per_series_rows_summed_by_group_rtol_1e-9": ok}}
        for bl in chunks:
            bl.close()
        del chunks, first
    return rec


if __name__ == "__main__":
    sys.exit(main())
