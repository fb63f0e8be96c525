#!/usr/bin/env python3
"""bench.py -- flow records/s through EWMA throughput-anomaly detection (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one complete TAD job (stage A filter/reduce, group, time sort, stddev_samp, EWMA,
anomaly compaction) over one synthetic flow table of BASELINE.json configs[1]: 100M records /
1M connections x 100 points per GPU (weak scaling: every rank holds that many rows of a table
whose connections are spread over all ranks).

ours:       `value`  = rows / device time per step, inputs resident in HBM (CUDA events recorded by
                       the library on its own stream: first kernel start -> last kernel end).
            `e2e`    = same job through the C ABI with HOST (pinned) column buffers: H2D of the
                       29 B/row inputs and D2H of the result rows inside the timed region.
reference:  the CPU oracle port (oracle/tad_oracle.c, the restated reference job; the reference
            itself is PySpark and cannot run in this image) on all host cores, bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "flow records/sec through EWMA anomaly detection"
BYTES_PER_ROW = 29          # src_ip4 dst_ip4 src_port2 dst_port2 proto1 flow_start4 flow_end4 value8
RESULT_ROW_BYTES = 46


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons: one streaming `nvidia-smi -lms 20` process; only the samples whose
    timestamps fall inside the timed region are kept."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.lines, self.proc, self.th = index, [], None, None
        self.t0 = self.t1 = None

    def _pump(self):
        try:
            for line in self.proc.stdout:
                self.lines.append((time.time(), line))
        except Exception:
            pass

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=3)
            except Exception:
                self.proc.kill()
        rows = []
        for ts, line in self.lines:
            f = [x.strip() for x in line.strip().split(",")]
            if len(f) >= 7:
                rows.append((ts, f[1:]))
        inside = [f for ts, f in rows if self.t0 is not None and self.t0 - 0.02 <= ts <= self.t1 + 0.02]
        use = inside if inside else [f for _, f in rows[-3:]]
        if not use:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(f[0]) for f in use if f[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(f[2 + i].lower().startswith("active") for f in use)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(use[0][1]) if use[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(use), "samples_in_timed_region": len(inside)}


def ncu_traffic(kernel, rows):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture (profiles/), valid for
    the 1e8-row workload it was taken on; None otherwise."""
    for name in ("r02_traffic.json", "r01_traffic.json"):          # newest capture of the shipped kernels first
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", name)))
            if d.get("rows") == rows and kernel in d["kernels"]:
                return d["kernels"][kernel]["dram_bytes_read"] + d["kernels"][kernel]["dram_bytes_write"]
        except Exception:
            pass
    return None


K1, K2, K3, M32 = 2654435761, 2246822519, 3266489917, 0xffffffff


def sample_mask(src_ip, dst_ip, frac):
    """Same pseudo-random subset of connections on every rank, for torch (int64 bit patterns) and numpy (unsigned) columns:
    a 20-bit hash of (sourceIP, destinationIP) below a threshold."""
    try:
        import torch
        is_t = isinstance(src_ip, torch.Tensor)
    except ImportError:
        is_t = False
    if is_t:
        a, b = src_ip.to(torch.int64) & M32, dst_ip.to(torch.int64) & M32
    else:
        import numpy as np
        a, b = src_ip.astype(np.uint64), dst_ip.astype(np.uint64)
    h = ((a * K1) ^ (b * K2)) & M32
    h = (h * K3) & M32
    h = (h ^ (h >> 15)) & 0xfffff
    return h < max(1, int(frac * (1 << 20)))


DUMP_BYTES = 64 << 20


def dump_sample(res, result_rows):
    """The rows of `res` (one job's result columns, or one rank's share of them) that --dump-outputs keeps: every row when
    the whole result (`result_rows` rows over all ranks) fits half of DUMP_BYTES as float64, else the connections that
    sample_mask selects with the largest power-of-two fraction that does.  Returns (rows, fraction)."""
    frac = 1.0
    while result_rows * frac * 8 * len(res) > DUMP_BYTES / 2:
        frac /= 2
    if frac < 1.0:
        m = sample_mask(res["src_ip"], res["dst_ip"], frac)
        res = {k: v[m] for k, v in res.items()}
    return res, frac


def write_outputs(out_dir, res, result_rows, frac):
    """DIR/<column>.npy, float64 (every result column is FP64 or an integer below 2^53), rows in canonical (key, flowEnd)
    order so that two builds compare element for element; cut to DUMP_BYTES in that order."""
    import numpy as np
    from oracle import tad_oracle
    res = tad_oracle.canonicalize(res)
    keep = min(len(res["flow_end"]), DUMP_BYTES // (8 * len(res)))
    os.makedirs(out_dir, exist_ok=True)
    for k, v in res.items():
        np.save(os.path.join(out_dir, k + ".npy"), v[:keep].astype(np.float64))
    return {"dir": out_dir, "rows": keep, "result_rows": result_rows, "connection_fraction": frac, "dtype": "float64"}


def parity_check(eng, dcols, cols_t, algo, global_rows, total_series, dist, rank, world, want_connections=3000):
    """One more (untimed) job on the bench table; the connections of a hash-selected sample are cross-checked bit for bit
    against the CPU oracle (the checker; tests/test_gpu_full_size.py does the same): the input rows of the sample are
    collected from every rank, the oracle runs stages A-E on them, and the result rows the engine produced for those
    connections (on whichever rank owns them) must be identical in every column."""
    import numpy as np
    from oracle import c_oracle, tad_oracle
    from theia_b200 import synth
    frac = min(1.0, want_connections / max(1, total_series))
    job = eng.submit(dcols, algo=algo, tad_id="parity", global_rows=global_rows)
    job.wait()
    res = job.result()
    job.release()
    m_in = sample_mask(cols_t["src_ip"], cols_t["dst_ip"], frac)
    sub = synth.torch_cols_to_numpy(cols_t, m_in)
    m_out = sample_mask(res["src_ip"], res["dst_ip"], frac)
    got = {k: v[m_out] for k, v in res.items()}
    if dist is not None:
        box = [None] * world if rank == 0 else None
        dist.gather_object((sub, got), box, dst=0)
        if rank != 0:
            return None
        sub = {k: np.concatenate([b[0][k] for b in box]) for k in sub}
        got = {k: np.concatenate([b[1][k] for b in box]) for k in got}
    cols, ns, npts = c_oracle.run_job(sub, algo={"EWMA": 0, "ARIMA": 1, "DBSCAN": 2}[algo])
    want, got = tad_oracle.canonicalize(cols), tad_oracle.canonicalize(got)
    ok = len(want["flow_end"]) == len(got["flow_end"])
    bad = []
    if ok:
        for c in want:
            if not np.array_equal(want[c], got[c], equal_nan=True):
                ok = False
                bad.append(c)
    return {"checked": int(ns), "input_rows": int(len(sub["value"])), "result_rows": int(len(want["flow_end"])),
            "ok": bool(ok), "against": "oracle/tad_oracle.c, every result column bit-exact", **({"differs": bad} if bad else {})}


def python_port_rate(points):
    """Single-core rate of the pure-Python restatement (numpy stages A/B + the per-series UDF loops the Spark workers
    would run, oracle/tad_oracle.py) on a 2e5-row sample: the 'local[1]'-style figure SURVEY section 8(d) asks for.
    Reported next to the C port; never fatal."""
    try:
        from oracle import tad_oracle
        from theia_b200 import synth
        t = synth.make_flows(max(1, 200_000 // points), points, seed=1)
        tad_oracle.run_job(t, tad_oracle.JobSpec())
        t0 = time.perf_counter()
        tad_oracle.run_job(t, tad_oracle.JobSpec())
        dt = time.perf_counter() - t0
        return {"value": len(t["value"]) / dt, "unit": "records/s", "cores": 1,
                "sample": "%d rows, oracle/tad_oracle.py" % len(t["value"])}
    except Exception as e:       # the bench line must not depend on this side figure
        return {"unavailable": repr(e)[:120]}


def native_decode_rate():
    """Host-side rate of the ClickHouse Native-format ingest (theia_b200/clickhouse_native.py): 1e6 flow rows of the eight
    engine columns, IPs as text.  A side figure for the transport that replaces JDBC; never fatal."""
    try:
        from theia_b200 import clickhouse_native as chn
        from theia_b200 import synth
        t = synth.make_flows(10_000, 100, seed=2)
        cols = [("sourceIP", "String", t["src_ip"]), ("destinationIP", "String", t["dst_ip"]),
                ("sourceTransportPort", "UInt16", t["src_port"]), ("destinationTransportPort", "UInt16", t["dst_port"]),
                ("protocolIdentifier", "UInt8", t["proto"]), ("flowStartSeconds", "DateTime", t["flow_start"]),
                ("flowEndSeconds", "DateTime", t["flow_end"]), ("throughput", "UInt64", t["value"])]
        n = len(t["value"])
        stream = b"".join(chn.write_native([(k, ty, v[lo:lo + 65536]) for k, ty, v in cols]) for lo in range(0, n, 65536))
        chn.flows_from_native(stream)
        t0 = time.perf_counter()
        chn.flows_from_native(stream)
        dt = time.perf_counter() - t0
        return {"value": n / dt, "unit": "records/s", "bytes_per_record": len(stream) / n,
                "sample": "%d rows in 64 Ki-row blocks, IPv4 addresses as text" % n}
    except Exception as e:
        return {"unavailable": repr(e)[:120]}


def bench_table_numpy(series, points, seed=1):
    """The bench table (BASELINE configs[1] shape) as numpy columns for the CPU arm: generated on the GPU when one is
    visible (the numpy generator needs minutes for 1e8 rows), else with numpy.  Untimed."""
    from theia_b200 import synth
    try:
        import torch
        if torch.cuda.is_available():
            cols_t = synth.make_flows_torch(series, points, seed=seed, device=torch.device("cuda", 0))
            t = synth.torch_cols_to_numpy(cols_t)
            del cols_t
            torch.cuda.empty_cache()
            return t
    except Exception:
        pass
    return synth.make_flows(series, points, seed=seed)


def cpu_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def run_reference(args):
    """CPU arm: the oracle port of the reference job (stages A-E) with all host threads, on the SAME table shape as our arm
    (full size unless --ref-series bounds it).  Runs in a process of its own (the GPU arm calls it through a subprocess):
    the OpenMP placement below binds threads -- including the calling one -- and must not leak into a process that drives
    GPUs (it pinned every rank's host threads to one core when it did)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = cpu_threads()                           # before any OpenMP runtime narrows the calling thread's mask
    # pin the OpenMP threads of the oracle port (one per hardware thread, no migration) before libgomp loads, so that the
    # baseline does not swing with the scheduler's mood from box to box
    os.environ.setdefault("OMP_PROC_BIND", "spread")
    os.environ.setdefault("OMP_PLACES", "threads")
    os.environ.pop("OMP_NUM_THREADS", None)         # torchrun sets it to 1 for every rank; the oracle asks for `cores` itself
    from oracle import c_oracle
    series = args.ref_series or args.series
    t = bench_table_numpy(series, args.points)
    rows = len(t["value"])
    c_oracle.build()
    for _ in range(min(args.warmup, 1)):           # one warm-up pass is enough for a CPU job of seconds
        c_oracle.run_job(t, algo=0, threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cols, ns, npts = c_oracle.run_job(t, algo=0, threads=cores)
    dt = (time.perf_counter() - t0) / args.steps
    v = rows / dt
    outputs = None
    if args.dump_outputs:
        n = len(cols["flow_end"])
        sub, frac = dump_sample(cols, n)
        outputs = write_outputs(args.dump_outputs, sub, n, frac)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "records/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "EWMA, %d records / %d connections x %d points per GPU (BASELINE configs[1])" % (args.series * args.points, args.series, args.points),
                   "sample": "each step runs the CPU path on %d connections x %d points = %d rows%s" % (
                       series, args.points, rows, "" if series == args.series else " (bounded sample)"),
                   "rows_per_step": rows, "same_table_shape_as_ours": series == args.series},
        "cpu_baseline": {"value": v, "unit": "records/s", "cores": cores, "threads_used": cores, "kind": "port",
                         "omp": {k: os.environ.get(k) for k in ("OMP_PROC_BIND", "OMP_PLACES", "OMP_NUM_THREADS")},
                         "sample": "%d rows per step, oracle/tad_oracle.c with OpenMP on %d threads; %d series, %d points found" % (
                             rows, cores, ns, npts),
                         "python_port_1core": python_port_rate(args.points)},
        "e2e": {"value": v, "unit": "records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, **({"outputs": outputs} if outputs else {})}))


def side_run(eng, dev, algo, series, points, steps, warmup, name):
    """One of the other BASELINE configurations on this GPU: device-resident synthetic table, `warmup` + `steps` jobs, the
    library's CUDA-event times, its own roofline figures and its own parity flag (sampled connections against the oracle;
    ARIMA: against oracle/arima_oracle.py on a handful of connections, flags and relative error)."""
    import torch
    from theia_b200 import synth
    from theia_b200.engine import DeviceColumns
    out = {"config": name, "algo": algo}
    try:
        cols_t = synth.make_flows_torch(series, points, seed=5, device=dev, noisy=(algo == "ARIMA"))
        rows = int(cols_t["value"].numel())
        torch.cuda.synchronize()
        dcols = DeviceColumns(rows, {k: v.data_ptr() for k, v in cols_t.items()})
        dcols.keepalive = cols_t
        ms, phase, launches, st = 0.0, {}, 0, None
        for i in range(warmup + steps):
            job = eng.submit(dcols, algo=algo, tad_id="side")
            st = job.wait()
            job.release()
            if i >= warmup:
                ms += st["device_ms"]
                launches += st["gpu_launches"]
                for k, v in st["phase_ms"].items():
                    phase[k] = phase.get(k, 0.0) + v
        ms /= steps
        per = {k: v / steps for k, v in phase.items() if v}
        peak, peak_src = peaks()
        kern = {k: per[k] for k in ("hist", "scatter", "group", "detect") if per.get(k, 0) > 0}
        dom = max(kern, key=kern.get)
        out.update({"records": rows, "value": rows / (ms * 1e-3), "unit": "records/s", "ms_per_step": ms, "steps": steps,
                    "warmup": warmup, "series": int(st["series"]), "series_per_s": int(st["series"]) / (ms * 1e-3),
                    "result_rows": int(st["result_rows"]), "gpu_launches": launches, "phase_ms": per, "dtype": "f64",
                    "roofline": {"bound": "hbm", "kernel": dom,
                                 **({"limiter": "FP64 compute, not HBM: ~100 likelihood evaluations x t Kalman-filter steps per fit; "
                                                "the HBM fraction below is reported for the contract only"} if algo == "ARIMA" else {}), "achieved": BYTES_PER_ROW * rows / (kern[dom] * 1e-3) / 1e9, "peak": peak,
                                 "unit": "GB/s", "frac": BYTES_PER_ROW * rows / (kern[dom] * 1e-3) / 1e9 / peak,
                                 "pipeline_frac": BYTES_PER_ROW * rows / (ms * 1e-3) / 1e9 / peak, "traffic": None,
                                 "peak_source": peak_src}})
        if algo == "ARIMA":
            out["fits_per_s"] = rows / (ms * 1e-3)            # one ARIMA(1,1,1) prefix fit per point (anomaly_detection.py:239-258)
            out["parity"] = arima_parity(eng, cols_t, series)
        else:
            out["parity"] = parity_check(eng, dcols, cols_t, algo, 0, series, None, 0, 1)
        del dcols, cols_t
        torch.cuda.empty_cache()
    except Exception as e:          # a side figure must not take the bench line down
        out["unavailable"] = repr(e)[:200]
    return out


def side_sharded(eng, dev, dist, rank, world, series_per_gpu, points, steps, warmup, name):
    """A larger sharded table through the same multi-GPU path as the headline (device-resident input); all ranks call this."""
    import torch
    from theia_b200 import synth
    from theia_b200.engine import DeviceColumns
    out = {"config": name, "algo": "EWMA", "n_gpus": world}
    try:
        free, _total = torch.cuda.mem_get_info()
        need = series_per_gpu * points * 220            # generator temporaries + columns + slots + entries + csr, bytes per row
        ok = torch.tensor([1 if free > need else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok[0]) == 0:
            out["unavailable"] = "not enough free HBM on some rank (%.0f GB free here)" % (free / 1e9)
            return out
        cols_t = synth.make_flows_torch_sharded(series_per_gpu, points, seed=7, device=dev, rank=rank, world=world)
        rows = int(cols_t["value"].numel())
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        dcols = DeviceColumns(rows, {k: v.data_ptr() for k, v in cols_t.items()})
        dcols.keepalive = cols_t
        global_rows = rows * world
        ms, phase, st = 0.0, {}, None
        for i in range(warmup + steps):
            job = eng.submit(dcols, algo="EWMA", tad_id="side", global_rows=global_rows)
            st = job.wait()
            job.release()
            if i >= warmup:
                ms += st["device_ms"]
                for k, v in st["phase_ms"].items():
                    phase[k] = phase.get(k, 0.0) + v
        t = torch.tensor([ms / steps], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
        parity = parity_check(eng, dcols, cols_t, "EWMA", global_rows, series_per_gpu * world, dist, rank, world)
        peak, peak_src = peaks()
        out.update({"records": global_rows, "rows_per_gpu": rows, "value": global_rows / (ms * 1e-3), "unit": "records/s",
                    "ms_per_step": ms, "steps": steps, "warmup": warmup, "dtype": "f64",
                    "phase_ms": {k: v / steps for k, v in phase.items() if v}, "parity": parity,
                    "roofline": {"bound": "hbm", "unit": "GB/s", "peak": peak * world, "peak_source": peak_src + " x %d GPUs" % world,
                                 "achieved": BYTES_PER_ROW * global_rows / (ms * 1e-3) / 1e9,
                                 "frac": BYTES_PER_ROW * global_rows / (ms * 1e-3) / 1e9 / (peak * world), "traffic": None,
                                 "kernel": "whole job (aggregate HBM-read roofline of the %d GPUs)" % world}})
        del dcols, cols_t
        torch.cuda.empty_cache()
    except Exception as e:          # a side figure must not take the bench line down
        out["unavailable"] = repr(e)[:200]
    return out


def arima_parity(eng, cols_t, series, want=3):
    """ARIMA: a handful of connections against the SciPy restatement of statsmodels' fit (oracle/arima_oracle.py; the C
    oracle has no ARIMA): share of identical flags, median / max relative error of algoCalc."""
    try:
        import numpy as np
        from oracle import arima_oracle, tad_oracle
        from theia_b200 import synth
        m = sample_mask(cols_t["src_ip"], cols_t["dst_ip"], min(1.0, want / series))
        sub = synth.torch_cols_to_numpy(cols_t, m)
        got, _ = eng.run(sub, algo="ARIMA", tad_id="parity", emit_all=True)
        res = tad_oracle.run_job(sub, tad_oracle.JobSpec(algo=tad_oracle.ALGO_ARIMA, emit_all=True),
                                 arima_fn=arima_oracle.calculate_arima)
        w, g = tad_oracle.canonicalize(dict(res.cols)), tad_oracle.canonicalize(got)
        if len(w["flow_end"]) != len(g["flow_end"]) or not np.array_equal(w["flow_end"], g["flow_end"]):
            return {"ok": False, "note": "different set of surviving series / points (%d vs %d rows)" % (len(g["flow_end"]), len(w["flow_end"]))}
        rel = np.abs(g["algo_calc"] - w["algo_calc"]) / np.maximum(np.abs(w["algo_calc"]), 1e-300)
        same = float(np.mean(g["anomaly"] == w["anomaly"]))
        return {"checked": int(len(np.unique(sub["src_ip"]))), "points": int(len(rel)), "flags_identical": same,
                "rel_err_median": float(np.median(rel)), "rel_err_max": float(rel.max()), "ok": bool(same >= 0.99),
                "against": "oracle/arima_oracle.py (SciPy restatement; parity unpinned below ~1e-3, DESIGN.md section 8)"}
    except Exception as e:
        return {"ok": None, "unavailable": repr(e)[:160]}


def run_ours(args):
    import numpy as np
    import torch
    from theia_b200 import synth
    from theia_b200.engine import DeviceColumns, TadEngine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    uid = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        buf = [TadEngine.get_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(buf, src=0)
        uid = buf[0]
    eng = TadEngine(device=local, world_size=world, rank=rank, nccl_unique_id=uid)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()              # early: nvidia-smi takes a second or more to enumerate the GPUs

    S, n = args.series, args.points
    cols_t = synth.make_flows_torch(S, n, seed=1 + rank, device=dev) if world == 1 else \
        synth.make_flows_torch_sharded(S, n, seed=1, device=dev, rank=rank, world=world)
    rows = int(cols_t["value"].numel())
    torch.cuda.synchronize()
    torch.cuda.empty_cache()         # the generator's temporaries go back to the driver: the engine allocates with cudaMalloc
    dcols = DeviceColumns(rows, {k: v.data_ptr() for k, v in cols_t.items()})
    dcols.keepalive = cols_t

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    global_rows = rows * world if world > 1 else 0      # what the host's SELECT count() tells every rank (equal shards)

    def step(cols):
        job = eng.submit(cols, algo=args.algo, tad_id="bench", global_rows=global_rows)
        st = job.wait()
        return job, st

    # ---- value: inputs resident in HBM ---------------------------------------------------------
    for _ in range(args.warmup):
        job, st = step(dcols)
        job.release()
    barrier()
    sampler.mark_begin()
    t0 = time.perf_counter()
    dev_ms, phase, launches, result_rows = 0.0, {}, 0, 0
    last = None
    for i in range(args.steps):
        job, st = step(dcols)
        dev_ms += st["device_ms"]
        launches += st["gpu_launches"]
        result_rows = st["result_rows"]
        for k, v in st["phase_ms"].items():
            phase[k] = phase.get(k, 0.0) + v
        if args.dump_outputs and i == args.steps - 1:
            last = job                   # its rows are fetched once the clock has stopped
        else:
            job.release()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None

    # ---- --dump-outputs: the result rows of the last timed step (all ranks' shares, sampled alike) ----------------------
    outputs = None
    if last is not None:
        res = last.result()
        last.release()
        n = torch.tensor([len(res["flow_end"])], device=dev, dtype=torch.int64)
        if dist is not None:
            dist.all_reduce(n)
        res, frac = dump_sample(res, int(n[0]))
        if dist is not None:
            box = [None] * world if rank == 0 else None
            dist.gather_object(res, box, dst=0)
            if rank == 0:
                res = {k: np.concatenate([b[k] for b in box]) for k in res}
        if rank == 0:
            outputs = write_outputs(args.dump_outputs, res, int(n[0]), frac)
    stats = torch.tensor([dev_ms / args.steps, wall_ms / args.steps], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    ms_dev, ms_wall = float(stats[0]), float(stats[1])
    tr = torch.tensor([rows], device=dev, dtype=torch.int64)
    if dist is not None:
        dist.all_reduce(tr)
    total_rows = int(tr[0])
    assert world == 1 or total_rows == global_rows, "shards are not balanced"

    # ---- parity: a sample of connections against the CPU oracle, at every N (untimed) -------------------------------
    parity = None
    if not args.no_parity:
        parity = parity_check(eng, dcols, cols_t, args.algo, global_rows, S * world, dist, rank, world)

    # ---- e2e: host (pinned) buffers through the C ABI, H2D + D2H inside the timed region --------
    if args.no_e2e:
        if rank == 0:
            print(json.dumps({"value": total_rows / (ms_dev * 1e-3), "ms_per_step": ms_dev, "wall_ms_per_step": ms_wall,
                              "phase_ms": {k: v / args.steps for k, v in phase.items()}, "parity": parity,
                              "note": "profiling run", **({"outputs": outputs} if outputs else {})}))
        eng.close()
        if dist is not None:
            dist.destroy_process_group()
        return
    hcols = eng.alloc_columns(rows)
    for name, tns in cols_t.items():
        hv = hcols.view(name)
        hv[:rows] = tns.cpu().numpy().view(hv.dtype)
    hcols.c.rows = rows
    for _ in range(max(1, args.warmup // 2)):
        job, st = step(hcols)
        job.result(copy=False)
        job.release()
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(1, args.steps // 2)
    for _ in range(e2e_steps):
        job, st = step(hcols)
        res = job.result(copy=False)
        d2h = int(st["result_rows"]) * RESULT_ROW_BYTES
        h2d_ms = st["phase_ms"]["h2d"]
        job.release()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    e2e_t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_ms = float(e2e_t[0])

    # ---- e2e, two jobs in flight: a second context (own stream + workspace) on the same GPU, jobs submitted
    # alternately so that the H2D of job i+1 overlaps the compute and D2H of job i (how the controller's 4
    # workers drive tad_submit).  Reported separately; `e2e.value` above is one job at a time.
    pipe_ms = None
    if world == 1 and not args.no_pipelined:
        eng2 = TadEngine(device=local)
        hcols2 = eng2.alloc_columns(rows)
        for name in cols_t:
            hcols2.view(name)[:rows] = hcols.view(name)[:rows]
        hcols2.c.rows = rows
        engines = [(eng, hcols), (eng2, hcols2)]
        for e_, c_ in engines:                       # warm both workspaces
            j_ = e_.submit(c_, algo="EWMA", tad_id="bench")
            j_.wait(); j_.result(copy=False); j_.release()
        torch.cuda.synchronize()
        n_pipe = max(4, args.steps)
        t0 = time.perf_counter()
        inflight = []
        for k in range(n_pipe):
            e_, c_ = engines[k % 2]
            if len(inflight) == 2:
                j_ = inflight.pop(0)
                j_.wait(); j_.result(copy=False); j_.release()
            inflight.append(e_.submit(c_, algo="EWMA", tad_id="bench"))
        for j_ in inflight:
            j_.wait(); j_.result(copy=False); j_.release()
        torch.cuda.synchronize()
        pipe_ms = (time.perf_counter() - t0) * 1e3 / n_pipe
        hcols2.free()
        eng2.close()

    if rank == 0:
        peak, peak_src = peaks()
        per = {k: v / args.steps for k, v in phase.items()}
        kern = {k: per[k] for k in ("hist", "scatter", "group", "detect") if per.get(k, 0) > 0}
        dom = max(kern, key=kern.get)
        alg_bytes = {"hist": 17, "scatter": 29, "group": 29, "detect": 29}[dom] * rows
        achieved = alg_bytes / (kern[dom] * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": total_rows / (ms_dev * 1e-3), "unit": "records/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "EWMA, %d records / %d connections x %d points per GPU (BASELINE configs[1])" % (rows, S, n),
                       "rows_per_gpu": rows, "l2": "inputs (%.1f GB) larger than L2" % (rows * BYTES_PER_ROW / 1e9),
                       "timing": "library CUDA events on its stream; wall clock per step %.3f ms" % ms_wall},
            "e2e": {"value": total_rows / (e2e_ms * 1e-3), "unit": "records/s",
                    "h2d_bytes_per_step": rows * BYTES_PER_ROW, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms, "h2d_ms": h2d_ms,
                    "two_jobs_in_flight": None if pipe_ms is None else
                    {"value": rows / (pipe_ms * 1e-3), "ms_per_step": pipe_ms,
                     "note": "two contexts on one GPU, H2D of job i+1 overlaps compute + D2H of job i"}},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic(dom, rows), "peak_source": peak_src,
                         "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed ncu --set full "
                                           "capture of the shipped build (profiles/r02_traffic.json, valid for the 1e8-row workload); "
                                           "ncu cannot run inside the timed bench",
                         "note": "achieved = algorithmic bytes (29 B/row; hist 17) / CUDA-event time of the phase; the group phase is "
                                 "three launches of one kernel template (capacity classes)",
                         "pipeline_frac": rows * BYTES_PER_ROW / (ms_dev * 1e-3) / 1e9 / peak},
            "phase_ms": per, "result_rows": result_rows, "clocks": clocks,
        }
        line["parity"] = parity
        if outputs:
            line["outputs"] = outputs
        line["phase_ms_meaning"] = {
            "h2d": "host->device column copies, with the partition kernels that run chunk by chunk behind them (0 for device-resident input)",
            "exchange": "several GPUs: gather of the peers' arrival counters (rows are pulled inside `group`); exact partition: exposed NCCL all-to-all",
            "sync": "several GPUs: waiting for the other ranks at the job's two barriers (arrival skew + barrier latency)"}
        if world == 1 and not args.no_cpu:
            # the CPU arm in a process of its own (see run_reference): the same table shape, 2 timed passes
            cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2", "--warmup", "1",
                   "--series", str(S), "--points", str(n), "--ref-series", str(args.ref_series)]
            env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
            try:
                out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
                ref = json.loads(out.stdout.strip().splitlines()[-1])
                line["cpu_baseline"] = ref["cpu_baseline"]
                line["cpu_baseline"]["ms_per_pass"] = ref["ms_per_step"]
            except Exception as e:
                line["cpu_baseline"] = {"unavailable": repr(e)[:200], "kind": "port"}
            line["native_ingest"] = native_decode_rate()
    hcols.free()
    del dcols, cols_t
    torch.cuda.empty_cache()
    big = None
    big_series = int(os.environ.get("TAD_BENCH_BIG_SIDE", "5000000" if world == 8 else "0"))   # connections per GPU; 0 = no side run
    if world > 1 and big_series > 0 and not args.no_sides and args.algo == "EWMA":
        # BASELINE configs[4] (1e10 records / 1e8 connections over 8 GPUs) at 40 % of its named size: 5e8 rows per GPU.  Every rank
        # takes part (the job is collective); rank 0 reports.  A watchdog guards the headline: should the side run not come back
        # (a rank failing alone would leave the others inside a collective), rank 0 prints the line without it and every rank exits.
        def bail():
            if rank == 0:
                line.setdefault("side", []).append({"config": "BASELINE configs[4] at 40 %", "unavailable": "side run exceeded its 300 s budget"})
                print(json.dumps(line), flush=True)
            os._exit(0)
        dog = threading.Timer(300.0, bail)
        dog.daemon = True
        dog.start()
        big = side_sharded(eng, dev, dist, rank, world, big_series, 100, steps=2, warmup=1,
                           name="BASELINE configs[4] at 40 %: 4e9 records / 4e7 connections hash-sharded over 8 GPUs (5e8 rows per GPU; "
                                "the named 1.25e9 rows per GPU need the memory plan of DESIGN.md section 6)")
        dog.cancel()
    if rank == 0:
        if big is not None:
            line.setdefault("side", []).append(big)
        if world == 1 and not args.no_sides and args.algo == "EWMA":
            # the other BASELINE configurations, measured in the same run on the same GPU (device-resident input)
            line["side"] = line.get("side", []) + [
                side_run(eng, dev, "DBSCAN", 10_000_000, 24, steps=3, warmup=1,
                         name="BASELINE configs[3]: DBSCAN over 10M connections x 24 points (240M records)"),
                side_run(eng, dev, "ARIMA", 20_000, 100, steps=1, warmup=1,
                         name="BASELINE configs[2] slice: ARIMA per-series fit + score, 20K connections x 100 points "
                              "(2M records; the named 1B-record size is reported as fits/s x its 1e7 connections)"),
            ]
        print(json.dumps(line))
    eng.close()
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--series", type=int, default=1_000_000)
    ap.add_argument("--points", type=int, default=100)
    ap.add_argument("--ref-series", type=int, default=0, help="connections in the CPU arm's table (0 = the full bench table)")
    ap.add_argument("--no-parity", action="store_true", help="skip the sampled oracle cross-check")
    ap.add_argument("--no-sides", action="store_true", help="skip the DBSCAN / ARIMA side measurements (N = 1 only)")
    ap.add_argument("--algo", default="EWMA", choices=["EWMA", "DBSCAN", "ARIMA"],
                    help="detector (the BASELINE metric is EWMA; the others are side measurements of configs[2]/[3])")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs: skip the host-buffer leg")
    ap.add_argument("--no-pipelined", action="store_true", help="skip the two-jobs-in-flight e2e figure")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result rows of the last timed step as DIR/<column>.npy (float64, canonical row order, "
                         "at most 64 MB: above that a fixed hash-selected subset of the connections)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
