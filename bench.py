#!/usr/bin/env python
"""bench.py -- series fitted+forecast per second on N B200s (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference-shaped CPU fan-out on the host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's forecasts to DIR/*.npy

A "step" is one pass of the hot path over one batch of synthetic series:
  value : device-resident y[N,T] -> forecast table, kernels + (N>1) one NCCL all_gather, timed with
          CUDA events on the launching stream, max over ranks.
  e2e   : the same call with HOST (pinned) buffers through the C ABI: H2D of y and D2H of the
          forecasts are inside the timed region.
One JSON line on stdout (rank 0).  See DESIGN.md section 5 for how each field is measured.
"""
import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "series fitted+forecast/sec"
UNIT = "series/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--series", type=int, default=1_000_000,
                    help="series per GPU (--scaling weak, default) or in total, block-sharded over the ranks (--scaling strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --series per GPU (driver default); strong: --series in total = BASELINE configs[3] as worded "
                         "(1 M groups over 8 GPUs + one all-gather of the forecast table)")
    ap.add_argument("--tc-variant", type=int, default=0, choices=[0, 1, 2],
                    help="tcgen05 kernel instantiation: 0 auto, 1 = 10 stages / 1 staging tile, 2 = 8 stages / 2 staging tiles")
    ap.add_argument("--calendars", type=int, default=0,
                    help="single GPU: ragged batch -- the series are split over this many distinct calendars (start dates "
                         "one day apart, same length) and fit in ONE launch (mmf_fit_forecast_ragged_f32)")
    ap.add_argument("--replicas", type=int, default=1,
                    help="single GPU diagnostic: store every forecast tile to this many LOCAL copies of the table through the "
                         "multi-destination epilogue (isolates its cost from NVLink)")
    ap.add_argument("--stream-solve", action="store_true",
                    help="experimental: solve the series with gaps beside the tcgen05 kernel (mmf_config.stream_solve = 1)")
    ap.add_argument("--no-traffic", action="store_true", help="skip the live ncu DRAM-traffic probe of the dominant kernel")
    ap.add_argument("--traffic-child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--t", type=int, default=1095)
    ap.add_argument("--horizon", type=int, default=28)
    ap.add_argument("--kernel", default="auto", choices=["auto", "warp", "tc"])
    ap.add_argument("--nan-frac", type=float, default=0.0)
    ap.add_argument("--mode", default="future", choices=["future", "holdout"],
                    help="future: fit all T rows, forecast `horizon` rows (BASELINE metric); holdout: the reference "
                         "contract -- hold out the last `horizon` rows, emit a fitted/forecast value for all T dates")
    ap.add_argument("--e2e-series", type=int, default=0, help="series per e2e step (0 = same as --series)")
    ap.add_argument("--gather", default="p2p", choices=["p2p", "nccl", "multicast", "multicast-bulk"],
                    help="N>1: how the forecast table reaches every rank: p2p = bulk stores from the fit kernel's epilogue "
                         "into every peer's copy over NVLink (default), nccl = one all_gather after the kernel")
    ap.add_argument("--graph", action="store_true",
                    help="replay each step as a CUDA graph (small batches are launch-bound); single GPU only")
    ap.add_argument("--pitch-floats", type=int, default=0,
                    help="row pitch of the device-resident y in floats (0 = T rounded up to 4; 32 | pitch = 128-B aligned rows)")
    ap.add_argument("--no-others", action="store_true",
                    help="skip the short extra measurements of the other BASELINE configurations (other_configs in the line)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-groups", type=int, default=0, help="groups per step of the reference arm (0 = 16 x cores)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the forecast table of the last timed step to DIR/forecast.npy "
                         "(and the e2e leg's last host output to DIR/e2e_forecast.npy), float32; tables larger than "
                         "30 MB are reduced to a fixed seeded sample of rows, the same on every run with the same arguments")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


DUMP_BYTES = 30_000_000      # per dumped table: forecast.npy and e2e_forecast.npy stay under 64 MB together


def dump_output(dirname, name, table):
    """Write ``table`` (rows x columns, torch tensor or NumPy array) to dirname/name.npy as float32, so that two builds
    of the project can be compared output for output.  A table over DUMP_BYTES keeps a fixed sample of its rows
    (numpy default_rng(0), in row order): the same rows on every run of the same shape."""
    import numpy as np
    import torch
    rows, cols = table.shape
    keep = max(1, DUMP_BYTES // (4 * cols))
    if rows > keep:
        idx = np.sort(np.random.default_rng(0).choice(rows, keep, replace=False))
        table = table[torch.from_numpy(idx).to(table.device)] if torch.is_tensor(table) else table[idx]
    if torch.is_tensor(table):
        table = table.cpu().numpy()
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, f"{name}.npy"), np.ascontiguousarray(table, dtype=np.float32))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            atexit.register(self.proc.kill)     # the sampler never outlives the bench, even when a step raises
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for ts, r in self.rows if t0 - 0.05 <= ts <= t1 + 0.15 and len(r) >= 9] or [r for _, r in self.rows if len(r) >= 9]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = [float(r[1]) for r in rows]
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(rows[0][2]), "reasons": sorted(reasons),
                "samples": len(rows), "power_w_max": max(float(r[3]) for r in rows)}


# =========================================================================================
def cpu_port_baseline(y_sample, start, t, h):
    """The oracle on a bounded sample, all host cores: the C restatement (oracle/mmf_oracle_c.c, float64
    accumulation, pthreads) when its library is there (build() compiles it), else the NumPy route."""
    import numpy as np
    from oracle import mmf_oracle as O

    grid = O.calendar_grid(start, t + h, "D")
    X = O.design_matrix(grid, t)
    cores = len(os.sched_getaffinity(0))
    n_s = y_sample.shape[0]
    so = os.path.join(ROOT, "oracle", "libmmf_oracle.so")
    if not os.path.exists(so):
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle")], capture_output=True)
    if os.path.exists(so):
        # pages first-touched by the pinned worker thread that later reads them: the same placement on every box
        # (round 1's sample lived on whichever NUMA node the rank had been bound to and moved 3.3x between boxes)
        y32 = O.numa_local_sample(np.ascontiguousarray(y_sample, dtype=np.float32))
        prep = {}
        out, st, used = O.fit_forecast_packed_c(y32, X, t, t, h, return_threads=True, prepared=prep)   # warm, same placement
        t0 = time.perf_counter()
        done = 0
        while time.perf_counter() - t0 < 12.0:
            O.fit_forecast_packed_c(y32, X, t, t, h, out=out, status=st, prepared=prep)
            done += n_s
        dt = time.perf_counter() - t0
        return {"value": done / dt, "unit": UNIT, "cores": used, "kind": "port",
                "sample": f"{done} series x {t} days ({done // n_s} passes over {n_s} distinct), C restatement of the oracle "
                          f"(float64 accumulation, one pass per series, {used} pthreads pinned one per core, sample pages "
                          f"first-touched by the thread that reads them), {dt:.1f} s"}
    O.fit_forecast_packed(y_sample[:256], X, t, t, h)                 # warm
    t0 = time.perf_counter()
    done = 0
    block = 20000
    while time.perf_counter() - t0 < 12.0:                            # cycle over the sample for ~12 s of CPU work
        lo = done % n_s
        O.fit_forecast_packed(y_sample[lo:lo + block], X, t, t, h)
        done += min(block, n_s - lo)
    dt = time.perf_counter() - t0
    return {"value": done / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{done} series x {t} days (cycling over {n_s} distinct), float64 NumPy oracle, vectorised packed "
                      f"route, BLAS threads, {dt:.1f} s"}


_REF = {}


def _ref_init(t, h):
    from oracle import mmf_oracle as O
    _REF["O"], _REF["t"], _REF["h"] = O, t, h


def _ref_one(args):
    """One Spark-task-shaped unit (reference 02:523-528 + 417-494): a group's rows arrive as an Arrow
    RecordBatch, become a pandas frame, go through the per-group UDF, and return as Arrow."""
    import pandas as pd
    import pyarrow as pa
    key, dates, vals = args
    O = _REF["O"]
    pdf = pd.DataFrame({"Product": key[0], "SKU": key[1], "Date": dates, "Demand": vals})
    batch = pa.RecordBatch.from_pandas(pdf, preserve_index=False)          # JVM -> Python worker hop
    out = O.build_tune_and_score_model(batch.to_pandas(), freq="D", horizon=_REF["h"], mode="future")
    return pa.RecordBatch.from_pandas(out, preserve_index=False).num_rows  # Python worker -> JVM hop


def run_reference(args):
    """--impl reference: the reference-shaped CPU fan-out (one Python UDF call per group, Arrow hop both
    ways, all host cores), the stand-in for Spark local[*] which needs a JVM + pyspark (absent)."""
    import multiprocessing as mp
    import numpy as np
    import mmf

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0))
    g = args.ref_groups or 16 * cores
    t, h = args.t, args.horizon
    y, start = mmf.synth.daily_store_item_demand(g, t, seed=1234)
    days = mmf.design.calendar_grid(start, t, "D")
    import datetime as dt
    dates = [dt.date.fromisoformat(str(d)) for d in days]
    work = [((f"store{i // 50}", f"item{i}"), dates, y[i]) for i in range(g)]
    with mp.get_context("fork").Pool(cores, initializer=_ref_init, initargs=(t, h)) as pool:
        for _ in range(max(args.warmup, 1)):
            pool.map(_ref_one, work[:cores * 2], chunksize=1)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            rows = pool.map(_ref_one, work, chunksize=1)
        dtot = time.perf_counter() - t0
    assert all(r == h for r in rows)
    value = g * args.steps / dtot
    sample = (f"{g} groups x {t} days per step, one oracle-UDF call per group with an Arrow RecordBatch round trip, "
              f"multiprocessing.Pool({cores}); reference SARIMAX+hyperopt UDF itself cannot run here (no statsmodels/"
              f"hyperopt/pyspark/JVM)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dtot / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{g} (store,item) groups x {t} days per step, {h}-day horizon, future mode "
                                   f"(bounded sample of the 1M-series workload)", "groups_per_step": g, "t": t,
                       "horizon": h, "parallelism": f"cpu fan-out x{cores}",
                       "same_config_note": "same metric, series length, horizon and mode as the GPU arm; a bounded number "
                                           f"of groups per step ({g} = 16 x cores): every group is an independent task of the "
                                           "same size, so series/s of the fan-out does not depend on how many groups a step holds"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def nvlink_counters(index):
    """Sum of the NVLink data counters of GPU `index` in bytes (tx, rx), or None: `nvidia-smi nvlink -gt d`."""
    try:
        r = subprocess.run(["nvidia-smi", "nvlink", "-gt", "d", "-i", str(index)], capture_output=True, text=True, timeout=20)
        tx = rx = 0
        seen = False
        for line in r.stdout.splitlines():
            parts = line.replace(":", " ").split()
            if "Tx" in parts or "Rx" in parts:
                val = float(parts[-2])
                mult = {"KiB": 1024.0, "MiB": 1024.0 ** 2, "GiB": 1024.0 ** 3, "B": 1.0}.get(parts[-1], 1024.0)
                if "Tx" in parts:
                    tx += val * mult
                else:
                    rx += val * mult
                seen = True
        return (tx, rx) if seen else None
    except Exception:
        return None


TRAFFIC_KERNELS = "fit_tc_kernel|fit_warp_kernel|predict_tc_kernel|solve_rows_kernel"


def traffic_child(args):
    """Child of the live traffic probe (runs under ncu): the same launch as a bench step on the same shape --
    values do not change the bytes a gap-free pass moves, so the input is a cheap random level + noise."""
    import torch
    import mmf
    torch.cuda.set_device(0)
    n, t, h = args.series, args.t, args.horizon
    ld = args.pitch_floats or ((t + 3) & ~3)
    g = torch.Generator(device="cuda").manual_seed(7)
    y = (torch.randn((n, ld), generator=g, device="cuda") * 100.0 + 10000.0).round_()[:, :t]
    if args.nan_frac > 0:
        y[torch.rand((n, t), generator=g, device="cuda") < args.nan_frac] = float("nan")
    _, start = mmf.synth.daily_store_item_demand(1, t, seed=0)
    eng = mmf.ForecastEngine(device=0, kernel=args.kernel, tc_variant=args.tc_variant)
    _, ps, npred = eng.plan_calendar(start, t, "D", h, args.mode)
    out = torch.empty((n, (npred + 3) & ~3), device="cuda")[:, :npred] if args.mode == "holdout" else torch.empty((n, h), device="cuda")
    eng.fit_forecast(y, ps, npred, out=out)
    torch.cuda.synchronize()
    torch.cuda.profiler.start()
    eng.fit_forecast(y, ps, npred, out=out)
    torch.cuda.synchronize()
    torch.cuda.profiler.stop()
    eng.close()


def live_traffic(args, n, kernel_name):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel on this run's shape, measured
    now: `ncu` around a child process that issues the same launch (the bench's own timed steps never run under a
    profiler).  Returns (bytes or None, note)."""
    import shutil
    import tempfile
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None, "ncu not found"
    log = os.path.join(tempfile.mkdtemp(prefix="mmf_ncu_"), "traffic.csv")
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum", "--clock-control", "none",
           "--profile-from-start", "off", "-k", f"regex:{TRAFFIC_KERNELS}", "--csv", "--print-units", "base",
           "--log-file", log, sys.executable, os.path.abspath(__file__), "--traffic-child", "--series", str(n),
           "--t", str(args.t), "--horizon", str(args.horizon), "--kernel", args.kernel, "--mode", args.mode,
           "--nan-frac", str(args.nan_frac), "--tc-variant", str(args.tc_variant), "--pitch-floats", str(args.pitch_floats)]
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=420, env=env)
        if r.returncode != 0 or not os.path.exists(log):
            return None, f"ncu probe failed (rc {r.returncode}): {(r.stderr or r.stdout)[-200:]!r}"
        import csv
        rows = []
        with open(log) as f:
            lines = [ln for ln in f if not ln.startswith("==")]
        for row in csv.DictReader(lines):
            rows.append(row)
        per = {}
        for row in rows:
            kn = row.get("Kernel Name", "")
            if kernel_name not in kn:
                continue
            m, v = row.get("Metric Name"), float(row.get("Metric Value", "0").replace(",", ""))
            per.setdefault(row.get("ID"), {})[m] = v
        if not per:
            return None, f"no {kernel_name} launch in the ncu log"
        tot = [d.get("dram__bytes_read.sum", 0.0) + d.get("dram__bytes_write.sum", 0.0) for d in per.values()]
        return sum(tot) / len(tot), (f"live: ncu dram__bytes_read.sum + dram__bytes_write.sum, {len(tot)} launch(es) of "
                                     f"{kernel_name} on this run's shape in a child process, this box")
    except Exception as exc:        # noqa: BLE001 -- the probe must never take the bench down
        return None, f"ncu probe failed: {exc!r}"


# =========================================================================================
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import mmf
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and rank == 0:
        print(f"# note: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    all_cpus = os.sched_getaffinity(0)
    numa_cpus = mmf.bind_to_gpu_numa(local)             # pinned staging buffers land on the GPU's NUMA node
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    t, h = args.t, args.horizon
    # weak: --series per GPU; strong: --series in total, equal contiguous blocks of ceil(total/world) rows per rank
    n = args.series if args.scaling == "weak" else -(-args.series // world)
    K, W = args.steps, max(args.warmup, 3)

    # ---- inputs: resident in HBM before the timed region; 4.4 GB per pass >> 126 MB L2
    y, start = mmf.synth.daily_store_item_demand_torch(n, t, seed=1234 + rank, nan_frac=args.nan_frac, device=dev,
                                                        ld=args.pitch_floats or None)
    torch.cuda.synchronize()
    # the all-gathered forecast table.  N>1: NVLink symmetric memory so the fit kernel itself can store every
    # forecast row into all ranks' copies (NVLS multicast or P2P); --gather nccl keeps the plain collective.
    gather = "none"
    sym = None
    if world > 1 and args.gather != "nccl":
        from mmf.sharding import SymmetricTable
        try:
            sym = SymmetricTable(n, h, dev, mode=args.gather)
            ok = torch.ones(1, device=dev)
        except Exception as exc:                          # no NVLink symmetric memory on this box
            sym, ok = None, torch.zeros(1, device=dev)
            print(f"# rank {rank}: symmetric memory unavailable ({exc!r}); falling back to NCCL all_gather", file=sys.stderr)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)         # all ranks take the same path
        if float(ok[0]) < 1.0:
            sym = None
    if sym is not None:
        table = sym.table
        gather = "fused-" + args.gather
    else:
        table = torch.zeros((world * n, h), dtype=torch.float32, device=dev)
        gather = "nccl-all_gather" if world > 1 else "none"
    mine = table[rank * n:(rank + 1) * n]

    eng = mmf.ForecastEngine(device=local, kernel=args.kernel, tc_variant=args.tc_variant, stream_solve=args.stream_solve)
    # ForecastEngine enqueues on torch's current stream for CUDA tensors, so the CUDA events below see the kernels
    _, ps, npred = eng.plan_calendar(start, t, "D", h, args.mode)
    if args.mode == "holdout":
        if world > 1:
            raise SystemExit("--mode holdout is a single-GPU diagnostic")
        table = torch.zeros((n, (npred + 3) & ~3), dtype=torch.float32, device=dev)[:, :npred]
        mine = table
    st = eng.fit_forecast(y, ps, npred, out=mine, want_stats=True)["stats"]
    launches_per_call, kernel_used = st.kernel_launches, st.kernel_used

    # inputs that fit a few L2s are rotated over distinct buffers so that every step streams from HBM
    in_bytes = n * t * 4
    n_rot = 1 if in_bytes >= 4 * 126e6 else int(min(64, -(-int(5 * 126e6) // in_bytes)))
    ys = [y] + [mmf.device_packed(y, device=dev) for _ in range(n_rot - 1)]      # same row pitch as y
    graphs = None
    if args.graph:
        if world > 1 or args.mode != "future":
            raise SystemExit("--graph is a single-GPU, future-mode option")
        graphs = [eng.capture(yy, ps, npred, out=mine)[0] for yy in ys]
    step_no = [0]

    ragged_rows = None
    if args.calendars > 0:
        if world > 1:
            raise SystemExit("--calendars is a single-GPU option")
        C_ = args.calendars
        ragged_rows = np.linspace(0, n, C_ + 1).astype(np.int64)
        starts = [np.datetime64(start, "D") - np.timedelta64(c, "D") for c in range(C_)]
        t0_plan = time.perf_counter()
        eng.plan_calendars(starts, [t] * C_, "D", h, mode=args.mode)
        ragged_plan_s = time.perf_counter() - t0_plan
    reps = None
    if args.replicas > 1 and world == 1:
        rep_tensors = [torch.zeros_like(mine) for _ in range(args.replicas - 1)]     # kept alive by the closure below
        reps = [mine.data_ptr()] + [r.data_ptr() for r in rep_tensors]

    def fit():
        i = step_no[0] % n_rot
        step_no[0] += 1
        if ragged_rows is not None:
            eng.fit_forecast_ragged(ys[i], ragged_rows, out=mine)
        elif reps is not None:
            assert len(rep_tensors) == args.replicas - 1
            eng.fit_forecast_bcast(ys[i], ps, npred, reps, h)
        elif graphs is not None:
            graphs[i].replay()
        elif sym is not None:
            sym.fit_into(eng, ys[i], ps, npred)         # forecasts land in every rank's table from the epilogue
        else:
            eng.fit_forecast(ys[i], ps, npred, out=mine)

    def exchange():
        if sym is not None:
            sym.barrier()                               # all peers' stores have landed
        elif world > 1:
            dist.all_gather_into_tensor(table, mine)    # in-place: mine is table's slice

    def step():
        fit()
        exchange()

    for _ in range(W):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:                       # start sampling BEFORE the barrier so every rank enters the timed loop together
        sampler.start()
        time.sleep(0.3)
    # NVLink byte counters of rank 0's GPU: read BEFORE the barrier (a subprocess; it must not skew rank 0's entry
    # into the timed loop) and again after the closing barrier
    nvl0 = nvlink_counters(local) if (rank == 0 and world > 1) else None
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * K + 2)]
    torch.cuda.profiler.start()          # `ncu --profile-from-start off` captures exactly the timed region
    wall0 = time.time()
    ev[0].record()
    for i in range(K):
        ev[2 + 2 * i].record()
        fit()
        ev[3 + 2 * i].record()
        exchange()
    ev[1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    torch.cuda.profiler.stop()
    wall1 = time.time()
    nvl1 = nvlink_counters(local) if nvl0 is not None else None
    total_ms = ev[0].elapsed_time(ev[1])
    kern_ms = [ev[2 + 2 * i].elapsed_time(ev[3 + 2 * i]) for i in range(K)]
    tt = torch.tensor([total_ms, sum(kern_ms) / K], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms, kern_ms_avg = float(tt[0]), float(tt[1])
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    if args.dump_outputs and rank == 0:                 # the table as the last timed step left it (every rank's is equal)
        dump_output(args.dump_outputs, "forecast", table)
    value = world * n * K / (total_ms * 1e-3)
    gather_check = None
    shard_only = None
    if world > 1:                                       # every rank's table must equal the NCCL-gathered one
        ref = torch.empty((world * n, h), dtype=torch.float32, device=dev)
        loc = torch.empty((n, h), dtype=torch.float32, device=dev)
        # the same K steps with every rank keeping its forecasts local (what the reference's distributed Delta
        # write would need): separates the fit's scaling from the cost of replicating the table to every GPU
        for _ in range(3):
            eng.fit_forecast(y, ps, npred, out=loc)
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(K):
            eng.fit_forecast(y, ps, npred, out=loc)
        s1.record()
        torch.cuda.synchronize()
        so = torch.tensor([s0.elapsed_time(s1)], device=dev, dtype=torch.float64)
        dist.all_reduce(so, op=dist.ReduceOp.MAX)
        nvlink = None
        if nvl0 is not None and nvl1 is not None:       # rank 0's GPU, driver counters around the timed region
            nvlink = {"tx_bytes_per_step": (nvl1[0] - nvl0[0]) / K, "rx_bytes_per_step": (nvl1[1] - nvl0[1]) / K,
                      "tx_GBps": (nvl1[0] - nvl0[0]) / (total_ms * 1e-3) / 1e9,
                      "rx_GBps": (nvl1[1] - nvl0[1]) / (total_ms * 1e-3) / 1e9,
                      "source": "nvidia-smi nvlink -gt d on rank 0's GPU before / after the timed region"}
        shard_only = {"value": world * n * K / (float(so[0]) * 1e-3), "unit": "series/s", "ms_per_step": float(so[0]) / K,
                      "nvlink": nvlink,
                      "note": "same K steps, forecasts kept on the fitting rank (no table replication); max over ranks",
                      "replication_bytes_in_per_gpu_per_step": (world - 1) * n * h * 4,
                      "replication_ingress_GBps_per_gpu": (world - 1) * n * h * 4 / (total_ms / K * 1e-3) / 1e9}
        dist.all_gather_into_tensor(ref, loc)
        diff = (ref - table).abs().max().reshape(1)
        dist.all_reduce(diff, op=dist.ReduceOp.MAX)
        gather_check = float(diff[0])
        del ref, loc

    # ---- roofline of the dominant kernel (algorithmic bytes: 4*T read + 4*H written per series)
    peak, peak_src = peaks()
    bytes_per_series = 4 * t + 4 * h if args.mode == "future" else 4 * (t - h) + 4 * t
    achieved = n * bytes_per_series / (kern_ms_avg * 1e-3) / 1e9
    dom_kernel = "fit_tc_kernel" if kernel_used == "tc" else "fit_warp_kernel"
    traffic, traffic_note = (None, "not probed")
    if rank == 0 and world == 1 and not args.no_traffic:
        traffic, traffic_note = live_traffic(args, n, dom_kernel)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_unit": "bytes per launch", "traffic_source": traffic_note,
                "algorithmic_bytes_per_launch": n * bytes_per_series,
                "kernel": dom_kernel,
                "peak_source": peak_src, "bytes_per_series": bytes_per_series,
                "kernel_ms": kern_ms_avg,
                "note": "CUDA events around each step's libmmf launches in the timed region, max over ranks"}

    # ---- e2e: host (pinned) buffers through the C ABI, H2D + D2H inside the timed region
    e2e = None
    if not args.no_e2e and args.mode == "future":
        ne = args.e2e_series or n
        # host narrowing: the library's automatic setting turns it on only when the process sees ONE GPU (several ranks of a
        # multi-GPU job would fight for host cores and memory bandwidth).  A single-process run on a multi-GPU box is the
        # same situation as a single-GPU box, so it asks for it explicitly (mmf_config.host_narrow = 1, "always try");
        # multi-rank runs keep the automatic setting.
        eng2 = mmf.ForecastEngine(device=local, kernel=args.kernel, host_narrow="on" if world == 1 else "auto")
        eng2.plan_calendar(start, t, "D", h, "future")
        yh = mmf.alloc_packed(ne, t)                      # pinned, pitched
        oh = mmf.pinned_empty((ne, h))
        yh[...] = y[:ne].cpu().numpy()
        Ke = min(K, 10)
        eng2.fit_forecast(yh, ps, npred, out=oh)
        h2d_actual = eng2.fit_forecast(yh, ps, npred, out=oh, want_stats=True)["stats"].h2d_bytes
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(Ke):
            eng2.fit_forecast(yh, ps, npred, out=oh)      # returns when the forecasts are in host memory
        te = time.perf_counter() - t0
        tte = torch.tensor([te], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tte, op=dist.ReduceOp.MAX)
        te = float(tte[0])
        if args.dump_outputs and rank == 0:
            dump_output(args.dump_outputs, "e2e_forecast", oh)
        chk = float(np.abs(oh[:4096] - table[rank * n: rank * n + 4096].cpu().numpy()).max())
        e2e = {"value": world * ne * Ke / te, "unit": UNIT, "h2d_bytes_per_step": int(h2d_actual),
               "d2h_bytes_per_step": ne * h * 4, "series_per_step_per_gpu": ne, "steps": Ke,
               "ms_per_step": 1e3 * te / Ke, "max_abs_diff_vs_device_path": chk,
               "host_input_bytes_per_step": ne * t * 4,
               "transport": ("float32 host buffer in; integer-valued chunks are narrowed to uint16 on host threads (exact or "
                             "not used) while the previous chunk's copy is in flight, widened on the device"
                             if h2d_actual < ne * t * 4 else "float32 host buffer in, float32 over PCIe"),
               "api": "mmf_fit_forecast_f32 with pinned host float32 y/out (ForecastEngine.fit_forecast on NumPy arrays)",
               "host_narrow": ("mmf_config.host_narrow = 1 (this is the only process feeding a GPU on this host)" if world == 1
                               else "automatic (off when the process sees several GPUs)"),
               "cpu_affinity": (f"{len(numa_cpus)} cores local to the GPU (NVML)" if numa_cpus else "unchanged")}
        # the same end-to-end call when the demand column arrives as uint16 (the recipe's demand is integer valued,
        # 01-data-generator.py:304): half the H2D bytes, widened on the device, bit-equal forecasts required
        try:
            yu = mmf.alloc_packed(ne, t, dtype=np.uint16)
            mmf.to_integer_demand(yh, np.uint16, out=yu)
            ou = mmf.pinned_empty((ne, h))
            for _ in range(2):
                eng2.fit_forecast(yu, ps, npred, out=ou)
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(Ke):
                eng2.fit_forecast(yu, ps, npred, out=ou)
            tu = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tu, op=dist.ReduceOp.MAX)
            tu = float(tu[0])
            e2e["uint16_ingest"] = {"value": world * ne * Ke / tu, "unit": UNIT, "h2d_bytes_per_step": ne * t * 2,
                                    "d2h_bytes_per_step": ne * h * 4, "ms_per_step": 1e3 * tu / Ke,
                                    "bit_equal_to_f32_ingest": bool(np.array_equal(ou, oh)),
                                    "api": "mmf_fit_forecast_int(MMF_DT_U16) with pinned host y/out"}
            del yu, ou
        except ValueError as exc:        # synthetic demand outside uint16: not applicable to this workload
            e2e["uint16_ingest"] = {"unavailable": str(exc)}
        eng2.close()

    # ---- the other BASELINE configurations, measured briefly in the same run (single GPU, default workload only): the
    # driver's record then also carries configs[1], configs[2], the reference's holdout contract and the gap path
    others = None
    default_run = (world == 1 and args.mode == "future" and args.nan_frac == 0.0 and args.calendars == 0 and args.replicas == 1
                   and not args.graph and n == 1_000_000 and t == 1095)
    if rank == 0 and default_run and not args.no_others:
        def timed(call, bytes_per_step, steps=20, warm=3):
            for _ in range(warm):
                call()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                call()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            return {"ms_per_step": ms, "roofline_frac": bytes_per_step / (ms * 1e-3) / 1e9 / peak}

        others = {}
        try:
            for name, ns in (("configs[1] 10k x 1095", 10_000), ("configs[2] 100k x 1095", 100_000)):
                rot = int(min(64, -(-int(5 * 126e6) // (ns * t * 4))))
                bufs = [mmf.device_packed(y[:ns], device=dev) for _ in range(rot)]       # distinct buffers: > 5x L2 in total
                o = torch.empty((ns, h), device=dev)
                k = [0]

                def small():
                    eng.fit_forecast(bufs[k[0] % rot], ps, npred, out=o)
                    k[0] += 1
                r = timed(small, ns * bytes_per_series, steps=50)
                r.update({"series_per_s": ns / (r["ms_per_step"] * 1e-3), "rotating_buffers": rot})
                # the same batch when the caller vouches for gap-free data (mmf_config.assume_finite: no fix-up launches)
                engf = mmf.ForecastEngine(device=local, kernel=args.kernel, assume_finite=True, tc_variant=args.tc_variant)
                engf.plan_calendar(start, t, "D", h, "future")

                def small_finite():
                    engf.fit_forecast(bufs[k[0] % rot], ps, npred, out=o)
                    k[0] += 1
                rf = timed(small_finite, ns * bytes_per_series, steps=50)
                r["assume_finite"] = {"ms_per_step": rf["ms_per_step"], "roofline_frac": rf["roofline_frac"]}
                engf.close()
                others[name] = r
                del bufs, o
            # the reference's contract: hold out the last `horizon` rows, a value for every date (02:484-494)
            engh = mmf.ForecastEngine(device=local, kernel=args.kernel)
            _, psh, nph = engh.plan_calendar(start, t, "D", h, "holdout")
            oh_ = torch.empty((n, (nph + 3) & ~3), device=dev)[:, :nph]
            r = timed(lambda: engh.fit_forecast(y, psh, nph, out=oh_), n * (4 * (t - h) + 4 * t), steps=10)
            r["series_per_s"] = n / (r["ms_per_step"] * 1e-3)
            others["holdout mode, 1M x 1095 (a value for all 1095 dates)"] = r
            del oh_
            engh.close()
            # series with gaps: 2 % of the values missing in every series
            yn = y.clone() if y.is_contiguous() else mmf.device_packed(y, device=dev)
            g2 = torch.Generator(device=dev).manual_seed(99)
            for i0 in range(0, n, 1 << 18):
                blk = yn[i0:i0 + (1 << 18)]
                blk[torch.rand(blk.shape, generator=g2, device=dev) < 0.02] = float("nan")
            r = timed(lambda: eng.fit_forecast(yn, ps, npred, out=mine), n * bytes_per_series, steps=10)
            r["series_per_s"] = n / (r["ms_per_step"] * 1e-3)
            others["2% of the values missing in every series, 1M x 1095"] = r
            # what the reference's asfreq actually produces (02:422-423): a few groups with some missing dates
            yn.copy_(y)
            rows = torch.randperm(n, generator=g2, device=dev)[: n // 50]
            first = torch.randint(30, t - 30, (rows.numel(),), generator=g2, device=dev)
            for k in range(10):
                yn[rows, first + k] = float("nan")
            r = timed(lambda: eng.fit_forecast(yn, ps, npred, out=mine), n * bytes_per_series, steps=10)
            r["series_per_s"] = n / (r["ms_per_step"] * 1e-3)
            others["2% of the series have a 10-day gap, 1M x 1095"] = r
            del yn
            eng.fit_forecast(y, ps, npred, out=mine)           # leave the table as the main measurement wrote it
            torch.cuda.synchronize()
        except Exception as exc:          # noqa: BLE001 -- the extras must never take the main line down
            others["error"] = repr(exc)

    cpu = None
    os.sched_setaffinity(0, all_cpus)                   # the CPU legs use every host core again
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_port_baseline(y[:100000].cpu().numpy(), start, t, h)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": (f"{n} (store,item) series x {t} days per GPU, {h}-day horizon, {args.mode} mode "
                                        f"(BASELINE configs[3] shape; weak scaling)" if args.scaling == "weak" else
                                        f"{world * n} (store,item) series x {t} days in total, {n} per GPU (block-sharded), "
                                        f"{h}-day horizon, {args.mode} mode (BASELINE configs[3] as worded; strong scaling)"),
                           "tc_variant": args.tc_variant, "local_replicas": args.replicas,
                           **({"calendars": args.calendars, "ragged_plan_seconds": ragged_plan_s,
                               "ragged": "one launch over all calendars (mmf_fit_forecast_ragged_f32); every step "
                                         "includes the call's one host synchronisation"} if args.calendars > 0 else {}),
                           "series_per_gpu": n, "t": t, "horizon": h, "nan_frac": args.nan_frac, "mode": args.mode,
                           "kernel": kernel_used,
                           "l2": (f"inputs {in_bytes / 1e9:.2f} GB per step per GPU > 126 MB L2" if n_rot == 1 else
                                  f"inputs {in_bytes / 1e6:.0f} MB per step: rotating over {n_rot} distinct buffers "
                                  f"({n_rot * in_bytes / 1e6:.0f} MB > 126 MB L2)"),
                           "cuda_graph": bool(args.graph),
                           "parallelism": f"series-sharded x{world}" + (f" + forecast table replicated to every rank via {gather}" if world > 1 else ""),
                           "gather": gather, "gather_max_abs_diff_vs_nccl": gather_check},
                **({"shard_only": shard_only} if shard_only is not None else {}),
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
                **({"other_configs": others} if others is not None else {}),
                "gpu_launches": launches_per_call * K, "clocks": clocks}
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.traffic_child:
        traffic_child(a)
    elif a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
