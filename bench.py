#!/usr/bin/env python
"""bench.py — scans/sec of the scan-to-submap registration hot path (BASELINE.json metric) on N B200s.

A "step" is one pass of the whole per-scan hot path of BASELINE configs[1] (64-beam ~130k pts/scan + 200 Hz IMU, single
submap, 1 x B200) over one batch of DISTINCT synthetic scans:
    IMU pre-integration of the 20 samples since the previous scan -> state prediction -> first voxel filter ->
    deskew/transform/range gate -> second voxel filters -> adaptive voxel filters -> Levenberg-Marquardt point-to-grid
    match with the pre-integration residual fused into the same solve,
followed by the configs[4] exchange step: every rank runs its share of loop-closure searches (sharded by submap owner)
and the constraint records are exchanged with one ncclAllGather issued from the C-ABI (at N = 1 the communicator has one
rank, so the per-GPU work is the same at every N: weak scaling).

  value  scans/s with the batch already resident in HBM (dl_frontend_match_batch_imu_samples_dev; the IMU samples, about
         1.3 kB per scan, are uploaded every step), device-timed with CUDA events on the library's streams, max over ranks.
  e2e    the same metric through the C-ABI calls that take HOST buffers (dl_frontend_submit_imu_samples / _collect_imu):
         pinned host scans copied to the device and results + states copied back inside the timed region (wall clock).
  roofline       achieved algorithmic GB/s of the dominant stage (per-stage CUDA events) vs the measured HBM peak.
  cpu_baseline   the oracle (CPU restatement of the same chain) on the host cores: pooled threads with a work queue, and the
                 reference's real mode (one thread); bounded sample (N=1, rank 0).
  configs2 / mode_F   extra keys: configs[2] (128-beam, 0.05 m grid, correlative + refine) and the full-cloud matcher mode.

`--impl reference` times the CPU chain alone (all host threads) and prints the same line with "impl": "reference".
`--dump-outputs DIR` writes what the last timed step returned (rank 0) as float64 .npy files, see dump_outputs(); the inputs are
seeded, so two builds run with the same arguments can be compared output for output.
Inputs per step exceed L2 (148 scans x 2.1 MB = 309 MB > 126 MB), so no explicit L2 flush.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

# stdout carries the ONE JSON line only. NCCL prints its version banner to stdout at NCCL_DEBUG=VERSION (the pool's boxes set
# it) and honours NCCL_DEBUG_FILE only above that level: raise VERSION to WARN (same banner, nothing else unless something is
# wrong) and point the log at stderr. Any other level the caller chose (INFO to see the transports, ...) is left alone.
if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from (which may be read-only)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "d-liom_b200"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "scans/sec (64-beam, 10 Hz) per GPU; pose RMSE vs reference CPU"
UNIT = "scans/s"
IMU_NOISE = [3.99e-2, 1.56e-2, 6.4e-5, 3.6e-5]     # D/config/kaist.lua:38-43
IMU_WEIGHT = 1.0


def oracle():
    """The CPU checker / baseline. Imported lazily and only on the cpu_baseline and --impl reference legs."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import orc
    orc.lib()
    return orc


def apply_pose(p7, pts):
    w, x, y, z = p7[3:]
    R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                  [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                  [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
    return pts @ R.T + p7[:3]


def physical_cores():
    try:
        ids = set()
        phys = core = None
        for line in open("/proc/cpuinfo"):
            if line.startswith("physical id"):
                phys = line.split(":")[1].strip()
            elif line.startswith("core id"):
                core = line.split(":")[1].strip()
            elif not line.strip():
                if phys is not None and core is not None:
                    ids.add((phys, core))
                phys = core = None
        return len(ids) or None
    except Exception:
        return None


def usable_cpus():
    """(threads to use, description): os.cpu_count() capped by the affinity mask and by the container's CFS quota. The pool's GPU
    boxes show 128 logical CPUs but run under `cpu.max = 1600000 100000` (16 CPUs' worth of time): 128 busy threads are then
    throttled to ~700 scans/s, 16 threads run at their full 1 100 scans/s (tools/cpu_scaling.py, profiles/r3_cpu_scaling.json) —
    the reference arm must use what the box really grants to be the best the host can do."""
    n = os.cpu_count() or 1
    note = f"os.cpu_count() = {n}"
    try:
        aff = len(os.sched_getaffinity(0))
        if aff < n:
            n, note = aff, note + f", affinity {aff}"
    except (AttributeError, OSError):
        pass
    quota = period = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]       # cgroup v2
        if q != "max":
            quota, period = float(q), float(p)
    except (OSError, ValueError):
        try:                                                              # cgroup v1
            quota = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        except (OSError, ValueError):
            pass
    if quota and period and quota > 0:
        cap = max(1, int(-(-quota // period)))
        note += f", cgroup quota {quota / period:g} CPUs"
        n = min(n, cap)
    return n, note


def build_workload(args, rank):
    """Submap cells (built with the oracle's range-data inserter, like the reference builds a submap: hit 0.55 /
    miss 0.49 / 2 free voxels, high-res max range 20 m) + the batch of DISTINCT scans to register, each with the IMU
    samples since the previous scan and the (perturbed) state there. Deterministic."""
    import imu_synth
    import synth
    orc = oracle()
    scene = synth.Scene(42)
    opts = orc.FrontEndOptions.defaults()
    hi, lo = orc.Grid(0.1), orc.Grid(0.45)
    origin = np.zeros((1, 3), np.float32)
    t0 = 2.0
    for k in range(args.map_scans):
        t = t0 + 0.1 * k
        rows = synth.make_scan(scene, args.beams, t)
        cur = synth.pose7(t)
        ing = orc.ingest_scan(opts, rows, origin, synth.pose7(t - 0.1), cur)
        local = apply_pose(cur, ing["returns_tracking"].astype(np.float64)).astype(np.float32)
        o = cur[:3].astype(np.float32)
        hi.insert_range_data(o, local[np.linalg.norm(local - o, axis=1) <= 20.0])
        lo.insert_range_data(o, local)
    rng = np.random.RandomState(45 + rank)
    span = 0.1 * max(args.map_scans - 2, 1)
    scans, truths, states_i, intervals = [], [], [], []
    for j in range(args.batch):
        # sweeps spread over the mapped stretch, all distinct (different end times -> different rays and noise), per-rank offset
        t = t0 + 0.05 + span * j / max(args.batch, 1) + 0.0007 * rank
        scans.append(synth.make_scan(scene, args.beams, t))
        truths.append(synth.pose7(t))
        si = imu_synth.state(t - 0.1, ba=rng.normal(0, 1e-2, 3), bg=rng.normal(0, 1e-3, 3))
        si[:3] += rng.uniform(-0.05, 0.05, 3)        # the previous scan's estimate is not the truth
        si[7:10] += rng.uniform(-0.5, 0.5, 3)        # -> the prediction is off by up to ~0.1 m, like the 0.1 m / 1 deg of SURVEY 8d
        states_i.append(si)
        intervals.append(imu_synth.samples(t - 0.1, t, ba=si[10:13], bg=si[13:16], noise=(IMU_NOISE[0], IMU_NOISE[1]),
                                           seed=1000 * rank + j))
    return {"orc": orc, "opts": opts, "hi": hi, "lo": lo, "origin": origin, "scans": scans, "truth": np.array(truths),
            "states_i": np.array(states_i), "intervals": intervals, "submap_pose": orc.IDENTITY_POSE.copy()}


def loop_closure_pairs(w, args, rank):
    """The configs[4] exchange step's work list for this rank: `pairs` recent nodes (filtered clouds of its own scans) against
    the submap it owns (submap id = rank), pose guesses a few metres off so that the coarse search has a window to cover."""
    orc = w["orc"]
    rng = np.random.RandomState(900 + rank)
    his, los, guesses, nodes = [], [], [], []
    o = w["opts"]
    for k in range(args.pairs):
        j = (k * 17) % len(w["scans"])
        si = w["states_i"][j]
        pts = orc.ingest_scan(o, w["scans"][j], w["origin"], si[:7], w["truth"][j])["returns_tracking"]
        hk, _ = orc.adaptive_voxel_filter(pts, o.hi_max_length, o.hi_min_num_points, o.hi_max_range)
        lk, _ = orc.adaptive_voxel_filter(pts, o.lo_max_length, o.lo_min_num_points, o.lo_max_range)
        g = np.array(w["truth"][j], np.float64)
        g[:3] += rng.uniform(-1, 1, 3) * [2.0, 2.0, 0.4]
        his.append(pts[hk]); los.append(pts[lk]); guesses.append(g); nodes.append(1000 * rank + j)
    return {"hi": his, "lo": los, "guesses": np.array(guesses), "nodes": nodes, "submaps": [rank] * args.pairs}


def pose_errors(a, b):
    dt = np.linalg.norm(a[:, :3] - b[:, :3], axis=1)
    qa = a[:, 3:7] / np.linalg.norm(a[:, 3:7], axis=1, keepdims=True)
    qb = b[:, 3:7] / np.linalg.norm(b[:, 3:7], axis=1, keepdims=True)
    d = np.abs(np.sum(qa * qb, axis=1)).clip(max=1.0)
    return dt, 2 * np.arccos(d)


def struct_rows(records, struct):
    """(len(records), k) float64 of a ctypes struct's scalar and array fields, in declaration order; nested structs and
    `reserved` are left out (integers up to 2^53 are exact in float64)."""
    rows = []
    for r in records:
        row = []
        for name, _ in struct._fields_:
            v = getattr(r, name)
            if name == "reserved" or isinstance(v, C.Structure):
                continue
            row.extend(v[:] if isinstance(v, C.Array) else [v])
        rows.append(row)
    return np.array(rows, np.float64)


def dump_outputs(path, dliom, results, states, table):
    """What the last timed step hands its caller, one float64 .npy per array (columns in the C struct's field order):
    states (B, 16) p q v ba bg after the solve; scan_results (B, 25) = dl_scan_result without its solve summary;
    solve_summary (B, 7) = dl_solve_summary; constraints (rows, 15) = the exchange step's dl_constraint_row table (not
    written with --pairs 0)."""
    os.makedirs(path, exist_ok=True)
    arrays = {"states": np.asarray(states, np.float64), "scan_results": struct_rows(results, dliom.ScanResult),
              "solve_summary": struct_rows([r.summary for r in results], dliom.SolveSummary)}
    if table is not None:
        arrays["constraints"] = struct_rows(table, dliom.ConstraintRow)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons at 2 Hz from before the warm-up to after the last timed region (a subprocess every
    500 ms; round 1 sampled at 10 Hz, which showed up as noise in a 33 ms timed region)."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.samples, self.stop_flag, self.mark = gpu_index, [], False, False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.QUERY}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 9:
                    self.samples.append((self.mark, f))
            except Exception:
                pass
            time.sleep(0.5)

    def summary(self):
        loaded = [f for m, f in self.samples if m] or [f for _, f in self.samples]
        if not loaded:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[1]) for s in loaded)
        reasons = set()
        for s in loaded:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(loaded[0][2]), "reasons": sorted(reasons),
                "samples": len(sm), "note": "nvidia-smi at 2 Hz while the timed loops run (median over those samples)"}


def cpu_chain(w, sel, threads):
    orc = w["orc"]
    return orc.frontend_batch_imu(w["opts"], [w["scans"][i] for i in sel], w["origin"], IMU_NOISE, w["states_i"][sel],
                                  [w["intervals"][i] for i in sel], w["submap_pose"], w["hi"], w["lo"], threads,
                                  imu_weight=IMU_WEIGHT)


def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path (oracle port of the same chain) on all host threads."""
    if rank != 0:
        return
    w = build_workload(args, 0)
    threads, cpu_note = usable_cpus()
    sample = max(args.batch, 8 * threads)   # >= 8 scans per pooled thread, handed out from a work queue
    sel = [i % args.batch for i in range(sample)]
    cpu_chain(w, sel[:threads], threads)    # spawn the pool
    times = []
    for step in range(args.warmup + args.steps):
        secs = cpu_chain(w, sel, threads)[0]
        if step >= args.warmup:
            times.append(secs)
    ms = 1e3 * float(np.median(times))
    value = sample / (ms / 1e3)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "impl": "reference",
            "config": workload_config(args, args.batch),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "physical_cores": physical_cores(), "kind": "port",
                             "cpus": cpu_note,
                             "sample": f"{sample} scans per step ({args.batch} distinct, cycled), median of {args.steps} steps, "
                                       f"persistent pool of {threads} threads fed from a work queue"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def workload_config(args, batch):
    return {"workload": f"configs[1]: {args.beams}-beam scans (~130k pts) + 200 Hz IMU (20 samples per scan, pre-integrated on the "
                        f"device inside the step) vs one submap (0.1 m / 0.45 m), whole front-end hot path, pipeline-faithful "
                        f"filters, IMU residual fused into the solve; + configs[4] exchange step ({args.pairs} loop-closure "
                        f"searches per rank, ncclAllGather of the constraint rows)",
            "imu": True, "scans_per_step_per_gpu": batch, "distinct_scans": batch, "beams": args.beams,
            "map_scans": args.map_scans, "row_bytes": 4 * args.row_floats,
            "row_layout": {3: "x y z (12 B) + per-point times as runs", 4: "x y z t (16 B)", 8: "RangeMeasurement (32 B)"}[args.row_floats],
            "l2_policy": f"inputs ({batch} x {130605 * 4 * args.row_floats / 1e6:.1f} MB) exceed the 126 MB L2; no explicit flush",
            "parallelism": f"scans sharded over {args.gpus} gpu(s); loop-closure pairs sharded by submap owner, one ncclAllGather per step",
            "exchange_thread": f"each step's exchange (searches + all-gather + table on the host) is issued from one of "
                               f"{args.exchange_threads} background host threads (own context + NCCL communicator each, step k -> "
                               "thread k mod T), like the reference's constraint-builder pool; every one of the K exchanges completes "
                               "inside the timed region"}


_T0 = time.perf_counter()


def note(msg):
    """Phase marker on stderr (stdout carries the JSON line only)."""
    print(f"[bench {time.perf_counter() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=148, help="scans per step per GPU (default: one per SM)")
    ap.add_argument("--beams", type=int, default=64)
    ap.add_argument("--map-scans", type=int, default=40)
    ap.add_argument("--pairs", type=int, default=8, help="loop-closure (node, submap) searches per rank and step")
    ap.add_argument("--exchange-threads", type=int, default=2,
                    help="host threads (each with its own context and NCCL communicator) that run the exchange steps; step k "
                         "goes to thread k mod T on every rank, so the collectives pair up")
    ap.add_argument("--cpu-sample", type=int, default=0, help="scans in the cpu_baseline sample (0 = 8 x threads)")
    ap.add_argument("--row-floats", type=int, default=3, choices=[3, 4, 8],
                    help="3: x y z rows + the per-point times as runs (12 B/point); 4: TimedPointCloud rows x y z t (what AddRangeData "
                         "receives); 8: RangeMeasurement rows")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[2] / mode-F / no-IMU extra measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step (rank 0) to DIR/<name>.npy (see dump_outputs())")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the device path's results: use it with --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import dliom
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = f"cuda:{local_rank}"
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    w = build_workload(args, rank)
    B = args.batch
    ctx, ctx2 = dliom.Context(local_rank), dliom.Context(local_rank)
    xctxs = [dliom.Context(local_rank) for _ in range(max(1, args.exchange_threads))]   # one context per exchange thread
    ctx3 = xctxs[0]
    hi, lo = ctx.grid(0.1), ctx.grid(0.45)
    hi.set_cells(*w["hi"].export())
    lo.set_cells(*w["lo"].export())
    fo = dliom.FrontendOptions.from_oracle(w["opts"])
    fo.range_row_floats = args.row_floats
    row_bytes = 4 * args.row_floats
    runs_bytes = 0
    if args.row_floats == 3:   # bare x y z rows; the times travel as ~2 k runs per sweep (bit-identical deskew)
        runs_bytes = dliom.TimeRuns([s["t"] for s in w["scans"]], pin=True).attach(fo)._time_runs.nbytes

    sizes = np.array([len(s) for s in w["scans"]], np.int64)
    cap = int(sizes.max())
    # pinned host staging (e2e) and the HBM-resident copy (value)
    host = torch.zeros((B, cap, row_bytes), dtype=torch.uint8).pin_memory()
    for b, s in enumerate(w["scans"]):
        host[b, :len(s)] = torch.from_numpy(s.view(np.uint8).reshape(-1, 32)[:, :row_bytes].copy())
    dev = host.to(device)
    fo.host_scan_stride_rows = cap   # the pinned staging tensor is (B, cap, row_bytes): one allocation, constant stride
    host_rows = dliom.HostScanBatch([host[b, :int(sizes[b])].numpy() for b in range(B)])
    host2 = host.clone().pin_memory()   # second pinned copy + second context for the streaming e2e loop (double buffering)
    host_rows2 = dliom.HostScanBatch([host2[b, :int(sizes[b])].numpy() for b in range(B)])
    imus = [dliom.ImuSamples(IMU_NOISE, w["intervals"], w["states_i"], imu_weight=IMU_WEIGHT, pin=True) for _ in range(2)]
    imu_bytes = int(imus[0].dt.nbytes + imus[0].acc.nbytes + imus[0].gyr.nbytes + imus[0].states.nbytes + imus[0].offsets.nbytes)
    stream = torch.cuda.ExternalStream(ctx.stream, device=device)

    res_bytes = B * C.sizeof(dliom.ScanResult)
    dev_lanes = [(c, torch.zeros(res_bytes, dtype=torch.uint8, device=device), torch.zeros((B, 16), dtype=torch.float64, device=device), im)
                 for c, im in zip((ctx, ctx2), imus)]

    # ---- the exchange step: NCCL communicators owned by the C-ABI library, created from ids that torch.distributed carries
    comms = []
    for xc in xctxs:
        idt = torch.zeros(128, dtype=torch.uint8, device=device)
        if rank == 0:
            idt.copy_(torch.tensor(list(dliom.comm_unique_id()), dtype=torch.uint8))
        if dist is not None:
            dist.broadcast(idt, 0)
        comms.append(dliom.Comm(xc, bytes(idt.cpu().numpy().tolist()), rank, world))
        xc.set_blocking_sync(True)   # exchange threads sleep in their waits: the box grants 16 CPUs for up to 8 ranks x 4 threads
    comm = comms[0]
    lc = loop_closure_pairs(w, args, rank) if args.pairs > 0 else None
    copt = dliom.ConstraintOptions.defaults(min_score=0.3, min_low_resolution_score=0.3, xy_window=3.0, z_window=0.5)
    exchange = {"ms": [], "found": 0, "bytes": 0, "rows": 0}

    plans = []
    if args.pairs > 0:
        plans = [xc.constraint_exchange_plan(cm, copt, args.pairs, lc["submaps"], lc["nodes"], lc["guesses"], lc["hi"], lc["lo"],
                                             [hi] * args.pairs, [lo] * args.pairs) for xc, cm in zip(xctxs, comms)]
    exchange_lock = threading.Lock()

    class ExchangeWorker(threading.Thread):
        """The exchange steps run on their own host thread and context, like the reference's constraint builder, whose searches
        run on a background thread pool next to the front end (constraint_builder_3d.cc:189-197): step k's search + all-gather
        overlaps the front end of step k+1 instead of blocking the thread that launches it. submit() queues one exchange,
        drain() returns when every queued exchange has completed (each one ends with a device sync and the table on the host)."""

        def __init__(self, plan):
            super().__init__(daemon=True)
            self.plan = plan
            self.cv = threading.Condition()
            self.pending = 0
            self.error = None
            self.stop = False
            self.table = None   # the constraint table of this worker's latest exchange
            self.start()

        def run(self):
            while True:
                with self.cv:
                    while self.pending == 0 and not self.stop:
                        self.cv.wait()
                    if self.stop:
                        return
                try:
                    table, info = self.plan()
                    self.table = table
                    with exchange_lock:
                        exchange["ms"].append(info.collective_ms)
                        exchange["found"] = info.found_total
                        exchange["bytes"] = int(info.bytes_received)
                        exchange["rows"] = len(table)
                except Exception as e:   # surfaced by drain()
                    self.error = e
                with self.cv:
                    self.pending -= 1
                    self.cv.notify_all()

        def submit(self):
            with self.cv:
                self.pending += 1
                self.cv.notify_all()

        def drain(self):
            with self.cv:
                while self.pending > 0:
                    self.cv.wait()
            if self.error is not None:
                raise self.error

        def close(self):
            with self.cv:
                self.stop = True
                self.cv.notify_all()

    workers = [ExchangeWorker(p) for p in plans]
    submitted = [0]

    def step_exchange():
        if workers:                # --pairs 0: front end only (experiments)
            workers[submitted[0] % len(workers)].submit()   # same assignment on every rank: the all-gathers pair up
            submitted[0] += 1

    def drain_exchange():
        for wk in workers:
            wk.drain()

    def step_dev(i, options=None, lanes=None):
        """One pass of the hot path over the HBM-resident batch. Successive steps alternate between two contexts (own
        streams, own scratch), so the latency-bound back half of step i overlaps the front half of step i+1."""
        c, out, st, im = (lanes or dev_lanes)[i % 2]
        c.frontend_match_batch_imu_samples_dev(options or fo, im, C.c_void_p(dev.data_ptr()), cap, sizes, w["origin"],
                                               w["submap_pose"], hi, lo, C.c_void_p(out.data_ptr()), C.c_void_p(st.data_ptr()))

    lanes = [(ctx, host_rows, imus[0]), (ctx2, host_rows2, imus[1])]

    def run_streaming(steps, with_exchange=True):
        """K batches through dl_frontend_submit_imu_samples / dl_frontend_collect_imu on two alternating contexts: batch i+1 is
        uploading while batch i computes; every batch's inputs cross PCIe and every batch's results are read back."""
        out = None
        for i in range(steps):
            c, rows, im = lanes[i & 1]
            if i >= 2:
                out = c.frontend_collect_imu()
            c.frontend_submit_imu_samples(fo, rows, w["origin"], im, w["submap_pose"], hi, lo)
            if with_exchange:
                step_exchange()
        for i in range(max(steps - 2, 0), steps):
            out = lanes[i & 1][0].frontend_collect_imu()
        if with_exchange:
            drain_exchange()
        return out

    def barrier():
        torch.cuda.synchronize()
        for c in [ctx, ctx2] + xctxs:
            c.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_device_loop(steps, options=None, with_exchange=True):
        """CUDA events on the launching streams: the first context's stream opens the region; the closing event is recorded on
        the same stream after it has been made to wait for the other contexts' streams (event waits, no host sync)."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        others = [torch.cuda.ExternalStream(c.stream, device=device) for c in [ctx2] + xctxs]
        barrier()
        gate = torch.cuda.Event()
        gate.record(stream)
        for s2 in others:
            s2.wait_event(gate)           # no context starts before e0
        e0.record(stream)
        for k in range(steps):
            step_dev(k, options)
            if with_exchange:
                step_exchange()
        if with_exchange:
            drain_exchange()          # every exchange of the region has run (and synchronised its context) before the closing event
        for s2 in others:
            tail = torch.cuda.Event()
            tail.record(s2)
            stream.wait_event(tail)
        e1.record(stream)
        barrier()
        return e0.elapsed_time(e1)

    note("workload built, contexts created")
    sampler = ClockSampler(local_rank)
    sampler.start()
    # ---- warm-up (both paths)
    warm = max(args.warmup, 1)   # at least one untimed pass: scratch arenas are sized on first use
    for k in range(2 * warm):
        step_dev(k)
        step_exchange()
    drain_exchange()
    run_streaming(max(warm, 2))
    barrier()
    res = ctx.fetch_results(C.c_void_p(dev_lanes[0][1].data_ptr()), B)
    states = dev_lanes[0][2].cpu().numpy()

    note("warm-up done")
    # ---- timed: device-resident
    sampler.mark = True
    ctx.set_profiling(True)
    ctx.read_profile()
    exchange["ms"].clear()
    launches0 = sum(c.launches for c in [ctx, ctx2] + xctxs)
    ms_total = timed_device_loop(args.steps)
    launches = sum(c.launches for c in [ctx, ctx2] + xctxs) - launches0
    profile = ctx.read_profile()
    ctx.set_profiling(False)
    if args.dump_outputs:   # read back before the later loops reuse the lanes; the last step ran on lane (steps - 1) % 2
        c_last, out_last, st_last, _ = dev_lanes[(args.steps - 1) % 2]
        last_step = (c_last.fetch_results(C.c_void_p(out_last.data_ptr()), B), st_last.cpu().numpy(),
                     workers[(submitted[0] - 1) % len(workers)].table if workers else None)
    collective_ms = float(np.median(exchange["ms"])) if exchange["ms"] else None
    note("device-resident loop done")
    # ---- timed: end to end (host buffers in, results out), streaming and blocking
    barrier()
    t0 = time.perf_counter()
    res_stream, states_stream = run_streaming(args.steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    sync_steps = max(3, min(args.steps, 20))
    barrier()
    t0 = time.perf_counter()
    for _ in range(sync_steps):
        res_e2e, states_e2e, _ = ctx.frontend_match_batch_imu_samples(fo, host_rows, w["origin"], imus[0], w["submap_pose"], hi, lo)
    barrier()
    e2e_sync_s = (time.perf_counter() - t0) / sync_steps
    sampler.mark = False
    stream_equal = bool(np.array_equal(states_stream, states_e2e) and
                        all(list(a.pose_estimate_local) == list(c.pose_estimate_local) and a.ok == c.ok and
                            a.num_returns == c.num_returns for a, c in zip(res_stream, res_e2e)))
    dev_equal = bool(np.array_equal(states, states_e2e))
    # ---- stage durations with NOTHING overlapping: one context, its sub-batches back to back on one stream, a synchronise between steps. These are
    # the kernels' own launch durations (what a roofline compares with a peak); the per-stage times of the timed region above are
    # stretched by whatever the other context / sub-batch stream / exchange runs at the same time.
    serial_steps = 6
    os.environ["DLIOM_SERIAL"] = "1"
    for _ in range(2):
        step_dev(0)
        ctx.synchronize()
    ctx.set_profiling(True)
    ctx.read_profile()
    for _ in range(serial_steps):
        step_dev(0)
        ctx.synchronize()
    profile_serial = ctx.read_profile()
    ctx.set_profiling(False)
    del os.environ["DLIOM_SERIAL"]
    barrier()
    note("e2e loops done")
    # ---- latency of ONE scan through the blocking call (what a 10 Hz single-trajectory node sees)
    one = dliom.HostScanBatch([host[0, :int(sizes[0])].numpy()])
    imu_one = dliom.ImuSamples(IMU_NOISE, w["intervals"][:1], w["states_i"][:1], imu_weight=IMU_WEIGHT)
    fo_one = dliom.FrontendOptions.from_oracle(w["opts"])
    fo_one.range_row_floats = args.row_floats
    if args.row_floats == 3:
        dliom.TimeRuns([w["scans"][0]["t"]]).attach(fo_one)
    lat = []
    for _ in range(25):
        t1 = time.perf_counter()
        ctx.frontend_match_batch_imu_samples(fo_one, one, w["origin"], imu_one, w["submap_pose"], hi, lo)
        lat.append((time.perf_counter() - t1) * 1e3)
    single_scan_ms = float(np.median(lat[5:]))
    # ---- the PCIe ceiling of the e2e number: the same pinned bytes copied with nothing else running
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dev.copy_(host, non_blocking=True)
    torch.cuda.synchronize()
    c0.record()
    for _ in range(5):
        dev.copy_(host, non_blocking=True)
    c1.record()
    torch.cuda.synchronize()
    h2d_gbs = 5 * host.numel() / (c0.elapsed_time(c1) * 1e-3) / 1e9

    note("latency + PCIe ceiling done")
    # ---- extra keys (N = 1 only): the same step without the exchange, the plain (no IMU) solve, mode F, configs[2]
    extras = {}
    if world == 1 and not args.no_extras:
        def fetch_lane0():
            ctx.synchronize()
            return ctx.fetch_results(C.c_void_p(dev_lanes[0][1].data_ptr()), B)
        extras = measure_extras(args, w, dliom, ctx, timed_device_loop, fetch_lane0, B, fo, hi, lo)

    note("extras done")
    t = torch.tensor([ms_total, e2e_s * 1e3, e2e_sync_s * 1e3, collective_ms or 0.0], dtype=torch.float64, device=device)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms_total, e2e_sync_ms, collective_ms_max = float(t[0]), float(t[1]), float(t[2]), float(t[3])
    ms_step = ms_total / args.steps
    value = world * B / (ms_step / 1e3)
    e2e_value = world * B / (e2e_ms_total / args.steps / 1e3)

    if rank == 0:
        # ---- roofline of the dominant stage from the per-stage CUDA-event times (algorithmic bytes, SURVEY 8d)
        n_raw = float(sizes.sum())
        n1 = sum(r.num_first_filter for r in res)
        n2 = sum(r.num_returns for r in res)
        evals = sum(r.summary.num_evaluations * (r.num_high_resolution + r.num_low_resolution) for r in res)
        adaptive_bytes = sum(12.0 * (r.num_cropped_high * r.num_passes_high + r.num_cropped_low * r.num_passes_low) +
                             12.0 * (r.num_high_resolution + r.num_low_resolution) for r in res)
        stage_bytes = {
            "voxel_filter_first": 16.0 * n_raw + 16.0 * n1,                          # 16 N_in + 16 N_out (SURVEY 8d's model; 12 B rows read less)
            "ingest_second_filter": 28.0 * n1 + 12.0 * n1 + 12.0 * n2,               # ingest 28 N + second pass 12 N_in + 12 N_out
            "adaptive_voxel_filter": adaptive_bytes,
            "nls_solve": 28.0 * evals,
            "imu_preintegrate_predict": float(imu_bytes),
        }
        steps_profiled = max(1, (args.steps + 1) // 2)   # the profiled context runs every other step of the timed region
        stages = {}
        for k, v in profile_serial.items():
            per_step = v[0] / serial_steps
            over = profile.get(k, (0.0, 0))[0] / steps_profiled
            stages[k] = {"ms_per_step": per_step, "ms_per_step_overlapped": over, "bytes_per_step": stage_bytes.get(k)}
        dom = max((k for k in stages if stage_bytes.get(k)), key=lambda k: stages[k]["ms_per_step"])
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_kind = "of measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "of fallback (6.65 TB/s)"
        achieved = (stages[dom]["bytes_per_step"] or 0.0) / (stages[dom]["ms_per_step"] * 1e-3) / 1e9
        achieved_over = (stages[dom]["bytes_per_step"] or 0.0) / (max(stages[dom]["ms_per_step_overlapped"], 1e-9) * 1e-3) / 1e9
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(dom)
        except Exception:
            pass
        roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic, "peak_kind": peak_kind,
                    "achieved_overlapped": achieved_over, "frac_overlapped": achieved_over / peak,
                    "units": "achieved = algorithmic bytes of one STEP (148 scans, SURVEY 8d's per-point figures) / the stage's own "
                             "device time per step: CUDA events around the stage's launches with nothing else on the GPU (one "
                             f"context, its two sub-batches of 74 scans back to back on one stream, {serial_steps} steps after the timed loops); achieved_overlapped divides by "
                             "the same events' time inside the timed region, where two contexts, two sub-batch streams and the "
                             "exchange share the GPU; traffic = ncu dram bytes of the stage's kernels per STEP (profiles/)",
                    "stages": {k: {"ms_per_step": round(v["ms_per_step"], 4),
                                   "ms_per_step_overlapped": round(v["ms_per_step_overlapped"], 4),
                                   "gbps": None if not v["bytes_per_step"] else round(v["bytes_per_step"] / (v["ms_per_step"] * 1e-3) / 1e9, 2)}
                               for k, v in stages.items()},
                    "stages_note": "ms_per_step: the stage alone; ms_per_step_overlapped: inside the timed region (they overlap "
                                   "there, so they sum to more than the step)",
                    "serial_step_ms": round(sum(v["ms_per_step"] for k, v in stages.items() if k != "imu_preintegrate_predict"), 4),
                    "whole_step_gbps": round(sum(v for v in stage_bytes.values()) / (ms_step * 1e-3) / 1e9, 1)}

        # ---- CPU baseline (oracle chain) on a bounded sample, and pose parity of the GPU batch against it
        cpu = None
        parity = None
        if world == 1:
            threads, cpu_note = usable_cpus()
            sample = args.cpu_sample or max(B, 8 * threads)
            sel = [i % B for i in range(sample)]
            cpu_chain(w, sel[:threads], threads)   # spawn the pool
            runs = [cpu_chain(w, sel, threads) for _ in range(3)]
            secs = float(np.median([r[0] for r in runs]))
            one_n = 16
            secs1 = cpu_chain(w, list(range(one_n)), 1)[0]
            cpu = {"value": sample / secs, "unit": UNIT, "cores": threads, "physical_cores": physical_cores(), "kind": "port",
                   "cpus": cpu_note,
                   "sample": f"{sample} scans ({B} distinct, cycled; {secs:.2f} s, median of 3), persistent pool of {threads} threads "
                             f"fed from a work queue",
                   "all_cores": sample / secs, "single_thread": one_n / secs1,
                   "single_thread_note": "the reference's real mode: one front-end thread, Ceres num_threads = 1"}
            want = cpu_chain(w, list(range(B)), threads)
            dt, dr = pose_errors(states, want[1])
            ok_cpu = want[3]
            parity = {"scans": B, "distinct_scans": B, "rmse_m": float(np.sqrt(np.mean(dt ** 2))),
                      "rmse_rad": float(np.sqrt(np.mean(dr ** 2))), "max_m": float(dt.max()), "max_rad": float(dr.max()),
                      "max_velocity_diff": float(np.abs(states[:, 7:10] - want[1][:, 7:10]).max()),
                      "max_bias_diff": float(np.abs(states[:, 10:] - want[1][:, 10:]).max()),
                      "same_iteration_counts": bool(all(r.summary.num_iterations == it for r, it in zip(res, want[4]))),
                      "all_ok": bool(all(r.ok == 1 for r in res) and all(ok_cpu == 1))}

        h2d = int(sizes.sum() * row_bytes) + imu_bytes + runs_bytes
        d2h = int(B * (C.sizeof(dliom.ScanResult) + 128))
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32 (indices, scores) + f64 (pre-integration, least squares)", "data": "synthetic",
                "config": workload_config(args, B),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": e2e_ms_total / args.steps,
                        "timing": "wall clock around K x (dl_frontend_submit_imu_samples, dl_frontend_collect_imu) on two alternating "
                                  "contexts + the exchange step: batch i+1 uploads while batch i computes; all K uploads, solves and "
                                  "result reads inside",
                        "sync_call": {"value": world * B / e2e_sync_ms * 1e3, "ms_per_step": e2e_sync_ms,
                                      "note": "one blocking dl_frontend_match_batch_imu_samples per step, nothing overlaps across steps"},
                        "streaming_equals_sync_results": stream_equal, "device_resident_equals_sync_results": dev_equal,
                        "pcie_h2d_gbs": round(h2d_gbs, 2), "copy_only_ms_per_step": round(h2d / h2d_gbs / 1e6, 3),
                        "pcie_note": "plain pinned cudaMemcpyAsync of the same buffers, measured in this run: the floor of e2e"},
                "collective": {"name": "ncclAllGather (dl_constraint_search_exchange)", "ranks": world,
                               "bytes": exchange["bytes"], "rows": exchange["rows"], "ms": collective_ms_max,
                               "searches_per_rank_per_step": args.pairs, "constraints_found": exchange["found"],
                               "note": "device time of the all-gather alone (CUDA events), median over the timed steps, max over "
                                       "ranks; the searches that feed it are inside the step time"},
                "latency": {"single_scan_ms": round(single_scan_ms, 3),
                            "note": "median wall time of dl_frontend_match_batch_imu_samples on ONE 64-beam scan (2.1 MB upload, result "
                                    "download); the CPU path takes 1000 / cpu_baseline.single_thread ms"},
                "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "parity_vs_cpu": parity,
                "clocks": sampler.summary()}
        line.update(extras)
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dliom, *last_step)
    note("line printed")
    sampler.stop_flag = True
    for wk in workers:
        wk.close()
        wk.join(timeout=5)
    for cm in comms:
        cm.close()
    if dist is not None:
        dist.destroy_process_group()
    note("done")


def measure_extras(args, w, dliom, ctx, timed_device_loop, fetch_lane0, B, fo, hi=None, lo=None):
    """Secondary measurements at N = 1: each is its own short device-timed loop over the same resident batch."""
    extras = {}
    steps = max(10, min(args.steps, 30))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    try:
        ms = timed_device_loop(steps, with_exchange=False)
        extras["front_end_only"] = {"value": B / (ms / steps / 1e3), "unit": UNIT, "ms_per_step": ms / steps,
                                    "note": "the same IMU-coupled step without the loop-closure exchange step"}
    except Exception as e:   # an extra must never take the headline down with it
        extras["front_end_only"] = {"error": str(e)}
    try:
        # mode F (SURVEY 8d): adaptive filters pass everything through, the matcher sees the whole filtered cloud
        ff = dliom.FrontendOptions.from_buffer_copy(fo)     # same rows / time runs as the headline step
        ff.high_resolution_adaptive_voxel_filter.min_num_points = 1e9
        ff.low_resolution_adaptive_voxel_filter.min_num_points = 1e9
        timed_device_loop(2, ff, with_exchange=False)
        ctx.set_profiling(True)
        ctx.read_profile()
        k = 6
        msf = timed_device_loop(k, ff, with_exchange=False)
        prof = ctx.read_profile()
        ctx.set_profiling(False)
        res = fetch_lane0()
        pts = sum(r.num_high_resolution + r.num_low_resolution for r in res)
        evals = sum(r.summary.num_evaluations * (r.num_high_resolution + r.num_low_resolution) for r in res)
        nls_ms = prof.get("nls_solve", (0.0, 0))[0] / (k / 2)
        achieved = 28.0 * evals / (nls_ms * 1e-3) / 1e9 if nls_ms > 0 else None
        extras["mode_F"] = {"value": B / (msf / k / 1e3), "unit": UNIT, "ms_per_step": msf / k,
                            "matcher_points_per_scan": pts / B, "evaluations_per_scan": sum(r.summary.num_evaluations for r in res) / B,
                            "stages_ms_per_step": {n: round(v[0] / (k / 2), 4) for n, v in prof.items()},
                            "roofline": {"bound": "hbm", "kernel": "nls_fused_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                                         "frac": None if achieved is None else achieved / peak, "traffic": None,
                                         "bytes_model": "28 B per point per evaluation (12 B point + 8 corners x 2 B), SURVEY 8d"},
                            "all_ok": bool(all(r.ok == 1 for r in res)),
                            "note": "full-cloud mode: adaptive filters pass-through (min_num_points = 1e9), the fused solve sees every "
                                    "point of the second voxel filter's output"}
    except Exception as e:
        extras["mode_F"] = {"error": str(e)}
    try:
        extras["configs2"] = measure_configs2(args, w, dliom, ctx, peak)
    except Exception as e:
        extras["configs2"] = {"error": repr(e)}
    try:
        extras["loop_closure"] = measure_loop_closure(args, w, dliom, ctx, hi, lo)
    except Exception as e:
        extras["loop_closure"] = {"error": repr(e)}
    return extras


def measure_loop_closure(args, w, dliom, ctx, hi, lo, submaps=32, nodes=8, steps=5):
    """BASELINE configs[3] shape: submaps x nodes (node, submap) constraint searches per step — coarse translation search over the
    stock 5 m x 5 m x 1 m window (214 221 leaves at 0.1 m) + least-squares refinement, ConstraintBuilder3D::ComputeConstraint —
    through the host-buffer call dl_constraint_search_batch (clouds and guesses in, constraints out), wall clock. Every pair
    searches the bench's one submap (the grids are what a search reads; 32 copies would only add HBM), with its own guess."""
    from concurrent.futures import ThreadPoolExecutor
    orc = w["orc"]
    lcw = loop_closure_pairs(w, argparse.Namespace(pairs=nodes), 0)
    rng = np.random.RandomState(31)
    his, los, guesses = [], [], []
    for s in range(submaps):
        for n in range(nodes):
            g = np.array(lcw["guesses"][n], np.float64)
            g[:3] += rng.uniform(-1, 1, 3) * [1.0, 1.0, 0.2]
            his.append(lcw["hi"][n]); los.append(lcw["lo"][n]); guesses.append(g)
    count = len(guesses)
    opt = dliom.ConstraintOptions.defaults(min_score=0.3, min_low_resolution_score=0.3)
    call = dict(pose_guesses=np.array(guesses), hi_clouds=his, lo_clouds=los, hi_grids=[hi] * count, lo_grids=[lo] * count)
    cons = ctx.constraint_search_batch(opt, **call)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        cons = ctx.constraint_search_batch(opt, **call)
        times.append(time.perf_counter() - t0)
    secs = float(np.median(times))
    found = sum(1 for c in cons if c.found)
    # CPU: the oracle's branch and bound (precomputation stack built once per submap, outside the timed sample) + its LM refine
    threads, cpu_note = usable_cpus()
    t0 = time.perf_counter()
    matcher = orc.FastCorrelativeScanMatcher(w["hi"], w["lo"], min_low_resolution_score=0.3)
    stack_s = time.perf_counter() - t0

    def cpu_pair(i):
        c = matcher.match(his[i], los[i], guesses[i], 0.3)
        if c.found:
            cp = np.array(c.pose[:])
            orc.ceres_match([his[i], los[i]], [w["hi"], w["lo"]], [5.0, 30.0], 10.0, 1.0, cp[:3], cp, max_iter=10)
        return bool(c.found)
    sample = list(range(min(count, 4 * threads)))
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        found_cpu = sum(ex.map(cpu_pair, sample))
    cpu_s = time.perf_counter() - t0
    same = all(bool(cons[i].found) == f for i, f in zip(sample, ThreadPoolExecutor(threads).map(cpu_pair, sample[:8])))
    return {"value": count / secs, "unit": "searches/s", "ms_per_step": 1e3 * secs, "searches_per_step": count,
            "workload": f"configs[3] shape: {submaps} x {nodes} (node, submap) pairs per step, window 5 m x 5 m x 1 m at 0.1 m = 214 221 "
                        f"leaves per search, min_score 0.3, {int(np.mean([len(c) for c in his]))} / {int(np.mean([len(c) for c in los]))} points "
                        f"(high / low resolution) per node; host buffers in, constraints out (wall clock, median of {steps})",
            "constraints_found": found,
            "cpu_baseline": {"value": len(sample) / cpu_s, "unit": "searches/s", "cores": threads, "cpus": cpu_note, "kind": "port",
                             "sample": f"{len(sample)} searches on {threads} threads ({cpu_s:.2f} s), found {found_cpu}; the "
                                       f"precomputation stack ({stack_s:.2f} s per submap, built once) is outside the sample"},
            "found_flags_equal_cpu_first8": bool(same)}


def measure_configs2(args, w, dliom, ctx, peak, num_scans=16, map_scans=12, steps=3):
    """BASELINE configs[2]: 128-beam scans (~256k pts) against a 0.05 m submap, correlative search (RT-CSM, 0.15 m / 1 deg
    window -> 7^3 x 11^3 = 456 533 candidates per scan) + least-squares refine, device-resident batch, plain (no IMU) solve."""
    import torch
    import synth
    orc = w["orc"]
    scene = synth.Scene(42)
    opts = orc.FrontEndOptions.defaults()
    origin = np.zeros((1, 3), np.float32)
    hi, lo = ctx.grid(0.05), ctx.grid(0.45)
    og = orc.Grid(0.05)
    ident = orc.IDENTITY_POSE.copy()
    t0 = 2.0
    for k in range(map_scans):       # the submap is built ON THE DEVICE (dl_submap_insert_range_data, bit-exact vs the oracle's inserter)
        t = t0 + 0.1 * k
        rows = synth.make_scan(scene, 128, t)
        cur = synth.pose7(t)
        ing = orc.ingest_scan(opts, rows, origin, synth.pose7(t - 0.1), cur)
        local = apply_pose(cur, ing["returns_tracking"].astype(np.float64)).astype(np.float32)
        ctx.submap_insert_range_data(hi, lo, ident, cur[:3].astype(np.float32), local, high_resolution_max_range=20)
        o3 = cur[:3].astype(np.float32)
        og.insert_range_data(o3, local[np.linalg.norm(local - o3, axis=1) <= 20.0])   # the checker's copy, for parity_scan0
    rng = np.random.RandomState(77)
    scans, prevs, curs = [], [], []
    for j in range(num_scans):
        t = t0 + 0.05 + 0.1 * (map_scans - 2) * j / num_scans
        scans.append(synth.make_scan(scene, 128, t))
        prevs.append(synth.pose7(t - 0.1))
        curs.append(synth.perturb_pose(synth.pose7(t), rng, 0.1, 0.5))
    prevs, curs = np.array(prevs), np.array(curs)
    fo = dliom.FrontendOptions.from_oracle(opts)
    fo.range_row_floats = 4
    fo.use_online_correlative_scan_matching = 1
    fo.real_time_correlative_scan_matcher = dliom.RtcsmOptions(0.15, np.deg2rad(1.0), 1e-1, 1e-1)
    sizes = np.array([len(s) for s in scans], np.int64)
    cap = int(sizes.max())
    host = torch.zeros((num_scans, cap, 16), dtype=torch.uint8)
    for b, sc in enumerate(scans):
        host[b, :len(sc)] = torch.from_numpy(sc.view(np.uint8).reshape(-1, 32)[:, :16].copy())
    dev = host.cuda()
    out = torch.zeros(num_scans * C.sizeof(dliom.ScanResult), dtype=torch.uint8, device="cuda")

    def step():
        ctx.frontend_match_batch_dev(fo, C.c_void_p(dev.data_ptr()), cap, sizes, origin, prevs, curs, ident, hi, lo,
                                     C.c_void_p(out.data_ptr()))
    step()
    ctx.synchronize()
    stream = torch.cuda.ExternalStream(ctx.stream)
    ctx.set_profiling(True)
    ctx.read_profile()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    ctx.synchronize()
    ms = e0.elapsed_time(e1) / steps
    prof = ctx.read_profile()
    ctx.set_profiling(False)
    res = ctx.fetch_results(C.c_void_p(out.data_ptr()), num_scans)
    # algorithmic bytes of the correlative stage: R (12 N + 2 N L) per scan (SURVEY 8d) with the window the library derived
    n_hi = np.array([r.num_high_resolution for r in res], np.float64)
    R, L = 11 ** 3, 7 ** 3
    csm_bytes = float(np.sum(R * (12.0 * n_hi + 2.0 * n_hi * L)))
    csm_ms = prof.get("rtcsm", (0.0, 0))[0] / steps
    achieved = csm_bytes / (csm_ms * 1e-3) / 1e9 if csm_ms > 0 else None
    # one scan against the oracle's exhaustive search (bit-exact score, same pose), ~seconds of CPU
    ing = orc.ingest_scan(opts, scans[0], origin, prevs[0], curs[0])
    pts = ing["returns_tracking"]
    hk, _ = orc.adaptive_voxel_filter(pts, opts.hi_max_length, opts.hi_min_num_points, opts.hi_max_range)
    init = np.concatenate([ing["current_pose"][:3].astype(np.float64), ing["current_pose"][3:].astype(np.float64)])
    want = orc.rtcsm_match(og, pts[hk], init, 0.15, np.deg2rad(1.0), 1e-1, 1e-1)
    return {"value": num_scans / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "scans_per_step": num_scans,
            "workload": "configs[2]: 128-beam scans (~256k pts), 0.05 m / 0.45 m submap built on the device, RT-CSM 0.15 m / 1 deg "
                        "(456 533 candidates per scan) + least-squares refine, plain solve",
            "points_per_scan": float(sizes.mean()), "correlative_points_per_scan": float(n_hi.mean()),
            "candidates_per_scan": R * L, "stages_ms_per_step": {n: round(v[0] / steps, 4) for n, v in prof.items()},
            "roofline": {"bound": "hbm", "kernel": "rtcsm_score_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": None if achieved is None else achieved / peak, "traffic": None,
                         "bytes_model": "R (12 N + 2 N L) per scan: the cloud once per rotation + one 2-byte voxel per (point, translation)",
                         "note": "voxel reads are L1/L2 hits by design (a translation window touches <= 8 bricks): the kernel is "
                                 "issue-bound, not HBM-bound; see profiles/"},
            "all_ok": bool(all(r.ok == 1 for r in res)),
            "parity_scan0": {"rtcsm_score_equal": bool(np.float32(res[0].rtcsm_score) == np.float32(want["score"])),
                             "gpu_score": float(res[0].rtcsm_score), "oracle_score": float(want["score"])}}


if __name__ == "__main__":
    main()
