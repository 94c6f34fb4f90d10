#!/usr/bin/env python
"""bench.py — events/s of the EventCalib hot path (detection: ingest -> windows -> DBSCAN -> circle fit; residual
evaluation: association -> J^T J / J^T r -> cost) on the BASELINE.json configurations.

    python bench.py [--config C2|C3|C4|C5] --gpus N --steps K --warmup W [--impl reference] [--events E] [--dump-outputs DIR]

  C2 (default; the configuration BASELINE.json's metric is quoted on): per GPU a synthetic 20 M-event DAVIS346 (346x260)
     circle-grid stream, 2 Mev/s, tiling windows of 1.5 ms (= 3 x MotionTimeStep), DBSCAN eps 4 / minPts 2, cluster filter,
     circle fit (fitCircle 1), then the residual evaluation of the same events.
  C3 640x480, 10 Mev/s, 10 ms tiling windows (~1e5 events each), 25 M events per GPU (= the 200 M-event stream of the
     configuration sharded over 8 GPUs); same stages as C2.
  C5 1280x720, 100 Mev/s, 20 % background noise + 5 % polarity flips, 1 ms tiling windows, the front end swept over
     eps in {2,3,4,6,8} x minPts in {2,3,5,8}: a 50 M-event stream x 20 sweep points = 1 G event passes per step and GPU.
  C4 the full dynamic calibration: a FIXED residual set (the C2 stream cut to --events, default 7 M), knots every 25 ms,
     exactly 50 LM iterations (normal equations + inter-GPU sum + solve + cost of the candidate), residuals sharded over
     the N GPUs (strong scaling).
One "step" = one pass of the hot path over the per-GPU stream (C4: one run of the LM loop, --lm-iters iterations).
N > 1: windows are independent, so rank r holds the r-th slice of a longer stream (weak scaling, no data-path collective);
value = all events of all ranks / max-over-ranks device time.

  value    device-resident: the packed 25-byte records are already in HBM when the timed region starts
  e2e      through the C ABI with HOST buffers: pinned-host records -> H2D -> front end -> D2H of the per-window
           summaries and candidate circles (+ the packed normal equations), every step
  parity   the same run checked against the reference's CPU path (oracle/_ref: the reference's own DBSCAN compiled in
           place + restated glue; oracle port if absent): per window the point / cluster / kept-cluster counts and the
           candidate pairs exact, circle centres and radii 1e-9 relative, residual count exact and cost 1e-9 relative.
           Any mismatch makes the run fail (exit code 1) after the line is printed.
  roofline / cpu_baseline / clocks: see DESIGN.md §Measurement.

--dump-outputs DIR writes, after the timed steps, what the last timed step computed (rank 0) as DIR/<name>.npy in float64:
per-window summaries, candidate circles, the clustered points with their labels and, with the residual evaluation, the
packed normal equations, the cost and the residual count (C4: the LM result).  A sweep leaves the outputs of its last
point.  The files stay under 64 MB: a larger array is cut to a fixed seeded sample of its rows, whose indices go to
DIR/<name>_rows.npy.  The inputs are generated from fixed seeds, so two builds run with the same arguments can be compared
file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "events/sec (detection+residual eval)"
UNIT = "events/s"
ALGO_BYTES_PER_EVENT = 29.0  # SURVEY.md §8(d): 25 B record read + 4 B label write
RTOL = 1e-9                  # north star: fitted circle centres / residuals within 1e-9 relative

CONFIGS = {
    "C2": dict(width=346, height=260, rate=2.0e6, window=1.5e-3, events=20_000_000, seed=1002, noise=0.05, flip=0.0,
               sweep=[(4.0, 2)], residual=True,
               what="synthetic %d-event DAVIS346 (346x260) circle-grid stream, %d tiling windows of 1.5 ms"),
    "C3": dict(width=640, height=480, rate=10.0e6, window=10e-3, events=25_000_000, seed=1003, noise=0.05, flip=0.0,
               sweep=[(4.0, 2)], residual=True,
               what="synthetic %d-event 640x480 circle-grid stream (1/8 of the 200 M-event configuration per GPU), %d tiling "
                    "windows of 10 ms"),
    "C5": dict(width=1280, height=720, rate=100.0e6, window=1e-3, events=50_000_000, seed=1005, noise=0.2, flip=0.05,
               sweep=[(float(e), m) for e in (2, 3, 4, 6, 8) for m in (2, 3, 5, 8)], residual=False,
               what="synthetic %d-event 1280x720 high-rate stream (100 Mev/s, 20 %% noise, 5 %% polarity flips), %d tiling "
                    "windows of 1 ms, front end swept over eps {2,3,4,6,8} x minPts {2,3,5,8} (20 passes = 1 G event passes "
                    "per step at the default size)"),
    "C4": dict(width=346, height=260, rate=2.0e6, window=1.5e-3, events=7_000_000, seed=1004, noise=0.05, flip=0.0,
               sweep=[(4.0, 2)], residual=True, what=""),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_BYTES = 60 << 20   # array bytes of --dump-outputs: under 64 MB with the .npy headers


def dump_outputs(dirname, arrays, large=()):
    """Writes every array as dirname/<name>.npy in float64.  The arrays named in `large` share what DUMP_BYTES leaves
    after the others; one that exceeds its share keeps a seeded sample of its rows (first axis), indices in <name>_rows.npy."""
    out = {k: np.asarray(v, np.float64) for k, v in arrays.items()}
    share = (DUMP_BYTES - sum(v.nbytes for k, v in out.items() if k not in large)) // max(1, len(large))
    for k in large:
        a = out[k]
        if a.nbytes > share:
            m = int(share // (a.nbytes // len(a) + 8))
            rows = np.sort(np.random.default_rng(0).choice(len(a), m, replace=False))
            out[k], out[k + "_rows"] = a[rows], rows.astype(np.float64)
    assert sum(v.nbytes for v in out.values()) <= DUMP_BYTES
    os.makedirs(dirname, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(dirname, k + ".npy"), v)


def frontend_outputs(ctx):
    """What a caller reads back after ecb_frontend_run: per-window summaries, candidate circles, points + labels."""
    s = ctx.summary()
    out = {"window_" + f: s[f] for f in s.dtype.names}
    out["candidates"] = ctx.candidates(max(1, int(s["n_candidates"].max())) if len(s) else 1)
    for pol in (0, 1):
        xy, lab = ctx.points(pol)
        out["points_xy_label_pol%d" % pol] = np.concatenate([xy, lab[:, None]], axis=1)
    return out


def make_workload(cfg, n_events, rank):
    from eventcalib_b200 import synth
    dur = n_events / cfg["rate"]
    t0 = 5.0 + rank * dur
    workers = max(1, min(16, (os.cpu_count() or 2) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))))
    ev = synth.make_stream(n_events, cfg["width"], cfg["height"], t0=t0, duration=dur, seed=cfg["seed"] + rank,
                           noise_frac=cfg["noise"], flip_frac=cfg["flip"], workers=workers)
    win = synth.tiling_windows(t0, t0 + dur, cfg["window"])
    return ev, win


def frontend_params(cfg, eps=4.0, min_pts=2, order_mode=1, median_mode=1):
    import eventcalib_b200 as ecb
    rthr = ecb.radius_threshold(cfg["width"], cfg["height"], 9, 4, True, 5.5, 1.75)
    return ecb.default_params(eps=eps, min_pts=min_pts, cluster_min=5, knn_num=3, fit_circle=1, radius_threshold=rthr,
                              rows_cols=36, order_mode=order_mode, median_mode=median_mode), rthr


def bind_to_gpu_numa_node(index):
    """Pins this process (and the pinned host buffers it allocates afterwards: first touch) to the CPUs of the NUMA node the
    GPU hangs off, so that 8 ranks x 500 MB of records per step do not all cross one node's memory controllers and the
    inter-socket link.  Returns {"node": n, "cpus": k} or None when the box exposes no NUMA topology (VMs report -1)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:      # NVML prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return {"node": node, "cpus": len(cpus)}
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        if os.environ.get("ECB_BENCH_NO_SAMPLER"):   # diagnosis only (does the sampler perturb the run?): the line then has no clocks
            return
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.p:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm)}
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


def truth_problem(cfg, ev_t0, ev_t1, traj_seed, seed=0, **kw):
    """Key frames / circles / one spline segment from the generator's ground truth (the host-side initialisation stage of the
    reference, EventCalibIni + the EventCalibSpline constructor, is outside the hot path)."""
    from eventcalib_b200 import calib_problem, synth
    cam, board = synth.Camera(cfg["width"], cfg["height"]), synth.Board()
    return calib_problem.build_from_truth(cam, synth.Trajectory(traj_seed, board, 78.0), board, ev_t0, ev_t1, seed=seed, **kw)


def cpu_reference(cfg, ev, win, budget_s=40.0, threads=None, detail=False, sweep=None):
    """The reference's CPU path on (a bounded sample of) the workload's windows, threaded like the reference
    (hardware_concurrency()-2 std::threads over windows, eventCameraCalib.cpp:172-190; Ceres num_threads = hw-2,
    EventCalibSpline.cpp:242):  detection = the reference's own DBSCAN from oracle/_ref + restated glue (oracle port if
    _ref is absent);  residual evaluation = association + one dual-number (Jet<37>) Jacobian evaluation with dense
    per-span J^T J + one cost-only evaluation (oracle/ecb_oracle_cost.cpp).
    Returns (cpu_baseline dict, per-sweep-point detail of the sample windows, residual-evaluation detail)."""
    import oracle
    oracle.build()
    kind = "reference" if oracle.have_ref() else "port"
    hw = os.cpu_count() or 4
    threads = threads or max(1, hw - 2)
    _, rthr = frontend_params(cfg)
    sweep = sweep or cfg["sweep"]
    base = dict(clusterMin=5, knn_num=3, fitCircle=1, Rthr=rthr, rows_cols=36, ref=True)
    # calibrate on a few windows, then size the sample for ~budget_s of wall time (all windows if they fit the budget)
    probe = win[: min(len(win), max(2, threads))]
    t0 = time.perf_counter()
    _, nev, _ = oracle.frontend_windows(ev["t"], ev["x"], ev["y"], ev["p"], probe, threads=threads, eps=sweep[0][0],
                                        minS=sweep[0][1], **base)
    dt = max(time.perf_counter() - t0, 1e-6)
    share = 0.55 if cfg["residual"] else 1.0  # detection's share of the CPU budget
    n_s = int(min(len(win), max(len(probe), share * budget_s / len(sweep) / (dt / len(probe)))))
    sample = win[:n_s]
    det, dt_det, nev = [], 0.0, 0
    for eps, mp in sweep:
        t0 = time.perf_counter()
        nev, counts, per, cand = oracle.frontend_windows_detail(ev["t"], ev["x"], ev["y"], ev["p"], sample, threads=threads,
                                                               eps=eps, minS=mp, cand_cap=64, **base)
        dt_det += time.perf_counter() - t0
        det.append(dict(eps=eps, min_pts=mp, counts=counts, n_cand=per, cand=cand))
    n_passes = nev * len(sweep)
    res, dt_res, n_res = None, 0.0, 0
    if cfg["residual"]:
        hi = int(np.searchsorted(ev["t"], sample[-1, 1], side="right"))
        rank_seed = int(round((ev["t"][0] - 5.0) / max(len(ev["t"]) / cfg["rate"], 1e-9)))
        pb = truth_problem(cfg, float(ev["t"][0]), float(ev["t"][hi - 1]), cfg["seed"] + rank_seed)
        P = oracle.CostProblem([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
        t0 = time.perf_counter()
        P.associate(ev["t"][:hi], ev["x"][:hi], ev["y"][:hi], pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
        c_jac, c_cost = P.eval_mt(pb["intrinsics"], pb["rot_cp"], pb["trans_cp"], threads)
        dt_res = time.perf_counter() - t0
        n_res = P.n_residuals
        res = dict(hi=hi, pb=pb, n_res=n_res, cost=c_cost, cost_jac=c_jac)
    dt = dt_det + dt_res
    cb = dict(value=n_passes / dt, unit=UNIT, cores=threads, kind=kind, seconds=dt,
              detection_events_per_s=n_passes / dt_det,
              sample="first %d of %d windows (%d events%s, %d residuals), %d std::threads of %d host cores; detection: %s%s" % (
                  n_s, len(win), nev, " x %d sweep points" % len(sweep) if len(sweep) > 1 else "", n_res, threads, hw,
                  "the reference's DBSCAN compiled in place + restated glue (oracle/_ref)" if kind == "reference" else "oracle port",
                  "; residual eval: single-thread association + Jet<37> Jacobian evaluation + cost-only evaluation (port)"
                  if cfg["residual"] else ""))
    if cfg["residual"]:
        cb["residual_eval_events_per_s"] = nev / dt_res
    return cb, (det if detail else None), res


def check_parity(ecb, cfg, ev, rec, win, det, res, local, order_mode=1, median_mode=1):
    """GPU (through the C ABI, its own context) against the CPU reference results of cpu_reference() on the same windows."""
    n_s = len(det[0]["counts"])
    sample = win[:n_s]
    hi = int(np.searchsorted(ev["t"], sample[-1, 1], side="right"))
    ctx = ecb.Context(local)
    ctx.set_sensor(cfg["width"], cfg["height"])
    ctx.load_events(rec[:hi])
    out = dict(windows=int(n_s), of_windows=int(len(win)), sweep_points=len(det), mismatches=0, status_or=0,
               max_rel_center_err=0.0, candidates=0, rtol=RTOL,
               checked="per window: points, raw clusters, kept clusters per polarity and candidate pairs exact; circle centres / "
                       "radii rtol 1e-9; vs the reference's CPU path (%s)" % ("oracle/_ref" if __import__("oracle").have_ref() else "oracle port"))
    for d in det:
        prm, _ = frontend_params(cfg, d["eps"], d["min_pts"], order_mode, median_mode)
        ctx.frontend_run(sample, prm)
        s = ctx.summary()
        k = max(64, int(s["n_candidates"].max()))
        c = ctx.candidates(k)
        out["status_or"] |= int(np.bitwise_or.reduce(s["status"])) if len(s) else 0
        bad = np.zeros(n_s, bool)
        cnt = d["counts"]
        bad |= (s["n_points"][:, 0] != cnt[:, 0]) | (s["n_points"][:, 1] != cnt[:, 1])
        bad |= (s["n_clusters"][:, 0] != cnt[:, 2]) | (s["n_clusters"][:, 1] != cnt[:, 3])
        bad |= (s["n_kept"][:, 0] != cnt[:, 4]) | (s["n_kept"][:, 1] != cnt[:, 5])
        bad |= s["n_candidates"] != d["n_cand"]
        kk = min(k, d["cand"].shape[1])
        m = np.arange(kk)[None, :] < np.minimum(d["n_cand"], kk)[:, None]
        g, r = c[:, :kk], d["cand"][:, :kk]
        bad |= ((g[..., :2] != r[..., :2]) & m[..., None]).any(axis=(1, 2))
        rel = np.abs(g[..., 2:] - r[..., 2:]) / np.maximum(np.abs(r[..., 2:]), 1e-300)
        rel = np.where(m[..., None], rel, 0.0)
        bad |= (rel > RTOL).any(axis=(1, 2))
        out["max_rel_center_err"] = max(out["max_rel_center_err"], float(rel[~bad].max()) if (~bad).any() else 0.0)
        out["mismatches"] += int(bad.sum())
        out["candidates"] += int(np.minimum(d["n_cand"], kk).sum())
        if bad.any():
            out.setdefault("first_bad", dict(eps=d["eps"], min_pts=d["min_pts"], window=int(np.nonzero(bad)[0][0])))
    if out["status_or"]:
        out["mismatches"] += 1
    if res is not None:
        pb = res["pb"]
        ctx.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
        n_res = ctx.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
        cost = ctx.cost_eval(pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])
        cj, _, _ = ctx.cost_normal_eq(pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])
        rel = max(abs(cost - res["cost"]) / abs(res["cost"]), abs(cj - res["cost_jac"]) / abs(res["cost_jac"]))
        out["residuals"] = {"gpu": int(n_res), "cpu": int(res["n_res"]), "cost_rel_err": float(rel)}
        if n_res != res["n_res"] or not rel <= RTOL:
            out["mismatches"] += 1
    ctx.close()
    return out


def run_reference(args, cfg, rank, world):
    """--impl reference: the reference's CPU implementation of the path, same config / metric, all host threads."""
    if rank != 0:
        return
    n_events = min(args.events, 4_000_000 if args.config in ("C2", "C4") else 2_000_000)
    ev, win = make_workload(cfg, n_events, 0)   # a bounded slice is enough for the CPU arm
    if args.config == "C4":
        return run_c4_reference(args, cfg, ev)
    vals = []
    for i in range(args.warmup + args.steps):
        cb, _, _ = cpu_reference(cfg, ev, win, budget_s=max(2.0, 40.0 / max(1, args.warmup + args.steps)))
        if i >= args.warmup:
            vals.append(cb)
    v = float(np.mean([c["value"] for c in vals]))
    secs = float(np.mean([c["seconds"] for c in vals]))
    cb = dict(vals[-1])
    cb["value"] = v
    cb.pop("seconds", None)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": secs * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32 pixels / f64 fit", "data": "synthetic",
            "config": {"workload": "%s per GPU: %s; CPU arm runs a bounded sample of it" % (
                args.config, cfg["what"] % (args.events, int(args.events / cfg["rate"] / cfg["window"])))},
            "cpu_baseline": cb, "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print_json(line)


# ------------------------------------------------------------------------------------------------- C4 ----
def c4_problem(cfg, ev, world):
    """The fixed calibration problem of C4: ONE spline segment over the whole stream (knots every 50 steps = 25 ms), key
    frames / circles from the ground truth, intrinsics +2 %, noisy poses."""
    return truth_problem(cfg, float(ev["t"][0]), float(ev["t"][-1]), cfg["seed"], seed=4)


def run_c4_reference(args, cfg, ev):
    import oracle
    oracle.build()
    hw = os.cpu_count() or 4
    threads = max(1, hw - 2)
    pb = c4_problem(cfg, ev, 1)
    P = oracle.CostProblem([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    P.associate(ev["t"], ev["x"], ev["y"], pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
    n_res = P.n_residuals
    ts = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        P.eval_mt(pb["intrinsics"], pb["rot_cp"], pb["trans_cp"], threads)   # one Jacobian + one cost-only evaluation
        if i >= args.warmup:
            ts.append(time.perf_counter() - t0)
    dt = float(np.mean(ts))
    v = n_res / dt
    cb = dict(value=v, unit="residuals x LM iterations / s", cores=threads, kind="port",
              sample="%d residuals of a %d-event stream; per LM iteration one Jet<37> Jacobian evaluation with dense per-span "
                     "J^T J and one cost-only evaluation on %d std::threads of %d host cores (the Ceres linear solve is not timed)" % (
                         n_res, len(ev["t"]), threads, hw))
    print_json({"impl": "reference", "metric": METRIC, "value": v, "unit": "residuals x LM iterations / s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": "C4: LM iterations of the dynamic calibration on a fixed residual set; CPU arm = residual / "
                                       "Jacobian evaluation of a bounded stream"},
                "cpu_baseline": cb, "e2e": {"value": v, "unit": "residuals x LM iterations / s", "h2d_bytes_per_step": 0,
                                            "d2h_bytes_per_step": 0}})


def run_c4(args, cfg, rank, world, local):
    """Strong scaling of the LM loop: the residuals of ONE fixed problem are split over the ranks by time; every iteration =
    solve + candidate cost (all ranks) + normal equations at the accepted point (inter-GPU sum fused into the span reduction)."""
    import torch
    import torch.distributed as dist
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ev, _ = make_workload(cfg, args.events, 0)       # every rank generates the same stream, keeps its time slice
    pb = c4_problem(cfg, ev, world)
    n = len(ev["t"])
    lo, hi = rank * n // world, (rank + 1) * n // world
    rec = synth.to_records({k: ev[k][lo:hi] for k in ("t", "x", "y", "p")})
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = ecb.Context(local, stream.cuda_stream)
    ctx.set_sensor(cfg["width"], cfg["height"])
    ctx.load_events(rec)
    ctx.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    n_res = ctx.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
    iters = args.lm_iters if args.lm_iters > 0 else 50
    solver = ecb.DeviceLm(ctx, [pb["n_cp"]], ecb.lm_options(max_iterations=iters, fixed_iterations=1))
    xch = setup_exchange(ctx, rank, world, dist, torch) if world > 1 else None
    if xch:
        solver.set_exchange(rank, xch["ptrs"])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_once():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        summ = solver.run(pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, summ

    for _ in range(max(1, min(args.warmup, 2))):
        run_once()
    sampler = ClockSampler(local) if rank == 0 else None
    l0 = ctx.launches
    runs = [run_once() for _ in range(args.steps)]
    launches = (ctx.launches - l0) // len(runs)
    clocks = sampler.stop() if sampler else None
    ms = float(np.mean([r[0] for r in runs]))
    summ = runs[-1][1]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {k: v for k, v in summ.items() if k != "reserved"})
    tot_res = n_res
    if world > 1:
        t = torch.tensor([float(n_res)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t)
        tot_res = int(t.item())
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu:
        # the device LM loop against the host state machine (ecb_lm_*) driving the same GPU evaluations, over the first 12
        # iterations (before convergence: afterwards both wander along the weakly determined k3..k5 directions at round-off
        # level, and rounding differences of the two solves are amplified by the conditioning, not by an error): same accept /
        # reject sequence, cost trajectory and intrinsics within 1e-9 (the Ceres solve itself is external: DESIGN.md §5)
        K = min(12, iters)
        i2, r2, t2, s2, tr2 = ctx.calibrate([pb["n_cp"]], pb["intrinsics"], pb["rot_cp"], pb["trans_cp"], ecb.lm_options(max_iterations=K))
        lm2 = ecb.DeviceLm(ctx, [pb["n_cp"]], ecb.lm_options(max_iterations=K))
        o2 = lm2.run(pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])
        lm2.close()
        rel = float(np.max(np.abs(o2["intrinsics"] - i2) / np.abs(i2)))
        same = len(o2["trace"]) == len(tr2) and bool(np.array_equal(o2["trace"][:, 3], tr2[:, 3]))
        relc = float(np.max(np.abs(o2["trace"][:, 0] - tr2[:, 0]) / tr2[:, 0])) if same else float("inf")
        parity = {"windows": 0, "mismatches": int(not (rel <= RTOL and relc <= RTOL and same)), "rtol": RTOL,
                  "checked": "device LM loop (state machine + band-arrow Cholesky on the GPU) vs the host LM state machine on the same GPU "
                             "evaluations, first %d iterations: accept / reject sequence %s, cost trajectory max rel. diff %.1e, "
                             "intrinsics max rel. diff %.1e" % (K, "equal" if same else "DIFFERS", relc, rel)}
    if rank == 0:
        it = summ["iterations"]
        unit = "residuals x LM iterations / s"
        value = tot_res * it / (ms * 1e-3)
        line = {"metric": METRIC, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic",
                "config": {"workload": "C4: full dynamic calibration on a fixed problem — %d residual blocks from a %d-event DAVIS346 "
                                       "stream, %d control points (knots every 25 ms, D = %d), intrinsics +2 %%, exactly %d LM iterations "
                                       "(tolerances off): per iteration band-arrow Cholesky solve on the device, candidate cost, normal "
                                       "equations of the accepted point with the inter-GPU sum fused into the span reduction" % (
                                           tot_res, n, pb["n_cp"], 9 + 6 * pb["n_cp"], it),
                           "residuals_all_gpus": int(tot_res), "control_points": int(pb["n_cp"]),
                           "parallelism": "residuals sharded by time x%d (strong scaling)" % world,
                           "l2": "residual records %.0f MB per GPU per evaluation" % (n_res * 56 / 1e6)},
                "gpu_launches": int(launches), "clocks": clocks,
                "lm": {k: (float(v) if isinstance(v, float) else int(v)) for k, v in summ.items()
                       if k in ("iterations", "successful_steps", "termination", "initial_cost", "final_cost", "gradient_max_norm", "radius")},
                "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 64,
                        "note": "the LM loop runs from device-resident residuals; per iteration only the accept / reject scalars "
                                "cross PCIe"}}
        line["lm"]["s_per_iteration"] = ms * 1e-3 / max(it, 1)
        line["lm"]["final_intrinsics"] = [float(v) for v in summ["intrinsics"]]
        line["lm"]["truth_intrinsics"] = [float(v) for v in pb["truth_intrinsics"]]
        if parity:
            line["parity"] = parity
        print_json(line)
    solver.close()
    if world > 1:
        teardown_exchange(ctx, xch, rank, dist, torch)
        dist.destroy_process_group()
    ctx.close()
    if parity and parity["mismatches"]:
        sys.exit(1)


def setup_exchange(ctx, rank, world, dist, torch):
    """Peer-mapped receive buffers of the fused normal-equation exchange (CUDA IPC handles gathered once through NCCL)."""
    if os.environ.get("ECB_NO_P2P"):
        return None
    ok, xch = 1, None
    try:
        my_buf = ctx.device_alloc(ctx.exchange_buffer_bytes(world))
        h = torch.from_numpy(ctx.ipc_export(my_buf)).cuda()
        hs = [torch.empty_like(h) for _ in range(world)]
        dist.all_gather(hs, h)
        ptrs = [my_buf if r == rank else ctx.ipc_open(hs[r].cpu().numpy()) for r in range(world)]
        xch = {"ptrs": ptrs, "epoch": 0, "buf": my_buf}
    except Exception as e:  # noqa: BLE001
        sys.stderr.write("rank %d: peer mapping unavailable (%s), using NCCL\n" % (rank, e))
        ok = 0
    t_ok = torch.tensor([ok], device="cuda")
    dist.all_reduce(t_ok, op=dist.ReduceOp.MIN)
    return xch if int(t_ok.item()) else None


def teardown_exchange(ctx, xch, rank, dist, torch):
    dist.barrier()
    torch.cuda.synchronize()
    if xch:
        for r_, p_ in enumerate(xch["ptrs"]):
            if r_ != rank:
                ctx.ipc_close(p_)
        dist.barrier()
        ctx.device_free(xch["buf"])


# ----------------------------------------------------------------------------------------------- main ----
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--events", type=int, default=0, help="events per GPU (default: the configuration's)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / parity leg")
    ap.add_argument("--cpu-budget", type=float, default=40.0, help="seconds of CPU work for the cpu_baseline / parity leg")
    ap.add_argument("--slices", type=int, default=0, help="time slices (contexts/streams/host threads) of the e2e pipeline")
    ap.add_argument("--order-mode", type=int, default=1, help="pid order: 0 first arrival, 1 libstdc++ unordered_set order (the reference's)")
    ap.add_argument("--median-mode", type=int, default=1, help="cluster centre: 0 canonical, 1 std::nth_element over BFS order (the reference's)")
    ap.add_argument("--slice-plan", default="", help="relative sizes of the e2e time slices, e.g. 1,2,3,3,2,1 (overrides --slices)")
    ap.add_argument("--lm-iters", type=int, default=0, help="LM iterations of C4 (default 50)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    cfg = CONFIGS[args.config]
    if args.events <= 0:
        args.events = cfg["events"]

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE line, the result JSON: everything else that writes to file descriptor 1 (NCCL prints its
    # version banner there) is sent to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    json_out = os.fdopen(json_fd, "w")
    global print_json

    def print_json(line):
        json_out.write(json.dumps(line) + "\n")
        json_out.flush()
    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
        return

    import torch
    import torch.distributed as dist
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    if args.config == "C4":
        return run_c4(args, cfg, rank, world, local)
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    WIDTH, HEIGHT = cfg["width"], cfg["height"]
    sweep = cfg["sweep"]
    ev, win = make_workload(cfg, args.events, rank)
    n = len(ev["t"])
    rec = synth.to_records(ev)
    # N > 1: host threads and the pinned record buffers of this rank on the GPU's own NUMA node (ECB_BENCH_NO_NUMA=1: off)
    numa = bind_to_gpu_numa_node(local) if world > 1 and not os.environ.get("ECB_BENCH_NO_NUMA") else None
    pinned = torch.empty(n * 25, dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[:] = rec.view(np.uint8).reshape(-1)
    d_raw = torch.empty(n * 25 + 16, dtype=torch.uint8, device="cuda")
    d_raw[: n * 25].copy_(pinned, non_blocking=False)
    # the PCIe ceiling of the end-to-end number: plain pinned -> device copy of the same records (outside every timed region)
    h2d_gbs = 0.0
    for _ in range(3):
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        c0.record()
        d_raw[: n * 25].copy_(pinned, non_blocking=True)
        c1.record()
        torch.cuda.synchronize()
        h2d_gbs = max(h2d_gbs, n * 25 / (c0.elapsed_time(c1) * 1e-3) / 1e9)
    h2d_all_gbs = h2d_gbs
    if world > 1:  # the host-side ceiling of the N-GPU end-to-end number: all ranks copying at once
        dist.barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        c0.record()
        for _ in range(2):
            d_raw[: n * 25].copy_(pinned, non_blocking=True)
        c1.record()
        torch.cuda.synchronize()
        t = torch.tensor([2 * n * 25 / (c0.elapsed_time(c1) * 1e-3) / 1e9], device="cuda", dtype=torch.float64)
        tmin = t.clone()
        dist.all_reduce(t)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        h2d_all_gbs = float(t.item())

    # one explicit (non-default) stream shared by torch (copies, NCCL, timing events) and the library's kernels
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = ecb.Context(local, stream.cuda_stream)
    ctx.set_sensor(WIDTH, HEIGHT)
    prms = [frontend_params(cfg, e_, m_, args.order_mode, args.median_mode)[0] for e_, m_ in sweep]
    ctx.load_events_device(d_raw.data_ptr(), n)

    # residual evaluation: key frames / circles / spline segments from the ground truth (host-side initialisation is
    # outside the hot path); rank r owns segment r (EventCalibSpline splits the map into segments at gaps,
    # EventCalibSpline.cpp:319-348); every rank knows all segments, holds only its own residuals
    do_res = cfg["residual"]
    last = {}   # scalars the last device-resident step returned (--dump-outputs)
    n_res, segs, mine, xch, xch_check = 0, None, None, None, None
    rot = np.zeros((0, 4))
    if do_res:
        dur = n / cfg["rate"]
        segs = [truth_problem(cfg, 5.0 + r * dur + 0.5 / cfg["rate"], 5.0 + (r + 1) * dur - 0.5 / cfg["rate"], cfg["seed"] + r, seed=r)
                for r in range(world)]
        mine = segs[rank]
        n_cp = [sg["n_cp"] for sg in segs]
        knots = [sg["knots"] for sg in segs]
        ctx.cost_setup(n_cp, knots, mine["radius"], mine["huber"])
        intr = mine["intrinsics"]
        rot = np.concatenate([sg["rot_cp"] for sg in segs])
        trans = np.concatenate([sg["trans_cp"] for sg in segs])
        n_res = ctx.cost_associate(mine["kf_t"], mine["circles"], mine["landmarks"], mine["step"])
        lay = ctx.cost_layout()
        d_ne = torch.zeros(lay["out_doubles"], dtype=torch.float64, device="cuda")
        h_ne = torch.empty(lay["out_doubles"], dtype=torch.float64, pin_memory=True)
        # N > 1: the inter-GPU sum of the normal equations AND of the scalar cost is fused into the span reduction
        # (peer-mapped receive buffers over NVLink); NCCL all-reduce is the fallback when peer mapping is unavailable
        if world > 1:
            xch = setup_exchange(ctx, rank, world, dist, torch)

        def normal_eq_all_ranks(i_, r_, t_):
            """packed J^T J / J^T r / cost of ALL ranks' residuals in d_ne (device)"""
            if xch:
                xch["epoch"] += 1
                ctx.cost_normal_eq_exchange(i_, r_, t_, rank, xch["ptrs"], xch["epoch"], d_ne.data_ptr(), want_cost=False)
            else:
                ctx.cost_normal_eq(i_, r_, t_, d_out=d_ne.data_ptr(), host=False)
                if world > 1:
                    dist.all_reduce(d_ne)

        if xch:  # once: the fused exchange against NCCL's all-reduce of the same evaluation
            normal_eq_all_ranks(intr, rot, trans)
            a_x = d_ne.clone()
            ctx.cost_normal_eq(intr, rot, trans, d_out=d_ne.data_ptr(), host=False)
            dist.all_reduce(d_ne)
            xch_check = float((a_x - d_ne).abs().max().item() / max(float(d_ne.abs().max().item()), 1e-300))

        d_kf_t = torch.from_numpy(np.ascontiguousarray(mine["kf_t"], np.float64)).cuda()
        d_kf_c = torch.from_numpy(np.ascontiguousarray(mine["circles"], np.float64)).cuda()
        d_lm = torch.from_numpy(np.ascontiguousarray(mine["landmarks"], np.float64)).cuda()

        def residual_eval():
            """one LM iteration's worth of evaluation: association + J^T J / J^T r + cost (both summed over the GPUs inside
            the fused exchange) + the cost-only evaluation of this rank's residuals"""
            # device-resident step: the key-frame tables are inputs like the records and lie in HBM (ecb_cost_associate_device);
            # the end-to-end step below uploads them from host arrays inside the timed region
            last["n_residuals"] = ctx.cost_associate_device(d_kf_t.data_ptr(), d_kf_c.data_ptr(), len(mine["kf_t"]),
                                                            mine["circles"].shape[1], d_lm.data_ptr(), mine["step"])
            normal_eq_all_ranks(intr, rot, trans)
            last["cost"] = ctx.cost_eval(intr, rot, trans)

    def step_device():
        ctx.load_events_device(d_raw.data_ptr(), n)
        for p_ in prms:
            ctx.frontend_run(win, p_)
        if do_res:
            residual_eval()

    # ---- end to end from host buffers: S time slices, each with its own context / stream / host thread, so the H2D copy
    # of slice k+1 overlaps the kernels of slice k (the C ABI is re-entrant per context; ctypes releases the GIL).
    from concurrent.futures import ThreadPoolExecutor
    if args.slices <= 0:  # 8 slices on one GPU; with N ranks on one host keep about one host thread per core
        args.slices = 8 if world == 1 else max(2, min(8, (os.cpu_count() or 16) // world))
    plan = [float(v) for v in args.slice_plan.split(",")] if args.slice_plan else [1.0] * max(1, min(args.slices, len(win)))
    S = len(plan)
    # Host waits: a slice thread spins in cudaStreamSynchronize by default.  When the ranks' slice threads outnumber the host
    # cores (8 ranks x 4 slices on the 32-core 8-GPU box) the spinning threads starve each other, so the slice contexts then
    # sleep on an event instead (ECB_BLOCKING_SYNC, read by ecb_ctx_create).  ECB_BENCH_SYNC=spin|block|yield overrides (yield: poll + sched_yield).
    sync_mode = os.environ.get("ECB_BENCH_SYNC", "auto")
    if sync_mode == "auto":
        # (8 ranks x 4 slices on 32 cores, e2e ms per step: yield 29.8, spin 30.4, block 31.9; 1 rank on 16 cores: spin 12.3,
        #  block 14.4 — profiles/r2t_n8_e2e_trace.md)
        sync_mode = "yield" if world * (S + 1) > (os.cpu_count() or 16) else "spin"
    if sync_mode in ("block", "yield"):
        os.environ["ECB_BLOCKING_SYNC"] = "1" if sync_mode == "block" else "2"
    cuts = np.round(np.cumsum([0.0] + plan) / sum(plan) * len(win)).astype(int)
    slices = []
    for j in range(S):
        w0, w1 = int(cuts[j]), int(cuts[j + 1])
        lo = int(np.searchsorted(ev["t"], win[w0, 0], side="left")) if j > 0 else 0
        slices.append(dict(w0=w0, w1=w1, lo=lo))
    for j in range(S):
        sl = slices[j]
        sl["hi"] = slices[j + 1]["lo"] if j + 1 < S else n
        sl["ctx"] = ecb.Context(local)          # own non-blocking stream
        sl["ctx"].set_sensor(WIDTH, HEIGHT)
        if do_res:
            sl["ctx"].cost_setup(n_cp, knots, mine["radius"], mine["huber"])
            ta, tb = ev["t"][sl["lo"]], ev["t"][sl["hi"] - 1]
            m = (mine["kf_t"] > ta - 6 * mine["step"]) & (mine["kf_t"] < tb + 6 * mine["step"])
            sl["kf_t"], sl["circles"] = mine["kf_t"][m].copy(), mine["circles"][m].copy()
    if do_res:
        d_parts = torch.zeros(S, lay["out_doubles"], dtype=torch.float64, device="cuda")
    # caller-owned host result buffers: every slice writes its windows' summaries / candidate circles in place
    h_summ = np.zeros(len(win), ecb.SUMMARY_DTYPE)
    h_cand = np.zeros((len(win), 48, 5))
    pool = ThreadPoolExecutor(S)

    trace = os.environ.get("ECB_BENCH_TRACE")
    stagger = float(os.environ.get("ECB_BENCH_STAGGER_US", "0")) * 1e-6
    t_origin = [0.0]
    load_done = [0.0] * S
    h2d_done = []   # per step: host time at which the LAST slice's records had arrived, relative to the step start

    def slice_work(j):
        sl = slices[j]
        c = sl["ctx"]
        if stagger:  # uploads enter the copy queue in slice order (the threads race otherwise): slice plans can then shape the ramp
            time.sleep(j * stagger)
        tm = [time.perf_counter()]
        c.load_events_ptr(pinned.data_ptr() + sl["lo"] * 25, sl["hi"] - sl["lo"])
        tm.append(time.perf_counter())
        cost = 0.0
        for p_ in prms:
            c.frontend_run(win[sl["w0"]:sl["w1"]], p_)
            out = c.summary(out=h_summ[sl["w0"]:sl["w1"]]), c.candidates(48, out=h_cand[sl["w0"]:sl["w1"]])
        tm.append(time.perf_counter())
        if do_res:
            c.cost_associate(sl["kf_t"], sl["circles"], mine["landmarks"], mine["step"])
            c.cost_normal_eq(intr, rot, trans, d_out=d_parts[j].data_ptr(), host=False)
            cost = c.cost_eval(intr, rot, trans)       # synchronises the slice's stream
        tm.append(time.perf_counter())
        if trace:
            sys.stderr.write("rank %d slice %d: start %.2f load_end %.2f frontend_end %.2f cost_end %.2f ms\n" % (
                (rank, j) + tuple((x - t_origin[0]) * 1e3 for x in tm)))
        load_done[j] = tm[1] - t_origin[0]   # when this slice's records (H2D + unpack) were on the device
        return out + (cost,)

    def step_e2e():
        t_origin[0] = time.perf_counter()
        res = list(pool.map(slice_work, range(S)))
        h2d_done.append(max(load_done))
        if do_res:
            torch.sum(d_parts, dim=0, out=d_ne)   # the packed buffer ends with the cost: summed with the rest
            if world > 1:
                dist.all_reduce(d_ne)
            h_ne.copy_(d_ne, non_blocking=False)
        return h_summ, h_cand

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    n_pass = n * len(sweep)   # events processed by one step on this GPU
    for _ in range(args.warmup):
        step_device()
    l0 = ctx.launches
    sampler = ClockSampler(local) if rank == 0 else None
    ms = timed(step_device, args.steps)
    launches = ctx.launches - l0
    value = world * n_pass * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        outs = frontend_outputs(ctx)
        if do_res:
            outs.update(last, normal_eq=d_ne.cpu().numpy())
        dump_outputs(args.dump_outputs, outs, large=("candidates", "points_xy_label_pol0", "points_xy_label_pol1"))

    # per-kernel durations, measured live with CUDA events on the launching stream (separate pass; the front-end stages
    # of a sweep are those of its last point)
    ctx.set_profiling(True)
    stage = {}
    for _ in range(args.steps):
        step_device()
        for k, v in ctx.stage_ms().items():
            stage.setdefault(k, []).append(v)
    ctx.set_profiling(False)
    stage = {k: float(np.mean(v)) for k, v in stage.items() if np.mean(v) > 0}

    if os.environ.get("ECB_BENCH_GAPS"):   # wall clock of every API call of the device-resident step against its kernels
        calls = [("load_events_device", lambda: ctx.load_events_device(d_raw.data_ptr(), n)),
                 ("frontend_run", lambda: ctx.frontend_run(win, prms[-1]))]
        if do_res:
            calls += [("cost_associate_device", lambda: ctx.cost_associate_device(d_kf_t.data_ptr(), d_kf_c.data_ptr(), len(mine["kf_t"]),
                                                                                  mine["circles"].shape[1], d_lm.data_ptr(), mine["step"])),
                      ("normal_eq", lambda: normal_eq_all_ranks(intr, rot, trans)),
                      ("cost_eval", lambda: ctx.cost_eval(intr, rot, trans))]
        acc = {k: [] for k, _ in calls}
        for _ in range(5):
            for k, f in calls:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                f()
                torch.cuda.synchronize()
                acc[k].append((time.perf_counter() - t0) * 1e3)
        sys.stderr.write("GAPS " + " ".join("%s %.3f" % (k, float(np.median(v))) for k, v in acc.items()) + "\n")

    # end to end through the C ABI with host buffers
    s, c = step_e2e()
    step_e2e()
    del h2d_done[:]
    ms_e2e = timed(step_e2e, args.steps)
    h2d_done_ms = float(np.mean(h2d_done)) * 1e3 if h2d_done else 0.0
    if world > 1:   # the step lasts as long as its slowest rank: report that rank's arrival time
        t_ = torch.tensor([h2d_done_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t_, op=dist.ReduceOp.MAX)
        h2d_done_ms = float(t_.item())
    clocks = sampler.stop() if sampler else None
    e2e_value = world * n_pass * args.steps / (ms_e2e * 1e-3)
    h2d = n * 25 + win.nbytes * len(sweep) + ((9 + 7 * len(rot)) * 8 * 2 if do_res else 0)
    d2h = (s.nbytes + c.nbytes) * len(sweep) + (h_ne.numel() * 8 if do_res else 0)

    if rank == 0:
        hbm, which = peaks()
        npts = int(s["n_points"].sum())
        # algorithmic bytes / flops per launch of each kernel (DESIGN.md §4): residual records are 56 B (obs 16, basis 32,
        # first control point 4, circle id 4)
        algo = {"ingest": n * 37.0, "window": n * 4.0 + npts * 8.0, "cluster": npts * 12.0, "pair": npts * 8.0,
                "order": npts * 8.0,
                "assoc": n * 12.0 * 2 + n_res * 68.0, "normal_eq": n_res * 56.0, "cost": n_res * 56.0}
        flops = {"normal_eq": n_res * NE_FLOP_PER_RESIDUAL, "cost": n_res * 150.0}
        tot = sum(stage.values())
        kernels = {}
        for k in stage:
            kernels[k] = {"ms": stage[k], "share": stage[k] / tot, "algo_gbs": algo[k] / (stage[k] * 1e-3) / 1e9 if k in algo else None}
            if k in flops:
                kernels[k]["algo_tflops"] = flops[k] / (stage[k] * 1e-3) / 1e12
        dom = max((k for k in stage if k in algo), key=lambda k: stage[k])
        # tier formula: SURVEY §8(d)'s per-unit figure (29 B / event) x the events one launch processes / the dominant
        # kernel's average launch duration
        achieved = n * ALGO_BYTES_PER_EVENT / (stage[dom] * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": "k_" + dom, "achieved": achieved, "peak": hbm, "unit": "GB/s",
                    "frac": achieved / hbm, "traffic": None, "peak_source": which,
                    "algorithmic_bytes_per_launch": n * ALGO_BYTES_PER_EVENT,
                    "kernel_own_bytes_per_launch": algo[dom],
                    "path_frac": (value / world) * ALGO_BYTES_PER_EVENT / 1e9 / hbm,
                    "limiter": LIMITERS.get(dom, "hbm"),
                    "note": "achieved = 29 B/event (SURVEY §8(d)) x events per launch / the dominant kernel's CUDA-event duration; "
                            "path_frac = the same bytes over the whole step.  HBM is the formal bound of the path, not the limiter "
                            "of this kernel (see `limiter`, `per_point` and profiles/): the sensor plane as a shared-memory bitmap "
                            "removed the sort traffic, what is left is instruction issue and shared-memory work per point",
                    "kernels": kernels}
        # DRAM bytes per launch and instruction counts of the dominant kernel from the committed `ncu --set full` capture
        # (profiles/), scaled to this run's event count when it differs
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            k = tr["kernels"].get("k_" + dom)
            if k and tr.get("config", "C2") == args.config:
                roofline["ncu"] = {m: k[m] for m in ("issue_active_pct", "warps_active_pct", "dram_throughput_pct", "fp64_pipe_active_pct",
                                                      "smem_bank_conflict_pct") if m in k}
                roofline["traffic"] = (k["dram_bytes_read"] + k["dram_bytes_write"]) * (n / float(tr["events"]))
                roofline["traffic_source"] = tr["source"] + ("" if n == tr["events"] else " (scaled from %d events)" % tr["events"])
                if "inst_executed" in k and npts:
                    roofline["per_point"] = {"warp_instructions": k["inst_executed"] * (n / float(tr["events"])) / npts,
                                             "smem_wavefronts": k.get("smem_wavefronts", 0) * (n / float(tr["events"])) / npts,
                                             "points": npts}
        except Exception:
            pass
        if "normal_eq" in stage:
            tf = flops["normal_eq"] / (stage["normal_eq"] * 1e-3) / 1e12
            roofline["cost_kernel"] = {"bound": "tensor", "kernel": "k_normal_eq (FP64 DMMA)", "unit": "TFLOP/s",
                                       "achieved": tf, "peak": 37.0, "frac": tf / 37.0,
                                       "flop_per_residual": NE_FLOP_PER_RESIDUAL,
                                       "flop_source": "executed FP64 flop per residual counted from SASS / ncu "
                                                      "(profiles/r2_normal_eq_flops.md), not SURVEY's 2.0 k estimate",
                                       "peak_source": "builder-measured FP64 DMMA m8n8k4 on this pool's B200 (profiles/r1_fp64_peak.txt); "
                                                      "MEASURED_PEAKS.json has no FP64 figure"}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "int32 pixels / f64 fit + f64 residuals", "data": "synthetic",
                "config": {"workload": "%s per GPU: %s, DBSCAN %s + cluster filter + circle fit (fitCircle 1; pid order %s, "
                                       "cluster centres %s)%s" % (
                                           args.config, cfg["what"] % (n, len(win)),
                                           "eps 4 minPts 2" if len(sweep) == 1 else "sweep",
                                           "= libstdc++ unordered_set order like the reference" if args.order_mode == 1 else "= first arrival",
                                           "= std::nth_element over BFS-ordered members like the reference" if args.median_mode == 1 else "canonical",
                                           ", then residual evaluation of the same events (association + J^T J/J^T r + cost, summed "
                                           "over the GPUs when N>1)" if do_res else ""),
                           "events_per_gpu": n, "event_passes_per_step_per_gpu": int(n_pass), "windows_per_gpu": int(len(win)),
                           "residuals_per_gpu": int(n_res),
                           "control_points": int(len(rot)), "parallelism": "windows / spline segments sharded x%d" % world,
                           "normal_eq_exchange": (("fused into the span reduction: P2P stores into peer-mapped receive buffers "
                                                   "over NVLink, one-shot sum in rank order, cost in the header (max rel. diff vs NCCL "
                                                   "all-reduce %.1e)" % xch_check)
                                                  if xch else ("NCCL all-reduce" if world > 1 and do_res else "single GPU")),
                           "l2": "inputs larger than L2 (%.0f MB of records per step)" % (n * 25 / 1e6),
                           "found_circles_per_window": float(s["n_candidates"].mean())},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
                "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / args.steps, "h2d_bytes_per_step": int(h2d),
                        "d2h_bytes_per_step": int(d2h), "pipeline": "%d time slices (relative sizes %s), one context/stream/host thread each "
                        "(H2D of slice k+1 overlaps the kernels of slice k); host waits: %s" % (S, ":".join("%g" % v for v in plan), sync_mode),
                        "h2d_copy_gbs": h2d_gbs, "pcie_floor_ms": h2d / (h2d_gbs * 1e9) * 1e3 if h2d_gbs > 0 else None,
                        # measured inside the timed steps: when the last record of the step had reached the (slowest) GPU; the
                        # rest of the step is the last slice's kernels + result copies
                        "h2d_done_ms": h2d_done_ms, "frac_h2d_done": h2d_done_ms / (ms_e2e / args.steps)}}
        if world > 1:
            floor = n * 25 * world / (h2d_all_gbs * 1e9) * 1e3
            line["e2e"]["numa"] = numa if numa else "not bound (single NUMA node or topology not exposed)"
            line["e2e"].update({"h2d_copy_gbs_all_ranks_concurrent": h2d_all_gbs, "host_floor_ms": floor,
                                "frac_of_host_ceiling": floor / (ms_e2e / args.steps)})
        rc = 0
        if not args.no_cpu and world == 1:
            cb, det, res = cpu_reference(cfg, ev, win, budget_s=args.cpu_budget, detail=True)
            cb.pop("seconds", None)
            line["cpu_baseline"] = cb
            line["parity"] = check_parity(ecb, cfg, ev, rec, win, det, res, local, args.order_mode, args.median_mode)
            rc = 1 if line["parity"]["mismatches"] else 0
        print_json(line)
    else:
        rc = 0
    if world > 1:
        teardown_exchange(ctx, xch, rank, dist, torch)
        dist.destroy_process_group()
    pool.shutdown()
    for sl in slices:
        sl["ctx"].close()
    ctx.close()
    if rc:
        sys.exit(rc)


# executed FP64 flop per residual of k_normal_eq (SASS count x ncu instruction counters, profiles/r2_normal_eq_flops.md):
# 80 DMMA m8n8k4 (512 flop) per 32 residuals = 1280; DFMA 258 x 2 + DMUL 175 + DADD 46 = 737 (rows 32 / 33 of the Gram matrix, closed-form residual + Jacobian)
NE_FLOP_PER_RESIDUAL = 2017.0
# what actually limits each kernel (ncu, profiles/): the `bound` key of the contract stays "hbm" (the formal bound of
# streaming integer work), this names the limiter
LIMITERS = {"cluster": "instruction issue + shared-memory wavefronts (bitmap stencil, union-find, kd-order emulation)",
            "pair": "instruction fetch + FP64 sqrt/div latency", "order": "shared-memory atomics + 64-bit integer hashing",
            "normal_eq": "FP64 pipe (DMMA + DFMA)", "assoc": "instruction issue", "ingest": "hbm", "cost": "hbm / FP64 latency",
            "window": "shared-memory atomics + barriers", "bfs": "L2 latency"}


if __name__ == "__main__":
    main()
