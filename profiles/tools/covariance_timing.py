"""Device time of ecb_covariance at the C4 size (bench.py --config C4: one spline segment over a 7 M-event stream, D = 843).

    python profiles/tools/covariance_timing.py [--events 7000000] [--reps 20] [--out FILE]

Two figures, each the median over --reps calls after 3 warm-up calls, host clock around a call that ends in a device
synchronise (ecb_covariance reads its result back):
  packed   d_packed given (the normal equations already on the device): assemble, equilibration, band-arrow factorisation,
           corner inverse, selected inversion, read-back of Z (band + cross + corner)
  full     d_packed = NULL: the normal-equation evaluation at x included
The normal equations are evaluated once into a device buffer for the first figure.  Prints one JSON line (also to --out).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception:  # noqa: BLE001
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--events", type=int, default=7_000_000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import bench
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth
    cfg = bench.CONFIGS["C4"]
    ev, _ = bench.make_workload(cfg, a.events, 0)
    pb = bench.c4_problem(cfg, ev, 1)
    ctx = ecb.Context(0)
    ctx.set_sensor(cfg["width"], cfg["height"])
    ctx.load_events(synth.to_records(ev))
    ctx.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    n_res = ctx.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
    n_cp = [pb["n_cp"]]
    x = (pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])
    lay = ctx.cost_layout()
    d_packed = ctx.device_alloc(8 * lay["out_doubles"])
    ctx.cost_normal_eq(*x, d_out=d_packed, host=False)
    ctx.synchronize()

    def timed(**kw):
        ts, out = [], None
        for k in range(3 + a.reps):
            ctx.synchronize()
            t0 = time.perf_counter()
            out = ctx.covariance(n_cp, *x, **kw)
            dt = time.perf_counter() - t0
            if k >= 3:
                ts.append(dt * 1e3)
        return float(np.median(ts)), float(np.min(ts)), float(np.max(ts)), out

    p_med, p_min, p_max, cp = timed(d_packed=d_packed)
    f_med, f_min, f_max, cf = timed()
    ctx.device_free(d_packed)
    assert cp["ok"] and cf["ok"]
    assert np.array_equal(cp["cov_band"], cf["cov_band"]), "packed and evaluated paths differ"
    res = {"tool": "covariance_timing", "gpu": gpu_info(), "events": a.events, "residuals": n_res, "control_points": int(pb["n_cp"]),
           "dimension": cp["dimension"], "reps": a.reps,
           "packed_ms": {"median": p_med, "min": p_min, "max": p_max},
           "full_ms": {"median": f_med, "min": f_min, "max": f_max},
           "min_relative_pivot": cp["min_relative_pivot"], "sigma2": cp["sigma2"],
           "std_intrinsics": cp["std_intrinsics"].tolist(),
           "note": "host clock around ecb_covariance (ends in a device synchronise and the read-back of "
                   "%d doubles of Z)" % (cp["cov_band"].size + cp["cov_cross"].size + 81)}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
