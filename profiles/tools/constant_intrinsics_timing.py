"""Cost of constant intrinsics at the C4 size (bench.py --config C4: one spline segment over a 7 M-event stream, D = 843).

    python profiles/tools/constant_intrinsics_timing.py [--events 7000000] [--reps 20] [--iters 50] [--out FILE]

For the masks none / k3 k4 k5 / all nine, alternated inside every repetition (so that the masks see the same machine state),
after 2 warm-up rounds:
  lm   the device LM (ecb_lm_device_*) with fixed_iterations and --iters iterations: host clock around begin + iterations +
       result (the read-back synchronises), per iteration.  A rejected iteration skips the normal equations at a new point,
       so the accepted-step count of each mask is reported with it.
  cov  ecb_covariance with the packed normal equations given (evaluated once at the starting point): host clock around the call
       (it ends in the read-back of Z).
Median / min / max over --reps repetitions.  Prints one JSON line (also to --out) with the card's name and power limit.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

MASKS = {"none": [], "k3 k4 k5": ["k3", "k4", "k5"], "all nine": ["fx", "fy", "cx", "cy", "k1", "k2", "k3", "k4", "k5"]}


def stats(v):
    return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--events", type=int, default=7_000_000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import bench
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth
    from covariance_timing import gpu_info
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
    d_packed = ctx.device_alloc(8 * ctx.cost_layout()["out_doubles"])
    ctx.cost_normal_eq(*x, d_out=d_packed, host=False)
    ctx.synchronize()
    opt = ecb.lm_options(max_iterations=a.iters, fixed_iterations=1)
    solvers = {}
    for name, names in MASKS.items():   # the device LM captures the context's mask when it is created
        ctx.set_constant_intrinsics(names)
        solvers[name] = ecb.DeviceLm(ctx, n_cp, opt)
    t_lm = {k: [] for k in MASKS}
    t_cov = {k: [] for k in MASKS}
    last = {}
    for rep in range(2 + a.reps):
        for name, names in MASKS.items():
            ctx.synchronize()
            t0 = time.perf_counter()
            out = solvers[name].run(*x)
            dt = time.perf_counter() - t0
            ctx.set_constant_intrinsics(names)
            ctx.synchronize()
            t1 = time.perf_counter()
            cov = ctx.covariance(n_cp, *x, d_packed=d_packed)
            dc = time.perf_counter() - t1
            if rep >= 2:
                t_lm[name].append(dt * 1e3 / out["iterations"])
                t_cov[name].append(dc * 1e3)
            last[name] = (out, cov)
    ctx.device_free(d_packed)
    per_mask = {}
    for name, names in MASKS.items():
        out, cov = last[name]
        const = [ecb.INTRINSIC_NAMES.index(nm) for nm in names]
        assert cov["ok"] and np.array_equal(out["intrinsics"][const], x[0][const])
        per_mask[name] = {"lm_ms_per_iteration": stats(t_lm[name]), "covariance_ms": stats(t_cov[name]),
                          "iterations": out["iterations"], "accepted_steps": out["successful_steps"],
                          "final_cost": out["final_cost"], "dimension": cov["dimension"],
                          "min_relative_pivot": cov["min_relative_pivot"], "std_intrinsics": cov["std_intrinsics"].tolist()}
    for s in solvers.values():
        s.close()
    res = {"tool": "constant_intrinsics_timing", "gpu": gpu_info(), "events": a.events, "residuals": n_res,
           "control_points": int(pb["n_cp"]), "reps": a.reps, "lm_iterations": a.iters, "masks": per_mask,
           "note": "host clock; masks alternated inside every repetition; device LM with fixed_iterations from the C4 starting "
                   "point; ecb_covariance at the starting point with the packed normal equations given"}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
