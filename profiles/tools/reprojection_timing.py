"""Cost of the reprojection report at the C4 size (bench.py --config C4: one spline segment over a 7 M-event stream, 6.7 M
residuals).

    python profiles/tools/reprojection_timing.py [--events 7000000] [--reps 20] [--out FILE]

For both rotation models, after 2 warm-up rounds, CUDA events on the context's stream around
  errors          ecb_cost_reprojection_errors into a device buffer (asynchronous; the events bracket the kernel)
  keyframe / circle / sensor_cell
                  ecb_cost_reprojection_groups (it ends in the read-back of the groups)
Median / min / max over --reps repetitions.  Bytes are derived from the shapes (see traffic()) and compared with the 7.7 TB/s of
HBM3e of one B200 (data sheet).  Prints one JSON line (also to --out) with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

HBM_BPS = 7.7e12


def stats(v):
    return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}


def traffic(n, n_groups, what):
    """DRAM bytes the algorithm needs for n records.  Reprojection pass: obs 16 + basis 32 + first control point 4 + circle 4
    read, e 8 written.  Grouping: the reprojection pass, key 8 + index 4 written (plus the event index 8 and its stamp 8 for key frames,
    the circle 4, or the observation 16), per 8-bit radix pass key + index read twice (histogram, scatter) and written once,
    then index 4 + e 8 read by the reduction."""
    res = 64 * n
    if what == "errors":
        return res
    key_in = {"keyframe": 16, "circle": 4, "sensor_cell": 16}[what]
    passes = (max(int(n_groups).bit_length(), 1) + 7) // 8
    return res + n * (key_in + 12) + passes * n * (8 + 12 + 12) + n * 12


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--events", type=int, default=7_000_000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    import bench
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth
    from covariance_timing import gpu_info
    cfg = bench.CONFIGS["C4"]
    ev, _ = bench.make_workload(cfg, a.events, 0)
    pb = bench.c4_problem(cfg, ev, 1)
    stream = torch.cuda.Stream(device=0)
    ctx = ecb.Context(0, stream=stream.cuda_stream)
    ctx.set_sensor(cfg["width"], cfg["height"])
    ctx.load_events(synth.to_records(ev))
    ctx.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    n = ctx.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
    d_e = torch.empty(n, dtype=torch.float64, device="cuda:0")
    rot = pb["rot_cp"].reshape(-1, 4)
    groups_of = {}
    out = {}
    for model in (0, 1):
        ctx.cost_set_rotation_model(model)
        r_cp = (rot / np.linalg.norm(rot, axis=1, keepdims=True)).ravel() if model else pb["rot_cp"]
        x = (pb["intrinsics"], r_cp, pb["trans_cp"])
        jobs = {"errors": lambda: ctx.reprojection_errors(*x, d_out=d_e.data_ptr(), host=False)}
        for by in ("keyframe", "circle", "sensor_cell"):
            jobs[by] = (lambda by=by: groups_of.__setitem__(by, ctx.reprojection_groups(*x, by, kf_t=pb["kf_t"], cell_px=16)))
        t = {k: [] for k in jobs}
        for rep in range(2 + a.reps):
            for k, f in jobs.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                stream.synchronize()
                e0.record(stream)
                f()
                e1.record(stream)
                e1.synchronize()
                if rep >= 2:
                    t[k].append(e0.elapsed_time(e1))
        e, n_invalid = ctx.reprojection_errors(*x)
        ok = e[~np.isnan(e)]
        res = {"n_invalid": n_invalid, "rms_px": float(np.sqrt(np.mean(ok * ok)))}
        for k in jobs:
            G = len(groups_of[k][0]) if k in groups_of else 0
            b = traffic(n, G, k)
            med = float(np.median(t[k]))
            res[k] = {"ms": stats(t[k]), "groups": G, "bytes": b, "GB_per_s": b / (med * 1e-3) / 1e9,
                      "share_of_hbm_peak": b / (med * 1e-3) / HBM_BPS}
            if k in groups_of:
                tot = groups_of[k][1]
                assert int(tot["count"]) + int(tot["n_invalid"]) == n and int(tot["n_invalid"]) == n_invalid
        out["quaternion" if model == 0 else "so3"] = res
    ctx.cost_set_rotation_model(0)
    line = json.dumps({"tool": "reprojection_timing", "gpu": gpu_info(), "events": a.events, "residuals": n,
                       "reps": a.reps, "cell_px": 16, "models": out,
                       "note": "CUDA events on the context's stream, median of reps after 2 warm-up rounds; the records (6.7 M x "
                               "64 B = 0.43 GB) exceed L2; bytes derived from shapes, peak 7.7 TB/s (data sheet)"})
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
