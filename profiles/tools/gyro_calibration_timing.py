"""Time of ecb_gyro_calibrate on a minute of data: a 60 s spline with knots every 25 ms (2 403 control points at the Greville
abscissae of the generator's trajectory) and a 1 kHz gyroscope (6 * 10^4 samples, synth.gyro_samples, 0.01 rad/s noise),
D = 0.1 s, M = 2 001 offsets: 1.2 * 10^8 evaluations of w_c in the scan.

    python profiles/tools/gyro_calibration_timing.py [--reps 10] [--out FILE]

For both rotation models, after 2 warm-up calls:
- the whole call: host clock around Context.gyro_calibrate (it ends in a synchronise), median over --reps calls;
- the scan alone: device time of the k_gyro_reduce<..., ScanOp> kernel per call, from torch.profiler (CUDA activities) over
  --reps calls in a pass of its own;
- for comparison, ecb_trajectory_motion_device at the same n x M query times, sorted (host clock around the call, which waits
  for its count), median over --reps calls.
Rates are w_c evaluations (scan) and queries (k_motion) per second.  Prints one JSON line with the GPU's name and power limit
(also to --out).
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
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def problem():
    from eventcalib_b200 import synth
    from scipy.spatial.transform import Rotation
    traj = synth.Trajectory(1004, synth.Board(), 92.0, (0.35, 0.35, 0.25))
    t0, t1, dt = 5.0, 65.0, 0.025
    inner = np.arange(t0, t1 + dt / 2, dt)
    kn = np.r_[[t0] * 3, inner, [inner[-1]] * 3]
    n_cp = len(kn) - 4
    grev = (kn[1:n_cp + 1] + kn[2:n_cp + 2] + kn[3:n_cp + 3]) / 3.0
    rot, trans = traj.quat_xyzw(grev)
    g = synth.gyro_samples(traj, t0 + 0.15, t1 - 0.15, 1000.0, Rotation.from_rotvec([0.3, -1.2, 2.0]).as_matrix(), 3.37e-3,
                           (0.02, -0.01, 0.005), 0.01, seed=1)
    return n_cp, kn, np.ascontiguousarray(rot), np.ascontiguousarray(trans), g


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import eventcalib_b200 as ecb
    n_cp, kn, rot, trans, g = problem()
    D, M, n = 0.1, 2001, len(g)
    ctx = ecb.Context(0)
    ctx.cost_setup([n_cp], [kn], 1.0, 1.0)
    res = {"tool": "gyro_calibration_timing", "gpu": gpu_info(), "n_samples": n, "n_offsets": M, "max_offset": D,
           "n_cp": n_cp, "reps": a.reps}
    grid = D * (2.0 * np.arange(M) - (M - 1)) / (M - 1)
    for so3 in (0, 1):
        ctx.cost_set_rotation_model(so3)
        tag = "so3" if so3 else "quat"
        for _ in range(2):
            out = ctx.gyro_calibrate(rot, g, D, M)
        times = []
        for _ in range(a.reps):
            ctx.synchronize()
            s = time.perf_counter()
            out = ctx.gyro_calibrate(rot, g, D, M)
            times.append(time.perf_counter() - s)
        assert out["ok"], out.get("message")
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(a.reps):
                ctx.gyro_calibrate(rot, g, D, M)
            ctx.synchronize()
        scan_us = sum(e.device_time_total for e in prof.key_averages() if "ScanOp" in e.key) / a.reps
        n_eval = out["n_used"] * M
        # k_motion at the same n x M times, sorted
        dt = (torch.from_numpy(g[:, 0]).cuda()[:, None] + torch.from_numpy(grid).cuda()[None, :]).reshape(-1)
        dt = torch.sort(dt).values.contiguous()
        dm = torch.empty((dt.numel(), 16), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        mt = []
        for k in range(a.reps + 2):
            s = time.perf_counter()
            ctx.trajectory_motion_device(rot, trans, dt.data_ptr(), dt.numel(), dm.data_ptr())
            if k >= 2:
                mt.append(time.perf_counter() - s)
        del dm, dt
        torch.cuda.empty_cache()
        res[tag] = {"call_ms_median": 1e3 * float(np.median(times)), "call_ms_min": 1e3 * min(times),
                    "call_ms_max": 1e3 * max(times), "scan_ms": scan_us / 1e3, "scan_evals_per_s": n_eval / (scan_us * 1e-6),
                    "motion_queries": n * M, "motion_ms_median": 1e3 * float(np.median(mt)),
                    "motion_queries_per_s": n * M / float(np.median(mt)), "n_used": out["n_used"],
                    "iterations": out["iterations"], "termination": out["termination"], "offset_error_s": out["offset"] - 3.37e-3,
                    "rms": out["rms"]}
    ctx.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
