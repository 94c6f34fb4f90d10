"""Device time of ecb_trajectory_motion_device and ecb_motion_covariance_device at the C4 size (bench.py --config C4: one
spline segment, D = 843).

    python profiles/tools/trajectory_motion_timing.py [--events 7000000] [--reps 20] [--out FILE]

ecb_covariance runs once per rotation model at the problem's starting point; then 10^6 and 10^7 query times, uniform over the
spline, sorted and the same times shuffled, go through the device variants (torch CUDA tensors): the motion alone at the same
point (control points as host arrays, uploaded by the call) and the motion with its 9 x 9 covariance.  CUDA events on the
context's stream bracket each call (no count, so no synchronise inside); median, min and max over --reps calls after 3 warm-up
calls.  The output (128 or 776 bytes a query: 1.3 or 7.8 GB at 10^7) is far larger than the 126 MB L2.

Shape-derived figures per query: bytes moved = 8 in + 128 motion (+ 648 covariance); FP64 operations of the contraction
Sigma_m = J Z_blk J^T as the kernel runs it (lower triangle of Z, sparse J), 2 per FMA; the motion and its Jacobian are not
counted (dual-number arithmetic with sin / cos / atan, not a fixed FMA count).  They are reported against 7.7 TB/s (HBM3e,
data sheet) and 36.4 TFLOP/s (FP64 DFMA measured on a B200, profiles/r1_fp64_peak.txt), with the bound that applies.  Prints
one JSON line (also to --out).
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12
FP64_FLOP_PER_S = 36.4e12
BYTES_MOTION = 8 + 16 * 8
BYTES_COV = 81 * 8


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception:  # noqa: BLE001
        return "unknown"


def sigma_flops_per_query():
    """FP64 operations of k_motion's motion_sigma: v_c = sum_{r >= c} Z_rc J_r (3 FMA for a rotation row of J, 2 for a
    translation row: v_w and a_w), then the rank-2 update of the upper triangle of Sigma_m by v_c and the column J_c"""
    fma = 0
    for c in range(24):
        fma += sum(3 if r % 6 < 3 else 2 for r in range(c, 24))
        kc = c % 6
        fma += 6 * 2 + 3 * 6 if kc < 3 else 9 * 2   # rotation column: 6 entries x 2 + 18 x 1; translation column: 9 x 2
    return 2 * fma


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
    assert torch.cuda.is_available(), "needs a GPU"
    cfg = bench.CONFIGS["C4"]
    ev, _ = bench.make_workload(cfg, a.events, 0)
    pb = bench.c4_problem(cfg, ev, 1)
    stream = torch.cuda.Stream()
    ctx = ecb.Context(0, stream=stream.cuda_stream)   # the events below are recorded on the same stream
    ctx.set_sensor(cfg["width"], cfg["height"])
    ctx.load_events(synth.to_records(ev))
    ctx.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    n_res = ctx.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
    n_cp = [pb["n_cp"]]
    x = (pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])
    kn = np.asarray(pb["knots"])
    rng = np.random.default_rng(0)
    flops = sigma_flops_per_query()
    res = {"tool": "trajectory_motion_timing", "gpu": gpu_info(), "events": a.events, "residuals": n_res,
           "control_points": int(pb["n_cp"]), "reps": a.reps, "bytes_per_query": {"motion": BYTES_MOTION,
                                                                                  "motion_covariance": BYTES_MOTION + BYTES_COV},
           "sigma_fp64_flop_per_query": flops, "runs": []}
    rot, trans = np.asarray(x[1], np.float64), np.asarray(x[2], np.float64)
    for so3 in (0, 1):
        ctx.cost_set_rotation_model(so3)
        cov = ctx.covariance(n_cp, *x)
        assert cov["ok"], cov
        for n in (1_000_000, 10_000_000):
            sorted_t = np.sort(rng.uniform(kn[0], kn[-1], n))
            for order in ("sorted", "shuffled"):
                t = sorted_t if order == "sorted" else rng.permutation(sorted_t)
                dt = torch.from_numpy(t).cuda()
                dm = torch.empty((n, 16), dtype=torch.float64, device="cuda")
                dc = torch.empty((n, 81), dtype=torch.float64, device="cuda")
                for with_cov in (False, True):
                    if with_cov:
                        def call(count):
                            return ctx.motion_covariance_device(dt.data_ptr(), n, dm.data_ptr(), dc.data_ptr(), count=count)
                    else:
                        def call(count):
                            return ctx.trajectory_motion_device(rot, trans, dt.data_ptr(), n, dm.data_ptr(), count=count)
                    torch.cuda.synchronize()
                    assert call(True) == n
                    ms = []
                    for k in range(3 + a.reps):
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record(stream)
                        call(False)
                        e1.record(stream)
                        e1.synchronize()
                        if k >= 3:
                            ms.append(e0.elapsed_time(e1))
                    # the device result equals the host variant on a sample
                    idx = rng.choice(n, 1000, replace=False)
                    di = torch.from_numpy(idx).cuda()
                    if with_cov:
                        h = ctx.motion_covariance(t[idx])
                        assert np.array_equal(h["cov"].reshape(-1, 81), dc[di].cpu().numpy())
                    else:
                        h = ctx.trajectory_motion(rot, trans, t[idx])
                    got = dm[di].cpu().numpy()
                    assert np.array_equal(np.concatenate([h["pose"], h["omega"], h["velocity"], h["acceleration"]], 1), got)
                    med = float(np.median(ms))
                    nbytes = BYTES_MOTION + (BYTES_COV if with_cov else 0)
                    t_bytes = n * nbytes / HBM_BYTES_PER_S * 1e3
                    t_flops = n * flops / FP64_FLOP_PER_S * 1e3 if with_cov else 0.0
                    res["runs"].append({"rotation_model": "so3" if so3 else "quaternion", "covariance": with_cov, "queries": n,
                                        "order": order, "ms": {"median": med, "min": float(np.min(ms)), "max": float(np.max(ms))},
                                        "bytes_floor_ms": t_bytes, "sigma_flop_floor_ms": t_flops,
                                        "bound": "bytes" if t_bytes >= t_flops else "fp64",
                                        "share_of_bound": max(t_bytes, t_flops) / med,
                                        "queries_per_s": n / (med * 1e-3),
                                        "achieved_GBps": n * nbytes / (med * 1e-3) / 1e9})
                del dt, dm, dc
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
