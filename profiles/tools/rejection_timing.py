"""Cost of outlier rejection (ecb_cost_reject) at the C4 size (bench.py --config C4: one spline segment over a 7 M-event stream,
6.7 M residuals).

    python profiles/tools/rejection_timing.py [--events 7000000] [--reps 20] [--out FILE] [--ptxas FILE]

For both rotation models, two cases: a threshold that removes about 1 % of the records (the 99th percentile of |r| at the start
point), and a mask that drops every tenth key frame.  Before every call the records are associated again, untimed; CUDA events
on the context's stream bracket ecb_cost_reject (it ends in a synchronise).  Median / min / max over --reps repetitions after 2
warm-up rounds.  Prints one JSON line (also to --out) with the card's name and power limit read in the same run; --ptxas writes
the -Xptxas -v lines of the two rejection kernels (compiled here for sm_100a).
"""
import argparse
import json
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def stats(v):
    return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}


def ptxas_report():
    """registers / spills of k_reject_count and k_reject_write from a compile of ecb_cost.cu into a temporary directory"""
    import tempfile
    from eventcalib_b200 import build as b
    with tempfile.TemporaryDirectory() as d:
        out = subprocess.run([b.NVCC] + b.COMMON + ["-Xptxas", "-v", "-c", os.path.join(b.CSRC, "ecb_cost.cu"), "-o",
                                                     os.path.join(d, "ecb_cost.o")], capture_output=True, text=True, check=True)
    lines = (out.stdout + out.stderr).splitlines()
    rep = {}
    for i, l in enumerate(lines):
        m = re.search(r"Function properties for \S*(k_reject_\w+?)E", l)
        if m:
            rep[m.group(1)] = " | ".join(s.strip() for s in lines[i + 1:i + 3])
    return rep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--events", type=int, default=7_000_000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="")
    ap.add_argument("--ptxas", action="store_true")
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

    def associate():
        return ctx.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])

    n = associate()
    K = len(pb["kf_t"])
    drop = (np.arange(K) % 10 == 5).astype(np.uint8)
    rot = pb["rot_cp"].reshape(-1, 4)
    out = {}
    for model in (0, 1):
        ctx.cost_set_rotation_model(model)
        r_cp = (rot / np.linalg.norm(rot, axis=1, keepdims=True)).ravel() if model else pb["rot_cp"]
        x = (pb["intrinsics"], r_cp, pb["trans_cp"])
        associate()
        thr = float(np.quantile(np.abs(ctx.cost_residuals(*x)), 0.99))
        jobs = {"threshold_1pct": dict(max_abs_r=thr), "drop_tenth_keyframes": dict(drop_keyframes=drop, kf_t=pb["kf_t"])}
        res = {}
        for k, kw in jobs.items():
            t, counts = [], None
            for rep in range(2 + a.reps):
                assert associate() == n
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                stream.synchronize()
                e0.record(stream)
                counts = ctx.reject_residuals(*x, **kw)
                e1.record(stream)
                e1.synchronize()
                if rep >= 2:
                    t.append(e0.elapsed_time(e1))
            res[k] = {"ms": stats(t), "kept": counts[0], "removed": counts[1],
                      "removed_share": counts[1] / n}
            if k == "threshold_1pct":
                res[k]["max_abs_r"] = thr
        out["quaternion" if model == 0 else "so3"] = res
    ctx.cost_set_rotation_model(0)
    rec = {"tool": "rejection_timing", "gpu": gpu_info(), "events": a.events, "residuals": n, "keyframes": K, "reps": a.reps,
           "models": out,
           "note": "CUDA events on the context's stream around ecb_cost_reject (ends in a synchronise), re-associated untimed "
                   "before every call; median of reps after 2 warm-up rounds"}
    if a.ptxas:
        rec["ptxas"] = ptxas_report()
    line = json.dumps(rec)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
