"""Cost of re-association (ecb_cost_reassociate) at the C4 size (bench.py --config C4: one spline segment over a 7 M-event stream).

    python profiles/tools/reassociation_timing.py [--events 7000000] [--reps 20] [--out FILE] [--ptxas]

For both rotation models, two windows: the association's own (max_dt = 0, 5 motion steps) and twice that.  Before every call the
records are associated again, untimed, so every call compares with the same records; CUDA events on the context's stream bracket
ecb_cost_reassociate (it ends in a synchronise).  The key-frame association (ecb_cost_associate) is timed the same way for scale.
Median / min / max over --reps repetitions after 2 warm-up rounds.  Prints one JSON line (also to --out) with the card's name and
power limit read in the same run; --ptxas adds the -Xptxas -v lines of k_reassoc_count (compiled here for sm_100a).
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
    """registers / spills of both instances of k_reassoc_count from a compile of ecb_cost.cu into a temporary directory"""
    import tempfile
    from eventcalib_b200 import build as b
    with tempfile.TemporaryDirectory() as d:
        out = subprocess.run([b.NVCC] + b.COMMON + ["-Xptxas", "-v", "-c", os.path.join(b.CSRC, "ecb_cost.cu"), "-o",
                                                     os.path.join(d, "ecb_cost.o")], capture_output=True, text=True, check=True)
    lines = (out.stdout + out.stderr).splitlines()
    rep = {}
    for i, l in enumerate(lines):
        m = re.search(r"Function properties for \S*(k_reassoc_count)ILi(\d)E", l)
        if m:
            rep["%s<%s>" % (m.group(1), m.group(2))] = " | ".join(s.strip() for s in lines[i + 1:i + 3])
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

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stream.synchronize()
        e0.record(stream)
        r = fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1), r

    n = associate()
    t_assoc = [timed(associate)[0] for _ in range(2 + a.reps)][2:]
    rot = pb["rot_cp"].reshape(-1, 4)
    window = 5 * pb["step"]
    out = {}
    for model in (0, 1):
        ctx.cost_set_rotation_model(model)
        r_cp = (rot / np.linalg.norm(rot, axis=1, keepdims=True)).ravel() if model else pb["rot_cp"]
        x = (pb["intrinsics"], r_cp, pb["trans_cp"])
        res = {}
        for name, max_dt in (("default_window", 0.0), ("twice_window", 2 * window)):
            t, counts = [], None
            for rep in range(2 + a.reps):
                assert associate() == n
                ms, counts = timed(lambda: ctx.reassociate(*x, max_dt=max_dt))
                if rep >= 2:
                    t.append(ms)
            res[name] = {"max_dt": max_dt, "ms": stats(t), "residuals": counts[0], "same": counts[1], "changed": counts[2],
                         "new": counts[3], "lost": counts[4]}
        out["quaternion" if model == 0 else "so3"] = res
    ctx.cost_set_rotation_model(0)
    rec = {"tool": "reassociation_timing", "gpu": gpu_info(), "events": a.events, "association_residuals": n,
           "keyframes": len(pb["kf_t"]), "circles": int(pb["circles"].shape[1]), "reps": a.reps,
           "association_ms": stats(t_assoc), "models": out,
           "note": "CUDA events on the context's stream around ecb_cost_reassociate (ends in a synchronise) at the problem's start "
                   "point, associated again untimed before every call; ecb_cost_associate timed the same way; median of reps "
                   "after 2 warm-up rounds"}
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
