"""The residual report (ecb_cost_residuals, ecb_cost_residual_groups): the raw residuals r_k against the restated oracle, the
grouped statistics against a numpy grouping of the GPU's own r, determinism, shards, error codes and the CLI files.
r is a distance on the board plane (units of the board points), not pixels."""
import math
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _raw_from_corrected(res, huber):
    """inverts the Huber corrector of the oracle's rows: res = r inside the band, sign(r) sqrt(delta |r|) outside"""
    return np.where(np.abs(res) <= huber, res, np.sign(res) * res * res / huber)


def _rho_half(r, huber):
    s = r * r
    return 0.5 * np.where(s > huber * huber, 2.0 * huber * np.abs(r) - huber * huber, s)


def _nearest_kf(kf, u):
    lo = np.searchsorted(kf, u, side="left")
    best = np.minimum(lo, len(kf) - 1)
    prev = np.maximum(lo - 1, 0)
    take_prev = (lo > 0) & ((lo >= len(kf)) | ((u - kf[prev]) <= (kf[np.minimum(lo, len(kf) - 1)] - u)))
    return np.where(take_prev, prev, best)


def _numpy_groups(r, key, n_groups, huber):
    out = []
    for g in range(n_groups):
        v = r[key == g]
        out.append(dict(count=len(v), n_downweighted=int(np.count_nonzero(v * v > huber * huber)), sum=math.fsum(v),
                        sum_sq=math.fsum(v * v), max_abs=float(np.abs(v).max()) if len(v) else 0.0,
                        cost=math.fsum(_rho_half(v, huber))))
    return out


def _check_groups(groups, ref, rtol=1e-12):
    assert len(groups) == len(ref)
    for g, q in zip(groups, ref):
        assert int(g["count"]) == q["count"] and int(g["n_downweighted"]) == q["n_downweighted"]
        assert float(g["max_abs"]) == q["max_abs"]
        for f in ("sum", "sum_sq", "cost"):
            assert abs(float(g[f]) - q[f]) <= rtol * abs(q[f]), (f, float(g[f]), q[f])


def _same(a, b):
    return a.tobytes() == b.tobytes()


@pytest.fixture(scope="module")
def assoc(oracle_mod):
    """the stream of test_gpu_cost plus one event exactly midway between two key-frame stamps (a copy of an event associated
    with the earlier frame): the tie must go to the earlier frame"""
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth, calib_problem
    ev = synth.make_stream(300000, 346, 260, t0=5.0, duration=0.3, seed=1004, return_truth=True)
    pb = calib_problem.build(ev, seed=3)
    kf = pb["kf_t"]
    P = oracle_mod.CostProblem([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    oe, oc = P.associate(ev["t"], ev["x"], ev["y"], kf, pb["circles"], pb["landmarks"], pb["step"])
    key0 = _nearest_kf(kf, ev["t"][oe])
    mid = None
    for i in range(1, len(kf) - 2):
        u = 0.5 * (kf[i] + kf[i + 1])
        if (u - kf[i]) == (kf[i + 1] - u) and np.any(key0 == i):
            mid = (u, int(oe[np.nonzero(key0 == i)[0][0]]), i)
            break
    assert mid is not None
    u, src, i_mid = mid
    ev2 = {k: np.append(ev[k], ev[k][src]) for k in ("t", "x", "y", "p")}
    ev2["t"][-1] = u
    order = np.argsort(ev2["t"], kind="stable")
    ev2 = {k: v[order] for k, v in ev2.items()}
    mid_index = int(np.nonzero(order == len(order) - 1)[0][0])
    c = ecb.Context(0)
    c.set_sensor(346, 260)
    c.load_events(synth.to_records(ev2))
    c.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    n = c.cost_associate(kf, pb["circles"], pb["landmarks"], pb["step"])
    P = oracle_mod.CostProblem([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    oe, oc = P.associate(ev2["t"], ev2["x"], ev2["y"], kf, pb["circles"], pb["landmarks"], pb["step"])
    assert n == len(oe) and np.any(oe == mid_index)
    Ps = oracle_mod.CostProblem([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"], so3=True)
    Ps.associate(ev2["t"], ev2["x"], ev2["y"], kf, pb["circles"], pb["landmarks"], pb["step"])
    yield dict(ctx=c, ev=ev2, pb=pb, P=P, Ps=Ps, n=n, mid_index=mid_index, i_mid=i_mid)
    c.close()


def _points(a, so3):
    pb = a["pb"]
    rot = pb["rot_cp"].reshape(-1, 4)
    if so3:
        rot = rot / np.linalg.norm(rot, axis=1, keepdims=True)
    x0 = (pb["intrinsics"], rot.ravel(), pb["trans_cp"])
    import eventcalib_b200 as ecb
    intr, rot1, trans1, summ, _ = a["ctx"].calibrate(pb["n_cp"], *x0, options=ecb.lm_options(max_iterations=8, rotation_model=int(so3)))
    assert summ["final_cost"] < summ["initial_cost"]
    return [x0, (intr, rot1, trans1)]


@pytest.mark.parametrize("so3", [False, True])
def test_association_residuals_and_groups(oracle_mod, assoc, so3):
    c, pb, ev = assoc["ctx"], assoc["pb"], assoc["ev"]
    huber = pb["huber"]
    P = assoc["Ps"] if so3 else assoc["P"]
    c.cost_set_rotation_model(int(so3))
    try:
        for x in _points(assoc, so3):
            # 1. r_k against the oracle's rows (corrector inverted), every record
            r = c.cost_residuals(*x)
            c_ref, _, _, res_ref, _ = P.normal_eq(*x, want_rows=True)
            r_ref = _raw_from_corrected(res_ref, huber)
            assert len(r) == assoc["n"]
            assert np.all(np.abs(r - r_ref) <= 1e-9 * np.maximum(1.0, np.abs(r_ref)))
            assert np.count_nonzero(r * r > huber * huber) > 0
            # ... and a sample against the reference's own functor, where it travelled with the repository
            if oracle_mod.have_ref_functor():
                ei, ci = c.cost_association()
                rng = np.random.default_rng(5)
                rot = np.asarray(x[1]).reshape(-1, 4)
                trans = np.asarray(x[2]).reshape(-1, 3)
                for k in rng.choice(len(r), 1000, replace=False):
                    e = ei[k]
                    sp, N = oracle_mod.basis(pb["knots"], ev["t"][e])
                    obs = np.array([ev["x"][e], ev["y"][e]], float)
                    lm = pb["landmarks"][ci[k]]
                    Q, T = rot[sp - 3:sp + 1], trans[sp - 3:sp + 1]
                    if so3:
                        beta = np.array([N[1] + N[2] + N[3], N[2] + N[3], N[3]])
                        _, _, rd = oracle_mod.ref_residual_jac_so3(x[0], Q, T, obs, lm, pb["radius"], beta, N)
                    else:
                        _, _, rd = oracle_mod.ref_residual_jac(x[0], Q, T, obs, lm, pb["radius"], N)
                    assert abs(r[k] - rd) <= 1e-9 * max(1.0, abs(rd))
            # 2. the cost three ways
            cost = c.cost_eval(*x)
            assert abs(math.fsum(_rho_half(r, huber)) - cost) <= 1e-12 * cost
            ei, ci = c.cost_association()
            keys = {"keyframe": (_nearest_kf(pb["kf_t"], ev["t"][ei]), len(pb["kf_t"])),
                    "circle": (ci, pb["circles"].shape[1]),
                    "sensor_cell": None}
            assert keys["keyframe"][0][np.nonzero(ei == assoc["mid_index"])[0][0]] == assoc["i_mid"]
            obs = np.stack([ev["x"][ei], ev["y"][ei]], 1).astype(float)
            for cell in (16, 7):
                ncx, ncy = -(-346 // cell), -(-260 // cell)
                keys["sensor_cell"] = (np.floor(obs[:, 1] / cell).astype(np.int64) * ncx + np.floor(obs[:, 0] / cell).astype(np.int64),
                                       ncx * ncy)
                assert np.any(obs[:, 0] % cell == 0)   # observations on cell edges
                for by, (key, G) in keys.items():
                    g, tot = c.residual_groups(*x, by, kf_t=pb["kf_t"], cell_px=cell)
                    assert len(g) == G
                    _check_groups(g, _numpy_groups(r, key, G, huber))
                    assert abs(float(g["cost"].sum()) - cost) <= 1e-12 * cost
                    assert abs(float(tot["cost"]) - cost) <= 1e-12 * cost
                    assert int(tot["count"]) == len(r) and float(tot["max_abs"]) == np.abs(r).max()
                    # 4. determinism
                    g2, tot2 = c.residual_groups(*x, by, kf_t=pb["kf_t"], cell_px=cell)
                    assert _same(g, g2) and _same(tot, tot2)
            assert _same(c.cost_residuals(*x), r)
    finally:
        c.cost_set_rotation_model(0)


def _explicit_problem():
    """two spline segments, non-integer observations, residuals far outside the Huber band, observations on cell edges and
    outside the sensor"""
    from eventcalib_b200 import synth, spline
    rng = np.random.default_rng(9)
    board = synth.Board()
    traj = synth.Trajectory(3, board, 78.0)
    knots, ncp, rot, trans, obs, lm, tt, sp = [], [], [], [], [], [], [], []
    for s, (a, b, n_cp) in enumerate([(1.0, 1.4, 7), (2.0, 2.25, 5)]):
        us = np.linspace(a, b, 40)
        kn = spline.knot_vector(us, n_cp)
        q, tw = traj.quat_xyzw(us)
        rot.append(spline.fit_control_points(kn, us, q, n_cp))
        trans.append(spline.fit_control_points(kn, us, tw, n_cp))
        knots.append(kn)
        ncp.append(n_cp)
        t = np.sort(rng.uniform(a, b, 5000))
        t[0], t[-1] = a, b
        tt.append(t)
        sp.append(np.full(len(t), s))
        o = np.stack([rng.uniform(10, 330, len(t)), rng.uniform(10, 250, len(t))], 1)
        o[:40] = np.stack([rng.integers(0, 22, 40) * 16.0, rng.integers(0, 17, 40) * 16.0], 1)   # on cell edges
        o[40:50] = [[-0.5, 10], [346.0, 10], [10, 260.0], [10, -1e-9], [400, 300], [345.999, 259.999], [0, 0], [-3, -3],
                    [1e6, 5], [5, 1e6]]
        obs.append(o)
        lm.append(board.centres()[rng.integers(0, 36, len(t))])
    return ncp, knots, np.concatenate(rot), np.concatenate(trans), *map(np.concatenate, (obs, lm, tt, sp))


def _explicit_ctx(ncp, knots, obs, lm, tt, sp, sensor=True):
    import eventcalib_b200 as ecb
    c = ecb.Context(0)
    if sensor:
        c.set_sensor(346, 260)
    c.cost_setup(ncp, knots, 1.75, 0.35)
    c.cost_set_residuals(obs, lm, tt, sp)
    return c


@pytest.mark.parametrize("so3", [False, True])
def test_explicit_residuals_and_shards(oracle_mod, so3):
    from eventcalib_b200 import synth
    ncp, knots, rot, trans, obs, lm, tt, sp = _explicit_problem()
    if so3:
        rot = (rot.reshape(-1, 4) / np.linalg.norm(rot.reshape(-1, 4), axis=1, keepdims=True)).ravel()
    x = (synth.Camera().intrinsics(), rot, trans)
    huber = 0.35
    c = _explicit_ctx(ncp, knots, obs, lm, tt, sp)
    c.cost_set_rotation_model(int(so3))
    P = oracle_mod.CostProblem(ncp, knots, 1.75, huber, so3=so3)
    P.set_residuals(obs, lm, tt, sp)
    r = c.cost_residuals(*x)
    _, _, _, res_ref, _ = P.normal_eq(*x, want_rows=True)
    r_ref = _raw_from_corrected(res_ref, huber)
    assert np.all(np.abs(r - r_ref) <= 1e-9 * np.maximum(1.0, np.abs(r_ref)))
    assert np.abs(r).max() > 100 * huber
    cost = c.cost_eval(*x)
    assert abs(math.fsum(_rho_half(r, huber)) - cost) <= 1e-12 * cost
    cell = 16
    ncx, ncy = 22, 17
    inside = (obs[:, 0] >= 0) & (obs[:, 0] < 346) & (obs[:, 1] >= 0) & (obs[:, 1] < 260)
    assert np.count_nonzero(~inside) >= 16
    key = np.where(inside, np.floor(np.where(inside, obs[:, 1], 0) / cell).astype(np.int64) * ncx +
                   np.floor(np.where(inside, obs[:, 0], 0) / cell).astype(np.int64), -1)
    g, tot = c.residual_groups(*x, "sensor_cell", cell_px=cell)
    _check_groups(g, _numpy_groups(r, key, ncx * ncy, huber))
    assert int(g["count"].sum()) == np.count_nonzero(inside)
    _check_groups([tot], _numpy_groups(r, np.zeros(len(r), np.int64), 1, huber))   # the outside records count in the total
    assert abs(float(tot["cost"]) - cost) <= 1e-12 * cost
    g2, tot2 = c.residual_groups(*x, "sensor_cell", cell_px=cell)
    assert _same(g, g2) and _same(tot, tot2)
    # 5. two contexts on device 0 holding contiguous halves (as the shards do), combined in rank order
    h = len(tt) // 2
    parts = [_explicit_ctx(ncp, knots, obs[a:b], lm[a:b], tt[a:b], sp[a:b]) for a, b in ((0, h), (h, len(tt)))]
    comb, ctot = None, None
    for p in parts:
        p.cost_set_rotation_model(int(so3))
        gp, tp = p.residual_groups(*x, "sensor_cell", cell_px=cell)
        if comb is None:
            comb, ctot = gp.copy(), tp.copy()
        else:
            for f in ("count", "n_downweighted", "sum", "sum_sq", "cost"):
                comb[f] += gp[f]
                ctot[f] += tp[f]
            comb["max_abs"] = np.maximum(comb["max_abs"], gp["max_abs"])
            ctot["max_abs"] = max(float(ctot["max_abs"]), float(tp["max_abs"]))
        p.close()
    for a_, b_ in ((comb, g), (ctot[None], tot[None])):
        for f in ("count", "n_downweighted", "max_abs"):
            assert np.array_equal(a_[f], b_[f])
        for f in ("sum", "sum_sq", "cost"):
            assert np.all(np.abs(a_[f] - b_[f]) <= 1e-12 * np.maximum(np.abs(b_[f]), 1e-300))
    c.close()


def test_error_codes_and_edge_cases(assoc):
    import ctypes as C
    import eventcalib_b200 as ecb
    a, pb = assoc["ctx"], assoc["pb"]
    x = (pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])
    lib = a.lib
    xs = [np.ascontiguousarray(v, np.float64) for v in x]
    kf = np.ascontiguousarray(pb["kf_t"], np.float64)
    K, n_circ = len(kf), pb["circles"].shape[1]

    def call(ctx, by, kf_ptr, nk, cell, groups=None, cap=0, total=None):
        ng = C.c_int(-7)
        rc = lib.ecb_cost_residual_groups(ctx.h, ecb._ptr(xs[0]), ecb._ptr(xs[1]), ecb._ptr(xs[2]), by, kf_ptr, nk, cell,
                                          ecb._ptr(groups) if groups is not None else None, cap, C.byref(ng),
                                          ecb._ptr(total) if total is not None else None)
        return rc, ng.value

    kfp = ecb._ptr(kf)
    # size queries
    assert call(a, 0, kfp, K, 16) == (ecb.OK, K)
    assert call(a, 1, None, 0, 16) == (ecb.OK, n_circ)
    assert call(a, 2, None, 0, 16) == (ecb.OK, 22 * 17)
    assert call(a, 2, None, 0, 1) == (ecb.OK, 346 * 260)
    # cap too small: ECB_ERR_ARG, n_groups still set, nothing written
    buf = np.full(n_circ, 7, ecb.RESIDUAL_GROUP_DTYPE)
    tot = np.full((), 7, ecb.RESIDUAL_GROUP_DTYPE)
    assert call(a, 1, None, 0, 16, buf, n_circ - 1, tot) == (ecb.ERR_ARG, n_circ)
    assert np.all(buf["count"] == 7) and int(tot["count"]) == 7
    assert call(a, 1, None, 0, 16, buf, n_circ, tot) == (ecb.OK, n_circ)
    assert int(tot["count"]) == assoc["n"]
    # argument errors
    assert call(a, 3, kfp, K, 16)[0] == ecb.ERR_ARG
    assert call(a, -1, kfp, K, 16)[0] == ecb.ERR_ARG
    assert call(a, 2, None, 0, 0)[0] == ecb.ERR_ARG
    assert call(a, 0, None, K, 16)[0] == ecb.ERR_ARG
    assert call(a, 0, kfp, K - 1, 16)[0] == ecb.ERR_ARG
    # explicit residuals have no key frame or circle; no sensor: no cells
    ncp, knots, rot, trans, obs, lm, tt, sp = _explicit_problem()
    e = _explicit_ctx(ncp, knots, obs, lm, tt, sp, sensor=False)
    assert call(e, 0, kfp, K, 16)[0] == ecb.ERR_STATE
    assert call(e, 1, None, 0, 16)[0] == ecb.ERR_STATE
    assert call(e, 2, None, 0, 16)[0] == ecb.ERR_STATE
    with pytest.raises(ecb.EcbError):
        e.residual_groups(*x, "sensor_cell")
    with pytest.raises(ValueError):
        e.residual_groups(*x, "span")
    # zero residuals: all-zero groups
    e.set_sensor(346, 260)
    e.cost_setup(ncp, knots, 1.75, 0.35)
    e.cost_set_residuals(np.zeros((0, 2)), np.zeros((0, 3)), np.zeros(0), np.zeros(0))
    xe = (x[0], rot, trans)
    assert len(e.cost_residuals(*xe)) == 0
    g, t = e.residual_groups(*xe, "sensor_cell", cell_px=32)
    assert len(g) == 11 * 9 and not np.any(g.view(np.uint8)) and not np.any(np.atleast_1d(t).view(np.uint8))
    e.close()
    # events loaded after the association: no key-frame grouping (the circle grouping needs no events)
    from eventcalib_b200 import synth
    b = ecb.Context(0)
    ev = assoc["ev"]
    b.set_sensor(346, 260)
    b.load_events(synth.to_records(ev))
    b.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    b.cost_associate(kf, pb["circles"], pb["landmarks"], pb["step"])
    g0, t0 = b.residual_groups(*x, "keyframe", kf_t=kf)
    b.load_events(synth.to_records(ev))
    assert call(b, 0, kfp, K, 16)[0] == ecb.ERR_STATE
    assert call(b, 1, None, 0, 16)[0] == ecb.OK
    b.cost_associate(kf, pb["circles"], pb["landmarks"], pb["step"])
    g1, t1 = b.residual_groups(*x, "keyframe", kf_t=kf)
    assert _same(g0, g1) and _same(t0, t1)
    # the device output variant: asynchronous into a caller's buffer, the same values as the host copy
    import torch
    d = torch.empty(assoc["n"], dtype=torch.float64, device="cuda:0")
    b.cost_residuals(*x, d_out=d.data_ptr(), host=False)
    b.synchronize()
    assert np.array_equal(d.cpu().numpy(), a.cost_residuals(*x))
    b.close()


def _run_cli(tmp_path, save, env_extra, devices="0"):
    from test_host_cli import CLI
    env = dict(os.environ, ECB_PIECES="4", ECB_NO_IMAGES="1", ECB_DEVICES=devices, **env_extra)
    env.pop("ECB_DEVICE", None)
    return subprocess.run([CLI, str(tmp_path / "cfg.yaml"), str(tmp_path / "ev.bin"), str(save)], capture_output=True, text=True,
                          stdin=subprocess.DEVNULL, timeout=600, env=env)


def _read(path):
    rows = [l.split() for l in path.read_text().splitlines() if not l.startswith("#")]
    return np.array(rows, float)


def test_cli_writes_residual_report(tmp_path):
    """ECB_RESIDUALS=1 on the stream of test_cli_writes_intrinsics_covariance"""
    from eventcalib_b200 import synth
    from test_host_cli import YAML, HOST
    import eventcalib_b200.build as bld
    bld.build()
    subprocess.check_call(["make", "-s", "-C", HOST])
    ev = synth.make_stream(2000000, 346, 260, t0=5.0, duration=1.0, seed=1001, return_truth=True, workers=4,
                           rot_amp=(0.35, 0.35, 0.3), orbit=True)
    synth.write_bin(str(tmp_path / "ev.bin"), ev)
    (tmp_path / "cfg.yaml").write_text(YAML.replace("fitCircle: 0", "fitCircle: 1"))
    r = _run_cli(tmp_path, tmp_path / "bad", {"ECB_RESIDUALS": "1", "ECB_RESIDUAL_CELL": "0"})
    assert r.returncode == 1 and "ECB_RESIDUAL_CELL" in r.stderr
    assert _run_cli(tmp_path, tmp_path / "bad", {"ECB_RESIDUAL_CELL": "x16"}).returncode == 1
    plain = tmp_path / "plain"
    r = _run_cli(tmp_path, plain, {})
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr
    assert not any((plain / f).exists() for f in ("ResidualsByKeyframe.txt", "ResidualsByCircle.txt", "ResidualMap.txt"))
    assert "Residuals:" not in r.stdout

    def run(save, devices):
        r = _run_cli(tmp_path, save, {"ECB_RESIDUALS": "1", "ECB_RESIDUAL_CELL": "20"}, devices)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr
        summ = [l for l in r.stdout.splitlines() if l.startswith("Solver Summary:")][0]
        n_res = int(summ.split("residuals ")[1].split(",")[0])
        final = float(summ.split("->")[1].split(",")[0])
        line = [l for l in r.stdout.splitlines() if l.startswith("Residuals:")][0]
        kf, circ, cells = (_read(save / f) for f in ("ResidualsByKeyframe.txt", "ResidualsByCircle.txt", "ResidualMap.txt"))
        return n_res, final, line, kf, circ, cells

    save = tmp_path / "out"
    n_res, final, line, kf, circ, cells = run(save, "0")
    assert kf.shape[1] == 7 and circ.shape == (36, 10) and cells.shape[1] == 8
    for f in ("ResidualsByKeyframe.txt", "ResidualsByCircle.txt", "ResidualMap.txt"):
        assert "not pixels" in (save / f).read_text()
    assert "# cell 20 px" in (save / "ResidualMap.txt").read_text()
    traj = _read(save / "TrajectoryByEvent.txt")
    assert set(np.round(traj[:, 0], 6)) <= set(np.round(kf[:, 0], 6)) and np.all(np.diff(kf[:, 0]) > 0)
    for tab, c_count, c_cost in ((kf, 1, 6), (circ, 4, 9), (cells, 2, 7)):
        assert int(tab[:, c_count].sum()) == n_res
        assert abs(tab[:, c_cost].sum() - final) <= 1e-7 * final
    assert np.all(cells[:, 0] % 20 == 0) and np.all(cells[:, 1] % 20 == 0) and np.all(cells[:, 2] > 0)
    # the totals line: count, RMS, mean, max |r|, down-weighted
    nums = line.replace("(", " ").replace(",", " ").split()
    count, rms, mean, mx, ndw = int(nums[1]), float(nums[3]), float(nums[5]), float(nums[8]), int(nums[10])
    assert count == n_res
    w = kf[:, 1]
    assert abs(rms - math.sqrt(np.sum(w * np.nan_to_num(kf[:, 3]) ** 2) / count)) <= 1e-9 * rms
    assert abs(mean - np.sum(w * np.nan_to_num(kf[:, 2])) / count) <= 1e-9 * max(abs(mean), 1e-12)
    assert mx == pytest.approx(np.nanmax(kf[:, 4]), rel=1e-9) and ndw == int(kf[:, 5].sum())
    import torch
    if torch.cuda.device_count() >= 2:   # 6. ShardedCalibSpline::residualGroups over two GPUs against one
        n2, final2, _, kf2, circ2, cells2 = run(tmp_path / "out2", "0,1")
        assert n2 == n_res
        for a_, b_, cc in ((kf, kf2, 1), (circ, circ2, 4), (cells, cells2, 2)):
            assert np.array_equal(a_[:, cc], b_[:, cc])
            np.testing.assert_allclose(b_[:, cc + 5], a_[:, cc + 5], rtol=1e-5)
