"""ecb_gyro_calibrate on the GPU, for both rotation models and a spline of two segments: the scan curve and the valid set
against numpy on trajectory_motion; exact recovery of rotation, offset and bias from a gyroscope synthesised from the spline;
agreement with scipy.optimize.least_squares and the residuals against a numpy restatement; the reported uncertainty under
noise; the offset held at 0; the failure statuses; the argument and state errors; determinism; two GPUs; the CLI's ECB_GYRO."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy.optimize import least_squares
from scipy.spatial.transform import Rotation

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R_TRUE = Rotation.from_rotvec([0.3, -1.2, 2.0])
B_TRUE = np.array([0.02, -0.01, 0.005])
D_TRUE = 3.37e-3


def _problem(kind):
    """noise-free control points of the generator's trajectory (build_from_truth), one segment over [5, 5.6] or two"""
    from eventcalib_b200 import synth, calib_problem
    board = synth.Board()
    traj = synth.Trajectory(1004, board, 92.0, (0.35, 0.35, 0.25))
    cam = synth.Camera(346, 260)
    spans = [(5.0, 5.30), (5.34, 5.64)] if kind == "two_segments" else [(5.0, 5.6)]
    pbs = [calib_problem.build_from_truth(cam, traj, board, a, b, seed=1, pose_noise=(0.0, 0.0)) for a, b in spans]
    return dict(so3=int(kind == "so3"), n_cp=[p["n_cp"] for p in pbs], knots=[np.asarray(p["knots"], np.float64) for p in pbs],
                rot=np.concatenate([p["rot_cp"] for p in pbs]), trans=np.concatenate([p["trans_cp"] for p in pbs]),
                radius=pbs[0]["radius"], huber=pbs[0]["huber"], traj=traj)


@pytest.fixture(scope="module", params=["quat", "so3", "two_segments"])
def spline(request):
    import eventcalib_b200 as ecb
    p = _problem(request.param)
    ctx = ecb.Context(0)
    ctx.cost_setup(p["n_cp"], p["knots"], p["radius"], p["huber"])
    ctx.cost_set_rotation_model(p["so3"])
    p["ctx"] = ctx
    yield p
    ctx.close()


def _omega(p, t):
    return p["ctx"].trajectory_motion(p["rot"], p["trans"], t)["omega"]


def _used(p, t, D):
    """the valid set: the first segment holding t - D is the first holding t + D"""
    def seg(u):
        return next((k for k, kn in enumerate(p["knots"]) if kn[0] <= u <= kn[-1]), -1)
    return np.array([np.isfinite(u) and seg(u - D) >= 0 and seg(u - D) == seg(u + D) for u in t])


def _gyro(p, rate=2000.0, R=R_TRUE, d=D_TRUE, b=B_TRUE, noise=0.0, seed=0, margin=0.05):
    """stamps at rate with jitter over the spline (and past its ends), readings R w_c(t + d) + b + noise; stamps whose t + d
    leaves the spline get w_c of the nearest inside time (they are unused anyway)"""
    rng = np.random.default_rng(seed)
    base = np.arange(p["knots"][0][0] - margin, p["knots"][-1][-1] + margin, 1.0 / rate)
    t = base + rng.uniform(-0.3, 0.3, len(base)) / rate
    w = _omega(p, t + d)
    bad = np.isnan(w[:, 0])
    w[bad] = _omega(p, np.clip(t[bad] + d, p["knots"][0][0], p["knots"][-1][-1]))
    w[np.isnan(w[:, 0])] = 0.0   # in the gap between two segments
    g = R.apply(w) + b + rng.normal(0.0, noise, w.shape)
    return np.column_stack([t, g])


def _rot_err(q, R=R_TRUE):
    return (Rotation.from_quat(q) * R.inv()).magnitude()


def test_scan_curve_and_valid_set(spline):
    """offset_cost against numpy (|w_c(t + d_m)| - |w_g|)^2 averaged over the used samples, w_c from trajectory_motion, to 1e-12
    relative; the valid set (NaN stamp, NaN reading, windows leaving the spline or crossing the gap) against numpy; residual rows
    NaN exactly for unused samples"""
    g = _gyro(spline, noise=0.01, seed=1)
    g[5, 0] = np.nan
    g[len(g) // 2, 2] = np.nan
    D, M = 0.02, 41
    out = spline["ctx"].gyro_calibrate(spline["rot"], g, D, M)
    assert out["ok"], out.get("message")
    used = _used(spline, g[:, 0], D) & np.isfinite(g).all(axis=1)
    assert not used[5] and not used[len(g) // 2]
    if len(spline["knots"]) == 2:   # samples whose window crosses the gap
        gap = (g[:, 0] + D > spline["knots"][0][-1]) & (g[:, 0] - D < spline["knots"][1][0])
        assert gap.sum() > 10 and not used[gap].any()
    assert out["n_used"] == used.sum() and out["n_unused"] == len(g) - used.sum()
    assert np.isnan(out["residuals"][~used]).all() and np.isfinite(out["residuals"][used]).all()
    grid = out["offset_grid"]
    assert grid[M // 2] == 0.0 and grid[0] == -D and grid[-1] == D
    t, wg = g[used, 0], np.linalg.norm(g[used, 1:], axis=1)
    ref = np.array([np.mean((np.linalg.norm(_omega(spline, t + d), axis=1) - wg) ** 2) for d in grid])
    np.testing.assert_allclose(out["offset_cost"], ref, rtol=1e-12, atol=0)
    assert out["scan_offset"] == grid[np.argmin(ref)]


def test_exact_recovery(spline):
    """a gyroscope synthesised from the spline itself (R_gc = Exp(0.3, -1.2, 2.0), d = 3.37 ms off the grid of D = 20 ms,
    M = 401, b = (0.02, -0.01, 0.005) rad/s, jittered stamps): rotation, offset and bias to 1e-9, rms <= 1e-9 rad/s"""
    out = spline["ctx"].gyro_calibrate(spline["rot"], _gyro(spline), 0.02, 401)
    assert out["ok"], out.get("message")
    assert out["n_params"] == 7 and out["status"] == 0
    print("exact recovery", _rot_err(out["q_gc"]), out["offset"] - D_TRUE, out["bias"] - B_TRUE, out["rms"], out["iterations"],
          out["termination"])
    assert _rot_err(out["q_gc"]) <= 1e-9
    assert abs(out["offset"] - D_TRUE) <= 1e-9
    assert np.abs(out["bias"] - B_TRUE).max() <= 1e-9
    assert out["rms"] <= 1e-9
    # the scan compares norms, which the bias shifts: its offset is a starting point only
    assert out["scan_offset"] in out["offset_grid"] and abs(out["scan_offset"] - D_TRUE) < 0.01
    np.testing.assert_allclose(out["R_gc"], Rotation.from_quat(out["q_gc"]).as_matrix(), rtol=0, atol=1e-15)


def _objective(p, g, q0):
    """r(delta, d, b) = Exp(delta) R(q0) w_c(t + d) + b - w_g over the used samples, w_c from trajectory_motion"""
    R0 = Rotation.from_quat(q0)

    def f(x):
        w = _omega(p, g[:, 0] + x[3])
        return ((Rotation.from_rotvec(x[:3]) * R0).apply(w) + x[4:] - g[:, 1:]).ravel()

    def jac(x):
        """[-[R w]x, R dw/dt, I3], dw/dt by central differences (h = 1e-6: error ~ 1e-9 relative)"""
        R, h = Rotation.from_rotvec(x[:3]) * R0, 1e-6
        a = R.apply(_omega(p, g[:, 0] + x[3]))
        J = np.zeros((len(g), 3, 7))
        J[:, 0, 1], J[:, 0, 2], J[:, 1, 0], J[:, 1, 2], J[:, 2, 0], J[:, 2, 1] = a[:, 2], -a[:, 1], -a[:, 2], a[:, 0], a[:, 1], -a[:, 0]
        J[:, :, 3] = R.apply((_omega(p, g[:, 0] + x[3] + h) - _omega(p, g[:, 0] + x[3] - h)) / (2 * h))
        J[:, :, 4:] = np.eye(3)
        return J.reshape(-1, 7)
    return f, jac


def test_agrees_with_scipy_and_numpy_residuals(spline):
    """with 0.01 rad/s noise: the solution equals scipy.optimize.least_squares on the same objective (started at the scan
    offset) to 1e-8 of the parameter vector's norm; the residuals at the solution equal R_gc w_c(t + d) + b - w_g to 1e-12 of
    max |w|; cost and rms are 1/2 sum |r|^2 and sqrt(sum |r|^2 / 3n)"""
    D = 0.02
    g = _gyro(spline, noise=0.01, seed=2)
    out = spline["ctx"].gyro_calibrate(spline["rot"], g, D, 401)
    assert out["ok"], out.get("message")
    used = _used(spline, g[:, 0], D)
    gu = g[used]
    f, jac = _objective(spline, gu, out["q_gc"])
    x0 = np.r_[0.0, 0.0, 0.0, out["scan_offset"], np.zeros(3)]
    ls = least_squares(f, x0, jac=jac, method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15,
                       x_scale=np.r_[1, 1, 1, 1e-3, 1e-2, 1e-2, 1e-2])
    q_ls = (Rotation.from_rotvec(ls.x[:3]) * Rotation.from_quat(out["q_gc"])).as_quat()
    q_ls *= np.sign(q_ls @ out["q_gc"])
    ours = np.r_[out["q_gc"], out["offset"], out["bias"]]
    theirs = np.r_[q_ls, ls.x[3], ls.x[4:]]
    print("scipy", np.abs(ours - theirs).max(), out["iterations"], out["termination"])
    assert np.abs(ours - theirs).max() <= 1e-8 * np.linalg.norm(theirs)
    w = _omega(spline, gu[:, 0] + out["offset"])
    r = Rotation.from_quat(out["q_gc"]).apply(w) + out["bias"] - gu[:, 1:]
    assert np.abs(out["residuals"][used] - r).max() <= 1e-12 * np.abs(w).max()
    assert abs(out["cost"] - 0.5 * (r ** 2).sum()) <= 1e-9 * out["cost"]
    assert abs(out["rms"] - np.sqrt((r ** 2).sum() / (3 * used.sum()))) <= 1e-9 * out["rms"]


def test_noise_uncertainty(spline):
    """0.01 rad/s Gaussian noise: every error within 5 reported standard deviations, sigma2 within 10 % of 1e-4; cov symmetric
    positive definite with std = sqrt(sigma2 diag cov)"""
    out = spline["ctx"].gyro_calibrate(spline["rot"], _gyro(spline, noise=0.01, seed=3), 0.02, 401)
    assert out["ok"], out.get("message")
    std = out["std"]
    dtheta = (Rotation.from_quat(out["q_gc"]) * R_TRUE.inv()).as_rotvec()   # left perturbation, gyroscope frame
    err = np.r_[dtheta, out["offset"] - D_TRUE, out["bias"] - B_TRUE]
    print("noise", err / std, out["sigma2"])
    assert (np.abs(err) <= 5 * std).all(), err / std
    assert abs(out["sigma2"] - 1e-4) <= 1e-5
    np.testing.assert_array_equal(out["cov"], out["cov"].T)
    assert np.linalg.eigvalsh(out["cov"]).min() > 0
    np.testing.assert_array_equal(std, np.sqrt(out["sigma2"] * np.diag(out["cov"])))


def test_offset_held_at_zero(spline):
    """D = 0 (one offset): the offset is exactly 0.0, 6 parameters, the offset's row and column of cov are 0"""
    out = spline["ctx"].gyro_calibrate(spline["rot"], _gyro(spline, d=0.0, noise=0.01, seed=4), 0.0, 1)
    assert out["ok"], out.get("message")
    assert out["offset"] == 0.0 and out["scan_offset"] == 0.0 and out["n_params"] == 6
    assert not out["cov"][3].any() and not out["cov"][:, 3].any() and out["std"][3] == 0.0
    assert _rot_err(out["q_gc"]) < 1e-2 and np.abs(out["bias"] - B_TRUE).max() < 1e-2
    assert len(out["offset_cost"]) == 1 and np.isfinite(out["offset_cost"][0])


def test_failure_statuses(spline):
    """rotation about one axis: rank deficient (cov NaN, the estimate still filled); a true offset outside +-D: the scan's
    minimum at the edge; fewer used samples than parameters; every one ECB_FAILED as ok=False with a message"""
    import eventcalib_b200 as ecb
    ctx = spline["ctx"]
    # one axis: every control point a rotation about u
    u = np.array([0.48, -0.6, 0.64])
    ang = 0.8 * np.sin(np.linspace(0.0, 6.0, len(spline["rot"])))
    rot1 = Rotation.from_rotvec(ang[:, None] * u).as_quat()
    p1 = dict(spline, rot=rot1)
    out = ctx.gyro_calibrate(rot1, _gyro(p1, d=0.0, noise=0.0), 0.02, 401)
    assert not out["ok"] and out["status"] == ecb.GYRO_RANK_DEFICIENT and "rank deficient" in out["message"]
    assert np.isnan(out["cov"]).all() and np.isnan(out["std"]).all() and np.isfinite(out["q_gc"]).all()
    # true offset 30 ms, window +-10 ms
    out = ctx.gyro_calibrate(spline["rot"], _gyro(spline, d=0.03), 0.01, 21)
    assert not out["ok"] and out["status"] == ecb.GYRO_OFFSET_AT_EDGE and out["scan_offset"] == 0.01
    assert np.isfinite(out["offset_cost"]).all() and np.isnan(out["q_gc"]).all()
    # too few
    g = _gyro(spline)
    kn = spline["knots"][0]
    few = g[(g[:, 0] > kn[0] + 0.1)][:3]
    for gg in (few, g[:0]):
        out = ctx.gyro_calibrate(spline["rot"], gg, 0.02, 401)
        assert not out["ok"] and out["status"] == ecb.GYRO_TOO_FEW_SAMPLES and out["n_used"] == len(gg)


def test_errors_and_determinism(spline):
    """ECB_ERR_STATE before cost_setup; every ECB_ERR_ARG case of the header; two identical calls are bit-identical"""
    import eventcalib_b200 as ecb
    ctx = spline["ctx"]
    g = _gyro(spline, noise=0.01, seed=5)
    a = ctx.gyro_calibrate(spline["rot"], g, 0.02, 401)
    b = ctx.gyro_calibrate(spline["rot"], g, 0.02, 401)
    for k, v in a.items():
        np.testing.assert_array_equal(v, b[k], err_msg=k)
    fresh = ecb.Context(0)
    try:
        with pytest.raises(ecb.EcbError) as e:
            fresh.gyro_calibrate(spline["rot"], g, 0.02, 401)
        assert e.value.code == ecb.ERR_STATE
    finally:
        fresh.close()
    lib, h = ctx.lib, ctx.h
    r, gg = np.ascontiguousarray(spline["rot"]), np.ascontiguousarray(g)
    out = ecb.GyroCalibration()

    def call(hh=h, rr=r, gp=gg, n=len(g), D=0.02, M=401, o=True):
        return lib.ecb_gyro_calibrate(hh, rr.ctypes.data_as(C.c_void_p) if rr is not None else None,
                                      gp.ctypes.data_as(C.c_void_p) if gp is not None else None, n, D, M,
                                      C.byref(out) if o else None, None, None)
    assert call() == ecb.OK
    for kw in (dict(hh=None), dict(o=False), dict(n=-1), dict(gp=None), dict(D=np.nan), dict(D=-1e-3), dict(D=np.inf),
               dict(M=400), dict(M=0), dict(M=-1), dict(M=65537), dict(D=0.0, M=3), dict(M=1)):
        assert call(**kw) == ecb.ERR_ARG, kw
    assert call(gp=None, n=0, D=0.0, M=1) == ecb.FAILED   # no samples: too few, not an argument error


def test_two_gpus():
    """the same calibration on two GPUs is bit-identical"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import eventcalib_b200 as ecb
    p = _problem("quat")
    outs, g = [], None
    for dev in (0, 1):
        c = ecb.Context(dev)
        try:
            c.cost_setup(p["n_cp"], p["knots"], p["radius"], p["huber"])
            p["ctx"] = c
            g = _gyro(p, noise=0.01, seed=6) if g is None else g
            outs.append(c.gyro_calibrate(p["rot"], g, 0.02, 401))
        finally:
            c.close()
    for k, v in outs[0].items():
        np.testing.assert_array_equal(v, outs[1][k], err_msg=k)


def test_cli_camera_gyroscope(tmp_path):
    """ECB_GYRO on the stream of test_cli_writes_trajectory_motion with a 1 kHz gyroscope of the generator's true trajectory
    (known R_gc, offset, bias, 0.005 rad/s noise): bad values or a bad file exit with code 1 before any output; every other file
    is byte for byte the one without the variable; CameraGyroscope.txt has the model header, the estimate and the scan curve;
    the estimate lies within 0.45 deg / 2 ms / 0.006 rad/s of the truth.  Measured on the first run (B200): 0.22 deg, +1.04 ms
    (the offset's reported deviation 0.19 ms: the event-calibrated spline lags the generator's trajectory), 0.0029 rad/s."""
    from eventcalib_b200 import synth
    from test_host_cli import YAML, CLI, HOST
    import eventcalib_b200.build as b
    b.build()
    subprocess.check_call(["make", "-s", "-C", HOST])
    ev = synth.make_stream(2000000, 346, 260, t0=5.0, duration=1.0, seed=1001, return_truth=True, workers=4,
                           rot_amp=(0.35, 0.35, 0.3), orbit=True)
    synth.write_bin(str(tmp_path / "ev.bin"), ev)
    (tmp_path / "cfg.yaml").write_text(YAML.replace("fitCircle: 0", "fitCircle: 1"))
    R, d, bias = Rotation.from_rotvec([0.4, -0.9, 1.7]), 2.5e-3, np.array([0.02, -0.01, 0.005])
    g = synth.gyro_samples(ev["trajectory"], 5.0, 6.0, 1000.0, R.as_matrix(), d, bias, 0.005, seed=7)
    with open(tmp_path / "gyro.txt", "w") as f:
        f.write("# t wx wy wz ax ay az\n\n")
        for row in g:
            f.write(" ".join("%.17g" % v for v in row) + " 0 0 9.81\n")
    (tmp_path / "bad.txt").write_text("# header\n5.0 0.1 0.2 0.3\n5.001 0.1 x 0.3\n")

    def run(out, code=0, **env_extra):
        env = dict(os.environ, ECB_PIECES="4", ECB_NO_IMAGES="1", ECB_DEVICES="0", **env_extra)
        env.pop("ECB_DEVICE", None)
        r = subprocess.run([CLI, str(tmp_path / "cfg.yaml"), str(tmp_path / "ev.bin"), str(out)], capture_output=True, text=True,
                           stdin=subprocess.DEVNULL, timeout=600, env=env)
        assert r.returncode == code, r.stdout[-2000:] + r.stderr
        return r

    good = str(tmp_path / "gyro.txt")
    for env, msg in ((dict(ECB_GYRO=str(tmp_path / "missing.txt")), "cannot open"),
                     (dict(ECB_GYRO=str(tmp_path / "bad.txt")), "line 3"),
                     *[(dict(ECB_GYRO=good, ECB_GYRO_MAX_OFFSET=v), "ECB_GYRO_MAX_OFFSET must be") for v in ("-1", "nan", "inf", "abc", "")]):
        r = run(tmp_path / "bad", code=1, **env)
        assert msg in r.stderr, (env, r.stderr)
        assert not (tmp_path / "bad").exists() and "Camera-gyroscope" not in r.stdout
    plain, with_gyro = tmp_path / "plain", tmp_path / "gyro"
    plain.mkdir()
    with_gyro.mkdir()
    run(plain)
    out = run(with_gyro, ECB_GYRO=good).stdout
    line = [l for l in out.splitlines() if l.startswith("Camera-gyroscope:")]
    assert len(line) == 1 and " ms (+- " in line[0] and " deg, bias " in line[0] and " rad/s, " in line[0], out[-2000:]
    files = sorted(p.name for p in plain.iterdir())
    assert sorted(p.name for p in with_gyro.iterdir()) == sorted(files + ["CameraGyroscope.txt"])
    for name in files:
        assert (plain / name).read_bytes() == (with_gyro / name).read_bytes(), name
    text = (with_gyro / "CameraGyroscope.txt").read_text().splitlines()
    assert text[0].startswith("# camera-gyroscope calibration: w_g(t) = R_gc w_c(t + offset) + bias")
    assert "rad/s" in text[1] and "gyroscope frame" in text[1]
    k = next(i for i, l in enumerate(text) if l.startswith("# scan"))
    kv = {l.split()[0]: np.array([float(v) for v in l.split()[1:]]) for l in text[2:k]}
    assert sorted(kv) == sorted(["q_gc", "R_gc", "rotation_std", "offset", "offset_std", "bias", "bias_std", "rms", "sigma2",
                                 "n_used", "n_unused", "scan_offset", "iterations", "termination"])
    scan = np.array([[float(v) for v in l.split()] for l in text[k + 1:]])
    assert scan.shape == (1001, 2) and scan[500, 0] == 0.0 and abs(scan[0, 0] + 0.05) < 1e-15 and np.isfinite(scan).all()
    assert kv["R_gc"].shape == (9,) and kv["n_used"][0] > 500
    np.testing.assert_allclose(kv["R_gc"].reshape(3, 3), Rotation.from_quat(kv["q_gc"]).as_matrix(), atol=1e-12)
    e_rot = np.degrees(_rot_err(kv["q_gc"], R))
    e_off, e_b = kv["offset"][0] - d, np.abs(kv["bias"] - bias).max()
    print("cli", e_rot, "deg", 1e3 * e_off, "ms", e_b, "rad/s", kv["rms"], kv["offset_std"], kv["rotation_std"], kv["bias_std"])
    assert e_rot <= 0.45 and abs(e_off) <= 2e-3 and e_b <= 0.006
