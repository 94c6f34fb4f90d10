"""ecb_trajectory_motion and ecb_motion_covariance on the GPU: the motion (pose, body angular velocity, world velocity and
acceleration) against the CPU-verified header (tests/helpers/motion_host.cpp, checked in test_motion_jacobian.py) and the 9 x 9
covariance against J Z_dense J^T, for both rotation models and two segments; the pose against pose_covariance's; the explicit
control-point call against the covariance call; host against device variants; independence of the batch; NaN rows; the state
and argument errors; two GPUs; the CLI's ECB_TRAJECTORY_MOTION output; the frame and units against the generator's trajectory."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_gpu_pose_covariance import _z_dense, _stream

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _host_lib():
    """the motion header built for the host (-ffp-contract=off, as test_motion_jacobian.py builds it)"""
    out = os.path.join(ROOT, "tests", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libmotion_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", so,
                           os.path.join(ROOT, "tests", "helpers", "motion_host.cpp")])
    lib = C.CDLL(so)
    lib.host_ders_basis.restype = lib.host_motion.restype = None
    lib.host_ders_basis.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.host_motion.argtypes = [C.c_void_p] * 5 + [C.c_int, C.c_void_p, C.c_void_p]
    return lib


def _P(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="module", params=["quat", "so3", "two_segments"])
def solved(request):
    """the calibrated problems of test_gpu_pose_covariance.py with their covariance computed on their own context"""
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth, calib_problem
    so3 = int(request.param == "so3")
    if request.param == "two_segments":
        ev = synth.make_stream(160000, 346, 260, t0=5.0, duration=0.64, seed=1004, return_truth=True, rot_amp=(0.35, 0.35, 0.25),
                               dist=92.0)
        a = calib_problem.build_from_truth(ev["camera"], ev["trajectory"], ev["board"], 5.0, 5.30, seed=1)
        b = calib_problem.build_from_truth(ev["camera"], ev["trajectory"], ev["board"], 5.34, 5.64, seed=2)
        pbs = [a, b]
        rot0 = np.concatenate([a["rot_cp"], b["rot_cp"]])
        trans0 = np.concatenate([a["trans_cp"], b["trans_cp"]])
        iters = 50
    else:
        ev = _stream(150000, 0.6) if so3 == 0 else _stream(100000, 0.4)
        a = calib_problem.build(ev, seed=2, intr_noise=0.02)
        pbs = [a]
        rot0 = a["rot_cp"].reshape(-1, 4)
        rot0 = rot0 / np.linalg.norm(rot0, axis=1, keepdims=True)
        trans0 = a["trans_cp"]
        iters = 20 if so3 == 0 else 12
    n_cp = [p["n_cp"] for p in pbs]
    knots = [np.asarray(p["knots"], np.float64) for p in pbs]
    ctx = ecb.Context(0)
    ctx.set_sensor(346, 260)
    ctx.load_events(synth.to_records(ev))
    ctx.cost_setup(n_cp, knots, a["radius"], a["huber"])
    ctx.cost_set_rotation_model(so3)
    kf_t = np.concatenate([p["kf_t"] for p in pbs])
    ctx.cost_associate(kf_t, np.concatenate([p["circles"] for p in pbs]), a["landmarks"], a["step"])
    i, r, t, _, _ = ctx.calibrate(n_cp, a["intrinsics"], rot0, trans0, ecb.lm_options(max_iterations=iters, rotation_model=so3))
    x = (i, np.asarray(r, np.float64).reshape(-1, 4), np.asarray(t, np.float64).reshape(-1, 3))
    assert ctx.covariance(n_cp, *x)["ok"]
    yield dict(ctx=ctx, so3=so3, n_cp=n_cp, knots=knots, x=x, kf_t=kf_t, Z=_z_dense(ctx, n_cp, x))
    ctx.close()


def _queries(knots, kf_t, seed=0):
    """key-frame stamps, random times inside each segment's knot range, every knot"""
    rng = np.random.default_rng(seed)
    return np.concatenate([kf_t, *[rng.uniform(k[0], k[-1], 200 // len(knots)) for k in knots], *knots])


def _reference(solved, lib, times):
    """(motion16, Sigma_m) per time from the host header and the dense Z; None outside every segment"""
    import oracle
    oracle.build()
    n_cp, knots, (_, rot, trans), Z = solved["n_cp"], solved["knots"], solved["x"], solved["Z"]
    cp_off = np.r_[0, np.cumsum(n_cp)[:-1]]
    out = []
    for u in times:
        s = next((k for k, kn in enumerate(knots) if kn[0] <= u <= kn[-1]), None)
        if s is None:
            out.append(None)
            continue
        kn = np.ascontiguousarray(knots[s])
        span, _ = oracle.basis(kn, u)
        N, Nd, Ndd = np.zeros(4), np.zeros(4), np.zeros(4)
        lib.host_ders_basis(_P(kn), span, u, _P(N), _P(Nd), _P(Ndd))
        c0 = cp_off[s] + span - 3
        Q, T = np.ascontiguousarray(rot[c0:c0 + 4]), np.ascontiguousarray(trans[c0:c0 + 4])
        m, J = np.zeros(16), np.zeros((9, 24))
        lib.host_motion(_P(Q), _P(T), _P(N), _P(Nd), _P(Ndd), solved["so3"], _P(m), _P(J))
        blk = Z[6 * c0:6 * c0 + 24, 6 * c0:6 * c0 + 24]
        out.append((m, J @ blk @ J.T))
    return out


def _motion_rows(d):
    return np.concatenate([d["pose"], d["omega"], d["velocity"], d["acceleration"]], axis=1)


def test_motion_covariance_matches_host_header(solved):
    """motion against the host header: the pose 1e-13, w / v / a 1e-11 of their largest value (device FMA contraction and the
    device's atan / sin / cos against glibc's are the only differences); Sigma_m against J Z_dense J^T to 1e-7 of its largest
    entry (the selected inverse against a dense inverse, as for the pose covariance); exact symmetry, PSD"""
    lib = _host_lib()
    ctx = solved["ctx"]
    times = _queries(solved["knots"], solved["kf_t"])
    got = ctx.motion_covariance(times)
    ref = _reference(solved, lib, times)
    valid = np.array([r is not None for r in ref])
    assert valid[len(solved["kf_t"]):].all() and valid.sum() > len(times) // 2
    assert got["n_valid"] == valid.sum()
    M = _motion_rows(got)
    assert np.isnan(M[~valid]).all() and np.isnan(got["cov"][~valid]).all()
    assert np.isfinite(M[valid]).all() and np.isfinite(got["cov"][valid]).all()
    Mr = np.array([r[0] for r in ref if r is not None])
    Sr = np.array([r[1] for r in ref if r is not None])
    M, S = M[valid], got["cov"][valid]
    for lo, hi, tol in ((0, 7, 1e-13), (7, 10, 1e-11), (10, 13, 1e-11), (13, 16, 1e-11)):
        scale = max(1.0, np.abs(Mr[:, lo:hi]).max())
        assert np.abs(M[:, lo:hi] - Mr[:, lo:hi]).max() <= tol * scale, (lo, np.abs(M[:, lo:hi] - Mr[:, lo:hi]).max() / scale)
    assert np.abs(S - Sr).max() <= 1e-7 * np.abs(Sr).max(), np.abs(S - Sr).max() / np.abs(Sr).max()
    np.testing.assert_array_equal(S, np.transpose(S, (0, 2, 1)))
    ev = np.linalg.eigvalsh(S)
    assert (ev[:, 0] >= -1e-12 * ev[:, -1]).all() and (ev[:, -1] > 0).all()
    # the pose column is pose_covariance's pose, bit for bit
    np.testing.assert_array_equal(got["pose"], ctx.pose_covariance(times)["pose"])


def test_trajectory_motion_is_motion_covariance(solved):
    """trajectory_motion at the covariance's point equals motion_covariance's motion bit for bit (NaN rows included)"""
    ctx, (_, rot, trans) = solved["ctx"], solved["x"]
    lo, hi = min(k[0] for k in solved["knots"]), max(k[-1] for k in solved["knots"])
    times = np.r_[_queries(solved["knots"], solved["kf_t"], seed=5), np.linspace(lo - 0.01, hi + 0.01, 5000), np.nan]
    a = ctx.trajectory_motion(rot, trans, times)
    b = ctx.motion_covariance(times)
    np.testing.assert_array_equal(_motion_rows(a), _motion_rows(b))
    assert a["n_valid"] == b["n_valid"]


def test_motion_outside_and_nan(solved):
    ctx, knots, (_, rot, trans) = solved["ctx"], solved["knots"], solved["x"]
    lo, hi = min(k[0] for k in knots), max(k[-1] for k in knots)
    inside = np.array([lo, knots[0][4], hi])   # first knot, an interior knot of the first segment, last knot
    times = np.array([lo - 1.0, inside[0], np.nan, inside[1], hi + 1e-9, inside[2], -np.inf, np.inf])
    if len(knots) == 2:   # the gap between the two segments
        times = np.r_[times, 0.5 * (knots[0][-1] + knots[1][0])]
    ok = np.isin(times, inside)
    for got in (ctx.motion_covariance(times), ctx.trajectory_motion(rot, trans, times)):
        M = _motion_rows(got)
        assert got["n_valid"] == 3
        assert np.isnan(M[~ok]).all() and np.isfinite(M[ok]).all()
        if "cov" in got:
            assert np.isnan(got["cov"][~ok]).all() and np.isfinite(got["cov"][ok]).all()
    empty = ctx.motion_covariance(np.zeros(0))
    assert empty["n_valid"] == 0 and empty["cov"].shape == (0, 9, 9)
    assert ctx.trajectory_motion(rot, trans, np.zeros(0))["n_valid"] == 0
    r, t = np.ascontiguousarray(rot), np.ascontiguousarray(trans)
    assert ctx.lib.ecb_motion_covariance(ctx.h, None, -1, None, None, None) == -2   # ECB_ERR_ARG
    assert ctx.lib.ecb_motion_covariance_device(ctx.h, None, -1, None, None, None) == -2
    assert ctx.lib.ecb_trajectory_motion(ctx.h, _P(r), _P(t), None, -1, None, None) == -2
    assert ctx.lib.ecb_trajectory_motion(ctx.h, None, _P(t), None, 0, None, None) == -2
    assert ctx.lib.ecb_trajectory_motion_device(ctx.h, _P(r), None, None, 0, None, None) == -2
    assert ctx.lib.ecb_trajectory_motion_device(ctx.h, _P(r), _P(t), None, 5, None, None) == -2   # no times


def test_motion_independent_of_batch(solved):
    """a time asked alone equals, bit for bit, the same time inside a shuffled batch of 10^6; a repeated call is identical; the
    device variants on torch tensors equal the host variants; every output may be left out"""
    import torch
    ctx, knots, (_, rot, trans) = solved["ctx"], solved["knots"], solved["x"]
    rng = np.random.default_rng(3)
    lo, hi = min(k[0] for k in knots), max(k[-1] for k in knots)
    probe = np.r_[solved["kf_t"][:5], knots[0][4], knots[-1][-1]]
    batch = np.r_[rng.uniform(lo - 0.01, hi + 0.01, 1_000_000 - len(probe)), probe]
    perm = rng.permutation(len(batch))
    batch = batch[perm]
    where = np.argsort(perm)[-len(probe):]
    big = ctx.motion_covariance(batch)
    Mb = _motion_rows(big)
    for k, u in enumerate(probe):
        one = ctx.motion_covariance([u])
        np.testing.assert_array_equal(_motion_rows(one)[0], Mb[where[k]])
        np.testing.assert_array_equal(one["cov"][0], big["cov"][where[k]])
        np.testing.assert_array_equal(_motion_rows(ctx.trajectory_motion(rot, trans, [u]))[0], Mb[where[k]])
    again = ctx.motion_covariance(batch)
    np.testing.assert_array_equal(again["cov"], big["cov"])
    np.testing.assert_array_equal(_motion_rows(again), Mb)
    assert again["n_valid"] == big["n_valid"]
    dt = torch.from_numpy(batch).cuda()
    dm = torch.empty((len(batch), 16), dtype=torch.float64, device="cuda")
    dc = torch.empty((len(batch), 81), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    assert ctx.motion_covariance_device(dt.data_ptr(), len(batch), dm.data_ptr(), dc.data_ptr()) == big["n_valid"]
    np.testing.assert_array_equal(dm.cpu().numpy(), Mb)
    np.testing.assert_array_equal(dc.cpu().numpy().reshape(-1, 9, 9), big["cov"])
    dm.zero_()
    assert ctx.trajectory_motion_device(rot, trans, dt.data_ptr(), len(batch), dm.data_ptr()) == big["n_valid"]
    np.testing.assert_array_equal(dm.cpu().numpy(), Mb)
    # asynchronous without a count; outputs left out
    dm.zero_()
    assert ctx.trajectory_motion_device(rot, trans, dt.data_ptr(), len(batch), dm.data_ptr(), count=False) is None
    ctx.synchronize()
    np.testing.assert_array_equal(dm.cpu().numpy(), Mb)
    assert ctx.motion_covariance_device(dt.data_ptr(), len(batch), 0, 0) == big["n_valid"]
    only_cov = ctx.motion_covariance_device(dt.data_ptr(), len(batch), 0, dc.data_ptr())
    assert only_cov == big["n_valid"]
    np.testing.assert_array_equal(dc.cpu().numpy().reshape(-1, 9, 9), big["cov"])
    nv = C.c_int64()
    cov_only = np.empty((1000, 9, 9))
    assert ctx.lib.ecb_motion_covariance(ctx.h, _P(np.ascontiguousarray(batch[:1000])), 1000, None, _P(cov_only),
                                         C.byref(nv)) == 0
    np.testing.assert_array_equal(cov_only, big["cov"][:1000])


def test_motion_state_errors():
    """ecb_trajectory_motion: ECB_ERR_STATE before ecb_cost_setup only.  ecb_motion_covariance: the rules of
    ecb_pose_covariance — before any covariance, after ecb_cost_setup, a rotation-model switch or a constant-intrinsics change"""
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth, calib_problem
    ev = _stream(150000, 0.6)
    pb = calib_problem.build(ev, seed=2, intr_noise=0.02)
    n_cp = [pb["n_cp"]]
    x = (pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])
    ctx = ecb.Context(0)
    t = np.array([pb["knots"][4]])

    def state_error(f):
        with pytest.raises(ecb.EcbError) as e:
            f()
        return e.value.code == ecb.ERR_STATE

    try:
        ctx.set_sensor(346, 260)
        ctx.load_events(synth.to_records(ev))
        assert state_error(lambda: ctx.trajectory_motion(x[1], x[2], t))   # before ecb_cost_setup
        assert state_error(lambda: ctx.motion_covariance(t))
        ctx.cost_setup(n_cp, [pb["knots"]], pb["radius"], pb["huber"])
        assert ctx.trajectory_motion(x[1], x[2], t)["n_valid"] == 1      # no covariance needed
        ctx.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
        assert state_error(lambda: ctx.motion_covariance(t))              # before any covariance
        assert ctx.covariance(n_cp, *x)["ok"]
        assert ctx.motion_covariance(t)["n_valid"] == 1
        ctx.cost_set_rotation_model(1)
        assert state_error(lambda: ctx.motion_covariance(t))
        assert ctx.trajectory_motion(x[1], x[2], t)["n_valid"] == 1
        ctx.cost_set_rotation_model(0)
        assert state_error(lambda: ctx.motion_covariance(t))              # still: the covariance was taken before the switch
        assert ctx.covariance(n_cp, *x)["ok"]
        assert ctx.motion_covariance(t)["n_valid"] == 1
        ctx.set_constant_intrinsics(["k4", "k5"])                      # Z of other free parameters
        assert state_error(lambda: ctx.motion_covariance(t))
        assert ctx.covariance(n_cp, *x)["ok"]
        assert ctx.motion_covariance(t)["n_valid"] == 1
        ctx.cost_setup(n_cp, [pb["knots"]], pb["radius"], pb["huber"])   # new knots
        assert state_error(lambda: ctx.motion_covariance(t))
        assert ctx.trajectory_motion(x[1], x[2], t)["n_valid"] == 1
    finally:
        ctx.close()


def test_motion_two_gpus():
    """the normal equations exchanged between two GPUs, ecb_covariance on each rank from the summed buffer: both ranks' motion
    and motion covariances are bit-identical"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth, calib_problem
    ev = _stream(120000, 0.5)
    pb = calib_problem.build(ev, seed=2, intr_noise=0.02)
    rec = synth.to_records(ev)
    n = len(rec)
    n_cp = [pb["n_cp"]]
    x = (pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])
    kn = np.asarray(pb["knots"])
    times = np.r_[pb["kf_t"], np.linspace(kn[0], kn[-1], 1000)]
    ranks = []
    for dev, (lo, hi) in enumerate(((0, n // 2 + 333), (n // 2 + 333, n))):
        c = ecb.Context(dev)
        c.set_sensor(346, 260)
        c.load_events(rec[lo:hi])
        c.cost_setup(n_cp, [pb["knots"]], pb["radius"], pb["huber"])
        c.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
        c.enable_peer_access(1 - dev)
        ranks.append(c)
    bufs = [c.device_alloc(c.exchange_buffer_bytes(2)) for c in ranks]
    outs = [c.device_alloc(8 * c.cost_layout()["out_doubles"]) for c in ranks]
    m = sum(c.cost_layout()["n_residuals"] for c in ranks)
    try:
        for r, c in enumerate(ranks):
            c.cost_normal_eq_exchange(*x, r, bufs, 1, outs[r], want_cost=False)
        covs = [c.covariance(n_cp, *x, d_packed=outs[r], n_residuals_total=m) for r, c in enumerate(ranks)]
        assert covs[0]["ok"] and covs[1]["ok"]
        mot = [c.motion_covariance(times) for c in ranks]
        traj = [c.trajectory_motion(x[1], x[2], times) for c in ranks]
    finally:
        for c, p, q in zip(ranks, bufs, outs):
            c.synchronize()
            c.device_free(p)
            c.device_free(q)
            c.close()
    assert mot[0]["n_valid"] == len(times)
    np.testing.assert_array_equal(mot[0]["cov"], mot[1]["cov"])
    np.testing.assert_array_equal(_motion_rows(mot[0]), _motion_rows(mot[1]))
    np.testing.assert_array_equal(_motion_rows(traj[0]), _motion_rows(traj[1]))
    np.testing.assert_array_equal(_motion_rows(traj[0]), _motion_rows(mot[0]))


def test_motion_frame_and_units():
    """on build_from_truth control points (noise-free key-frame poses, 15 control points over 0.4 s), w_b and v_w at interior
    times agree with central differences of the generator's Trajectory (w_b = Log(R(t-h)^T R(t+h)) / 2h of R_wb, v_w of t_wb)
    within 5 % relative RMS, for both rotation models.  Measured: 0.23 % for w_b and 0.21 % for v_w (the spline's fit of the
    sinusoids); a world-frame w, a flipped sign or another time unit is off by 100 % or more."""
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth, calib_problem
    from scipy.spatial.transform import Rotation
    board = synth.Board()
    traj = synth.Trajectory(1004, board, 92.0, (0.35, 0.35, 0.25))
    pb = calib_problem.build_from_truth(synth.Camera(346, 260), traj, board, 5.0, 5.4, seed=1, pose_noise=(0.0, 0.0))
    kn = np.asarray(pb["knots"], np.float64)
    t = np.linspace(kn[0] + 0.05, kn[-1] - 0.05, 400)
    h = 1e-5
    Rm, tm = traj.pose(t - h)
    Rp, tp = traj.pose(t + h)
    w_ref = np.array([Rotation.from_matrix(a.T @ b).as_rotvec() for a, b in zip(Rm, Rp)]) / (2 * h)
    v_ref = (tp - tm) / (2 * h)

    def rel(a, b):
        return np.sqrt(((a - b) ** 2).sum() / (b ** 2).sum())

    ctx = ecb.Context(0)
    try:
        ctx.cost_setup([pb["n_cp"]], [kn], pb["radius"], pb["huber"])
        for so3 in (0, 1):
            ctx.cost_set_rotation_model(so3)
            got = ctx.trajectory_motion(pb["rot_cp"], pb["trans_cp"], t)
            assert got["n_valid"] == len(t)
            ew, ev_ = rel(got["omega"], w_ref), rel(got["velocity"], v_ref)
            assert ew < 0.05 and ev_ < 0.05, (so3, ew, ev_)
            assert rel(-got["omega"], w_ref) > 1.0
    finally:
        ctx.close()


def test_cli_writes_trajectory_motion(tmp_path):
    """ECB_TRAJECTORY_MOTION=200 on the stream of test_cli_writes_trajectory_covariance: TrajectoryMotion.txt has the units
    header, 19 columns (stamp, w_b, v_w, a_w, 9 deviations), stamps t0 + k / 200 inside the segments, positive finite deviations;
    a "Trajectory motion:" line; every other output file is byte for byte the one without the variable.  An invalid rate ends
    the program with exit code 1 before any file work."""
    from eventcalib_b200 import synth
    from test_host_cli import YAML, CLI, HOST
    import eventcalib_b200.build as b
    b.build()
    subprocess.check_call(["make", "-s", "-C", HOST])
    ev = synth.make_stream(2000000, 346, 260, t0=5.0, duration=1.0, seed=1001, return_truth=True, workers=4,
                           rot_amp=(0.35, 0.35, 0.3), orbit=True)
    synth.write_bin(str(tmp_path / "ev.bin"), ev)
    (tmp_path / "cfg.yaml").write_text(YAML.replace("fitCircle: 0", "fitCircle: 1"))

    def run(out, code=0, **env_extra):
        env = dict(os.environ, ECB_PIECES="4", ECB_NO_IMAGES="1", ECB_DEVICES="0", **env_extra)
        env.pop("ECB_DEVICE", None)
        r = subprocess.run([CLI, str(tmp_path / "cfg.yaml"), str(tmp_path / "ev.bin"), str(out)], capture_output=True, text=True,
                           stdin=subprocess.DEVNULL, timeout=600, env=env)
        assert r.returncode == code, r.stdout[-2000:] + r.stderr
        return r

    for bad in ("0", "-5", "abc", "inf", "nan", "200Hz", ""):
        r = run(tmp_path / "bad", code=1, ECB_TRAJECTORY_MOTION=bad)
        assert "ECB_TRAJECTORY_MOTION must be a positive finite number" in r.stderr
        assert not (tmp_path / "bad").exists()
    plain, with_motion = tmp_path / "plain", tmp_path / "motion"
    plain.mkdir()
    with_motion.mkdir()
    run(plain)
    out = run(with_motion, ECB_TRAJECTORY_MOTION="200").stdout
    line = [l for l in out.splitlines() if l.startswith("Trajectory motion:")]
    assert len(line) == 1 and "at 200 Hz" in line[0]
    files = sorted(p.name for p in plain.iterdir())
    assert sorted(p.name for p in with_motion.iterdir()) == sorted(files + ["TrajectoryMotion.txt"])
    for name in files:
        assert (plain / name).read_bytes() == (with_motion / name).read_bytes(), name
    lines = (with_motion / "TrajectoryMotion.txt").read_text().splitlines()
    head = [l for l in lines if l.startswith("#")]
    rows = np.array([[float(v) for v in l.split()] for l in lines if not l.startswith("#")])
    assert len(head) == 2 and "rad/s" in head[1] and "board units/s^2" in head[1]
    assert rows.shape[1] == 19 and len(rows) > 100
    assert int(line[0].split()[2]) == len(rows)
    k = (rows[:, 0] - rows[0, 0]) * 200.0
    assert np.abs(k - np.round(k)).max() < 1e-4 and (np.diff(rows[:, 0]) > 0).all()   # printed with 10 decimals
    assert np.isfinite(rows).all() and (rows[:, 10:] > 0).all()
    wmax = np.sqrt((rows[:, 1:4] ** 2).sum(1)).max()
    assert abs(wmax - float(line[0].split("max |omega|")[1].split()[0])) <= 1e-6 * wmax
