"""ecb_pose_covariance on the GPU: the 6 x 6 pose covariance Sigma(t) = J Z_blk J^T against J from the CPU-verified header
(tests/helpers/pose_host.cpp, checked in test_pose_jacobian.py) times a dense inverse of the GPU normal equations, for both
rotation models and two segments; poses against EventCalibSpline::evaluate; NaN rows outside the splines; independence of the
batch; the state errors; two GPUs; the CLI's ECB_TRAJECTORY_COVARIANCE=1 output."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import lm_oracle

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _host_libs():
    """the pose header built for the host, and the façade's EventCalibSpline::evaluate"""
    import eventcalib_b200.build as b
    b.build()
    out = os.path.join(ROOT, "tests", "_build")
    os.makedirs(out, exist_ok=True)
    pose_so, fac_so = os.path.join(out, "libpose_host.so"), os.path.join(out, "libfacade_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", pose_so,
                           os.path.join(ROOT, "tests", "helpers", "pose_host.cpp")])
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", fac_so,
                           os.path.join(ROOT, "tests", "helpers", "facade_host.cpp"),
                           "-L" + os.path.join(ROOT, "eventcalib_b200"), "-lecb",
                           "-Wl,-rpath," + os.path.join(ROOT, "eventcalib_b200")])
    lib, fac = C.CDLL(pose_so), C.CDLL(fac_so)
    lib.host_pose_jacobian.restype = None
    return lib, fac


def _P(a):
    return a.ctypes.data_as(C.c_void_p)


def _stream(n_events, duration):
    from eventcalib_b200 import synth
    return synth.make_stream(n_events, 346, 260, t0=5.0, duration=duration, seed=1004, return_truth=True,
                             rot_amp=(0.35, 0.35, 0.25), dist=92.0)


def _z_dense(ctx, n_cp, x):
    """Z = H^-1 (band rows first, intrinsics last) from a dense inverse of the GPU's assembled normal equations at x"""
    _, Hs, gs = ctx.cost_normal_eq(*x)
    maps, Ct = lm_oracle._index_map(n_cp)
    D = 9 + 6 * Ct
    A, _ = lm_oracle.assemble(Hs, gs, maps, D)
    perm = np.r_[9:D, 0:9]
    H = A[np.ix_(perm, perm)]
    d = np.diag(H)
    s = np.where(d > 0, 1.0 / np.sqrt(np.where(d > 0, d, 1.0)), 1.0)
    return np.linalg.inv(H * s[:, None] * s[None, :]) * s[:, None] * s[None, :]


@pytest.fixture(scope="module", params=["quat", "so3", "two_segments"])
def solved(request):
    """a calibrated problem of test_gpu_covariance.py with its covariance computed on its own context"""
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
    cov = ctx.covariance(n_cp, *x)
    assert cov["ok"]
    yield dict(ctx=ctx, so3=so3, n_cp=n_cp, knots=knots, x=x, kf_t=kf_t, cov=cov, Z=_z_dense(ctx, n_cp, x))
    ctx.close()


def _queries(knots, kf_t, seed=0):
    """key-frame stamps, random times inside each segment's knot range (not in the gap between segments), every knot"""
    rng = np.random.default_rng(seed)
    return np.concatenate([kf_t, *[rng.uniform(k[0], k[-1], 200 // len(knots)) for k in knots], *knots])


def _reference(solved, lib, fac, times):
    """(pose, Sigma_ref) per time from the host header and the dense Z; None outside every segment"""
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
        span, N = oracle.basis(knots[s], u)
        c0 = cp_off[s] + span - 3
        Q, T = np.ascontiguousarray(rot[c0:c0 + 4]), np.ascontiguousarray(trans[c0:c0 + 4])
        pose, J = np.zeros(7), np.zeros((6, 24))
        lib.host_pose_jacobian(_P(Q), _P(T), _P(N), solved["so3"], _P(pose), _P(J))
        q4, t3 = np.zeros(4), np.zeros(3)
        kn = np.ascontiguousarray(knots[s])
        assert fac.fh_eval(_P(kn), int(n_cp[s]), _P(np.ascontiguousarray(rot[cp_off[s]:cp_off[s] + n_cp[s]])),
                           _P(np.ascontiguousarray(trans[cp_off[s]:cp_off[s] + n_cp[s]])), solved["so3"], C.c_double(u), _P(q4),
                           _P(t3)) == 1
        blk = Z[6 * c0:6 * c0 + 24, 6 * c0:6 * c0 + 24]
        out.append((np.r_[t3, q4], J @ blk @ J.T))
    return out


def test_pose_covariance_matches_dense_reference(solved):
    lib, fac = _host_libs()
    times = _queries(solved["knots"], solved["kf_t"])
    got = solved["ctx"].pose_covariance(times)
    ref = _reference(solved, lib, fac, times)
    valid = np.array([r is not None for r in ref])
    # the random times and the knots lie inside a segment by construction; a key frame may not (it then has no pose either)
    assert valid[len(solved["kf_t"]):].all() and valid.sum() > len(times) // 2
    assert got["n_valid"] == valid.sum()
    assert np.isnan(got["cov"][~valid]).all() and np.isfinite(got["cov"][valid]).all()
    ref = [r for r in ref if r is not None]
    got = {"cov": got["cov"][valid], "pose": got["pose"][valid]}
    S, Sr = got["cov"], np.array([r[1] for r in ref])
    assert np.abs(S - Sr).max() <= 1e-7 * np.abs(Sr).max(), np.abs(S - Sr).max() / np.abs(Sr).max()
    np.testing.assert_array_equal(S, np.transpose(S, (0, 2, 1)))
    ev = np.linalg.eigvalsh(S)
    assert (ev[:, 0] >= -1e-12 * ev[:, -1]).all() and (ev[:, -1] > 0).all()
    pose_ref = np.array([r[0] for r in ref])
    assert np.abs(got["pose"] - pose_ref).max() <= 1e-13 * max(1.0, np.abs(pose_ref).max())


def test_pose_covariance_outside_and_nan(solved):
    ctx, knots = solved["ctx"], solved["knots"]
    lo, hi = min(k[0] for k in knots), max(k[-1] for k in knots)
    inside = np.array([lo, knots[0][4], hi])   # first knot, an interior knot of the first segment, last knot
    times = np.array([lo - 1.0, inside[0], np.nan, inside[1], hi + 1e-9, inside[2], -np.inf, np.inf])
    if len(knots) == 2:   # the gap between the two segments
        times = np.r_[times, 0.5 * (knots[0][-1] + knots[1][0])]
    got = ctx.pose_covariance(times)
    ok = np.isin(times, inside)
    assert got["n_valid"] == 3
    assert np.isnan(got["pose"][~ok]).all() and np.isnan(got["cov"][~ok]).all()
    assert np.isfinite(got["pose"][ok]).all() and np.isfinite(got["cov"][ok]).all()
    empty = ctx.pose_covariance(np.zeros(0))
    assert empty["n_valid"] == 0 and empty["cov"].shape == (0, 6, 6)
    assert ctx.lib.ecb_pose_covariance(ctx.h, None, -1, None, None, None) == -2   # ECB_ERR_ARG


def test_pose_covariance_independent_of_batch(solved):
    """a time asked alone equals, bit for bit, the same time inside a shuffled batch of 10^6; a repeated call is identical; the
    device variant on torch tensors equals the host variant"""
    import torch
    ctx, knots = solved["ctx"], solved["knots"]
    rng = np.random.default_rng(3)
    lo, hi = min(k[0] for k in knots), max(k[-1] for k in knots)
    probe = np.r_[solved["kf_t"][:5], knots[0][4], knots[-1][-1]]
    batch = np.r_[rng.uniform(lo - 0.01, hi + 0.01, 1_000_000 - len(probe)), probe]
    perm = rng.permutation(len(batch))
    batch = batch[perm]
    where = np.argsort(perm)[-len(probe):]
    big = ctx.pose_covariance(batch)
    for k, u in enumerate(probe):
        one = ctx.pose_covariance([u])
        np.testing.assert_array_equal(one["pose"][0], big["pose"][where[k]])
        np.testing.assert_array_equal(one["cov"][0], big["cov"][where[k]])
    again = ctx.pose_covariance(batch)
    np.testing.assert_array_equal(again["cov"], big["cov"])
    np.testing.assert_array_equal(again["pose"], big["pose"])
    assert again["n_valid"] == big["n_valid"]
    dt = torch.from_numpy(batch).cuda()
    dp = torch.empty((len(batch), 7), dtype=torch.float64, device="cuda")
    dc = torch.empty((len(batch), 36), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    nv = ctx.pose_covariance_device(dt.data_ptr(), len(batch), dp.data_ptr(), dc.data_ptr())
    assert nv == big["n_valid"]
    np.testing.assert_array_equal(dp.cpu().numpy(), big["pose"])
    np.testing.assert_array_equal(dc.cpu().numpy().reshape(-1, 6, 6), big["cov"])


def test_pose_covariance_state_errors():
    """ECB_ERR_STATE before any covariance, after a rank-deficient covariance, after a new ecb_cost_setup and after a
    rotation-model switch"""
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth, calib_problem
    ev = _stream(150000, 0.6)
    pb = calib_problem.build(ev, seed=2, intr_noise=0.02)
    n_cp = [pb["n_cp"]]
    x = (pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])
    ctx = ecb.Context(0)
    t = np.array([pb["knots"][4]])

    def state_error():
        with pytest.raises(ecb.EcbError) as e:
            ctx.pose_covariance(t)
        return e.value.code == ecb.ERR_STATE

    try:
        ctx.set_sensor(346, 260)
        ctx.load_events(synth.to_records(ev))
        assert state_error()   # before ecb_cost_setup
        ctx.cost_setup(n_cp, [pb["knots"]], pb["radius"], pb["huber"])
        ctx.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
        assert state_error()   # before any covariance
        assert ctx.covariance(n_cp, *x)["ok"]
        assert ctx.pose_covariance(t)["n_valid"] == 1
        # rank deficient: 4 consecutive spans without residuals (test_covariance_rank_deficient_and_deterministic)
        ei, ci = ctx.cost_association()
        obs = np.stack([ev["x"][ei], ev["y"][ei]], 1).astype(np.float64)
        lm = np.asarray(pb["landmarks"], np.float64)[ci]
        tt = ev["t"][ei].astype(np.float64)
        order = np.argsort(tt, kind="stable")
        obs, lm, tt = obs[order], lm[order], tt[order]
        c, kn = pb["n_cp"] // 2, np.asarray(pb["knots"])
        gap = (tt >= kn[c]) & (tt < kn[c + 4])
        ctx.cost_set_residuals(obs[~gap], lm[~gap], tt[~gap], np.zeros((~gap).sum(), np.int32))
        assert not ctx.covariance(n_cp, *x)["ok"]
        assert state_error()
        ctx.cost_set_residuals(obs, lm, tt, np.zeros(len(tt), np.int32))
        assert ctx.covariance(n_cp, *x)["ok"]
        assert ctx.pose_covariance(t)["n_valid"] == 1
        ctx.cost_set_rotation_model(1)   # the rotation tangent changed meaning
        assert state_error()
        ctx.cost_set_rotation_model(0)
        assert state_error()             # still: the covariance was taken before the switch
        assert ctx.covariance(n_cp, *x)["ok"]
        assert ctx.pose_covariance(t)["n_valid"] == 1
        ctx.cost_setup(n_cp, [pb["knots"]], pb["radius"], pb["huber"])   # new knots
        assert state_error()
    finally:
        ctx.close()


def test_pose_covariance_two_gpus():
    """the normal equations exchanged between two GPUs, ecb_covariance on each rank from the summed buffer: both ranks' pose
    covariances are bit-identical"""
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
        poses = [c.pose_covariance(times) for c in ranks]
    finally:
        for c, p, q in zip(ranks, bufs, outs):
            c.synchronize()
            c.device_free(p)
            c.device_free(q)
            c.close()
    assert poses[0]["n_valid"] == len(times)
    np.testing.assert_array_equal(poses[0]["cov"], poses[1]["cov"])
    np.testing.assert_array_equal(poses[0]["pose"], poses[1]["pose"])


def test_cli_writes_trajectory_covariance(tmp_path):
    """ECB_TRAJECTORY_COVARIANCE=1 (with ECB_COVARIANCE=1) on the stream of test_cli_writes_intrinsics_covariance:
    TrajectoryCovariance.txt has TrajectoryByEvent.txt's stamps line for line, symmetric positive semi-definite matrices, the
    sigma2 of IntrinsicsCovariance.txt; the switch alone computes the covariance itself and writes the same file"""
    from eventcalib_b200 import synth
    from test_host_cli import YAML, CLI, HOST
    import eventcalib_b200.build as b
    b.build()
    subprocess.check_call(["make", "-s", "-C", HOST])
    ev = synth.make_stream(2000000, 346, 260, t0=5.0, duration=1.0, seed=1001, return_truth=True, workers=4,
                           rot_amp=(0.35, 0.35, 0.3), orbit=True)
    synth.write_bin(str(tmp_path / "ev.bin"), ev)
    (tmp_path / "cfg.yaml").write_text(YAML.replace("fitCircle: 0", "fitCircle: 1"))

    def run(out, **env_extra):
        env = dict(os.environ, ECB_PIECES="4", ECB_NO_IMAGES="1", ECB_DEVICES="0", **env_extra)
        env.pop("ECB_DEVICE", None)
        r = subprocess.run([CLI, str(tmp_path / "cfg.yaml"), str(tmp_path / "ev.bin"), str(out)], capture_output=True, text=True,
                           stdin=subprocess.DEVNULL, timeout=600, env=env)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr
        return r.stdout

    both, alone = tmp_path / "both", tmp_path / "alone"
    run(both, ECB_COVARIANCE="1", ECB_TRAJECTORY_COVARIANCE="1")
    out_alone = run(alone, ECB_TRAJECTORY_COVARIANCE="1")
    assert "Intrinsics standard deviation:" not in out_alone and not (alone / "IntrinsicsCovariance.txt").exists()
    text = (both / "TrajectoryCovariance.txt").read_text()
    assert text == (alone / "TrajectoryCovariance.txt").read_text()
    lines = text.splitlines()
    head = [l for l in lines if l.startswith("#")]
    rows = [l.split() for l in lines if not l.startswith("#")]
    tum = [l.split() for l in (both / "TrajectoryByEvent.txt").read_text().splitlines()]
    assert len(rows) == len(tum) > 10
    assert [r[0] for r in rows] == [t[0] for t in tum]
    sigma2 = float(head[-1].split("=")[-1])
    icov = [l for l in (both / "IntrinsicsCovariance.txt").read_text().splitlines() if not l.startswith("#")]
    assert sigma2 == float(icov[0]) > 0
    S = np.array([[float(v) for v in r[1:]] for r in rows]).reshape(-1, 6, 6)
    np.testing.assert_array_equal(S, np.transpose(S, (0, 2, 1)))
    ev_ = np.linalg.eigvalsh(S)
    assert (ev_[:, 0] >= -1e-12 * ev_[:, -1]).all() and (ev_[:, -1] > 0).all()
