"""Constant intrinsics on the GPU (ecb_cost_set_constant_intrinsics): the host LM loop (ecb_calibrate) against the reduced dense
restatement of tests/test_constant_intrinsics_lm.py driven by the oracle, the device LM against the host state machine, the
covariance against a dense inverse of the GPU normal equations with the constant rows and columns deleted, the pose covariance
from that Z, the default (mask 0) bit for bit, two GPUs, and the CLI's ECB_CONSTANT_INTRINSICS."""
import os
import subprocess

import numpy as np
import pytest

import lm_oracle
from test_constant_intrinsics_lm import assert_matches_reduced, solve_reduced

K345 = 0b111000000
NB = 24


def _stream(n_events, duration):
    from eventcalib_b200 import synth
    return synth.make_stream(n_events, 346, 260, t0=5.0, duration=duration, seed=1004, return_truth=True,
                             rot_amp=(0.35, 0.35, 0.25), dist=92.0)


def _problem(layout):
    """(ev, n_cp, knots, pb of the first segment, rot0, trans0, kf_t, circles): the problems of test_gpu_calibrate.py /
    test_gpu_covariance.py — one segment (quaternion or SO(3) sizes) or the two-segment one"""
    from eventcalib_b200 import calib_problem
    if layout == "two":
        ev = _stream(160000, 0.64)
        a = calib_problem.build_from_truth(ev["camera"], ev["trajectory"], ev["board"], 5.0, 5.30, seed=1)
        b = calib_problem.build_from_truth(ev["camera"], ev["trajectory"], ev["board"], 5.34, 5.64, seed=2)
        pbs = [a, b]
    else:
        ev = _stream(150000, 0.6) if layout == "quat" else _stream(100000, 0.4)
        pbs = [calib_problem.build(ev, seed=2, intr_noise=0.02)]
    a = pbs[0]
    rot0 = np.concatenate([p["rot_cp"] for p in pbs]).reshape(-1, 4)
    rot0 = rot0 / np.linalg.norm(rot0, axis=1, keepdims=True)
    return dict(ev=ev, n_cp=[p["n_cp"] for p in pbs], knots=[np.asarray(p["knots"], np.float64) for p in pbs], pb=a, rot0=rot0,
                trans0=np.concatenate([p["trans_cp"] for p in pbs]).reshape(-1, 3), kf_t=np.concatenate([p["kf_t"] for p in pbs]),
                circles=np.concatenate([p["circles"] for p in pbs]))


def _context(pr, so3=0, mask_names=None, device=0, records=None):
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth
    ctx = ecb.Context(device)
    if mask_names is not None:
        ctx.set_constant_intrinsics(mask_names)   # a property of the context: set before cost_setup, it survives it
    ctx.set_sensor(346, 260)
    ctx.load_events(synth.to_records(pr["ev"]) if records is None else records)
    a = pr["pb"]
    ctx.cost_setup(pr["n_cp"], pr["knots"], a["radius"], a["huber"])
    ctx.cost_set_rotation_model(so3)
    ctx.cost_associate(pr["kf_t"], pr["circles"], a["landmarks"], a["step"])
    return ctx


def _names(mask):
    import eventcalib_b200 as ecb
    return [nm for i, nm in enumerate(ecb.INTRINSIC_NAMES) if (mask >> i) & 1]


def _const(mask):
    return np.array([(mask >> i) & 1 for i in range(9)], bool)


@pytest.mark.gpu
def test_calibrate_with_constant_intrinsics_matches_reduced_restatement(oracle_mod):
    """ecb_calibrate (GPU evaluations, host solve) with k3 k4 k5 constant against the reduced dense restatement driven by the
    oracle on the problem of test_calibrate_matches_oracle_lm"""
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth, calib_problem
    ev = _stream(150000, 0.6)
    pb = calib_problem.build(ev, seed=2, intr_noise=0.02)
    ctx = ecb.Context(0)
    try:
        ctx.set_sensor(346, 260)
        ctx.load_events(synth.to_records(ev))
        ctx.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
        ctx.set_constant_intrinsics(["k3", "k4", "k5"])
        n = ctx.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
        P = oracle_mod.CostProblem([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
        P.associate(ev["t"], ev["x"], ev["y"], pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
        assert n == P.n_residuals
        K = 20
        i1, r1, t1, summ, tr1 = ctx.calibrate([pb["n_cp"]], pb["intrinsics"], pb["rot_cp"], pb["trans_cp"],
                                              ecb.lm_options(max_iterations=K))
    finally:
        ctx.close()
    i2, r2, t2, tr2, _ = solve_reduced(P, [pb["n_cp"]], pb["intrinsics"], pb["rot_cp"], pb["trans_cp"], K345, max_iterations=K)
    assert_matches_reduced(tr1, i1, r1, t1, tr2, i2, r2, t2, pb["intrinsics"], K345)
    assert summ["final_cost"] < summ["initial_cost"]


@pytest.mark.gpu
@pytest.mark.parametrize("so3,layout", [(0, "quat"), (1, "so3"), (0, "two"), (1, "two")])
def test_device_lm_with_constant_intrinsics_matches_host(so3, layout):
    """the device LM against the host state machine, k3 k4 k5 constant, run to termination: the criteria of
    test_device_lm_matches_host_state_machine, and the constant intrinsics == their start values on both loops"""
    import eventcalib_b200 as ecb
    pr = _problem(layout)
    intr0 = pr["pb"]["intrinsics"]
    ctx = _context(pr, so3, ["k3", "k4", "k5"])
    try:
        opt = ecb.lm_options(max_iterations=50, rotation_model=so3)
        i1, r1, t1, s1, tr1 = ctx.calibrate(pr["n_cp"], intr0, pr["rot0"], pr["trans0"], opt)
        lm = ecb.DeviceLm(ctx, pr["n_cp"], opt)
        out = lm.run(intr0, pr["rot0"], pr["trans0"])
        lm.close()
    finally:
        ctx.close()
    c = _const(K345)
    np.testing.assert_array_equal(i1[c], intr0[c])
    np.testing.assert_array_equal(out["intrinsics"][c], intr0[c])
    assert s1["termination"] != 7
    tr2 = out["trace"]
    assert len(tr1) == len(tr2) and out["iterations"] == s1["iterations"] and out["successful_steps"] == s1["successful_steps"]
    assert out["termination"] == s1["termination"]
    np.testing.assert_array_equal(tr1[:, 3], tr2[:, 3])
    np.testing.assert_allclose(tr1[:, 0], tr2[:, 0], rtol=1e-9)
    np.testing.assert_allclose(tr1[:, 2], tr2[:, 2], rtol=1e-6)
    np.testing.assert_allclose(out["intrinsics"], i1, rtol=1e-9)
    np.testing.assert_allclose(out["rot_cp"], r1.reshape(-1, 4), rtol=0, atol=1e-9)
    np.testing.assert_allclose(out["trans_cp"], t1.reshape(-1, 3), rtol=1e-9, atol=1e-9)
    assert out["final_cost"] < out["initial_cost"]


@pytest.mark.gpu
def test_device_lm_all_intrinsics_constant():
    """known intrinsics: only the trajectory is fitted; the intrinsics come back unchanged and the cost still decreases"""
    import eventcalib_b200 as ecb
    pr = _problem("quat")
    intr0 = pr["pb"]["intrinsics"]
    ctx = _context(pr, 0, list(ecb.INTRINSIC_NAMES))
    try:
        lm = ecb.DeviceLm(ctx, pr["n_cp"], ecb.lm_options(max_iterations=20))
        out = lm.run(intr0, pr["rot0"], pr["trans0"])
        lm.close()
        i1, _, _, s1, _ = ctx.calibrate(pr["n_cp"], intr0, pr["rot0"], pr["trans0"], ecb.lm_options(max_iterations=20))
    finally:
        ctx.close()
    np.testing.assert_array_equal(out["intrinsics"], intr0)
    np.testing.assert_array_equal(i1, intr0)
    assert out["final_cost"] < out["initial_cost"] and s1["final_cost"] < s1["initial_cost"]


@pytest.mark.gpu
def test_zero_mask_is_bit_identical_to_the_default():
    """a context that set k3 k4 k5 and then cleared the mask against a fresh one: ecb_calibrate, DeviceLm and ecb_covariance
    bit for bit"""
    import eventcalib_b200 as ecb
    pr = _problem("quat")
    intr0 = pr["pb"]["intrinsics"]
    opt = ecb.lm_options(max_iterations=12)
    res = []
    for names in (None, ["k3", "k4", "k5"]):
        ctx = _context(pr, 0, names)
        try:
            if names:
                ctx.set_constant_intrinsics([])
            cal = ctx.calibrate(pr["n_cp"], intr0, pr["rot0"], pr["trans0"], opt)
            lm = ecb.DeviceLm(ctx, pr["n_cp"], opt)
            dev = lm.run(intr0, pr["rot0"], pr["trans0"])
            lm.close()
            cov = ctx.covariance(pr["n_cp"], *cal[:3])
        finally:
            ctx.close()
        res.append((cal, dev, cov))
    (c0, d0, v0), (c1, d1, v1) = res
    for a, b in zip(c0[:3] + (c0[4],), c1[:3] + (c1[4],)):
        np.testing.assert_array_equal(a, b)
    assert c0[3] == c1[3]
    for k in ("intrinsics", "rot_cp", "trans_cp", "trace", "final_cost", "iterations"):
        np.testing.assert_array_equal(d0[k], d1[k])
    assert v0["ok"] and v1["ok"]
    for k in ("cov_intrinsics", "cov_band", "cov_cross", "sigma2", "min_relative_pivot", "dimension"):
        np.testing.assert_array_equal(v0[k], v1[k])


def _dense_reduced(ctx, n_cp, x, mask):
    """the GPU's assembled normal equations at x (control points first, intrinsics last) with the constant intrinsics' rows and
    columns deleted, equilibrated: returns s and the scaled inverse, both scattered back to D with 1 / 0 at the constant ones"""
    cost, Hs, gs = ctx.cost_normal_eq(*x)
    maps, C = lm_oracle._index_map(n_cp)
    D = 9 + 6 * C
    A, _ = lm_oracle.assemble(Hs, gs, maps, D)
    perm = np.r_[9:D, 0:9]
    H = A[np.ix_(perm, perm)]
    keep = np.r_[np.ones(D - 9, bool), ~_const(mask)]
    Hr = H[np.ix_(keep, keep)]
    sr = 1.0 / np.sqrt(np.diag(Hr))
    Mr = Hr * sr[:, None] * sr[None, :]
    assert np.linalg.cond(Mr) < 1e8   # so that the bound of the comparison says something
    s = np.ones(D)
    s[keep] = sr
    Minv = np.zeros((D, D))
    Minv[np.ix_(keep, keep)] = np.linalg.inv(Mr)
    return cost, s, Minv


def _calibrated(pr, so3, mask, iters):
    """a context with the mask set and the problem calibrated with it (the iteration counts of test_gpu_covariance.py)"""
    import eventcalib_b200 as ecb
    ctx = _context(pr, so3, _names(mask))
    i, r, t, _, _ = ctx.calibrate(pr["n_cp"], pr["pb"]["intrinsics"], pr["rot0"], pr["trans0"],
                                  ecb.lm_options(max_iterations=iters, rotation_model=so3))
    return ctx, (i, np.asarray(r).reshape(-1, 4), np.asarray(t).reshape(-1, 3))


@pytest.mark.gpu
@pytest.mark.parametrize("so3,layout,iters", [(0, "quat", 20), (1, "so3", 12), (0, "two", 50)])
def test_covariance_with_constant_intrinsics_matches_reduced_dense_inverse(so3, layout, iters):
    from test_gpu_covariance import _compare
    pr = _problem(layout)
    ctx, x = _calibrated(pr, so3, K345, iters)
    try:
        cov = ctx.covariance(pr["n_cp"], *x)
        again = ctx.covariance(pr["n_cp"], *x)
        cost, s, Minv = _dense_reduced(ctx, pr["n_cp"], x, K345)
        m = ctx.cost_layout()["n_residuals"]
        if layout == "quat":   # the measured values DESIGN.md §5 quotes (printed, not asserted): with and without k3 k4 k5
            ctx.set_constant_intrinsics([])
            free = ctx.covariance(pr["n_cp"], *x)
            ctx.set_constant_intrinsics(["k3", "k4", "k5"])
            for tag, c in (("all free", free), ("k3 k4 k5 constant", cov)):
                print("\n[constant intrinsics] %s: sigma(k1) %.6g sigma(k2) %.6g min_relative_pivot %.6g sigma(fx) %.6g" % (
                    tag, c["std_intrinsics"][4], c["std_intrinsics"][5], c["min_relative_pivot"], c["std_intrinsics"][0]))
    finally:
        ctx.close()
    assert cov["ok"] and cov["deficient_index"] == -1
    _compare(cov, pr["n_cp"], s, Minv)
    c = _const(K345)
    assert not cov["cov_intrinsics"][c].any() and not cov["cov_intrinsics"][:, c].any() and not cov["cov_cross"][c].any()
    assert not np.signbit(cov["cov_intrinsics"][c]).any() and not np.signbit(cov["cov_cross"][c]).any()   # +0.0 exactly
    np.testing.assert_array_equal(cov["std_intrinsics"][c], 0.0)
    D = 9 + 6 * sum(pr["n_cp"])
    assert cov["dimension"] == D - 3 and cov["n_residuals"] == m and cov["cost"] == cost
    assert cov["sigma2"] == pytest.approx(2 * cost / (m - (D - 3)), rel=1e-15)
    assert 1e-12 < cov["min_relative_pivot"] <= 1.0 + 1e-12
    for k in ("cov_intrinsics", "cov_band", "cov_cross", "sigma2", "min_relative_pivot"):
        np.testing.assert_array_equal(cov[k], again[k])


@pytest.mark.gpu
def test_pose_covariance_after_masked_covariance():
    """Sigma = J Z'_blk J^T at the key-frame stamps with Z' the reduced dense inverse; ECB_ERR_STATE once the mask changes"""
    import eventcalib_b200 as ecb
    from test_gpu_pose_covariance import _host_libs, _reference
    pr = _problem("quat")
    ctx, x = _calibrated(pr, 0, K345, 20)
    try:
        assert ctx.covariance(pr["n_cp"], *x)["ok"]
        _, s, Minv = _dense_reduced(ctx, pr["n_cp"], x, K345)
        got = ctx.pose_covariance(pr["kf_t"])
        ctx.set_constant_intrinsics(["k3", "k4", "k5"])   # the same mask again: Z still holds
        assert ctx.pose_covariance(pr["kf_t"][:3])["n_valid"] >= 0
        ctx.set_constant_intrinsics(["k4", "k5"])
        with pytest.raises(ecb.EcbError) as e:
            ctx.pose_covariance(pr["kf_t"][:3])
        assert e.value.code == ecb.ERR_STATE
    finally:
        ctx.close()
    lib, fac = _host_libs()
    solved = dict(so3=0, n_cp=pr["n_cp"], knots=pr["knots"], x=x, Z=Minv * s[:, None] * s[None, :])
    ref = _reference(solved, lib, fac, pr["kf_t"])
    valid = np.array([r is not None for r in ref])
    assert valid.sum() > len(valid) // 2 and got["n_valid"] == valid.sum()
    S, Sr = got["cov"][valid], np.array([r[1] for r in ref if r is not None])
    assert np.abs(S - Sr).max() <= 1e-7 * np.abs(Sr).max(), np.abs(S - Sr).max() / np.abs(Sr).max()


@pytest.mark.gpu
def test_two_gpus_with_constant_intrinsics():
    """device LM and covariance with k3 k4 k5 constant over two GPUs: ranks bit-identical, equal to one GPU to 1e-9"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth
    pr = _problem("quat")
    rec = synth.to_records(pr["ev"])
    n = len(rec)
    K = 10
    opt = ecb.lm_options(max_iterations=K, fixed_iterations=1)
    x0 = (pr["pb"]["intrinsics"], pr["rot0"], pr["trans0"])
    one = _context(pr, 0, ["k3", "k4", "k5"])
    try:
        lm1 = ecb.DeviceLm(one, pr["n_cp"], opt)
        ref = lm1.run(*x0)
        lm1.close()
        x = (ref["intrinsics"], ref["rot_cp"], ref["trans_cp"])
        ref_cov = one.covariance(pr["n_cp"], *x)
    finally:
        one.close()
    ranks, lms = [], []
    for dev, (lo, hi) in enumerate(((0, n // 2 + 333), (n // 2 + 333, n))):
        c = _context(pr, 0, ["k3", "k4", "k5"], device=dev, records=rec[lo:hi])
        c.enable_peer_access(1 - dev)
        ranks.append(c)
    bufs = [c.device_alloc(c.exchange_buffer_bytes(2)) for c in ranks]        # the LM's exchange
    bufs_cov = [c.device_alloc(c.exchange_buffer_bytes(2)) for c in ranks]    # the covariance's (its epochs start at 1)
    outs_ne = [c.device_alloc(8 * c.cost_layout()["out_doubles"]) for c in ranks]
    m = sum(c.cost_layout()["n_residuals"] for c in ranks)
    try:
        for r, c in enumerate(ranks):
            lm = ecb.DeviceLm(c, pr["n_cp"], opt)
            lm.set_exchange(r, bufs)
            lms.append(lm)
        for lm in lms:
            lm.begin(*x0)
        for lm in lms:
            lm.iterate(K + 1)
        outs = [lm.result() for lm in lms]
        for r, c in enumerate(ranks):
            c.cost_normal_eq_exchange(*x, r, bufs_cov, 1, outs_ne[r], want_cost=False)
        covs = [c.covariance(pr["n_cp"], *x, d_packed=outs_ne[r], n_residuals_total=m) for r, c in enumerate(ranks)]
    finally:
        for lm in lms:
            lm.close()
        for c, p, p2, q in zip(ranks, bufs, bufs_cov, outs_ne):
            c.synchronize()
            for ptr in (p, p2, q):
                c.device_free(ptr)
            c.close()
    for k in ("intrinsics", "rot_cp", "trans_cp", "trace"):
        np.testing.assert_array_equal(outs[0][k], outs[1][k])
    np.testing.assert_array_equal(outs[0]["intrinsics"][_const(K345)], x0[0][_const(K345)])
    np.testing.assert_array_equal(outs[0]["trace"][:, 3], ref["trace"][:, 3])
    np.testing.assert_allclose(outs[0]["trace"][:, 0], ref["trace"][:, 0], rtol=1e-9)
    np.testing.assert_allclose(outs[0]["intrinsics"], ref["intrinsics"], rtol=1e-9)
    assert covs[0]["ok"] and covs[1]["ok"] and covs[0]["dimension"] == ref_cov["dimension"]
    for k in ("cov_intrinsics", "cov_band", "cov_cross", "sigma2", "cost", "min_relative_pivot"):
        np.testing.assert_array_equal(covs[0][k], covs[1][k])
    d = np.sqrt(np.diag(ref_cov["cov_intrinsics"]))
    d = np.where(d > 0, d, 1.0)
    np.testing.assert_allclose(covs[0]["cov_intrinsics"] / np.outer(d, d), ref_cov["cov_intrinsics"] / np.outer(d, d), rtol=0,
                               atol=1e-9)
    assert not covs[0]["cov_intrinsics"][_const(K345)].any()


def _cli(tmp_path, env_extra, cfg=None, ev=None):
    from test_host_cli import CLI
    env = dict(os.environ, ECB_PIECES="4", ECB_NO_IMAGES="1", ECB_DEVICES="0", **env_extra)
    env.pop("ECB_DEVICE", None)
    return subprocess.run([CLI, str(cfg or tmp_path / "cfg.yaml"), str(ev or tmp_path / "ev.bin"), str(tmp_path / "out")],
                          capture_output=True, text=True, stdin=subprocess.DEVNULL, timeout=600, env=env)


def test_cli_refuses_unknown_names_and_reference_signatures(tmp_path):
    """before any file or GPU work: an unknown name, or the switch together with ECB_REFERENCE_SIGNATURES, exits with 1"""
    from test_host_cli import HOST
    subprocess.check_call(["make", "-s", "-C", HOST])
    r = _cli(tmp_path, {"ECB_CONSTANT_INTRINSICS": "k3,kappa,k5"})
    assert r.returncode == 1 and "kappa" in r.stderr, r.stderr
    r = _cli(tmp_path, {"ECB_CONSTANT_INTRINSICS": "k3", "ECB_REFERENCE_SIGNATURES": "1"})
    assert r.returncode == 1 and "ECB_REFERENCE_SIGNATURES" in r.stderr, r.stderr


@pytest.mark.gpu
def test_cli_constant_intrinsics_with_covariance(tmp_path):
    """ECB_CONSTANT_INTRINSICS=k3,k4,k5 ECB_COVARIANCE=1 on the stream of test_cli_writes_intrinsics_covariance"""
    from eventcalib_b200 import synth
    from test_host_cli import YAML, HOST
    import eventcalib_b200.build as b
    b.build()
    subprocess.check_call(["make", "-s", "-C", HOST])
    ev = synth.make_stream(2000000, 346, 260, t0=5.0, duration=1.0, seed=1001, return_truth=True, workers=4,
                           rot_amp=(0.35, 0.35, 0.3), orbit=True)
    synth.write_bin(str(tmp_path / "ev.bin"), ev)
    (tmp_path / "cfg.yaml").write_text(YAML.replace("fitCircle: 0", "fitCircle: 1"))
    r = _cli(tmp_path, {"ECB_CONSTANT_INTRINSICS": "k3,k4,k5", "ECB_COVARIANCE": "1"})
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr
    lines = r.stdout.splitlines()
    ci = [l for l in lines if l.startswith("Constant intrinsics:")]
    assert len(ci) == 1
    tok = ci[0].split(":", 1)[1].split()
    assert tok[0::3] == ["k3", "k4", "k5"] and tok[1::3] == ["="] * 3
    const = np.array(tok[2::3], float)
    after = [l for l in lines if l.startswith("Intrinsics after optimization:")][0]
    intr = np.array(after.split(":", 1)[1].split(), float)
    assert lines.index(ci[0]) < lines.index(after)
    np.testing.assert_array_equal(intr[6:9], [float("%.12g" % v) for v in const])
    txt = (tmp_path / "out" / "IntrinsicsCovariance.txt").read_text().splitlines()
    rows = [l.split() for l in txt if not l.startswith("#")]
    assert [len(v) for v in rows] == [1] + [9] * 9 + [9]
    Z = np.array(rows[1:10], float)
    std = np.array(rows[10], float)
    assert not Z[6:].any() and not Z[:, 6:].any()
    np.testing.assert_array_equal(std[6:], 0.0)
    assert np.all(std[:6] > 0) and np.linalg.eigvalsh(Z[:6, :6]).min() > 0
    head = txt[0].split(",")   # "# sigma2 = 2 cost / (residuals - parameters), <m> residuals, <dimension> parameters"
    n_res, n_par = int(head[1].split()[0]), int(head[2].split()[0])
    assert n_par % 6 == 0 and n_par > 6 and n_res > n_par   # D - 3 with D = 6 C + 9 (without the switch: D, = 3 mod 6)
    assert float(rows[0][0]) > 0
