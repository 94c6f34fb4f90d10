"""ecb_covariance on the GPU: the selected inverse of the Jacobi-equilibrated normal equations against a dense inverse of the
same (assembled GPU) normal equations, both rotation models, two segments, rank deficiency, determinism, two GPUs, and the CLI's
ECB_COVARIANCE=1 output."""
import os
import subprocess

import numpy as np
import pytest

import lm_oracle

pytestmark = pytest.mark.gpu
NB, NI = 24, 9


def _stream(n_events, duration):
    from eventcalib_b200 import synth
    return synth.make_stream(n_events, 346, 260, t0=5.0, duration=duration, seed=1004, return_truth=True,
                             rot_amp=(0.35, 0.35, 0.25), dist=92.0)


def _load(ctx, ev, n_cp, knots, pb):
    from eventcalib_b200 import synth
    ctx.set_sensor(346, 260)
    ctx.load_events(synth.to_records(ev))
    ctx.cost_setup(n_cp, knots, pb["radius"], pb["huber"])


def _dense(ctx, n_cp, x):
    """H assembled from the GPU's packed normal equations at x, intrinsics last; S; the scaled inverse M^-1 = S^-1 Z S^-1"""
    cost, Hs, gs = ctx.cost_normal_eq(*x)
    maps, C = lm_oracle._index_map(n_cp)
    D = 9 + 6 * C
    A, _ = lm_oracle.assemble(Hs, gs, maps, D)
    perm = np.r_[9:D, 0:9]
    H = A[np.ix_(perm, perm)]
    d = np.diag(H)
    s = np.where(d > 0, 1.0 / np.sqrt(np.where(d > 0, d, 1.0)), 1.0)
    M = H * s[:, None] * s[None, :]
    return cost, s, M, np.linalg.inv(M)


def _compare(cov, n_cp, s, Minv, bound=1e-8):
    """every returned entry against the dense inverse, in the scaled space: max |S^-1 dZ S^-1| <= bound max |S^-1 Z S^-1|"""
    n = 6 * sum(n_cp)
    seg_of = np.repeat(np.arange(len(n_cp)), [6 * c for c in n_cp])
    ref_b = np.zeros((n, NB))
    got_b = np.zeros((n, NB))
    for r in range(NB):
        j = np.arange(n - r)
        same = seg_of[j] == seg_of[j + r]
        ref_b[j, r] = np.where(same, Minv[j + r, j], 0.0)
        got_b[j, r] = cov["cov_band"][j, r] / (s[j] * s[j + r])
        # entries across segments and past the end are exactly 0
        assert not cov["cov_band"][j[~same], r].any() and not cov["cov_band"][n - r:, r].any()
    got_x = cov["cov_cross"] / (s[n:, None] * s[None, :n])
    got_c = cov["cov_intrinsics"] / (s[n:, None] * s[None, n:])
    scale = max(np.abs(ref_b).max(), np.abs(Minv[n:, :n]).max(), np.abs(Minv[n:, n:]).max())
    err = max(np.abs(got_b - ref_b).max(), np.abs(got_x - Minv[n:, :n]).max(), np.abs(got_c - Minv[n:, n:]).max())
    assert err <= bound * scale, (err, scale)
    np.testing.assert_array_equal(cov["cov_intrinsics"], cov["cov_intrinsics"].T)


@pytest.mark.parametrize("so3", [0, 1])
def test_covariance_matches_dense_inverse(ctx, so3):
    import eventcalib_b200 as ecb
    from eventcalib_b200 import calib_problem
    ev = _stream(150000, 0.6) if so3 == 0 else _stream(100000, 0.4)
    pb = calib_problem.build(ev, seed=2, intr_noise=0.02)
    rot0 = pb["rot_cp"].reshape(-1, 4)
    rot0 = rot0 / np.linalg.norm(rot0, axis=1, keepdims=True)
    n_cp = [pb["n_cp"]]
    _load(ctx, ev, n_cp, [pb["knots"]], pb)
    ctx.cost_set_rotation_model(so3)
    try:
        ctx.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
        i, r, t, summ, _ = ctx.calibrate(n_cp, pb["intrinsics"], rot0, pb["trans_cp"],
                                         ecb.lm_options(max_iterations=20 if so3 == 0 else 12, rotation_model=so3))
        x = (i, r, t)
        cov = ctx.covariance(n_cp, *x)
        cost, s, M, Minv = _dense(ctx, n_cp, x)
        c_eval = ctx.cost_eval(*x)
        m = ctx.cost_layout()["n_residuals"]
    finally:
        ctx.cost_set_rotation_model(0)
    assert cov["ok"] and cov["deficient_index"] == -1
    assert np.linalg.cond(M) < 1e8   # so that the bound below says something
    _compare(cov, n_cp, s, Minv)
    D = 9 + 6 * sum(n_cp)
    assert cov["dimension"] == D and cov["n_residuals"] == m
    assert cov["cost"] == cost and abs(cov["cost"] - c_eval) <= 1e-9 * c_eval
    assert cov["sigma2"] == pytest.approx(2 * cost / (m - D), rel=1e-15)
    assert 1e-12 < cov["min_relative_pivot"] <= 1.0 + 1e-12
    std = cov["std_intrinsics"]
    assert np.all(np.isfinite(std)) and np.all(std > 0)
    np.testing.assert_allclose(std, np.sqrt(cov["sigma2"] * np.diag(cov["cov_intrinsics"])), rtol=1e-15)
    # the 6 x 6 block of a control point from the band helper equals the dense one
    c = len(r) // 2
    blk = ecb.control_point_covariance(cov, c)
    ref = Minv[6 * c:6 * c + 6, 6 * c:6 * c + 6] * s[6 * c:6 * c + 6, None] * s[None, 6 * c:6 * c + 6]
    assert np.abs(blk - ref).max() <= 1e-7 * np.abs(ref).max()


def test_covariance_two_segments(ctx):
    """the two-segment problem of test_device_lm_two_segments_and_convergence: one selected-inversion CTA per segment, band
    entries across the segments 0, the corner (the intrinsics' covariance) summed over both"""
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth, calib_problem
    ev = synth.make_stream(160000, 346, 260, t0=5.0, duration=0.64, seed=1004, return_truth=True, rot_amp=(0.35, 0.35, 0.25), dist=92.0)
    cam, traj, board = ev["camera"], ev["trajectory"], ev["board"]
    a = calib_problem.build_from_truth(cam, traj, board, 5.0, 5.30, seed=1)
    b = calib_problem.build_from_truth(cam, traj, board, 5.34, 5.64, seed=2)
    n_cp = [a["n_cp"], b["n_cp"]]
    _load(ctx, ev, n_cp, [a["knots"], b["knots"]], a)
    ctx.cost_associate(np.concatenate([a["kf_t"], b["kf_t"]]), np.concatenate([a["circles"], b["circles"]]), a["landmarks"], a["step"])
    i, r, t, _, _ = ctx.calibrate(n_cp, a["intrinsics"], np.concatenate([a["rot_cp"], b["rot_cp"]]),
                                  np.concatenate([a["trans_cp"], b["trans_cp"]]), ecb.lm_options(max_iterations=50))
    cov = ctx.covariance(n_cp, i, r, t)
    _, s, M, Minv = _dense(ctx, n_cp, (i, r, t))
    assert cov["ok"]
    _compare(cov, n_cp, s, Minv)
    n0 = 6 * n_cp[0]
    for j in range(n0 - NB + 1, n0):
        assert not cov["cov_band"][j, n0 - j:].any()
    np.testing.assert_allclose(cov["cov_intrinsics"], Minv[-9:, -9:] * s[-9:, None] * s[None, -9:], rtol=1e-7,
                               atol=1e-9 * np.abs(cov["cov_intrinsics"]).max())


def test_covariance_rank_deficient_and_deterministic(ctx):
    """explicit residuals with 4 consecutive spans left empty: the control point they share has no residuals, its pivot is 0,
    the call fails and names a row of that control point; the same residuals without the gap succeed, twice bit for bit"""
    from eventcalib_b200 import calib_problem
    ev = _stream(150000, 0.6)
    pb = calib_problem.build(ev, seed=2, intr_noise=0.02)
    n_cp = [pb["n_cp"]]
    _load(ctx, ev, n_cp, [pb["knots"]], pb)
    ctx.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
    ei, ci = ctx.cost_association()
    obs = np.stack([ev["x"][ei], ev["y"][ei]], 1).astype(np.float64)
    lm = np.asarray(pb["landmarks"], np.float64)[ci]
    tt = ev["t"][ei].astype(np.float64)
    order = np.argsort(tt, kind="stable")
    obs, lm, tt = obs[order], lm[order], tt[order]
    x = (pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])
    c = pb["n_cp"] // 2
    kn = np.asarray(pb["knots"])
    gap = (tt >= kn[c]) & (tt < kn[c + 4])    # spans c-3 .. c: every span control point c takes part in
    assert gap.sum() > 0 and (~gap).sum() > 0
    ctx.cost_set_residuals(obs[~gap], lm[~gap], tt[~gap], np.zeros((~gap).sum(), np.int32))
    bad = ctx.covariance(n_cp, *x)
    assert not bad["ok"] and 6 * c <= bad["deficient_index"] < 6 * c + 6, (bad["deficient_index"], c)
    assert "cov_band" not in bad and bad["min_relative_pivot"] == 0.0
    ctx.cost_set_residuals(obs, lm, tt, np.zeros(len(tt), np.int32))
    one = ctx.covariance(n_cp, *x)
    two = ctx.covariance(n_cp, *x)
    assert one["ok"] and one["deficient_index"] == -1
    for k in ("cov_intrinsics", "cov_band", "cov_cross"):
        np.testing.assert_array_equal(one[k], two[k])
    assert one["sigma2"] == two["sigma2"] and one["min_relative_pivot"] == two["min_relative_pivot"]


def test_covariance_two_gpus_from_exchanged_normal_equations():
    """the events split over two GPUs, the normal equations summed by the exchange into a device buffer on each, ecb_covariance
    on that buffer: both ranks bit-identical, equal to the one-GPU result within the bound of the dense comparison"""
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
    one = ecb.Context(0)
    one.set_sensor(346, 260)
    one.load_events(rec)
    one.cost_setup(n_cp, [pb["knots"]], pb["radius"], pb["huber"])
    one.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
    ref = one.covariance(n_cp, *x)
    _, s, _, _ = _dense(one, n_cp, x)
    one.close()
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
        for r, c in enumerate(ranks):   # enqueued on both devices before either waits
            c.cost_normal_eq_exchange(*x, r, bufs, 1, outs[r], want_cost=False)
        covs = [c.covariance(n_cp, *x, d_packed=outs[r], n_residuals_total=m) for r, c in enumerate(ranks)]
    finally:
        for c, p, q in zip(ranks, bufs, outs):
            c.synchronize()
            c.device_free(p)
            c.device_free(q)
            c.close()
    assert covs[0]["ok"] and covs[1]["ok"]
    for k in ("cov_intrinsics", "cov_band", "cov_cross", "sigma2", "cost", "min_relative_pivot"):
        np.testing.assert_array_equal(covs[0][k], covs[1][k])
    assert covs[0]["n_residuals"] == ref["n_residuals"] == m
    nn = 6 * sum(n_cp)
    sb = s[:nn, None] * np.array([[s[j + r] if j + r < nn else 1.0 for r in range(NB)] for j in range(nn)])
    parts = [(covs[0]["cov_band"] / sb, ref["cov_band"] / sb),
             (covs[0]["cov_cross"] / (s[nn:, None] * s[None, :nn]), ref["cov_cross"] / (s[nn:, None] * s[None, :nn])),
             (covs[0]["cov_intrinsics"] / (s[nn:, None] * s[None, nn:]), ref["cov_intrinsics"] / (s[nn:, None] * s[None, nn:]))]
    scale = max(np.abs(b).max() for _, b in parts)
    assert max(np.abs(a - b).max() for a, b in parts) <= 1e-8 * scale


def test_cli_writes_intrinsics_covariance(tmp_path):
    """ECB_COVARIANCE=1 on the stream of test_cli_end_to_end_calibration: IntrinsicsCovariance.txt holds sigma2, a symmetric
    positive definite 9 x 9 Z and the standard deviations, which the extra stdout line repeats"""
    from eventcalib_b200 import synth
    from test_host_cli import YAML, CLI, HOST
    import eventcalib_b200.build as b
    b.build()
    subprocess.check_call(["make", "-s", "-C", HOST])
    ev = synth.make_stream(2000000, 346, 260, t0=5.0, duration=1.0, seed=1001, return_truth=True, workers=4,
                           rot_amp=(0.35, 0.35, 0.3), orbit=True)
    synth.write_bin(str(tmp_path / "ev.bin"), ev)
    (tmp_path / "cfg.yaml").write_text(YAML.replace("fitCircle: 0", "fitCircle: 1"))
    save = tmp_path / "out"

    def run(devices, out):
        env = dict(os.environ, ECB_PIECES="4", ECB_COVARIANCE="1", ECB_NO_IMAGES="1", ECB_DEVICES=devices)
        env.pop("ECB_DEVICE", None)
        r = subprocess.run([CLI, str(tmp_path / "cfg.yaml"), str(tmp_path / "ev.bin"), str(out)], capture_output=True, text=True,
                           stdin=subprocess.DEVNULL, timeout=600, env=env)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr
        lines = r.stdout.splitlines()
        k = [n for n, l in enumerate(lines) if l.startswith("Intrinsics after optimization:")][0]
        assert lines[k + 1].startswith("Intrinsics standard deviation:")
        return np.array(lines[k + 1].split(":")[1].split(), float)

    std_out = run("0", save)
    rows = [l.split() for l in (save / "IntrinsicsCovariance.txt").read_text().splitlines() if not l.startswith("#")]
    assert [len(v) for v in rows] == [1] + [9] * 9 + [9]
    sigma2 = float(rows[0][0])
    Z = np.array(rows[1:10], float)
    std = np.array(rows[10], float)
    assert sigma2 > 0
    np.testing.assert_array_equal(Z, Z.T)
    assert np.linalg.eigvalsh(Z).min() > 0
    np.testing.assert_allclose(std, np.sqrt(sigma2 * np.diag(Z)), rtol=1e-12)
    np.testing.assert_allclose(std_out, std, rtol=1e-9)
    import torch
    if torch.cuda.device_count() >= 2:   # two shards: normal equations exchanged, every shard inverts the sum
        np.testing.assert_allclose(run("0,1", tmp_path / "out2"), std_out, rtol=1e-6)
