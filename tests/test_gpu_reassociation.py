"""Re-association at a calibrated point (ecb_cost_reassociate): the records against a numpy restatement (candidates, spline pose,
back-projection, nearest landmark, event-to-rim error), the counts, invariants, the interplay with rejection, the groupings, the
LM loops, shards, the error codes, the quality on a fast-motion stream with a known camera, and the CLI."""
import ctypes as C
import math

import numpy as np
import pytest

import lm_oracle
from test_gpu_reprojection import _numpy_e, _poses  # noqa: F401
from test_gpu_residuals import _nearest_kf, _read, _run_cli, _explicit_problem

pytestmark = pytest.mark.gpu

GATE = 5.0


def _same(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


@pytest.fixture(scope="module")
def prob():
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth, calib_problem
    ev = synth.make_stream(100000, 346, 260, t0=5.0, duration=0.3, seed=1004, return_truth=True)
    pb = calib_problem.build(ev, seed=3, kf_every=16 * 5e-4)   # key frames 16 steps apart: the 5-step window leaves gaps
    c = ecb.Context(0)
    c.set_sensor(346, 260)
    c.load_events(synth.to_records(ev))
    c.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    yield dict(ctx=c, ev=ev, pb=pb)
    c.close()


def _associate(c, pb):
    return c.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])


def _start(pb, so3):
    rot = pb["rot_cp"].reshape(-1, 4)
    rot = (rot / np.linalg.norm(rot, axis=1, keepdims=True)).ravel() if so3 else pb["rot_cp"]
    return (pb["intrinsics"], rot, pb["trans_cp"])


def _candidates(ev, pb, max_dt):
    """events in the segment and near their key frame (the association's window test when max_dt == 0)"""
    kn, kf, u = pb["knots"], pb["kf_t"], ev["t"]
    dt = u - kf[_nearest_kf(kf, u)]
    near = (dt * dt < 5 * pb["step"] * 5 * pb["step"]) if max_dt == 0 else (np.abs(dt) <= max_dt)
    return np.nonzero((u >= kn[0]) & (u <= kn[-1]) & near)[0]


def _numpy_reassoc(ev, pb, x, so3, oracle_mod, max_dt=0.0, gate=GATE):
    """(kept events, their circles, ambiguous events): the restated decision of every candidate; an event within 1e-9 relative
    of the gate or of a nearest-landmark tie is ambiguous"""
    intr = np.asarray(x[0], float)
    rot, trans = np.asarray(x[1]).reshape(-1, 4), np.asarray(x[2]).reshape(-1, 3)
    cand = _candidates(ev, pb, max_dt)
    n = len(cand)
    obs = np.stack([ev["x"][cand], ev["y"][cand]], 1).astype(float)
    tt = ev["t"][cand]
    N, c0 = np.zeros((n, 4)), np.zeros(n, np.int64)
    for k in range(n):
        s, N[k] = oracle_mod.basis(pb["knots"], tt[k])
        c0[k] = s - 3
    idx = c0[:, None] + np.arange(4)
    R, t = _poses(rot[idx], trans[idx], N, so3)
    xn, yn = (obs[:, 0] - intr[2]) / intr[0], (obs[:, 1] - intr[3]) / intr[1]
    r2 = xn * xn + yn * yn
    k5 = intr[4:]
    s = 1 + r2 * (k5[0] + r2 * (k5[1] + r2 * (k5[2] + r2 * (k5[3] + r2 * k5[4]))))
    Xr = R.apply(np.stack([xn * s, yn * s, np.ones(n)], 1))
    with np.errstate(divide="ignore", invalid="ignore"):
        Xw = (-t[:, 2] / Xr[:, 2])[:, None] * Xr + t
    L = pb["landmarks"]
    D = np.sqrt(((Xw[:, None, :] - L[None, :, :]) ** 2).sum(-1))
    ci = np.argmin(D, axis=1)
    d2 = np.sort(D, axis=1)[:, :2]
    tie = d2[:, 1] - d2[:, 0] <= 1e-9 * d2[:, 1]
    e, _, _ = _numpy_e(intr, x[1], x[2], [pb["knots"]], obs, L[ci], tt, np.zeros(n, np.int64), pb["radius"], so3, oracle_mod, [0])
    near_gate = np.abs(np.abs(e) - gate) <= 1e-9 * gate
    finite = np.isfinite(Xw).all(1)
    keep = finite & np.isfinite(e) & (np.abs(e) < gate)
    amb = cand[finite & (tie | near_gate)]
    return cand[keep], ci[keep], amb, cand


def _counts(ei0, ci0, ei, ci):
    prev = dict(zip(ei0.tolist(), ci0.tolist()))
    same = sum(1 for i, c in zip(ei.tolist(), ci.tolist()) if prev.get(i) == c)
    changed = sum(1 for i, c in zip(ei.tolist(), ci.tolist()) if i in prev and prev[i] != c)
    new = sum(1 for i in ei.tolist() if i not in prev)
    return len(ei), same, changed, new, len(ei0) - same - changed


@pytest.mark.parametrize("so3", [False, True])
def test_matches_numpy(prob, oracle_mod, so3):
    import eventcalib_b200 as ecb
    c, ev, pb = prob["ctx"], prob["ev"], prob["pb"]
    c.cost_set_rotation_model(int(so3))
    try:
        x0 = _start(pb, so3)
        _associate(c, pb)
        x1 = c.calibrate(pb["n_cp"], *x0, options=ecb.lm_options(max_iterations=8, rotation_model=int(so3)))[:3]
        window = 5 * pb["step"]
        for x, max_dt in ((x0, 0.0), (x1, 0.0), (x1, 2 * window)):
            _associate(c, pb)
            ei0, ci0 = c.cost_association()
            counts = c.reassociate(*x, max_dt=max_dt)
            ei, ci = c.cost_association()
            assert counts == _counts(ei0, ci0, ei, ci)
            assert c.cost_layout()["n_residuals"] == len(ei)
            ke, kc, amb, cand = _numpy_reassoc(ev, pb, x, so3, oracle_mod, max_dt)
            print("\nso3 %d max_dt %g: %d candidates, %d kept, %d ambiguous; counts %s" % (so3, max_dt, len(cand), len(ei), len(amb),
                                                                                       counts))
            assert len(amb) <= max(3, len(cand) // 10000)
            assert len(ei) > 0
            g_ok, n_ok = ~np.isin(ei, amb), ~np.isin(ke, amb)
            assert np.array_equal(ei[g_ok], ke[n_ok]) and np.array_equal(ci[g_ok], kc[n_ok])
            if len(amb) == 0:
                assert counts == _counts(ei0, ci0, ke, kc)
    finally:
        c.cost_set_rotation_model(0)


def test_invariants(prob):
    import eventcalib_b200 as ecb
    c, ev, pb = prob["ctx"], prob["ev"], prob["pb"]
    x0 = _start(pb, False)
    _associate(c, pb)
    x = c.calibrate(pb["n_cp"], *x0, options=ecb.lm_options(max_iterations=8))[:3]
    cand = _candidates(ev, pb, 0.0)
    sets = {}
    for max_dt in (0.0, 2 * 5 * pb["step"]):
        _associate(c, pb)
        n, *_ = c.reassociate(*x, max_dt=max_dt)
        ei, ci = c.cost_association()
        e, bad = c.reprojection_errors(*x)
        assert len(e) == n and bad == 0 and np.all(np.abs(e) < GATE)
        assert np.all(np.diff(ei) > 0)
        r1 = c.cost_residuals(*x)
        again = c.reassociate(*x, max_dt=max_dt)
        assert again == (n, n, 0, 0, 0)
        ei2, ci2 = c.cost_association()
        assert _same(ei, ei2) and _same(ci, ci2) and _same(r1, c.cost_residuals(*x))
        sets[max_dt] = set(ei.tolist())
    assert sets[0.0] <= set(cand.tolist())
    assert sets[0.0] <= sets[2 * 5 * pb["step"]] and len(sets[2 * 5 * pb["step"]]) > len(sets[0.0])


def test_interplay(prob, oracle_mod):
    """rejection undone, the groupings, ecb_calibrate against the dense LM restatement, a device LM created before the call"""
    import eventcalib_b200 as ecb
    c, ev, pb = prob["ctx"], prob["ev"], prob["pb"]
    kf = pb["kf_t"]
    x0 = _start(pb, False)
    _associate(c, pb)
    x = c.calibrate(pb["n_cp"], *x0, options=ecb.lm_options(max_iterations=8))[:3]
    n, *_ = c.reassociate(*x)
    ei, ci = c.cost_association()
    thr = float(np.quantile(np.abs(c.cost_residuals(*x)), 0.8))
    kept, removed = c.reject_residuals(*x, max_abs_r=thr, drop_keyframes=(np.arange(len(kf)) % 4 == 0), kf_t=kf)
    assert removed > 0 and kept + removed == n
    counts = c.reassociate(*x)
    assert counts == (n, kept, 0, removed, 0)
    e2, c2 = c.cost_association()
    assert _same(ei, e2) and _same(ci, c2)
    for by in ("keyframe", "circle", "sensor_cell"):
        groups, total = c.residual_groups(*x, by, kf_t=kf if by == "keyframe" else None)
        assert int(groups["count"].sum()) == int(total["count"]) == n
    # the LM on the new records against the dense restatement driven by the oracle given them explicitly
    P = oracle_mod.CostProblem([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    obs = np.stack([ev["x"][ei], ev["y"][ei]], 1).astype(float)
    P.set_residuals(obs, pb["landmarks"][ci], ev["t"][ei], np.zeros(len(ei), np.int32))
    K = 10
    i1, r1, t1, summ, tr1 = c.calibrate([pb["n_cp"]], *x, ecb.lm_options(max_iterations=K))
    i2, r2, t2, tr2, term = lm_oracle.solve(P, [pb["n_cp"]], *x, max_iterations=K)
    tr2 = np.array(tr2)
    assert len(tr1) == len(tr2)
    np.testing.assert_array_equal(tr1[:, 3], tr2[:, 3])
    np.testing.assert_allclose(tr1[:, 0], tr2[:, 0], rtol=1e-9)
    # k3 .. k5 (19, 15, -539 here) are weakly determined by this short stream: the banded and the dense solve of the same steps
    # leave them 3e-9 apart (relative) after 10 iterations, while every other intrinsic agrees to 1e-9
    np.testing.assert_allclose(i1[:6], i2[:6], rtol=1e-9)
    np.testing.assert_allclose(i1[6:], i2[6:], rtol=1e-8)
    np.testing.assert_allclose(r1.reshape(-1, 4), r2, rtol=0, atol=1e-9)
    np.testing.assert_allclose(t1.reshape(-1, 3), t2, rtol=1e-9, atol=1e-9)
    # a device LM created before a re-association reads the new records: the same run as one created after it
    _associate(c, pb)
    la2 = ecb.DeviceLm(c, pb["n_cp"], ecb.lm_options(max_iterations=K))
    c.reassociate(*x)
    lb = ecb.DeviceLm(c, pb["n_cp"], ecb.lm_options(max_iterations=K))
    da, db = la2.run(*x), lb.run(*x)
    for f in ("intrinsics", "rot_cp", "trans_cp", "trace"):
        assert _same(da[f], db[f])
    for o in (la2, lb):
        o.close()


def test_shards(prob):
    """three contexts on one GPU holding contiguous thirds of the events against one: records and counts bit for bit, the normal
    equations summed by the exchange against the single context's"""
    import torch
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth
    ev, pb, one = prob["ev"], prob["pb"], prob["ctx"]
    x0 = _start(pb, False)
    _associate(one, pb)
    x = one.calibrate(pb["n_cp"], *x0, options=ecb.lm_options(max_iterations=8))[:3]
    rec = synth.to_records(ev)
    n_ev = len(ev["t"])
    cuts = [0, n_ev // 3 + 11, 2 * n_ev // 3 - 5, n_ev]
    ranks = []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        c = ecb.Context(0)
        c.set_sensor(346, 260)
        c.load_events(rec[lo:hi])
        c.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
        ranks.append(c)
    lay = one.cost_layout()
    nbytes = ranks[0].exchange_buffer_bytes(3)
    bufs = [c.device_alloc(nbytes) for c in ranks]
    outs = [torch.zeros(lay["out_doubles"], dtype=torch.float64, device="cuda") for _ in ranks]
    try:
        for epoch, max_dt in ((1, 0.0), (2, 2 * 5 * pb["step"])):
            _associate(one, pb)
            for c in ranks:
                _associate(c, pb)
            c1 = one.reassociate(*x, max_dt=max_dt)
            cr = [c.reassociate(*x, max_dt=max_dt) for c in ranks]
            assert tuple(sum(v) for v in zip(*cr)) == c1
            ei = np.concatenate([c.cost_association()[0] + lo for c, lo in zip(ranks, cuts)])
            ci = np.concatenate([c.cost_association()[1] for c in ranks])
            e1, ci1 = one.cost_association()
            assert _same(ei, e1) and _same(ci, ci1)
            assert _same(np.concatenate([c.cost_residuals(*x) for c in ranks]), one.cost_residuals(*x))
            for r in range(3):
                ranks[r].cost_normal_eq_exchange(*x, r, bufs, epoch, outs[r].data_ptr(), want_cost=False, phases=1)
            cs = [ranks[r].cost_normal_eq_exchange(*x, r, bufs, epoch, outs[r].data_ptr(), want_cost=True, phases=2) for r in range(3)]
            assert cs[0] == cs[1] == cs[2]
            a = outs[0].cpu().numpy()
            cost, H, g = one.cost_normal_eq(*x)
            ns = lay["total_spans"]
            blk = a[:ns * 1122].reshape(ns, 1122)
            assert abs(a[ns * 1122] - cost) <= 1e-12 * cost
            assert np.abs(blk[:, :1089].reshape(ns, 33, 33) - H).max() <= 1e-12 * np.abs(H).max()
            assert np.abs(blk[:, 1089:] - g).max() <= 1e-12 * np.abs(g).max()
    finally:
        for c, p in zip(ranks, bufs):
            c.synchronize()
            c.device_free(p)
            c.close()


def test_error_codes(prob):
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth
    c, ev, pb = prob["ctx"], prob["ev"], prob["pb"]
    xs = [np.ascontiguousarray(v, np.float64) for v in _start(pb, False)]
    lib = c.lib

    def call(ctx, gate, max_dt, x=xs):
        out = [C.c_int64(-7) for _ in range(5)]
        rc = lib.ecb_cost_reassociate(ctx.h, ecb._ptr(x[0]), ecb._ptr(x[1]), ecb._ptr(x[2]), gate, max_dt, *[C.byref(v) for v in out])
        return rc, tuple(v.value for v in out)

    n = _associate(c, pb)
    for gate, max_dt in ((math.nan, 0.0), (0.0, 0.0), (-1.0, 0.0), (5.0, math.nan), (5.0, -1e-300)):
        assert call(c, gate, max_dt)[0] == ecb.ERR_ARG
    assert c.cost_layout()["n_residuals"] == n  # nothing changed by a refused call
    # zero kept events
    assert call(c, 1e-300, 0.0) == (ecb.OK, (0, 0, 0, 0, n))
    assert c.cost_layout()["n_residuals"] == 0 and len(c.cost_association()[0]) == 0
    _, total = c.residual_groups(*xs, "keyframe", kf_t=pb["kf_t"])
    assert int(total["count"]) == 0
    rc, counts = call(c, GATE, 0.0)
    assert rc == ecb.OK and counts[1:] == (0, 0, counts[0], 0) and counts[0] > 0
    # no ecb_cost_setup; records of ecb_cost_set_residuals; no association
    e = ecb.Context(0)
    assert call(e, GATE, 0.0)[0] == ecb.ERR_STATE
    ncp, knots, rot, trans, obs, lm, tt, sp = _explicit_problem()
    e.cost_setup(ncp, knots, 1.75, 0.35)
    xe = [np.ascontiguousarray(v, np.float64) for v in (pb["intrinsics"], rot, trans)]
    assert call(e, GATE, 0.0, xe)[0] == ecb.ERR_STATE
    e.cost_set_residuals(obs, lm, tt, sp)
    assert call(e, GATE, 0.0, xe)[0] == ecb.ERR_STATE
    e.close()
    # events loaded since the association
    b = ecb.Context(0)
    b.set_sensor(346, 260)
    b.load_events(synth.to_records(ev))
    b.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    _associate(b, pb)
    assert call(b, GATE, 0.0)[0] == ecb.OK
    b.load_events(synth.to_records(ev))
    assert call(b, GATE, 0.0)[0] == ecb.ERR_STATE
    b.close()


@pytest.mark.xfail(strict=False, reason="measured on a B200: the re-associated solve ends 0.80 px from the generator's fx / fy / "
                                         "cx / cy (norm) against 0.74 px for the key-frame association alone, event-to-rim RMS "
                                         "0.8118 px both; the claim does not hold on this stream")
def test_quality_fast_motion():
    """the camera orbits the board with large rotations and the key-frame window is 5 ms, so a circle moves by several pixels
    between its key frame and the events of the window: one re-association round and a solve must end no farther from the
    generator's fx / fy / cx / cy than the solve on the key-frame association, with an event-to-rim RMS that does not increase.
    The generator's detected circles are the exact projections of the circle centres and none is missed, so of the three defects
    of the key-frame association only the stale circle is present here."""
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth, calib_problem
    ev = synth.make_stream(600000, 346, 260, t0=5.0, duration=0.5, seed=1007, return_truth=True, rot_amp=(0.35, 0.35, 0.3),
                           orbit=True)
    pb = calib_problem.build(ev, seed=5, step=1e-3)
    c = ecb.Context(0)
    c.set_sensor(346, 260)
    c.load_events(synth.to_records(ev))
    c.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    opt = ecb.lm_options(max_iterations=50)
    n1 = _associate(c, pb)
    i1, r1, t1, _, _ = c.calibrate(pb["n_cp"], pb["intrinsics"], pb["rot_cp"], pb["trans_cp"], options=opt)
    e1, _ = c.reprojection_errors(i1, r1, t1)
    counts = c.reassociate(i1, r1, t1)
    i2, r2, t2, _, _ = c.calibrate(pb["n_cp"], i1, r1, t1, options=opt)
    e2, _ = c.reprojection_errors(i2, r2, t2)
    truth = pb["truth_intrinsics"]
    d1, d2 = np.abs(i1[:4] - truth[:4]), np.abs(i2[:4] - truth[:4])
    rms1, rms2 = (math.sqrt(np.nanmean(v * v)) for v in (e1, e2))
    print("\nkey-frame association: %d records, fx fy cx cy error %s px (norm %.4f), event-to-rim RMS %.6f px"
          % (n1, np.array2string(d1, precision=4), np.linalg.norm(d1), rms1))
    print("re-association %s: fx fy cx cy error %s px (norm %.4f), event-to-rim RMS %.6f px"
          % (counts, np.array2string(d2, precision=4), np.linalg.norm(d2), rms2))
    c.close()
    assert np.linalg.norm(d2) <= np.linalg.norm(d1) and rms2 <= rms1


def test_cli_reassociate(tmp_path):
    """ECB_REASSOCIATE=1: the round's line, its summary, the report files of the final solve; the first solve unchanged; the error
    exits before any GPU work"""
    import subprocess
    from eventcalib_b200 import synth
    from test_host_cli import YAML, HOST
    import eventcalib_b200.build as bld
    bld.build()
    subprocess.check_call(["make", "-s", "-C", HOST])
    (tmp_path / "cfg.yaml").write_text(YAML.replace("fitCircle: 0", "fitCircle: 1"))
    for bad in ("0", "-1", "1.5", "x", "2x", ""):
        r = _run_cli(tmp_path, tmp_path / "bad", {"ECB_REASSOCIATE": bad})
        assert r.returncode == 1 and "ECB_REASSOCIATE" in r.stderr, bad
    r = _run_cli(tmp_path, tmp_path / "bad", {"ECB_REASSOCIATE": "1", "ECB_REFERENCE_SIGNATURES": "1"})
    assert r.returncode == 1 and "ECB_REFERENCE_SIGNATURES" in r.stderr
    assert not (tmp_path / "bad").exists() or not any((tmp_path / "bad").iterdir())
    ev = synth.make_stream(2000000, 346, 260, t0=5.0, duration=1.0, seed=1001, return_truth=True, workers=4,
                           rot_amp=(0.35, 0.35, 0.3), orbit=True)
    synth.write_bin(str(tmp_path / "ev.bin"), ev)
    plain = _run_cli(tmp_path, tmp_path / "plain", {"ECB_RESIDUALS": "1"})
    assert plain.returncode == 0, plain.stdout[-2000:] + plain.stderr
    assert "Re-association" not in plain.stdout and "after re-association" not in plain.stdout
    r = _run_cli(tmp_path, tmp_path / "out", {"ECB_REASSOCIATE": "1", "ECB_RESIDUALS": "1", "ECB_COVARIANCE": "1"})
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr
    lines = r.stdout.splitlines()
    first = [l for l in lines if l.startswith("Solver Summary:")]
    ra = [l for l in lines if l.startswith("Re-association 1:")]
    second = [l for l in lines if l.startswith("Solver Summary (after re-association 1):")]
    assert len(first) == len(ra) == len(second) == 1
    assert lines.index(first[0]) < lines.index(ra[0]) < lines.index(second[0])
    assert first[0] == [l for l in plain.stdout.splitlines() if l.startswith("Solver Summary:")][0]
    nums = [int(v) for v in ra[0].replace("(", " ").replace(")", " ").replace(",", " ").split() if v.isdigit()]
    n, same, changed, new, lost = nums
    n_first = int(first[0].split("residuals ")[1].split(",")[0])
    assert n == same + changed + new and n_first == same + changed + lost
    assert int(second[0].split("residuals ")[1].split(",")[0]) == n
    final = float(second[0].split("->")[1].split(",")[0])
    kf = _read(tmp_path / "out" / "ResidualsByKeyframe.txt")
    assert int(kf[:, 1].sum()) == n
    assert abs(kf[:, 6].sum() - final) <= 1e-7 * final
    assert ("%d residuals" % n) in (tmp_path / "out" / "IntrinsicsCovariance.txt").read_text()
