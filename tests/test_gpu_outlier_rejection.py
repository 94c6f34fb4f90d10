"""Outlier rejection (ecb_cost_reject): the decisions against a numpy mask built from the GPU's own r, the kept records against
a context given them explicitly, the no-op, shards, a calibration with mislabelled key frames, the error codes and the CLI."""
import ctypes as C
import math

import numpy as np
import pytest

from test_gpu_residuals import _explicit_ctx, _explicit_problem, _nearest_kf, _read, _run_cli
from test_outlier_policy import apply_policy, policy_lib

pytestmark = pytest.mark.gpu


def _same(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


@pytest.fixture(scope="module")
def prob():
    """the stream of test_gpu_residuals (without its midpoint event)"""
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth, calib_problem
    ev = synth.make_stream(300000, 346, 260, t0=5.0, duration=0.3, seed=1004, return_truth=True)
    pb = calib_problem.build(ev, seed=3)
    c = ecb.Context(0)
    c.set_sensor(346, 260)
    c.load_events(synth.to_records(ev))
    c.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    yield dict(ctx=c, ev=ev, pb=pb)
    c.close()


def _associate(c, pb):
    return c.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])


def _explicit_of(ev, pb, ei, ci):
    """the records (event ei, circle ci) as explicit residual blocks"""
    obs = np.stack([ev["x"][ei], ev["y"][ei]], 1).astype(float)
    return obs, pb["landmarks"][ci], ev["t"][ei], np.zeros(len(ei), np.int32)


def _check_normal_eq(c, ref, x):
    cost, H, g = c.cost_normal_eq(*x)
    cost_r, H_r, g_r = ref.cost_normal_eq(*x)
    assert abs(cost - cost_r) <= 1e-12 * cost_r
    assert abs(c.cost_eval(*x) - ref.cost_eval(*x)) <= 1e-12 * cost_r
    assert np.abs(H - H_r).max() <= 1e-12 * np.abs(H_r).max() and np.abs(g - g_r).max() <= 1e-12 * np.abs(g_r).max()


@pytest.mark.parametrize("so3", [False, True])
def test_decisions_match_numpy(prob, so3):
    import eventcalib_b200 as ecb
    c, ev, pb = prob["ctx"], prob["ev"], prob["pb"]
    kf = pb["kf_t"]
    K = len(kf)
    c.cost_set_rotation_model(int(so3))
    try:
        rot = pb["rot_cp"].reshape(-1, 4)
        rot = (rot / np.linalg.norm(rot, axis=1, keepdims=True)).ravel() if so3 else pb["rot_cp"]
        x0 = (pb["intrinsics"], rot, pb["trans_cp"])
        _associate(c, pb)
        i8, r8, t8, _, _ = c.calibrate(pb["n_cp"], *x0, options=ecb.lm_options(max_iterations=8, rotation_model=int(so3)))
        every7 = (np.arange(K) % 7 == 3).astype(np.uint8)
        for x in (x0, (i8, r8, t8)):
            n = _associate(c, pb)
            ei0, ci0 = c.cost_association()
            r0 = c.cost_residuals(*x)
            key = _nearest_kf(kf, ev["t"][ei0])
            a = np.abs(r0)
            cases = [(math.inf, None), (float(np.quantile(a, 0.99)), None), (float(np.quantile(a, 0.9)), every7),
                     (math.inf, every7), (pb["huber"], None), (0.0, None)]
            for thr, drop in cases:
                if drop is not None or thr != math.inf:
                    assert _associate(c, pb) == n
                keep = a <= thr
                if drop is not None:
                    keep &= drop[key] == 0
                kept, removed = c.reject_residuals(*x, max_abs_r=thr, drop_keyframes=drop, kf_t=kf if drop is not None else None)
                assert (kept, removed) == (int(keep.sum()), n - int(keep.sum()))
                assert c.cost_layout()["n_residuals"] == kept
                ei, ci = c.cost_association()
                assert np.array_equal(ei, ei0[keep]) and np.array_equal(ci, ci0[keep])
                assert _same(c.cost_residuals(*x), r0[keep])
                if 0 < kept:
                    ref = ecb.Context(0)
                    ref.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
                    ref.cost_set_rotation_model(int(so3))
                    ref.cost_set_residuals(*_explicit_of(ev, pb, ei, ci))
                    _check_normal_eq(c, ref, x)
                    ref.close()
    finally:
        c.cost_set_rotation_model(0)


def test_explicit_records():
    from eventcalib_b200 import synth
    ncp, knots, rot, trans, obs, lm, tt, sp = _explicit_problem()
    x = (synth.Camera().intrinsics(), rot, trans)
    c = _explicit_ctx(ncp, knots, obs, lm, tt, sp)
    r0 = c.cost_residuals(*x)
    thr = float(np.quantile(np.abs(r0), 0.8))
    keep = np.abs(r0) <= thr
    assert c.reject_residuals(*x, max_abs_r=thr) == (int(keep.sum()), int((~keep).sum()))
    assert _same(c.cost_residuals(*x), r0[keep])
    ref = _explicit_ctx(ncp, knots, obs[keep], lm[keep], tt[keep], sp[keep])
    _check_normal_eq(c, ref, x)
    assert _same(c.residual_groups(*x, "sensor_cell")[0], ref.residual_groups(*x, "sensor_cell")[0])
    c.close()
    ref.close()


def test_noop_is_bit_identical(prob):
    """max_abs_r = inf and no mask: ecb_calibrate, the device LM and ecb_covariance as on a context that never called it; a device
    LM created before a real rejection stays valid"""
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth
    ev, pb = prob["ev"], prob["pb"]
    ctxs = []
    for _ in range(2):
        c = ecb.Context(0)
        c.set_sensor(346, 260)
        c.load_events(synth.to_records(ev))
        c.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
        n = _associate(c, pb)
        ctxs.append(c)
    a, b = ctxs
    x = (pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])
    assert a.reject_residuals(*x) == (n, 0)
    assert a.reject_residuals(*x) == (n, 0)
    opt = ecb.lm_options(max_iterations=10)
    ra, rb = a.calibrate(pb["n_cp"], *x, options=opt), b.calibrate(pb["n_cp"], *x, options=opt)
    for u, v in zip(ra[:3], rb[:3]):
        assert _same(u, v)
    assert ra[3] == rb[3] and _same(ra[4], rb[4])
    la, lb = ecb.DeviceLm(a, pb["n_cp"], opt), ecb.DeviceLm(b, pb["n_cp"], opt)
    da, db = la.run(*x), lb.run(*x)
    for f in ("intrinsics", "rot_cp", "trans_cp", "trace"):
        assert _same(da[f], db[f])
    ca, cb = a.covariance(pb["n_cp"], *ra[:3]), b.covariance(pb["n_cp"], *ra[:3])
    assert ca["ok"] and cb["ok"]
    for f in ("cov_intrinsics", "cov_band", "cov_cross"):
        assert _same(ca[f], cb[f])
    # a device LM created before a rejection reads the kept records: the same run as one created after it
    thr = float(np.quantile(np.abs(a.cost_residuals(*x)), 0.95))
    kept, removed = a.reject_residuals(*x, max_abs_r=thr)
    assert removed > 0
    lc = ecb.DeviceLm(a, pb["n_cp"], opt)
    d_before, d_after = la.run(*x), lc.run(*x)
    for f in ("intrinsics", "rot_cp", "trans_cp", "trace"):
        assert _same(d_before[f], d_after[f])
    assert a.covariance(pb["n_cp"], *ra[:3])["n_residuals"] == kept
    for o in (la, lb, lc):
        o.close()
    for c in ctxs:
        c.close()


def test_shards(prob):
    """two contexts on one GPU holding contiguous halves of the events, the same threshold and mask: their kept records
    concatenated equal one context's, the exchange sums the single context's normal equations, also with one half emptied"""
    import torch
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth
    ev, pb, one = prob["ev"], prob["pb"], prob["ctx"]
    kf = pb["kf_t"]
    K = len(kf)
    x = (pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])
    rec = synth.to_records(ev)
    n_ev = len(ev["t"])
    cut = n_ev // 2 + 777
    ranks = []
    for lo, hi in ((0, cut), (cut, n_ev)):
        c = ecb.Context(0)
        c.set_sensor(346, 260)
        c.load_events(rec[lo:hi])
        c.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
        ranks.append(c)
    lay = one.cost_layout()
    nbytes = ranks[0].exchange_buffer_bytes(2)
    bufs = [c.device_alloc(nbytes) for c in ranks]
    outs = [torch.zeros(lay["out_doubles"], dtype=torch.float64, device="cuda") for _ in ranks]
    try:
        _associate(one, pb)
        thr = float(np.quantile(np.abs(one.cost_residuals(*x)), 0.97))
        for epoch in (1, 2):
            _associate(one, pb)
            for c in ranks:
                _associate(c, pb)
            if epoch == 1:
                drop = (np.arange(K) % 5 == 1).astype(np.uint8)
            else:   # every key frame that rank 1's records count under and later ones: rank 1 keeps nothing
                j0 = int(_nearest_kf(kf, ev["t"][ranks[1].cost_association()[0] + cut]).min())
                drop = (np.arange(K) >= j0).astype(np.uint8)
            t = thr
            k1, _ = one.reject_residuals(*x, max_abs_r=t, drop_keyframes=drop, kf_t=kf)
            kr = [c.reject_residuals(*x, max_abs_r=t, drop_keyframes=drop, kf_t=kf)[0] for c in ranks]
            assert sum(kr) == k1
            ei = np.concatenate([ranks[0].cost_association()[0], ranks[1].cost_association()[0] + cut])
            ci = np.concatenate([c.cost_association()[1] for c in ranks])
            e1, c1 = one.cost_association()
            assert np.array_equal(ei, e1) and np.array_equal(ci, c1)
            assert _same(np.concatenate([c.cost_residuals(*x) for c in ranks]), one.cost_residuals(*x))
            if epoch == 2:
                assert kr[1] == 0 and ranks[1].cost_layout()["n_residuals"] == 0
            for r in (0, 1):   # two ranks on ONE device: all send sides first, then the receive sides
                ranks[r].cost_normal_eq_exchange(*x, r, bufs, epoch, outs[r].data_ptr(), want_cost=False, phases=1)
            cs = [ranks[r].cost_normal_eq_exchange(*x, r, bufs, epoch, outs[r].data_ptr(), want_cost=True, phases=2) for r in (0, 1)]
            assert cs[0] == cs[1]
            a = outs[0].cpu().numpy()
            assert np.array_equal(a, outs[1].cpu().numpy())
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


def test_mislabelled_keyframes_are_dropped():
    """five key frames whose circle ids are shifted by one grid row (a wrong grid order): calibrate, apply the policy (k = 3),
    calibrate again from that solution.  The dropped key frames are exactly the corrupted ones, and fx / fy / cx / cy move toward
    the generator's camera and back to the solution of the uncorrupted problem.  The camera orbits the board with large rotations:
    under the default, nearly fronto-parallel motion the focal length is not determined by the data (the uncorrupted solve then
    ends 65 px from the generator's fx, and so does the solve after rejection), which says nothing about the rejection."""
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth, calib_problem
    ev = synth.make_stream(600000, 346, 260, t0=5.0, duration=0.5, seed=1007, return_truth=True, rot_amp=(0.35, 0.35, 0.3),
                           orbit=True)
    pb = calib_problem.build(ev, seed=5)
    K = len(pb["kf_t"])
    bad = np.array([K // 6, K // 3, K // 2, 2 * K // 3, 5 * K // 6])
    circ = pb["circles"].copy()
    circ[bad] = np.roll(circ[bad], 4, axis=1)   # the 4 circles of a row: every id one row off
    c = ecb.Context(0)
    c.set_sensor(346, 260)
    c.load_events(synth.to_records(ev))
    c.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    opt = ecb.lm_options(max_iterations=50)
    x0 = (pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])
    c.cost_associate(pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
    i0 = c.calibrate(pb["n_cp"], *x0, options=opt)[0]
    c.cost_associate(pb["kf_t"], circ, pb["landmarks"], pb["step"])
    i1, r1, t1, s1, _ = c.calibrate(pb["n_cp"], *x0, options=opt)
    groups, _ = c.residual_groups(i1, r1, t1, "keyframe", kf_t=pb["kf_t"])
    s, thr, drop = apply_policy(policy_lib(), groups, 3.0)
    kept, removed = c.reject_residuals(i1, r1, t1, max_abs_r=thr, drop_keyframes=drop, kf_t=pb["kf_t"])
    assert sorted(np.nonzero(drop)[0].tolist()) == sorted(bad.tolist())
    i2, r2, t2, s2, _ = c.calibrate(pb["n_cp"], i1, r1, t1, options=opt)
    truth = pb["truth_intrinsics"]
    e0, e1, e2 = (np.abs(v[:4] - truth[:4]) for v in (i0, i1, i2))
    print("\nmislabelled key frames %s of %d; s %.6g, threshold %.6g, records removed %d of %d" % (bad.tolist(), K, s, thr, removed,
                                                                                                  kept + removed))
    print("fx fy cx cy error, uncorrupted:      %s px" % np.array2string(e0, precision=4))
    print("fx fy cx cy error before rejection: %s px" % np.array2string(e1, precision=4))
    print("fx fy cx cy error after rejection:  %s px" % np.array2string(e2, precision=4))
    assert np.all(e2 < e1)
    assert np.all(np.abs(i2[:4] - i0[:4]) < np.abs(i1[:4] - i0[:4]))
    c.close()


def test_error_codes(prob):
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth
    c, ev, pb = prob["ctx"], prob["ev"], prob["pb"]
    kf = np.ascontiguousarray(pb["kf_t"], np.float64)
    K = len(kf)
    xs = [np.ascontiguousarray(v, np.float64) for v in (pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])]
    lib = c.lib
    drop = np.zeros(K, np.uint8)

    def call(ctx, thr, kf_ptr, drop_ptr, nk):
        kept, removed = C.c_int64(-7), C.c_int64(-7)
        rc = lib.ecb_cost_reject(ctx.h, ecb._ptr(xs[0]), ecb._ptr(xs[1]), ecb._ptr(xs[2]), thr, kf_ptr, drop_ptr, nk,
                                 C.byref(kept), C.byref(removed))
        return rc, kept.value, removed.value

    n = _associate(c, pb)
    kfp, dp = ecb._ptr(kf), ecb._ptr(drop)
    assert call(c, math.nan, None, None, 0)[0] == ecb.ERR_ARG
    assert call(c, -1e-300, None, None, 0)[0] == ecb.ERR_ARG
    assert call(c, 1.0, None, dp, K)[0] == ecb.ERR_ARG
    assert call(c, 1.0, kfp, dp, K - 1)[0] == ecb.ERR_ARG
    assert c.cost_layout()["n_residuals"] == n    # nothing removed by a refused call
    assert call(c, math.inf, kfp, dp, K) == (ecb.OK, n, 0)
    assert call(c, math.inf, None, None, 0) == (ecb.OK, n, 0)
    # no ecb_cost_setup
    e = ecb.Context(0)
    assert call(e, 1.0, None, None, 0)[0] == ecb.ERR_STATE
    # a key-frame mask on explicit records
    ncp, knots, rot, trans, obs, lm, tt, sp = _explicit_problem()
    e.cost_setup(ncp, knots, 1.75, 0.35)
    e.cost_set_residuals(obs, lm, tt, sp)
    xe = [np.ascontiguousarray(v, np.float64) for v in (pb["intrinsics"], rot, trans)]
    rc = lib.ecb_cost_reject(e.h, ecb._ptr(xe[0]), ecb._ptr(xe[1]), ecb._ptr(xe[2]), 1.0, kfp, dp, K, None, None)
    assert rc == ecb.ERR_STATE
    # zero records: OK, both counts 0
    e.cost_set_residuals(np.zeros((0, 2)), np.zeros((0, 3)), np.zeros(0), np.zeros(0))
    assert e.reject_residuals(*xe, max_abs_r=0.0) == (0, 0)
    e.close()
    # a mask after events were loaded since the association; the threshold alone needs no events
    b = ecb.Context(0)
    b.set_sensor(346, 260)
    b.load_events(synth.to_records(ev))
    b.cost_setup([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    _associate(b, pb)
    b.load_events(synth.to_records(ev))
    assert call(b, 1.0, kfp, dp, K)[0] == ecb.ERR_STATE
    assert call(b, math.inf, None, None, 0)[0] == ecb.OK
    b.close()


def test_cli_reject(tmp_path):
    """ECB_REJECT=3 on the stream of test_cli_writes_residual_report: the rejection line, the second summary, the report files of
    the second solve; the two error exits"""
    import subprocess
    from eventcalib_b200 import synth
    from test_host_cli import YAML, HOST
    import eventcalib_b200.build as bld
    bld.build()
    subprocess.check_call(["make", "-s", "-C", HOST])
    (tmp_path / "cfg.yaml").write_text(YAML.replace("fitCircle: 0", "fitCircle: 1"))
    for bad in ("0", "-3", "inf", "nan", "3x", ""):
        r = _run_cli(tmp_path, tmp_path / "bad", {"ECB_REJECT": bad})
        assert r.returncode == 1 and "ECB_REJECT" in r.stderr, bad
    r = _run_cli(tmp_path, tmp_path / "bad", {"ECB_REJECT": "3", "ECB_REFERENCE_SIGNATURES": "1"})
    assert r.returncode == 1 and "ECB_REFERENCE_SIGNATURES" in r.stderr
    ev = synth.make_stream(2000000, 346, 260, t0=5.0, duration=1.0, seed=1001, return_truth=True, workers=4,
                           rot_amp=(0.35, 0.35, 0.3), orbit=True)
    synth.write_bin(str(tmp_path / "ev.bin"), ev)

    def run(save, devices):
        r = _run_cli(tmp_path, save, {"ECB_REJECT": "3", "ECB_RESIDUALS": "1", "ECB_COVARIANCE": "1"}, devices)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr
        lines = r.stdout.splitlines()
        first = [l for l in lines if l.startswith("Solver Summary:")]
        rej = [l for l in lines if l.startswith("Outlier rejection:")]
        second = [l for l in lines if l.startswith("Solver Summary (after rejection):")]
        assert len(first) == len(rej) == len(second) == 1
        assert lines.index(first[0]) < lines.index(rej[0]) < lines.index(second[0])
        return r.stdout, first[0], rej[0], second[0]

    save = tmp_path / "out"
    out, first, rej, second = run(save, "0")
    n_all = int(first.split("residuals ")[1].split(",")[0])
    n_kept = int(second.split("residuals ")[1].split(",")[0])
    removed = int(rej.split("records removed ")[1].split(" ")[0])
    assert rej.split(" of ")[-1].split(" ")[0] == str(n_all) and n_kept == n_all - removed
    k = float(rej.split("k ")[1].split(",")[0])
    s = float(rej.split(", s ")[1].split(",")[0])
    thr = float(rej.split("threshold ")[1].split(",")[0])
    assert k == 3 and thr == pytest.approx(3 * s, rel=1e-7)
    # the reports describe the second solve: counts and sum of costs against its summary line
    final = float(second.split("->")[1].split(",")[0])
    kf = _read(save / "ResidualsByKeyframe.txt")
    assert int(kf[:, 1].sum()) == n_kept
    assert abs(kf[:, 6].sum() - final) <= 1e-7 * final
    cov = (save / "IntrinsicsCovariance.txt").read_text()
    assert ("%d residuals" % n_kept) in cov
    import torch
    if torch.cuda.device_count() >= 2:   # ShardedCalibSpline::rejectOutliers over two GPUs against one
        out2, first2, rej2, second2 = run(tmp_path / "out2", "0,1")
        assert rej2.split("key frames dropped")[1] == rej.split("key frames dropped")[1]
        assert int(second2.split("residuals ")[1].split(",")[0]) == n_kept
