"""The reprojection report (ecb_cost_reprojection_errors, ecb_cost_reprojection_groups, ecb_keyframe_reprojection): e_k of every
record against a numpy restatement (spline pose, back-projection onto the board, rim point, forward model by bisection and
brentq on the monotone branch of the inverse radial polynomial), its sign against r_k, the groupings against numpy groupings of
the GPU's own e, intrinsics that fold inside the sensor, determinism, shards, error codes, the key-frame centres and the CLI."""
import math
import os

import numpy as np
import pytest
from scipy.optimize import brentq
from scipy.spatial.transform import Rotation

from test_gpu_residuals import assoc, _explicit_ctx, _explicit_problem, _nearest_kf, _points, _read, _run_cli, _same  # noqa: F401

pytestmark = pytest.mark.gpu


def _fold(k):
    h = np.array([1.0] + [(2 * i + 3) * k[i] for i in range(5)])
    r = np.roots(h[::-1])
    r = r[(np.abs(r.imag) <= 1e-12 * np.abs(r)) & (r.real > 0)].real
    return math.sqrt(r.min()) if len(r) else math.inf


def _g(k, rho):
    u = rho * rho
    return rho * (1 + u * (k[0] + u * (k[1] + u * (k[2] + u * (k[3] + u * k[4])))))


def _distort(k, rho_u, fold):
    """rho_d with g(rho_d) = rho_u on [0, fold) by bisection to full precision (NaN past g(fold))"""
    hi0 = fold if np.isfinite(fold) else max(1.0, float(np.nanmax(rho_u, initial=0.0))) * 4.0
    lo, hi = np.zeros_like(rho_u), np.full_like(rho_u, hi0)
    for _ in range(200):
        m = 0.5 * (lo + hi)
        below = _g(k, m) < rho_u
        lo, hi = np.where(below, m, lo), np.where(below, hi, m)
    out = 0.5 * (lo + hi)
    out[~(rho_u < (_g(k, fold) if np.isfinite(fold) else np.inf))] = np.nan
    return out


def _poses(Q, T, N, so3):
    """spline poses of n records: Q[n,4,4], T[n,4,3], N[n,4] -> (Rotation, t[n,3])"""
    t = np.einsum("nj,njc->nc", N, T)
    if not so3:
        return Rotation.from_quat(np.einsum("nj,njc->nc", N, Q)), t
    beta = np.cumsum(N[:, ::-1], axis=1)[:, ::-1][:, 1:]
    R = Rotation.from_quat(Q[:, 0])
    for j in range(1, 4):
        rel = Rotation.from_quat(Q[:, j - 1]).inv() * Rotation.from_quat(Q[:, j])
        R = R * Rotation.from_rotvec(beta[:, j - 1:j] * rel.as_rotvec())
    return R, t


def _project(intr, R, t, P, fold):
    """pixels of world points P at poses (R, t); NaN where not projectable"""
    pc = R.inv().apply(P - t)
    with np.errstate(divide="ignore", invalid="ignore"):
        xu, yu = pc[:, 0] / pc[:, 2], pc[:, 1] / pc[:, 2]
        ru = np.hypot(xu, yu)
        rd = _distort(intr[4:], ru, fold)
        sc = np.where(ru > 0, rd / ru, 1.0)
    q = np.stack([intr[0] * xu * sc + intr[2], intr[1] * yu * sc + intr[3]], 1)
    q[~(pc[:, 2] > 0)] = np.nan
    return q, ru


def _numpy_e(intr, rot, trans, knots_list, obs, L, tt, sp, radius, so3, oracle_mod, cp_off):
    rot, trans = np.asarray(rot).reshape(-1, 4), np.asarray(trans).reshape(-1, 3)
    n = len(obs)
    N, c0 = np.zeros((n, 4)), np.zeros(n, np.int64)
    for i in range(n):
        s, Ni = oracle_mod.basis(knots_list[sp[i]], tt[i])
        N[i], c0[i] = Ni, cp_off[sp[i]] + s - 3
    idx = c0[:, None] + np.arange(4)
    R, t = _poses(rot[idx], trans[idx], N, so3)
    fold = _fold(intr[4:])
    x, y = (obs[:, 0] - intr[2]) / intr[0], (obs[:, 1] - intr[3]) / intr[1]
    r2 = x * x + y * y
    k = intr[4:]
    s = 1 + r2 * (k[0] + r2 * (k[1] + r2 * (k[2] + r2 * (k[3] + r2 * k[4]))))
    Xr = R.apply(np.stack([x * s, y * s, np.ones(n)], 1))
    with np.errstate(divide="ignore", invalid="ignore"):
        Xw = (-t[:, 2] / Xr[:, 2])[:, None] * Xr + t
        d = Xw - L
        nd = np.linalg.norm(d, axis=1)
        P = L + radius * d / nd[:, None]
    q, ru = _project(intr, R, t, P, fold)
    e = np.sign(nd - radius) * np.hypot(q[:, 0] - obs[:, 0], q[:, 1] - obs[:, 1])
    e[~(np.sqrt(r2) < fold) | ~(nd > 0)] = np.nan
    e[~np.isfinite(e)] = np.nan
    return e, ru, fold


def _numpy_groups(e, key, G):
    out = []
    for g in range(G):
        v = e[key == g]
        ok = v[~np.isnan(v)]
        out.append(dict(count=len(ok), n_invalid=len(v) - len(ok), sum=math.fsum(ok), sum_sq=math.fsum(ok * ok),
                        max_abs=float(np.abs(ok).max()) if len(ok) else 0.0))
    return out


def _check_groups(groups, ref, rtol=1e-12):
    assert len(groups) == len(ref)
    for g, q in zip(groups, ref):
        assert int(g["count"]) == q["count"] and int(g["n_invalid"]) == q["n_invalid"]
        assert float(g["max_abs"]) == q["max_abs"]
        for f in ("sum", "sum_sq"):
            assert abs(float(g[f]) - q[f]) <= rtol * max(abs(q[f]), 1e-300) + 1e-300, (f, float(g[f]), q[f])


def _assoc_records(a):
    c, ev, pb = a["ctx"], a["ev"], a["pb"]
    ei, ci = c.cost_association()
    obs = np.stack([ev["x"][ei], ev["y"][ei]], 1).astype(float)
    return ei, ci, obs, pb["landmarks"][ci], ev["t"][ei]


def _keys(a, ei, ci, obs, cell):
    pb, ev = a["pb"], a["ev"]
    ncx, ncy = -(-346 // cell), -(-260 // cell)
    return {"keyframe": (_nearest_kf(pb["kf_t"], ev["t"][ei]), len(pb["kf_t"])),
            "circle": (ci, pb["circles"].shape[1]),
            "sensor_cell": (np.floor(obs[:, 1] / cell).astype(np.int64) * ncx + np.floor(obs[:, 0] / cell).astype(np.int64),
                            ncx * ncy)}


@pytest.mark.parametrize("so3", [False, True])
def test_reprojection_errors_and_groups(oracle_mod, assoc, so3):
    c, pb = assoc["ctx"], assoc["pb"]
    c.cost_set_rotation_model(int(so3))
    try:
        ei, ci, obs, L, tt = _assoc_records(assoc)
        sp = np.zeros(len(ei), np.int64)
        for x in _points(assoc, so3):
            e, bad = c.reprojection_errors(*x)
            e_ref, ru, fold = _numpy_e(np.asarray(x[0]), x[1], x[2], [pb["knots"]], obs, L, tt, sp, pb["radius"], so3, oracle_mod, [0])
            assert len(e) == assoc["n"] and bad == int(np.isnan(e).sum())
            assert np.array_equal(np.isnan(e), np.isnan(e_ref))
            ok = ~np.isnan(e)
            assert ok.sum() > 0.99 * len(e)
            err = np.abs(e[ok] - e_ref[ok])
            assert err.max() <= 1e-9, err.max()
            # brentq on the monotone branch for a sample
            rng = np.random.default_rng(11)
            k = np.asarray(x[0])[4:]
            for i in rng.choice(np.nonzero(ok)[0], 200, replace=False):
                rd = brentq(lambda r: _g(k, r) - ru[i], 0.0, fold, xtol=1e-16, rtol=1e-15)
                rd_b = _distort(k, np.array([ru[i]]), fold)[0]
                assert abs(rd - rd_b) * x[0][0] <= 1e-10
            # sign against the residual of the same record
            r = c.cost_residuals(*x)
            m = ok & (np.abs(r) > 1e-9)
            assert np.array_equal(np.sign(e[m]), np.sign(r[m]))
            # the groupings against numpy groupings of the GPU's own e
            for cell in (16, 7):
                for by, (key, G) in _keys(assoc, ei, ci, obs, cell).items():
                    g, tot = c.reprojection_groups(*x, by, kf_t=pb["kf_t"], cell_px=cell)
                    _check_groups(g, _numpy_groups(e, key, G))
                    _check_groups([tot], _numpy_groups(e, np.zeros(len(e), np.int64), 1))
                    g2, tot2 = c.reprojection_groups(*x, by, kf_t=pb["kf_t"], cell_px=cell)
                    assert _same(g, g2) and _same(tot, tot2)
            e2, _ = c.reprojection_errors(*x)
            assert _same(e, e2)
        # the residual report is unchanged by a reprojection call in between
        r0 = c.cost_residuals(*x)
        g0, t0 = c.residual_groups(*x, "circle")
        c.reprojection_groups(*x, "keyframe", kf_t=pb["kf_t"])
        assert _same(c.cost_residuals(*x), r0)
        g1, t1 = c.residual_groups(*x, "circle")
        assert _same(g0, g1) and _same(t0, t1)
    finally:
        c.cost_set_rotation_model(0)


def test_fold_inside_the_sensor(oracle_mod, assoc):
    import eventcalib_b200 as ecb
    c, pb = assoc["ctx"], assoc["pb"]
    intr = np.array(pb["intrinsics"], float)
    ei, ci, obs, L, tt = _assoc_records(assoc)
    rho_ev = np.hypot((obs[:, 0] - intr[2]) / intr[0], (obs[:, 1] - intr[3]) / intr[1])
    # scale k5 until the model folds inside the sensor and inside the outer tenth of the associated events
    scale = 1.0
    while not ecb.inverse_radial_fold(intr[4:] * np.r_[1, 1, 1, 1, scale]) < min(0.6, np.quantile(rho_ev, 0.9)):
        scale *= 1.25
        assert scale < 1e4
    intr[8] *= scale
    assert abs(ecb.inverse_radial_fold(intr[4:]) - _fold(intr[4:])) <= 1e-12 * _fold(intr[4:])
    x = (intr, pb["rot_cp"], pb["trans_cp"])
    e, bad = c.reprojection_errors(*x)
    e_ref, _, _ = _numpy_e(intr, x[1], x[2], [pb["knots"]], obs, L, tt, np.zeros(len(ei), np.int64), pb["radius"], False,
                           oracle_mod, [0])
    assert np.array_equal(np.isnan(e), np.isnan(e_ref))
    assert bad == int(np.isnan(e_ref).sum()) > 0
    # at the fold g' = 0 and the inverse is ill-conditioned: the values are compared where the event lies 2 % inside it
    fold = _fold(intr[4:])
    ok = ~np.isnan(e) & (rho_ev < 0.98 * fold)
    assert ok.sum() > 0.5 * len(e) and np.abs(e[ok] - e_ref[ok]).max() <= 1e-9
    for by, (key, G) in _keys(assoc, ei, ci, obs, 16).items():
        g, tot = c.reprojection_groups(*x, by, kf_t=pb["kf_t"])
        _check_groups(g, _numpy_groups(e, key, G))
        assert int(tot["n_invalid"]) == bad and int(tot["count"]) == len(e) - bad


@pytest.mark.parametrize("so3", [False, True])
def test_explicit_records_and_shards(oracle_mod, so3):
    from eventcalib_b200 import synth
    ncp, knots, rot, trans, obs, lm, tt, sp = _explicit_problem()
    if so3:
        rot = (rot.reshape(-1, 4) / np.linalg.norm(rot.reshape(-1, 4), axis=1, keepdims=True)).ravel()
    x = (synth.Camera().intrinsics(), rot, trans)
    c = _explicit_ctx(ncp, knots, obs, lm, tt, sp)
    c.cost_set_rotation_model(int(so3))
    e, bad = c.reprojection_errors(*x)
    e_ref, _, _ = _numpy_e(x[0], rot, trans, knots, obs, lm, tt, sp.astype(np.int64), 1.75, so3, oracle_mod, np.r_[0, np.cumsum(ncp)[:-1]])
    assert np.array_equal(np.isnan(e), np.isnan(e_ref)) and bad == int(np.isnan(e).sum())
    ok = ~np.isnan(e)
    assert np.abs(e[ok] - e_ref[ok]).max() <= 1e-9
    cell, ncx = 16, 22
    inside = (obs[:, 0] >= 0) & (obs[:, 0] < 346) & (obs[:, 1] >= 0) & (obs[:, 1] < 260)
    key = np.where(inside, np.floor(np.where(inside, obs[:, 1], 0) / cell).astype(np.int64) * ncx +
                   np.floor(np.where(inside, obs[:, 0], 0) / cell).astype(np.int64), -1)
    g, tot = c.reprojection_groups(*x, "sensor_cell", cell_px=cell)
    _check_groups(g, _numpy_groups(e, key, 22 * 17))
    _check_groups([tot], _numpy_groups(e, np.zeros(len(e), np.int64), 1))
    # two contexts holding contiguous halves (as the shards do), combined in rank order
    h = len(tt) // 2
    comb, ctot = None, None
    for a_, b_ in ((0, h), (h, len(tt))):
        p = _explicit_ctx(ncp, knots, obs[a_:b_], lm[a_:b_], tt[a_:b_], sp[a_:b_])
        p.cost_set_rotation_model(int(so3))
        gp, tp = p.reprojection_groups(*x, "sensor_cell", cell_px=cell)
        if comb is None:
            comb, ctot = gp.copy(), tp.copy()
        else:
            for f in ("count", "n_invalid", "sum", "sum_sq"):
                comb[f] += gp[f]
                ctot[f] += tp[f]
            comb["max_abs"] = np.maximum(comb["max_abs"], gp["max_abs"])
            ctot["max_abs"] = max(float(ctot["max_abs"]), float(tp["max_abs"]))
        p.close()
    for a_, b_ in ((comb, g), (ctot[None], tot[None])):
        for f in ("count", "n_invalid", "max_abs"):
            assert np.array_equal(a_[f], b_[f])
        for f in ("sum", "sum_sq"):
            assert np.all(np.abs(a_[f] - b_[f]) <= 1e-12 * np.maximum(np.abs(b_[f]), 1e-300))
    c.close()


def test_error_codes_and_zero_records(assoc):
    import ctypes as C
    import eventcalib_b200 as ecb
    a, pb = assoc["ctx"], assoc["pb"]
    xs = [np.ascontiguousarray(v, np.float64) for v in (pb["intrinsics"], pb["rot_cp"], pb["trans_cp"])]
    x = tuple(xs)
    lib = a.lib
    kf = np.ascontiguousarray(pb["kf_t"], np.float64)
    K, n_circ = len(kf), pb["circles"].shape[1]

    def call(ctx, by, kf_ptr, nk, cell, groups=None, cap=0, total=None):
        ng = C.c_int(-7)
        rc = lib.ecb_cost_reprojection_groups(ctx.h, ecb._ptr(xs[0]), ecb._ptr(xs[1]), ecb._ptr(xs[2]), by, kf_ptr, nk, cell,
                                              ecb._ptr(groups) if groups is not None else None, cap, C.byref(ng),
                                              ecb._ptr(total) if total is not None else None)
        return rc, ng.value

    kfp = ecb._ptr(kf)
    assert call(a, 0, kfp, K, 16) == (ecb.OK, K)
    assert call(a, 1, None, 0, 16) == (ecb.OK, n_circ)
    assert call(a, 2, None, 0, 16) == (ecb.OK, 22 * 17)
    buf = np.full(n_circ, 7, ecb.REPROJECTION_GROUP_DTYPE)
    tot = np.full((), 7, ecb.REPROJECTION_GROUP_DTYPE)
    assert call(a, 1, None, 0, 16, buf, n_circ - 1, tot) == (ecb.ERR_ARG, n_circ)
    assert np.all(buf["count"] == 7) and int(tot["count"]) == 7
    assert call(a, 1, None, 0, 16, buf, n_circ, tot) == (ecb.OK, n_circ)
    assert int(tot["count"]) + int(tot["n_invalid"]) == assoc["n"]
    assert call(a, 3, kfp, K, 16)[0] == ecb.ERR_ARG
    assert call(a, -1, kfp, K, 16)[0] == ecb.ERR_ARG
    assert call(a, 2, None, 0, 0)[0] == ecb.ERR_ARG
    assert call(a, 0, None, K, 16)[0] == ecb.ERR_ARG
    assert call(a, 0, kfp, K - 1, 16)[0] == ecb.ERR_ARG
    assert lib.ecb_cost_reprojection_errors(a.h, None, ecb._ptr(xs[1]), ecb._ptr(xs[2]), None, None, None) == ecb.ERR_ARG
    assert lib.ecb_inverse_radial_fold(None, None) == ecb.ERR_ARG
    ncp, knots, rot, trans, obs, lm, tt, sp = _explicit_problem()
    e = _explicit_ctx(ncp, knots, obs, lm, tt, sp, sensor=False)
    assert call(e, 0, kfp, K, 16)[0] == ecb.ERR_STATE
    assert call(e, 1, None, 0, 16)[0] == ecb.ERR_STATE
    assert call(e, 2, None, 0, 16)[0] == ecb.ERR_STATE
    with pytest.raises(ValueError):
        e.reprojection_groups(*x, "span")
    # zero records: empty e, all-zero groups
    e.set_sensor(346, 260)
    e.cost_setup(ncp, knots, 1.75, 0.35)
    e.cost_set_residuals(np.zeros((0, 2)), np.zeros((0, 3)), np.zeros(0), np.zeros(0))
    xe = (x[0], rot, trans)
    ev, bad = e.reprojection_errors(*xe)
    assert len(ev) == 0 and bad == 0
    g, t = e.reprojection_groups(*xe, "sensor_cell", cell_px=32)
    assert len(g) == 11 * 9 and not np.any(g.view(np.uint8)) and not np.any(np.atleast_1d(t).view(np.uint8))
    e.close()
    # no ecb_cost_setup
    b = ecb.Context(0)
    assert lib.ecb_cost_reprojection_errors(b.h, *(ecb._ptr(v) for v in xs), None, None, None) == ecb.ERR_STATE
    circ = np.ascontiguousarray(pb["circles"], np.float64)
    lmk = np.ascontiguousarray(pb["landmarks"], np.float64)
    out = [np.zeros(K * n_circ * 2), np.zeros(K * n_circ)]
    kf_args = (ecb._ptr(kf), ecb._ptr(circ), K, n_circ, ecb._ptr(lmk), ecb._ptr(out[0]), ecb._ptr(out[1]), None)
    assert lib.ecb_keyframe_reprojection(b.h, *(ecb._ptr(v) for v in xs), *kf_args) == ecb.ERR_STATE
    b.close()
    assert lib.ecb_keyframe_reprojection(a.h, *(ecb._ptr(v) for v in xs), ecb._ptr(kf), ecb._ptr(circ), 0, n_circ,
                                         ecb._ptr(lmk), None, None, None) == ecb.ERR_ARG
    # the device output variant equals the host copy
    import torch
    d = torch.empty(assoc["n"], dtype=torch.float64, device="cuda:0")
    a.reprojection_errors(*x, d_out=d.data_ptr(), host=False)
    a.synchronize()
    assert _same(d.cpu().numpy(), a.reprojection_errors(*x)[0])


@pytest.mark.parametrize("so3", [False, True])
def test_keyframe_reprojection(oracle_mod, assoc, so3):
    c, pb = assoc["ctx"], assoc["pb"]
    c.cost_set_rotation_model(int(so3))
    try:
        for x in _points(assoc, so3):
            kf = np.array(pb["kf_t"], float)
            circ = np.array(pb["circles"], float)
            K, n = circ.shape[:2]
            circ[1, 3, 2] = -1.0   # absent features
            circ[4, :5, 2] = -1.0
            kf[-1] = pb["knots"][-1] + 1.0   # a stamp outside every segment
            proj, err, tot = c.keyframe_reprojection(*x, kf, circ, pb["landmarks"])
            intr = np.asarray(x[0])
            rot, trans = np.asarray(x[1]).reshape(-1, 4), np.asarray(x[2]).reshape(-1, 3)
            fold = _fold(intr[4:])
            ref = np.full((K, n, 2), np.nan)
            for k in range(K - 1):
                s, N = oracle_mod.basis(pb["knots"], kf[k])
                R, t = _poses(rot[None, s - 3:s + 1], trans[None, s - 3:s + 1], N[None], so3)
                R = Rotation.from_quat(np.repeat(R.as_quat(), n, 0))
                q, _ = _project(intr, R, np.repeat(t, n, 0), pb["landmarks"], fold)
                ref[k] = q
            ref[circ[:, :, 2] < 0] = np.nan
            assert np.array_equal(np.isnan(proj), np.isnan(ref))
            assert np.isnan(proj[1, 3]).all() and np.isnan(proj[4, :5]).all() and np.isnan(proj[-1]).all()
            ok = ~np.isnan(ref[:, :, 0])
            assert np.abs(proj[ok] - ref[ok]).max() <= 1e-9
            e_ref = np.hypot(ref[:, :, 0] - circ[:, :, 0], ref[:, :, 1] - circ[:, :, 1])
            assert np.array_equal(np.isnan(err), np.isnan(e_ref)) and np.abs(err[ok] - e_ref[ok]).max() <= 1e-9
            present = circ[:, :, 2] >= 0
            v = err[present]
            assert int(tot["count"]) == int((~np.isnan(v)).sum()) and int(tot["n_invalid"]) == int(np.isnan(v).sum()) >= 1
            vv = v[~np.isnan(v)]
            assert abs(float(tot["sum_sq"]) - math.fsum(vv * vv)) <= 1e-12 * math.fsum(vv * vv)
            assert float(tot["max_abs"]) == vv.max()
            p2, e2, t2 = c.keyframe_reprojection(*x, kf, circ, pb["landmarks"])
            assert _same(p2, proj) and _same(e2, err) and _same(t2, tot)
    finally:
        c.cost_set_rotation_model(0)


def test_cli_writes_reprojection_report(tmp_path):
    """ECB_REPROJECTION=1 on the stream of test_cli_writes_residual_report"""
    import subprocess
    from eventcalib_b200 import synth
    from test_host_cli import YAML, HOST
    import eventcalib_b200.build as bld
    bld.build()
    subprocess.check_call(["make", "-s", "-C", HOST])
    ev = synth.make_stream(2000000, 346, 260, t0=5.0, duration=1.0, seed=1001, return_truth=True, workers=4,
                           rot_amp=(0.35, 0.35, 0.3), orbit=True)
    synth.write_bin(str(tmp_path / "ev.bin"), ev)
    (tmp_path / "cfg.yaml").write_text(YAML.replace("fitCircle: 0", "fitCircle: 1"))
    files = ("ReprojectionByKeyframe.txt", "ReprojectionByCircle.txt", "ReprojectionMap.txt")
    plain = tmp_path / "plain"
    r0 = _run_cli(tmp_path, plain, {})
    assert r0.returncode == 0, r0.stdout[-2000:] + r0.stderr
    assert "Reprojection:" not in r0.stdout and not any((plain / f).exists() for f in files)

    def run(save, devices):
        r = _run_cli(tmp_path, save, {"ECB_REPROJECTION": "1", "ECB_RESIDUAL_CELL": "20"}, devices)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr
        summ = [l for l in r.stdout.splitlines() if l.startswith("Solver Summary:")][0]
        n_res = int(summ.split("residuals ")[1].split(",")[0])
        line = [l for l in r.stdout.splitlines() if l.startswith("Reprojection:")][0]
        return r, n_res, line, [_read(save / f) for f in files]

    save = tmp_path / "out"
    r, n_res, line, (kf, circ, cells) = run(save, "0")
    # without the switch the output set is the same, but for the report
    assert sorted(p.name for p in plain.iterdir()) == sorted(p.name for p in save.iterdir() if p.name not in files)
    assert kf.shape[1] == 8 and circ.shape == (36, 11) and cells.shape[1] == 7
    assert "# cell 20 px" in (save / "ReprojectionMap.txt").read_text()
    traj = _read(save / "TrajectoryByEvent.txt")
    assert set(np.round(traj[:, 0], 6)) <= set(np.round(kf[:, 0], 6)) and np.all(np.diff(kf[:, 0]) > 0)
    for tab, cc in ((kf, 1), (circ, 4), (cells, 2)):
        assert int(tab[:, cc].sum() + tab[:, cc + 1].sum()) == n_res
    assert np.all(cells[:, 0] % 20 == 0) and np.all(cells[:, 1] % 20 == 0)
    # the line: events, RMS, mean, max |e|, invalid; centres, RMS; fold and corner radius
    w = line.replace(",", " ").replace(";", " ").split()
    count, rms, mean, mx, bad = int(w[1]), float(w[4]), float(w[7]), float(w[11]), int(w[14])
    ccount, crms = int(w[15]), float(w[19])
    fold_px, corner_px = float(w[23]), float(w[29])
    assert count + bad == n_res and count == int(kf[:, 1].sum()) and bad == int(kf[:, 2].sum())
    cnt = kf[:, 1]
    assert abs(rms - math.sqrt(np.sum(cnt * np.nan_to_num(kf[:, 4]) ** 2) / count)) <= 1e-7 * rms
    assert abs(mean - np.sum(cnt * np.nan_to_num(kf[:, 3])) / count) <= 1e-7 * max(abs(mean), 1e-12)
    assert mx == pytest.approx(np.nanmax(kf[:, 5]), rel=1e-9)
    assert ccount == int(kf[:, 6].sum()) == int(circ[:, 9].sum()) > 0
    assert abs(crms - math.sqrt(np.sum(kf[:, 6] * np.nan_to_num(kf[:, 7]) ** 2) / ccount)) <= 1e-7 * crms
    assert corner_px > 0 and fold_px > 0
    import torch
    if torch.cuda.device_count() >= 2:   # ShardedCalibSpline::reprojectionGroups over two GPUs against one
        _, n2, _, (kf2, circ2, cells2) = run(tmp_path / "out2", "0,1")
        assert n2 == n_res
        for a_, b_, cc in ((kf, kf2, 1), (circ, circ2, 4), (cells, cells2, 2)):
            assert np.array_equal(a_[:, cc:cc + 2], b_[:, cc:cc + 2])
            np.testing.assert_allclose(b_[:, cc + 3], a_[:, cc + 3], rtol=1e-5)
        np.testing.assert_allclose(kf2[:, 7], kf[:, 7], rtol=1e-5)
