"""The motion header eventcalib_b200/csrc/ecb_motion.h (host build, -ffp-contract=off) for both rotation models:
- the derivative basis of orders 1 and 2 against scipy.interpolate.BSpline(...).derivative() on clamped non-uniform knots, order
  0 bit for bit against the port's basis;
- v_w and a_w against central differences of the spline position;
- w_b against Log(R(t-h)^T R(t+h)) / 2h of a numpy restatement of the spline rotation, with quaternion control points of norms
  != 1 and, for SO(3), a run of near-identical control points (the small-angle branch of Log and Exp);
- B_j against central differences along each control point's tangent (oracle.quat_plus / oracle.so3_plus);
- the pose bit for bit against ecb_pose_eval.
Times: the first knot, the last knot, exactly on interior knots, inside spans."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy.interpolate import BSpline
from scipy.spatial.transform import Rotation

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_CP = 8


def _lib():
    so = os.path.join(ROOT, "tests", "_build", "libmotion_host.so")
    os.makedirs(os.path.dirname(so), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", so,
                           os.path.join(ROOT, "tests", "helpers", "motion_host.cpp")])
    lib = C.CDLL(so)
    for f in (lib.host_ders_basis, lib.host_motion, lib.host_pose_eval):
        f.restype = None
    lib.host_ders_basis.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.host_motion.argtypes = [C.c_void_p] * 5 + [C.c_int, C.c_void_p, C.c_void_p]
    lib.host_pose_eval.argtypes = [C.c_void_p] * 3 + [C.c_int, C.c_void_p]
    return lib


def _P(a):
    return a.ctypes.data_as(C.c_void_p)


def _spline(oracle_mod, so3, seed, flat=False):
    """clamped cubic knots over [5, 6] (non-uniform: from random stamps); rotation control points along a smooth curve (unit
    for SO(3), norms 0.9 .. 1.1 for the quaternion model, whose spline normalises), translations random.  flat: control points
    2 .. 5 equal up to rotations of 1e-12 rad, so relative rotations take the small-angle branch of Log / Exp."""
    rng = np.random.default_rng(seed)
    us = np.sort(rng.uniform(5.0, 6.0, 40))
    us[0], us[-1] = 5.0, 6.0
    kn = oracle_mod.knots(us, N_CP)
    rv = np.cumsum(rng.normal(0.0, 0.25, (N_CP, 3)), axis=0)
    if flat:
        rv[2:6] = rv[2] + rng.normal(0.0, 1e-12, (4, 3))
    rot = Rotation.from_rotvec(rv).as_quat()
    rot *= np.sign(rot[:, 3:4])
    for k in range(1, N_CP):   # one sign per quaternion: a continuous curve
        if rot[k] @ rot[k - 1] < 0:
            rot[k] = -rot[k]
    if not so3:
        rot *= rng.uniform(0.9, 1.1, (N_CP, 1))
    trans = rng.normal(0.0, 0.5, (N_CP, 3))
    return np.ascontiguousarray(kn), np.ascontiguousarray(rot), np.ascontiguousarray(trans)


def _times(kn):
    rng = np.random.default_rng(7)
    inside = [kn[s] + (kn[s + 1] - kn[s]) * rng.uniform(0.1, 0.9) for s in range(3, N_CP)]
    return [kn[0], kn[-1], *kn[4:N_CP], *inside]


def _rotation_np(kn, rot, u, so3, oracle_mod):
    """restatement of the spline rotation at u (a scipy Rotation)"""
    span, N = oracle_mod.basis(kn, u)
    Q = rot[span - 3:span + 1]
    if not so3:
        return Rotation.from_quat(N @ Q)
    beta = np.cumsum(N[::-1])[::-1][1:]   # cumulative basis b1 .. b3
    R = Rotation.from_quat(Q[0])
    for j in range(1, 4):
        rel = Rotation.from_quat(Q[j - 1]).inv() * Rotation.from_quat(Q[j])
        R = R * Rotation.from_rotvec(beta[j - 1] * rel.as_rotvec())
    return R


def _motion(lib, oracle_mod, kn, rot, trans, u, so3, want_J=False):
    span, N = oracle_mod.basis(kn, u)
    Nh, Nd, Ndd = np.zeros(4), np.zeros(4), np.zeros(4)
    lib.host_ders_basis(_P(kn), span, u, _P(Nh), _P(Nd), _P(Ndd))
    Q, T = np.ascontiguousarray(rot[span - 3:span + 1]), np.ascontiguousarray(trans[span - 3:span + 1])
    m, J = np.zeros(16), np.zeros((9, 24))
    lib.host_motion(_P(Q), _P(T), _P(Nh), _P(Nd), _P(Ndd), so3, _P(m), _P(J) if want_J else None)
    return dict(span=span, N=N, Nh=Nh, Nd=Nd, Ndd=Ndd, Q=Q, T=T, m=m, J=J)


def test_derivative_basis_against_scipy(oracle_mod):
    """order 0 bit for bit the port's basis (so the pose is the evaluation's); orders 1 and 2 equal scipy's derivative of each
    basis function to 1e-12 of the largest value (both are exact formulas in FP64: only rounding differs)"""
    lib = _lib()
    for seed in range(4):
        kn, _, _ = _spline(oracle_mod, 0, seed)
        basis = [BSpline(kn, np.eye(N_CP)[j], 3) for j in range(N_CP)]
        d1 = [b.derivative(1) for b in basis]
        d2 = [b.derivative(2) for b in basis]
        for u in _times(kn):
            span, N = oracle_mod.basis(kn, u)
            Nh, Nd, Ndd = np.zeros(4), np.zeros(4), np.zeros(4)
            lib.host_ders_basis(_P(kn), span, u, _P(Nh), _P(Nd), _P(Ndd))
            np.testing.assert_array_equal(Nh, N)
            idx = range(span - 3, span + 1)
            ref1 = np.array([float(d1[j](u)) for j in idx])
            ref2 = np.array([float(d2[j](u)) for j in idx])
            assert np.abs(Nd - ref1).max() <= 1e-12 * np.abs(ref1).max(), (seed, u, Nd - ref1)
            assert np.abs(Ndd - ref2).max() <= 1e-12 * np.abs(ref2).max(), (seed, u, Ndd - ref2)
            # every other basis function has zero derivatives at u: the four carry the whole sum
            assert abs(sum(float(d1[j](u)) for j in range(N_CP)) - Nd.sum()) <= 1e-12 * np.abs(ref1).max()


@pytest.mark.parametrize("so3", [0, 1])
def test_velocity_acceleration_against_finite_differences(oracle_mod, so3):
    """v_w and a_w against central differences of the position sum N_j(t) T_j (scipy BSpline, which extrapolates the end
    spans past the first and last knot).  v: h = 1e-5, truncation h^2 |p'''| / 6 ~ 1e-9 and rounding eps |p| / h ~ 1e-11,
    tolerance 1e-7 of |v|max.  a: h = 1e-4; inside a span p is cubic, but across an interior knot p''' jumps and the central
    second difference is off by ~ h |jump p'''| / 6 ~ 1e-3 of |a| (knot spacing ~ 0.2), rounding 4 eps |p| / h^2 ~ 1e-8:
    tolerance 3e-3 of |a|max at interior knots, 1e-6 elsewhere."""
    lib = _lib()
    for seed in range(3):
        kn, rot, trans = _spline(oracle_mod, so3, seed)
        pos = BSpline(kn, trans, 3)
        for u in _times(kn):
            r = _motion(lib, oracle_mod, kn, rot, trans, u, so3)
            v, a = r["m"][10:13], r["m"][13:16]
            h = 1e-5
            v_fd = (pos(u + h) - pos(u - h)) / (2 * h)
            assert np.abs(v - v_fd).max() <= 1e-7 * max(1.0, np.abs(v).max()), (seed, u, v - v_fd)
            h = 1e-4
            a_fd = (pos(u + h) - 2 * pos(u) + pos(u - h)) / h ** 2
            on_knot = kn[0] < u < kn[-1] and np.isin(u, kn)
            tol = 3e-3 if on_knot else 1e-6
            assert np.abs(a - a_fd).max() <= tol * max(1.0, np.abs(a).max()), (seed, u, a - a_fd)


@pytest.mark.parametrize("so3", [0, 1])
@pytest.mark.parametrize("flat", [False, True])
def test_angular_velocity_against_finite_differences(oracle_mod, so3, flat):
    """w_b against Log(R(t-h)^T R(t+h)) / 2h (symmetric: error h^2 |w''| / 6 ~ 1e-9 at h = 1e-5, rounding eps / h ~ 1e-11); at
    the first and last knot, where t -/+ h leaves the spline, Log(R(t)^T R(t+h)) / h one-sided (error h |w'| / 2 ~ 1e-6 at
    h = 1e-7, rounding eps / h ~ 1e-9).  Tolerances 1e-7 and 2e-5 of max(1, |w|)."""
    lib = _lib()
    for seed in range(3):
        kn, rot, trans = _spline(oracle_mod, so3, seed, flat=flat)
        for u in _times(kn):
            w = _motion(lib, oracle_mod, kn, rot, trans, u, so3)["m"][7:10]
            if u == kn[0] or u == kn[-1]:
                h = 1e-7 if u == kn[0] else -1e-7
                R0, R1 = _rotation_np(kn, rot, u, so3, oracle_mod), _rotation_np(kn, rot, u + h, so3, oracle_mod)
                w_fd, tol = (R0.inv() * R1).as_rotvec() / h, 2e-5
            else:
                h = 1e-5
                R0, R1 = _rotation_np(kn, rot, u - h, so3, oracle_mod), _rotation_np(kn, rot, u + h, so3, oracle_mod)
                w_fd, tol = (R0.inv() * R1).as_rotvec() / (2 * h), 1e-7
            assert np.abs(w - w_fd).max() <= tol * max(1.0, np.abs(w).max()), (so3, flat, seed, u, w - w_fd)


@pytest.mark.parametrize("so3", [0, 1])
@pytest.mark.parametrize("flat", [False, True])
def test_motion_jacobian_against_finite_differences(oracle_mod, so3, flat):
    """the 9 x 24 J against central differences of (w_b, v_w, a_w) along each control point's tangent (the Plus of the rotation
    model for rotations, additive for translations), h = 1e-6: truncation h^2 |d^3 w| ~ 1e-12, rounding eps |w| / h ~ 1e-10,
    tolerance 1e-7 of |J|max.  The translation rows are Nd_j I3 and Ndd_j I3 exactly; w_b has no translation part."""
    lib = _lib()
    plus = oracle_mod.so3_plus if so3 else oracle_mod.quat_plus
    h = 1e-6
    for seed in range(3):
        kn, rot, trans = _spline(oracle_mod, so3, seed, flat=flat)
        for u in _times(kn):
            r = _motion(lib, oracle_mod, kn, rot, trans, u, so3, want_J=True)
            J, Q, T = r["J"], r["Q"], r["T"]
            fd = np.zeros((9, 24))
            for j in range(4):
                for k in range(6):
                    out = []
                    for sgn in (1.0, -1.0):
                        Qp, Tp = Q.copy(), T.copy()
                        d = np.zeros(3)
                        d[k % 3] = sgn * h
                        if k < 3:
                            Qp[j] = plus(Q[j], d)
                        else:
                            Tp[j] = T[j] + d
                        m = np.zeros(16)
                        lib.host_motion(_P(Qp), _P(Tp), _P(r["Nh"]), _P(r["Nd"]), _P(r["Ndd"]), so3, _P(m), None)
                        out.append(m[7:16])
                    fd[:, 6 * j + k] = (out[0] - out[1]) / (2 * h)
            err = np.abs(J - fd).max()
            assert err <= 1e-7 * np.abs(J).max(), (so3, flat, seed, u, err)
            for j in range(4):
                np.testing.assert_array_equal(J[3:6, 6 * j + 3:6 * j + 6], r["Nd"][j] * np.eye(3))
                np.testing.assert_array_equal(J[6:9, 6 * j + 3:6 * j + 6], r["Ndd"][j] * np.eye(3))
                assert not J[:3, 6 * j + 3:6 * j + 6].any() and not J[3:, 6 * j:6 * j + 3].any()


@pytest.mark.parametrize("so3", [0, 1])
def test_motion_pose_is_pose_eval(oracle_mod, so3):
    """the pose columns equal ecb_pose_eval at the port's basis, bit for bit"""
    lib = _lib()
    for seed in range(3):
        for flat in (False, True):
            kn, rot, trans = _spline(oracle_mod, so3, seed, flat=flat)
            for u in _times(kn):
                r = _motion(lib, oracle_mod, kn, rot, trans, u, so3)
                pose = np.zeros(7)
                lib.host_pose_eval(_P(r["Q"]), _P(r["T"]), _P(np.ascontiguousarray(r["N"])), so3, _P(pose))
                np.testing.assert_array_equal(r["m"][:7], pose)
