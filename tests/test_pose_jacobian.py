"""The pose and 6 x 24 pose Jacobian of eventcalib_b200/csrc/ecb_pose.h (host build) for both rotation models: the Jacobian
against central finite differences of a numpy restatement of the spline pose, perturbed along each control point's tangent
(oracle.quat_plus / oracle.so3_plus, translation additive) and mapped back with Log(R^T R) and t - t^; the pose against
EventCalibSpline::evaluate.  Times: the first knot, the last knot, exactly on an interior knot, inside a span."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_CP = 8


def _lib():
    so = os.path.join(ROOT, "tests", "_build", "libpose_host.so")
    os.makedirs(os.path.dirname(so), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", so,
                           os.path.join(ROOT, "tests", "helpers", "pose_host.cpp")])
    lib = C.CDLL(so)
    lib.host_pose_jacobian.restype = None
    return lib


def _facade():
    import eventcalib_b200.build as b
    b.build()
    so = os.path.join(ROOT, "tests", "_build", "libfacade_host.so")
    os.makedirs(os.path.dirname(so), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so,
                           os.path.join(ROOT, "tests", "helpers", "facade_host.cpp"),
                           "-L" + os.path.join(ROOT, "eventcalib_b200"), "-lecb",
                           "-Wl,-rpath," + os.path.join(ROOT, "eventcalib_b200")])
    return C.CDLL(so)


def _P(a):
    return np.ascontiguousarray(a, np.float64).ctypes.data_as(C.c_void_p)


def _spline(oracle_mod, so3, seed):
    """clamped cubic knots over [5, 6]; rotation control points along a smooth curve (unit for SO(3), norms 0.9 .. 1.1 for the
    quaternion model, whose spline normalises), translations random"""
    rng = np.random.default_rng(seed)
    us = np.sort(rng.uniform(5.0, 6.0, 40))
    us[0], us[-1] = 5.0, 6.0
    kn = oracle_mod.knots(us, N_CP)
    rv = np.cumsum(rng.normal(0.0, 0.25, (N_CP, 3)), axis=0)
    rot = Rotation.from_rotvec(rv).as_quat()
    rot *= np.sign(rot[:, 3:4])
    for k in range(1, N_CP):   # one sign per quaternion: a continuous curve
        if rot[k] @ rot[k - 1] < 0:
            rot[k] = -rot[k]
    if not so3:
        rot *= rng.uniform(0.9, 1.1, (N_CP, 1))
    trans = rng.normal(0.0, 0.5, (N_CP, 3))
    return kn, rot, trans


def _pose_np(Q, T, N, so3):
    """restatement of the spline pose: (Rotation, translation)"""
    t = N @ T
    if not so3:
        return Rotation.from_quat(N @ Q), t
    beta = np.cumsum(N[::-1])[::-1][1:]   # cumulative basis b1 .. b3
    R = Rotation.from_quat(Q[0])
    for j in range(1, 4):
        rel = Rotation.from_quat(Q[j - 1]).inv() * Rotation.from_quat(Q[j])
        R = R * Rotation.from_rotvec(beta[j - 1] * rel.as_rotvec())
    return R, t


def _times(kn):
    rng = np.random.default_rng(7)
    return [kn[0], kn[-1], kn[5], 0.5 * (kn[4] + kn[5]) + 0.1 * (kn[5] - kn[4]) * rng.uniform()]


@pytest.mark.parametrize("so3", [0, 1])
def test_pose_jacobian_against_finite_differences(oracle_mod, so3):
    lib = _lib()
    plus = oracle_mod.so3_plus if so3 else oracle_mod.quat_plus
    h = 1e-6
    for seed in range(3):
        kn, rot, trans = _spline(oracle_mod, so3, seed)
        for u in _times(kn):
            span, N = oracle_mod.basis(kn, u)
            Q, T = rot[span - 3:span + 1].copy(), trans[span - 3:span + 1].copy()
            pose, J = np.zeros(7), np.zeros((6, 24))
            lib.host_pose_jacobian(_P(Q), _P(T), _P(N), so3, pose.ctypes.data_as(C.c_void_p), J.ctypes.data_as(C.c_void_p))
            R0, t0 = _pose_np(Q, T, N, so3)
            assert np.abs(pose[:3] - t0).max() <= 1e-13 * max(1.0, np.abs(t0).max())
            assert min(np.abs(pose[3:] - R0.as_quat()).max(), np.abs(pose[3:] + R0.as_quat()).max()) <= 1e-13
            fd = np.zeros((6, 24))
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
                        R, t = _pose_np(Qp, Tp, N, so3)
                        out.append(np.r_[(R0.inv() * R).as_rotvec(), t - t0])
                    fd[:, 6 * j + k] = (out[0] - out[1]) / (2 * h)
            err = np.abs(J - fd).max()
            assert err <= 1e-7 * np.abs(J).max(), (so3, seed, u, err)
            # translation rows are N_j I3 exactly, rotation rows have no translation part
            for j in range(4):
                np.testing.assert_array_equal(J[3:, 6 * j + 3:6 * j + 6], N[j] * np.eye(3))
                assert not J[:3, 6 * j + 3:6 * j + 6].any() and not J[3:, 6 * j:6 * j + 3].any()


@pytest.mark.parametrize("so3", [0, 1])
def test_pose_matches_evaluate(oracle_mod, so3):
    lib, fh = _lib(), _facade()
    for seed in range(3):
        kn, rot, trans = _spline(oracle_mod, so3, seed)
        for u in _times(kn):
            span, N = oracle_mod.basis(kn, u)
            pose, J = np.zeros(7), np.zeros((6, 24))
            lib.host_pose_jacobian(_P(rot[span - 3:span + 1]), _P(trans[span - 3:span + 1]), _P(N), so3,
                                   pose.ctypes.data_as(C.c_void_p), J.ctypes.data_as(C.c_void_p))
            q4, t3 = np.zeros(4), np.zeros(3)
            assert fh.fh_eval(_P(kn), N_CP, _P(rot), _P(trans), so3, C.c_double(u), q4.ctypes.data_as(C.c_void_p),
                              t3.ctypes.data_as(C.c_void_p)) == 1
            ref = np.r_[t3, q4]
            assert np.abs(pose - ref).max() <= 1e-13 * np.abs(ref).max(), (so3, u, pose - ref)
