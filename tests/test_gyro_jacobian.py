"""The angular acceleration of ecb_motion.h and the gyroscope residual of ecb_gyro.h (host build, -ffp-contract=off), for both
rotation models, on the splines of test_motion_jacobian.py (quaternion control points of norms != 1; for SO(3) also a run of
near-identical control points, the small-angle branch of Log / Exp):
- dw/dt against central differences of w, at the first and last knot, exactly on interior knots and inside spans;
- w of ecb_angular_velocity, with and without dw/dt, bit for bit the w of ecb_motion_eval;
- the 3 x 7 Jacobian of r = R_gc w_c(t + d) + b - w_g against finite differences, R_gc perturbed as Exp(delta) R_gc;
- the ctypes result struct against the header's layout."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

from test_motion_jacobian import _lib as _motion_lib, _motion, _spline, _times

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    so = os.path.join(ROOT, "tests", "_build", "libgyro_host.so")
    os.makedirs(os.path.dirname(so), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", so,
                           os.path.join(ROOT, "tests", "helpers", "gyro_host.cpp")])
    lib = C.CDLL(so)
    lib.host_angular_velocity.restype = lib.host_gyro_residual.restype = None
    lib.host_angular_velocity.argtypes = [C.c_void_p] * 4 + [C.c_int] + [C.c_void_p] * 3
    lib.host_gyro_residual.argtypes = [C.c_void_p] * 7
    return lib


def _P(a):
    return a.ctypes.data_as(C.c_void_p)


def _omega(glib, mlib, oracle_mod, kn, rot, trans, u, so3):
    """(w, dw/dt, w without dw/dt, ecb_motion_eval's w) at u"""
    r = _motion(mlib, oracle_mod, kn, rot, trans, u, so3)
    w, wd, w1 = np.zeros(3), np.zeros(3), np.zeros(3)
    glib.host_angular_velocity(_P(r["Q"]), _P(r["Nh"]), _P(r["Nd"]), _P(r["Ndd"]), so3, _P(w), _P(wd), _P(w1))
    return w, wd, w1, r["m"][7:10]


@pytest.mark.parametrize("so3", [0, 1])
@pytest.mark.parametrize("flat", [False, True])
def test_angular_acceleration_against_finite_differences(oracle_mod, so3, flat):
    """dw/dt against (w(t+h) - w(t-h)) / 2h inside spans, h = 1e-5 (truncation h^2 |w'''| / 6 ~ 1e-8, rounding eps |w| / h ~
    1e-10).  On a knot w'' jumps, so a symmetric difference is off by h |jump w''| / 4; there each side that lies on the spline
    is checked with the one-sided s (-3 w(t) + 4 w(t+sh) - w(t+2sh)) / 2h, which sees one polynomial piece only (error
    h^2 |w'''| / 3): dw/dt is continuous, so both sides agree with it.  Tolerance 1e-6 of max(1, |dw/dt|)."""
    glib, mlib = _lib(), _motion_lib()
    h = 1e-5
    for seed in range(3):
        kn, rot, trans = _spline(oracle_mod, so3, seed, flat=flat)

        def w_at(u):
            return _omega(glib, mlib, oracle_mod, kn, rot, trans, u, so3)[0]

        for u in _times(kn):
            _, wd, _, _ = _omega(glib, mlib, oracle_mod, kn, rot, trans, u, so3)
            if u in kn:
                sides = [s for s in (1.0, -1.0) if kn[0] <= u + 2 * s * h <= kn[-1]]
                fds = [s * (-3 * w_at(u) + 4 * w_at(u + s * h) - w_at(u + 2 * s * h)) / (2 * h) for s in sides]
            else:
                fds = [(w_at(u + h) - w_at(u - h)) / (2 * h)]
            for fd in fds:
                assert np.abs(wd - fd).max() <= 1e-6 * max(1.0, np.abs(wd).max()), (so3, flat, seed, u, wd - fd)


@pytest.mark.parametrize("so3", [0, 1])
def test_angular_velocity_is_motion_eval(oracle_mod, so3):
    """w of ecb_angular_velocity, with and without the derivative, bit for bit ecb_motion_eval's"""
    glib, mlib = _lib(), _motion_lib()
    for seed in range(3):
        for flat in (False, True):
            kn, rot, trans = _spline(oracle_mod, so3, seed, flat=flat)
            for u in _times(kn):
                w, _, w1, ref = _omega(glib, mlib, oracle_mod, kn, rot, trans, u, so3)
                np.testing.assert_array_equal(w, ref)
                np.testing.assert_array_equal(w1, ref)


@pytest.mark.parametrize("so3", [0, 1])
def test_gyro_residual_jacobian_against_finite_differences(oracle_mod, so3):
    """r(delta, d, b) = Exp(delta) R_gc w_c(t + d) + b - w_g with w_c from the spline: the analytic J = [-[R w_c]x, R dw_c/dt, I3]
    against central differences, h = 1e-6 (rotation and bias: exact up to rounding eps |w| / h ~ 1e-10; offset: truncation
    h^2 |w'''| / 6).  Tolerance 1e-7 of max(1, |J|max).  The residual itself is R_gc w_c + b - w_g."""
    glib, mlib = _lib(), _motion_lib()
    rng = np.random.default_rng(11)
    h = 1e-6
    for seed in range(3):
        kn, rot, trans = _spline(oracle_mod, so3, seed)
        for u in [u for u in _times(kn) if u not in kn]:   # inside spans: w_c is smooth over t + d +- h
            q = Rotation.from_rotvec(rng.normal(0.0, 1.5, 3)).as_quat()
            b, wg = rng.normal(0.0, 0.05, 3), rng.normal(0.0, 1.0, 3)

            def res(delta, d, bb, want_J=False):
                w, wd, _, _ = _omega(glib, mlib, oracle_mod, kn, rot, trans, u + d, so3)
                qq = np.ascontiguousarray((Rotation.from_rotvec(delta) * Rotation.from_quat(q)).as_quat())
                r, J = np.zeros(3), np.zeros((3, 7))
                glib.host_gyro_residual(_P(qq), _P(np.ascontiguousarray(bb)), _P(w), _P(wd), _P(wg), _P(r),
                                        _P(J) if want_J else None)
                return r, J, w

            r0, J, w = res(np.zeros(3), 0.0, b, True)
            np.testing.assert_allclose(r0, Rotation.from_quat(q).apply(w) + b - wg, rtol=0, atol=1e-13 * max(1.0, np.abs(w).max()))
            fd = np.zeros((3, 7))
            for k in range(7):
                e = np.zeros(7)
                e[k] = h
                rp = res(e[:3], e[3], b + e[4:])[0]
                rm = res(-e[:3], -e[3], b - e[4:])[0]
                fd[:, k] = (rp - rm) / (2 * h)
            assert np.abs(J - fd).max() <= 1e-7 * max(1.0, np.abs(J).max()), (so3, seed, u, J - fd)
            np.testing.assert_array_equal(J[:, 4:], np.eye(3))


def test_gyro_struct_matches_header(tmp_path):
    """the ctypes GyroCalibration has the size and field offsets of the header's ecb_gyro_calibration"""
    import eventcalib_b200 as ecb
    src = tmp_path / "size.c"
    fields = [f[0] for f in ecb.GyroCalibration._fields_]
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "eventcalib_b200.h"\nint main(void) {\n'
                   '    printf("%zu", sizeof(ecb_gyro_calibration));\n'
                   + "".join('    printf(" %%zu", offsetof(ecb_gyro_calibration, %s));\n' % f for f in fields) + "    return 0;\n}\n")
    exe = tmp_path / "size"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(v) for v in subprocess.check_output([str(exe)], text=True).split()]
    assert got == [C.sizeof(ecb.GyroCalibration)] + [getattr(ecb.GyroCalibration, f).offset for f in fields]
