"""The forward camera model of eventcalib_b200/csrc/ecb_camera.h (host build): the fold of the inverse radial polynomial against
numpy's roots, the pixel -> inverse polynomial -> distort -> pixel round trip on every pixel of the DAVIS346 sensor, the invalid
range past the fold, and the exact cases k = 0 and rho_u = 0.  Two cameras: the synthetic one and the sample result of the
reference (parameter/cvcalib/example.xml:60-67), whose polynomial folds 2 % outside the sensor's corner (345, 0), where the
fixed-point iteration of OpenCV-style undistortion fails by more than 20 px."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, H = 346, 260
EXAMPLE = np.array([367.862391528, 368.850785864, 168.446433308, 138.747524029,
                    0.227345275939, 2.56983530177, -20.0008686649, 77.8547449903, -112.37955919])


@pytest.fixture(scope="module")
def lib():
    so = os.path.join(ROOT, "tests", "_build", "libcamera_host.so")
    os.makedirs(os.path.dirname(so), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", so,
                           os.path.join(ROOT, "tests", "helpers", "camera_host.cpp")])
    lib = C.CDLL(so)
    lib.host_fold.restype = None
    lib.host_distort_radius.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_int, C.c_void_p]
    lib.host_project.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    return lib


def _P(a):
    return a.ctypes.data_as(C.c_void_p)


def _synthetic():
    from eventcalib_b200 import synth
    return synth.Camera().intrinsics()


CAMERAS = {"synthetic": _synthetic, "example": lambda: EXAMPLE.copy()}


def _fold(lib, k):
    k = np.ascontiguousarray(k, np.float64)
    rho, g = C.c_double(), C.c_double()
    lib.host_fold(_P(k), C.byref(rho), C.byref(g))
    return rho.value, g.value


def _fold_numpy(k):
    """smallest positive real root of h(u) = 1 + 3 k1 u + ... + 11 k5 u^5, as rho = sqrt(u)"""
    h = np.array([1.0] + [(2 * i + 3) * k[i] for i in range(5)])
    r = np.roots(h[::-1])
    r = r[(np.abs(r.imag) <= 1e-12 * np.abs(r)) & (r.real > 0)].real
    return np.sqrt(r.min()) if len(r) else np.inf


def _g(k, rho):
    u = rho * rho
    return rho * (1 + u * (k[0] + u * (k[1] + u * (k[2] + u * (k[3] + u * k[4])))))


def _project(lib, intr, p):
    p = np.ascontiguousarray(p, np.float64)
    uv = np.zeros((len(p), 2))
    nv = lib.host_project(_P(intr), _P(p), len(p), _P(uv))
    return uv, nv


@pytest.mark.parametrize("cam", list(CAMERAS))
def test_fold_against_numpy_roots(lib, cam):
    intr = CAMERAS[cam]()
    k = intr[4:]
    rho, g = _fold(lib, k)
    ref = _fold_numpy(k)
    if cam == "example":
        assert abs(rho - 0.6237) < 1e-4   # the reference's sample result folds at rho_d = 0.6237
    if np.isfinite(ref):
        assert abs(rho - ref) <= 1e-12 * ref, (rho, ref)
        assert g == _g(k, rho)
    else:
        assert rho == np.inf and g == np.inf
    # more cases: random polynomials, with and without a positive root, and lower degrees
    rng = np.random.default_rng(1)
    for _ in range(200):
        kk = rng.normal(0, 1, 5) * rng.choice([0.0, 1.0, 10.0], 5)
        rho, _ = _fold(lib, kk)
        ref = _fold_numpy(kk)
        if np.isfinite(ref):
            assert abs(rho - ref) <= 1e-9 * ref, (kk, rho, ref)
        else:
            assert rho == np.inf, (kk, rho)
    assert _fold(lib, np.zeros(5)) == (np.inf, np.inf)


def _fixed_point(k, xu, yu, iters):
    xd, yd = xu.copy(), yu.copy()
    for _ in range(iters):
        u = xd * xd + yd * yd
        s = 1 + u * (k[0] + u * (k[1] + u * (k[2] + u * (k[3] + u * k[4]))))
        xd, yd = xu / s, yu / s
    return xd, yd


@pytest.mark.parametrize("cam", list(CAMERAS))
def test_round_trip_every_pixel(lib, cam):
    intr = CAMERAS[cam]()
    fx, fy, cx, cy, k = intr[0], intr[1], intr[2], intr[3], intr[4:]
    v, u = np.mgrid[0:H, 0:W].astype(np.float64)
    u, v = u.ravel(), v.ravel()
    assert {(0.0, 0.0), (W - 1.0, 0.0), (0.0, H - 1.0), (W - 1.0, H - 1.0)} <= set(zip(u, v))
    xd, yd = (u - cx) / fx, (v - cy) / fy
    r2 = xd * xd + yd * yd
    s = 1 + r2 * (k[0] + r2 * (k[1] + r2 * (k[2] + r2 * (k[3] + r2 * k[4]))))
    rho, _ = _fold(lib, k)
    assert np.sqrt(r2).max() < rho    # the whole sensor is inside the fold
    for depth in (1.0, 37.5):
        p = np.stack([xd * s * depth, yd * s * depth, np.full_like(xd, depth)], 1)
        uv, nv = _project(lib, intr, p)
        assert nv == len(p)
        err = np.hypot(uv[:, 0] - u, uv[:, 1] - v)
        assert err.max() <= 1e-9, (cam, err.max(), u[err.argmax()], v[err.argmax()])
    if cam == "example":   # the corners where the fixed-point iteration fails
        for px in ((0.0, 0.0), (345.0, 0.0)):
            i = int(np.nonzero((u == px[0]) & (v == px[1]))[0][0])
            fxd, fyd = _fixed_point(k, np.array([xd[i] * s[i]]), np.array([yd[i] * s[i]]), 200)
            assert np.hypot(fx * fxd[0] + cx - px[0], fy * fyd[0] + cy - px[1]) > 20.0


@pytest.mark.parametrize("cam", list(CAMERAS))
def test_invalid_past_the_fold(lib, cam):
    intr = CAMERAS[cam]()
    k = np.ascontiguousarray(intr[4:])
    rho, g = _fold(lib, k)
    if not np.isfinite(rho):   # scale k5 until the synthetic camera folds (a larger k5 magnitude with the sign that folds)
        k = k.copy()
        k[4] = -abs(k[4]) * 50 - 1.0
        rho, g = _fold(lib, k)
    assert np.isfinite(rho) and np.isfinite(g)
    ru = np.array([0.0, 0.5 * g, g * (1 - 1e-12), g, np.nextafter(g, np.inf), 2 * g, np.inf, np.nan, -1e-3])
    rd = np.zeros(len(ru))
    nv = lib.host_distort_radius(_P(k), rho, g, _P(ru), len(ru), _P(rd))
    assert nv == 3
    assert np.all(np.isnan(rd[3:]))
    assert rd[0] == 0.0 and 0 < rd[1] < rd[2] < rho
    assert abs(_g(k, rd[1]) - ru[1]) <= 1e-15 and abs(_g(k, rd[2]) - ru[2]) <= 1e-14
    # a camera-frame point whose undistorted radius is past the fold, or behind / on the camera plane, is not projectable
    ip = np.r_[intr[:4], k]
    pts = np.array([[1.01 * g, 0.0, 1.0], [0.0, 3.0 * g, 1.0], [0.1, 0.1, 0.0], [0.1, 0.1, -1.0], [np.nan, 0.0, 1.0],
                    [0.5 * g, 0.0, 1.0]])
    uv, nv = _project(lib, ip, pts)
    assert nv == 1 and np.all(np.isnan(uv[:5])) and np.all(np.isfinite(uv[5]))


def test_exact_cases(lib):
    intr = np.array([300.0, 310.0, 170.0, 130.0, 0.0, 0.0, 0.0, 0.0, 0.0])
    rng = np.random.default_rng(3)
    ru = np.r_[0.0, rng.uniform(0, 3, 1000), 1e-300, 1e100]
    rd = np.zeros(len(ru))
    assert lib.host_distort_radius(_P(intr[4:].copy()), np.inf, np.inf, _P(ru), len(ru), _P(rd)) == len(ru)
    assert np.array_equal(rd, ru)   # k = 0: rho_d = rho_u exactly
    p = np.c_[rng.uniform(-1, 1, (1000, 2)), rng.uniform(0.5, 2, 1000)]
    uv, nv = _project(lib, intr, p)
    assert nv == len(p)
    assert np.array_equal(uv[:, 0], intr[0] * (p[:, 0] / p[:, 2]) + intr[2])
    assert np.array_equal(uv[:, 1], intr[1] * (p[:, 1] / p[:, 2]) + intr[3])
    for cam in CAMERAS.values():   # rho_u = 0: the principal point, exactly
        c = cam()
        uv, nv = _project(lib, c, np.array([[0.0, 0.0, 2.0]]))
        assert nv == 1 and uv[0, 0] == c[2] and uv[0, 1] == c[3]
        rd = np.ones(1)
        rho, g = _fold(lib, c[4:])
        assert lib.host_distort_radius(_P(c[4:].copy()), rho, g, _P(np.zeros(1)), 1, _P(rd)) == 1 and rd[0] == 0.0
