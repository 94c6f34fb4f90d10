"""The outlier policy of the C++ façade (ecb::outlierRejection, host build): s = the lower median of the key frames' RMS over the
key frames with records, key frames with RMS > k s dropped, record threshold k s."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def policy_lib():
    import eventcalib_b200.build as b
    b.build()
    so = os.path.join(ROOT, "tests", "_build", "liboutlier_policy_host.so")
    os.makedirs(os.path.dirname(so), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so,
                           os.path.join(ROOT, "tests", "helpers", "outlier_policy_host.cpp"),
                           "-L" + os.path.join(ROOT, "eventcalib_b200"), "-lecb",
                           "-Wl,-rpath," + os.path.join(ROOT, "eventcalib_b200")])
    lib = C.CDLL(so)
    lib.host_outlier_policy.restype = C.c_double
    lib.host_outlier_policy.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_void_p]
    return lib


@pytest.fixture(scope="module")
def lib():
    return policy_lib()


def apply_policy(lib, groups, k):
    """ecb::outlierRejection on residual_groups(by="keyframe") output: (s, threshold, drop)"""
    g = np.ascontiguousarray(groups)
    thr = C.c_double(0.0)
    drop = np.zeros(max(len(g), 1), np.uint8)
    s = lib.host_outlier_policy(g.ctypes.data_as(C.c_void_p), len(g), float(k), C.byref(thr), drop.ctypes.data_as(C.c_void_p))
    return s, thr.value, drop[:len(g)]


def _policy(lib, count, rms, k):
    """groups with the given counts and RMS (sum_sq = count rms^2); returns (s, threshold, drop)"""
    import eventcalib_b200 as ecb
    count = np.asarray(count, np.int64)
    g = np.zeros(len(count), ecb.RESIDUAL_GROUP_DTYPE)
    g["count"] = count
    g["sum_sq"] = count * np.asarray(rms, float) ** 2
    return apply_policy(lib, g, k)


def test_lower_median_odd_and_even(lib):
    # odd: 5 frames, median element 2 of the sorted RMS
    s, t, d = _policy(lib, [4, 4, 4, 4, 4], [0.5, 0.1, 0.3, 0.2, 0.4], 2.0)
    assert s == 0.3 and t == 0.6 and list(d) == [0, 0, 0, 0, 0]
    # even: 4 frames, the LOWER median (element 1 of 4), not the mean of the middle two
    s, t, d = _policy(lib, [4, 4, 4, 4], [0.4, 0.1, 0.3, 0.2], 1.5)
    assert s == 0.2 and t == pytest.approx(0.3, abs=0, rel=1e-15)
    assert list(d) == [1, 0, int(0.3 > t), 0]


def test_empty_keyframes_are_ignored(lib):
    # the empty frames would make the lower median 0 if they took part; they are never dropped either
    s, t, d = _policy(lib, [0, 0, 0, 5, 5, 5], [0, 0, 0, 0.2, 0.1, 0.3], 3.0)
    assert s == 0.2 and t == pytest.approx(0.6, rel=1e-15)
    assert list(d) == [0, 0, 0, 0, 0, 0]
    s, t, d = _policy(lib, [0, 0], [0, 0], 3.0)   # no records at all
    assert s == 0.0 and t == 0.0 and list(d) == [0, 0]


def test_tie_at_threshold_is_kept(lib):
    # RMS exactly k s: kept (the comparison is strictly greater)
    s, t, d = _policy(lib, [1, 1, 1], [1.0, 2.0, 3.0], 1.5)
    assert s == 2.0 and t == 3.0 and list(d) == [0, 0, 0]
    s, t, d = _policy(lib, [1, 1, 1], [1.0, 2.0, np.nextafter(3.0, 4.0)], 1.5)
    assert list(d) == [0, 0, 1]


def test_one_huge_record_drops_its_frame(lib):
    # 9 frames of 200 records at RMS 0.1; one frame holds 199 such records and one of 50: its RMS is 3.6, far above 3 x 0.1
    count = [200] * 9
    rms = [0.1] * 9
    big = np.sqrt((199 * 0.01 + 50.0 ** 2) / 200)
    rms[4] = big
    s, t, d = _policy(lib, count, rms, 3.0)
    assert s == pytest.approx(0.1, rel=1e-15) and list(d) == [0, 0, 0, 0, 1, 0, 0, 0, 0]


def test_all_frames_equal_drop_none(lib):
    s, t, d = _policy(lib, [3] * 7, [0.25] * 7, 1.0)
    assert s == 0.25 and t == 0.25 and not np.any(d)
