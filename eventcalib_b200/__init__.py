"""eventcalib_b200 — Python mirror of the C ABI in ``include/eventcalib_b200.h``.

The product is the CUDA library ``libecb.so`` (built in-tree by ``eventcalib_b200.build``); this module only
binds it with ctypes for the tests, ``bench.py`` and ``__graft_entry__``.  There is no CPU fallback: if the
library is missing or no CUDA device is present, every compute call raises.
"""
import ctypes as C
import math
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libecb.so")

OK, FAILED, ERR_CUDA, ERR_ARG, ERR_UNSUPPORTED, ERR_STATE = 0, 1, -1, -2, -3, -4
PB_DUPLICATE, PB_CLUSTER_CAP, PB_RANGE = 2, 4, 8


class EcbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("ecb error %d: %s" % (code, msg))
        self.code = code


class FrontendParams(C.Structure):
    _fields_ = [("dbscan_eps", C.c_double), ("dbscan_min_pts", C.c_uint32), ("cluster_min", C.c_uint32),
                ("knn_num", C.c_int32), ("fit_circle", C.c_int32), ("radius_threshold", C.c_double),
                ("rows_cols", C.c_uint32), ("order_mode", C.c_int32), ("max_clusters", C.c_uint32),
                ("median_mode", C.c_uint32)]


class LmOptions(C.Structure):
    _fields_ = [("max_iterations", C.c_int32), ("jacobi_scaling", C.c_int32), ("fixed_iterations", C.c_int32),
                ("rotation_model", C.c_int32), ("function_tolerance", C.c_double), ("gradient_tolerance", C.c_double),
                ("parameter_tolerance", C.c_double), ("initial_radius", C.c_double), ("max_radius", C.c_double),
                ("min_radius", C.c_double), ("min_relative_decrease", C.c_double), ("min_lm_diagonal", C.c_double),
                ("max_lm_diagonal", C.c_double)]


class LmSummary(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("successful_steps", C.c_int32), ("termination", C.c_int32),
                ("reserved", C.c_int32), ("initial_cost", C.c_double), ("final_cost", C.c_double),
                ("gradient_max_norm", C.c_double), ("radius", C.c_double)]


class WindowSummary(C.Structure):
    _fields_ = [("ev_lo", C.c_int64), ("ev_hi", C.c_int64), ("n_points", C.c_int32 * 2), ("n_clusters", C.c_int32 * 2),
                ("n_kept", C.c_int32 * 2), ("n_candidates", C.c_int32), ("status", C.c_uint32),
                ("point_offset", C.c_int64 * 2)]


class CovarianceSummary(C.Structure):
    _fields_ = [("cost", C.c_double), ("sigma2", C.c_double), ("min_relative_pivot", C.c_double), ("n_residuals", C.c_int64),
                ("dimension", C.c_int32), ("deficient_index", C.c_int32)]


class GyroCalibration(C.Structure):
    """ecb_gyro_calibration: camera-gyroscope rotation, time offset and bias with their covariance"""
    _fields_ = [("q_gc", C.c_double * 4), ("offset", C.c_double), ("bias", C.c_double * 3), ("cov", C.c_double * 49),
                ("std", C.c_double * 7), ("sigma2", C.c_double), ("cost", C.c_double), ("rms", C.c_double),
                ("scan_offset", C.c_double), ("n_used", C.c_int64), ("n_unused", C.c_int64), ("iterations", C.c_int32),
                ("termination", C.c_int32), ("n_params", C.c_int32), ("status", C.c_int32)]


GYRO_OK, GYRO_TOO_FEW_SAMPLES, GYRO_OFFSET_AT_EDGE, GYRO_RANK_DEFICIENT = 0, 1, 2, 3


class ResidualGroup(C.Structure):
    """ecb_residual_group: statistics of a group of raw residuals r (board units, not pixels)"""
    _fields_ = [("count", C.c_int64), ("n_downweighted", C.c_int64), ("sum", C.c_double), ("sum_sq", C.c_double),
                ("max_abs", C.c_double), ("cost", C.c_double)]


RESIDUAL_GROUP_DTYPE = np.dtype([("count", "<i8"), ("n_downweighted", "<i8"), ("sum", "<f8"), ("sum_sq", "<f8"),
                                 ("max_abs", "<f8"), ("cost", "<f8")])
assert RESIDUAL_GROUP_DTYPE.itemsize == C.sizeof(ResidualGroup)
RESIDUALS_BY = {"keyframe": 0, "circle": 1, "sensor_cell": 2}

# ecb_reprojection_group: statistics of a group of reprojection errors e (pixels); count / sum / sum_sq / max_abs over the valid
# records, n_invalid = the records that cannot be projected (NaN)
REPROJECTION_GROUP_DTYPE = np.dtype([("count", "<i8"), ("n_invalid", "<i8"), ("sum", "<f8"), ("sum_sq", "<f8"),
                                     ("max_abs", "<f8")])


# the order of every intrinsics array (ecb_residual.h): bit i of a constant-intrinsics mask is INTRINSIC_NAMES[i].  In the spline
# stage k1 .. k5 are the coefficients of the inverse radial polynomial, not OpenCV's distortion coefficients.
INTRINSIC_NAMES = ("fx", "fy", "cx", "cy", "k1", "k2", "k3", "k4", "k5")


def constant_intrinsics_mask(names):
    """Bit mask of ecb_cost_set_constant_intrinsics from an iterable of INTRINSIC_NAMES (a string: comma- or space-separated
    names); empty means none.  An unknown name raises ValueError."""
    if isinstance(names, str):
        names = names.replace(",", " ").split()
    mask = 0
    for nm in names:
        if nm not in INTRINSIC_NAMES:
            raise ValueError("unknown intrinsic %r (names: %s)" % (nm, " ".join(INTRINSIC_NAMES)))
        mask |= 1 << INTRINSIC_NAMES.index(nm)
    return mask


SUMMARY_DTYPE = np.dtype([("ev_lo", "<i8"), ("ev_hi", "<i8"), ("n_points", "<i4", 2), ("n_clusters", "<i4", 2),
                          ("n_kept", "<i4", 2), ("n_candidates", "<i4"), ("status", "<u4"), ("point_offset", "<i8", 2)])
assert SUMMARY_DTYPE.itemsize == C.sizeof(WindowSummary)

# every symbol include/eventcalib_b200.h declares (checked by tests/test_abi.py)
SYMBOLS = ["ecb_ctx_create", "ecb_ctx_destroy", "ecb_last_error", "ecb_launch_count", "ecb_synchronize", "ecb_version", "ecb_device_count",
           "ecb_set_sensor", "ecb_load_events_host", "ecb_load_events_device", "ecb_num_events", "ecb_frontend_run",
           "ecb_frontend_summary", "ecb_frontend_total_points", "ecb_frontend_points", "ecb_frontend_candidates",
           "ecb_frontend_clusters", "ecb_frontend_rectify", "ecb_frontend_device_ptrs", "ecb_dbscan_run", "ecb_dbscan_run_batch",
           "ecb_dbscan_run_ordered", "ecb_dbscan_run_batch_ordered", "ecb_dbscan_run_nd",
           "ecb_fit_circles", "ecb_set_profiling", "ecb_stage_ms", "ecb_cost_setup", "ecb_cost_set_rotation_model",
           "ecb_cost_set_constant_intrinsics", "ecb_cost_layout",
           "ecb_cost_associate", "ecb_cost_associate_device", "ecb_cost_get_association", "ecb_cost_set_residuals", "ecb_cost_eval", "ecb_cost_normal_eq",
           "ecb_exchange_buffer_bytes", "ecb_cost_normal_eq_exchange", "ecb_device_alloc", "ecb_device_free", "ecb_ipc_export",
           "ecb_ipc_open", "ecb_ipc_close", "ecb_enable_peer_access", "ecb_lm_default_options", "ecb_lm_create",
           "ecb_lm_destroy", "ecb_lm_dimension", "ecb_lm_set_constant_intrinsics", "ecb_lm_begin", "ecb_lm_propose", "ecb_lm_feedback", "ecb_lm_update",
           "ecb_lm_state", "ecb_lm_trace", "ecb_calibrate", "ecb_lm_device_create", "ecb_lm_device_destroy",
           "ecb_lm_device_set_exchange", "ecb_lm_device_begin", "ecb_lm_device_iterate", "ecb_lm_device_running",
           "ecb_lm_device_result", "ecb_calibrate_device", "ecb_covariance", "ecb_pose_covariance",
           "ecb_pose_covariance_device", "ecb_cost_residuals", "ecb_cost_residual_groups", "ecb_cost_reject",
           "ecb_cost_reassociate", "ecb_inverse_radial_fold", "ecb_cost_reprojection_errors", "ecb_cost_reprojection_groups", "ecb_keyframe_reprojection",
           "ecb_trajectory_motion", "ecb_trajectory_motion_device", "ecb_motion_covariance", "ecb_motion_covariance_device",
           "ecb_gyro_calibrate"]

_lib = None


def load_library():
    """Loads libecb.so; raises if the CUDA extension was not built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("ECB_LIBRARY", LIB_PATH)  # A/B builds of the same library (profiles/tools/ab_build.py)
    if not os.path.exists(path):
        raise EcbError(ERR_CUDA, "libecb.so not built (run `python -m eventcalib_b200.build`); there is no CPU fallback")
    lib = C.CDLL(path)
    vp, i32, i64, u32, dbl = C.c_void_p, C.c_int, C.c_int64, C.c_uint32, C.c_double
    lib.ecb_ctx_create.argtypes = [i32, vp, C.POINTER(vp)]
    lib.ecb_ctx_destroy.argtypes = [vp]
    lib.ecb_ctx_destroy.restype = None
    lib.ecb_last_error.argtypes = [vp]
    lib.ecb_last_error.restype = C.c_char_p
    lib.ecb_launch_count.argtypes = [vp]
    lib.ecb_launch_count.restype = C.c_uint64
    lib.ecb_synchronize.argtypes = [vp]
    lib.ecb_version.restype = C.c_char_p
    lib.ecb_set_sensor.argtypes = [vp, i32, i32]
    lib.ecb_load_events_host.argtypes = [vp, vp, i64]
    lib.ecb_load_events_device.argtypes = [vp, vp, i64]
    lib.ecb_num_events.argtypes = [vp]
    lib.ecb_num_events.restype = i64
    lib.ecb_frontend_run.argtypes = [vp, vp, i32, C.POINTER(FrontendParams)]
    lib.ecb_frontend_summary.argtypes = [vp, vp, i32]
    lib.ecb_frontend_total_points.argtypes = [vp, i32]
    lib.ecb_frontend_total_points.restype = i64
    lib.ecb_frontend_points.argtypes = [vp, i32, vp, vp]
    lib.ecb_frontend_candidates.argtypes = [vp, vp, i32]
    lib.ecb_frontend_clusters.argtypes = [vp, i32, i32, vp, vp, vp, i32]
    lib.ecb_frontend_device_ptrs.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(i32)]
    lib.ecb_frontend_rectify.argtypes = [vp, vp, i32, i32, vp, dbl, i32, i32, i32, vp, vp]
    lib.ecb_cost_set_rotation_model.argtypes = [vp, i32]
    lib.ecb_cost_set_constant_intrinsics.argtypes = [vp, u32]
    lib.ecb_exchange_buffer_bytes.argtypes = [vp, i32]
    lib.ecb_exchange_buffer_bytes.restype = C.c_size_t
    lib.ecb_cost_normal_eq_exchange.argtypes = [vp, vp, vp, vp, i32, i32, vp, C.c_uint64, i32, vp, vp]
    lib.ecb_device_alloc.argtypes = [vp, C.c_size_t, C.POINTER(vp)]
    lib.ecb_device_free.argtypes = [vp, vp]
    lib.ecb_ipc_export.argtypes = [vp, vp, vp]
    lib.ecb_ipc_open.argtypes = [vp, vp, C.POINTER(vp)]
    lib.ecb_ipc_close.argtypes = [vp, vp]
    lib.ecb_enable_peer_access.argtypes = [vp, i32]
    lib.ecb_dbscan_run.argtypes = [vp, vp, i32, dbl, u32, vp, C.POINTER(C.c_int32)]
    lib.ecb_dbscan_run_batch.argtypes = [vp, vp, vp, i32, dbl, u32, vp, vp, vp]
    lib.ecb_dbscan_run_ordered.argtypes = [vp, vp, i32, dbl, u32, vp, C.POINTER(C.c_int32), vp, vp]
    lib.ecb_dbscan_run_batch_ordered.argtypes = [vp, vp, vp, i32, dbl, u32, vp, vp, vp, vp, vp]
    lib.ecb_dbscan_run_nd.argtypes = [vp, vp, i32, i32, dbl, u32, vp, C.POINTER(C.c_int32), vp, vp]
    lib.ecb_fit_circles.argtypes = [vp, vp, vp, i32, vp]
    lib.ecb_set_profiling.argtypes = [vp, i32]
    lib.ecb_stage_ms.argtypes = [vp, vp]
    lib.ecb_cost_setup.argtypes = [vp, i32, vp, vp, dbl, dbl]
    lib.ecb_cost_layout.argtypes = [vp, vp, vp, vp, vp]
    lib.ecb_cost_associate.argtypes = [vp, vp, vp, i32, i32, vp, dbl, vp]
    lib.ecb_cost_associate_device.argtypes = [vp, vp, vp, i32, i32, vp, dbl, vp]
    lib.ecb_cost_get_association.argtypes = [vp, vp, vp, i64]
    lib.ecb_cost_set_residuals.argtypes = [vp, vp, vp, vp, vp, i64]
    lib.ecb_cost_eval.argtypes = [vp, vp, vp, vp, vp]
    lib.ecb_cost_normal_eq.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    lib.ecb_cost_residuals.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.ecb_cost_residual_groups.argtypes = [vp, vp, vp, vp, i32, vp, i32, i32, vp, i32, C.POINTER(C.c_int), vp]
    lib.ecb_cost_reject.argtypes = [vp, vp, vp, vp, dbl, vp, vp, i32, C.POINTER(i64), C.POINTER(i64)]
    lib.ecb_cost_reassociate.argtypes = [vp, vp, vp, vp, dbl, dbl] + [C.POINTER(i64)] * 5
    lib.ecb_inverse_radial_fold.argtypes = [vp, C.POINTER(dbl)]
    lib.ecb_cost_reprojection_errors.argtypes = [vp, vp, vp, vp, vp, vp, C.POINTER(i64)]
    lib.ecb_cost_reprojection_groups.argtypes = [vp, vp, vp, vp, i32, vp, i32, i32, vp, i32, C.POINTER(C.c_int), vp]
    lib.ecb_keyframe_reprojection.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, vp, vp, vp, vp]
    lib.ecb_lm_default_options.argtypes = [C.POINTER(LmOptions)]
    lib.ecb_lm_default_options.restype = None
    lib.ecb_lm_create.argtypes = [i32, vp, C.POINTER(LmOptions)]
    lib.ecb_lm_create.restype = vp
    lib.ecb_lm_destroy.argtypes = [vp]
    lib.ecb_lm_destroy.restype = None
    lib.ecb_lm_dimension.argtypes = [vp]
    lib.ecb_lm_set_constant_intrinsics.argtypes = [vp, u32]
    lib.ecb_lm_begin.argtypes = [vp, vp, vp, vp, vp]
    lib.ecb_lm_propose.argtypes = [vp, vp, vp, vp]
    lib.ecb_lm_feedback.argtypes = [vp, dbl]
    lib.ecb_lm_update.argtypes = [vp, vp]
    lib.ecb_lm_state.argtypes = [vp, vp, vp, vp, C.POINTER(LmSummary)]
    lib.ecb_lm_trace.argtypes = [vp, vp, i32]
    lib.ecb_calibrate.argtypes = [vp, i32, vp, vp, vp, vp, C.POINTER(LmOptions), C.POINTER(LmSummary), vp, i32]
    lib.ecb_lm_device_create.argtypes = [vp, i32, vp, C.POINTER(LmOptions), C.POINTER(vp)]
    lib.ecb_lm_device_destroy.argtypes = [vp]
    lib.ecb_lm_device_destroy.restype = None
    lib.ecb_lm_device_set_exchange.argtypes = [vp, i32, i32, vp]
    lib.ecb_lm_device_begin.argtypes = [vp, vp, vp, vp]
    lib.ecb_lm_device_iterate.argtypes = [vp, i32]
    lib.ecb_lm_device_running.argtypes = [vp]
    lib.ecb_lm_device_result.argtypes = [vp, vp, vp, vp, C.POINTER(LmSummary), vp, i32]
    lib.ecb_calibrate_device.argtypes = [vp, vp, vp, vp, C.POINTER(LmSummary), vp, i32]
    lib.ecb_covariance.argtypes = [vp, i32, vp, vp, vp, vp, vp, i64, vp, vp, vp, C.POINTER(CovarianceSummary)]
    lib.ecb_pose_covariance.argtypes = [vp, vp, i64, vp, vp, C.POINTER(C.c_int64)]
    lib.ecb_pose_covariance_device.argtypes = [vp, vp, i64, vp, vp, C.POINTER(C.c_int64)]
    lib.ecb_trajectory_motion.argtypes = [vp, vp, vp, vp, i64, vp, C.POINTER(C.c_int64)]
    lib.ecb_trajectory_motion_device.argtypes = [vp, vp, vp, vp, i64, vp, C.POINTER(C.c_int64)]
    lib.ecb_motion_covariance.argtypes = [vp, vp, i64, vp, vp, C.POINTER(C.c_int64)]
    lib.ecb_motion_covariance_device.argtypes = [vp, vp, i64, vp, vp, C.POINTER(C.c_int64)]
    lib.ecb_gyro_calibrate.argtypes = [vp, vp, vp, i64, C.c_double, i32, C.POINTER(GyroCalibration), vp, vp]
    _lib = lib
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def inverse_radial_fold(k):
    """rho_fold of the inverse radial polynomial k[5] = k1 .. k5 (ecb_inverse_radial_fold): g(rho) = rho s(rho^2) increases on
    [0, rho_fold) only, so the forward model (projection) exists for distorted radii below it; inf when g increases everywhere.
    Normalised units: rho_fold * fx is the radius in pixels."""
    k = np.ascontiguousarray(k, np.float64)
    if k.shape != (5,):
        raise ValueError("k must hold the 5 coefficients k1 .. k5")
    rho = C.c_double(0.0)
    rc = load_library().ecb_inverse_radial_fold(_ptr(k), C.byref(rho))
    if rc != OK:
        raise EcbError(rc, "ecb_inverse_radial_fold")
    return rho.value


def default_params(eps=4.0, min_pts=2, cluster_min=5, knn_num=3, fit_circle=0, radius_threshold=15.511363636363637,
                   rows_cols=36, order_mode=0, max_clusters=0, median_mode=0):
    """CirclesEventFrame::Params defaults + parameter/event_calibration/example.yaml.
    order_mode=1, median_mode=1 reproduce the reference's pid order and std::nth_element medians."""
    return FrontendParams(eps, min_pts, cluster_min, knn_num, fit_circle, radius_threshold, rows_cols, order_mode,
                          max_clusters, median_mode)


def radius_threshold(width, height, rows, cols, asymmetric, square, radius):
    """circleRadiusThreshold_ of the CirclesEventFrame ctor (CirclesEventFrame.cpp:16-33)."""
    c2 = 2.0 * cols if asymmetric else float(cols)
    W, H = float(width), float(height)
    return min(max(W, H) / max(float(rows), c2), min(W, H) / min(float(rows), c2)) / square * radius * 1.5


class Context:
    """One CUDA device + stream + buffers (``ecb_ctx``)."""

    def __init__(self, device=0, stream=None):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.ecb_ctx_create(device, C.c_void_p(stream) if stream else None, C.byref(h))
        if rc != OK:
            raise EcbError(rc, "ecb_ctx_create failed: no usable CUDA device %d (there is no CPU fallback)" % device)
        self.h = h
        self.n_win = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.ecb_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc < 0 or rc == FAILED:
            raise EcbError(rc, self.lib.ecb_last_error(self.h).decode())
        return rc

    @property
    def launches(self):
        return int(self.lib.ecb_launch_count(self.h))

    def synchronize(self):
        self._chk(self.lib.ecb_synchronize(self.h))

    STAGES = ["ingest", "bounds", "window", "cluster", "pair", "assoc", "normal_eq", "cost", "order", "bfs"]

    def set_profiling(self, on=True):
        self._chk(self.lib.ecb_set_profiling(self.h, int(on)))

    def stage_ms(self):
        out = np.zeros(len(self.STAGES), np.float32)
        self._chk(self.lib.ecb_stage_ms(self.h, _ptr(out)))
        return dict(zip(self.STAGES, out.tolist()))

    # ---- ingest ----
    def set_sensor(self, width, height):
        self._chk(self.lib.ecb_set_sensor(self.h, width, height))

    def load_events(self, records):
        """records: numpy structured array / bytes of packed 25-byte reference records (host)."""
        buf = np.ascontiguousarray(records)
        n = buf.nbytes // 25
        self._keep = buf
        self._chk(self.lib.ecb_load_events_host(self.h, _ptr(buf), n))
        return n

    def load_events_ptr(self, host_ptr, n):
        """host_ptr: address of n packed records in (ideally pinned) host memory."""
        self._chk(self.lib.ecb_load_events_host(self.h, C.c_void_p(host_ptr), n))
        return n

    def load_events_device(self, dptr, n):
        self._chk(self.lib.ecb_load_events_device(self.h, C.c_void_p(dptr), n))

    # ---- front end ----
    def frontend_run(self, windows, params=None):
        win = np.ascontiguousarray(windows, np.float64).reshape(-1, 2)
        params = params or default_params()
        self._chk(self.lib.ecb_frontend_run(self.h, _ptr(win), len(win), C.byref(params)))
        self.n_win = len(win)

    def summary(self, out=None):
        """per-window summaries; `out` (optional): a caller-owned SUMMARY_DTYPE array of n_win entries to fill"""
        if out is None:
            out = np.zeros(self.n_win, SUMMARY_DTYPE)
        assert out.dtype == SUMMARY_DTYPE and out.flags.c_contiguous and len(out) == self.n_win
        if self.n_win:
            self._chk(self.lib.ecb_frontend_summary(self.h, _ptr(out), self.n_win))
        return out

    def points(self, polarity):
        n = int(self.lib.ecb_frontend_total_points(self.h, polarity))
        xy = np.zeros((max(n, 1), 2))
        lab = np.zeros(max(n, 1), np.int32)
        self._chk(self.lib.ecb_frontend_points(self.h, polarity, _ptr(xy), _ptr(lab)))
        return xy[:n], lab[:n]

    def candidates(self, max_cand=64, out=None):
        if out is None:
            out = np.zeros((self.n_win, max_cand, 5))
        assert out.dtype == np.float64 and out.flags.c_contiguous and out.shape == (self.n_win, max_cand, 5)
        if self.n_win:
            self._chk(self.lib.ecb_frontend_candidates(self.h, _ptr(out), max_cand))
        return out

    def rectify(self, window_index, image_points, rows=9, cols=4, asymmetric=True, inlier_threshold=3.0):
        """rectifyFeatures for frames of the last front-end run; image_points [n_frames][n_circles][5][2]"""
        wi = np.ascontiguousarray(window_index, np.int32)
        img = np.ascontiguousarray(image_points, np.float64)
        nf, nc = img.shape[0], img.shape[1]
        assert img.shape == (nf, nc, 5, 2) and len(wi) == nf
        out = np.zeros((max(nf, 1), nc, 3))
        ok = np.zeros(max(nf, 1), np.int32)
        self._chk(self.lib.ecb_frontend_rectify(self.h, _ptr(wi), nf, nc, _ptr(img), float(inlier_threshold), rows, cols,
                                                int(asymmetric), _ptr(out), _ptr(ok)))
        return out[:nf], ok[:nf]

    def clusters(self, window, polarity, cap=512):
        raw = np.zeros(cap, np.int32)
        size = np.zeros(cap, np.int32)
        med = np.zeros(cap, np.int32)
        n = self._chk(self.lib.ecb_frontend_clusters(self.h, window, polarity, _ptr(raw), _ptr(size), _ptr(med), cap))
        return raw[:n], size[:n], med[:n]

    # ---- DBSCAN::Run boundary ----
    def dbscan(self, xy, eps, min_pts):
        """Returns (status, labels, n_clusters) like DBSCAN::Run: status 0 SUCCESS / 1 FAILED."""
        xy = np.ascontiguousarray(xy, np.float64).reshape(-1, 2)
        n = len(xy)
        labels = np.full(max(n, 1), -1, np.int32)
        nc = C.c_int32(0)
        rc = self.lib.ecb_dbscan_run(self.h, _ptr(xy), n, float(eps), int(min_pts), _ptr(labels), C.byref(nc))
        if rc == FAILED:
            return FAILED, labels[:0], 0
        self._chk(rc)
        return OK, labels[:n], nc.value

    def dbscan_ordered(self, xy, eps, min_pts):
        """DBSCAN::Run with `Clusters` as ordered lists (the reference's member order) and `Noise`."""
        xy = np.ascontiguousarray(xy, np.float64).reshape(-1, 2)
        n = len(xy)
        labels = np.full(max(n, 1), -1, np.int32)
        sizes = np.zeros(max(n, 1), np.int32)
        members = np.zeros(max(n, 1), np.uint32)
        nc = C.c_int32(0)
        rc = self.lib.ecb_dbscan_run_ordered(self.h, _ptr(xy), n, float(eps), int(min_pts), _ptr(labels), C.byref(nc),
                                             _ptr(sizes), _ptr(members))
        if rc == FAILED:
            return FAILED, labels[:0], [], labels[:0]
        self._chk(rc)
        off = np.concatenate([[0], np.cumsum(sizes[:nc.value])])
        clusters = [members[off[c]:off[c + 1]].copy() for c in range(nc.value)]
        return OK, labels[:n], clusters, np.nonzero(labels[:n] < 0)[0].astype(np.uint32)

    def dbscan_nd(self, pts, eps, min_pts, ordered=True):
        """DBSCAN<T,Float>::Run(V, dim, eps, min) for dim = pts.shape[1] (1..4): (status, labels, clusters, noise)."""
        pts = np.ascontiguousarray(pts, np.float64)
        n, dim = pts.shape
        labels = np.full(max(n, 1), -1, np.int32)
        sizes = np.zeros(max(n, 1), np.int32)
        members = np.zeros(max(n, 1), np.uint32)
        nc = C.c_int32(0)
        rc = self.lib.ecb_dbscan_run_nd(self.h, _ptr(pts), n, dim, float(eps), int(min_pts), _ptr(labels), C.byref(nc),
                                        _ptr(sizes) if ordered else None, _ptr(members) if ordered else None)
        if rc == FAILED:
            return FAILED, labels[:0], [], labels[:0]
        self._chk(rc)
        off = np.concatenate([[0], np.cumsum(sizes[:nc.value])])
        clusters = [members[off[c]:off[c + 1]].copy() for c in range(nc.value)] if ordered else nc.value
        return OK, labels[:n], clusters, np.nonzero(labels[:n] < 0)[0].astype(np.uint32)

    def dbscan_batch_ordered(self, xy, offsets, eps, min_pts):
        xy = np.ascontiguousarray(xy, np.float64).reshape(-1, 2)
        off = np.ascontiguousarray(offsets, np.int64)
        k = len(off) - 1
        labels = np.full(max(len(xy), 1), -1, np.int32)
        sizes = np.zeros(max(len(xy), 1), np.int32)
        members = np.zeros(max(len(xy), 1), np.uint32)
        nc = np.zeros(max(k, 1), np.int32)
        st = np.zeros(max(k, 1), np.uint32)
        self._chk(self.lib.ecb_dbscan_run_batch_ordered(self.h, _ptr(xy), _ptr(off), k, float(eps), int(min_pts),
                                                        _ptr(labels), _ptr(nc), _ptr(st), _ptr(sizes), _ptr(members)))
        out = []
        for j in range(k):
            o = np.concatenate([[0], np.cumsum(sizes[off[j]:off[j] + nc[j]])]) + off[j]
            out.append([members[o[c]:o[c + 1]].copy() for c in range(nc[j])])
        return labels[:len(xy)], nc[:k], st[:k], out

    def dbscan_batch(self, xy, offsets, eps, min_pts):
        xy = np.ascontiguousarray(xy, np.float64).reshape(-1, 2)
        off = np.ascontiguousarray(offsets, np.int64)
        k = len(off) - 1
        labels = np.full(max(len(xy), 1), -1, np.int32)
        nc = np.zeros(max(k, 1), np.int32)
        st = np.zeros(max(k, 1), np.uint32)
        self._chk(self.lib.ecb_dbscan_run_batch(self.h, _ptr(xy), _ptr(off), k, float(eps), int(min_pts), _ptr(labels),
                                                _ptr(nc), _ptr(st)))
        return labels[:len(xy)], nc[:k], st[:k]

    def fit_circles(self, xy, offsets):
        xy = np.ascontiguousarray(xy, np.float64).reshape(-1, 2)
        off = np.ascontiguousarray(offsets, np.int64)
        k = len(off) - 1
        out = np.zeros((max(k, 1), 3))
        self._chk(self.lib.ecb_fit_circles(self.h, _ptr(xy), _ptr(off), k, _ptr(out)))
        return out[:k]

    # ---- cost evaluation ----
    def cost_setup(self, n_cp, knots, radius=1.75, huber=0.35):
        n_cp = np.ascontiguousarray(np.atleast_1d(n_cp), np.int32)
        kn = np.ascontiguousarray(np.concatenate([np.asarray(k, np.float64).ravel() for k in knots])
                                  if isinstance(knots, (list, tuple)) else knots, np.float64)
        assert len(kn) == int(n_cp.sum()) + 4 * len(n_cp)
        self._chk(self.lib.ecb_cost_setup(self.h, len(n_cp), _ptr(n_cp), _ptr(kn), float(radius), float(huber)))

    def cost_set_rotation_model(self, use_so3):
        """0: normalised quaternion spline (useSO3: 0); 1: cumulative SO(3) spline + LocalParameterizationSO3 (useSO3: 1)"""
        self._chk(self.lib.ecb_cost_set_rotation_model(self.h, int(use_so3)))

    def set_constant_intrinsics(self, names):
        """Holds the named intrinsics (INTRINSIC_NAMES; empty: none) at their start values in calibrate() and DeviceLm (captured
        when a DeviceLm is created), and conditions covariance() on them: their rows and columns of Z are zeros and
        dimension counts the free parameters.  Kept by the context across cost_setup."""
        self._chk(self.lib.ecb_cost_set_constant_intrinsics(self.h, constant_intrinsics_mask(names)))

    # ---- fused reduce + inter-GPU exchange of the normal equations ----
    def exchange_buffer_bytes(self, n_ranks):
        return int(self.lib.ecb_exchange_buffer_bytes(self.h, n_ranks))

    def device_alloc(self, nbytes):
        p = C.c_void_p()
        self._chk(self.lib.ecb_device_alloc(self.h, nbytes, C.byref(p)))
        return p.value

    def device_free(self, ptr):
        self._chk(self.lib.ecb_device_free(self.h, C.c_void_p(ptr)))

    def ipc_export(self, ptr):
        h = np.zeros(64, np.uint8)
        self._chk(self.lib.ecb_ipc_export(self.h, C.c_void_p(ptr), _ptr(h)))
        return h

    def ipc_open(self, handle):
        h = np.ascontiguousarray(handle, np.uint8)
        p = C.c_void_p()
        self._chk(self.lib.ecb_ipc_open(self.h, _ptr(h), C.byref(p)))
        return p.value

    def enable_peer_access(self, peer_device):
        """several GPUs driven from ONE process: lets this context's kernels store into buffers of `peer_device`"""
        self._chk(self.lib.ecb_enable_peer_access(self.h, int(peer_device)))

    def ipc_close(self, ptr):
        self._chk(self.lib.ecb_ipc_close(self.h, C.c_void_p(ptr)))

    def cost_normal_eq_exchange(self, intr, rot, trans, rank, recv_ptrs, epoch, d_out, want_cost=True, phases=3):
        """normal equations with the inter-GPU sum fused in; recv_ptrs: device pointers of every rank's receive buffer"""
        a = [np.ascontiguousarray(v, np.float64) for v in (intr, rot, trans)]
        ptrs = (C.c_void_p * len(recv_ptrs))(*[C.c_void_p(p) for p in recv_ptrs])
        cost = C.c_double(0)
        self._chk(self.lib.ecb_cost_normal_eq_exchange(self.h, _ptr(a[0]), _ptr(a[1]), _ptr(a[2]), rank, len(recv_ptrs), ptrs,
                                                       C.c_uint64(epoch), int(phases), C.c_void_p(d_out),
                                                       C.cast(C.byref(cost), C.c_void_p) if want_cost else None))
        return cost.value if want_cost else None

    def cost_layout(self):
        cp, sp = C.c_int32(), C.c_int32()
        nr, nd = C.c_int64(), C.c_int64()
        self._chk(self.lib.ecb_cost_layout(self.h, C.byref(cp), C.byref(sp), C.byref(nr), C.byref(nd)))
        return dict(total_cp=cp.value, total_spans=sp.value, n_residuals=nr.value, out_doubles=nd.value)

    def cost_associate(self, kf_t, circles, landmarks, step):
        kf_t = np.ascontiguousarray(kf_t, np.float64)
        circles = np.ascontiguousarray(circles, np.float64)
        lm = np.ascontiguousarray(landmarks, np.float64)
        n = C.c_int64(0)
        self._chk(self.lib.ecb_cost_associate(self.h, _ptr(kf_t), _ptr(circles), len(kf_t), circles.shape[1], _ptr(lm),
                                              float(step), C.byref(n)))
        return n.value

    def cost_associate_device(self, d_kf_t, d_circles, n_keyframes, n_circles, d_landmarks, step):
        """the same with device pointers (integers) of the three tables"""
        n = C.c_int64(0)
        self._chk(self.lib.ecb_cost_associate_device(self.h, C.c_void_p(d_kf_t), C.c_void_p(d_circles), int(n_keyframes),
                                                     int(n_circles), C.c_void_p(d_landmarks), float(step), C.byref(n)))
        return n.value

    def cost_association(self):
        n = self.cost_layout()["n_residuals"]
        ev = np.zeros(max(n, 1), np.int64)
        ci = np.zeros(max(n, 1), np.int32)
        self._chk(self.lib.ecb_cost_get_association(self.h, _ptr(ev), _ptr(ci), n))
        return ev[:n], ci[:n]

    def cost_set_residuals(self, obs, lm, t, spline):
        obs = np.ascontiguousarray(obs, np.float64)
        lm = np.ascontiguousarray(lm, np.float64)
        t = np.ascontiguousarray(t, np.float64)
        sp = np.ascontiguousarray(spline, np.int32)
        self._chk(self.lib.ecb_cost_set_residuals(self.h, _ptr(obs), _ptr(lm), _ptr(t), _ptr(sp), len(t)))

    def cost_eval(self, intr, rot, trans):
        intr = np.ascontiguousarray(intr, np.float64)
        rot = np.ascontiguousarray(rot, np.float64)
        trans = np.ascontiguousarray(trans, np.float64)
        c = C.c_double(0)
        self._chk(self.lib.ecb_cost_eval(self.h, _ptr(intr), _ptr(rot), _ptr(trans), C.byref(c)))
        return c.value

    def cost_normal_eq(self, intr, rot, trans, d_out=None, host=True):
        """Returns (cost, H[n_spans,33,33], g[n_spans,33]) when host=True, else leaves the packed result in d_out."""
        intr = np.ascontiguousarray(intr, np.float64)
        rot = np.ascontiguousarray(rot, np.float64)
        trans = np.ascontiguousarray(trans, np.float64)
        lay = self.cost_layout()
        c = C.c_double(0)
        if not host:
            self._chk(self.lib.ecb_cost_normal_eq(self.h, _ptr(intr), _ptr(rot), _ptr(trans), C.c_void_p(d_out), None, None))
            return None
        out = np.zeros(lay["out_doubles"])
        self._chk(self.lib.ecb_cost_normal_eq(self.h, _ptr(intr), _ptr(rot), _ptr(trans),
                                              C.c_void_p(d_out) if d_out else None, _ptr(out), C.byref(c)))
        ns = lay["total_spans"]
        blk = out[:ns * 1122].reshape(ns, 1122)
        return c.value, blk[:, :1089].reshape(ns, 33, 33).copy(), blk[:, 1089:].copy()

    def cost_residuals(self, intr, rot, trans, d_out=None, host=True):
        """Raw residuals r_k = ||X_w - L|| - radius of every record at the point (ecb_cost_residuals), in the order of
        cost_association(): a distance on the board plane in the units of the board points, NOT pixels.  Returns an ndarray
        (float64, n_residuals) when host=True; else leaves them in d_out (device pointer, or None for the context's own buffer),
        enqueued on the context's stream, and returns None."""
        return self._record_report(self.lib.ecb_cost_residuals, intr, rot, trans, d_out, host)

    def residual_groups(self, intr, rot, trans, by, kf_t=None, cell_px=16):
        """Statistics of the raw residuals (board units, not pixels) per group (ecb_cost_residual_groups).  by: "keyframe"
        (kf_t: the stamps given to cost_associate), "circle" or "sensor_cell" (cells of cell_px pixels, row major).  Returns
        (groups, total) as numpy structured arrays of RESIDUAL_GROUP_DTYPE (count, n_downweighted, sum, sum_sq, max_abs, cost);
        total has shape () and covers every record."""
        return self._group_report(self.lib.ecb_cost_residual_groups, RESIDUAL_GROUP_DTYPE, intr, rot, trans, by, kf_t, cell_px)

    def reject_residuals(self, intr, rot, trans, max_abs_r=math.inf, drop_keyframes=None, kf_t=None):
        """Removes outliers from this context's records (ecb_cost_reject): record k goes when not |r_k| <= max_abs_r (r_k as
        cost_residuals returns it at the point; NaN always goes) or when drop_keyframes[j] is true for its key frame j (the
        grouping of residual_groups(by="keyframe"); kf_t: the stamps given to cost_associate).  The kept records keep their
        order, and every later call on the context sees only them until the next association or cost_set_residuals.
        Returns (n_kept, n_removed)."""
        a = [np.ascontiguousarray(v, np.float64) for v in (intr, rot, trans)]
        kf = np.ascontiguousarray(kf_t, np.float64) if kf_t is not None else None
        drop = np.ascontiguousarray(np.asarray(drop_keyframes) != 0, np.uint8) if drop_keyframes is not None else None
        if drop is not None and kf is not None and len(kf) != len(drop):
            raise ValueError("drop_keyframes and kf_t must have one entry per key frame")
        nk = len(drop) if drop is not None else (len(kf) if kf is not None else 0)
        kept, removed = C.c_int64(0), C.c_int64(0)
        self._chk(self.lib.ecb_cost_reject(self.h, _ptr(a[0]), _ptr(a[1]), _ptr(a[2]), float(max_abs_r), _ptr(kf), _ptr(drop), nk,
                                           C.byref(kept), C.byref(removed)))
        return kept.value, removed.value

    def reassociate(self, intr, rot, trans, gate_px=5.0, max_dt=0.0):
        """Re-associates the loaded events with the board circles at a calibrated point (ecb_cost_reassociate): every candidate
        event of the association (max_dt = 0: its window; > 0: |t - t_kf| <= max_dt) is matched to the landmark nearest to its
        back-projection at its own pose on the spline and kept when its event-to-rim error is below gate_px pixels.  The kept
        events replace the records (event order, the layout of cost_associate); key frames and landmarks stay the association's.
        Returns (n_residuals, n_same, n_changed, n_new, n_lost), the last four against the records held before the call."""
        a = [np.ascontiguousarray(v, np.float64) for v in (intr, rot, trans)]
        out = [C.c_int64(0) for _ in range(5)]
        self._chk(self.lib.ecb_cost_reassociate(self.h, _ptr(a[0]), _ptr(a[1]), _ptr(a[2]), float(gate_px), float(max_dt),
                                                *[C.byref(v) for v in out]))
        return tuple(v.value for v in out)

    def reprojection_errors(self, intr, rot, trans, d_out=None, host=True):
        """Reprojection errors e_k of every record in pixels (ecb_cost_reprojection_errors), in the order of cost_residuals():
        e_k = sign(|d| - radius) |q - o|, o the event pixel and q the projection of the residual's rim point, NaN where it cannot
        be projected.  Returns (e as float64 ndarray, n_invalid) when host=True; else leaves e in d_out (device pointer, or None
        for the context's own buffer), enqueued on the context's stream, and returns None."""
        bad = C.c_int64(0)
        e = self._record_report(self.lib.ecb_cost_reprojection_errors, intr, rot, trans, d_out, host, C.byref(bad) if host else None)
        return (e, bad.value) if host else None

    def reprojection_groups(self, intr, rot, trans, by, kf_t=None, cell_px=16):
        """Statistics of the reprojection errors (pixels) per group (ecb_cost_reprojection_groups): the groups of residual_groups.
        Returns (groups, total) as numpy structured arrays of REPROJECTION_GROUP_DTYPE (count, n_invalid, sum, sum_sq,
        max_abs; count and the sums over the valid records only); total has shape () and covers every record."""
        return self._group_report(self.lib.ecb_cost_reprojection_groups, REPROJECTION_GROUP_DTYPE, intr, rot, trans, by, kf_t,
                                  cell_px)

    def _record_report(self, fn, intr, rot, trans, d_out, host, *extra):
        """one value per record (fn: ecb_cost_residuals or ecb_cost_reprojection_errors; extra: its arguments after h_out): an
        ndarray when host, else None with the values left in d_out"""
        a = [np.ascontiguousarray(v, np.float64) for v in (intr, rot, trans)]
        d = C.c_void_p(d_out) if d_out else None
        if not host:
            self._chk(fn(self.h, _ptr(a[0]), _ptr(a[1]), _ptr(a[2]), d, None, *extra))
            return None
        n = self.cost_layout()["n_residuals"]
        out = np.zeros(max(n, 1))
        self._chk(fn(self.h, _ptr(a[0]), _ptr(a[1]), _ptr(a[2]), d, _ptr(out), *extra))
        return out[:n]

    def _group_report(self, fn, dtype, intr, rot, trans, by, kf_t, cell_px):
        """the groups of one report (fn: ecb_cost_residual_groups or ecb_cost_reprojection_groups, dtype: its group record): the
        size query, then the filled call"""
        if by not in RESIDUALS_BY:
            raise ValueError("by must be one of %s" % ", ".join(RESIDUALS_BY))
        a = [np.ascontiguousarray(v, np.float64) for v in (intr, rot, trans)]
        kf = np.ascontiguousarray(kf_t, np.float64) if kf_t is not None else None
        nk = len(kf) if kf is not None else 0
        args = (self.h, _ptr(a[0]), _ptr(a[1]), _ptr(a[2]), RESIDUALS_BY[by], _ptr(kf), nk, int(cell_px))
        ng = C.c_int(0)
        self._chk(fn(*args, None, 0, C.byref(ng), None))
        groups = np.zeros(max(ng.value, 1), dtype)
        total = np.zeros((), dtype)
        self._chk(fn(*args, _ptr(groups), ng.value, C.byref(ng), _ptr(total)))
        return groups[:ng.value], total

    def keyframe_reprojection(self, intr, rot, trans, kf_t, circles, landmarks):
        """Circle centres of the key frames reprojected at their stamps (ecb_keyframe_reprojection): kf_t[K], circles[K][n][3]
        (cx, cy, r; r < 0 = absent) and landmarks[n][3] as for cost_associate.  Returns (proj[K, n, 2], err[K, n] = |proj -
        (cx, cy)| in pixels, total of REPROJECTION_GROUP_DTYPE over the present features); NaN for an absent feature, a stamp
        outside every segment, or a point that cannot be projected."""
        a = [np.ascontiguousarray(v, np.float64) for v in (intr, rot, trans)]
        kf = np.ascontiguousarray(kf_t, np.float64)
        circ = np.ascontiguousarray(circles, np.float64)
        lm = np.ascontiguousarray(landmarks, np.float64)
        K, n = circ.shape[0], circ.shape[1]
        if circ.shape != (K, n, 3) or kf.shape != (K,) or lm.shape != (n, 3):
            raise ValueError("kf_t[K], circles[K][n][3] and landmarks[n][3] expected")
        proj, err = np.zeros((K, n, 2)), np.zeros((K, n))
        total = np.zeros((), REPROJECTION_GROUP_DTYPE)
        self._chk(self.lib.ecb_keyframe_reprojection(self.h, _ptr(a[0]), _ptr(a[1]), _ptr(a[2]), _ptr(kf), _ptr(circ), K, n,
                                                     _ptr(lm), _ptr(proj), _ptr(err), _ptr(total)))
        return proj, err, total

    def calibrate(self, n_cp, intr, rot, trans, options=None, trace_rows=256):
        """EventCalibSpline::optimize on one GPU: returns (intr, rot, trans, summary dict, trace[rows,4])."""
        n_cp = np.ascontiguousarray(np.atleast_1d(n_cp), np.int32)
        intr = np.array(intr, np.float64, copy=True)
        rot = np.array(rot, np.float64, copy=True)
        trans = np.array(trans, np.float64, copy=True)
        opt = options or lm_options()
        summ = LmSummary()
        tr = np.zeros((trace_rows, 4))
        self._chk(self.lib.ecb_calibrate(self.h, len(n_cp), _ptr(n_cp), _ptr(intr), _ptr(rot), _ptr(trans), C.byref(opt),
                                         C.byref(summ), _ptr(tr), trace_rows))
        rows = int(np.count_nonzero(tr[:, 2]))
        return intr, rot, trans, {f[0]: getattr(summ, f[0]) for f in LmSummary._fields_}, tr[:rows]

    def covariance(self, n_cp, intr, rot, trans, d_packed=None, n_residuals_total=0):
        """Covariance Z = H^-1 of the parameters at x (ecb_covariance): the selected inverse on the band / arrow pattern.
        Returns a dict: ok, cov_intrinsics [9,9], cov_band [6C,24] (Z(j+r, j) at [j, r]), cov_cross [9,6C], cost, sigma2,
        min_relative_pivot, n_residuals, dimension, deficient_index and std_intrinsics = sqrt(sigma2 diag Z_cc).  A rank-deficient
        system gives ok=False, the index of the failing pivot and no arrays.  d_packed: device pointer of an already-summed packed
        buffer (several GPUs); n_residuals_total: residual count over all ranks (0: this context's).  control_point_covariance()
        takes the 6 x 6 block of one control point out of the result."""
        n_cp = np.ascontiguousarray(np.atleast_1d(n_cp), np.int32)
        a = [np.ascontiguousarray(v, np.float64) for v in (intr, rot, trans)]
        n = 6 * int(n_cp.sum())
        zc, zb, zx = np.zeros((9, 9)), np.zeros((n, 24)), np.zeros((9, n))
        s = CovarianceSummary()
        rc = self.lib.ecb_covariance(self.h, len(n_cp), _ptr(n_cp), _ptr(a[0]), _ptr(a[1]), _ptr(a[2]),
                                     C.c_void_p(d_packed) if d_packed else None, int(n_residuals_total), _ptr(zc), _ptr(zb),
                                     _ptr(zx), C.byref(s))
        if rc != FAILED:
            self._chk(rc)
        out = {f[0]: getattr(s, f[0]) for f in CovarianceSummary._fields_}
        out["ok"] = rc == OK
        if rc == OK:
            out.update(cov_intrinsics=zc, cov_band=zb, cov_cross=zx, std_intrinsics=np.sqrt(s.sigma2 * np.diag(zc)))
        return out

    def pose_covariance(self, times):
        """6 x 6 covariance Sigma(t) of the trajectory's pose at the given times (ecb_pose_covariance), from the last successful
        covariance() on this context.  Returns a dict: pose (n, 7) = tx ty tz qx qy qz qw, cov (n, 6, 6) over (dtheta body
        frame, dp world frame), n_valid.  Times outside every segment, and NaN, give NaN rows.  Not scaled by sigma2."""
        t = np.ascontiguousarray(np.atleast_1d(times), np.float64)
        n = len(t)
        pose, cov = np.empty((n, 7)), np.empty((n, 6, 6))
        nv = C.c_int64()
        self._chk(self.lib.ecb_pose_covariance(self.h, _ptr(t), n, _ptr(pose), _ptr(cov), C.byref(nv)))
        return {"pose": pose, "cov": cov, "n_valid": nv.value}

    def pose_covariance_device(self, d_times, n, d_pose, d_cov, count=True):
        """ecb_pose_covariance_device on raw device pointers (e.g. torch CUDA tensors' data_ptr()): n float64 times in, n x 7
        poses and n x 36 covariances out (either pointer may be 0).  Enqueued on the context's stream; with count=True it waits
        and returns the number of valid queries, else returns None at once."""
        nv = C.c_int64()
        self._chk(self.lib.ecb_pose_covariance_device(self.h, C.c_void_p(d_times) if d_times else None, int(n),
                                                      C.c_void_p(d_pose) if d_pose else None,
                                                      C.c_void_p(d_cov) if d_cov else None, C.byref(nv) if count else None))
        return nv.value if count else None

    def trajectory_motion(self, rot, trans, times):
        """Motion of the trajectory at the given times (ecb_trajectory_motion) at the control points rot (4 per point, x y z w)
        and trans (3 per point), in the layout of cost_eval and the rotation model of this context; needs cost_setup only.
        Returns a dict: pose (n, 7) = tx ty tz qx qy qz qw, omega (n, 3) body-frame angular velocity in radians per time unit,
        velocity (n, 3) and acceleration (n, 3) in the world frame, n_valid.  Times outside every segment, and NaN, give NaN
        rows."""
        r, tr = (np.ascontiguousarray(v, np.float64) for v in (rot, trans))
        t = np.ascontiguousarray(np.atleast_1d(times), np.float64)
        n = len(t)
        motion = np.empty((n, 16))
        nv = C.c_int64()
        self._chk(self.lib.ecb_trajectory_motion(self.h, _ptr(r), _ptr(tr), _ptr(t), n, _ptr(motion), C.byref(nv)))
        return _motion_dict(motion, nv.value)

    def trajectory_motion_device(self, rot, trans, d_times, n, d_motion, count=True):
        """ecb_trajectory_motion_device: control points as host arrays, raw device pointers (e.g. torch CUDA tensors'
        data_ptr()) for n float64 times in and n x 16 motion rows out (the pointer may be 0).  Enqueued on the context's stream;
        with count=True it waits and returns the number of valid queries, else returns None at once."""
        r, tr = (np.ascontiguousarray(v, np.float64) for v in (rot, trans))
        nv = C.c_int64()
        self._chk(self.lib.ecb_trajectory_motion_device(self.h, _ptr(r), _ptr(tr), C.c_void_p(d_times) if d_times else None,
                                                        int(n), C.c_void_p(d_motion) if d_motion else None,
                                                        C.byref(nv) if count else None))
        return nv.value if count else None

    def motion_covariance(self, times):
        """Motion of the trajectory and its 9 x 9 covariance over (omega, velocity, acceleration) at the given times
        (ecb_motion_covariance), at the point and with the Z of the last successful covariance() on this context.  Returns the
        dict of trajectory_motion plus cov (n, 9, 9).  Not scaled by sigma2."""
        t = np.ascontiguousarray(np.atleast_1d(times), np.float64)
        n = len(t)
        motion, cov = np.empty((n, 16)), np.empty((n, 9, 9))
        nv = C.c_int64()
        self._chk(self.lib.ecb_motion_covariance(self.h, _ptr(t), n, _ptr(motion), _ptr(cov), C.byref(nv)))
        out = _motion_dict(motion, nv.value)
        out["cov"] = cov
        return out

    def motion_covariance_device(self, d_times, n, d_motion, d_cov, count=True):
        """ecb_motion_covariance_device on raw device pointers: n float64 times in, n x 16 motion rows and n x 81 covariances
        out (either pointer may be 0).  Enqueued on the context's stream; with count=True it waits and returns the number of
        valid queries, else returns None at once."""
        nv = C.c_int64()
        self._chk(self.lib.ecb_motion_covariance_device(self.h, C.c_void_p(d_times) if d_times else None, int(n),
                                                        C.c_void_p(d_motion) if d_motion else None,
                                                        C.c_void_p(d_cov) if d_cov else None, C.byref(nv) if count else None))
        return nv.value if count else None

    def gyro_calibrate(self, rot, gyro, max_offset, n_offsets):
        """Camera-gyroscope calibration (ecb_gyro_calibrate) at the rotation control points rot (4 per point, x y z w, layout of
        cost_eval, rotation model of this context); needs cost_setup only.  gyro (n, 4) = t wx wy wz: gyroscope stamps (time
        units of the knots) and readings (rad per time unit, gyroscope frame).  Model w_g = R_gc w_c(t + offset) + bias; the
        offset is searched on n_offsets (odd) points over [-max_offset, max_offset] (max_offset 0 with n_offsets 1: held at 0),
        then refined with the rotation and the bias by least squares.  Returns a dict: ok, status (GYRO_*), message (when not
        ok), q_gc (x y z w), R_gc (3, 3), offset, bias, cov (7, 7) over (rotation tangent, offset, bias), not scaled by sigma2,
        std, sigma2, cost, rms, scan_offset, offset_grid and offset_cost (the scan), residuals (n, 3) (NaN rows for unused
        samples), n_used, n_unused, iterations, termination (ECB_LM_* code), n_params.  A failed calibration (too few samples,
        the scan's minimum at the edge of the grid, a rank-deficient system) gives ok=False with what was computed; other
        errors raise."""
        r = np.ascontiguousarray(rot, np.float64)
        g = np.ascontiguousarray(np.asarray(gyro, np.float64).reshape(-1, 4))
        n, M = len(g), int(n_offsets)
        res = np.full((n, 3), np.nan)
        cost = np.full(max(M, 0), np.nan)
        s = GyroCalibration()
        rc = self.lib.ecb_gyro_calibrate(self.h, _ptr(r), _ptr(g), n, float(max_offset), M, C.byref(s), _ptr(cost), _ptr(res))
        if rc != FAILED:
            self._chk(rc)
        q = np.array(s.q_gc)
        out = {"ok": rc == OK, "status": s.status, "q_gc": q, "offset": s.offset, "bias": np.array(s.bias),
               "cov": np.array(s.cov).reshape(7, 7), "std": np.array(s.std), "sigma2": s.sigma2, "cost": s.cost, "rms": s.rms,
               "scan_offset": s.scan_offset, "offset_cost": cost, "residuals": res, "n_used": s.n_used, "n_unused": s.n_unused,
               "iterations": s.iterations, "termination": s.termination, "n_params": s.n_params,
               "offset_grid": (max_offset * (2.0 * np.arange(M) - (M - 1)) / (M - 1)) if M > 1 else np.zeros(M)}
        x, y, z, w = q
        out["R_gc"] = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                                [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                                [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
        if rc == FAILED:
            out["message"] = self.lib.ecb_last_error(self.h).decode()
        return out


def _motion_dict(motion, n_valid):
    """the columns of a motion row (ecb_trajectory_motion): pose 7, omega 3, velocity 3, acceleration 3"""
    return {"pose": motion[:, :7], "omega": motion[:, 7:10], "velocity": motion[:, 10:13], "acceleration": motion[:, 13:16],
            "n_valid": n_valid}


def control_point_covariance(cov, c):
    """6 x 6 block Z of control point c (rotation tangent 3, translation 3) from the band of Context.covariance()"""
    band = cov["cov_band"]
    out = np.empty((6, 6))
    for a in range(6):
        for b in range(6):
            lo, hi = min(a, b), max(a, b)
            out[a, b] = band[6 * c + lo, hi - lo]
    return out


def lm_options(**kw):
    o = LmOptions()
    load_library().ecb_lm_default_options(C.byref(o))
    for k, v in kw.items():
        setattr(o, k, v)
    return o


class DeviceLm:
    """EventCalibSpline::optimize with the LM state machine and the band-arrow Cholesky solve on the device (ecb_lm_device_*):
    the host enqueues the iterations and reads the result once.  ctx must hold the residual set (cost_setup + association)."""

    def __init__(self, ctx, n_cp, options=None):
        self.ctx = ctx
        self.lib = ctx.lib
        self.n_cp = np.ascontiguousarray(np.atleast_1d(n_cp), np.int32)
        self.C = int(self.n_cp.sum())
        self.opt = options or lm_options()
        h = C.c_void_p()
        ctx._chk(self.lib.ecb_lm_device_create(ctx.h, len(self.n_cp), _ptr(self.n_cp), C.byref(self.opt), C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            if getattr(self.ctx, "h", None):   # the context owns the device: destroy before it (a closed context took it along)
                self.lib.ecb_lm_device_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_exchange(self, rank, recv_ptrs):
        """several GPUs: device pointers of every rank's receive buffer (own buffer at [rank]), see Context.exchange_buffer_bytes"""
        ptrs = (C.c_void_p * len(recv_ptrs))(*[C.c_void_p(p) for p in recv_ptrs])
        self._keep = ptrs
        self.ctx._chk(self.lib.ecb_lm_device_set_exchange(self.h, rank, len(recv_ptrs), ptrs))

    def begin(self, intr, rot, trans):
        a = [np.ascontiguousarray(v, np.float64) for v in (intr, rot, trans)]
        self.ctx._chk(self.lib.ecb_lm_device_begin(self.h, _ptr(a[0]), _ptr(a[1]), _ptr(a[2])))

    def iterate(self, n):
        self.ctx._chk(self.lib.ecb_lm_device_iterate(self.h, int(n)))

    def running(self):
        rc = self.lib.ecb_lm_device_running(self.h)
        if rc < 0:
            self.ctx._chk(rc)
        return rc == 1

    def result(self, trace_rows=256):
        i, r, t = np.zeros(9), np.zeros((self.C, 4)), np.zeros((self.C, 3))
        s = LmSummary()
        tr = np.zeros((trace_rows, 4))
        self.ctx._chk(self.lib.ecb_lm_device_result(self.h, _ptr(i), _ptr(r), _ptr(t), C.byref(s), _ptr(tr), trace_rows))
        out = {f[0]: getattr(s, f[0]) for f in LmSummary._fields_}
        out.update(intrinsics=i, rot_cp=r, trans_cp=t, trace=tr[:int(np.count_nonzero(tr[:, 2]))])
        return out

    def run(self, intr, rot, trans, trace_rows=256):
        """begin + all iterations + result; with fixed_iterations the whole loop is enqueued without a host round trip"""
        self.begin(intr, rot, trans)
        total = self.opt.max_iterations + 1
        if self.opt.fixed_iterations:
            self.iterate(total)
        else:
            done = 0
            while done < total:
                k = min(8, total - done)
                self.iterate(k)
                done += k
                if done < total and not self.running():
                    break
        return self.result(trace_rows)


class LmState:
    """Host-only LM state machine (ecb_lm_*), for callers that all-reduce the normal equations between GPUs."""

    def __init__(self, n_cp, options=None):
        self.lib = load_library()
        self.n_cp = np.ascontiguousarray(np.atleast_1d(n_cp), np.int32)
        self.C = int(self.n_cp.sum())
        self.h = C.c_void_p(self.lib.ecb_lm_create(len(self.n_cp), _ptr(self.n_cp), C.byref(options or lm_options())))

    def __del__(self):
        try:
            self.lib.ecb_lm_destroy(self.h)
        except Exception:
            pass

    def set_constant_intrinsics(self, names):
        """intrinsics held at their start values (INTRINSIC_NAMES; empty: none); before begin(), EcbError(ERR_STATE) after"""
        rc = self.lib.ecb_lm_set_constant_intrinsics(self.h, constant_intrinsics_mask(names))
        if rc != OK:
            raise EcbError(rc, "ecb_lm_set_constant_intrinsics: %s" % ("call it before begin()" if rc == ERR_STATE else "bad mask"))

    def begin(self, intr, rot, trans, packed):
        a = [np.ascontiguousarray(v, np.float64) for v in (intr, rot, trans, packed)]
        return self.lib.ecb_lm_begin(self.h, *[_ptr(v) for v in a])

    def propose(self):
        ci, cr, ct = np.zeros(9), np.zeros((self.C, 4)), np.zeros((self.C, 3))
        st = self.lib.ecb_lm_propose(self.h, _ptr(ci), _ptr(cr), _ptr(ct))
        return st, ci, cr, ct

    def feedback(self, cost):
        return self.lib.ecb_lm_feedback(self.h, float(cost))

    def update(self, packed):
        p = np.ascontiguousarray(packed, np.float64)
        return self.lib.ecb_lm_update(self.h, _ptr(p))

    def state(self):
        i, r, t = np.zeros(9), np.zeros((self.C, 4)), np.zeros((self.C, 3))
        s = LmSummary()
        self.lib.ecb_lm_state(self.h, _ptr(i), _ptr(r), _ptr(t), C.byref(s))
        return i, r, t, {f[0]: getattr(s, f[0]) for f in LmSummary._fields_}

    def trace(self, rows=512):
        tr = np.zeros((rows, 4))
        n = self.lib.ecb_lm_trace(self.h, _ptr(tr), rows)
        return tr[:n]
