"""Deterministic synthetic circle-grid event streams in the reference's binary format.

The generator is shared by the tests, ``bench.py`` and the CLI demo; it is NOT part of the oracle.
It follows SURVEY.md §8(d): a pinhole camera whose ground-truth model *is* the calibration model of
``EventCalibSpline::unDistort`` (EventCalibSpline.hpp:36-63) looks at the asymmetric 9x4 circle board of
``parameter/event_calibration/example.yaml`` (square 5.5 cm, radius 1.75 cm; centres as in
EventCalibIni.cpp:99-106) along a smooth 6-DoF trajectory.  Each event is a rim sample with Gaussian
radial jitter, rounded to the integer pixel; the leading half-rim (w.r.t. the circle's image motion) has
polarity 1, the trailing half 0; a fraction of events is uniform background noise.  Timestamps are
strictly increasing float64 seconds.

Record format (Event.hpp:41-47 / EventStream.cpp:47-50): 25 bytes, packed, little endian:
``f64 t, f64 x, f64 y, u8 polarity``; no header.
"""
from dataclasses import dataclass, field

import numpy as np

RECORD = np.dtype([("t", "<f8"), ("x", "<f8"), ("y", "<f8"), ("p", "u1")])
assert RECORD.itemsize == 25


def inverse_radial_distortion(k):
    """PinholeCamera::inverseRadialDistortion (core/sensor/src/PinholeCamera.cpp:70-95), 4 radial terms in."""
    k0, k1, k2, k3 = [float(v) for v in k]
    b = np.zeros(5)
    b[0] = -k0
    b[1] = 3 * k0 * k0 - k1
    b[2] = -12 * k0 ** 3 + 8 * k0 * k1 - k2
    b[3] = 55 * k0 ** 4 - 55 * k0 * k0 * k1 + 5 * k1 * k1 + 10 * k0 * k2 - k3
    b[4] = -273 * k0 ** 5 + 364 * k0 ** 3 * k1 - 78 * k0 * k1 * k1 - 78 * k0 * k0 * k2 + 12 * k1 * k2 + 12 * k0 * k3
    return b


@dataclass
class Board:
    rows: int = 9
    cols: int = 4
    square: float = 5.5
    radius: float = 1.75
    asymmetric: bool = True

    def centres(self):
        c = []
        for i in range(self.rows):
            for j in range(self.cols):
                if self.asymmetric:
                    c.append(((2 * j + i % 2) * self.square, i * self.square, 0.0))
                else:
                    c.append((j * self.square, i * self.square, 0.0))
        return np.array(c)


@dataclass
class Camera:
    width: int = 346
    height: int = 260
    radial: tuple = (-0.34991902, -0.014698517, 0.59684463, 0.0)  # unit_test_inverseDistortion.cpp:10
    f: float = field(default=0.0)

    def __post_init__(self):
        if self.f == 0.0:
            self.f = 359.67525 * (self.width / 346.0)
        self.cx = (self.width - 1) / 2.0
        self.cy = (self.height - 1) / 2.0
        self.inv_poly = inverse_radial_distortion(self.radial)

    def intrinsics(self):
        """The 9-vector of EventCalibSpline (EventCalibSpline.hpp:24-34): fx fy cx cy k1..k5."""
        return np.concatenate([[self.f, self.f, self.cx, self.cy], self.inv_poly])

    def s(self, r2):
        b = self.inv_poly
        return 1 + r2 * (b[0] + r2 * (b[1] + r2 * (b[2] + r2 * (b[3] + r2 * b[4]))))

    def distort(self, xu, yu, iters=14):
        """invert the undistortion polynomial: find xd with xd * s(|xd|^2) = xu (fixed point)."""
        xd, yd = xu.copy(), yu.copy()
        for _ in range(iters):
            sc = self.s(xd * xd + yd * yd)
            xd, yd = xu / sc, yu / sc
        return xd, yd


class Trajectory:
    """Smooth camera pose (R_wb, t_wb) in the board frame: sum of sinusoids, board always in view."""

    def __init__(self, seed, board: Board, dist=75.0, rot_amp=None, orbit=False):
        r = np.random.default_rng(seed)
        c = board.centres()
        self.mid = np.array([c[:, 0].mean(), c[:, 1].mean(), 0.0])
        self.dist = dist
        self.orbit = orbit  # True: the camera orbits the board centre and keeps looking at it (large tilts stay in view)
        self.w = r.uniform(1.5, 4.5, size=(6, 3))  # rad/s
        self.ph = r.uniform(0, 2 * np.pi, size=(6, 3))
        self.amp_t = np.array([3.0, 3.0, 6.0]) / 3.0  # cm per sinusoid
        self.amp_r = np.array(rot_amp if rot_amp is not None else [0.10, 0.10, 0.15]) / 3.0  # rad per sinusoid

    def _sig(self, t, k):
        return np.sin(self.w[k][None, :] * t[:, None] + self.ph[k][None, :]).sum(axis=1)

    def pose(self, t):
        t = np.atleast_1d(np.asarray(t, np.float64))
        tw = np.stack([self.mid[0] + self.amp_t[0] * self._sig(t, 0), self.mid[1] + self.amp_t[1] * self._sig(t, 1),
                       -self.dist + self.amp_t[2] * self._sig(t, 2)], axis=1)
        a = self.amp_r[0] * self._sig(t, 3)
        b = self.amp_r[1] * self._sig(t, 4)
        c = np.pi / 2 + self.amp_r[2] * self._sig(t, 5)
        ca, sa, cb, sb, cc, sc = np.cos(a), np.sin(a), np.cos(b), np.sin(b), np.cos(c), np.sin(c)
        n = len(t)
        Rz = np.zeros((n, 3, 3)); Rx = np.zeros((n, 3, 3)); Ry = np.zeros((n, 3, 3))
        Rz[:, 0, 0] = cc; Rz[:, 0, 1] = -sc; Rz[:, 1, 0] = sc; Rz[:, 1, 1] = cc; Rz[:, 2, 2] = 1
        Rx[:, 0, 0] = 1; Rx[:, 1, 1] = ca; Rx[:, 1, 2] = -sa; Rx[:, 2, 1] = sa; Rx[:, 2, 2] = ca
        Ry[:, 0, 0] = cb; Ry[:, 0, 2] = sb; Ry[:, 1, 1] = 1; Ry[:, 2, 0] = -sb; Ry[:, 2, 2] = cb
        R = Rz @ Rx @ Ry
        if self.orbit:
            tw = (self.mid[None, :] - R[:, :, 2] * (self.dist + self.amp_t[2] * self._sig(t, 2))[:, None]
                  + R[:, :, 0] * (self.amp_t[0] * self._sig(t, 0))[:, None] + R[:, :, 1] * (self.amp_t[1] * self._sig(t, 1))[:, None])
        return R, tw

    def _dsig(self, t, k):
        return (self.w[k][None, :] * np.cos(self.w[k][None, :] * t[:, None] + self.ph[k][None, :])).sum(axis=1)

    def angular_velocity(self, t):
        """body-frame angular velocity w_b of pose()'s rotation (R_wb^T dR_wb/dt = [w_b]x), rad/s, analytic: for
        R = Rz(c) Rx(a) Ry(b), w_b = Ry^T Rx^T (c' e_z) + Ry^T (a' e_x) + b' e_y"""
        t = np.atleast_1d(np.asarray(t, np.float64))
        a, b = self.amp_r[0] * self._sig(t, 3), self.amp_r[1] * self._sig(t, 4)
        da, db, dc = self.amp_r[0] * self._dsig(t, 3), self.amp_r[1] * self._dsig(t, 4), self.amp_r[2] * self._dsig(t, 5)
        ca, sa, cb, sb = np.cos(a), np.sin(a), np.cos(b), np.sin(b)
        return np.stack([cb * da - sb * ca * dc, sa * dc + db, sb * da + cb * ca * dc], axis=1)

    def quat_xyzw(self, t):
        R, tw = self.pose(t)
        q = np.zeros((len(R), 4))
        for i, M in enumerate(R):
            tr = M.trace()
            if tr > 0:
                s = np.sqrt(tr + 1.0) * 2
                q[i] = [(M[2, 1] - M[1, 2]) / s, (M[0, 2] - M[2, 0]) / s, (M[1, 0] - M[0, 1]) / s, 0.25 * s]
            else:
                k = int(np.argmax(np.diag(M)))
                j, l = (k + 1) % 3, (k + 2) % 3
                s = np.sqrt(1.0 + M[k, k] - M[j, j] - M[l, l]) * 2
                v = np.zeros(4)
                v[k] = 0.25 * s
                v[j] = (M[j, k] + M[k, j]) / s
                v[l] = (M[l, k] + M[k, l]) / s
                v[3] = (M[l, j] - M[j, l]) / s
                q[i] = v
        # continuity of sign
        for i in range(1, len(q)):
            if np.dot(q[i], q[i - 1]) < 0:
                q[i] = -q[i]
        return q, tw


def project(cam: Camera, R, tw, Xw):
    """world point(s) -> pixel through the ground-truth model. R: (n,3,3) R_wb, tw: (n,3), Xw: (n,3)."""
    Xc = np.einsum("nji,nj->ni", R, Xw - tw)  # R^T (Xw - t)
    xu = Xc[:, 0] / Xc[:, 2]
    yu = Xc[:, 1] / Xc[:, 2]
    xd, yd = cam.distort(xu, yu)
    return cam.f * xd + cam.cx, cam.f * yd + cam.cy


def _gen_chunk(args):
    (s, e, n_events, width, height, t0, duration, seed, noise_frac, flip_frac, jitter, board, dist, k, rot_amp, traj_seed, orbit) = args
    cam = Camera(width, height)
    traj = Trajectory(traj_seed, board, dist, rot_amp, orbit)
    centres = board.centres()
    rng = np.random.default_rng([seed, k])
    dt = duration / n_events
    m = e - s
    t = t0 + (np.arange(s, e) + rng.uniform(0.05, 0.95, m)) * dt
    k = rng.integers(0, len(centres), m)
    th = rng.uniform(0, 2 * np.pi, m)
    R, tw = traj.pose(t)
    C = centres[k]
    rim = C + board.radius * np.stack([np.cos(th), np.sin(th), np.zeros(m)], axis=1)
    u, v = project(cam, R, tw, rim)
    cu, cv = project(cam, R, tw, C)
    R2, tw2 = traj.pose(t + 1e-4)
    cu2, cv2 = project(cam, R2, tw2, C)
    nx, ny = u - cu, v - cv
    nn = np.sqrt(nx * nx + ny * ny) + 1e-12
    pol = ((nx * (cu2 - cu) + ny * (cv2 - cv)) > 0)
    j = rng.normal(0, jitter, m)
    u = u + nx / nn * j
    v = v + ny / nn * j
    noise = rng.uniform(0, 1, m) < noise_frac
    nz = int(noise.sum())
    u[noise] = rng.uniform(0, width - 1, nz)
    v[noise] = rng.uniform(0, height - 1, nz)
    pol[noise] = rng.uniform(0, 1, nz) < 0.5
    if flip_frac > 0:
        fl = rng.uniform(0, 1, m) < flip_frac
        pol[fl] = ~pol[fl]
    return (t, np.clip(np.rint(u), 0, width - 1), np.clip(np.rint(v), 0, height - 1), pol.astype(np.uint8))


def make_stream(n_events, width=346, height=260, t0=5.0, duration=0.5, seed=1001, noise_frac=0.05, flip_frac=0.0,
                jitter=0.7, board: Board = None, dist=None, chunk=1 << 19, return_truth=False, workers=1, rot_amp=None, traj_seed=None,
                orbit=False):
    """Returns dict(t, x, y, p) float64/uint8 arrays (time sorted, integer-valued pixel coordinates).
    Deterministic in (seed, n_events, chunk) — independent of `workers` (processes used to generate chunks)."""
    board = board or Board()
    if dist is None:
        dist = 78.0
    if traj_seed is None:
        traj_seed = seed
    jobs = [(s, min(n_events, s + chunk), n_events, width, height, t0, duration, seed, noise_frac, flip_frac, jitter,
             board, dist, k, rot_amp, traj_seed, orbit) for k, s in enumerate(range(0, n_events, chunk))]
    if workers > 1 and len(jobs) > 1:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(min(workers, len(jobs))) as pool:
            parts = pool.map(_gen_chunk, jobs)
    else:
        parts = [_gen_chunk(j) for j in jobs]
    T = np.concatenate([p[0] for p in parts])
    X = np.concatenate([p[1] for p in parts])
    Y = np.concatenate([p[2] for p in parts])
    P = np.concatenate([p[3] for p in parts])
    out = dict(t=T, x=X, y=Y, p=P, width=width, height=height)
    if return_truth:
        out.update(camera=Camera(width, height), trajectory=Trajectory(traj_seed, board, dist, rot_amp, orbit), board=board)
    return out


def to_records(ev):
    """Pack a stream into the reference's 25-byte records (numpy structured array)."""
    rec = np.empty(len(ev["t"]), RECORD)
    rec["t"] = ev["t"]
    rec["x"] = ev["x"]
    rec["y"] = ev["y"]
    rec["p"] = ev["p"]
    return rec


def write_bin(path, ev):
    to_records(ev).tofile(path)


def read_bin(path):
    rec = np.fromfile(path, RECORD)
    return dict(t=rec["t"].copy(), x=rec["x"].copy(), y=rec["y"].copy(), p=rec["p"].copy())


def tiling_windows(t_begin, t_end, length):
    """Fixed tiling windows [k*L, (k+1)*L) expressed as the reference's CLOSED intervals: the upper bound is the
    largest double below the next window's start, so consecutive windows never share an event."""
    n = int(np.floor((t_end - t_begin) / length + 1e-9))
    a = t_begin + np.arange(n) * length
    b = np.nextafter(t_begin + (np.arange(n) + 1) * length, -np.inf)
    return np.stack([a, b], axis=1)


def gyro_samples(traj, t0, t1, rate, R_gc=np.eye(3), offset=0.0, bias=(0.0, 0.0, 0.0), noise=0.0, seed=0):
    """A gyroscope rigidly mounted with the camera of traj: stamps t = t0 + k / rate <= t1 on the gyroscope clock, readings
    w_g = R_gc w_b(t + offset) + bias + N(0, noise^2) (rad/s, gyroscope frame; R_gc rotates camera-frame vectors into the
    gyroscope frame, gyroscope stamp t is event time t + offset).  Returns (n, 4) = t wx wy wz."""
    t = t0 + np.arange(int(np.floor((t1 - t0) * rate)) + 1) / rate
    w = traj.angular_velocity(t + offset) @ np.asarray(R_gc, np.float64).T + np.asarray(bias, np.float64)
    w += np.random.default_rng(seed).normal(0.0, noise, w.shape)
    return np.column_stack([t, w])
