// The forward camera model of the spline stage: board point -> pixel, the inverse of the back-projection in ecb_residual.h.
//
// The spline stage models distortion by the INVERSE radial polynomial (EventCalibSpline.hpp:36-63): a distorted normalised
// point x_d = ((u - cx) / fx, (v - cy) / fy) undistorts to x_u = x_d s(|x_d|^2), s(u) = 1 + k1 u + k2 u^2 + ... + k5 u^5.  In
// radii, rho_u = g(rho_d) = rho_d s(rho_d^2).  Projecting needs the inverse of g, and g need not be monotone: its derivative is
// h(rho^2) with h(u) = 1 + 3 k1 u + 5 k2 u^2 + 7 k3 u^3 + 9 k4 u^4 + 11 k5 u^5.  rho_fold^2 is the smallest positive real root of
// h (+inf when there is none); g is strictly increasing on [0, rho_fold), so it has an inverse on [0, g(rho_fold)) and nowhere
// beyond.  A fitted polynomial can fold just outside the sensor, where the fixed-point iteration x_d <- x_u / s(|x_d|^2) of
// OpenCV-style undistortion no longer converges; ecb_distort_radius uses safeguarded Newton inside the bracket [0, rho_fold].
//
// Everything here is plain C++ (host and device) so that the host build of the tests can check it without a GPU.
// ecb_inverse_radial_fold_host runs on the host once per call; the kernels receive rho_fold and g(rho_fold).
#pragma once
#include <math.h>

#include "ecb_pose.h"

#ifndef ECB_HD
#ifdef __CUDACC__
#define ECB_HD __host__ __device__ __forceinline__
#else
#define ECB_HD inline
#endif
#endif

// g(rho) = rho s(rho^2) for k[5] = k1 .. k5
ECB_HD double ecb_radial_g(const double *k, double rho) {
    const double u = rho * rho;
    return rho * (1.0 + u * (k[0] + u * (k[1] + u * (k[2] + u * (k[3] + u * k[4])))));
}

// g'(rho) = h(rho^2)
ECB_HD double ecb_radial_dg(const double *k, double rho) {
    const double u = rho * rho;
    return 1.0 + u * (3.0 * k[0] + u * (5.0 * k[1] + u * (7.0 * k[2] + u * (9.0 * k[3] + u * 11.0 * k[4]))));
}

// The fold of the camera (rho_fold, g(rho_fold)); fold = +inf and g_fold = +inf when g increases everywhere
struct EcbFold {
    double rho, g;
};

namespace ecb_camera_detail {

inline double poly(const double *a, int n, double x) {  // a[0] + a[1] x + ... + a[n] x^n
    double v = a[n];
    for (int i = n - 1; i >= 0; --i) v = v * x + a[i];
    return v;
}

// bisection of a sign change of p on [lo, hi] to full precision: stops when the midpoint is an end point (deterministic)
inline double bisect(const double *a, int n, double lo, double hi) {
    double plo = poly(a, n, lo);
    for (int it = 0; it < 2100; ++it) {
        const double m = 0.5 * (lo + hi);
        if (!(m > lo && m < hi)) break;
        const double pm = poly(a, n, m);
        if (pm == 0.0) return m;
        if ((pm < 0.0) == (plo < 0.0)) {
            lo = m;
            plo = pm;
        } else {
            hi = m;
        }
    }
    return hi;  // the first point at or past the sign change
}

// the real roots of p (degree n, a[n] != 0) in the open interval (lo, hi), ascending: p is monotone between consecutive roots of
// p', so the roots of p' (by recursion) split (lo, hi) into pieces holding at most one sign change each.  Roots of even
// multiplicity (no sign change) are not reported.  Returns the count (<= n).
inline int real_roots(const double *a, int n, double lo, double hi, double *out) {
    if (n < 1) return 0;
    double ends[7];
    int ne = 0;
    ends[ne++] = lo;
    if (n >= 2) {
        double d[5];
        for (int i = 1; i <= n; ++i) d[i - 1] = i * a[i];
        ne += real_roots(d, n - 1, lo, hi, ends + 1);
    }
    ends[ne++] = hi;
    int cnt = 0;
    for (int i = 0; i + 1 < ne; ++i) {
        const double pa = poly(a, n, ends[i]), pb = poly(a, n, ends[i + 1]);
        if (pa == 0.0 && i > 0 && ends[i] > lo) {  // a critical point that is itself a root (counted once)
            if (cnt == 0 || out[cnt - 1] != ends[i]) out[cnt++] = ends[i];
            continue;
        }
        if ((pa < 0.0 && pb > 0.0) || (pa > 0.0 && pb < 0.0)) out[cnt++] = bisect(a, n, ends[i], ends[i + 1]);
    }
    return cnt;
}

}  // namespace ecb_camera_detail

// rho_fold of the inverse radial polynomial k[5] (host): the square root of the smallest positive real root of h, by an exact
// isolation of the real roots of h on (0, B] (B: Cauchy's bound on the roots) and bisection to full precision.  Deterministic.
inline EcbFold ecb_inverse_radial_fold_host(const double *k) {
    const double a[6] = {1.0, 3.0 * k[0], 5.0 * k[1], 7.0 * k[2], 9.0 * k[3], 11.0 * k[4]};
    int n = 5;
    while (n > 0 && a[n] == 0.0) --n;
    EcbFold f{INFINITY, INFINITY};
    if (n == 0) return f;
    double bound = 0.0;  // every root has |u| <= 1 + max_i |a_i / a_n|
    for (int i = 0; i < n; ++i) bound = fmax(bound, fabs(a[i] / a[n]));
    bound = 1.0 + bound;
    if (!(bound < INFINITY)) return f;
    double roots[5];
    const int nr = ecb_camera_detail::real_roots(a, n, 0.0, bound * 2.0, roots);
    for (int i = 0; i < nr; ++i)
        if (roots[i] > 0.0) {
            f.rho = sqrt(roots[i]);
            f.g = ecb_radial_g(k, f.rho);
            break;
        }
    return f;
}

// rho_d in [0, rho_fold) with g(rho_d) = rho_u: safeguarded Newton in the bracket [0, rho_fold] (a bisection step whenever
// Newton leaves it), at most ECB_DISTORT_ITERS steps.  rho_u = 0 gives 0 and k = 0 gives rho_u, both exactly.  false (rho_d
// untouched) when rho_u >= g(rho_fold) or rho_u is not finite.
constexpr int ECB_DISTORT_ITERS = 100;
ECB_HD bool ecb_distort_radius(const double *k, EcbFold fold, double rho_u, double &rho_d) {
    if (!(rho_u >= 0.0 && rho_u < fold.g && rho_u < INFINITY)) return false;
    if (rho_u == 0.0) {
        rho_d = 0.0;
        return true;
    }
    double lo = 0.0, hi = fold.rho;
    if (!(hi < INFINITY)) {  // g increases everywhere: a finite bracket by doubling (g is an unbounded polynomial)
        hi = rho_u;
        for (int i = 0; i < 2100 && ecb_radial_g(k, hi) < rho_u; ++i) hi *= 2.0;
    }
    double x = fmin(rho_u, hi);
    for (int it = 0; it < ECB_DISTORT_ITERS; ++it) {
        const double f = ecb_radial_g(k, x) - rho_u;
        if (f == 0.0) break;
        if (f < 0.0) lo = x; else hi = x;
        double xn = x - f / ecb_radial_dg(k, x);
        if (!(xn > lo && xn < hi)) xn = 0.5 * (lo + hi);
        if (xn == x) break;
        x = xn;
    }
    rho_d = x;
    return true;
}

// pixel of a camera-frame point p (intrinsics fx fy cx cy k1 .. k5 as in ecb_residual.h); false when p.z <= 0, when its
// undistorted radius is at or past g(rho_fold), or for a non-finite input
ECB_HD bool ecb_project(const double *intr, EcbFold fold, const double p[3], double &u, double &v) {
    if (!(p[2] > 0.0)) return false;
    const double xu = p[0] / p[2], yu = p[1] / p[2];
    const double rho_u = sqrt(xu * xu + yu * yu);
    double rho_d;
    if (!ecb_distort_radius(intr + 4, fold, rho_u, rho_d)) return false;
    const double sc = rho_u > 0.0 ? rho_d / rho_u : 1.0;
    u = intr[0] * (xu * sc) + intr[2];
    v = intr[1] * (yu * sc) + intr[3];
    return true;
}

// v -> R(q) v for a unit quaternion q (x y z w); conj: R(q)^T v
ECB_HD void ecb_quat_rotate(const double q[4], const double v[3], bool conj, double o[3]) {
    const double s = conj ? -1.0 : 1.0;
    const double x = s * q[0], y = s * q[1], z = s * q[2], w = q[3];
    const double u0 = 2.0 * (y * v[2] - z * v[1]), u1 = 2.0 * (z * v[0] - x * v[2]), u2 = 2.0 * (x * v[1] - y * v[0]);
    o[0] = v[0] + w * u0 + (y * u2 - z * u1);
    o[1] = v[1] + w * u1 + (z * u0 - x * u2);
    o[2] = v[2] + w * u2 + (x * u1 - y * u0);
}

// X_w: the event pixel (ou, ov) back-projected onto the board plane z = 0 at the pose (q, t), with the operations of the residual
// (ecb_residual.h: unDistort, the third row of R(q), the ray-plane depth, q * v + t), so that X_w - L is the residual's d.
// Not finite when the ray is parallel to the plane.
ECB_HD void ecb_board_point(const double *intr, const double q[4], const double t[3], double ou, double ov, double Xw[3]) {
    const double q0 = q[0], q1 = q[1], q2 = q[2], q3 = q[3];
    const double x = (ou - intr[2]) * (1.0 / intr[0]), y = (ov - intr[3]) * (1.0 / intr[1]);
    const double r2 = x * x + y * y, r4 = r2 * r2, r6 = r4 * r2, r8 = r6 * r2, r10 = r8 * r2;
    const double s = 1.0 + intr[4] * r2 + intr[5] * r4 + intr[6] * r6 + intr[7] * r8 + intr[8] * r10;
    const double X0 = x * s, X1 = y * s;
    const double R30 = 2.0 * (q0 * q2 - q3 * q1), R31 = 2.0 * (q1 * q2 + q3 * q0), R32 = 1.0 - 2.0 * (q0 * q0 + q1 * q1);
    const double lam = -t[2] * (1.0 / (R30 * X0 + R31 * X1 + R32));
    const double v0 = lam * X0, v1 = lam * X1, v2 = lam;
    const double uv0 = 2.0 * (q1 * v2 - q2 * v1), uv1 = 2.0 * (q2 * v0 - q0 * v2), uv2 = 2.0 * (q0 * v1 - q1 * v0);
    Xw[0] = v0 + q3 * uv0 + (q1 * uv2 - q2 * uv1) + t[0];
    Xw[1] = v1 + q3 * uv1 + (q2 * uv0 - q0 * uv2) + t[1];
    Xw[2] = v2 + q3 * uv2 + (q0 * uv1 - q1 * uv0) + t[2];
}

// Reprojection error of one residual record, in pixels (the residual's correspondence seen in the image):
//   X_w = back-projection of the event pixel o onto the board plane z = 0 at the pose (q, t) (as in ecb_residual.h),
//   d = X_w - L, rim point P = L + radius d / |d|, p_c = R^T (P - t), q_px = its projection,
//   e = sign(|d| - radius) |q_px - o|   (> 0: the event lies outside the projected rim).
// NaN when |d| = 0, when the event's own distorted radius is at or past rho_fold (the model folds inside the sensor there), when
// P cannot be projected, or when a value is not finite.  This is not the distance to the projected ellipse of the circle.
ECB_HD double ecb_rim_reprojection(const double *intr, EcbFold fold, const double q[4], const double t[3], double ou, double ov,
                                   double lx, double ly, double lz, double radius) {
    const double fx = intr[0], fy = intr[1], cx = intr[2], cy = intr[3];
    const double x = (ou - cx) / fx, y = (ov - cy) / fy;
    const double r2 = x * x + y * y;
    if (!(sqrt(r2) < fold.rho)) return NAN;
    const double s = 1.0 + r2 * (intr[4] + r2 * (intr[5] + r2 * (intr[6] + r2 * (intr[7] + r2 * intr[8]))));
    const double X[3] = {x * s, y * s, 1.0};
    double Xr[3];
    ecb_quat_rotate(q, X, false, Xr);
    const double lam = -t[2] / Xr[2];
    const double d0 = lam * Xr[0] + t[0] - lx, d1 = lam * Xr[1] + t[1] - ly, d2 = lam * Xr[2] + t[2] - lz;
    const double nd = sqrt(d0 * d0 + d1 * d1 + d2 * d2);
    if (!(nd > 0.0 && nd < INFINITY)) return NAN;
    const double a = radius / nd;
    const double P[3] = {lx + a * d0 - t[0], ly + a * d1 - t[1], lz + a * d2 - t[2]};
    double pc[3], u, v;
    ecb_quat_rotate(q, P, true, pc);
    if (!ecb_project(intr, fold, pc, u, v)) return NAN;
    const double e = sqrt((u - ou) * (u - ou) + (v - ov) * (v - ov));
    if (!(e < INFINITY)) return NAN;
    return nd > radius ? e : (nd < radius ? -e : 0.0);
}
