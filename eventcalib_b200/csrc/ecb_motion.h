// Motion of the trajectory spline at one time — body angular velocity, world velocity and acceleration — and its 9 x 24
// Jacobian with respect to the tangent parameters of the 4 control points that carry it: what ecb_trajectory_motion and
// ecb_motion_covariance evaluate.
//
// Definition.  For a time t, let s be the first segment whose knot range holds t (EventCalibSpline::time2splineIdx) and i its
// span (BsplineReal::findSpan).  N_j, Nd_j and Ndd_j are the cubic basis functions N_{i-3..i} and their first and second time
// derivatives on the same clamped, non-uniform knots (NURBS-book algorithm A2.3, BsplineReal::dersBasisFuns with derivative
// limit 2; N bit for bit the basis of basis_dev).
//   pose   (R^, t^) = ecb_pose_eval, bit for bit what ecb_pose_covariance returns.
//   v_w    = sum Nd_j T_j,  a_w = sum Ndd_j T_j: world frame, translation units per time unit and per time unit squared.
//   w_b    body-frame angular velocity, R^T dR/dt = [w_b]x, radians per time unit:
//          quaternion model (q = q~ / |q~|, q~ = sum N_j Q_j):  w_b = 2 vec(q~^* (x) q~') / |q~|^2 with q~' = sum Nd_j Q_j (the
//          q q^T part of the normalisation drops out, vec(q^* (x) q) = 0);
//          SO(3) model (R = R0 E1 E2 E3, E_k = Exp(b_k d_k), d_k = Log(R_{k-1}^-1 R_k), ecb_so3::spline_rotation):
//          w_b = sum_k b'_k (E_{k+1} .. E3)^T d_k, b' the cumulative sum of Nd as b is of N.
//   dw_b/dt body angular acceleration (ecb_angular_velocity<true>, for the gyroscope calibration), from N, Nd and Ndd.
// The covariance of (w_b, v_w, a_w) is Sigma_m(t) = J Z_blk J^T (9 x 9).  J (9 x 24) is the derivative with respect to the tangent
// parameters of control points i-3 .. i in the order and rotation model of ecb_covariance (per control point: rotation tangent
// 3, translation 3).  J is sparse: the w_b rows of control point j are a 3 x 3 block B_j = d w_b / d delta_j (zero in the
// translation columns), the v_w and a_w rows are Nd_j I3 and Ndd_j I3 (zero in the rotation columns).  B_j comes from w_b
// evaluated in the dual numbers of ecb_so3 with control point j lifted along its tangent: dq(delta) (x) Q_j for quaternions
// (Ceres' EigenQuaternionParameterization), Q_j (x) exp(delta) for SO(3).  No sigma^2 scaling, as for ecb_pose_covariance.
//
// Plain C++ for host and device, so that the host build (tests) can check it against finite differences without a GPU.
#pragma once
#include "ecb_pose.h"

// the operations of basis_dev without contraction on the device (its N, bit for bit); the host build uses -ffp-contract=off
#ifdef __CUDA_ARCH__
#define ECB_MOT_MUL(a, b) __dmul_rn(a, b)
#define ECB_MOT_ADD(a, b) __dadd_rn(a, b)
#define ECB_MOT_DIV(a, b) __ddiv_rn(a, b)
#else
#define ECB_MOT_MUL(a, b) ((a) * (b))
#define ECB_MOT_ADD(a, b) ((a) + (b))
#define ECB_MOT_DIV(a, b) ((a) / (b))
#endif

// NURBS-book A2.3 for degree 3 and derivatives up to 2: N, Nd, Ndd = the basis N_{span-3..span}(u) and its first and second
// derivative in u.  knots: one clamped knot vector, span as find_span_dev returns it.
ECB_HD void ecb_ders_basis(const double *knots, int span, double u, double N[4], double Nd[4], double Ndd[4]) {
    double ndu[4][4], left[4], right[4];
    ndu[0][0] = 1.0;
#pragma unroll
    for (int j = 1; j <= 3; ++j) {  // the order of operations of basis_dev
        left[j] = u - knots[span + 1 - j];
        right[j] = knots[span + j] - u;
        double saved = 0.0;
#pragma unroll
        for (int r = 0; r < j; ++r) {
            ndu[j][r] = right[r + 1] + left[j - r];
            const double temp = ECB_MOT_DIV(ndu[r][j - 1], ndu[j][r]);
            ndu[r][j] = ECB_MOT_ADD(saved, ECB_MOT_MUL(right[r + 1], temp));
            saved = ECB_MOT_MUL(left[j - r], temp);
        }
        ndu[j][j] = saved;
    }
    double ders[3][4];
#pragma unroll
    for (int j = 0; j <= 3; ++j) ders[0][j] = ndu[j][3];
#pragma unroll
    for (int r = 0; r <= 3; ++r) {
        double a[2][4];
        int s1 = 0, s2 = 1;
        a[0][0] = 1.0;
#pragma unroll
        for (int k = 1; k <= 2; ++k) {
            double d = 0.0;
            const int rk = r - k, pk = 3 - k;
            if (r >= k) {
                a[s2][0] = a[s1][0] / ndu[pk + 1][rk];
                d = a[s2][0] * ndu[rk][pk];
            }
            const int j1 = rk >= -1 ? 1 : -rk;
            const int j2 = (r - 1 <= pk) ? k - 1 : 3 - r;
#pragma unroll
            for (int j = j1; j <= j2; ++j) {
                a[s2][j] = (a[s1][j] - a[s1][j - 1]) / ndu[pk + 1][rk + j];
                d += a[s2][j] * ndu[rk + j][pk];
            }
            if (r <= pk) {
                a[s2][k] = -a[s1][k - 1] / ndu[pk + 1][r];
                d += a[s2][k] * ndu[r][pk];
            }
            ders[k][r] = d;
            const int t = s1;
            s1 = s2;
            s2 = t;
        }
    }
#pragma unroll
    for (int j = 0; j <= 3; ++j) {
        N[j] = ders[0][j];
        Nd[j] = 3.0 * ders[1][j];
        Ndd[j] = 6.0 * ders[2][j];
    }
}

namespace ecb_motion {

using ecb_so3::Quat;

// R^T w for the unit quaternion q:  w - 2 s (v x w) + 2 v x (v x w),  q = (v, s)
template <class S>
ECB_HD void rotate_inv(const Quat<S> &q, S w[3]) {
    const S c0 = q.y * w[2] - q.z * w[1], c1 = q.z * w[0] - q.x * w[2], c2 = q.x * w[1] - q.y * w[0];  // v x w
    const S e0 = q.y * c2 - q.z * c1, e1 = q.z * c0 - q.x * c2, e2 = q.x * c1 - q.y * c0;              // v x (v x w)
    w[0] = w[0] - 2.0 * (q.w * c0) + 2.0 * e0;
    w[1] = w[1] - 2.0 * (q.w * c1) + 2.0 * e1;
    w[2] = w[2] - 2.0 * (q.w * c2) + 2.0 * e2;
}

// quaternion model: w = 2 vec(q~^* (x) q~') / |q~|^2; vec(a (x) b) = a_w b_v + b_w a_v + a_v x b_v with a = q~^* = (-q~_v, q~_w).
// DOT: also wd = dw/dt = 2 vec(q~^* (x) q~'') / |q~|^2 - 2 (q~ . q~') / |q~|^2 w (vec(q~'^* (x) q~') = 0), q~'' = sum Ndd_j Q_j.
template <class S, bool DOT = false>
ECB_HD void omega_quat(const Quat<S> R[4], const double N[4], const double Nd[4], S w[3], const double *Ndd = nullptr,
                       S *wd = nullptr) {
    S p[4], d[4], e[4];
    const S zero = ecb_so3::Lift<S>::of(0.0);
#pragma unroll
    for (int c = 0; c < 4; ++c) p[c] = d[c] = e[c] = zero;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const S Rc[4] = {R[j].x, R[j].y, R[j].z, R[j].w};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            p[c] = p[c] + N[j] * Rc[c];
            d[c] = d[c] + Nd[j] * Rc[c];
            if constexpr (DOT) e[c] = e[c] + Ndd[j] * Rc[c];
        }
    }
    const S n2 = p[0] * p[0] + p[1] * p[1] + p[2] * p[2] + p[3] * p[3];
    const S s = 2.0 / n2;
    w[0] = s * (p[3] * d[0] - d[3] * p[0] - (p[1] * d[2] - p[2] * d[1]));
    w[1] = s * (p[3] * d[1] - d[3] * p[1] - (p[2] * d[0] - p[0] * d[2]));
    w[2] = s * (p[3] * d[2] - d[3] * p[2] - (p[0] * d[1] - p[1] * d[0]));
    if constexpr (DOT) {
        const S f = (p[0] * d[0] + p[1] * d[1] + p[2] * d[2] + p[3] * d[3]) * s;
        wd[0] = s * (p[3] * e[0] - e[3] * p[0] - (p[1] * e[2] - p[2] * e[1])) - f * w[0];
        wd[1] = s * (p[3] * e[1] - e[3] * p[1] - (p[2] * e[0] - p[0] * e[2])) - f * w[1];
        wd[2] = s * (p[3] * e[2] - e[3] * p[2] - (p[0] * e[1] - p[1] * e[0])) - f * w[2];
    }
}

// SO(3) model: w_1 = b'_1 d_1, w_k = E_k^T w_{k-1} + b'_k d_k, w_b = w_3 (= sum_k b'_k (E_{k+1} .. E3)^T d_k).
// DOT: also wd = dw/dt from d(E_k^T)/dt = -[b'_k d_k]x E_k^T: wd_1 = b''_1 d_1, wd_k = E_k^T wd_{k-1} + (E_k^T w_{k-1}) x (b'_k d_k)
// + b''_k d_k, b'' the cumulative sum of Ndd (Sommer et al., CVPR 2020).
template <class S, bool DOT = false>
ECB_HD void omega_so3(const Quat<S> R[4], const double beta[3], const double dbeta[3], S w[3], const double *ddbeta = nullptr,
                      S *wd = nullptr) {
#pragma unroll
    for (int k = 1; k <= 3; ++k) {
        S d[3];
        ecb_so3::so3_log(ecb_so3::qmul(ecb_so3::qinv(R[k - 1]), R[k]), d);
        if (k > 1) {
            const S bd[3] = {beta[k - 1] * d[0], beta[k - 1] * d[1], beta[k - 1] * d[2]};
            const Quat<S> E = ecb_so3::so3_exp(bd);
            rotate_inv(E, w);
            if constexpr (DOT) {
                const S v[3] = {dbeta[k - 1] * d[0], dbeta[k - 1] * d[1], dbeta[k - 1] * d[2]};
                rotate_inv(E, wd);
                wd[0] = wd[0] + (w[1] * v[2] - w[2] * v[1]) + ddbeta[k - 1] * d[0];
                wd[1] = wd[1] + (w[2] * v[0] - w[0] * v[2]) + ddbeta[k - 1] * d[1];
                wd[2] = wd[2] + (w[0] * v[1] - w[1] * v[0]) + ddbeta[k - 1] * d[2];
            }
#pragma unroll
            for (int c = 0; c < 3; ++c) w[c] = w[c] + dbeta[k - 1] * d[c];
        } else {
#pragma unroll
            for (int c = 0; c < 3; ++c) w[c] = dbeta[0] * d[c];
            if constexpr (DOT)
#pragma unroll
                for (int c = 0; c < 3; ++c) wd[c] = ddbeta[0] * d[c];
        }
    }
}

}  // namespace ecb_motion

// pose q (x y z w), t; angular velocity w; velocity v; acceleration a
struct EcbMotion {
    double q[4], t[3], w[3], v[3], a[3];
};

// Q: 4 rotation control points (x y z w each), T: 4 translation control points, N / Nd / Ndd: ecb_ders_basis;
// so3: 0 normalised quaternion spline, 1 cumulative SO(3) spline.
ECB_HD void ecb_motion_eval(const double *Q, const double *T, const double N[4], const double Nd[4], const double Ndd[4], int so3,
                            EcbMotion &m) {
    ecb_pose_eval(Q, T, N, so3, m.q, m.t);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        double v = 0.0, a = 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            v += Nd[j] * T[3 * j + c];
            a += Ndd[j] * T[3 * j + c];
        }
        m.v[c] = v;
        m.a[c] = a;
    }
    ecb_so3::Quat<double> R[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) R[j] = ecb_so3::Quat<double>{Q[4 * j], Q[4 * j + 1], Q[4 * j + 2], Q[4 * j + 3]};
    if (so3) {
        double beta[3], dbeta[3];
        ecb_so3::cumulative_basis(N, beta);
        ecb_so3::cumulative_basis(Nd, dbeta);
        ecb_motion::omega_so3<double>(R, beta, dbeta, m.w);
    } else {
        ecb_motion::omega_quat<double>(R, N, Nd, m.w);
    }
}

// B[r][k] = d w_r / d delta_k of control point j (0 .. 3): w_b in dual numbers with Q_j lifted along its tangent
ECB_HD void ecb_motion_jacobian(const double *Q, const double N[4], const double Nd[4], int so3, int j, double B[3][3]) {
    using ecb_so3::D3;
    using ecb_so3::mk;
    ecb_so3::Quat<D3> R[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) R[i] = ecb_so3::Quat<D3>{mk(Q[4 * i]), mk(Q[4 * i + 1]), mk(Q[4 * i + 2]), mk(Q[4 * i + 3])};
    const double x = Q[4 * j], y = Q[4 * j + 1], z = Q[4 * j + 2], w = Q[4 * j + 3];
    // column k of d Q_j(delta) / d delta at 0: (e_k / 2, 0) applied on the right for SO(3) (ecb_so3::rotation_tangent), the
    // Plus Jacobian columns (e_k, 0) (x) Q_j of EigenQuaternionParameterization (ecb_pose.h) for quaternions
    const double P3[3][4] = {{0.5 * w, 0.5 * z, -0.5 * y, -0.5 * x}, {-0.5 * z, 0.5 * w, 0.5 * x, -0.5 * y},
                             {0.5 * y, -0.5 * x, 0.5 * w, -0.5 * z}};
    const double P4[3][4] = {{w, -z, y, -x}, {z, w, -x, -y}, {-y, x, w, -z}};
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (i == j)
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const double *P = so3 ? P3[k] : P4[k];
                R[i].x.d[k] = P[0];
                R[i].y.d[k] = P[1];
                R[i].z.d[k] = P[2];
                R[i].w.d[k] = P[3];
            }
    D3 om[3];
    if (so3) {
        double beta[3], dbeta[3];
        ecb_so3::cumulative_basis(N, beta);
        ecb_so3::cumulative_basis(Nd, dbeta);
        ecb_motion::omega_so3<D3>(R, beta, dbeta, om);
    } else {
        ecb_motion::omega_quat<D3>(R, N, Nd, om);
    }
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int k = 0; k < 3; ++k) B[r][k] = om[r].d[k];
}

// Body angular velocity w (bit for bit ecb_motion_eval's: the same omega_quat / omega_so3) and, with DOT, its time derivative wd
// (body angular acceleration, radians per time unit squared) from the rotation control points Q and N / Nd / Ndd of
// ecb_ders_basis; so3 as for ecb_motion_eval.  Without DOT, Ndd and wd are not read.
template <bool DOT>
ECB_HD void ecb_angular_velocity(const double *Q, const double N[4], const double Nd[4], const double Ndd[4], int so3, double w[3],
                                 double wd[3]) {
    ecb_so3::Quat<double> R[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) R[j] = ecb_so3::Quat<double>{Q[4 * j], Q[4 * j + 1], Q[4 * j + 2], Q[4 * j + 3]};
    if (so3) {
        double beta[3], dbeta[3], ddbeta[3];
        ecb_so3::cumulative_basis(N, beta);
        ecb_so3::cumulative_basis(Nd, dbeta);
        if constexpr (DOT) ecb_so3::cumulative_basis(Ndd, ddbeta);
        ecb_motion::omega_so3<double, DOT>(R, beta, dbeta, w, ddbeta, wd);
    } else {
        ecb_motion::omega_quat<double, DOT>(R, N, Nd, w, Ndd, wd);
    }
}
