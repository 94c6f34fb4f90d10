// Pose of the trajectory spline at one time and its 6 x 24 Jacobian with respect to the tangent parameters of the 4 control
// points that carry it — what ecb_pose_covariance needs to propagate the calibration's covariance to a pose.
//
// Definition.  For a time t, let s be the first segment whose knot range holds t (EventCalibSpline::time2splineIdx) and i its
// span (BsplineReal::findSpan).  The pose (R^, t^) at t is what EventCalibSpline::evaluate returns for the rotation model in
// use: quaternion model normalised sum N_j q_j, SO(3) model the cumulative spline ecb_so3::rotation_value, translation
// sum N_j t_j.  The tangent of the output has 6 values: dtheta, a body-frame rotation perturbation R = R^ Exp(dtheta) in
// radians, then dp = t - t^ in the world frame, in the units of the translation control points.  The output covariance is
// Sigma(t) = J Z_blk J^T.  J (6 x 24) is the derivative of (dtheta, dp) with respect to the tangent parameters of control
// points i-3 .. i in the order of ecb_covariance (per control point: rotation tangent 3, translation 3); the rotation tangent
// is the one of the model that was active when ecb_covariance ran: dq(delta) (x) q for quaternions, T (x) exp(delta) for SO(3).
// Z_blk is the 24 x 24 block of Z for those control points, read from the band.  No sigma^2 scaling: as for ecb_covariance,
// the covariance is sigma2 Sigma with sigma2 from ecb_covariance_summary.
//
// J is sparse: the rotation rows of control point j are a 3 x 3 block A_j (zero in the translation columns), the translation
// rows are N_j I3 (zero in the rotation columns).  The header is plain C++ so that the host build (tests) can check it against
// finite differences without a GPU.
#pragma once
#include "ecb_so3.h"

struct EcbPoseJac {
    double q[4];        // rotation x y z w
    double t[3];        // translation
    double A[4][3][3];  // A[j][r][k] = d dtheta_r / d delta_k of control point j; the translation block of j is N_j I3
};

// dtheta of a first-order change dq of the unit quaternion q:  q (x) (dtheta / 2, 1) = q + dq  =>  dtheta = 2 vec(q^* (x) dq)
ECB_HD void ecb_pose_dtheta(const double q[4], const double dq[4], double out[3]) {
    // vec(a (x) b) = a_w b_v + b_w a_v + a_v x b_v with a = q^* = (-q_v, q_w)
    out[0] = 2.0 * (q[3] * dq[0] - dq[3] * q[0] - (q[1] * dq[2] - q[2] * dq[1]));
    out[1] = 2.0 * (q[3] * dq[1] - dq[3] * q[1] - (q[2] * dq[0] - q[0] * dq[2]));
    out[2] = 2.0 * (q[3] * dq[2] - dq[3] * q[2] - (q[0] * dq[1] - q[1] * dq[0]));
}

// The pose alone (rotation q = x y z w, translation t): the sums of ecb_pose_jacobian, without the Jacobian.
ECB_HD void ecb_pose_eval(const double *Q, const double *T, const double N[4], int so3, double q[4], double t[3]) {
    for (int c = 0; c < 3; ++c) {
        double v = 0.0;
        for (int j = 0; j < 4; ++j) v += N[j] * T[3 * j + c];
        t[c] = v;
    }
    if (so3) {
        double beta[3];
        ecb_so3::cumulative_basis(N, beta);
        ecb_so3::rotation_value(Q, beta, q);
        return;
    }
    double n2 = 0.0;
    for (int c = 0; c < 4; ++c) {
        double v = 0.0;
        for (int j = 0; j < 4; ++j) v += N[j] * Q[4 * j + c];
        q[c] = v;
        n2 += v * v;
    }
    const double nz = sqrt(n2);
    for (int c = 0; c < 4; ++c) q[c] /= nz;
}

// Q: 4 rotation control points (x y z w each), T: 4 translation control points, N: the 4 basis values N_{i-3..i}(t);
// so3: 0 normalised quaternion spline, 1 cumulative SO(3) spline.
ECB_HD void ecb_pose_jacobian(const double *Q, const double *T, const double N[4], int so3, EcbPoseJac &o) {
    for (int c = 0; c < 3; ++c) {  // EventCalibSpline::evaluate, same order of the sum
        double v = 0.0;
        for (int j = 0; j < 4; ++j) v += N[j] * T[3 * j + c];
        o.t[c] = v;
    }
    if (so3) {
        double beta[3];
        ecb_so3::cumulative_basis(N, beta);
        ecb_so3::rotation_value(Q, beta, o.q);
#pragma unroll 1
        for (int j = 0; j < 4; ++j) {  // one dual-number spline at a time (unrolled, the four need more than 255 registers)
            double dq[4][3];
            ecb_so3::rotation_tangent(Q, beta, j, dq);
            for (int k = 0; k < 3; ++k) {
                const double d[4] = {dq[0][k], dq[1][k], dq[2][k], dq[3][k]};
                double th[3];
                ecb_pose_dtheta(o.q, d, th);
                for (int r = 0; r < 3; ++r) o.A[j][r][k] = th[r];
            }
        }
        return;
    }
    double n2 = 0.0;
    for (int c = 0; c < 4; ++c) {
        double v = 0.0;
        for (int j = 0; j < 4; ++j) v += N[j] * Q[4 * j + c];
        o.q[c] = v;
        n2 += v * v;
    }
    const double nz = sqrt(n2);
    for (int c = 0; c < 4; ++c) o.q[c] /= nz;
    // q = q~ / |q~| with q~ = sum N_j Q_j:  dq = (I - q q^T) dq~ / |q~|.  The q q^T part adds nothing to dtheta (vec(q^* (x) q)
    // = 0), so dtheta = 2 vec(q^* (x) dq~) / |q~| with dq~ = N_j P(Q_j) delta, P the 4 x 3 Plus Jacobian of Ceres'
    // EigenQuaternionParameterization (ecb_residual.h): its columns are (delta, 0) (x) Q_j for delta = e_0, e_1, e_2.
    for (int j = 0; j < 4; ++j) {
        const double x = Q[4 * j], y = Q[4 * j + 1], z = Q[4 * j + 2], w = Q[4 * j + 3];
        const double P[3][4] = {{w, -z, y, -x}, {z, w, -x, -y}, {-y, x, w, -z}};
        const double s = N[j] / nz;
        for (int k = 0; k < 3; ++k) {
            const double d[4] = {s * P[k][0], s * P[k][1], s * P[k][2], s * P[k][3]};
            double th[3];
            ecb_pose_dtheta(o.q, d, th);
            for (int r = 0; r < 3; ++r) o.A[j][r][k] = th[r];
        }
    }
}
