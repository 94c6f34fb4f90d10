// Host build of the product's motion header (eventcalib_b200/csrc/ecb_motion.h) so the CPU test suite can compare the derivative
// basis, the motion and its Jacobian with scipy and finite differences without a GPU.
#include "../../eventcalib_b200/csrc/ecb_motion.h"

extern "C" void host_ders_basis(const double *knots, int span, double u, double *N, double *Nd, double *Ndd) {
    ecb_ders_basis(knots, span, u, N, Nd, Ndd);
}

// motion16 = tx ty tz qx qy qz qw, wx wy wz, vx vy vz, ax ay az; J = the dense 9 x 24 Jacobian, row major (rows w_b, v_w, a_w;
// columns per control point: rotation tangent 3, translation 3)
extern "C" void host_motion(const double *Q, const double *T, const double *N, const double *Nd, const double *Ndd, int so3,
                            double *motion16, double *J) {
    EcbMotion m;
    ecb_motion_eval(Q, T, N, Nd, Ndd, so3, m);
    const double row[16] = {m.t[0], m.t[1], m.t[2], m.q[0], m.q[1], m.q[2], m.q[3], m.w[0],
                            m.w[1], m.w[2], m.v[0], m.v[1], m.v[2], m.a[0], m.a[1], m.a[2]};
    for (int i = 0; i < 16; ++i) motion16[i] = row[i];
    if (!J) return;
    for (int e = 0; e < 9 * 24; ++e) J[e] = 0.0;
    for (int j = 0; j < 4; ++j) {
        double B[3][3];
        ecb_motion_jacobian(Q, N, Nd, so3, j, B);
        for (int k = 0; k < 3; ++k) {
            for (int r = 0; r < 3; ++r) J[r * 24 + 6 * j + k] = B[r][k];
            J[(3 + k) * 24 + 6 * j + 3 + k] = Nd[j];
            J[(6 + k) * 24 + 6 * j + 3 + k] = Ndd[j];
        }
    }
}

// the pose header's ecb_pose_eval, for the bit-for-bit comparison with the motion's pose
extern "C" void host_pose_eval(const double *Q, const double *T, const double *N, int so3, double *pose7) {
    double q[4], t[3];
    ecb_pose_eval(Q, T, N, so3, q, t);
    for (int c = 0; c < 3; ++c) pose7[c] = t[c];
    for (int c = 0; c < 4; ++c) pose7[3 + c] = q[c];
}
