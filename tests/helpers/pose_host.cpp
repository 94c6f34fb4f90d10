// Host build of the product's pose / pose-Jacobian header (eventcalib_b200/csrc/ecb_pose.h) so the CPU test suite can compare
// it with finite differences and with EventCalibSpline::evaluate without a GPU.
#include "../../eventcalib_b200/csrc/ecb_pose.h"
// pose7 = tx ty tz qx qy qz qw; J = the dense 6 x 24 Jacobian, row major (rows dtheta, dp; columns per control point:
// rotation tangent 3, translation 3)
extern "C" void host_pose_jacobian(const double *Q, const double *T, const double *N, int so3, double *pose7, double *J) {
    EcbPoseJac o;
    ecb_pose_jacobian(Q, T, N, so3, o);
    for (int c = 0; c < 3; ++c) pose7[c] = o.t[c];
    for (int c = 0; c < 4; ++c) pose7[3 + c] = o.q[c];
    for (int e = 0; e < 6 * 24; ++e) J[e] = 0.0;
    for (int j = 0; j < 4; ++j)
        for (int k = 0; k < 3; ++k) {
            for (int r = 0; r < 3; ++r) J[r * 24 + 6 * j + k] = o.A[j][r][k];
            J[(3 + k) * 24 + 6 * j + 3 + k] = N[j];
        }
}
