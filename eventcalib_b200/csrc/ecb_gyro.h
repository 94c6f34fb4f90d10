// One gyroscope sample against the trajectory's angular velocity: the residual and its 3 x 7 Jacobian that ecb_gyro_calibrate
// sums into its normal equations.
//
// Model: w_g = R_gc w_c(t + d) + b + noise, with w_c the body-frame angular velocity of the spline (ecb_angular_velocity),
// R_gc the rotation from camera to gyroscope frame, d the time offset (gyroscope stamp t is event time t + d) and b the bias.
//   r = R_gc w_c(t + d) + b - w_g
//   J = dr / d(delta, d, b) = [ -[R_gc w_c]x, R_gc dw_c/dt, I3 ] with R_gc = Exp(delta) R^_gc (left perturbation, gyroscope frame).
//
// Plain C++ for host and device, so that the host build (tests) can check it against finite differences without a GPU.
#pragma once
#include "ecb_so3.h"

// row-major rotation matrix of the unit quaternion q = (x y z w)
ECB_HD void ecb_gyro_rotation(const double q[4], double R[9]) {
    const double x = q[0], y = q[1], z = q[2], w = q[3];
    R[0] = 1.0 - 2.0 * (y * y + z * z), R[1] = 2.0 * (x * y - z * w), R[2] = 2.0 * (x * z + y * w);
    R[3] = 2.0 * (x * y + z * w), R[4] = 1.0 - 2.0 * (x * x + z * z), R[5] = 2.0 * (y * z - x * w);
    R[6] = 2.0 * (x * z - y * w), R[7] = 2.0 * (y * z + x * w), R[8] = 1.0 - 2.0 * (x * x + y * y);
}

// r (3) of one sample; with J (3 x 7 row major, columns delta 3, d, b 3) also its Jacobian, which needs wdc = dw_c/dt
ECB_HD void ecb_gyro_residual(const double R[9], const double b[3], const double wc[3], const double wdc[3], const double wg[3],
                              double r[3], double *J) {
    double a[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        a[i] = R[3 * i] * wc[0] + R[3 * i + 1] * wc[1] + R[3 * i + 2] * wc[2];
        r[i] = a[i] + b[i] - wg[i];
    }
    if (!J) return;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        double *Ji = J + 7 * i;
        Ji[0] = Ji[1] = Ji[2] = 0.0;
        Ji[3] = R[3 * i] * wdc[0] + R[3 * i + 1] * wdc[1] + R[3 * i + 2] * wdc[2];
        Ji[4] = Ji[5] = Ji[6] = 0.0;
        Ji[4 + i] = 1.0;
    }
    // -[a]x
    J[1] = a[2], J[2] = -a[1];
    J[7] = -a[2], J[9] = a[0];
    J[14] = a[1], J[15] = -a[0];
}
