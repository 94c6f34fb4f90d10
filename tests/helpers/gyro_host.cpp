// Host build of the product's angular-acceleration and gyroscope headers (eventcalib_b200/csrc/ecb_motion.h, ecb_gyro.h) so the
// CPU test suite can check dw/dt and the gyroscope residual's Jacobian against finite differences without a GPU.
#include "../../eventcalib_b200/csrc/ecb_gyro.h"
#include "../../eventcalib_b200/csrc/ecb_motion.h"

// w and dw/dt (ecb_angular_velocity<true>); w alone (ecb_angular_velocity<false>) into w_only
extern "C" void host_angular_velocity(const double *Q, const double *N, const double *Nd, const double *Ndd, int so3, double *w,
                                      double *wd, double *w_only) {
    ecb_angular_velocity<true>(Q, N, Nd, Ndd, so3, w, wd);
    double unused[3];
    ecb_angular_velocity<false>(Q, N, Nd, Ndd, so3, w_only, unused);
}

// r (3) and J (3 x 7) of one sample at R_gc = q (x y z w), bias b
extern "C" void host_gyro_residual(const double *q, const double *b, const double *wc, const double *wdc, const double *wg,
                                   double *r, double *J) {
    double R[9];
    ecb_gyro_rotation(q, R);
    ecb_gyro_residual(R, b, wc, wdc, wg, r, J);
}
