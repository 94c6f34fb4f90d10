// Host build of the product's forward camera model (eventcalib_b200/csrc/ecb_camera.h) so the CPU test suite can check the fold,
// the distortion and the projection without a GPU.
#include "../../eventcalib_b200/csrc/ecb_camera.h"

// rho_fold and g(rho_fold) of k[5]
extern "C" void host_fold(const double *k, double *rho, double *g) {
    const EcbFold f = ecb_inverse_radial_fold_host(k);
    *rho = f.rho;
    *g = f.g;
}

// rho_d of n radii rho_u (NaN where invalid); returns the number of valid ones
extern "C" int host_distort_radius(const double *k, double rho, double g, const double *rho_u, int n, double *rho_d) {
    int nv = 0;
    for (int i = 0; i < n; ++i) {
        double d = NAN;
        if (ecb_distort_radius(k, EcbFold{rho, g}, rho_u[i], d)) ++nv;
        rho_d[i] = d;
    }
    return nv;
}

// pixels uv[n][2] of camera-frame points p[n][3] (NaN where not projectable); returns the number of valid ones
extern "C" int host_project(const double *intr, const double *p, int n, double *uv) {
    const EcbFold f = ecb_inverse_radial_fold_host(intr + 4);
    int nv = 0;
    for (int i = 0; i < n; ++i) {
        double u = NAN, v = NAN;
        if (ecb_project(intr, f, p + 3 * i, u, v)) ++nv; else u = v = NAN;
        uv[2 * i] = u;
        uv[2 * i + 1] = v;
    }
    return nv;
}
