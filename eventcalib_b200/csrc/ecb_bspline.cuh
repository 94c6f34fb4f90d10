// Cubic B-spline span search and basis on the device (BsplineReal.hpp:208-231, 107-145), shared by the cost evaluation
// (ecb_cost.cu) and the pose covariance (ecb_pose_cov.cu).  knots: one clamped knot vector of nk = n_cp + 4 entries.
#pragma once
#include <cuda_runtime.h>

__device__ __forceinline__ int find_span_dev(const double *knots, int nk, double u) {  // BsplineReal.hpp:208-231
    const int degree = 3;
    const int n = nk - 2 - degree;
    if (u == knots[n + 1]) return n;
    int low = degree, high = n + 1, mid = (low + high) / 2;
    while (u < knots[mid] || u >= knots[mid + 1]) {
        if (u < knots[mid]) high = mid; else low = mid;
        mid = (low + high) / 2;
    }
    return mid;
}

// same span (the one with knots[mid] <= u < knots[mid+1] is unique) from a proportional guess and a short walk: the
// reference's interior knots are nearly uniform (NURBS-book eq. 9.68), so the dependent-load chain of the bisection goes away
__device__ __forceinline__ int find_span_guess(const double *knots, int nk, double u) {
    const int degree = 3;
    const int n = nk - 2 - degree;
    if (u == knots[n + 1]) return n;
    const double k0 = knots[degree], k1 = knots[n + 1];
    int mid = degree + (int) ((u - k0) / (k1 - k0) * (double) (n + 1 - degree));
    mid = max(degree, min(n, mid));
    for (int s = 0; s < 8 && mid > degree && u < knots[mid]; ++s) --mid;
    for (int s = 0; s < 8 && mid < n && u >= knots[mid + 1]; ++s) ++mid;
    if (u < knots[mid] || u >= knots[mid + 1]) return find_span_dev(knots, nk, u);
    return mid;
}

__device__ __forceinline__ void basis_dev(const double *knots, int span, double u, double *N) {  // BsplineReal.hpp:107-145
    double ndu[4][4], left[4], right[4];
    ndu[0][0] = 1;
#pragma unroll
    for (int j = 1; j <= 3; j++) {
        left[j] = u - knots[span + 1 - j];
        right[j] = knots[span + j] - u;
        double saved = 0.0;
#pragma unroll
        for (int r = 0; r < j; ++r) {
            ndu[j][r] = right[r + 1] + left[j - r];
            double temp = __ddiv_rn(ndu[r][j - 1], ndu[j][r]);
            ndu[r][j] = __dadd_rn(saved, __dmul_rn(right[r + 1], temp));
            saved = __dmul_rn(left[j - r], temp);
        }
        ndu[j][j] = saved;
    }
#pragma unroll
    for (int j = 0; j <= 3; j++) N[j] = ndu[j][3];
}
