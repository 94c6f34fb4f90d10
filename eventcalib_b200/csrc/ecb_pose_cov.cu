// Covariance of the trajectory's pose at any time: Sigma(t) = J Z_blk J^T (definition in ecb_pose.h), from the Z and x that the
// last successful ecb_covariance left on the context and the knots of ecb_cost_setup.
//
//   k_pose_cov   one thread per query: segment (first whose knot range holds t), span and basis (ecb_bspline.cuh), pose and
//                6 x 24 Jacobian (ecb_pose.h), then Sigma from the lower triangle of the 24 x 24 block of Z in the band
//                (300 doubles, 160 KB for the whole band at D = 843: it stays in L2 / L1, and sorted queries read the same
//                block as their neighbours).  Each query is computed alone in a fixed order: its output does not depend on
//                the batch.  FP64.
#include <algorithm>

#include "ecb_bspline.cuh"
#include "ecb_common.cuh"
#include "ecb_pose.h"

namespace {

constexpr int POSE_THREADS = 128;
constexpr int64_t POSE_CHUNK = 1 << 20;  // queries per staged round of the host variant

// Sigma = sum_c (v_c J_c^T + J_c v_c^T) with v_c = sum_{r > c} Z_rc J_r + Z_cc J_c / 2 over the columns J_c of J: only the
// lower triangle of Z is read, and Sigma comes out exactly symmetric.  Zc(c) points at Z(c .. 23, c) of the block.
__device__ __forceinline__ void pose_sigma(const EcbPoseJac &P, const double N[4], const double *__restrict__ Zb, double S[6][6]) {
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int l = 0; l < 6; ++l) S[i][l] = 0.0;
#pragma unroll
    for (int c = 0; c < 24; ++c) {
        const double *Zc = Zb + c * 24;  // band column c of the block: Z(c + r, c) at Zc[r]
        double v[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll
        for (int r = c; r < 24; ++r) {
            double z = __ldg(Zc + (r - c));
            if (r == c) z *= 0.5;
            const int jr = r / 6, kr = r % 6;
            if (kr < 3) {
                v[0] += z * P.A[jr][0][kr];
                v[1] += z * P.A[jr][1][kr];
                v[2] += z * P.A[jr][2][kr];
            } else {
                v[kr] += z * N[jr];
            }
        }
        const int jc = c / 6, kc = c % 6;
        if (kc < 3) {  // J_c = (A_jc[:, kc], 0)
            const double a[3] = {P.A[jc][0][kc], P.A[jc][1][kc], P.A[jc][2][kc]};
#pragma unroll
            for (int i = 0; i < 3; ++i) {
#pragma unroll
                for (int l = i; l < 3; ++l) S[i][l] += v[i] * a[l] + a[i] * v[l];
#pragma unroll
                for (int l = 3; l < 6; ++l) S[i][l] += a[i] * v[l];
            }
        } else {  // J_c = N_jc e_kc
            const double nn = N[jc];
#pragma unroll
            for (int i = 0; i < 6; ++i) {
                if (i < kc) S[i][kc] += v[i] * nn;
                else if (i == kc) S[i][i] += 2.0 * v[i] * nn;
                else S[kc][i] += nn * v[i];
            }
        }
    }
}

template <int SO3>
__global__ void __launch_bounds__(POSE_THREADS) k_pose_cov(const double *__restrict__ times, int64_t n, EcbSplineView sv,
                                                           const double *__restrict__ x, const double *__restrict__ Zb,
                                                           double *__restrict__ pose, double *__restrict__ cov,
                                                           unsigned long long *__restrict__ n_valid) {
    const int64_t k = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    bool valid = false;
    if (k < n) {
        const double u = times[k];
        const double *kn = nullptr;
        int nk = 0;
        const int s = sv.segment(u, &kn, &nk);
        valid = s >= 0;
        double out[7], S[6][6];
        if (valid) {
            const int span = find_span_dev(kn, nk, u);
            double N[4];
            basis_dev(kn, span, u, N);
            const int c0 = sv.cp_off[s] + span - 3;
            // the Jacobian of each thread in shared memory (43 doubles: an odd stride, conflict-free): in registers, next to the
            // dual numbers of the SO(3) tangent, it would spill
            __shared__ EcbPoseJac sP[POSE_THREADS];
            EcbPoseJac &P = sP[threadIdx.x];
            ecb_pose_jacobian(x + 9 + 4 * (size_t) c0, x + 9 + 4 * (size_t) sv.total_cp + 3 * (size_t) c0, N, SO3, P);
            pose_sigma(P, N, Zb + (size_t) c0 * 6 * 24, S);
            out[0] = P.t[0], out[1] = P.t[1], out[2] = P.t[2];
            out[3] = P.q[0], out[4] = P.q[1], out[5] = P.q[2], out[6] = P.q[3];
        } else {
#pragma unroll
            for (int i = 0; i < 7; ++i) out[i] = NAN;
#pragma unroll
            for (int i = 0; i < 6; ++i)
#pragma unroll
                for (int l = i; l < 6; ++l) S[i][l] = NAN;
        }
        if (pose) {
            double *p = pose + 7 * k;
#pragma unroll
            for (int i = 0; i < 7; ++i) p[i] = out[i];
        }
        if (cov) {
            double *p = cov + 36 * k;
#pragma unroll
            for (int i = 0; i < 6; ++i)
#pragma unroll
                for (int l = 0; l < 6; ++l) p[6 * i + l] = i <= l ? S[i][l] : S[l][i];
        }
    }
    if (n_valid) {
        const unsigned m = __ballot_sync(0xffffffffu, valid);
        if ((threadIdx.x & 31) == 0 && m) atomicAdd(n_valid, (unsigned long long) __popc(m));
    }
}

// the Z, x and knots a query reads; ECB_ERR_STATE unless the last ecb_covariance succeeded after the last ecb_cost_setup /
// ecb_cost_set_rotation_model
int pose_state(ecb_ctx *ctx, EcbSplineView &sv, EcbCovView &cv) {
    if (ecb_cost_spline_view(ctx, &sv) != ECB_OK) return ecb_fail(ctx, ECB_ERR_STATE, "pose covariance: ecb_cost_setup first");
    if (ecb_covariance_view(ctx, &cv) != ECB_OK)
        return ecb_fail(ctx, ECB_ERR_STATE, "pose covariance: no successful ecb_covariance on this context");
    if (cv.spline_gen != ctx->spline_gen || cv.so3 != sv.so3 || cv.total_cp != sv.total_cp)
        return ecb_fail(ctx, ECB_ERR_STATE, "pose covariance: ecb_cost_setup or ecb_cost_set_rotation_model ran after ecb_covariance");
    return ECB_OK;
}

int pose_launch(ecb_ctx *ctx, const EcbSplineView &sv, const EcbCovView &cv, const double *d_times, int64_t n, double *d_pose,
                double *d_cov, unsigned long long *d_count) {
    if (n == 0) return ECB_OK;
    const int64_t blocks = (n + POSE_THREADS - 1) / POSE_THREADS;
    auto kern = cv.so3 ? k_pose_cov<1> : k_pose_cov<0>;
    kern<<<(unsigned) blocks, POSE_THREADS, 0, ctx->stream>>>(d_times, n, sv, cv.x, cv.Zb, d_pose, d_cov, d_count);
    ECB_LAUNCHED(ctx);
    return ecb_check(ctx, cudaGetLastError(), "k_pose_cov");
}

}  // namespace

extern "C" {

int ecb_pose_covariance_device(ecb_ctx *ctx, const double *d_times, int64_t n, double *d_pose, double *d_cov, int64_t *n_valid) {
    if (!ctx || n < 0 || (n > 0 && !d_times)) return ECB_ERR_ARG;
    if (n > (int64_t) INT32_MAX * POSE_THREADS) return ecb_fail(ctx, ECB_ERR_ARG, "pose covariance: %lld queries in one call", (long long) n);
    cudaSetDevice(ctx->device);
    EcbSplineView sv;
    EcbCovView cv;
    int rc;
    if ((rc = pose_state(ctx, sv, cv))) return rc;
    unsigned long long *d_count = nullptr;
    if (n_valid) {
        if ((rc = ecb_reserve(ctx, ctx->pose_io, 8))) return rc;
        d_count = (unsigned long long *) ctx->pose_io.p;
        ECB_CUDA(ctx, cudaMemsetAsync(d_count, 0, 8, ctx->stream));
    }
    if ((rc = pose_launch(ctx, sv, cv, d_times, n, d_pose, d_cov, d_count))) return rc;
    if (n_valid) {
        unsigned long long c = 0;
        if ((rc = ecb_d2h(ctx, &c, d_count, 8))) return rc;
        *n_valid = (int64_t) c;
    }
    return ECB_OK;
}

int ecb_pose_covariance(ecb_ctx *ctx, const double *times, int64_t n, double *pose, double *cov, int64_t *n_valid) {
    if (!ctx || n < 0 || (n > 0 && !times)) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    EcbSplineView sv;
    EcbCovView cv;
    int rc;
    if ((rc = pose_state(ctx, sv, cv))) return rc;
    const int64_t chunk = std::min<int64_t>(std::max<int64_t>(n, 1), POSE_CHUNK);
    // staging: count | times | pose | cov
    if ((rc = ecb_reserve(ctx, ctx->pose_io, 8 + (size_t) chunk * (1 + 7 + 36) * 8))) return rc;
    unsigned long long *d_count = (unsigned long long *) ctx->pose_io.p;
    double *d_t = (double *) ctx->pose_io.p + 1, *d_p = d_t + chunk, *d_c = d_p + 7 * chunk;
    ECB_CUDA(ctx, cudaMemsetAsync(d_count, 0, 8, ctx->stream));
    for (int64_t lo = 0; lo < n; lo += chunk) {
        const int64_t m = std::min(chunk, n - lo);
        ECB_CUDA(ctx, cudaMemcpyAsync(d_t, times + lo, (size_t) m * 8, cudaMemcpyHostToDevice, ctx->stream));
        if ((rc = pose_launch(ctx, sv, cv, d_t, m, pose ? d_p : nullptr, cov ? d_c : nullptr, d_count))) return rc;
        if (pose && (rc = ecb_d2h(ctx, pose + 7 * lo, d_p, (size_t) m * 56))) return rc;
        if (cov && (rc = ecb_d2h(ctx, cov + 36 * lo, d_c, (size_t) m * 288))) return rc;
    }
    unsigned long long c = 0;
    if ((rc = ecb_d2h(ctx, &c, d_count, 8))) return rc;
    if (n_valid) *n_valid = (int64_t) c;
    return ECB_OK;
}

}  // extern "C"
