// Covariance of the trajectory's pose at any time: Sigma(t) = J Z_blk J^T (definition in ecb_pose.h), from the Z and x that the
// last successful ecb_covariance left on the context and the knots of ecb_cost_setup.
//
//   k_pose_cov   one thread per query: segment (first whose knot range holds t), span and basis (ecb_bspline.cuh), pose and
//                6 x 24 Jacobian (ecb_pose.h), then Sigma from the lower triangle of the 24 x 24 block of Z in the band
//                (300 doubles, 160 KB for the whole band at D = 843: it stays in L2 / L1, and sorted queries read the same
//                block as their neighbours).  Each query is computed alone in a fixed order: its output does not depend on
//                the batch.  FP64.
//   k_motion     the same per query for the motion (ecb_motion.h): pose, w_b, v_w, a_w from the derivative basis, and with
//                COV the 9 x 24 Jacobian (in shared memory) and Sigma_m = J Z_blk J^T like k_pose_cov.  Each warp stages its
//                32 output rows in shared memory and stores them as one contiguous range.  FP64.
#include <algorithm>

#include "ecb_bspline.cuh"
#include "ecb_common.cuh"
#include "ecb_motion.h"
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
int pose_state(ecb_ctx *ctx, EcbSplineView &sv, EcbCovView &cv, const char *what = "pose covariance") {
    if (ecb_cost_spline_view(ctx, &sv) != ECB_OK) return ecb_fail(ctx, ECB_ERR_STATE, "%s: ecb_cost_setup first", what);
    if (ecb_covariance_view(ctx, &cv) != ECB_OK)
        return ecb_fail(ctx, ECB_ERR_STATE, "%s: no successful ecb_covariance on this context", what);
    if (cv.spline_gen != ctx->spline_gen || cv.so3 != sv.so3 || cv.total_cp != sv.total_cp)
        return ecb_fail(ctx, ECB_ERR_STATE, "%s: ecb_cost_setup or ecb_cost_set_rotation_model ran after ecb_covariance", what);
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

// ---- motion of the trajectory (definition in ecb_motion.h) ----------------------------------------------------------------
constexpr int MOTION_THREADS = 128;
constexpr int MOT_ROW = 16, MOT_STRIDE = 17;  // doubles of a motion row, and its stride in the staging (odd: conflict-free)
constexpr int COV_ROW = 81, JAC_STRIDE = 37;  // doubles of a 9 x 9 Sigma_m; of the 4 blocks B_j of a thread (36, odd stride)
static_assert(32 * JAC_STRIDE <= 32 * COV_ROW, "the staged covariances reuse the Jacobians' space");
// shared doubles per warp: the staged motion rows and, with the covariance, the Jacobians that the staged Sigma_m then replace
constexpr int motion_warp_doubles(int cov) { return 32 * MOT_STRIDE + (cov ? 32 * COV_ROW : 0); }

// pose_sigma for the 9 rows (w_b, v_w, a_w): Sigma = sum_c (v_c J_c^T + J_c v_c^T), v_c = sum_{r > c} Z_rc J_r + Z_cc J_c / 2,
// upper triangle only.  The column J_c of a rotation tangent is (B_jc[:, kc], 0, 0); of a translation it is Nd_jc e_p +
// Ndd_jc e_q with p = kc (v_w row), q = kc + 3 (a_w row).  sB: B_j[r][k] at sB[9 j + 3 r + k].
__device__ __forceinline__ void motion_sigma(const double *sB, const double Nd[4], const double Ndd[4],
                                             const double *__restrict__ Zb, double S[9][9]) {
#pragma unroll
    for (int i = 0; i < 9; ++i)
#pragma unroll
        for (int l = 0; l < 9; ++l) S[i][l] = 0.0;
#pragma unroll
    for (int c = 0; c < 24; ++c) {
        const double *Zc = Zb + c * 24;  // band column c of the block: Z(c + r, c) at Zc[r]
        double v[9] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll
        for (int r = c; r < 24; ++r) {
            double z = __ldg(Zc + (r - c));
            if (r == c) z *= 0.5;
            const int jr = r / 6, kr = r % 6;
            if (kr < 3) {
                v[0] += z * sB[9 * jr + kr];
                v[1] += z * sB[9 * jr + 3 + kr];
                v[2] += z * sB[9 * jr + 6 + kr];
            } else {
                v[kr] += z * Nd[jr];
                v[kr + 3] += z * Ndd[jr];
            }
        }
        const int jc = c / 6, kc = c % 6;
        if (kc < 3) {
            const double a[3] = {sB[9 * jc + kc], sB[9 * jc + 3 + kc], sB[9 * jc + 6 + kc]};
#pragma unroll
            for (int i = 0; i < 3; ++i) {
#pragma unroll
                for (int l = i; l < 3; ++l) S[i][l] += v[i] * a[l] + a[i] * v[l];
#pragma unroll
                for (int l = 3; l < 9; ++l) S[i][l] += a[i] * v[l];
            }
        } else {
            const int p = kc, q = kc + 3;
            const double nd = Nd[jc], ndd = Ndd[jc];
#pragma unroll
            for (int i = 0; i < 9; ++i) {
                if (i < p) S[i][p] += v[i] * nd;
                else if (i == p) S[p][p] += 2.0 * v[p] * nd;
                else S[p][i] += nd * v[i];
                if (i < q) S[i][q] += v[i] * ndd;
                else if (i == q) S[q][q] += 2.0 * v[q] * ndd;
                else S[q][i] += ndd * v[i];
            }
        }
    }
}

// One thread per query; a warp stages its 32 output rows in shared memory and stores them as one contiguous range.
// rot / trans: the control points (layout of ecb_cost_eval); Zb: the band of Z (COV only).
template <int SO3, int COV>
__global__ void __launch_bounds__(MOTION_THREADS) k_motion(const double *__restrict__ times, int64_t n, EcbSplineView sv,
                                                           const double *__restrict__ rot, const double *__restrict__ trans,
                                                           const double *__restrict__ Zb, double *__restrict__ motion,
                                                           double *__restrict__ cov, unsigned long long *__restrict__ n_valid) {
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *wbuf = smem + warp * motion_warp_doubles(COV);
    double *sM = wbuf + lane * MOT_STRIDE;
    double *sC = wbuf + 32 * MOT_STRIDE;  // COV: B of lane at sC + lane * JAC_STRIDE, then its Sigma_m at sC + lane * COV_ROW
    const int64_t k0 = (int64_t) blockIdx.x * MOTION_THREADS + warp * 32, k = k0 + lane;
    bool valid = false;
    double S[9][9];
    if (k < n) {
        const double u = times[k];
        const double *kn = nullptr;
        int nk = 0;
        const int s = sv.segment(u, &kn, &nk);
        valid = s >= 0;
        if (valid) {
            const int span = find_span_dev(kn, nk, u);
            double N[4], Nd[4], Ndd[4];
            ecb_ders_basis(kn, span, u, N, Nd, Ndd);
            const size_t c0 = (size_t) (sv.cp_off[s] + span - 3);
            const double *Q = rot + 4 * c0, *T = trans + 3 * c0;
            EcbMotion m;
            ecb_motion_eval(Q, T, N, Nd, Ndd, SO3, m);
            const double row[MOT_ROW] = {m.t[0], m.t[1], m.t[2], m.q[0], m.q[1], m.q[2], m.q[3], m.w[0],
                                         m.w[1], m.w[2], m.v[0], m.v[1], m.v[2], m.a[0], m.a[1], m.a[2]};
#pragma unroll
            for (int i = 0; i < MOT_ROW; ++i) sM[i] = row[i];
            if constexpr (COV != 0) {
                // the Jacobian of each thread in shared memory: in registers, next to the dual numbers of w_b, it would spill
                double *sB = sC + lane * JAC_STRIDE;
#pragma unroll 1
                for (int j = 0; j < 4; ++j) {
                    double B[3][3];
                    ecb_motion_jacobian(Q, N, Nd, SO3, j, B);
#pragma unroll
                    for (int r = 0; r < 3; ++r)
#pragma unroll
                        for (int c = 0; c < 3; ++c) sB[9 * j + 3 * r + c] = B[r][c];
                }
                motion_sigma(sB, Nd, Ndd, Zb + c0 * 6 * 24, S);
            }
        } else {
#pragma unroll
            for (int i = 0; i < MOT_ROW; ++i) sM[i] = NAN;
#pragma unroll
            for (int i = 0; i < 9; ++i)
#pragma unroll
                for (int l = 0; l < 9; ++l) S[i][l] = NAN;
        }
    }
    const int rows = (int) max((int64_t) 0, min((int64_t) 32, n - k0));
    if (motion) {
        __syncwarp();
        double *out = motion + k0 * MOT_ROW;
        for (int e = lane; e < rows * MOT_ROW; e += 32) out[e] = wbuf[(e / MOT_ROW) * MOT_STRIDE + e % MOT_ROW];
    }
    if constexpr (COV != 0) {
        __syncwarp();  // every lane has read its Jacobian
        if (k < n) {
            double *p = sC + lane * COV_ROW;
#pragma unroll
            for (int i = 0; i < 9; ++i)
#pragma unroll
                for (int l = 0; l < 9; ++l) p[9 * i + l] = i <= l ? S[i][l] : S[l][i];
        }
        __syncwarp();
        double *out = cov + k0 * COV_ROW;
        for (int e = lane; e < rows * COV_ROW; e += 32) out[e] = sC[e];
    }
    if (n_valid) {
        const unsigned msk = __ballot_sync(0xffffffffu, valid);
        if (lane == 0 && msk) atomicAdd(n_valid, (unsigned long long) __popc(msk));
    }
}

struct MotionArgs {
    EcbSplineView sv;
    const double *rot, *trans, *Zb;  // device: control points; the band of Z (nullptr: no covariance)
};

// k_motion<SO3, COV> with COV = d_cov != nullptr
int motion_launch(ecb_ctx *ctx, const MotionArgs &a, const double *d_times, int64_t n, double *d_motion, double *d_cov,
                  unsigned long long *d_count) {
    if (n == 0) return ECB_OK;
    const bool c = d_cov != nullptr;
    auto kern = a.sv.so3 ? (c ? k_motion<1, 1> : k_motion<1, 0>) : (c ? k_motion<0, 1> : k_motion<0, 0>);
    const size_t smem = (size_t) (MOTION_THREADS / 32) * motion_warp_doubles(c) * 8;
    ECB_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem)  /* constant: race-free */);
    const int64_t blocks = (n + MOTION_THREADS - 1) / MOTION_THREADS;
    kern<<<(unsigned) blocks, MOTION_THREADS, smem, ctx->stream>>>(d_times, n, a.sv, a.rot, a.trans, a.Zb, d_motion, d_cov, d_count);
    ECB_LAUNCHED(ctx);
    return ecb_check(ctx, cudaGetLastError(), "k_motion");
}

// motion_io = count | control points (cp doubles) | host staging (stage doubles); the count is zeroed
int motion_reserve(ecb_ctx *ctx, size_t cp, size_t stage, unsigned long long **d_count, double **d_cp, double **d_stage) {
    int rc;
    if ((rc = ecb_reserve(ctx, ctx->motion_io, (1 + cp + stage) * 8))) return rc;
    *d_count = (unsigned long long *) ctx->motion_io.p;
    *d_cp = (double *) ctx->motion_io.p + 1;
    *d_stage = *d_cp + cp;
    return ecb_check(ctx, cudaMemsetAsync(*d_count, 0, 8, ctx->stream), "motion count");
}

// h_rot / h_trans (host, ecb_trajectory_motion): uploaded into motion_io and used instead of a.rot / a.trans
int motion_device(ecb_ctx *ctx, MotionArgs a, const double *h_rot, const double *h_trans, const double *d_times, int64_t n,
                  double *d_motion, double *d_cov, int64_t *n_valid) {
    if (n > (int64_t) INT32_MAX * MOTION_THREADS) return ecb_fail(ctx, ECB_ERR_ARG, "motion: %lld queries in one call", (long long) n);
    const size_t C = (size_t) a.sv.total_cp, cp = h_rot ? 7 * C : 0;
    unsigned long long *d_count;
    double *d_cp, *d_stage;
    int rc;
    if ((rc = motion_reserve(ctx, cp, 0, &d_count, &d_cp, &d_stage))) return rc;
    if (h_rot) {
        if ((rc = ecb_h2d(ctx, d_cp, h_rot, 32 * C)) || (rc = ecb_h2d(ctx, d_cp + 4 * C, h_trans, 24 * C))) return rc;
        a.rot = d_cp, a.trans = d_cp + 4 * C;
    }
    if ((rc = motion_launch(ctx, a, d_times, n, d_motion, d_cov, n_valid ? d_count : nullptr))) return rc;
    if (n_valid) {
        unsigned long long c = 0;
        if ((rc = ecb_d2h(ctx, &c, d_count, 8))) return rc;
        *n_valid = (int64_t) c;
    }
    return ECB_OK;
}

// the host variants: times, motion and cov staged through motion_io in chunks, as ecb_pose_covariance does
int motion_host(ecb_ctx *ctx, MotionArgs a, const double *h_rot, const double *h_trans, const double *times, int64_t n,
                double *motion, double *cov, int64_t *n_valid) {
    const size_t C = (size_t) a.sv.total_cp, cp = h_rot ? 7 * C : 0;
    const int64_t chunk = std::min<int64_t>(std::max<int64_t>(n, 1), POSE_CHUNK);
    unsigned long long *d_count;
    double *d_cp, *d_t;
    int rc;
    if ((rc = motion_reserve(ctx, cp, (size_t) chunk * (1 + MOT_ROW + (cov ? COV_ROW : 0)), &d_count, &d_cp, &d_t))) return rc;
    if (h_rot) {
        if ((rc = ecb_h2d(ctx, d_cp, h_rot, 32 * C)) || (rc = ecb_h2d(ctx, d_cp + 4 * C, h_trans, 24 * C))) return rc;
        a.rot = d_cp, a.trans = d_cp + 4 * C;
    }
    double *d_m = d_t + chunk, *d_c = d_m + MOT_ROW * chunk;
    for (int64_t lo = 0; lo < n; lo += chunk) {
        const int64_t m = std::min(chunk, n - lo);
        ECB_CUDA(ctx, cudaMemcpyAsync(d_t, times + lo, (size_t) m * 8, cudaMemcpyHostToDevice, ctx->stream));
        if ((rc = motion_launch(ctx, a, d_t, m, motion ? d_m : nullptr, cov ? d_c : nullptr, d_count))) return rc;
        if (motion && (rc = ecb_d2h(ctx, motion + MOT_ROW * lo, d_m, (size_t) m * MOT_ROW * 8))) return rc;
        if (cov && (rc = ecb_d2h(ctx, cov + COV_ROW * lo, d_c, (size_t) m * COV_ROW * 8))) return rc;
    }
    unsigned long long c = 0;
    if ((rc = ecb_d2h(ctx, &c, d_count, 8))) return rc;
    if (n_valid) *n_valid = (int64_t) c;
    return ECB_OK;
}

// the knots and the rotation model of ecb_cost_setup, the control points given by the caller
int trajectory_args(ecb_ctx *ctx, MotionArgs &a) {
    if (ecb_cost_spline_view(ctx, &a.sv) != ECB_OK) return ecb_fail(ctx, ECB_ERR_STATE, "trajectory motion: ecb_cost_setup first");
    a.rot = a.trans = a.Zb = nullptr;
    return ECB_OK;
}

// the knots of ecb_cost_setup, x and Z of the last successful ecb_covariance (the ECB_ERR_STATE rules of ecb_pose_covariance)
int covariance_args(ecb_ctx *ctx, MotionArgs &a) {
    EcbCovView cv;
    int rc;
    if ((rc = pose_state(ctx, a.sv, cv, "motion covariance"))) return rc;
    a.rot = cv.x + 9;
    a.trans = cv.x + 9 + 4 * (size_t) cv.total_cp;
    a.Zb = cv.Zb;
    return ECB_OK;
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

int ecb_trajectory_motion(ecb_ctx *ctx, const double *rot_cp, const double *trans_cp, const double *times, int64_t n,
                          double *motion, int64_t *n_valid) {
    if (!ctx || n < 0 || !rot_cp || !trans_cp || (n > 0 && !times)) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    MotionArgs a;
    int rc;
    if ((rc = trajectory_args(ctx, a))) return rc;
    return motion_host(ctx, a, rot_cp, trans_cp, times, n, motion, nullptr, n_valid);
}

int ecb_trajectory_motion_device(ecb_ctx *ctx, const double *rot_cp, const double *trans_cp, const double *d_times, int64_t n,
                                 double *d_motion, int64_t *n_valid) {
    if (!ctx || n < 0 || !rot_cp || !trans_cp || (n > 0 && !d_times)) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    MotionArgs a;
    int rc;
    if ((rc = trajectory_args(ctx, a))) return rc;
    return motion_device(ctx, a, rot_cp, trans_cp, d_times, n, d_motion, nullptr, n_valid);
}

int ecb_motion_covariance(ecb_ctx *ctx, const double *times, int64_t n, double *motion, double *cov, int64_t *n_valid) {
    if (!ctx || n < 0 || (n > 0 && !times)) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    MotionArgs a;
    int rc;
    if ((rc = covariance_args(ctx, a))) return rc;
    return motion_host(ctx, a, nullptr, nullptr, times, n, motion, cov, n_valid);
}

int ecb_motion_covariance_device(ecb_ctx *ctx, const double *d_times, int64_t n, double *d_motion, double *d_cov,
                                 int64_t *n_valid) {
    if (!ctx || n < 0 || (n > 0 && !d_times)) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    MotionArgs a;
    int rc;
    if ((rc = covariance_args(ctx, a))) return rc;
    return motion_device(ctx, a, nullptr, nullptr, d_times, n, d_motion, d_cov, n_valid);
}

}  // extern "C"
