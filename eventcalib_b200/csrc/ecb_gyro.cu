// Camera-gyroscope calibration (ecb_gyro_calibrate): rotation R_gc, time offset d and bias b from the trajectory's body angular
// velocity.  Model and parameters in ecb_gyro.h and include/eventcalib_b200.h.
//   k_gyro_used      one thread per sample: stamp and reading finite, t - D and t + D in the same segment (the valid set,
//                    fixed for the whole call so that costs at different offsets compare like for like).
//   k_gyro_reduce    a sum over the used samples of a per-sample quantity, templated on it (Op): the scan's
//                    (|w_c(t + d_m)| - |w_g|)^2 with one grid row (blockIdx.y) per offset, the sums of the initial rotation,
//                    the normal equations.  Each thread adds its strided samples in order, a warp by a shuffle tree, a block's
//                    warps in order: one partial per block and row.  k_gyro_final adds a row's partials in block order.  The
//                    grid depends on the used-sample count only and no floating-point atomic is used, so repeated calls (and
//                    two GPUs) give bit-identical sums.  w_c only where the Op needs no dw_c/dt: no translation, no output row.
//   k_gyro_residual  one thread per sample: r_i at the solution, NaN rows for unused samples.
// The host part: the valid set, the scan, Horn's closed-form rotation, Levenberg-Marquardt on 7 (or 6) parameters, each
// iteration one normal-equation evaluation on the GPU, and the covariance.  FP64.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "../../include/ecb/calib_init.hpp"
#include "ecb_bspline.cuh"
#include "ecb_common.cuh"
#include "ecb_gyro.h"
#include "ecb_motion.h"

namespace {

constexpr int GYRO_THREADS = 256;
constexpr int NP = 7;  // delta 3, d, b 3

// offset d_m of the scan grid (the host and the device compute it alike)
__host__ __device__ __forceinline__ double gyro_offset(double D, int M, int m) {
    return M > 1 ? D * (double) (2 * m - (M - 1)) / (double) (M - 1) : 0.0;
}

// w_c at u and, with DOT, dw_c/dt (ecb_angular_velocity); NaN outside every segment
template <int SO3, bool DOT>
__device__ __forceinline__ void gyro_omega(const EcbSplineView &sv, const double *__restrict__ rot, double u, double w[3],
                                           double wd[3]) {
    const double *kn = nullptr;
    int nk = 0;
    const int s = sv.segment(u, &kn, &nk);
    if (s < 0) {
        w[0] = w[1] = w[2] = wd[0] = wd[1] = wd[2] = NAN;
        return;
    }
    const int span = find_span_dev(kn, nk, u);
    double N[4], Nd[4], Ndd[4];
    ecb_ders_basis(kn, span, u, N, Nd, Ndd);
    ecb_angular_velocity<DOT>(rot + 4 * (size_t) (sv.cp_off[s] + span - 3), N, Nd, Ndd, SO3, w, wd);
}

// a sample: s = t wx wy wz (gyroscope), wc = w_c(t + d), wd = dw_c/dt there (DOT only); acc: the K sums
struct ScanOp {  // (|w_c(t + d_m)| - |w_g|)^2 at every offset of the grid
    static constexpr int K = 1, PER_THREAD = 4;
    static constexpr bool DOT = false;
    double D;
    int M;
    __device__ double offset(int m) const { return gyro_offset(D, M, m); }
    __device__ void add(const double *s, const double wc[3], const double *, double *acc) const {
        const double e = sqrt(wc[0] * wc[0] + wc[1] * wc[1] + wc[2] * wc[2]) - sqrt(s[1] * s[1] + s[2] * s[2] + s[3] * s[3]);
        acc[0] += e * e;
    }
};

struct SumsOp {  // sum w_c (3), sum w_g (3), sum w_c w_g^T (9, row major) at one offset
    static constexpr int K = 15, PER_THREAD = 1;
    static constexpr bool DOT = false;
    double d;
    __device__ double offset(int) const { return d; }
    __device__ void add(const double *s, const double wc[3], const double *, double *acc) const {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            acc[i] += wc[i];
            acc[3 + i] += s[1 + i];
#pragma unroll
            for (int j = 0; j < 3; ++j) acc[6 + 3 * i + j] += wc[i] * s[1 + j];
        }
    }
};

struct NormalOp {  // J^T J (upper triangle, row major: 28), J^T r (7), 1/2 |r|^2 at (R, d, b)
    static constexpr int K = 28 + NP + 1, PER_THREAD = 1;
    static constexpr bool DOT = true;
    double R[9], b[3], d;
    __device__ double offset(int) const { return d; }
    __device__ void add(const double *s, const double wc[3], const double *wd, double *acc) const {
        double r[3], J[3 * NP];
        ecb_gyro_residual(R, b, wc, wd, s + 1, r, J);
        int e = 0;
#pragma unroll
        for (int i = 0; i < NP; ++i)
#pragma unroll
            for (int j = i; j < NP; ++j) acc[e++] += J[i] * J[j] + J[NP + i] * J[NP + j] + J[2 * NP + i] * J[2 * NP + j];
#pragma unroll
        for (int i = 0; i < NP; ++i) acc[28 + i] += J[i] * r[0] + J[NP + i] * r[1] + J[2 * NP + i] * r[2];
        acc[28 + NP] += 0.5 * (r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
    }
};

__global__ void k_gyro_used(const double *__restrict__ g, int64_t n, EcbSplineView sv, double D, uint8_t *__restrict__ used) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double *s = g + 4 * i;
    bool ok = isfinite(s[0]) && isfinite(s[1]) && isfinite(s[2]) && isfinite(s[3]);
    if (ok) {
        const double *kn = nullptr;
        int nk = 0;
        const int lo = sv.segment(s[0] - D, &kn, &nk);
        ok = lo >= 0 && lo == sv.segment(s[0] + D, &kn, &nk);
    }
    used[i] = ok;
}

// smp: the used samples (4 doubles each), nu of them; partial[(row * gridDim.x + block) * K + k]
template <int SO3, class Op>
__global__ void __launch_bounds__(GYRO_THREADS) k_gyro_reduce(const double *__restrict__ smp, int64_t nu, EcbSplineView sv,
                                                              const double *__restrict__ rot, Op op, double *__restrict__ partial) {
    __shared__ double swarp[GYRO_THREADS / 32][Op::K];
    const double d = op.offset(blockIdx.y);
    double acc[Op::K];
#pragma unroll
    for (int k = 0; k < Op::K; ++k) acc[k] = 0.0;
    for (int64_t i = (int64_t) blockIdx.x * GYRO_THREADS + threadIdx.x; i < nu; i += (int64_t) gridDim.x * GYRO_THREADS) {
        const double *s = smp + 4 * i;
        double wc[3], wd[3];
        gyro_omega<SO3, Op::DOT>(sv, rot, s[0] + d, wc, wd);
        op.add(s, wc, wd, acc);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < Op::K; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_down_sync(0xffffffffu, acc[k], o);
        if (lane == 0) swarp[warp][k] = acc[k];
    }
    __syncthreads();
    if (threadIdx.x < Op::K) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < GYRO_THREADS / 32; ++w) v += swarp[w][threadIdx.x];
        partial[((size_t) blockIdx.y * gridDim.x + blockIdx.x) * Op::K + threadIdx.x] = v;
    }
}

// out[row * K + k] = sum over blocks b in order of partial[(row * bx + b) * K + k]
__global__ void k_gyro_final(const double *__restrict__ partial, int64_t bx, int K, int rows, double *__restrict__ out) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= rows * K) return;
    const int row = e / K, k = e % K;
    double v = 0.0;
    for (int64_t b = 0; b < bx; ++b) v += partial[((size_t) row * bx + b) * K + k];
    out[e] = v;
}

template <int SO3>
__global__ void k_gyro_residual(const double *__restrict__ g, int64_t n, const uint8_t *__restrict__ used, EcbSplineView sv,
                                const double *__restrict__ rot, NormalOp x, double *__restrict__ res) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double r[3] = {NAN, NAN, NAN};
    if (used[i]) {
        const double *s = g + 4 * i;
        double wc[3], wd[3];
        gyro_omega<SO3, false>(sv, rot, s[0] + x.d, wc, wd);
        ecb_gyro_residual(x.R, x.b, wc, nullptr, s + 1, r, nullptr);
    }
    res[3 * i] = r[0], res[3 * i + 1] = r[1], res[3 * i + 2] = r[2];
}

// device buffers of one call, carved from ctx->gyro_io
struct GyroDev {
    EcbSplineView sv;
    double *rot, *raw, *smp, *partial, *fin, *res;
    uint8_t *used;
    int64_t n, nu;
};

template <class Op>
int64_t blocks_of(int64_t nu) {
    return std::max<int64_t>(1, (nu + (int64_t) GYRO_THREADS * Op::PER_THREAD - 1) / ((int64_t) GYRO_THREADS * Op::PER_THREAD));
}

// the rows x Op::K sums of Op over the used samples, into out
template <class Op>
int gyro_reduce(ecb_ctx *ctx, const GyroDev &g, const Op &op, int rows, std::vector<double> &out) {
    const int64_t bx = blocks_of<Op>(g.nu);
    auto kern = g.sv.so3 ? k_gyro_reduce<1, Op> : k_gyro_reduce<0, Op>;
    kern<<<dim3((unsigned) bx, (unsigned) rows), GYRO_THREADS, 0, ctx->stream>>>(g.smp, g.nu, g.sv, g.rot, op, g.partial);
    ECB_LAUNCHED(ctx);
    ECB_CUDA(ctx, cudaGetLastError());
    const int total = rows * Op::K;
    k_gyro_final<<<(total + 127) / 128, 128, 0, ctx->stream>>>(g.partial, bx, Op::K, rows, g.fin);
    ECB_LAUNCHED(ctx);
    ECB_CUDA(ctx, cudaGetLastError());
    out.resize((size_t) total);
    return ecb_d2h(ctx, out.data(), g.fin, (size_t) total * 8);
}

struct GyroX {  // the parameters: R_gc (x y z w), d, b
    double q[4], d, b[3];
};

NormalOp normal_op(const GyroX &x) {
    NormalOp op;
    ecb_gyro_rotation(x.q, op.R);
    for (int i = 0; i < 3; ++i) op.b[i] = x.b[i];
    op.d = x.d;
    return op;
}

// H = J^T J (7 x 7, full), g = J^T r, cost at x
int normal_eq(ecb_ctx *ctx, const GyroDev &gd, const GyroX &x, double H[NP][NP], double g[NP], double *cost) {
    std::vector<double> s;
    int rc;
    if ((rc = gyro_reduce(ctx, gd, normal_op(x), 1, s))) return rc;
    int e = 0;
    for (int i = 0; i < NP; ++i)
        for (int j = i; j < NP; ++j) H[i][j] = H[j][i] = s[(size_t) e++];
    for (int i = 0; i < NP; ++i) g[i] = s[(size_t) (28 + i)];
    *cost = s[28 + NP];
    return ECB_OK;
}

// L L^T = A (n x n, row major); false unless every pivot is positive and finite; *min_rel = least pivot L_kk^2 / A_kk
bool cholesky(int n, const double *A, double *L, double *min_rel) {
    double mr = INFINITY;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j <= i; ++j) {
            double s = A[i * n + j];
            for (int k = 0; k < j; ++k) s -= L[i * n + k] * L[j * n + k];
            if (i == j) {
                if (!(s > 0.0) || !isfinite(s)) {
                    if (min_rel) *min_rel = 0.0;
                    return false;
                }
                mr = std::min(mr, s / A[i * n + i]);
                L[i * n + i] = sqrt(s);
            } else {
                L[i * n + j] = s / L[j * n + j];
            }
        }
    if (min_rel) *min_rel = mr;
    return true;
}

void chol_solve(int n, const double *L, const double *b, double *x) {
    double y[NP];
    for (int i = 0; i < n; ++i) {
        double s = b[i];
        for (int k = 0; k < i; ++k) s -= L[i * n + k] * y[k];
        y[i] = s / L[i * n + i];
    }
    for (int i = n - 1; i >= 0; --i) {
        double s = y[i];
        for (int k = i + 1; k < n; ++k) s -= L[k * n + i] * x[k];
        x[i] = s / L[i * n + i];
    }
}

// x (+) delta over the 7 parameters: R = Exp(delta_0..2) R, d += delta_3, b += delta_4..6
GyroX plus(const GyroX &x, const double delta[NP]) {
    const ecb_so3::Quat<double> e = ecb_so3::so3_exp<double>(delta);
    const ecb_so3::Quat<double> q = ecb_so3::qmul(e, ecb_so3::Quat<double>{x.q[0], x.q[1], x.q[2], x.q[3]});
    const double nq = sqrt(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w);
    GyroX y;
    y.q[0] = q.x / nq, y.q[1] = q.y / nq, y.q[2] = q.z / nq, y.q[3] = q.w / nq;
    y.d = x.d + delta[3];
    for (int i = 0; i < 3; ++i) y.b[i] = x.b[i] + delta[4 + i];
    return y;
}

// the 8 ambient coordinates (q 4, d, b 3)
void ambient(const GyroX &x, double a[8]) {
    for (int i = 0; i < 4; ++i) a[i] = x.q[i];
    a[4] = x.d;
    for (int i = 0; i < 3; ++i) a[5 + i] = x.b[i];
}

// max |x - Plus(x, -g)| over the ambient coordinates (the projected gradient of ecb_lm)
double gradient_max_norm(const GyroX &x, const double g[NP]) {
    double ng[NP], a[8], c[8], m = 0.0;
    for (int i = 0; i < NP; ++i) ng[i] = -g[i];
    ambient(x, a);
    ambient(plus(x, ng), c);
    for (int i = 0; i < 8; ++i) m = std::max(m, fabs(a[i] - c[i]));
    return m;
}

// Horn's closed-form rotation q (x y z w) minimising sum |R a_i - b_i|^2 from C = sum a_i b_i^T (centred), row major
void horn(const double C[9], double q[4]) {
    const double Sxx = C[0], Sxy = C[1], Sxz = C[2], Syx = C[3], Syy = C[4], Syz = C[5], Szx = C[6], Szy = C[7], Szz = C[8];
    // Horn (1987) N over (w x y z); R(q) maximises q^T N q: the smallest eigenvector of -N
    const double N[16] = {Sxx + Syy + Szz, Syz - Szy,        Szx - Sxz,        Sxy - Syx,
                          Syz - Szy,       Sxx - Syy - Szz,  Sxy + Syx,        Szx + Sxz,
                          Szx - Sxz,       Sxy + Syx,        -Sxx + Syy - Szz, Syz + Szy,
                          Sxy - Syx,       Szx + Sxz,        Syz + Szy,        -Sxx - Syy + Szz};
    std::vector<double> M(16), v;
    for (int i = 0; i < 16; ++i) M[(size_t) i] = -N[i];
    ecb::smallestEigenvector(4, M, v);
    const double s = v[0] < 0.0 ? -1.0 : 1.0, nv = sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2] + v[3] * v[3]);
    q[0] = s * v[1] / nv, q[1] = s * v[2] / nv, q[2] = s * v[3] / nv, q[3] = s * v[0] / nv;
}

// ctx->gyro_io = rot 4C | samples 4n | used samples 4n | partials | sums | residuals 3n | flags n (bytes)
int gyro_alloc(ecb_ctx *ctx, const EcbSplineView &sv, int64_t n, int M, bool want_res, GyroDev &g) {
    const size_t C = (size_t) sv.total_cp, N = (size_t) n;
    const size_t part = (size_t) std::max<int64_t>(blocks_of<ScanOp>(n) * M * ScanOp::K, blocks_of<NormalOp>(n) * NormalOp::K);
    const size_t fin = std::max<size_t>((size_t) M, NormalOp::K);
    const size_t doubles = 4 * C + 8 * N + part + fin + (want_res ? 3 * N : 0);
    int rc;
    if ((rc = ecb_reserve(ctx, ctx->gyro_io, doubles * 8 + N + 8))) return rc;
    double *p = (double *) ctx->gyro_io.p;
    g.rot = p, p += 4 * C;
    g.raw = p, p += 4 * N;
    g.smp = p, p += 4 * N;
    g.partial = p, p += part;
    g.fin = p, p += fin;
    g.res = want_res ? p : nullptr, p += want_res ? 3 * N : 0;
    g.used = (uint8_t *) p;
    g.n = n;
    g.nu = 0;
    return ECB_OK;
}

void fill_nan(ecb_gyro_calibration *o) {
    const double nan = NAN;
    for (double &v : o->q_gc) v = nan;
    o->offset = nan;
    for (double &v : o->bias) v = nan;
    for (double &v : o->cov) v = nan;
    for (double &v : o->std) v = nan;
    o->sigma2 = o->cost = o->rms = o->scan_offset = nan;
}

}  // namespace

extern "C" {

int ecb_gyro_calibrate(ecb_ctx *ctx, const double *rot_cp, const double *gyro, int64_t n, double max_offset, int32_t n_offsets,
                       ecb_gyro_calibration *out, double *offset_cost, double *residuals) {
    if (!ctx || !out) return ECB_ERR_ARG;
    if (n < 0 || (n > 0 && !gyro) || !rot_cp) return ecb_fail(ctx, ECB_ERR_ARG, "gyroscope calibration: bad n, gyro or rot_cp");
    if (!(max_offset >= 0.0) || !isfinite(max_offset))
        return ecb_fail(ctx, ECB_ERR_ARG, "gyroscope calibration: max_offset must be finite and >= 0, got %g", max_offset);
    if (n_offsets < 1 || n_offsets > 65535 || n_offsets % 2 == 0 || (n_offsets > 1) != (max_offset > 0.0))
        return ecb_fail(ctx, ECB_ERR_ARG,
                        "gyroscope calibration: n_offsets must be odd in 1 .. 65535, 1 exactly when max_offset is 0 (got %d, %g)",
                        (int) n_offsets, max_offset);
    cudaSetDevice(ctx->device);
    EcbSplineView sv;
    if (ecb_cost_spline_view(ctx, &sv) != ECB_OK) return ecb_fail(ctx, ECB_ERR_STATE, "gyroscope calibration: ecb_cost_setup first");
    memset(out, 0, sizeof *out);
    fill_nan(out);
    const double D = max_offset;
    const int M = n_offsets, np = D > 0.0 ? 7 : 6;
    int P[NP];  // the estimated parameters among (delta 3, d, b 3)
    for (int i = 0, k = 0; i < NP; ++i)
        if (i != 3 || np == 7) P[k++] = i;
    out->n_params = np;
    out->termination = ECB_LM_RUNNING;
    if (offset_cost)
        for (int m = 0; m < M; ++m) offset_cost[m] = NAN;

    // the valid set
    GyroDev g;
    g.sv = sv;
    int rc;
    if ((rc = gyro_alloc(ctx, sv, n, M, residuals != nullptr, g))) return rc;
    if ((rc = ecb_h2d(ctx, g.rot, rot_cp, 32 * (size_t) sv.total_cp))) return rc;
    std::vector<uint8_t> used((size_t) n);
    std::vector<double> smp;
    if (n > 0) {
        ECB_CUDA(ctx, cudaMemcpyAsync(g.raw, gyro, (size_t) n * 32, cudaMemcpyHostToDevice, ctx->stream));
        k_gyro_used<<<(unsigned) ((n + 255) / 256), 256, 0, ctx->stream>>>(g.raw, n, sv, D, g.used);
        ECB_LAUNCHED(ctx);
        ECB_CUDA(ctx, cudaGetLastError());
        if ((rc = ecb_d2h(ctx, used.data(), g.used, (size_t) n))) return rc;
        for (int64_t i = 0; i < n; ++i)
            if (used[(size_t) i]) smp.insert(smp.end(), gyro + 4 * i, gyro + 4 * i + 4);
    }
    g.nu = (int64_t) smp.size() / 4;
    out->n_used = g.nu;
    out->n_unused = n - g.nu;
    if (g.nu < np) {
        out->status = ECB_GYRO_TOO_FEW_SAMPLES;
        return ecb_fail(ctx, ECB_FAILED, "gyroscope calibration: %lld used samples, fewer than the %d parameters", (long long) g.nu, np);
    }
    ECB_CUDA(ctx, cudaMemcpyAsync(g.smp, smp.data(), smp.size() * 8, cudaMemcpyHostToDevice, ctx->stream));

    // scan of the offset grid
    std::vector<double> s;
    ScanOp scan;
    scan.D = D, scan.M = M;
    if ((rc = gyro_reduce(ctx, g, scan, M, s))) return rc;
    int best = 0;
    for (int m = 0; m < M; ++m) {
        s[(size_t) m] /= (double) g.nu;
        if (s[(size_t) m] < s[(size_t) best]) best = m;
    }
    if (offset_cost) memcpy(offset_cost, s.data(), (size_t) M * 8);
    GyroX x;
    x.d = out->scan_offset = gyro_offset(D, M, best);
    if (M > 1 && (best == 0 || best == M - 1)) {
        out->status = ECB_GYRO_OFFSET_AT_EDGE;
        return ecb_fail(ctx, ECB_FAILED, "gyroscope calibration: the scan's least cost is at offset %g, the edge of +-%g: widen max_offset",
                        x.d, D);
    }

    // initial rotation (Horn) and bias at the scan offset
    SumsOp sums;
    sums.d = x.d;
    if ((rc = gyro_reduce(ctx, g, sums, 1, s))) return rc;
    const double nu = (double) g.nu;
    double Cc[9], R[9];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) Cc[3 * i + j] = s[(size_t) (6 + 3 * i + j)] - s[(size_t) i] * s[(size_t) (3 + j)] / nu;
    horn(Cc, x.q);
    ecb_gyro_rotation(x.q, R);
    for (int i = 0; i < 3; ++i)
        x.b[i] = (s[(size_t) (3 + i)] - (R[3 * i] * s[0] + R[3 * i + 1] * s[1] + R[3 * i + 2] * s[2])) / nu;

    // Levenberg-Marquardt: the trust-region rules of ecb_lm.cu on the dense np x np system
    ecb_lm_options opt;
    ecb_lm_default_options(&opt);
    double H[NP][NP], gr[NP], cost;
    if ((rc = normal_eq(ctx, g, x, H, gr, &cost))) return rc;
    if (np == 6) gr[3] = 0.0;
    double scale[NP], diag[NP];
    for (int i = 0; i < np; ++i) scale[i] = 1.0 / (1.0 + sqrt(H[P[i]][P[i]]));
    double radius = opt.initial_radius, decrease_factor = 2.0;
    bool reuse_diagonal = false;
    int iteration = 0, invalid_steps = 0, termination = ECB_LM_RUNNING;
    if (gradient_max_norm(x, gr) <= opt.gradient_tolerance) termination = ECB_LM_GRADIENT_TOLERANCE;
    while (termination == ECB_LM_RUNNING) {
        if (iteration >= opt.max_iterations) {
            termination = ECB_LM_NO_CONVERGENCE;
            break;
        }
        ++iteration;
        if (!reuse_diagonal)
            for (int i = 0; i < np; ++i)
                diag[i] = std::min(std::max(H[P[i]][P[i]] * scale[i] * scale[i], opt.min_lm_diagonal), opt.max_lm_diagonal);
        double Hs[NP * NP], A[NP * NP], L[NP * NP], gs[NP], y[NP], step[NP];
        for (int i = 0; i < np; ++i) {
            gs[i] = gr[P[i]] * scale[i];
            for (int j = 0; j < np; ++j) A[i * np + j] = Hs[i * np + j] = H[P[i]][P[j]] * scale[i] * scale[j];
            A[i * np + i] += diag[i] / radius;
        }
        double model_cost_change = 0.0;
        bool ok = cholesky(np, A, L, nullptr);
        if (ok) {
            chol_solve(np, L, gs, y);
            double a = 0.0, b = 0.0;
            for (int i = 0; i < np; ++i) step[i] = -y[i];
            for (int i = 0; i < np; ++i) {
                double hd = 0.0;
                for (int j = 0; j < np; ++j) hd += Hs[i * np + j] * step[j];
                a += step[i] * gs[i];
                b += step[i] * hd;
            }
            model_cost_change = -(a + 0.5 * b);
            ok = model_cost_change > 0.0 && isfinite(model_cost_change);
        }
        if (!ok) {  // invalid step: shrink the region and try again
            if (++invalid_steps > 5) {
                termination = ECB_LM_FAILURE;
                break;
            }
            radius /= decrease_factor;
            decrease_factor *= 2.0;
            reuse_diagonal = true;
            continue;
        }
        invalid_steps = 0;
        double delta[NP] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        for (int i = 0; i < np; ++i) delta[P[i]] = step[i] * scale[i];
        const GyroX c = plus(x, delta);
        double ax[8], ac[8], xn = 0.0, sn = 0.0;
        ambient(x, ax);
        ambient(c, ac);
        for (int i = 0; i < 8; ++i) xn += ax[i] * ax[i], sn += (ac[i] - ax[i]) * (ac[i] - ax[i]);
        double Hc[NP][NP], gc[NP], candidate_cost = INFINITY;  // |d| > D: rejected like a cost increase
        if (fabs(c.d) <= D) {
            if ((rc = normal_eq(ctx, g, c, Hc, gc, &candidate_cost))) return rc;
            if (np == 6) gc[3] = 0.0;
        }
        // The parameter and function tolerances are tested after the step is accepted or rejected, not before as in ecb_lm:
        // the candidate's normal equations are already evaluated, and on this small problem the last successful step is worth
        // keeping (it moves the estimate by up to the parameter tolerance).
        const bool small_step = sqrt(sn) <= opt.parameter_tolerance * (sqrt(xn) + opt.parameter_tolerance);
        const bool small_change = fabs(cost - candidate_cost) <= opt.function_tolerance * cost;
        const double rho = (cost - candidate_cost) / model_cost_change;
        if (rho > opt.min_relative_decrease) {
            x = c;
            memcpy(H, Hc, sizeof H);
            memcpy(gr, gc, sizeof gr);
            cost = candidate_cost;
            radius = std::min(opt.max_radius, radius / std::max(1.0 / 3.0, 1.0 - pow(2.0 * rho - 1.0, 3)));
            decrease_factor = 2.0;
            reuse_diagonal = false;
        } else {
            radius /= decrease_factor;
            decrease_factor *= 2.0;
            reuse_diagonal = true;
        }
        if (small_step) termination = ECB_LM_PARAMETER_TOLERANCE;
        else if (small_change) termination = ECB_LM_FUNCTION_TOLERANCE;
        else if (rho > opt.min_relative_decrease && gradient_max_norm(x, gr) <= opt.gradient_tolerance)
            termination = ECB_LM_GRADIENT_TOLERANCE;
        else if (radius < opt.min_radius) termination = ECB_LM_MIN_RADIUS;
    }
    for (int i = 0; i < 4; ++i) out->q_gc[i] = x.q[i];
    out->offset = x.d;
    for (int i = 0; i < 3; ++i) out->bias[i] = x.b[i];
    out->cost = cost;
    out->rms = sqrt(2.0 * cost / (3.0 * nu));
    out->sigma2 = 2.0 * cost / (3.0 * nu - np);
    out->iterations = iteration;
    out->termination = termination;
    if (residuals) {
        if (n > 0) {
            const NormalOp op = normal_op(x);
            auto kern = sv.so3 ? k_gyro_residual<1> : k_gyro_residual<0>;
            kern<<<(unsigned) ((n + 255) / 256), 256, 0, ctx->stream>>>(g.raw, n, g.used, sv, g.rot, op, g.res);
            ECB_LAUNCHED(ctx);
            ECB_CUDA(ctx, cudaGetLastError());
        }
        if ((rc = ecb_d2h(ctx, residuals, g.res, (size_t) n * 24))) return rc;
    }

    // covariance Z = (J^T J)^-1 over the estimated parameters; the offset's row and column 0 when it is held
    double Hr[NP * NP], L[NP * NP], min_rel = 0.0;
    for (int i = 0; i < np; ++i)
        for (int j = 0; j < np; ++j) Hr[i * np + j] = H[P[i]][P[j]];
    if (!cholesky(np, Hr, L, &min_rel) || min_rel < 1e-12) {
        out->status = ECB_GYRO_RANK_DEFICIENT;
        return ecb_fail(ctx, ECB_FAILED, "gyroscope calibration: J^T J is rank deficient (least relative pivot %g): does the motion "
                        "rotate about more than one axis?", min_rel);
    }
    for (double &v : out->cov) v = 0.0;
    for (int j = 0; j < np; ++j) {
        double e[NP] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0}, z[NP];
        e[j] = 1.0;
        chol_solve(np, L, e, z);
        for (int i = 0; i <= j; ++i) out->cov[P[i] * NP + P[j]] = out->cov[P[j] * NP + P[i]] = z[i];
    }
    for (int i = 0; i < NP; ++i) out->std[i] = sqrt(out->sigma2 * out->cov[i * NP + i]);
    out->status = ECB_GYRO_OK;
    return ECB_OK;
}

}  // extern "C"
