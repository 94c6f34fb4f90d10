// The Levenberg-Marquardt loop of EventCalibSpline::optimize (event_camera_calib/src/EventCalibSpline.cpp:197-247) with the
// trust-region state machine AND the linear solve on the device.  The host only enqueues kernels: per iteration
//
//   k_lm_iter_begin   iteration counter, "still running" flag
//   k_lm_build        Jacobi-scaled, damped system  S H S + diag / radius  (band + arrow) and the scaled gradient as an extra row
//   k_lm_factor       banded Cholesky, one CTA per spline segment: a 24 x 24 sliding window of the Schur complement in shared
//                     memory, one column per barrier; the 9 intrinsics rows and the right-hand side ride along as 10 arrow rows
//                     (so the forward substitution is part of the factorisation)
//   k_lm_corner       9 x 9 Schur complement of the intrinsics (sum of the segments' contributions in segment order), its
//                     Cholesky factor and the intrinsics part of the step
//   k_lm_backsub      back substitution, one warp per segment
//   k_lm_step         step, model cost change  -(J d).(r + J d / 2)  from the UNDAMPED system, candidate x+ = Plus(x, d)
//   k_cost            cost of the candidate (ecb_cost.cu), summed over the GPUs through the peer buffers when there are several
//   k_lm_decide       rho, accept / reject, radius update, termination tests
//   k_lm_commit, k_normal_eq (+ fused inter-GPU sum), k_lm_assemble, k_lm_gradnorm   — run only when the step was accepted:
//                     every kernel reads a device flag and returns at once otherwise, so no host round trip decides anything
//
// and reads the result back once at the end.  With several GPUs (one process per GPU, or several contexts of one process) the
// state machine is replicated: every rank sums the same packed normal equations and candidate costs in rank order, so all
// ranks take bit-identical decisions.
//
// The trust-region logic is the one of the host state machine ecb_lm_* (ecb_lm.cu), i.e. Ceres 1.x's TrustRegionMinimizer +
// LevenbergMarquardtStrategy restated [external — Ceres is not in /root/reference; SURVEY.md Appendix C]; tests compare the two.
// Unknown ordering of the tangent system: control point c owns rows 6c .. 6c+5 (rotation tangent, translation), the 9
// intrinsics come last (the arrow).  Band storage is column major: Hb[j * 24 + r] = H(j + r, j), r = 0 .. 23.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <climits>
#include <vector>

#include "ecb_common.cuh"
#include "ecb_so3.h"

int ecb_cost_dev_eval(ecb_ctx *ctx, const double *d_params, const int *d_go, double *d_cost);
int ecb_cost_dev_normal_eq(ecb_ctx *ctx, const double *d_params, const int *d_go, double *d_out);
int ecb_cost_dev_normal_eq_exchange(ecb_ctx *ctx, const double *d_params, const int *d_go, int rank, int n_ranks,
                                    void *const *recv_buffers, const unsigned long long *d_epoch, unsigned long long epoch,
                                    int phases, double *d_out, unsigned *d_err);
int ecb_cost_dev_scalar_exchange(ecb_ctx *ctx, const int *d_go, int rank, int n_ranks, void *const *recv_buffers,
                                 const unsigned long long *d_epoch, double *d_value, unsigned *d_err);
extern "C" int ecb_cost_layout(ecb_ctx *ctx, int32_t *total_cp, int32_t *total_spans, int64_t *n_residuals, int64_t *out_doubles);

namespace {

constexpr int NB = 24;               // band rows per column (half bandwidth 23 + diagonal)
constexpr int NI = 9;                // intrinsics
constexpr int NA = NI + 1;           // arrow rows of the factorisation: intrinsics + right-hand side
constexpr int OUT_STRIDE = 33 * 33 + 33;
constexpr int FACTOR_THREADS = 256;  // 595 window elements (300 band + 240 arrow + 55 corner), up to 3 per thread
constexpr int TRACE_CAP = 1024;

struct LmScalars {
    double cost, radius, decrease_factor, model_cost_change, candidate_cost, gradient_max_norm, step_norm, x_norm, initial_cost;
    int iteration, successful, termination, invalid_steps, reuse_diagonal;
    int running, step_valid, accepted, go_cost, factor_fail, trace_rows, pad0;
    unsigned xerr;
    unsigned long long epoch_ne, epoch_sc;
};

struct LmDims {
    int C, n, D, n_spans, n_seg;
    const int *cp_seg, *cp_local;                    // per control point: segment, index inside the segment
    const int *seg_cp_off, *seg_ncp, *seg_span_off;  // per segment
};

struct LmBufs {
    double *x, *cand, *ne;            // parameters (intr 9 | rot 4C | trans 3C) at x / candidate; packed normal equations at x
    double *Hb, *Ha, *Hc, *g;         // J^T J (band column major, arrow 9 x n, corner 9 x 9 full) and J^T r at x, unscaled
    double *scale, *diag, *step, *delta;
    double *Lb, *La, *Cc0, *dC, *Lc, *xi, *ysol;  // factorisation workspace (Lc: 1 / L(j, j) of the band)
    double *trace;
    LmScalars *s;
    double *Lcc;                      // k_lm_corner stores its 9 x 9 factor here when set (the covariance; NULL in the LM)
};

__device__ __forceinline__ void record(LmScalars *s, double *trace, double accepted) {
    if (s->trace_rows < TRACE_CAP) {
        double *t = trace + 4 * (size_t) s->trace_rows;
        t[0] = s->cost;
        t[1] = s->gradient_max_norm;
        t[2] = s->radius;
        t[3] = accepted;
    }
    ++s->trace_rows;
}

// EigenQuaternionParameterization::Plus [external: Ceres], storage x y z w: x+ = [sin|d|/|d| d, cos|d|] (x) x
__device__ __forceinline__ void quat_plus_dev(const double *x, const double *d, double *out) {
    const double nd = sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
    if (nd > 0.0) {
        const double s = sin(nd) / nd;
        const double ax = s * d[0], ay = s * d[1], az = s * d[2], aw = cos(nd);
        const double bx = x[0], by = x[1], bz = x[2], bw = x[3];
        out[3] = aw * bw - ax * bx - ay * by - az * bz;
        out[0] = aw * bx + ax * bw + ay * bz - az * by;
        out[1] = aw * by + ay * bw + az * bx - ax * bz;
        out[2] = aw * bz + az * bw + ax * by - ay * bx;
    } else {
        for (int i = 0; i < 4; ++i) out[i] = x[i];
    }
}

// local index (0 .. 32) of tangent component k (0..5) of the control point at offset o (0..3) inside a span block
__device__ __forceinline__ int local_idx(int o, int k) { return k < 3 ? 9 + 3 * o + k : 21 + 3 * o + (k - 3); }

// ---- packed per-span normal equations -> band / arrow / corner / gradient, spans added in ascending order (the host
// state machine's order, ecb_lm.cu assemble); the rows / columns of constant intrinsics (cmask) come out as exact zeros ---------
__global__ void k_lm_assemble(LmDims d, LmBufs b, const int *go, uint32_t cmask) {
    if (go && *go == 0) return;
    const int n = d.n;
    const long long total = (long long) n * NB + (long long) NI * n + NI * NI + d.D;
    for (long long e = (long long) blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long) gridDim.x * blockDim.x) {
        if (e < (long long) n * NB) {  // band: column j, row i = j + r
            const int j = (int) (e / NB), r = (int) (e % NB), i = j + r;
            double v = 0.0;
            if (i < n) {
                const int ci = i / 6, ki = i % 6, cj = j / 6, kj = j % 6;
                if (d.cp_seg[ci] == d.cp_seg[cj]) {
                    const int sg = d.cp_seg[ci], li = d.cp_local[ci], lj = d.cp_local[cj];
                    const int s0 = max(0, li - 3), s1 = min(lj, d.seg_ncp[sg] - 4);
                    for (int ls = s0; ls <= s1; ++ls) {
                        const double *B = b.ne + (size_t) (d.seg_span_off[sg] + ls) * OUT_STRIDE;
                        v += B[local_idx(li - ls, ki) * 33 + local_idx(lj - ls, kj)];
                    }
                }
            }
            b.Hb[e] = v;
        } else if (e < (long long) n * NB + (long long) NI * n) {  // arrow: intrinsic r, column j
            const long long q = e - (long long) n * NB;
            const int r = (int) (q / n), j = (int) (q % n);
            const int cj = j / 6, kj = j % 6, sg = d.cp_seg[cj], lj = d.cp_local[cj];
            const int s0 = max(0, lj - 3), s1 = min(lj, d.seg_ncp[sg] - 4);
            double v = 0.0;
            for (int ls = s0; ls <= s1; ++ls) v += b.ne[(size_t) (d.seg_span_off[sg] + ls) * OUT_STRIDE + r * 33 + local_idx(lj - ls, kj)];
            b.Ha[q] = ecb_zero_constant(cmask, r, -1, v);
        } else if (e < (long long) n * NB + (long long) NI * n + NI * NI) {  // corner
            const int q = (int) (e - (long long) n * NB - (long long) NI * n), r = q / NI, c = q % NI;
            double v = 0.0;
            for (int s = 0; s < d.n_spans; ++s) v += b.ne[(size_t) s * OUT_STRIDE + max(r, c) * 33 + min(r, c)];
            b.Hc[q] = ecb_zero_constant(cmask, r, c, v);
        } else {  // gradient
            const int i = (int) (e - (long long) n * NB - (long long) NI * n - NI * NI);
            double v = 0.0;
            if (i < n) {
                const int ci = i / 6, ki = i % 6, sg = d.cp_seg[ci], li = d.cp_local[ci];
                const int s0 = max(0, li - 3), s1 = min(li, d.seg_ncp[sg] - 4);
                for (int ls = s0; ls <= s1; ++ls) v += b.ne[(size_t) (d.seg_span_off[sg] + ls) * OUT_STRIDE + 1089 + local_idx(li - ls, ki)];
            } else {
                for (int s = 0; s < d.n_spans; ++s) v += b.ne[(size_t) s * OUT_STRIDE + 1089 + (i - n)];
                v = ecb_zero_constant(cmask, i - n, -1, v);
            }
            b.g[i] = v;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) b.s->cost = b.ne[(size_t) d.n_spans * OUT_STRIDE];
}

__device__ __forceinline__ double h_diag(const LmDims &d, const LmBufs &b, int i) {
    return i < d.n ? b.Hb[(size_t) i * NB] : b.Hc[(i - d.n) * NI + (i - d.n)];
}

// after the first assembly: Jacobi scaling from the first Jacobian, initial trust region
__global__ void k_lm_init(LmDims d, LmBufs b, ecb_lm_options o) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < d.D; i += gridDim.x * blockDim.x)
        b.scale[i] = o.jacobi_scaling ? 1.0 / (1.0 + sqrt(h_diag(d, b, i))) : 1.0;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        LmScalars *s = b.s;
        s->radius = o.initial_radius;
        s->decrease_factor = 2.0;
        s->reuse_diagonal = 0;
        s->iteration = 0;
        s->successful = 0;
        s->termination = ECB_LM_RUNNING;
        s->running = 1;
        s->invalid_steps = 0;
        s->trace_rows = 0;
        s->initial_cost = s->cost;
        s->accepted = 1;  // the gradient norms of the starting point are computed next
    }
}

// max |x - Plus(x, -g)| over the ambient parameters (Ceres' projected gradient), the trace row of an evaluation at an accepted
// point, and the gradient-tolerance test
__global__ void __launch_bounds__(1024) k_lm_gradnorm(LmDims d, LmBufs b, ecb_lm_options o, const int *go) {
    __shared__ double sh[1024];
    if (go && *go == 0) return;
    double m = 0.0;
    const double *intr = b.x, *rot = b.x + 9, *trans = b.x + 9 + 4 * (size_t) d.C;
    for (int c = threadIdx.x; c < d.C + 1; c += blockDim.x) {
        if (c == d.C) {
            for (int i = 0; i < 9; ++i) {
                const double v = intr[i] + (-b.g[d.n + i]);
                m = fmax(m, fabs(intr[i] - v));
            }
            continue;
        }
        double ng[3] = {-b.g[6 * c], -b.g[6 * c + 1], -b.g[6 * c + 2]}, q[4];
        if (o.rotation_model == 1) ecb_so3::plus(rot + 4 * c, ng, q);
        else quat_plus_dev(rot + 4 * c, ng, q);
        for (int k = 0; k < 4; ++k) m = fmax(m, fabs(rot[4 * c + k] - q[k]));
        for (int k = 0; k < 3; ++k) {
            const double t = trans[3 * c + k], v = t + (-b.g[6 * c + 3 + k]);
            m = fmax(m, fabs(t - v));
        }
    }
    sh[threadIdx.x] = m;
    __syncthreads();
    for (int s = 512; s > 0; s >>= 1) {
        if ((int) threadIdx.x < s) sh[threadIdx.x] = fmax(sh[threadIdx.x], sh[threadIdx.x + s]);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        LmScalars *s = b.s;
        s->gradient_max_norm = sh[0];
        record(s, b.trace, 1.0);
        if (!o.fixed_iterations && s->running && s->gradient_max_norm <= o.gradient_tolerance) {
            s->termination = ECB_LM_GRADIENT_TOLERANCE;
            s->running = 0;
        }
        s->accepted = 0;
    }
}

__global__ void k_lm_iter_begin(LmBufs b, ecb_lm_options o) {
    LmScalars *s = b.s;
    s->accepted = 0;
    s->go_cost = 0;
    s->step_valid = 0;
    s->factor_fail = 0;
    if (!s->running) return;
    if (s->iteration >= o.max_iterations) {
        s->termination = ECB_LM_NO_CONVERGENCE;
        s->running = 0;
        return;
    }
    ++s->iteration;
    s->step_valid = 1;
}

// scaled + damped system into the factorisation workspace
__global__ void k_lm_build(LmDims d, LmBufs b, ecb_lm_options o) {
    const LmScalars *s = b.s;
    if (!s->running) return;
    const int n = d.n;
    const double radius = s->radius;
    const bool reuse = s->reuse_diagonal != 0;
    const long long total = (long long) n * NB + (long long) NA * n + NA * NA;
    for (long long e = (long long) blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long) gridDim.x * blockDim.x) {
        if (e < (long long) n * NB) {
            const int j = (int) (e / NB), r = (int) (e % NB), i = j + r;
            double v = 0.0;
            if (i < n) {
                v = b.Hb[e] * b.scale[i] * b.scale[j];
                if (r == 0) {
                    double dg = b.diag[j];
                    if (!reuse) {
                        dg = fmin(fmax(b.Hb[e] * b.scale[j] * b.scale[j], o.min_lm_diagonal), o.max_lm_diagonal);
                        b.diag[j] = dg;
                    }
                    v += dg / radius;
                }
            }
            b.Lb[e] = v;
        } else if (e < (long long) n * NB + (long long) NA * n) {
            const long long q = e - (long long) n * NB;
            const int r = (int) (q / n), j = (int) (q % n);
            b.La[q] = r < NI ? b.Ha[q] * b.scale[n + r] * b.scale[j] : b.g[j] * b.scale[j];  // row 9: the scaled gradient
        } else {
            const int q = (int) (e - (long long) n * NB - (long long) NA * n), r = q / NA, c = q % NA;
            double v = 0.0;
            if (r < NI && c < NI) {
                v = b.Hc[r * NI + c] * b.scale[n + r] * b.scale[n + c];
                if (r == c) {
                    double dg = b.diag[n + r];
                    if (!reuse) {
                        dg = fmin(fmax(b.Hc[r * NI + r] * b.scale[n + r] * b.scale[n + r], o.min_lm_diagonal), o.max_lm_diagonal);
                        b.diag[n + r] = dg;
                    }
                    v += dg / radius;
                }
            } else if (r == NI && c < NI) {
                v = b.g[n + c] * b.scale[n + c];
            }
            b.Cc0[q] = v;
        }
    }
}

// Banded Cholesky of one segment's block of the band with the arrow rows carried along — BLOCKED by control point (6 columns
// per step; a residual couples 4 consecutive control points, so the band is block-banded: column 6 jb + k has no entry below
// row 6 jb + 23 and a 24-row window holds everything a block column touches).  Per block step:
//   1. warp 0 factorises the 6-column panel in registers: lane = one window row (24 band rows, 10 arrow rows; lanes 0 and 1
//      carry the two extra arrow rows), row-wise Crout — for column k the pivot row's entries are broadcast by shuffles,
//      l_rk = (a_rk - sum_{m<k} l_rm l_km) / sqrt(pivot) — no shared memory, no CTA barrier inside the panel;
//   2. all threads apply the rank-6 update to the trailing 18 x 18 band window, the 10 x 18 arrow window and the 10 x 10
//      corner sum, shifted by 6 into the other buffer, while the 6 entering rows / columns (raw entries, loaded one step
//      ahead during the panel phase) are appended.
// The updates are subtracted in ascending column order like a column-by-column right-looking factorisation, which this
// replaces (one column and one CTA barrier per step: 0.62 ms at D = 843; blocked: 139 steps instead of 834,
// profiles/r2s_lm_exchange_timing.md).  1 / L(j, j) is kept for the back substitution.
constexpr int FB = 6;                         // block = the 6 tangent parameters of one control point
constexpr int PANEL_ROWS = NB + NA;           // 24 band rows + 10 arrow rows
constexpr int N_ELEM = 300 + 240 + 55;        // window elements: band lower triangle, arrow, corner lower triangle
constexpr int EPT = (N_ELEM + FACTOR_THREADS - 1) / FACTOR_THREADS;

__global__ void __launch_bounds__(FACTOR_THREADS) k_lm_factor(LmDims d, LmBufs b) {
    __shared__ double W[2][NB * NB];
    __shared__ double A[2][NA * NB];
    __shared__ double P[PANEL_ROWS * FB];  // the factorised panel: P[row * 6 + k]; rows 0..23 band (0..5 = L11), 24..33 arrow
    __shared__ int s_fail;
    LmScalars *s = b.s;
    if (!s->running) return;
    const int sg = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const int j0 = 6 * d.seg_cp_off[sg], ns = 6 * d.seg_ncp[sg], n = d.n;
    double *Lb = b.Lb + (size_t) j0 * NB;
    // this thread's window elements: kind 0 band (r >= c), 1 arrow (r = arrow row, c = column), 2 corner (r >= c)
    int kind[EPT], er[EPT], ec[EPT];
#pragma unroll
    for (int q = 0; q < EPT; ++q) {
        const int e = tid + q * FACTOR_THREADS;
        kind[q] = 3, er[q] = 0, ec[q] = 0;
        if (e < 300 || (e >= 540 && e < N_ELEM)) {
            const int t = e < 300 ? e : e - 540;
            int r = (int) ((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
            while (r * (r + 1) / 2 > t) --r;
            while ((r + 1) * (r + 2) / 2 <= t) ++r;
            kind[q] = e < 300 ? 0 : 2, er[q] = r, ec[q] = t - r * (r + 1) / 2;
        } else if (e < 540) {
            kind[q] = 1, er[q] = (e - 300) / NB, ec[q] = (e - 300) % NB;
        }
    }
    // raw entries of the 6 rows / columns that enter the window after block step jb (global rows j + 24 .. j + 29)
    auto raw = [&](int q, int j) -> double {
        if (kind[q] == 0 && er[q] >= NB - FB) {
            const int i = j + FB + er[q];  // global row
            return i < ns ? Lb[(size_t) (j + FB + ec[q]) * NB + (er[q] - ec[q])] : 0.0;
        }
        if (kind[q] == 1 && ec[q] >= NB - FB) {
            const int c = j + FB + ec[q];
            return c < ns ? b.La[(size_t) er[q] * n + j0 + c] : 0.0;
        }
        return 0.0;
    };
    if (tid == 0) s_fail = 0;
#pragma unroll
    for (int q = 0; q < EPT; ++q) {  // initial window: rows / columns 0 .. 23 of the segment
        if (kind[q] == 0) W[0][er[q] * NB + ec[q]] = er[q] < ns ? Lb[(size_t) ec[q] * NB + (er[q] - ec[q])] : 0.0;
        if (kind[q] == 1) A[0][er[q] * NB + ec[q]] = ec[q] < ns ? b.La[(size_t) er[q] * n + j0 + ec[q]] : 0.0;
    }
    double acc = 0.0;  // corner update sum_j a_r a_c (the thread's kind-2 element, if any)
    __syncthreads();
    int cur = 0;
    for (int j = 0; j < ns; j += FB) {
        const double *Wc = W[cur], *Ac = A[cur];
        double *Wn = W[cur ^ 1], *An = A[cur ^ 1];
        double pre[EPT];
#pragma unroll
        for (int q = 0; q < EPT; ++q) pre[q] = raw(q, j);  // in flight during the panel phase
        if (tid < 32) {
            // ---- 1. panel: lane -> window row (band rows 0..23 | arrow rows 0..7), second row of lanes 0, 1: arrow rows 8, 9
            const bool band = lane < NB;
            double a1[FB], a2[FB];
#pragma unroll
            for (int k = 0; k < FB; ++k) {
                a1[k] = band ? (k <= lane ? Wc[lane * NB + k] : 0.0) : Ac[(lane - NB) * NB + k];
                a2[k] = lane < 2 ? Ac[(8 + lane) * NB + k] : 0.0;
            }
            bool bad = false;
#pragma unroll
            for (int k = 0; k < FB; ++k) {
                const double piv = __shfl_sync(0xffffffffu, a1[k], k);
                if (!(piv > 0.0)) bad = true;  // not positive definite (uniform)
                const double rs = rsqrt(piv);  // <= 1 ulp; sqrt + division were 3/4 of the panel's dependent chain
                a1[k] *= rs;  // rows above the diagonal of a band column hold zeros: harmless
                a2[k] *= rs;
                if (lane == 0) b.Lc[j0 + j + k] = rs;  // 1 / L(j + k, j + k)
#pragma unroll
                for (int m = k + 1; m < FB; ++m) {
                    const double lmk = __shfl_sync(0xffffffffu, a1[k], m);  // L(j + m, j + k): row m of the diagonal block
                    if (!band || lane >= m) a1[m] -= a1[k] * lmk;
                    a2[m] -= a2[k] * lmk;
                }
            }
            if (bad) s_fail = 1;
#pragma unroll
            for (int k = 0; k < FB; ++k) {
                P[lane * FB + k] = (band && k > lane) ? 0.0 : a1[k];
                if (lane < 2) P[(32 + lane) * FB + k] = a2[k];
                if (band) {  // column j + k of L: L(j + r, j + k) at band offset r - k
                    if (lane >= k && j + lane < ns) Lb[(size_t) (j + k) * NB + (lane - k)] = a1[k];
                } else {
                    b.La[(size_t) (lane - NB) * n + j0 + j + k] = a1[k];
                }
                if (lane < 2) b.La[(size_t) (8 + lane) * n + j0 + j + k] = a2[k];
            }
        }
        __syncthreads();
        if (s_fail) break;
        // ---- 2. rank-6 update of the trailing window, shifted by one block into the other buffer
#pragma unroll
        for (int q = 0; q < EPT; ++q) {
            const int r = er[q], c = ec[q];
            if (kind[q] == 0) {
                double v;
                if (r < NB - FB) {
                    v = Wc[(r + FB) * NB + (c + FB)];
                    const double *pr = P + (r + FB) * FB, *pc = P + (c + FB) * FB;
#pragma unroll
                    for (int k = 0; k < FB; ++k) v -= pr[k] * pc[k];
                } else {
                    v = pre[q];
                }
                Wn[r * NB + c] = v;
            } else if (kind[q] == 1) {
                double v;
                if (c < NB - FB) {
                    v = Ac[r * NB + c + FB];
                    const double *pr = P + (NB + r) * FB, *pc = P + (c + FB) * FB;
#pragma unroll
                    for (int k = 0; k < FB; ++k) v -= pr[k] * pc[k];
                } else {
                    v = pre[q];
                }
                An[r * NB + c] = v;
            } else if (kind[q] == 2) {
                const double *pr = P + (NB + r) * FB, *pc = P + (NB + c) * FB;
#pragma unroll
                for (int k = 0; k < FB; ++k) acc += pr[k] * pc[k];
            }
        }
        __syncthreads();
        cur ^= 1;
    }
    if (s_fail && tid == 0) atomicExch(&s->factor_fail, 1);
#pragma unroll
    for (int q = 0; q < EPT; ++q)
        if (kind[q] == 2) b.dC[(size_t) sg * NA * NA + er[q] * NA + ec[q]] = acc;
}

// Schur complement of the intrinsics, its Cholesky factor with the right-hand side row, and the intrinsics part of M^-1 gs
__global__ void k_lm_corner(LmDims d, LmBufs b) {
    LmScalars *s = b.s;
    if (!s->running || threadIdx.x != 0 || blockIdx.x != 0) return;
    double Cw[NA][NA];
    for (int r = 0; r < NA; ++r)
        for (int c = 0; c <= r; ++c) {
            double v = b.Cc0[r * NA + c];
            for (int sg = 0; sg < d.n_seg; ++sg) v -= b.dC[(size_t) sg * NA * NA + r * NA + c];
            Cw[r][c] = v;
        }
    bool ok = s->factor_fail == 0;
    for (int r = 0; r < NA && ok; ++r)
        for (int c = 0; c <= r && c < NI; ++c) {
            double v = Cw[r][c];
            for (int k = 0; k < c; ++k) v -= Cw[r][k] * Cw[c][k];
            if (r == c) {
                if (!(v > 0.0)) {
                    ok = false;
                    break;
                }
                Cw[r][r] = sqrt(v);
            } else {
                Cw[r][c] = v / Cw[c][c];
            }
        }
    if (b.Lcc)  // a failed row keeps its non-positive pivot, later rows their partial Schur complement
        for (int r = 0; r < NI; ++r)
            for (int c = 0; c <= r; ++c) b.Lcc[r * NI + c] = Cw[r][c];
    if (!ok) {
        s->factor_fail = 1;
        return;
    }
    double xi[NI];
    for (int r = NI - 1; r >= 0; --r) {  // L^T xi = y, y = row 9
        double v = Cw[NI][r];
        for (int k = r + 1; k < NI; ++k) v -= Cw[k][r] * xi[k];
        xi[r] = v / Cw[r][r];
    }
    for (int r = 0; r < NI; ++r) b.xi[r] = xi[r];
}

// back substitution of one segment, L^T x = y - A^T xi, column oriented: as soon as x_j is known every lane adds its term
// L(j, j - 1 - r) x_j to the pending sum of row j - 1 - r and the sums move down one lane — one shuffle and three FP64
// operations on the critical path per unknown instead of a five-level shuffle tree and a division.  Warp 0 runs the
// recurrence out of shared memory; warps 1 .. 3 stage the next chunk of L, y and 1 / L(j, j) meanwhile (coalesced loads,
// two buffers), so no global-memory latency sits on the sequential chain (0.35 ms at D = 843 before, ncu).
constexpr int BS_THREADS = 128, BS_CHUNK = 64, BS_ROW = NB + 1;  // per step: 23 band terms, y, 1 / diag  (25 doubles)

__global__ void __launch_bounds__(BS_THREADS) k_lm_backsub(LmDims d, LmBufs b) {
    __shared__ double buf[2][BS_CHUNK * BS_ROW];
    const LmScalars *s = b.s;
    if (!s->running || s->factor_fail) return;
    const int sg = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const int j0 = 6 * d.seg_cp_off[sg], ns = 6 * d.seg_ncp[sg], n = d.n;
    const double *Lb = b.Lb + (size_t) j0 * NB;
    // right-hand side with the arrow part taken out:  ya_j = y_j - sum_k A(k, j) xi_k   (y = arrow row 9 after the factorisation)
    {
        double xi[NI];
#pragma unroll
        for (int k = 0; k < NI; ++k) xi[k] = b.xi[k];
        for (int j = tid; j < ns; j += BS_THREADS) {
            double v = b.La[(size_t) NI * n + j0 + j];
#pragma unroll
            for (int k = 0; k < NI; ++k) v -= b.La[(size_t) k * n + j0 + j] * xi[k];
            b.ysol[j0 + j] = v;
        }
    }
    __syncthreads();
    // chunk q covers the unknowns j = hi(q) - 1 ... hi(q) - BS_CHUNK (descending), hi(q) = ns - q * BS_CHUNK
    const int n_chunks = (ns + BS_CHUNK - 1) / BS_CHUNK;
    auto stage = [&](int q, int first_thread, int n_threads) {  // slot t of the chunk = unknown j = hi - 1 - t
        const int hi = ns - q * BS_CHUNK;
        double *o = buf[q & 1];
        for (int e = tid - first_thread; e < BS_CHUNK * BS_ROW; e += n_threads) {
            const int t = e / BS_ROW, r = e - t * BS_ROW, j = hi - 1 - t;
            double v = 0.0;
            if (j >= 0) {
                if (r < NB - 1) {  // L(j, j - 1 - r): column j - 1 - r, band offset 1 + r
                    const int c = j - 1 - r;
                    if (c >= 0) v = Lb[(size_t) c * NB + 1 + r];
                } else if (r == NB - 1) {
                    v = b.ysol[j0 + j];
                } else {
                    v = b.Lc[j0 + j];
                }
            }
            o[e] = v;
        }
    };
    stage(0, 0, BS_THREADS);
    __syncthreads();
    double acc = 0.0;  // warp 0, at the start of step j: lane r holds sum_{i > row} L(i, row) x_i collected so far for row = j - r
    for (int q = 0; q < n_chunks; ++q) {
        if (tid >= 32) {
            if (q + 1 < n_chunks) stage(q + 1, 32, BS_THREADS - 32);
        } else {
            const double *c = buf[q & 1];
            const int hi = ns - q * BS_CHUNK, steps = min(BS_CHUNK, hi);
            double l = lane < NB - 1 ? c[lane] : 0.0, y = c[NB - 1], rd = c[NB];
            for (int t = 0; t < steps; ++t) {
                const double *nx = c + (t + 1 < BS_CHUNK ? (t + 1) * BS_ROW : 0);  // next step's operands, loaded ahead of the chain
                const double l1 = lane < NB - 1 ? nx[lane] : 0.0, y1 = nx[NB - 1], rd1 = nx[NB];
                const double xj = (y - __shfl_sync(0xffffffffu, acc, 0)) * rd;
                if (lane == 0) b.ysol[j0 + hi - 1 - t] = xj;
                acc = __shfl_down_sync(0xffffffffu, acc, 1);  // lane r: row j - 1 - r (independent of x_j: off the critical path)
                if (lane == 31) acc = 0.0;
                acc += l * xj;                                // + L(j, j - 1 - r) x_j
                l = l1, y = y1, rd = rd1;
            }
        }
        __syncthreads();
    }
}

// step = -M^-1 gs, model cost change from the undamped scaled system, candidate parameters
__global__ void __launch_bounds__(1024) k_lm_step(LmDims d, LmBufs b, ecb_lm_options o) {
    __shared__ double sh[3][1024];
    LmScalars *s = b.s;
    if (!s->running) return;
    const int n = d.n, D = d.D, tid = threadIdx.x, nthr = blockDim.x;
    const bool solved = s->factor_fail == 0;
    if (solved) {
        for (int i = tid; i < D; i += nthr) b.step[i] = i < n ? -b.ysol[i] : -b.xi[i - n];
    }
    __syncthreads();
    double a = 0.0, bb = 0.0;
    if (solved) {
        for (int i = tid; i < D; i += nthr) {
            double hd = 0.0;  // (S H S step)_i
            const double si = b.scale[i];
            if (i < n) {
                for (int r = 0; r < NB && i + r < n; ++r) hd += b.Hb[(size_t) i * NB + r] * si * b.scale[i + r] * b.step[i + r];
                for (int r = 1; r < NB && i - r >= 0; ++r) hd += b.Hb[(size_t) (i - r) * NB + r] * si * b.scale[i - r] * b.step[i - r];
                for (int k = 0; k < NI; ++k) hd += b.Ha[(size_t) k * n + i] * si * b.scale[n + k] * b.step[n + k];
            } else {
                const int k = i - n;
                for (int j = 0; j < n; ++j) hd += b.Ha[(size_t) k * n + j] * si * b.scale[j] * b.step[j];
                for (int c = 0; c < NI; ++c) hd += b.Hc[k * NI + c] * si * b.scale[n + c] * b.step[n + c];
            }
            a += b.step[i] * (b.g[i] * si);
            bb += b.step[i] * hd;
        }
    }
    sh[0][tid] = a;
    sh[1][tid] = bb;
    __syncthreads();
    for (int st = 512; st > 0; st >>= 1) {
        if (tid < st) {
            sh[0][tid] += sh[0][tid + st];
            sh[1][tid] += sh[1][tid + st];
        }
        __syncthreads();
    }
    const double mcc = -(sh[0][0] + 0.5 * sh[1][0]);
    const bool valid = solved && mcc > 0.0 && isfinite(mcc);
    __syncthreads();
    double xn = 0.0, sn = 0.0;
    if (valid) {
        for (int i = tid; i < D; i += nthr) b.delta[i] = b.step[i] * b.scale[i];
        __syncthreads();
        const double *intr = b.x, *rot = b.x + 9, *trans = b.x + 9 + 4 * (size_t) d.C;
        double *cintr = b.cand, *crot = b.cand + 9, *ctrans = b.cand + 9 + 4 * (size_t) d.C;
        for (int c = tid; c < d.C + 1; c += nthr) {
            if (c == d.C) {
                for (int i = 0; i < 9; ++i) {
                    const double v = intr[i] + b.delta[n + i];
                    cintr[i] = v;
                    xn += intr[i] * intr[i];
                    sn += (intr[i] - v) * (intr[i] - v);
                }
                continue;
            }
            double q[4];
            if (o.rotation_model == 1) ecb_so3::plus(rot + 4 * c, b.delta + 6 * c, q);
            else quat_plus_dev(rot + 4 * c, b.delta + 6 * c, q);
            for (int k = 0; k < 4; ++k) {
                crot[4 * c + k] = q[k];
                xn += rot[4 * c + k] * rot[4 * c + k];
                sn += (rot[4 * c + k] - q[k]) * (rot[4 * c + k] - q[k]);
            }
            for (int k = 0; k < 3; ++k) {
                const double t = trans[3 * c + k], v = t + b.delta[6 * c + 3 + k];
                ctrans[3 * c + k] = v;
                xn += t * t;
                sn += (t - v) * (t - v);
            }
        }
    }
    sh[0][tid] = xn;
    sh[1][tid] = sn;
    __syncthreads();
    for (int st = 512; st > 0; st >>= 1) {
        if (tid < st) {
            sh[0][tid] += sh[0][tid + st];
            sh[1][tid] += sh[1][tid + st];
        }
        __syncthreads();
    }
    if (tid == 0) {
        if (valid) {
            s->model_cost_change = mcc;
            s->x_norm = sqrt(sh[0][0]);
            s->step_norm = sqrt(sh[1][0]);
            s->invalid_steps = 0;
            s->go_cost = 1;
        } else {  // invalid step: shrink the region; the next iteration tries again (Ceres: HandleInvalidStep)
            s->step_valid = 0;
            if (++s->invalid_steps > 5) {
                s->termination = ECB_LM_FAILURE;
                s->running = 0;
            } else {
                s->radius /= s->decrease_factor;
                s->decrease_factor *= 2.0;
                s->reuse_diagonal = 1;
                record(s, b.trace, -1.0);
            }
        }
    }
}

__global__ void k_lm_decide(LmBufs b, ecb_lm_options o) {
    LmScalars *s = b.s;
    s->accepted = 0;
    if (!s->running || !s->step_valid) return;
    const double candidate_cost = s->candidate_cost;
    if (!o.fixed_iterations) {
        if (s->step_norm <= o.parameter_tolerance * (s->x_norm + o.parameter_tolerance)) {
            s->termination = ECB_LM_PARAMETER_TOLERANCE;
            s->running = 0;
            return;
        }
        if (fabs(s->cost - candidate_cost) <= o.function_tolerance * s->cost) {
            s->termination = ECB_LM_FUNCTION_TOLERANCE;
            s->running = 0;
            return;
        }
    }
    const double rho = (s->cost - candidate_cost) / s->model_cost_change;
    if (rho > o.min_relative_decrease) {
        s->accepted = 1;  // k_lm_commit moves x, the normal equations are evaluated at the new point
        ++s->successful;
        const double t = 2.0 * rho - 1.0;
        s->radius = fmin(o.max_radius, s->radius / fmax(1.0 / 3.0, 1.0 - t * t * t));
        s->decrease_factor = 2.0;
        s->reuse_diagonal = 0;
        return;
    }
    s->radius /= s->decrease_factor;
    s->decrease_factor *= 2.0;
    s->reuse_diagonal = 1;
    record(s, b.trace, 0.0);
    if (s->radius < o.min_radius) {
        if (o.fixed_iterations) {
            s->radius = o.min_radius;  // benchmark mode (config C4): exactly max_iterations iterations, no early exit
        } else {
            s->termination = ECB_LM_MIN_RADIUS;
            s->running = 0;
        }
    }
}

__global__ void k_lm_commit(LmBufs b, size_t n_params) {
    if (!b.s->accepted) return;
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < n_params; i += (size_t) gridDim.x * blockDim.x) b.x[i] = b.cand[i];
}

__global__ void k_lm_epoch(const int *go, unsigned long long *epoch) {
    if (*go) ++*epoch;
}

__global__ void k_lm_set_cost(LmBufs b, const double *v) { b.s->candidate_cost = *v; }

// ---- covariance of the parameters: Z = H^-1 on the band / arrow pattern (selected inversion) -----------------------------------
// ecb_covariance runs k_lm_assemble, k_lm_build, k_lm_factor and k_lm_corner unchanged on M = S H S with S = diag(H)^-1/2 (1 where
// the diagonal is 0) and no damping (radius = +inf: the damping term dg / radius adds exactly 0), then the kernels below.
// Constant intrinsics (cmask): their rows / columns of H are zero after k_lm_assemble; k_cov_begin gives them a unit diagonal, so
// M is the free block and an identity block that the factorisation keeps apart exactly, and Z of the free block is the inverse of
// H restricted to the free parameters.  k_cov_corner and k_cov_selinv write exact zeros into their rows / columns of Z.
constexpr double COV_MIN_PIVOT = 1e-12;  // relative pivot L(j, j)^2 / M(j, j) at or below which the system counts as rank deficient
constexpr int COV_THREADS = 256;
constexpr int CW = NB - 1 + NI;          // selected-inversion window: 23 band rows + 9 intrinsics = 32

struct CovBufs {
    double *Zb, *Zx, *Zc;  // outputs, unscaled: band (column major like Hb), cross 9 x n, corner 9 x 9
    double *Zcs, *Lcc;     // scaled corner of Z, corner factor of k_lm_corner
    double *res;           // cost, min relative pivot, first deficient index (-1: none)
};

// Jacobi equilibration to a unit diagonal and the state the LM kernels read
__global__ void k_cov_begin(LmDims d, LmBufs b, uint32_t cmask) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < d.D; i += gridDim.x * blockDim.x) {
        if (i >= d.n && ((cmask >> (i - d.n)) & 1u)) b.Hc[(i - d.n) * (NI + 1)] = 1.0;  // constant intrinsic: unit diagonal
        const double h = h_diag(d, b, i);
        b.scale[i] = h > 0.0 ? 1.0 / sqrt(h) : 1.0;
        if (i < d.n) b.Lc[i] = 0.0;  // a pivot the factorisation does not reach (it stops a segment at a failed pivot) stays 0
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        LmScalars *s = b.s;
        s->running = 1;
        s->radius = INFINITY;
        s->reuse_diagonal = 0;
        s->factor_fail = 0;
    }
}

// relative pivots of the factorisation: their minimum and the first index j with L(j, j)^2 / M(j, j) <= COV_MIN_PIVOT (or a
// failed pivot); the band comes first in the factorisation, so a band failure is reported before the intrinsics
__global__ void __launch_bounds__(1024) k_cov_pivots(LmDims d, LmBufs b, CovBufs c) {
    __shared__ double smin[1024];
    __shared__ int sbad[1024];
    const int tid = threadIdx.x;
    double mn = INFINITY;
    int bad = INT_MAX;
    for (int i = tid; i < d.D; i += blockDim.x) {
        double rel;
        if (i < d.n) {
            const double rc = b.Lc[i], m = b.Hb[(size_t) i * NB] * b.scale[i] * b.scale[i];
            if (rc == 0.0) continue;  // behind a failed pivot of the same segment
            rel = (isfinite(rc) && m > 0.0) ? 1.0 / (rc * rc * m) : 0.0;
        } else {
            const int r = i - d.n;
            const double l = c.Lcc[r * NI + r], m = b.Cc0[r * NA + r];
            rel = (l > 0.0 && m > 0.0) ? l * l / m : 0.0;
        }
        mn = fmin(mn, rel);
        if (!(rel > COV_MIN_PIVOT)) bad = min(bad, i);
    }
    smin[tid] = mn;
    sbad[tid] = bad;
    __syncthreads();
    for (int st = 512; st > 0; st >>= 1) {
        if (tid < st) {
            smin[tid] = fmin(smin[tid], smin[tid + st]);
            sbad[tid] = min(sbad[tid], sbad[tid + st]);
        }
        __syncthreads();
    }
    if (tid == 0) {
        c.res[0] = b.s->cost;
        c.res[1] = smin[0];
        c.res[2] = sbad[0] == INT_MAX ? -1.0 : (double) sbad[0];
    }
}

// Z_cc = (L_cc L_cc^T)^-1 of the 9 x 9 Schur factor: W = L_cc^-1 column by column (one thread each), Z_cc = W^T W
__global__ void k_cov_corner(LmDims d, LmBufs b, CovBufs c, uint32_t cmask) {
    __shared__ double W[NI][NI];
    if (c.res[2] >= 0.0) return;
    const int t = threadIdx.x;
    if (t < NI) {
        for (int r = 0; r < NI; ++r) {
            double v = r == t ? 1.0 : 0.0;
            for (int k = t; k < r; ++k) v -= c.Lcc[r * NI + k] * W[k][t];
            W[r][t] = r < t ? 0.0 : v / c.Lcc[r * NI + r];
        }
    }
    __syncthreads();
    if (t < NI * NI) {
        const int r = t / NI, q = t % NI, lo = max(r, q);
        double v = 0.0;
        for (int k = lo; k < NI; ++k) v += W[k][r] * W[k][q];
        c.Zcs[t] = v;
        c.Zc[t] = ecb_zero_constant(cmask, r, q, v * (b.scale[d.n + min(r, q)] * b.scale[d.n + lo]));  // the same rounding for (r, q) and (q, r): symmetric
    }
}

// Selected inversion (Takahashi) of one segment, blocked by control point like k_lm_factor.  With B the 6 columns of the block
// and K the rows L couples to them (the next 18 band rows of the segment and the 9 intrinsics), Z L = L^-T gives
//   Z_{R,B} = -Z_{R,K} T,   Z_BB = L_BB^-T L_BB^-1 - Z_{K,B}^T T,   T = L_KB L_BB^-1,
// for R = the next 23 band rows + the intrinsics (the band reach of the block's last column).  Every Z_{R,K} lies in the
// 32 x 32 window of Z the previous block left in shared memory; the window then slides up by one block.  The result equals the
// scalar recurrence Z_ij = -(1 / L_jj) sum_{k in N(j)} Z_ik L_kj run column by column.  Outputs are unscaled by S on the way out.
__global__ void __launch_bounds__(COV_THREADS) k_cov_selinv(LmDims d, LmBufs b, CovBufs c, uint32_t cmask) {
    __shared__ double Zw[2][CW * CW];  // window: index w < 23 -> band row j0 + 6 + w of the segment, w >= 23 -> intrinsic w - 23
    __shared__ double LB[FB][FB], LK[NB - FB + NI][FB], T[NB - FB + NI][FB], Wb[FB][FB], Y[CW][FB], ZB[FB][FB], rdg[FB];
    if (c.res[2] >= 0.0) return;
    const int sg = blockIdx.x, tid = threadIdx.x, n = d.n;
    const int js = 6 * d.seg_cp_off[sg], ns = 6 * d.seg_ncp[sg];
    constexpr int NK = NB - FB + NI;   // 27 coupled rows: window indices 0..17 and 23..31
    auto kwin = [](int q) { return q < NB - FB ? q : q + (NB - 1) - (NB - FB); };
    for (int e = tid; e < CW * CW; e += COV_THREADS) {  // the last block's window: rows past the segment are 0, the corner is Z_cc
        const int r = e / CW, q = e % CW;
        Zw[0][e] = (r >= NB - 1 && q >= NB - 1) ? c.Zcs[(r - (NB - 1)) * NI + (q - (NB - 1))] : 0.0;
    }
    int cur = 0;
    for (int j0 = ns - FB; j0 >= 0; j0 -= FB) {
        const double *Zp = Zw[cur];
        double *Zn = Zw[cur ^ 1];
        const int g0 = js + j0;  // global index of the block's first column
        // L of the block: L_BB (6 x 6 lower), L_KB (27 x 6), 1 / L(j, j)
        if (tid < FB * FB) {
            const int r = tid / FB, k = tid % FB;
            LB[r][k] = r >= k ? b.Lb[(size_t) (g0 + k) * NB + (r - k)] : 0.0;
            if (r == 0) rdg[k] = b.Lc[g0 + k];
        } else if (tid < FB * FB + NK * FB) {
            const int q = (tid - FB * FB) / FB, k = (tid - FB * FB) % FB;
            LK[q][k] = q < NB - FB ? (j0 + FB + q < ns ? b.Lb[(size_t) (g0 + k) * NB + (FB + q - k)] : 0.0)
                                   : b.La[(size_t) (q - (NB - FB)) * n + g0 + k];
        }
        __syncthreads();
        if (tid < NK) {  // T row q: T_q L_BB = L_Kq, columns right to left
            double t[FB];
#pragma unroll
            for (int k = FB - 1; k >= 0; --k) {
                double v = LK[tid][k];
#pragma unroll
                for (int m = k + 1; m < FB; ++m) v -= t[m] * LB[m][k];
                t[k] = v * rdg[k];
            }
#pragma unroll
            for (int k = 0; k < FB; ++k) T[tid][k] = t[k];
        } else if (tid >= 32 && tid < 32 + FB) {  // column k of W = L_BB^-1
            const int k = tid - 32;
#pragma unroll
            for (int r = 0; r < FB; ++r) {
                double v = r == k ? 1.0 : 0.0;
                for (int m = k; m < r; ++m) v -= LB[r][m] * Wb[m][k];
                Wb[r][k] = r < k ? 0.0 : v * rdg[r];
            }
        }
        __syncthreads();
        if (tid < CW * FB) {  // Z_{R,B} = -Z_{R,K} T
            const int w = tid / FB, k = tid % FB;
            double v = 0.0;
#pragma unroll 9
            for (int q = 0; q < NK; ++q) v += Zp[w * CW + kwin(q)] * T[q][k];
            Y[w][k] = -v;
        }
        __syncthreads();
        if (tid < FB * FB) {  // Z_BB (lower triangle, mirrored)
            const int r = tid / FB, k = tid % FB;
            if (r >= k) {
                double v = 0.0;
                for (int m = r; m < FB; ++m) v += Wb[m][r] * Wb[m][k];
                for (int q = 0; q < NK; ++q) v -= Y[kwin(q)][r] * T[q][k];
                ZB[r][k] = v;
                ZB[k][r] = v;
            }
        }
        __syncthreads();
        // outputs of the block's 6 columns, and the window of the next block (band rows j0 - 6 + 6 .. , i.e. B first)
        for (int e = tid; e < FB * NB + NI * FB; e += COV_THREADS) {
            if (e < FB * NB) {
                const int k = e / NB, r = e % NB, i = j0 + k + r;  // row inside the segment
                double v = 0.0;
                if (i < ns) v = (i < j0 + FB ? ZB[i - j0][k] : Y[i - j0 - FB][k]) * b.scale[js + i] * b.scale[g0 + k];
                c.Zb[(size_t) (g0 + k) * NB + r] = v;
            } else {
                const int a = (e - FB * NB) / FB, k = (e - FB * NB) % FB;
                c.Zx[(size_t) a * n + g0 + k] = ecb_zero_constant(cmask, a, -1, Y[NB - 1 + a][k] * b.scale[n + a] * b.scale[g0 + k]);
            }
        }
        for (int e = tid; e < CW * CW; e += COV_THREADS) {
            const int r = e / CW, q = e % CW;
            const int orr = r < FB ? -1 : (r < NB - 1 ? r - FB : r), oq = q < FB ? -1 : (q < NB - 1 ? q - FB : q);
            double v;
            if (orr < 0 && oq < 0) v = ZB[r][q];
            else if (orr < 0) v = Y[oq][r];
            else if (oq < 0) v = Y[orr][q];
            else v = Zp[orr * CW + oq];
            Zn[e] = v;
        }
        __syncthreads();
        cur ^= 1;
    }
}

}  // namespace

struct ecb_lm_device {
    ecb_ctx *ctx = nullptr;
    ecb_lm_options opt;
    LmDims dims;
    LmBufs bufs;
    DevBuf mem, tab;
    size_t n_params = 0, ne_doubles = 0;
    int rank = 0, n_ranks = 1;
    void *recv[ECB_MAX_PEERS] = {};
    double *d_cand_cost = nullptr;
    uint32_t generation = 0;
    uint32_t const_intrinsics = 0;  // the context's constant intrinsics at creation
    bool begun = false;
    // ECB_LM_TIMING=1: CUDA events around the phases of every enqueued iteration (solve | candidate cost | scalar exchange |
    // decide + commit | normal equations (+ exchange) | assemble), averaged and printed to stderr by ecb_lm_device_result
    std::vector<cudaEvent_t> tev;
    int t_iters = 0;
};
constexpr int LM_TPH = 7;  // events per timed iteration

extern "C" {

int ecb_lm_device_create(ecb_ctx *ctx, int n_splines, const int32_t *n_cp, const ecb_lm_options *opt, ecb_lm_device **out) {
    if (!ctx || !out || n_splines < 1 || !n_cp) return ECB_ERR_ARG;
    *out = nullptr;
    if (!ctx->cost) return ecb_fail(ctx, ECB_ERR_STATE, "ecb_cost_setup first");
    int32_t tcp = 0, tsp = 0;
    int64_t nd = 0;
    int rc = ecb_cost_layout(ctx, &tcp, &tsp, nullptr, &nd);
    if (rc) return rc;
    int C = 0;
    for (int s = 0; s < n_splines; ++s) C += n_cp[s];
    if (C != tcp) return ecb_fail(ctx, ECB_ERR_ARG, "spline layout differs from ecb_cost_setup");
    cudaSetDevice(ctx->device);
    ecb_lm_device *lm = new ecb_lm_device();
    lm->ctx = ctx;
    lm->const_intrinsics = ctx->const_intrinsics;
    if (opt) lm->opt = *opt; else ecb_lm_default_options(&lm->opt);
    const int n = 6 * C, D = n + NI;
    // integer tables
    std::vector<int> tabv;
    std::vector<int> cp_seg(C), cp_local(C), seg_cp_off(n_splines), seg_ncp(n_splines), seg_span_off(n_splines);
    int co = 0, so = 0;
    for (int s = 0; s < n_splines; ++s) {
        seg_cp_off[s] = co;
        seg_ncp[s] = n_cp[s];
        seg_span_off[s] = so;
        for (int k = 0; k < n_cp[s]; ++k) cp_seg[co + k] = s, cp_local[co + k] = k;
        co += n_cp[s];
        so += n_cp[s] - 3;
    }
    for (auto *v : {&cp_seg, &cp_local, &seg_cp_off, &seg_ncp, &seg_span_off}) tabv.insert(tabv.end(), v->begin(), v->end());
    if ((rc = ecb_reserve(ctx, lm->tab, tabv.size() * 4))) {
        delete lm;
        return rc;
    }
    cudaMemcpyAsync(lm->tab.p, tabv.data(), tabv.size() * 4, cudaMemcpyHostToDevice, ctx->stream);
    ecb_stream_sync(ctx);
    const int *t = (const int *) lm->tab.p;
    lm->dims.C = C;
    lm->dims.n = n;
    lm->dims.D = D;
    lm->dims.n_spans = tsp;
    lm->dims.n_seg = n_splines;
    lm->dims.cp_seg = t;
    lm->dims.cp_local = t + C;
    lm->dims.seg_cp_off = t + 2 * C;
    lm->dims.seg_ncp = t + 2 * C + n_splines;
    lm->dims.seg_span_off = t + 2 * C + 2 * n_splines;
    lm->n_params = 9 + 7 * (size_t) C;
    lm->ne_doubles = (size_t) nd;
    // one allocation for all double arrays
    size_t off = 0;
    auto take = [&](size_t cnt) {
        const size_t o = off;
        off += (cnt + 1) & ~(size_t) 1;
        return o;
    };
    const size_t o_x = take(lm->n_params), o_cand = take(lm->n_params), o_ne = take(lm->ne_doubles + 2);
    const size_t o_Hb = take((size_t) n * NB), o_Ha = take((size_t) NI * n), o_Hc = take(NI * NI), o_g = take(D);
    const size_t o_scale = take(D), o_diag = take(D), o_step = take(D), o_delta = take(D);
    const size_t o_Lb = take((size_t) n * NB), o_La = take((size_t) NA * n), o_Cc0 = take(NA * NA);
    const size_t o_dC = take((size_t) n_splines * NA * NA), o_Lc = take((size_t) std::max(n, NA * NA)), o_xi = take(NI + 1), o_ysol = take(D);
    const size_t o_trace = take((size_t) TRACE_CAP * 4), o_cc = take(2), o_s = take((sizeof(LmScalars) + 7) / 8 + 2);
    if ((rc = ecb_reserve(ctx, lm->mem, off * 8))) {
        delete lm;
        return rc;
    }
    cudaMemsetAsync(lm->mem.p, 0, off * 8, ctx->stream);
    double *m = (double *) lm->mem.p;
    lm->bufs = LmBufs{m + o_x, m + o_cand, m + o_ne, m + o_Hb, m + o_Ha, m + o_Hc, m + o_g, m + o_scale, m + o_diag, m + o_step,
                      m + o_delta, m + o_Lb, m + o_La, m + o_Cc0, m + o_dC, m + o_Lc, m + o_xi, m + o_ysol, m + o_trace,
                      (LmScalars *) (m + o_s)};
    lm->d_cand_cost = m + o_cc;
    *out = lm;
    return ecb_check(ctx, ecb_stream_sync(ctx), "device LM allocation");
}

void ecb_lm_device_destroy(ecb_lm_device *lm) {
    if (!lm) return;
    cudaSetDevice(lm->ctx->device);
    cudaStreamSynchronize(lm->ctx->stream);
    if (lm->mem.p) cudaFree(lm->mem.p);
    if (lm->tab.p) cudaFree(lm->tab.p);
    delete lm;
}

int ecb_lm_device_set_exchange(ecb_lm_device *lm, int rank, int n_ranks, void *const *recv_buffers) {
    if (!lm || n_ranks < 1 || n_ranks > ECB_MAX_PEERS || rank < 0 || rank >= n_ranks) return ECB_ERR_ARG;
    if (n_ranks > 1 && !recv_buffers) return ECB_ERR_ARG;
    lm->rank = rank;
    lm->n_ranks = n_ranks;
    for (int p = 0; p < n_ranks && recv_buffers; ++p) lm->recv[p] = recv_buffers[p];
    return ECB_OK;
}

// normal equations of ALL ranks at x -> ne; gated by the `accepted` flag
static int lmdev_normal_eq(ecb_lm_device *lm) {
    ecb_ctx *ctx = lm->ctx;
    LmScalars *s = lm->bufs.s;
    if (lm->n_ranks > 1) {
        k_lm_epoch<<<1, 1, 0, ctx->stream>>>(&s->accepted, &s->epoch_ne);
        ECB_LAUNCHED(ctx);
        return ecb_cost_dev_normal_eq_exchange(ctx, lm->bufs.x, &s->accepted, lm->rank, lm->n_ranks, lm->recv, &s->epoch_ne, 0,
                                               ECB_EXCHANGE_BOTH, lm->bufs.ne, &s->xerr);
    }
    return ecb_cost_dev_normal_eq(ctx, lm->bufs.x, &s->accepted, lm->bufs.ne);
}

int ecb_lm_device_begin(ecb_lm_device *lm, const double *intrinsics, const double *rot_cp, const double *trans_cp) {
    if (!lm || !intrinsics || !rot_cp || !trans_cp) return ECB_ERR_ARG;
    ecb_ctx *ctx = lm->ctx;
    cudaSetDevice(ctx->device);
    int rc;
    const size_t C = (size_t) lm->dims.C;
    if ((rc = ecb_h2d(ctx, lm->bufs.x, intrinsics, 72))) return rc;
    if ((rc = ecb_h2d(ctx, lm->bufs.x + 9, rot_cp, 32 * C))) return rc;
    if ((rc = ecb_h2d(ctx, lm->bufs.x + 9 + 4 * C, trans_cp, 24 * C))) return rc;
    // fresh state; exchange epochs of this run start above everything earlier runs left in the receive buffers
    LmScalars h;
    memset(&h, 0, sizeof h);
    h.accepted = 1;
    h.running = 1;
    ++lm->generation;
    h.epoch_ne = h.epoch_sc = ((unsigned long long) lm->generation << 40) * 2ull;
    if ((rc = ecb_h2d(ctx, lm->bufs.s, &h, sizeof h))) return rc;
    if ((rc = lmdev_normal_eq(lm))) return rc;
    const int blocks = ctx->sm_count * 2;
    k_lm_assemble<<<blocks, 256, 0, ctx->stream>>>(lm->dims, lm->bufs, nullptr, lm->const_intrinsics);
    ECB_LAUNCHED(ctx);
    k_lm_init<<<std::min(blocks, (lm->dims.D + 255) / 256), 256, 0, ctx->stream>>>(lm->dims, lm->bufs, lm->opt);
    ECB_LAUNCHED(ctx);
    k_lm_gradnorm<<<1, 1024, 0, ctx->stream>>>(lm->dims, lm->bufs, lm->opt, nullptr);
    ECB_LAUNCHED(ctx);
    lm->begun = true;
    return ecb_check(ctx, cudaGetLastError(), "device LM begin");
}

int ecb_lm_device_iterate(ecb_lm_device *lm, int n_iterations) {
    if (!lm || n_iterations < 0) return ECB_ERR_ARG;
    if (!lm->begun) return ecb_fail(lm->ctx, ECB_ERR_STATE, "ecb_lm_device_begin first");
    ecb_ctx *ctx = lm->ctx;
    cudaSetDevice(ctx->device);
    LmScalars *s = lm->bufs.s;
    const int blocks = ctx->sm_count * 2;
    int rc;
    static const bool timing = getenv("ECB_LM_TIMING") && atoi(getenv("ECB_LM_TIMING")) != 0;
    auto mark = [&](int k) {
        if (!timing || lm->t_iters >= 64) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, ctx->stream);
        lm->tev.push_back(e);
        if (k == LM_TPH - 1) ++lm->t_iters;
    };
    for (int it = 0; it < n_iterations; ++it) {
        mark(0);
        k_lm_iter_begin<<<1, 1, 0, ctx->stream>>>(lm->bufs, lm->opt);
        k_lm_build<<<blocks, 256, 0, ctx->stream>>>(lm->dims, lm->bufs, lm->opt);
        k_lm_factor<<<lm->dims.n_seg, FACTOR_THREADS, 0, ctx->stream>>>(lm->dims, lm->bufs);
        k_lm_corner<<<1, 32, 0, ctx->stream>>>(lm->dims, lm->bufs);
        k_lm_backsub<<<lm->dims.n_seg, BS_THREADS, 0, ctx->stream>>>(lm->dims, lm->bufs);
        k_lm_step<<<1, 1024, 0, ctx->stream>>>(lm->dims, lm->bufs, lm->opt);
        ctx->launches += 6;
        mark(1);
        if ((rc = ecb_cost_dev_eval(ctx, lm->bufs.cand, &s->go_cost, lm->d_cand_cost))) return rc;
        mark(2);
        if (lm->n_ranks > 1) {
            k_lm_epoch<<<1, 1, 0, ctx->stream>>>(&s->go_cost, &s->epoch_sc);
            ECB_LAUNCHED(ctx);
            if ((rc = ecb_cost_dev_scalar_exchange(ctx, &s->go_cost, lm->rank, lm->n_ranks, lm->recv, &s->epoch_sc, lm->d_cand_cost, &s->xerr)))
                return rc;
        }
        mark(3);
        k_lm_set_cost<<<1, 1, 0, ctx->stream>>>(lm->bufs, lm->d_cand_cost);
        k_lm_decide<<<1, 1, 0, ctx->stream>>>(lm->bufs, lm->opt);
        k_lm_commit<<<std::min(blocks, (int) ((lm->n_params + 255) / 256)), 256, 0, ctx->stream>>>(lm->bufs, lm->n_params);
        ctx->launches += 3;
        mark(4);
        if ((rc = lmdev_normal_eq(lm))) return rc;
        mark(5);
        k_lm_assemble<<<blocks, 256, 0, ctx->stream>>>(lm->dims, lm->bufs, &s->accepted, lm->const_intrinsics);
        k_lm_gradnorm<<<1, 1024, 0, ctx->stream>>>(lm->dims, lm->bufs, lm->opt, &s->accepted);
        ctx->launches += 2;
        mark(6);
    }
    return ecb_check(ctx, cudaGetLastError(), "device LM iteration");
}

// 1 while the state machine is still running (synchronises)
int ecb_lm_device_running(ecb_lm_device *lm) {
    if (!lm) return ECB_ERR_ARG;
    cudaSetDevice(lm->ctx->device);
    LmScalars h;
    const int rc = ecb_d2h(lm->ctx, &h, lm->bufs.s, sizeof h);
    if (rc) return rc;
    return h.running ? 1 : 0;
}

int ecb_lm_device_result(ecb_lm_device *lm, double *intrinsics, double *rot_cp, double *trans_cp, ecb_lm_summary *summary,
                         double *trace, int trace_rows) {
    if (!lm) return ECB_ERR_ARG;
    ecb_ctx *ctx = lm->ctx;
    cudaSetDevice(ctx->device);
    int rc;
    LmScalars h;
    if ((rc = ecb_d2h(ctx, &h, lm->bufs.s, sizeof h))) return rc;
    const size_t C = (size_t) lm->dims.C;
    std::vector<double> x(lm->n_params);
    if ((rc = ecb_d2h(ctx, x.data(), lm->bufs.x, lm->n_params * 8))) return rc;
    if (intrinsics) memcpy(intrinsics, x.data(), 72);
    if (rot_cp) memcpy(rot_cp, x.data() + 9, 32 * C);
    if (trans_cp) memcpy(trans_cp, x.data() + 9 + 4 * C, 24 * C);
    if (summary) {
        summary->iterations = h.iteration;
        summary->successful_steps = h.successful;
        summary->termination = (h.termination == ECB_LM_RUNNING && h.iteration >= lm->opt.max_iterations) ? ECB_LM_NO_CONVERGENCE : h.termination;
        summary->reserved = 0;
        summary->initial_cost = h.initial_cost;
        summary->final_cost = h.cost;
        summary->gradient_max_norm = h.gradient_max_norm;
        summary->radius = h.radius;
    }
    if (trace && trace_rows > 0) {
        const int rows = std::min(std::min(h.trace_rows, TRACE_CAP), trace_rows);
        if (rows > 0 && (rc = ecb_d2h(ctx, trace, lm->bufs.trace, (size_t) rows * 32))) return rc;
    }
    if (!lm->tev.empty()) {
        static const char *name[LM_TPH - 1] = {"solve", "candidate cost", "scalar exchange", "decide + commit", "normal equations", "assemble"};
        double sum[LM_TPH - 1] = {0};
        const bool each = atoi(getenv("ECB_LM_TIMING")) > 1;
        for (int it = 0; it < lm->t_iters; ++it) {
            if (each) fprintf(stderr, "[ecb lm timing] rank %d it %2d:", lm->rank, it);
            for (int k = 0; k + 1 < LM_TPH; ++k) {
                float ms = 0;
                cudaEventElapsedTime(&ms, lm->tev[(size_t) it * LM_TPH + k], lm->tev[(size_t) it * LM_TPH + k + 1]);
                sum[k] += ms;
                if (each) fprintf(stderr, " %.3f", ms);
            }
            if (each) fprintf(stderr, "\n");
        }
        fprintf(stderr, "[ecb lm timing] rank %d of %d, %d iterations, ms / iteration:", lm->rank, lm->n_ranks, lm->t_iters);
        for (int k = 0; k + 1 < LM_TPH; ++k) fprintf(stderr, " %s %.4f |", name[k], sum[k] / std::max(lm->t_iters, 1));
        fprintf(stderr, "\n");
        for (cudaEvent_t e : lm->tev) cudaEventDestroy(e);
        lm->tev.clear();
        lm->t_iters = 0;
    }
    if (h.xerr) return ecb_fail(ctx, ECB_ERR_STATE, "device LM: inter-GPU exchange timed out waiting for ranks (mask 0x%x)", h.xerr);
    return ECB_OK;
}

// the whole loop: begin, max_iterations iterations (enqueued in chunks; the state machine stops by itself), result
int ecb_calibrate_device(ecb_lm_device *lm, double *intrinsics, double *rot_cp, double *trans_cp, ecb_lm_summary *summary,
                         double *trace, int trace_rows) {
    if (!lm || !intrinsics || !rot_cp || !trans_cp) return ECB_ERR_ARG;
    int rc = ecb_lm_device_begin(lm, intrinsics, rot_cp, trans_cp);
    if (rc) return rc;
    const int total = lm->opt.max_iterations + 1;  // the extra pass lets the state machine report NO_CONVERGENCE itself
    const int chunk = lm->opt.fixed_iterations ? total : 8;
    for (int done = 0; done < total; done += chunk) {
        if ((rc = ecb_lm_device_iterate(lm, std::min(chunk, total - done)))) return rc;
        if (!lm->opt.fixed_iterations && done + chunk < total) {
            const int run = ecb_lm_device_running(lm);
            if (run < 0) return run;
            if (!run) break;
        }
    }
    return ecb_lm_device_result(lm, intrinsics, rot_cp, trans_cp, summary, trace, trace_rows);
}

}  // extern "C"

// ---- ecb_covariance ------------------------------------------------------------------------------------------------------------
// The workspace (the LM's factorisation buffers for this spline layout + the outputs) stays on the context between calls.
struct CovWork {
    std::vector<int32_t> n_cp;
    ecb_lm_device *lm = nullptr;
    DevBuf out;
    CovBufs c;
    // set when a call succeeds: the rotation model it differentiated in and ctx->spline_gen (ecb_pose_covariance reads Z and x)
    bool valid = false;
    int so3 = 0;
    uint64_t spline_gen = 0;
};

extern "C" void ecb_covariance_free(ecb_ctx *ctx) {
    if (!ctx || !ctx->cov) return;
    CovWork *w = (CovWork *) ctx->cov;
    ecb_lm_device_destroy(w->lm);
    if (w->out.p) cudaFree(w->out.p);
    delete w;
    ctx->cov = nullptr;
}

extern "C" int ecb_covariance(ecb_ctx *ctx, int n_splines, const int32_t *n_cp, const double *intrinsics, const double *rot_cp,
                              const double *trans_cp, const void *d_packed, int64_t n_residuals_total, double *cov_intrinsics,
                              double *cov_band, double *cov_cross, ecb_covariance_summary *summary) {
    if (!ctx || n_splines < 1 || !n_cp || !intrinsics || !rot_cp || !trans_cp || n_residuals_total < 0) return ECB_ERR_ARG;
    if (!ctx->cost) return ecb_fail(ctx, ECB_ERR_STATE, "ecb_cost_setup first");
    cudaSetDevice(ctx->device);
    int rc;
    std::vector<int32_t> key(n_cp, n_cp + n_splines);
    CovWork *w = (CovWork *) ctx->cov;
    if (!w || w->n_cp != key) {
        ecb_covariance_free(ctx);
        w = new CovWork();
        w->n_cp = key;
        if ((rc = ecb_lm_device_create(ctx, n_splines, n_cp, nullptr, &w->lm))) {
            delete w;
            return rc;
        }
        const size_t n = (size_t) w->lm->dims.n;
        const size_t cnt[6] = {n * NB, NI * n, NI * NI, NI * NI, NI * NI, 4};
        size_t total = 0;
        for (size_t k : cnt) total += k;
        if ((rc = ecb_reserve(ctx, w->out, total * 8))) {
            ecb_lm_device_destroy(w->lm);
            delete w;
            return rc;
        }
        double *p = (double *) w->out.p;
        double **dst[6] = {&w->c.Zb, &w->c.Zx, &w->c.Zc, &w->c.Zcs, &w->c.Lcc, &w->c.res};
        for (int k = 0; k < 6; ++k) *dst[k] = p, p += cnt[k];
        ctx->cov = w;
    }
    w->valid = false;
    ecb_lm_device *lm = w->lm;
    const LmDims &d = lm->dims;
    const size_t C = (size_t) d.C;
    LmBufs b = lm->bufs;
    b.Lcc = w->c.Lcc;
    if ((rc = ecb_h2d(ctx, b.x, intrinsics, 72))) return rc;
    if ((rc = ecb_h2d(ctx, b.x + 9, rot_cp, 32 * C))) return rc;
    if ((rc = ecb_h2d(ctx, b.x + 9 + 4 * C, trans_cp, 24 * C))) return rc;
    if (d_packed) {
        b.ne = (double *) d_packed;  // already summed over the ranks: every rank factorises the same system
    } else {
        ECB_CUDA(ctx, cudaMemsetAsync(b.ne, 0, (lm->ne_doubles + 2) * 8, ctx->stream));
        if ((rc = ecb_cost_dev_normal_eq(ctx, b.x, nullptr, b.ne))) return rc;
    }
    const int blocks = ctx->sm_count * 2;
    const uint32_t cmask = ctx->const_intrinsics;
    k_lm_assemble<<<blocks, 256, 0, ctx->stream>>>(d, b, nullptr, cmask);
    k_cov_begin<<<std::min(blocks, (d.D + 255) / 256), 256, 0, ctx->stream>>>(d, b, cmask);
    k_lm_build<<<blocks, 256, 0, ctx->stream>>>(d, b, lm->opt);
    k_lm_factor<<<d.n_seg, FACTOR_THREADS, 0, ctx->stream>>>(d, b);
    k_lm_corner<<<1, 32, 0, ctx->stream>>>(d, b);
    k_cov_pivots<<<1, 1024, 0, ctx->stream>>>(d, b, w->c);
    k_cov_corner<<<1, 96, 0, ctx->stream>>>(d, b, w->c, cmask);
    k_cov_selinv<<<d.n_seg, COV_THREADS, 0, ctx->stream>>>(d, b, w->c, cmask);
    ctx->launches += 8;
    if ((rc = ecb_check(ctx, cudaGetLastError(), "covariance kernels"))) return rc;
    double res[3];
    if ((rc = ecb_d2h(ctx, res, w->c.res, sizeof res))) return rc;
    int64_t m = n_residuals_total;
    if (m == 0 && (rc = ecb_cost_layout(ctx, nullptr, nullptr, &m, nullptr))) return rc;
    const int deficient = (int) res[2];
    const int dim = d.D - __builtin_popcount(cmask);  // free parameters
    if (summary) {
        summary->cost = res[0];
        summary->n_residuals = m;
        summary->dimension = dim;
        summary->sigma2 = m > dim ? 2.0 * res[0] / (double) (m - dim) : NAN;
        summary->min_relative_pivot = res[1];
        summary->deficient_index = deficient;
    }
    if (deficient >= 0)
        return ecb_fail(ctx, ECB_FAILED, "covariance: normal equations rank deficient at parameter %d (relative pivot <= %g)", deficient,
                        COV_MIN_PIVOT);
    if (cov_intrinsics && (rc = ecb_d2h(ctx, cov_intrinsics, w->c.Zc, NI * NI * 8))) return rc;
    if (cov_band && (rc = ecb_d2h(ctx, cov_band, w->c.Zb, (size_t) d.n * NB * 8))) return rc;
    if (cov_cross && (rc = ecb_d2h(ctx, cov_cross, w->c.Zx, (size_t) NI * d.n * 8))) return rc;
    EcbSplineView sv;
    if ((rc = ecb_cost_spline_view(ctx, &sv))) return rc;
    w->valid = true;
    w->so3 = sv.so3;
    w->spline_gen = ctx->spline_gen;
    return ECB_OK;
}

extern "C" int ecb_covariance_view(ecb_ctx *ctx, EcbCovView *v) {
    const CovWork *w = (const CovWork *) ctx->cov;
    if (!w || !w->valid) return ECB_ERR_STATE;
    v->Zb = w->c.Zb;
    v->x = w->lm->bufs.x;
    v->total_cp = w->lm->dims.C;
    v->so3 = w->so3;
    v->spline_gen = w->spline_gen;
    return ECB_OK;
}
