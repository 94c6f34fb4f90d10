// Host-side Levenberg-Marquardt step around the GPU normal equations (EventCalibSpline::optimize,
// event_camera_calib/src/EventCalibSpline.cpp:197-247: HuberLoss, EigenQuaternionParameterization on every rotation
// control point, SPARSE_NORMAL_CHOLESKY, function/gradient tolerance 1e-10, Ceres defaults otherwise).
//
// The trust-region logic restates Ceres 1.x's TrustRegionMinimizer + LevenbergMarquardtStrategy
// [external — Ceres is NOT in /root/reference; SURVEY.md Appendix C]: Jacobi column scaling 1/(1+||J_col||) from the
// first Jacobian, D^2 = clamp(diag(J^T J), 1e-6, 1e32) / radius, step from (J^T J + D^2) y = J^T r, step = -y,
// model_cost_change = -(J d).(r + J d / 2), accept iff rho > 1e-3, radius /= max(1/3, 1 - (2 rho - 1)^3) on success,
// radius /= 2, 4, 8 ... on failure.  Everything is computed from the packed J^T J / J^T r the GPU returns, so the
// Jacobian itself never leaves the device.
//
// Linear algebra: the tangent-space system is a block band (half bandwidth 23: a residual touches 4 consecutive control
// points x 6) bordered by the 9 dense intrinsics rows -> banded Cholesky + 9x9 Schur complement, O(D * 33^2) per solve.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "ecb_common.cuh"
#include "ecb_so3.h"

namespace {

constexpr int BW = 23;          // half bandwidth of the control-point block band
constexpr int NI = 9;           // intrinsics
constexpr int OUT_STRIDE = 33 * 33 + 33;

struct BandArrow {              // symmetric [[B, A^T], [A, C]]: B n x n banded (lower), A 9 x n, C 9 x 9
    int n = 0;
    std::vector<double> B, A, C;
    void resize(int n_) {
        n = n_;
        B.assign((size_t) n * (BW + 1), 0.0);
        A.assign((size_t) NI * n, 0.0);
        C.assign(NI * NI, 0.0);
    }
    void zero() {
        std::fill(B.begin(), B.end(), 0.0);
        std::fill(A.begin(), A.end(), 0.0);
        std::fill(C.begin(), C.end(), 0.0);
    }
    double &b(int i, int j) { return B[(size_t) i * (BW + 1) + (i - j)]; }  // i >= j, i - j <= BW
    double get(int i, int j) const {                                          // full symmetric accessor, D = n + 9
        if (i < j) std::swap(i, j);
        if (i < n) return (i - j <= BW) ? B[(size_t) i * (BW + 1) + (i - j)] : 0.0;
        if (j < n) return A[(size_t) (i - n) * n + j];
        return C[(i - n) * NI + (j - n)];
    }
    void add(int i, int j, double v) {  // i >= j
        if (i < n) b(i, j) += v;
        else if (j < n) A[(size_t) (i - n) * n + j] += v;
        else C[(i - n) * NI + (j - n)] += v;
    }
    // y = M x
    void mul(const double *x, double *y) const {
        const int D = n + NI;
        for (int i = 0; i < D; ++i) y[i] = 0.0;
        for (int i = 0; i < n; ++i)
            for (int d = 0; d <= BW && d <= i; ++d) {
                const double v = B[(size_t) i * (BW + 1) + d];
                y[i] += v * x[i - d];
                if (d) y[i - d] += v * x[i];
            }
        for (int r = 0; r < NI; ++r) {
            double s = 0.0;
            for (int j = 0; j < n; ++j) {
                const double v = A[(size_t) r * n + j];
                s += v * x[j];
                y[j] += v * x[n + r];
            }
            for (int c = 0; c < NI; ++c) s += C[std::max(r, c) * NI + std::min(r, c)] * x[n + c];  // only the lower triangle is stored
            y[n + r] += s;
        }
    }
};

// in-place Cholesky of a BandArrow and solve; returns false if not positive definite
struct BandArrowChol {
    BandArrow L;
    bool factor(const BandArrow &M) {
        L = M;
        const int n = L.n;
        for (int i = 0; i < n; ++i) {
            const int j0 = std::max(0, i - BW);
            for (int j = j0; j <= i; ++j) {
                double s = L.b(i, j);
                const int k0 = std::max(j0, std::max(0, j - BW));
                for (int k = k0; k < j; ++k) s -= L.b(i, k) * L.b(j, k);
                if (i == j) {
                    if (!(s > 0.0)) return false;
                    L.b(i, i) = sqrt(s);
                } else {
                    L.b(i, j) = s / L.b(j, j);
                }
            }
        }
        // Y = A L^-T  (rows of A): forward substitution per row
        for (int r = 0; r < NI; ++r) {
            double *y = &L.A[(size_t) r * n];
            for (int j = 0; j < n; ++j) {
                double s = y[j];
                for (int k = std::max(0, j - BW); k < j; ++k) s -= y[k] * L.b(j, k);
                y[j] = s / L.b(j, j);
            }
        }
        // S = C - Y Y^T, dense Cholesky
        for (int r = 0; r < NI; ++r)
            for (int c = 0; c <= r; ++c) {
                double s = L.C[r * NI + c];
                const double *yr = &L.A[(size_t) r * n], *yc = &L.A[(size_t) c * n];
                for (int j = 0; j < n; ++j) s -= yr[j] * yc[j];
                for (int k = 0; k < c; ++k) s -= L.C[r * NI + k] * L.C[c * NI + k];
                if (r == c) {
                    if (!(s > 0.0)) return false;
                    L.C[r * NI + r] = sqrt(s);
                } else {
                    L.C[r * NI + c] = s / L.C[c * NI + c];
                }
            }
        return true;
    }
    void solve(const double *b, double *x) const {
        const int n = L.n;
        std::vector<double> z(n + NI);
        for (int i = 0; i < n; ++i) {
            double s = b[i];
            for (int k = std::max(0, i - BW); k < i; ++k) s -= L.B[(size_t) i * (BW + 1) + (i - k)] * z[k];
            z[i] = s / L.B[(size_t) i * (BW + 1)];
        }
        for (int r = 0; r < NI; ++r) {
            double s = b[n + r];
            const double *y = &L.A[(size_t) r * n];
            for (int j = 0; j < n; ++j) s -= y[j] * z[j];
            for (int k = 0; k < r; ++k) s -= L.C[r * NI + k] * z[n + k];
            z[n + r] = s / L.C[r * NI + r];
        }
        for (int r = NI - 1; r >= 0; --r) {
            double s = z[n + r];
            for (int k = r + 1; k < NI; ++k) s -= L.C[k * NI + r] * x[n + k];
            x[n + r] = s / L.C[r * NI + r];
        }
        for (int i = 0; i < n; ++i)
            for (int r = 0; r < NI; ++r) z[i] -= L.A[(size_t) r * n + i] * x[n + r];
        for (int i = n - 1; i >= 0; --i) {
            double s = z[i];
            for (int k = i + 1; k <= std::min(n - 1, i + BW); ++k) s -= L.B[(size_t) k * (BW + 1) + (k - i)] * x[k];
            x[i] = s / L.B[(size_t) i * (BW + 1)];
        }
    }
};

void quat_plus(const double *x, const double *d, double *out) {  // EigenQuaternionParameterization::Plus [external: Ceres]
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

}  // namespace

struct ecb_lm {
    ecb_lm_options opt;
    int n_splines = 0, C = 0, n_spans = 0, D = 0;
    std::vector<int> span_cp0;      // first control point of every global span
    std::vector<double> intr, rot, trans;          // current x
    std::vector<double> c_intr, c_rot, c_trans;    // candidate
    BandArrow H;                    // J^T J at x (unscaled)
    std::vector<double> g;          // J^T r at x (unscaled), internal order
    std::vector<double> scale, diag, step, delta;
    double cost = 0, radius = 0, decrease_factor = 2, model_cost_change = 0, candidate_cost = 0;
    bool have_scale = false, reuse_diagonal = false, begun = false;
    uint32_t const_mask = 0;        // constant intrinsics (ecb_lm_set_constant_intrinsics)
    int iteration = 0, successful = 0, termination = ECB_LM_RUNNING, invalid_steps = 0;
    double gradient_max_norm = 0, step_norm = 0, x_norm = 0;
    std::vector<double> trace;
    BandArrowChol chol;

    int gidx(int cp, int k) const { return 6 * cp + k; }
    void plus(const double *d, std::vector<double> &oi, std::vector<double> &orot, std::vector<double> &otr) const {
        oi.resize(9);
        orot.resize(4 * (size_t) C);
        otr.resize(3 * (size_t) C);
        for (int i = 0; i < 9; ++i) oi[i] = intr[i] + d[6 * C + i];
        for (int c = 0; c < C; ++c) {
            if (opt.rotation_model == 1) ecb_so3::plus(&rot[4 * c], &d[6 * c], &orot[4 * c]);  // LocalParameterizationSO3::Plus
            else quat_plus(&rot[4 * c], &d[6 * c], &orot[4 * c]);
            for (int k = 0; k < 3; ++k) otr[3 * c + k] = trans[3 * c + k] + d[6 * c + 3 + k];
        }
    }
    void assemble(const double *packed) {
        H.zero();
        std::fill(g.begin(), g.end(), 0.0);
        int map[33];
        for (int s = 0; s < n_spans; ++s) {
            const int cp0 = span_cp0[s];
            for (int l = 0; l < 9; ++l) map[l] = 6 * C + l;
            for (int j = 0; j < 4; ++j)
                for (int k = 0; k < 3; ++k) {
                    map[9 + 3 * j + k] = 6 * (cp0 + j) + k;
                    map[21 + 3 * j + k] = 6 * (cp0 + j) + 3 + k;
                }
            const double *B = packed + (size_t) s * OUT_STRIDE, *gs = B + 1089;
            for (int a = 0; a < 33; ++a) {
                g[map[a]] += gs[a];
                for (int b = 0; b < 33; ++b) {
                    const int i = map[a], j = map[b];
                    if (i >= j) H.add(i, j, B[a * 33 + b]);
                }
            }
        }
        if (const_mask) {  // constant intrinsics: their rows / columns of J^T J and entries of J^T r become exact zeros
            const int n = H.n;
            for (int r = 0; r < NI; ++r) {
                for (int j = 0; j < n; ++j) H.A[(size_t) r * n + j] = ecb_zero_constant(const_mask, r, -1, H.A[(size_t) r * n + j]);
                for (int c = 0; c < NI; ++c) H.C[r * NI + c] = ecb_zero_constant(const_mask, r, c, H.C[r * NI + c]);
                g[n + r] = ecb_zero_constant(const_mask, r, -1, g[n + r]);
            }
        }
        cost = packed[(size_t) n_spans * OUT_STRIDE];
    }
    void gradient_norms() {
        // max |x - Plus(x, -g)| over the ambient parameters (Ceres projected gradient)
        std::vector<double> ng(D), pi, pr, pt;
        for (int i = 0; i < D; ++i) ng[i] = -g[i];
        plus(ng.data(), pi, pr, pt);
        double m = 0;
        for (int i = 0; i < 9; ++i) m = std::max(m, fabs(intr[i] - pi[i]));
        for (size_t i = 0; i < rot.size(); ++i) m = std::max(m, fabs(rot[i] - pr[i]));
        for (size_t i = 0; i < trans.size(); ++i) m = std::max(m, fabs(trans[i] - pt[i]));
        gradient_max_norm = m;
    }
    void record(double accepted) {
        trace.push_back(cost);
        trace.push_back(gradient_max_norm);
        trace.push_back(radius);
        trace.push_back(accepted);
    }
};

extern "C" {

void ecb_lm_default_options(ecb_lm_options *o) {
    if (!o) return;
    o->max_iterations = 50;
    o->function_tolerance = 1e-10;   // EventCalibSpline.cpp:239-240 (Sophus epsilon)
    o->gradient_tolerance = 1e-10;
    o->parameter_tolerance = 1e-8;
    o->initial_radius = 1e4;
    o->max_radius = 1e16;
    o->min_radius = 1e-32;
    o->min_relative_decrease = 1e-3;
    o->min_lm_diagonal = 1e-6;
    o->max_lm_diagonal = 1e32;
    o->jacobi_scaling = 1;
    o->fixed_iterations = 0;
    o->rotation_model = 0;
}

ecb_lm *ecb_lm_create(int n_splines, const int32_t *n_cp, const ecb_lm_options *opt) {
    if (n_splines < 1 || !n_cp) return nullptr;
    ecb_lm *lm = new ecb_lm();
    if (opt) lm->opt = *opt; else ecb_lm_default_options(&lm->opt);
    lm->n_splines = n_splines;
    int co = 0;
    for (int s = 0; s < n_splines; ++s) {
        for (int k = 0; k < n_cp[s] - 3; ++k) lm->span_cp0.push_back(co + k);
        co += n_cp[s];
    }
    lm->C = co;
    lm->n_spans = (int) lm->span_cp0.size();
    lm->D = 6 * co + 9;
    lm->H.resize(6 * co);
    lm->g.assign(lm->D, 0.0);
    lm->scale.assign(lm->D, 1.0);
    lm->diag.assign(lm->D, 0.0);
    lm->step.assign(lm->D, 0.0);
    lm->delta.assign(lm->D, 0.0);
    lm->radius = lm->opt.initial_radius;
    return lm;
}

void ecb_lm_destroy(ecb_lm *lm) { delete lm; }

int ecb_lm_dimension(const ecb_lm *lm) { return lm ? lm->D : 0; }

// intrinsics held at their start values (bit i = intrinsic i); before ecb_lm_begin only
int ecb_lm_set_constant_intrinsics(ecb_lm *lm, uint32_t mask) {
    if (!lm || mask > ECB_ALL_INTRINSICS) return ECB_ERR_ARG;
    if (lm->begun) return ECB_ERR_STATE;
    lm->const_mask = mask;
    return ECB_OK;
}

// first evaluation at x (iteration 0)
int ecb_lm_begin(ecb_lm *lm, const double *intr, const double *rot, const double *trans, const double *packed) {
    if (!lm || !intr || !rot || !trans || !packed) return ECB_ERR_ARG;
    lm->intr.assign(intr, intr + 9);
    lm->rot.assign(rot, rot + 4 * (size_t) lm->C);
    lm->trans.assign(trans, trans + 3 * (size_t) lm->C);
    lm->begun = true;
    lm->assemble(packed);
    lm->iteration = 0;
    lm->successful = 0;
    lm->radius = lm->opt.initial_radius;
    lm->decrease_factor = 2.0;
    lm->reuse_diagonal = false;
    lm->termination = ECB_LM_RUNNING;
    lm->trace.clear();
    if (lm->opt.jacobi_scaling)
        for (int i = 0; i < lm->D; ++i) lm->scale[i] = 1.0 / (1.0 + sqrt(lm->H.get(i, i)));
    else
        std::fill(lm->scale.begin(), lm->scale.end(), 1.0);
    lm->gradient_norms();
    lm->record(1.0);
    if (!lm->opt.fixed_iterations && lm->gradient_max_norm <= lm->opt.gradient_tolerance) lm->termination = ECB_LM_GRADIENT_TOLERANCE;
    return lm->termination;
}

// Solves for the trust-region step at the current x and writes the candidate parameters.
// Returns ECB_LM_RUNNING (evaluate the candidate's cost, then ecb_lm_feedback) or a termination code.
int ecb_lm_propose(ecb_lm *lm, double *c_intr, double *c_rot, double *c_trans) {
    if (!lm) return ECB_ERR_ARG;
    if (lm->termination != ECB_LM_RUNNING) return lm->termination;
    for (;;) {
        if (lm->iteration >= lm->opt.max_iterations) return lm->termination = ECB_LM_NO_CONVERGENCE;
        ++lm->iteration;
        const int D = lm->D;
        // scaled system: Hs = S H S, gs = S g;  diagonal D^2 = clamp(diag(Hs)) / radius
        if (!lm->reuse_diagonal)
            for (int i = 0; i < D; ++i) {
                const double d = lm->H.get(i, i) * lm->scale[i] * lm->scale[i];
                lm->diag[i] = std::min(std::max(d, lm->opt.min_lm_diagonal), lm->opt.max_lm_diagonal);
            }
        BandArrow M = lm->H;
        const int n = M.n;
        for (int i = 0; i < n; ++i)
            for (int d = 0; d <= BW && d <= i; ++d) M.B[(size_t) i * (BW + 1) + d] *= lm->scale[i] * lm->scale[i - d];
        for (int r = 0; r < NI; ++r) {
            for (int j = 0; j < n; ++j) M.A[(size_t) r * n + j] *= lm->scale[n + r] * lm->scale[j];
            for (int c = 0; c < NI; ++c) M.C[r * NI + c] *= lm->scale[n + r] * lm->scale[n + c];
        }
        BandArrow Hs = M;
        for (int i = 0; i < n; ++i) M.B[(size_t) i * (BW + 1)] += lm->diag[i] / lm->radius;
        for (int r = 0; r < NI; ++r) M.C[r * NI + r] += lm->diag[n + r] / lm->radius;
        std::vector<double> gs(D), y(D), Hd(D);
        for (int i = 0; i < D; ++i) gs[i] = lm->g[i] * lm->scale[i];
        bool ok = lm->chol.factor(M);
        if (ok) {
            lm->chol.solve(gs.data(), y.data());
            for (int i = 0; i < D; ++i) lm->step[i] = -y[i];
            Hs.mul(lm->step.data(), Hd.data());
            double a = 0, b = 0;
            for (int i = 0; i < D; ++i) {
                a += lm->step[i] * gs[i];
                b += lm->step[i] * Hd[i];
            }
            lm->model_cost_change = -(a + 0.5 * b);
            ok = lm->model_cost_change > 0.0 && std::isfinite(lm->model_cost_change);
        }
        if (!ok) {  // invalid step: shrink the region and try again (Ceres: HandleInvalidStep)
            if (++lm->invalid_steps > 5) return lm->termination = ECB_LM_FAILURE;
            lm->radius /= lm->decrease_factor;
            lm->decrease_factor *= 2.0;
            lm->reuse_diagonal = true;
            lm->record(-1.0);
            continue;
        }
        lm->invalid_steps = 0;
        for (int i = 0; i < D; ++i) lm->delta[i] = lm->step[i] * lm->scale[i];
        lm->plus(lm->delta.data(), lm->c_intr, lm->c_rot, lm->c_trans);
        memcpy(c_intr, lm->c_intr.data(), 72);
        memcpy(c_rot, lm->c_rot.data(), lm->c_rot.size() * 8);
        memcpy(c_trans, lm->c_trans.data(), lm->c_trans.size() * 8);
        double xn = 0, sn = 0;
        for (int i = 0; i < 9; ++i) {
            xn += lm->intr[i] * lm->intr[i];
            sn += (lm->intr[i] - lm->c_intr[i]) * (lm->intr[i] - lm->c_intr[i]);
        }
        for (size_t i = 0; i < lm->rot.size(); ++i) {
            xn += lm->rot[i] * lm->rot[i];
            sn += (lm->rot[i] - lm->c_rot[i]) * (lm->rot[i] - lm->c_rot[i]);
        }
        for (size_t i = 0; i < lm->trans.size(); ++i) {
            xn += lm->trans[i] * lm->trans[i];
            sn += (lm->trans[i] - lm->c_trans[i]) * (lm->trans[i] - lm->c_trans[i]);
        }
        lm->x_norm = sqrt(xn);
        lm->step_norm = sqrt(sn);
        return ECB_LM_RUNNING;
    }
}

// candidate_cost evaluated at the proposed parameters.  Returns 1: step accepted (x moved; evaluate the normal
// equations at the new x and call ecb_lm_update), 0: rejected (call ecb_lm_propose again), >= 2: terminated.
int ecb_lm_feedback(ecb_lm *lm, double candidate_cost) {
    if (!lm) return ECB_ERR_ARG;
    if (lm->termination != ECB_LM_RUNNING) return lm->termination;
    lm->candidate_cost = candidate_cost;
    if (!lm->opt.fixed_iterations) {
        if (lm->step_norm <= lm->opt.parameter_tolerance * (lm->x_norm + lm->opt.parameter_tolerance))
            return lm->termination = ECB_LM_PARAMETER_TOLERANCE;
        if (fabs(lm->cost - candidate_cost) <= lm->opt.function_tolerance * lm->cost)
            return lm->termination = ECB_LM_FUNCTION_TOLERANCE;
    }
    const double rho = (lm->cost - candidate_cost) / lm->model_cost_change;
    if (rho > lm->opt.min_relative_decrease) {
        lm->intr = lm->c_intr;
        lm->rot = lm->c_rot;
        lm->trans = lm->c_trans;
        ++lm->successful;
        lm->radius = lm->radius / std::max(1.0 / 3.0, 1.0 - pow(2.0 * rho - 1.0, 3));
        lm->radius = std::min(lm->opt.max_radius, lm->radius);
        lm->decrease_factor = 2.0;
        lm->reuse_diagonal = false;
        return 1;
    }
    lm->radius /= lm->decrease_factor;
    lm->decrease_factor *= 2.0;
    lm->reuse_diagonal = true;
    lm->record(0.0);
    if (lm->radius < lm->opt.min_radius) {
        if (!lm->opt.fixed_iterations) return lm->termination = ECB_LM_MIN_RADIUS;
        lm->radius = lm->opt.min_radius;  // benchmark mode (config C4): exactly max_iterations iterations, no early exit
    }
    return 0;
}

// normal equations at the accepted x
int ecb_lm_update(ecb_lm *lm, const double *packed) {
    if (!lm || !packed) return ECB_ERR_ARG;
    lm->assemble(packed);
    lm->gradient_norms();
    lm->record(1.0);
    if (!lm->opt.fixed_iterations && lm->gradient_max_norm <= lm->opt.gradient_tolerance)
        return lm->termination = ECB_LM_GRADIENT_TOLERANCE;
    return lm->termination;
}

int ecb_lm_state(const ecb_lm *lm, double *intr, double *rot, double *trans, ecb_lm_summary *sum) {
    if (!lm) return ECB_ERR_ARG;
    if (intr) memcpy(intr, lm->intr.data(), 72);
    if (rot) memcpy(rot, lm->rot.data(), lm->rot.size() * 8);
    if (trans) memcpy(trans, lm->trans.data(), lm->trans.size() * 8);
    if (sum) {
        sum->iterations = lm->iteration;
        sum->successful_steps = lm->successful;
        sum->termination = lm->termination;
        sum->final_cost = lm->cost;
        sum->initial_cost = lm->trace.empty() ? lm->cost : lm->trace[0];
        sum->gradient_max_norm = lm->gradient_max_norm;
        sum->radius = lm->radius;
    }
    return ECB_OK;
}

// per recorded evaluation: cost, gradient_max_norm, radius, accepted(1)/rejected(0)/invalid(-1)
int ecb_lm_trace(const ecb_lm *lm, double *out, int cap_rows) {
    if (!lm) return 0;
    const int rows = std::min((int) (lm->trace.size() / 4), cap_rows);
    if (out) memcpy(out, lm->trace.data(), (size_t) rows * 32);
    return rows;
}

int ecb_cost_layout(ecb_ctx *ctx, int32_t *total_cp, int32_t *total_spans, int64_t *n_residuals, int64_t *out_doubles);
int ecb_cost_eval(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, double *cost);
int ecb_cost_normal_eq(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, void *d_out,
                       double *h_out, double *cost);

// Single-GPU driver: the whole optimize() loop (GPU evaluations through ctx, host solve).  n_cp as given to ecb_cost_setup.
int ecb_calibrate(ecb_ctx *ctx, int n_splines, const int32_t *n_cp, double *intrinsics, double *rot_cp, double *trans_cp,
                  const ecb_lm_options *opt, ecb_lm_summary *summary, double *trace, int trace_rows) {
    if (!ctx || !intrinsics || !rot_cp || !trans_cp) return ECB_ERR_ARG;
    int64_t nd = 0;
    int32_t tcp = 0;
    int rc = ecb_cost_layout(ctx, &tcp, nullptr, nullptr, &nd);
    if (rc) return rc;
    ecb_lm *lm = ecb_lm_create(n_splines, n_cp, opt);
    if (!lm || lm->C != tcp) {
        ecb_lm_destroy(lm);
        return ecb_fail(ctx, ECB_ERR_ARG, "spline layout differs from ecb_cost_setup");
    }
    ecb_lm_set_constant_intrinsics(lm, ctx->const_intrinsics);
    std::vector<double> packed((size_t) nd), ci(9), cr(4 * (size_t) tcp), ct(3 * (size_t) tcp);
    rc = ecb_cost_normal_eq(ctx, intrinsics, rot_cp, trans_cp, nullptr, packed.data(), nullptr);
    int st = rc ? rc : ecb_lm_begin(lm, intrinsics, rot_cp, trans_cp, packed.data());
    while (st == ECB_LM_RUNNING) {
        st = ecb_lm_propose(lm, ci.data(), cr.data(), ct.data());
        if (st != ECB_LM_RUNNING) break;
        double cc = 0;
        if ((rc = ecb_cost_eval(ctx, ci.data(), cr.data(), ct.data(), &cc))) {
            st = rc;
            break;
        }
        const int fb = ecb_lm_feedback(lm, cc);
        if (fb == 1) {
            if ((rc = ecb_cost_normal_eq(ctx, ci.data(), cr.data(), ct.data(), nullptr, packed.data(), nullptr))) {
                st = rc;
                break;
            }
            st = ecb_lm_update(lm, packed.data());
        } else if (fb == 0) {
            st = ECB_LM_RUNNING;
        } else {
            st = fb;
        }
    }
    ecb_lm_state(lm, intrinsics, rot_cp, trans_cp, summary);
    if (trace) ecb_lm_trace(lm, trace, trace_rows);
    ecb_lm_destroy(lm);
    return st < 0 ? st : ECB_OK;
}

}  // extern "C"
