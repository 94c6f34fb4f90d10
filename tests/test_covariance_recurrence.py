"""CPU restatement of ecb_covariance: Jacobi-equilibrated band / arrow Cholesky factor and the selected inversion (Takahashi) on
band / arrow storage, checked against a dense inverse.  Pins the recurrence the GPU kernels (ecb_lmdev.cu: k_cov_corner,
k_cov_selinv) implement, both in the column-by-column form and in the blocked-by-control-point form the kernel runs.

Ordering: control point c owns tangent rows 6c .. 6c+5, the 9 intrinsics come last.  Band storage: Zb[j, r] = Z(j + r, j),
r = 0 .. 23, 0 past the end of a segment; cross Zx[a, j] = Z(intrinsic a, j); corner Zc (9 x 9)."""
import numpy as np
import pytest

import lm_oracle

NB, NI = 24, 9


def equilibrate(H):
    d = np.diag(H)
    s = np.where(d > 0, 1.0 / np.sqrt(np.where(d > 0, d, 1.0)), 1.0)
    return s, H * s[:, None] * s[None, :]


def band_arrow_factor(M, n):
    """Cholesky factor of M (band rows first, arrow last) in band / arrow storage; asserts that nothing falls outside it."""
    L = np.linalg.cholesky(M)
    Lb = np.zeros((n, NB))
    for r in range(NB):
        Lb[:n - r, r] = np.diag(L[:n, :n], -r)
    La = L[n:, :n].copy()
    Lc = L[n:, n:].copy()
    outside = np.tril(L[:n, :n], -NB)
    assert not outside.any(), "the factor has fill outside the band"
    return Lb, La, Lc


def selinv_columns(Lb, La, Lc, seg_rows):
    """The scalar recurrence: for j from a segment's last band row down to its first, N(j) = band rows j+1 .. j+23 of the
    segment + the 9 intrinsics,  Z_ij = -(1 / L_jj) sum_{k in N(j)} Z_ik L_kj,  Z_jj = 1 / L_jj^2 - (1 / L_jj) sum L_kj Z_kj."""
    n = Lb.shape[0]
    Wc = np.linalg.inv(Lc)
    Zc = Wc.T @ Wc
    Zb, Zx = np.zeros((n, NB)), np.zeros((NI, n))

    def z(i, k):  # Z on the stored pattern; i, k >= the current column
        if i >= n and k >= n:
            return Zc[i - n, k - n]
        if i >= n:
            return Zx[i - n, k]
        if k >= n:
            return Zx[k - n, i]
        lo, hi = min(i, k), max(i, k)
        assert hi - lo < NB
        return Zb[lo, hi - lo]

    for j0, j1 in seg_rows:
        for j in range(j1 - 1, j0 - 1, -1):
            N = list(range(j + 1, min(j + NB, j1))) + [n + a for a in range(NI)]
            l = np.array([Lb[j, k - j] if k < n else La[k - n, j] for k in N])
            ZN = np.array([[z(i, k) for k in N] for i in N])
            y = -(ZN @ l) / Lb[j, 0]
            for i, v in zip(N, y):
                if i < n:
                    Zb[j, i - j] = v
                else:
                    Zx[i - n, j] = v
            Zb[j, 0] = 1.0 / Lb[j, 0] ** 2 - (l @ y) / Lb[j, 0]
    return Zb, Zx, Zc


def selinv_blocked(Lb, La, Lc, seg_rows):
    """k_cov_selinv's form: per control point block B (6 columns), K = the next 18 band rows + the intrinsics, R = the next 23
    band rows + the intrinsics,  T = L_KB L_BB^-1,  Z_RB = -Z_RK T,  Z_BB = L_BB^-T L_BB^-1 - Z_KB^T T, over a sliding
    32 x 32 window of Z."""
    n = Lb.shape[0]
    Wc = np.linalg.inv(Lc)
    Zc = Wc.T @ Wc
    Zb, Zx = np.zeros((n, NB)), np.zeros((NI, n))
    kidx = list(range(18)) + list(range(23, 32))
    for j0s, j1s in seg_rows:
        ns = j1s - j0s
        win = np.zeros((32, 32))
        win[23:, 23:] = Zc
        for j0 in range(ns - 6, -1, -6):
            g0 = j0s + j0
            LB = np.zeros((6, 6))
            for r in range(6):
                for k in range(r + 1):
                    LB[r, k] = Lb[g0 + k, r - k]
            LK = np.zeros((27, 6))
            for q in range(18):
                if j0 + 6 + q < ns:
                    for k in range(6):
                        LK[q, k] = Lb[g0 + k, 6 + q - k]
            LK[18:] = La[:, g0:g0 + 6]
            WB = np.linalg.inv(LB)
            T = LK @ WB
            Y = -win[:, kidx] @ T
            ZB = WB.T @ WB - Y[kidx].T @ T
            for k in range(6):
                for r in range(NB):
                    i = j0 + k + r
                    if i < ns:
                        Zb[g0 + k, r] = ZB[i - j0, k] if i < j0 + 6 else Y[i - j0 - 6, k]
            Zx[:, g0:g0 + 6] = Y[23:]
            nw = np.zeros((32, 32))
            old = list(range(17)) + list(range(23, 32))
            new = list(range(6, 23)) + list(range(23, 32))
            nw[:6, :6] = ZB
            nw[np.ix_(new, list(range(6)))] = Y[old]
            nw[np.ix_(list(range(6)), new)] = Y[old].T
            nw[np.ix_(new, new)] = win[np.ix_(old, old)]
            win = nw
    return Zb, Zx, Zc


def covariance(H, n_cp):
    """Z = S (S H S)^-1 S on the band / arrow pattern (unscaled), via the factor and the selected inversion."""
    n = 6 * int(sum(n_cp))
    s, M = equilibrate(H)
    Lb, La, Lc = band_arrow_factor(M, n)
    seg = np.cumsum([0] + [6 * c for c in n_cp])
    rows = list(zip(seg[:-1], seg[1:]))
    out = []
    for fn in (selinv_columns, selinv_blocked):
        Zb, Zx, Zc = fn(Lb, La, Lc, rows)
        out.append((Zb * s[:n, None] * np.array([[s[j + r] if j + r < n else 0.0 for r in range(NB)] for j in range(n)]),
                    Zx * s[n:, None] * s[None, :n], Zc * s[n:, None] * s[None, n:]))
    return out, s, M


def dense_pattern(Z, n_cp):
    """the band / cross / corner entries of a dense Z, band entries across segments set to 0"""
    n = 6 * int(sum(n_cp))
    seg_of = np.repeat(np.arange(len(n_cp)), [6 * c for c in n_cp])
    Zb = np.zeros((n, NB))
    for j in range(n):
        for r in range(NB):
            if j + r < n and seg_of[j + r] == seg_of[j]:
                Zb[j, r] = Z[j + r, j]
    return Zb, Z[n:, :n], Z[n:, n:]


def random_problem(n_cp, rng, rows_per_span=40):
    """H = J^T J of random span blocks (4 consecutive control points + the intrinsics), columns scaled over 8 decades"""
    n = 6 * sum(n_cp)
    D = n + NI
    colscale = 10.0 ** rng.uniform(-4, 4, D)
    H = np.zeros((D, D))
    co = 0
    for c in n_cp:
        for s in range(c - 3):
            idx = np.r_[6 * (co + s): 6 * (co + s + 4), n:D]
            J = rng.standard_normal((rows_per_span, len(idx))) * colscale[idx]
            H[np.ix_(idx, idx)] += J.T @ J
        co += c
    return H


def check(H, n_cp, rtol=1e-10):
    (cols, blocked), s, M = covariance(H, n_cp)
    Z = np.linalg.inv(H)
    ref = dense_pattern(Z, n_cp)
    for got in (cols, blocked):
        for g, r, name in zip(got, ref, ("band", "cross", "corner")):
            # compare in the scaled space, where the entries are O(1 / smallest eigenvalue of M)
            if name == "band":
                n = g.shape[0]
                sr = np.array([[s[j + q] if j + q < n else 1.0 for q in range(NB)] for j in range(n)])
                gs, rs = g / (s[:n, None] * sr), r / (s[:n, None] * sr)
            elif name == "cross":
                gs, rs = g / (s[-NI:, None] * s[None, :-NI]), r / (s[-NI:, None] * s[None, :-NI])
            else:
                gs, rs = g / (s[-NI:, None] * s[None, -NI:]), r / (s[-NI:, None] * s[None, -NI:])
            assert np.abs(gs - rs).max() <= rtol * np.abs(rs).max(), name
    return cols, blocked, M


@pytest.mark.parametrize("n_cp", [[4], [9], [7, 5], [6, 4, 8]])
def test_selected_inverse_matches_dense_inverse(n_cp):
    rng = np.random.default_rng(sum(n_cp) * 7 + len(n_cp))
    H = random_problem(n_cp, rng)
    cols, blocked, M = check(H, n_cp)
    # the two forms of the recurrence agree with each other to round-off, and band entries across segments are 0
    for a, b in zip(cols, blocked):
        assert np.abs(a - b).max() <= 1e-9 * np.abs(a).max()
    n0 = 6 * n_cp[0]
    if len(n_cp) > 1:
        for j in range(n0 - NB + 1, n0):
            assert not cols[0][j, n0 - j:].any() and not blocked[0][j, n0 - j:].any()
    assert np.allclose(np.diag(M), 1.0)


def test_zero_column_is_rank_deficient():
    """a control point without residuals: zero diagonal, scale 1, the pivot of its first row is exactly 0"""
    rng = np.random.default_rng(5)
    n_cp = [12]
    H = random_problem(n_cp, rng)
    c = 6
    H[6 * c:6 * c + 6, :] = 0
    H[:, 6 * c:6 * c + 6] = 0
    s, M = equilibrate(H)
    assert np.all(s[6 * c:6 * c + 6] == 1.0) and M[6 * c, 6 * c] == 0.0
    with pytest.raises(np.linalg.LinAlgError):
        np.linalg.cholesky(M)


def test_oracle_normal_equations_at_the_converged_point(oracle_mod):
    """the first problem of test_gpu_calibrate.py at the point the reference LM loop converges to (function tolerance):
    cond(S H S) ~ 1e7 while cond(H) ~ 1e15, the recurrence still matches the dense inverse"""
    from eventcalib_b200 import synth, calib_problem
    ev = synth.make_stream(150000, 346, 260, t0=5.0, duration=0.6, seed=1004, return_truth=True, rot_amp=(0.35, 0.35, 0.25),
                           dist=92.0)
    pb = calib_problem.build(ev, seed=2, intr_noise=0.02)
    P = oracle_mod.CostProblem([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"])
    P.associate(ev["t"], ev["x"], ev["y"], pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
    i, r, t, _, term = lm_oracle.solve(P, [pb["n_cp"]], pb["intrinsics"], pb["rot_cp"], pb["trans_cp"], max_iterations=50)
    cost, Hs, gs = P.normal_eq(i, r, t)
    maps, C = lm_oracle._index_map([pb["n_cp"]])
    D = 9 + 6 * C
    A, _ = lm_oracle.assemble(Hs, gs, maps, D)
    # lm_oracle orders the intrinsics first; ecb_covariance orders them last
    perm = np.r_[9:D, 0:9]
    H = A[np.ix_(perm, perm)]
    _, M = equilibrate(H)
    assert np.linalg.cond(M) < 1e8 < np.linalg.cond(H)
    cols, _, _ = check(H, [pb["n_cp"]], rtol=1e-8)
    sigma2 = 2 * cost / (P.n_residuals - D)
    std = np.sqrt(sigma2 * np.diag(cols[2]))
    # the distortion terms are the weakly determined ones: k5's deviation is orders of magnitude above fx's
    assert std[8] > 100 * std[0] > 0
