"""CPU tests of constant intrinsics in the host LM state machine (ecb_lm_set_constant_intrinsics, eventcalib_b200/csrc/ecb_lm.cu),
driven by the oracle's normal equations like tests/test_lm_host.py.  The reference is solve_reduced below: the dense loop of
tests/lm_oracle.py on the REDUCED problem (the rows and columns of the constant intrinsics deleted from A and b, the step
scattered back with zeros, |x| of the full ambient vector), i.e. what Ceres does with a SubsetManifold on the intrinsics block."""
import numpy as np
import pytest

import lm_oracle

MASKS = {"k3 k4 k5": 0b111000000, "cx cy": 0b000001100, "all nine": 0b111111111}


def solve_reduced(P, n_cp_list, intr, rot, trans, mask, max_iterations=50, ftol=1e-10, gtol=1e-10, ptol=1e-8, fixed=False,
                  so3=False):
    """lm_oracle.solve with the constant intrinsics (bit i of mask = intrinsic i) removed from the tangent space"""
    lm_oracle.SO3[0] = bool(so3)
    maps, C = lm_oracle._index_map(n_cp_list)
    D = 9 + 6 * C
    free = np.array([i for i in range(D) if not (i < 9 and (mask >> i) & 1)], int)
    intr, rot, trans = np.array(intr, float), np.array(rot, float).reshape(C, 4), np.array(trans, float).reshape(C, 3)

    def reduced(H, g):
        A, b = lm_oracle.assemble(H, g, maps, D)
        return A[np.ix_(free, free)], b[free]

    def scatter(v):
        out = np.zeros(D)
        out[free] = v
        return out

    cost, H, g = P.normal_eq(intr, rot, trans)
    A, b = reduced(H, g)
    scale = 1.0 / (1.0 + np.sqrt(np.diag(A)))
    radius, dec = 1e4, 2.0
    trace = []

    def gmax():
        pi, pr, pt = lm_oracle.plus(intr, rot, trans, -scatter(b))
        return max(np.abs(intr - pi).max(), np.abs(rot - pr).max(), np.abs(trans - pt).max())

    trace.append((cost, gmax(), radius, 1.0))
    if not fixed and trace[-1][1] <= gtol:
        return intr, rot, trans, trace, "gradient"
    it, reuse, diag, term = 0, False, None, "running"
    while True:
        if it >= max_iterations:
            term = "no_convergence"
            break
        it += 1
        As = A * scale[:, None] * scale[None, :]
        gs = b * scale
        if not reuse:
            diag = np.clip(np.diag(As), 1e-6, 1e32)
        M = As + np.diag(diag / radius)
        try:
            L = np.linalg.cholesky(M)
            step = -np.linalg.solve(L.T, np.linalg.solve(L, gs))
            mcc = -(step @ gs + 0.5 * step @ (As @ step))
            ok = mcc > 0 and np.isfinite(mcc)
        except np.linalg.LinAlgError:
            ok = False
        if not ok:
            radius /= dec
            dec *= 2
            reuse = True
            trace.append((cost, trace[-1][1], radius, -1.0))
            continue
        ci, cr, ct = lm_oracle.plus(intr, rot, trans, scatter(step * scale))
        xn = np.sqrt((intr ** 2).sum() + (rot ** 2).sum() + (trans ** 2).sum())   # ambient |x|, constant intrinsics included
        sn = np.sqrt(((intr - ci) ** 2).sum() + ((rot - cr) ** 2).sum() + ((trans - ct) ** 2).sum())
        cc = P.cost(ci, cr, ct)
        if not fixed:
            if sn <= ptol * (xn + ptol):
                term = "parameter"
                break
            if abs(cost - cc) <= ftol * cost:
                term = "function"
                break
        rho = (cost - cc) / mcc
        if rho > 1e-3:
            intr, rot, trans = ci, cr, ct
            radius = min(1e16, radius / max(1.0 / 3.0, 1.0 - (2 * rho - 1) ** 3))
            dec, reuse = 2.0, False
            cost, H, g = P.normal_eq(intr, rot, trans)
            A, b = reduced(H, g)
            trace.append((cost, gmax(), radius, 1.0))
            if not fixed and trace[-1][1] <= gtol:
                term = "gradient"
                break
        else:
            radius /= dec
            dec *= 2
            reuse = True
            trace.append((cost, trace[-1][1], radius, 0.0))
            if radius < 1e-32:
                term = "min_radius"
                break
    return intr, rot, trans, trace, term


def names_of(mask):
    import eventcalib_b200 as ecb
    return [nm for i, nm in enumerate(ecb.INTRINSIC_NAMES) if (mask >> i) & 1]


def assert_matches_reduced(tr1, i1, r1, t1, tr2, i2, r2, t2, intr0, mask):
    """the criteria of the comparison with solve_reduced: accept / reject sequence, cost trajectory, free parameters, and the
    constant intrinsics equal to their start values"""
    tr2 = np.asarray(tr2)
    assert len(tr1) == len(tr2)
    np.testing.assert_array_equal(tr1[:, 3], tr2[:, 3])
    np.testing.assert_allclose(tr1[:, 0], tr2[:, 0], rtol=1e-9)
    const = np.array([(mask >> i) & 1 for i in range(9)], bool)
    np.testing.assert_array_equal(i1[const], np.asarray(intr0)[const])
    np.testing.assert_array_equal(i2[const], np.asarray(intr0)[const])
    np.testing.assert_allclose(i1[~const], i2[~const], rtol=1e-9)
    np.testing.assert_allclose(np.reshape(r1, (-1, 4)), r2, rtol=0, atol=1e-9)
    np.testing.assert_allclose(np.reshape(t1, (-1, 3)), t2, rtol=1e-9, atol=1e-9)


def _packed(c, H, g):
    ns = H.shape[0]
    out = np.zeros(ns * 1122 + 2)
    blk = out[:ns * 1122].reshape(ns, 1122)
    blk[:, :1089] = H.reshape(ns, 1089)
    blk[:, 1089:] = g
    out[ns * 1122] = c
    return out


@pytest.fixture(scope="module")
def problems(oracle_mod):
    """the problem of test_lm_host.py for both rotation models (SO(3) control points normalised)"""
    from eventcalib_b200 import synth, calib_problem
    ev = synth.make_stream(60000, 346, 260, t0=5.0, duration=0.4, seed=77, return_truth=True, rot_amp=(0.35, 0.35, 0.25),
                           dist=92.0)
    pb = calib_problem.build(ev, seed=1, intr_noise=0.01)
    out = {}
    for so3 in (0, 1):
        P = oracle_mod.CostProblem([pb["n_cp"]], [pb["knots"]], pb["radius"], pb["huber"], so3=bool(so3))
        P.associate(ev["t"], ev["x"], ev["y"], pb["kf_t"], pb["circles"], pb["landmarks"], pb["step"])
        rot0 = pb["rot_cp"].reshape(-1, 4)
        if so3:
            rot0 = rot0 / np.linalg.norm(rot0, axis=1, keepdims=True)
        out[so3] = (pb, P, rot0)
    return out


def _run(pb, P, rot0, names=None, pre=None, **opt):
    import eventcalib_b200 as ecb
    lm = ecb.LmState([pb["n_cp"]], ecb.lm_options(**opt))
    for nm in (pre or []):
        lm.set_constant_intrinsics(nm)
    if names is not None:
        lm.set_constant_intrinsics(names)
    x = (pb["intrinsics"], rot0, pb["trans_cp"])
    st = lm.begin(*x, _packed(*P.normal_eq(*x)))
    while st == 0:
        st, ci, cr, ct = lm.propose()
        if st != 0:
            break
        fb = lm.feedback(P.cost(ci, cr, ct))
        if fb == 1:
            st = lm.update(_packed(*P.normal_eq(ci, cr, ct)))
        elif fb == 0:
            st = 0
        else:
            st = fb
    return lm


@pytest.mark.parametrize("so3", [0, 1])
@pytest.mark.parametrize("which", list(MASKS))
def test_lm_with_constant_intrinsics_matches_reduced_restatement(problems, which, so3):
    pb, P, rot0 = problems[so3]
    mask = MASKS[which]
    K = 12
    lm = _run(pb, P, rot0, names_of(mask), max_iterations=K, rotation_model=so3)
    i1, r1, t1, summ = lm.state()
    i2, r2, t2, tr2, _ = solve_reduced(P, [pb["n_cp"]], pb["intrinsics"], rot0, pb["trans_cp"], mask, max_iterations=K, so3=so3)
    assert_matches_reduced(lm.trace(), i1, r1, t1, tr2, i2, r2, t2, pb["intrinsics"], mask)
    assert summ["final_cost"] < summ["initial_cost"]


def test_zero_mask_is_the_default(problems):
    """k5 set, then cleared, before begin: trace and result bit-identical to a state machine that never had a mask"""
    pb, P, rot0 = problems[0]
    ref = _run(pb, P, rot0, max_iterations=8)
    got = _run(pb, P, rot0, names=[], pre=[["k5"]], max_iterations=8)
    np.testing.assert_array_equal(got.trace(), ref.trace())
    for a, b in zip(got.state()[:3], ref.state()[:3]):
        np.testing.assert_array_equal(a, b)
    assert got.state()[3] == ref.state()[3]


def test_errors(problems):
    import eventcalib_b200 as ecb
    pb, P, rot0 = problems[0]
    lm = ecb.LmState([pb["n_cp"]], ecb.lm_options(max_iterations=2))
    assert lm.lib.ecb_lm_set_constant_intrinsics(lm.h, 0x200) == ecb.ERR_ARG
    assert lm.lib.ecb_lm_set_constant_intrinsics(lm.h, 0x1FF) == ecb.OK
    with pytest.raises(ValueError, match="k6"):
        lm.set_constant_intrinsics(["k1", "k6"])
    with pytest.raises(ValueError, match="K3"):
        ecb.constant_intrinsics_mask("fx,K3")
    assert ecb.constant_intrinsics_mask("k3, k4 k5") == 0b111000000 == ecb.constant_intrinsics_mask(("k3", "k4", "k5"))
    assert ecb.constant_intrinsics_mask([]) == 0
    x = (pb["intrinsics"], rot0, pb["trans_cp"])
    lm.begin(*x, _packed(*P.normal_eq(*x)))
    with pytest.raises(ecb.EcbError) as e:
        lm.set_constant_intrinsics(["k5"])
    assert e.value.code == ecb.ERR_STATE
    assert lm.lib.ecb_lm_set_constant_intrinsics(lm.h, 0) == ecb.ERR_STATE
