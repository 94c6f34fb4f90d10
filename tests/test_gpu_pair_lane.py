"""k_pair against the oracle's extractFeatures: candidate pairs and circles on windows that reach each shape of the kernel.
One lane per positive cluster with more positive clusters than a CTA has lanes, knn_num 1 / 3 / 8 (8 takes the KNN_MAX
candidate arrays), fitCircle 0 and 1 and clusters far wider than a warp; and kept-cluster tables too large for shared
memory (global scratch, a warp per cluster)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RTOL = 1e-9
SMEM_TABLE_CAP = 96 * 1024   # k_pair keeps its kept-cluster tables (44 B per entry) in shared memory up to this size
LANE_MAX_POINTS = 4096       # and runs a lane per cluster up to this many points per (window, polarity)


def _run(ctx, oracle_mod, ev, win, width, height, fit_circle, knn_num, eps=4.0, min_pts=2, cluster_min=5):
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth
    ctx.set_sensor(width, height)
    ctx.load_events(synth.to_records(ev))
    rthr = ecb.radius_threshold(width, height, 9, 4, True, 5.5, 1.75)
    prm = ecb.default_params(eps=eps, min_pts=min_pts, cluster_min=cluster_min, knn_num=knn_num, fit_circle=fit_circle,
                             radius_threshold=rthr, order_mode=1, median_mode=1)
    ctx.frontend_run(win, prm)
    summ = ctx.summary()
    pts = [ctx.points(0), ctx.points(1)]
    cand = ctx.candidates(max(64, int(summ["n_candidates"].max())))
    st = dict(max_kept=int(summ["n_kept"].max()), max_points=int(summ["n_points"].max()), max_size=0, candidates=0)
    for w in range(len(win)):
        s = summ[w]
        assert s["status"] == 0
        V = [pts[pol][0][int(s["point_offset"][pol]):int(s["point_offset"][pol]) + int(s["n_points"][pol])] for pol in (0, 1)]
        r = oracle_mod.extract(V[1], V[0], eps=eps, minS=min_pts, clusterMin=cluster_min, knn_num=knn_num,
                               fitCircle=fit_circle, Rthr=rthr, canonical_median=False)
        assert s["n_candidates"] == len(r["cand"]), "window %d" % w
        if len(r["cand"]):
            g = cand[w, :len(r["cand"])]
            assert np.array_equal(g[:, :2], r["cand"][:, :2]), "window %d" % w
            np.testing.assert_allclose(g[:, 2:], r["cand"][:, 2:], rtol=RTOL, atol=0)
        st["max_size"] = max([st["max_size"]] + [len(c) for c in r["p_clusters"]] + [len(c) for c in r["n_clusters"]])
        st["candidates"] += len(r["cand"])
    return st


@pytest.mark.parametrize("knn_num", [1, 3, 8])
@pytest.mark.parametrize("fit_circle", [0, 1])
def test_many_clusters_per_window(ctx, oracle_mod, fit_circle, knn_num):
    """Noisy DAVIS346 windows: over a hundred kept clusters per polarity, more than a CTA has lanes."""
    from eventcalib_b200 import synth
    ev = synth.make_stream(16000, 346, 260, t0=0.0, duration=0.003, seed=78, noise_frac=0.7, flip_frac=0.1)
    win = synth.tiling_windows(0.0, 0.003, 1.5e-3)
    st = _run(ctx, oracle_mod, ev, win, 346, 260, fit_circle, knn_num, eps=2.0, cluster_min=2)
    assert st["max_kept"] > 100 and st["max_points"] <= LANE_MAX_POINTS and st["candidates"] > 0, st


@pytest.mark.parametrize("knn_num", [1, 3, 8])
@pytest.mark.parametrize("fit_circle", [0, 1])
def test_large_clusters(ctx, oracle_mod, fit_circle, knn_num):
    """640x480 windows of 2 ms: clusters of about a hundred members, which one lane sums alone."""
    from eventcalib_b200 import synth
    ev = synth.make_stream(30000, 640, 480, t0=0.0, duration=0.004, seed=1003)
    win = synth.tiling_windows(0.0, 0.004, 2e-3)
    st = _run(ctx, oracle_mod, ev, win, 640, 480, fit_circle, knn_num)
    assert st["max_size"] > 32 and st["max_points"] <= LANE_MAX_POINTS and st["candidates"] > 30 * len(win), st


@pytest.mark.parametrize("fit_circle", [0, 1])
def test_tables_beyond_shared_memory(ctx, oracle_mod, fit_circle):
    """One 1280x720 window with thousands of kept clusters per polarity: the kept-cluster tables live in global scratch."""
    from eventcalib_b200 import synth
    ev = synth.make_stream(600000, 1280, 720, t0=0.0, duration=0.002, seed=79, noise_frac=0.8, flip_frac=0.05)
    win = np.array([[0.0, 0.001]])
    st = _run(ctx, oracle_mod, ev, win, 1280, 720, fit_circle, 3, eps=2.0, cluster_min=2)
    assert st["max_kept"] * 44 > SMEM_TABLE_CAP and st["candidates"] > 0, st
