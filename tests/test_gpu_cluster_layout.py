"""k_cluster's two shared-memory layouts against the oracle, on both sides of every limit the launcher picks by.

The launcher keeps r_st (per point: rank of a pid, then the seed mask and the member lists) in 16-bit words when the batch's
largest problem is below 2^15 points and within the fast kd path (n <= 6 points per thread); otherwise it keeps the wide
32-bit layout, whose slow kd path packs a node pid and two tie flags into one word.  On a 346 x 260 sensor with eps 4 the
narrow layout fits four CTAs per SM up to 1 458 points per problem (no kept-cluster tables, as in ecb_dbscan_run).
Labels must equal the oracle's bit for bit, and a window's results must not depend on the layout its batch ran with.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W, H = 346, 260
KD_PT = 6
FOUR_CTA_MAX_N = 1458  # 346 x 260, eps 4, max_k 1: 4 x (dynamic + 672 static + 1 KB reserved) <= 228 KB


def _points(rng, n):
    """n distinct pixels spanning the whole sensor (corners included): rings of dots with exact-eps gaps, plus noise."""
    pts = set()
    while len(pts) < 3 * n:
        cx, cy, r = rng.integers(10, W - 10), rng.integers(10, H - 10), rng.integers(3, 9)
        a = rng.uniform(0, 2 * np.pi, 4 * r)
        pts.update(zip(np.rint(cx + r * np.cos(a)).astype(int).tolist(), np.rint(cy + r * np.sin(a)).astype(int).tolist()))
        pts.update(zip(rng.integers(0, W, 8).tolist(), rng.integers(0, H, 8).tolist()))
    corners = [(0, 0), (W - 1, H - 1)]
    rest = sorted(pts - set(corners))
    pick = [rest[i] for i in rng.choice(len(rest), n - 2, replace=False)] + corners
    out = np.array(pick, np.float64)
    rng.shuffle(out)
    return out


def _check_batch(ctx, oracle_mod, sizes, seed, eps=4, min_pts=2):
    rng = np.random.default_rng(seed)
    sets = [_points(rng, n) for n in sizes]
    off = np.concatenate([[0], np.cumsum(sizes)])
    lab, nc, st = ctx.dbscan_batch(np.concatenate(sets), off, eps, min_pts)
    assert not st.any()
    for k, s in enumerate(sets):
        ref = oracle_mod.dbscan(s, eps, min_pts)
        assert nc[k] == len(ref["clusters"])
        assert np.array_equal(lab[off[k]:off[k + 1]], ref["labels"]), "labels differ (n=%d)" % len(s)


@pytest.mark.parametrize("threads", [256, 320])
@pytest.mark.parametrize("side", [0, 1])
def test_kd_fast_path_limit(ctx, oracle_mod, monkeypatch, threads, side):
    # n_cap = KD_PT * threads: narrow layout, fast kd path; one point more: wide layout, slow kd path
    monkeypatch.setenv("ECB_CL_THREADS", str(threads))
    n = KD_PT * threads + side
    _check_batch(ctx, oracle_mod, [n, n - 1, n // 2, 64], seed=threads + side)


@pytest.mark.parametrize("n", [FOUR_CTA_MAX_N - 1, FOUR_CTA_MAX_N, FOUR_CTA_MAX_N + 1])
def test_four_cta_footprint_limit(ctx, oracle_mod, n):
    # up to the limit: 4 CTAs x 256 threads; past it: 3 x 320, both in the narrow layout
    _check_batch(ctx, oracle_mod, [n, 1235, 700], seed=n)


def test_narrow_and_wide_on_the_same_problems(ctx, oracle_mod):
    # the same point sets once in a narrow batch and once with a problem that makes the batch wide
    rng = np.random.default_rng(7)
    sets = [_points(rng, n) for n in (1235, 900, 1400)]
    big = _points(rng, 4000)
    for group in (sets, sets + [big]):
        off = np.concatenate([[0], np.cumsum([len(s) for s in group])])
        lab, nc, st = ctx.dbscan_batch(np.concatenate(group), off, 4, 2)
        assert not st.any()
        for k, s in enumerate(group):
            assert np.array_equal(lab[off[k]:off[k + 1]], oracle_mod.dbscan(s, 4, 2)["labels"])


def test_frontend_windows_alone_and_with_an_oversized_window(ctx, oracle_mod):
    """DAVIS346 windows at the benchmark's density run in the narrow layout; one long window added to the batch switches
    the whole batch to the wide layout.  Labels, kept-cluster tables (ids, sizes, medians) and candidates of the shared
    windows must not change."""
    import eventcalib_b200 as ecb
    from eventcalib_b200 import synth
    ev = synth.make_stream(24000, W, H, t0=5.0, duration=0.012, seed=1002, noise_frac=0.05)
    win = synth.tiling_windows(5.0, 5.012, 1.5e-3)
    ctx.set_sensor(W, H)
    ctx.load_events(synth.to_records(ev))
    rthr = ecb.radius_threshold(W, H, 9, 4, True, 5.5, 1.75)
    prm = ecb.default_params(fit_circle=1, radius_threshold=rthr, order_mode=1, median_mode=1)
    runs = []
    for windows in (win, np.concatenate([win, [[5.0, 5.006]]])):
        ctx.frontend_run(windows, prm)
        s = ctx.summary()
        pts = [ctx.points(0), ctx.points(1)]
        out = {"cand": ctx.candidates(64)[:len(win)], "summ": s[:len(win)], "n_points": s["n_points"].max(axis=1)}
        for w in range(len(win)):
            for pol in (0, 1):
                o, k = int(s["point_offset"][w][pol]), int(s["n_points"][w][pol])
                out[w, pol] = (pts[pol][0][o:o + k], pts[pol][1][o:o + k]) + ctx.clusters(w, pol)
        runs.append(out)
    alone, mixed = runs
    assert alone["n_points"].max() <= KD_PT * 256 < mixed["n_points"][-1]
    assert np.array_equal(alone["cand"], mixed["cand"])
    for f in ("n_clusters", "n_kept", "n_candidates", "status"):
        assert np.array_equal(alone["summ"][f], mixed["summ"][f])
    for w in range(len(win)):
        for pol in (0, 1):
            for a, b in zip(alone[w, pol], mixed[w, pol]):
                assert np.array_equal(a, b), "window %d pol %d differs between the layouts" % (w, pol)
            # and the labels are the oracle's
            assert np.array_equal(alone[w, pol][1], oracle_mod.dbscan(alone[w, pol][0], 4, 2)["labels"])
