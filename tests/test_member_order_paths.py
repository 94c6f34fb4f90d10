"""The restatement behind k_bfs_order's small-cluster path (eventcalib_b200/csrc/ecb_bfs.cu: bfs_small), checked on the CPU
against the UNMODIFIED reference DBSCAN (oracle/_ref: dbscan.h + kdtree.cpp compiled in place):

  * the kd-tree is the reference's insertion tree (kdtree.cpp:106-146: pid order, axis = depth % 2, `<` goes left);
  * v is on the result list of u's range query iff d(u, v) <= eps and every ancestor of v that has v on its FAR side as seen
    from u passes `fabs(dx) < range` (find_nearest, kdtree.cpp:148-179);
  * the query meets nodes in pre-order, near child first, so two met nodes are ordered by their root paths written as near (0) /
    far (1) bits, left-aligned, the shorter path first when one continues the other with "near" only; the result list holds
    the later visit first (head insertion, kdtree.cpp:469-486);
  * a cluster's member list is the FIFO order of expandCluster (dbscan.h:229-259) replayed from those neighbour lists.

This is pure Python over the same integer decisions the kernel takes (floor(eps^2), ceil(eps)); the CUDA kernel itself is
compared with the reference in tests/test_gpu_frontend.py and tests/test_gpu_golden.py."""
import math
import os

import numpy as np
import pytest


def _tree(P):
    """parent, side (0 left / 1 right) and depth of every node of the reference's insertion tree"""
    n = len(P)
    left, right = [-1] * n, [-1] * n
    parent, side, depth = [-1] * n, [0] * n, [0] * n
    for i in range(1, n):
        cur, d = 0, 0
        while True:
            ax = d & 1
            go_left = P[i][ax] < P[cur][ax]
            nxt = left[cur] if go_left else right[cur]
            if nxt < 0:
                if go_left:
                    left[cur] = i
                else:
                    right[cur] = i
                parent[i], side[i], depth[i] = cur, 0 if go_left else 1, d + 1
                break
            cur, d = nxt, d + 1
    return parent, side, depth


def _path_key(P, parent, side, depth, u, v, epsc):
    """(visible, key) of v in u's range query; key orders the met nodes by visit time"""
    chain = []
    c = v
    while parent[c] >= 0:
        chain.append((parent[c], side[c]))
        c = parent[c]
    bits = []
    for a, sd in reversed(chain):            # root first
        ax = depth[a] & 1
        dx = P[u][ax] - P[a][ax]
        far = (dx <= 0) == (sd == 1)         # the near child is the left one iff dx <= 0
        if far and not (abs(dx) < epsc):
            return False, None
        bits.append(1 if far else 0)
    return True, (tuple(bits + [0] * (64 - len(bits))), len(bits))


def _member_order(P, members, eps):
    eps2i, epsc = math.floor(eps * eps), math.ceil(eps)
    parent, side, depth = _tree(P)
    members = sorted(int(m) for m in members)
    nbr = {}
    for u in members:
        seen = []
        for v in members:
            if v == u:
                continue
            ex, ey = P[v][0] - P[u][0], P[v][1] - P[u][1]
            if ex * ex + ey * ey > eps2i:
                continue
            ok, key = _path_key(P, parent, side, depth, u, v, epsc)
            if ok:
                seen.append((key, v))
        nbr[u] = [v for _, v in sorted(seen, reverse=True)]   # later visit first
    order, got = [members[0]], {members[0]}
    h = 0
    while h < len(order):
        for v in nbr[order[h]]:
            if v not in got:
                got.add(v)
                order.append(v)
        h += 1
    return order


def _cloud(rng, kind, n, eps=4.0):
    if kind == "ring":      # circle-edge clusters like the calibration board's
        pts = set()
        for cx, cy, r in ((30, 30, 6.0), (60, 34, 8.5), (40, 70, 5.0), (80, 80, 10.0)):
            for a in rng.uniform(0, 2 * np.pi, n // 4):
                pts.add((int(round(cx + r * math.cos(a))), int(round(cy + r * math.sin(a)))))
        pts = list(pts)
    elif kind == "lattice":  # many points exactly eps apart along the axes: the tie rule decides the edges
        st = max(1, int(eps))
        pts = [(st * i + int(rng.integers(0, 2)), st * j) for i in range(12) for j in range(12) if rng.random() < 0.8]
        pts = list(dict.fromkeys(pts))
    else:                    # dense random blob
        pts = list({(int(x), int(y)) for x, y in rng.integers(0, int(8 * eps) + 8, size=(n, 2))})
    rng.shuffle(pts)
    return [tuple(p) for p in pts]


@pytest.mark.parametrize("kind", ["ring", "lattice", "blob"])
@pytest.mark.parametrize("eps", [1.0, 2.0, 2.5, 3.0, 4.0, 4.5, 8.0])
def test_member_order_from_root_paths(oracle_mod, kind, eps):
    if not oracle_mod.have_ref():
        pytest.skip("oracle/_ref (the reference compiled in place) is not available")
    rng = np.random.default_rng(int(eps * 10) + len(kind))
    checked = 0
    for trial in range(12):
        P = _cloud(rng, kind, 160, eps)
        ref = oracle_mod.ref_dbscan(np.array(P, np.float64), eps, 2)
        for members in ref["clusters"]:
            if len(members) < 3:
                continue
            assert _member_order(P, members, eps) == [int(m) for m in members]
            checked += 1
    assert checked >= 6


def test_member_order_of_the_stored_reference_clusters():
    """The same restatement against the member lists the unmodified reference DBSCAN returned, as stored in
    tests/golden/dbscan_reference.npz (tests/golden/make_golden.py): runs where the reference itself is absent."""
    g =np.load(os.path.join(os.path.dirname(__file__), "golden", "dbscan_reference.npz"))
    checked = 0
    for k in range(int(g["n_cases"])):
        eps, mp = (float(v) for v in g["par_%d" % k])
        if mp != 2:
            continue
        P = [tuple(p) for p in g["pts_%d" % k].astype(float).tolist()]
        off = np.concatenate([[0], np.cumsum(g["sizes_%d" % k])])
        for c in range(len(off) - 1):
            members = [int(m) for m in g["members_%d" % k][off[c]:off[c + 1]]]
            if len(members) >= 3:
                assert _member_order(P, members, eps) == members, "case %d cluster %d" % (k, c)
                checked += 1
    assert checked >= 6
