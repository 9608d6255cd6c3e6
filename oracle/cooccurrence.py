"""Host reference of K16 (pg_pair_dist_hist) and of the statistics built on it (co_occurrence's ``occ``, Ripley's K
and L).

hist[b, a-1, c-1] = ordered pairs (i, j), i a query row, j any point, id_i != id_j, type_i = a, type_j = c, whose
squared distance d2 = fl(fl(dx*dx) + fl(dy*dy)) falls into bin b of the squared thresholds t2 = fl(t*t): b = 0 for
d2 <= t2[0], b for t2[b-1] < d2 <= t2[b]; pairs past the last threshold and types outside 1..T count nowhere.
numpy evaluates every float64 operation on its own (no FMA contraction), so ``_d2`` is the library's rule, and
``searchsorted(t2, d2, side="left")`` is the first b with d2 <= t2[b].

``pair_hist_brute`` takes every pair, in chunks of query rows. ``pair_hist`` takes the candidates of cKDTree's
sparse_distance_matrix at a radius a little above t_max, then decides every candidate by the same exact rule; the CPU
tests check that both agree, so the cheaper one serves slide-sized inputs.
"""
from __future__ import annotations

import numpy as np


def squared(thresholds) -> np.ndarray:
    t = np.asarray(thresholds, dtype=np.float64)
    return t * t


def _d2(ax, ay, bx, by):
    dx = ax - bx
    dy = ay - by
    return dx * dx + dy * dy


def _accumulate(hist, t2, n_types, ta, tb, d2):
    """Add the pairs (type ta, type tb, squared distance d2) - equal-length 1-D arrays - to hist [B*T*T]."""
    k = len(t2)
    ok = (ta >= 1) & (ta <= n_types) & (tb >= 1) & (tb <= n_types) & (d2 <= t2[-1])
    b = np.searchsorted(t2, d2[ok], side="left")
    key = (b * n_types + (ta[ok].astype(np.int64) - 1)) * n_types + (tb[ok].astype(np.int64) - 1)
    hist += np.bincount(key, minlength=k * n_types * n_types).astype(np.int64)


def _prep(xy, types, n_query, ids):
    xy = np.asarray(xy, dtype=np.float64).reshape(-1, 2)
    types = np.asarray(types, dtype=np.int64).reshape(-1)
    n = xy.shape[0]
    nq = n if n_query is None else int(n_query)
    ids = np.arange(n, dtype=np.int64) if ids is None else np.asarray(ids, dtype=np.int64).reshape(-1)
    return xy, types, nq, ids


def type_count(types, n_types, n_query=None) -> np.ndarray:
    t = np.asarray(types, dtype=np.int64).reshape(-1)
    t = t[: len(t) if n_query is None else int(n_query)]
    t = t[(t >= 1) & (t <= n_types)]
    return np.bincount(t - 1, minlength=n_types).astype(np.int64)


def pair_hist_brute(xy, types, thresholds, n_types, n_query=None, ids=None, chunk=1024) -> np.ndarray:
    """int64 [B, T, T] from every pair (i < n_query, j any)."""
    xy, types, nq, ids = _prep(xy, types, n_query, ids)
    t2 = squared(thresholds)
    hist = np.zeros(len(t2) * n_types * n_types, dtype=np.int64)
    for i0 in range(0, nq, chunk):
        i1 = min(nq, i0 + chunk)
        d2 = _d2(xy[i0:i1, 0, None], xy[i0:i1, 1, None], xy[None, :, 0], xy[None, :, 1])
        ta = np.broadcast_to(types[i0:i1, None], d2.shape)
        tb = np.broadcast_to(types[None, :], d2.shape)
        keep = ids[i0:i1, None] != ids[None, :]
        _accumulate(hist, t2, n_types, ta[keep], tb[keep], d2[keep])
    return hist.reshape(len(t2), n_types, n_types)


def pair_hist_sets(xq, tq, idq, xc, tc, idc, thresholds, n_types, chunk=200_000) -> np.ndarray:
    """int64 [B, T, T] of the ordered pairs (i in the query set, j in the candidate set, id_i != id_j); candidates from
    cKDTree at t_max (1 + 1e-9) plus a hair (its ndarray output keeps pairs at distance 0), every one decided by the
    exact rule."""
    from scipy.spatial import cKDTree

    xq = np.asarray(xq, dtype=np.float64).reshape(-1, 2)
    xc = np.asarray(xc, dtype=np.float64).reshape(-1, 2)
    tq, tc = np.asarray(tq, dtype=np.int64), np.asarray(tc, dtype=np.int64)
    idq, idc = np.asarray(idq, dtype=np.int64), np.asarray(idc, dtype=np.int64)
    t2 = squared(thresholds)
    hist = np.zeros(len(t2) * n_types * n_types, dtype=np.int64)
    if len(xq) == 0 or len(xc) == 0:
        return hist.reshape(len(t2), n_types, n_types)
    reach = float(np.sqrt(t2[-1])) * (1.0 + 1e-9) + 1e-300
    tree_c = cKDTree(xc)
    for i0 in range(0, len(xq), chunk):
        i1 = min(len(xq), i0 + chunk)
        m = cKDTree(xq[i0:i1]).sparse_distance_matrix(tree_c, reach, output_type="ndarray")
        i = m["i"].astype(np.int64) + i0
        j = m["j"].astype(np.int64)
        keep = idq[i] != idc[j]
        i, j = i[keep], j[keep]
        _accumulate(hist, t2, n_types, tq[i], tc[j], _d2(xq[i, 0], xq[i, 1], xc[j, 0], xc[j, 1]))
    return hist.reshape(len(t2), n_types, n_types)


def pair_hist(xy, types, thresholds, n_types, n_query=None, ids=None) -> np.ndarray:
    """int64 [B, T, T]: the same histogram as pair_hist_brute, for slide-sized inputs."""
    xy, types, nq, ids = _prep(xy, types, n_query, ids)
    return pair_hist_sets(xy[:nq], types[:nq], ids[:nq], xy, types, ids, thresholds, n_types)


def occurrence(count) -> np.ndarray:
    """occ[a, c, b] = count[a, c, b] * S_b / (R_ab * R_cb) in float64; R = row sums, S = the interval's total; NaN where
    R_ab or R_cb is 0."""
    cnt = np.asarray(count, dtype=np.int64)
    t, _, nb = cnt.shape
    occ = np.full(cnt.shape, np.nan)
    for b in range(nb):
        c = cnt[:, :, b]
        s = float(c.sum())
        row = c.sum(axis=1)
        for a in range(t):
            for d in range(t):
                if row[a] and row[d]:
                    occ[a, d, b] = float(c[a, d]) * s / (float(row[a]) * float(row[d]))
    return occ


def ripley_k(count, n, area) -> np.ndarray:
    """K[a, c, r] = area C[a, c, r] / (n_a n_c), diagonal area C[a, a, r] / (n_a (n_a - 1)); NaN where that is 0."""
    cnt = np.asarray(count, dtype=np.int64)
    n = np.asarray(n, dtype=np.int64)
    k = np.full(cnt.shape, np.nan)
    for a in range(len(n)):
        for c in range(len(n)):
            den = int(n[a]) * (int(n[a]) - 1) if a == c else int(n[a]) * int(n[c])
            if den > 0:
                k[a, c] = float(area) * cnt[a, c].astype(np.float64) / float(den)
    return k
