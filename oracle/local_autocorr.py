"""Oracle of K18 (pg_local_autocorr): local Moran's I_i and Getis-Ord Gi / Gi* restated in numpy / scipy.sparse, with
esda's conditional randomisation on K15's keyed permutations.

The observed statistics come from explicit weight matrices: W from the CSR (entries with an id outside [0, n) and self
entries dropped; binary, or each row divided by its sum), W* = that binary W plus the identity for Gi* (then row-
normalised), lags as W @ z, and W_i / S1_i as row sums of W and of W squared - Ord & Getis's forms with x(i) and S(i)
written on the centred z = x - mean. ``textbook_g`` keeps the forms on the raw x for the tests that show both agree.
Permuted statistics follow include/pathgraph.h: r_p = oracle.enrichment.permutations(n - 1, seed, [p])[:, :K], node
i's j-th neighbour r_p[j] + (r_p[j] >= i), the sum over j < d_i."""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp

from . import enrichment as oe

EPS = 2.0 ** -53
MODES = ("moran", "gi", "gi_star")


def graph(row_ptr, col, n: int) -> tuple[np.ndarray, np.ndarray]:
    """(rows, cols) int64 of the kept entries: ids in [0, n), not on the diagonal, in CSR order."""
    rp = np.asarray(row_ptr, dtype=np.int64)
    c = np.asarray(col, dtype=np.int64)
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(rp))
    ok = (c >= 0) & (c < n) & (c != rows)
    return rows[ok], c[ok]


def degrees(row_ptr, col, n: int) -> np.ndarray:
    rows, _ = graph(row_ptr, col, n)
    return np.bincount(rows, minlength=n).astype(np.int64)


def weights(row_ptr, col, n: int, transformation: bool, star: bool = False) -> sp.csr_matrix:
    """float64 [n, n]: 1 per kept entry (duplicates add), plus 1 on the diagonal with ``star``; row-normalised with
    ``transformation``."""
    rows, c = graph(row_ptr, col, n)
    if star:
        rows = np.concatenate([rows, np.arange(n, dtype=np.int64)])
        c = np.concatenate([c, np.arange(n, dtype=np.int64)])
    w = sp.csr_matrix((np.ones(rows.shape[0]), (rows, c)), shape=(n, n))
    if transformation:
        s = np.asarray(w.sum(axis=1)).ravel()
        w = sp.diags(np.divide(1.0, s, out=np.zeros_like(s), where=s > 0)) @ w
    return sp.csr_matrix(w)


def centred(x) -> np.ndarray:
    x = np.asarray(x, dtype=np.float64)
    return x - x.mean(axis=0) if x.shape[0] else x.copy()


def magnitudes(x, z) -> np.ndarray:
    """|z| + mean |x| per column: what the bound scales. A centred value carries the error of the mean as well as its
    own, and a mean of n values is off by up to n 2^-53 mean |x| whatever order it is summed in."""
    return np.abs(z) + (np.abs(x).mean(axis=0) if x.shape[0] else 0.0)


def _sqrt_pos(v):
    v = np.asarray(v, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        return np.where(v > 0, np.sqrt(np.where(v > 0, v, 1.0)), np.nan)


def observed(mode: str, row_ptr, col, x, transformation: bool) -> dict:
    """stat, lag [n, F] and the magnitude |stat| would have with |z| everywhere in its numerator (for the bound)."""
    x = np.asarray(x, dtype=np.float64)
    n = x.shape[0]
    z = centred(x)
    az = magnitudes(x, z)
    m2 = (z * z).sum(axis=0)
    nn = float(n)
    w = weights(row_ptr, col, n, transformation)
    lag, alag = w @ z, abs(w) @ az
    with np.errstate(divide="ignore", invalid="ignore"):
        if mode == "moran":
            c = np.where(m2 != 0, (nn - 1.0) / m2, np.nan)
            stat, mag = c * z * lag, np.abs(c) * az * alag
        elif mode == "gi_star":
            ws = weights(row_ptr, col, n, transformation, star=True)
            wi = np.asarray(ws.sum(axis=1)).ravel()[:, None]
            s1 = np.asarray(ws.multiply(ws).sum(axis=1)).ravel()[:, None]
            den = _sqrt_pos(m2 / nn if n else np.full_like(m2, np.nan)) * _sqrt_pos((nn * s1 - wi * wi) / (nn - 1.0))
            if n < 2:
                den = den * np.nan
            stat, mag = (ws @ z) / den, (abs(ws) @ az) / np.abs(den)
        else:
            wi = np.asarray(w.sum(axis=1)).ravel()[:, None]
            s1 = np.asarray(w.multiply(w).sum(axis=1)).ravel()[:, None]
            si = _sqrt_pos((m2 - z * z * nn / (nn - 1.0)) / (nn - 1.0))
            den = si * _sqrt_pos(((nn - 1.0) * s1 - wi * wi) / (nn - 2.0))
            if n < 3:
                den = den * np.nan
            stat = (lag + wi * z / (nn - 1.0)) / den
            mag = (alag + wi * az / (nn - 1.0)) / np.abs(den)
    return {"stat": stat, "lag": lag, "mag": mag, "z": z, "m2": m2}


def finish(mode: str, transformation: bool, n: int, d, zi, m2, s, zn=None) -> np.ndarray:
    """The statistic of nodes with degrees d [k], centred values zi [k, F] and neighbour sums s [..., k, F]: the degree
    forms of include/pathgraph.h (the kernel's), shared by the observed and the permuted sums. ``zn`` replaces z_i in
    the numerator only (the bound's magnitudes)."""
    zn = zi if zn is None else zn
    d = np.asarray(d, dtype=np.float64)[:, None]
    nn = float(n)
    with np.errstate(divide="ignore", invalid="ignore"):
        if mode == "moran":
            w = np.where(d > 0, 1.0 / d, 0.0) if transformation else 1.0
            c = np.where(m2 != 0, (nn - 1.0) / m2, np.nan)
            return c * zn * (w * s)
        if mode == "gi_star":
            w = 1.0 / (d + 1.0) if transformation else 1.0
            wi = 1.0 if transformation else d + 1.0
            s1 = w if transformation else d + 1.0
            den = _sqrt_pos(m2 / nn) * _sqrt_pos((nn * s1 - wi * wi) / (nn - 1.0))
            return (w * zn + w * s) / (den if n >= 2 else np.nan)
        w = 1.0 / d if transformation else 1.0
        wi = np.where(d > 0, 1.0, 0.0) if transformation else d
        s1 = 1.0 / d if transformation else d
        si = _sqrt_pos((m2 - zi * zi * nn / (nn - 1.0)) / (nn - 1.0))
        den = np.where(d > 0, si * _sqrt_pos(((nn - 1.0) * s1 - wi * wi) / (nn - 2.0)), np.nan)
        return (w * s + wi * zn / (nn - 1.0)) / (den if n >= 3 else np.nan)


def draws(n: int, seed: int, perms, k: int) -> np.ndarray:
    """int64 [len(perms), k]: r_p[j] = pi'_p(j), pi'_p K15's bijection of [0, n - 1) - the first k columns of
    oracle.enrichment.permutations(n - 1, seed, perms), evaluated for j < k only (K << n on a slide)."""
    perms = np.asarray(list(perms), dtype=np.uint64).reshape(-1)
    m = n - 1
    if k == 0 or m < 1:
        return np.zeros((len(perms), 0), dtype=np.int64)
    h = oe.half_bits(m)
    mask, sh = np.uint64((1 << h) - 1), np.uint64(h)
    rounds = np.arange(oe.ROUNDS, dtype=np.uint64)
    with np.errstate(over="ignore"):
        keys = oe.splitmix64(np.uint64(seed) ^ (np.uint64(64) * perms[:, None] + rounds[None, :]))
    out = np.empty((len(perms), k), dtype=np.uint64)
    cur = np.broadcast_to(np.arange(k, dtype=np.uint64), out.shape).copy()
    todo = np.ones(out.shape, dtype=bool)
    while todo.any():
        rows, cols = np.nonzero(todo)
        v = cur[rows, cols]
        lo, ro = v >> sh, v & mask
        for r in range(oe.ROUNDS):
            lo, ro = ro, lo ^ (oe.splitmix64(ro ^ keys[rows, r]) & mask)
        v = (lo << sh) | ro
        cur[rows, cols] = v
        ok = v < np.uint64(m)
        out[rows[ok], cols[ok]] = v[ok]
        todo[rows[ok], cols[ok]] = False
    return out.astype(np.int64)


def permuted_sums(z, az, d, nodes, r) -> tuple[np.ndarray, np.ndarray]:
    """Neighbour sums of z [n, F] (and of the magnitudes az) for the given nodes under draws r [P, K]:
    [P, len(nodes), F]."""
    z = np.asarray(z, dtype=np.float64)
    nodes = np.asarray(nodes, dtype=np.int64)
    dn = np.asarray(d, dtype=np.int64)[nodes]
    owner = np.repeat(np.arange(nodes.shape[0]), dn)
    j = np.arange(int(dn.sum())) - np.repeat(np.cumsum(dn) - dn, dn)
    p = r.shape[0]
    s = np.zeros((p, nodes.shape[0], z.shape[1]))
    a = np.zeros_like(s)
    for k in range(p):
        rj = r[k, j]
        src = rj + (rj >= nodes[owner])
        m = sp.csr_matrix((np.ones(owner.shape[0]), (owner, src)), shape=(nodes.shape[0], z.shape[0]))
        s[k] = m @ z
        a[k] = m @ az
    return s, a


def scale(n: int, d) -> np.ndarray:
    """Relative agreement bound of a fixed-order float64 evaluation, per node: 8 (d_i + n + 16) 2^-53."""
    return 8.0 * (np.asarray(d, dtype=np.float64) + n + 16.0) * EPS


def local_autocorr(row_ptr, col, x, mode: str = "moran", transformation: bool = True, n_perms: int = 0, seed: int = 0,
                   nodes=None, perms=None) -> dict:
    """The outputs of pg_local_autocorr for x [n, F] ([F, n] like the kernel's, except sims [P, F, n]) with per-value
    bounds. ``nodes`` / ``perms`` restrict the permutation outputs to a sample (sims then [len(perms), F, len(nodes)])."""
    x = np.asarray(x, dtype=np.float64)
    n, f = x.shape
    ob = observed(mode, row_ptr, col, x, transformation)
    z, m2 = ob["z"], ob["m2"]
    d = degrees(row_ptr, col, n)
    sc = scale(n, d)[:, None]
    out = {"stat": ob["stat"].T, "lag": ob["lag"].T, "bound": (sc * ob["mag"]).T, "d": d,
           "mean": x.mean(axis=0) if n else np.full(f, np.nan), "m2": m2,
           "mean_bound": scale(n, 0) * (np.abs(x).mean(axis=0) if n else np.zeros(f))}
    az = magnitudes(x, z)
    out["lag_bound"] = (sc * (abs(weights(row_ptr, col, n, transformation)) @ az)).T
    nodes = np.arange(n) if nodes is None else np.asarray(nodes, dtype=np.int64)
    perms = list(range(n_perms)) if perms is None else list(perms)
    k = int(d.max()) if n else 0
    r = draws(n, seed, perms, k)
    s, a = permuted_sums(z, az, d, nodes, r)
    zi, dn = z[nodes], d[nodes]
    sims = finish(mode, transformation, n, dn, zi, m2, s)
    mag = np.abs(finish(mode, transformation, n, dn, zi, m2, a, zn=az[nodes]))
    sims[:, dn == 0] = np.nan
    out["sims"] = np.moveaxis(sims, 2, 1)                          # [P, F, nodes]
    out["sims_bound"] = np.moveaxis(scale(n, dn)[None, :, None] * mag, 2, 1)
    stat = out["stat"][:, nodes]
    with np.errstate(invalid="ignore"):
        if len(perms):
            out["n_ge"] = np.where(np.isnan(stat), 0, (out["sims"] >= stat[None]).sum(0))
            out["perm_mean"] = out["sims"].mean(axis=0)
            out["perm_var"] = out["sims"].var(axis=0)
        else:
            out["n_ge"] = np.zeros(stat.shape, dtype=np.int64)
            out["perm_mean"] = np.full(stat.shape, np.nan)
            out["perm_var"] = np.full(stat.shape, np.nan)
    out["nodes"] = nodes
    return out


def textbook_g(row_ptr, col, x, transformation: bool, star: bool) -> dict:
    """Ord & Getis (1995) on the raw values of a column x [n]: G_i = sum_j w_ij x_j / sum_j x_j (j != i unless star),
    and the z-score (sum_j w_ij x_j - W_i xbar) / (S sqrt((m S1_i - W_i^2) / (m - 1))), where xbar and S (ddof 0) are
    taken over the m = n values (Gi*) or the m = n - 1 values other than x_i (Gi)."""
    x = np.asarray(x, dtype=np.float64)
    n = x.shape[0]
    w = weights(row_ptr, col, n, transformation, star=star)
    wi = np.asarray(w.sum(axis=1)).ravel()
    s1 = np.asarray(w.multiply(w).sum(axis=1)).ravel()
    num = w @ x
    if star:
        m, xbar = float(n), np.full(n, x.mean())
        s = np.full(n, x.std())
        den_g = np.full(n, x.sum())
    else:
        m = n - 1.0
        xbar = (x.sum() - x) / m
        s = np.sqrt((((x * x).sum() - x * x) / m) - xbar * xbar)
        den_g = x.sum() - x
    with np.errstate(divide="ignore", invalid="ignore"):
        return {"G": num / den_g, "Z": (num - wi * xbar) / (s * np.sqrt((m * s1 - wi * wi) / (m - 1.0)))}
