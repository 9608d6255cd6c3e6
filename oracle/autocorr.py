"""Oracle of K17 (pg_spatial_autocorr): Moran's I and Geary's C restated in numpy / scipy.sparse from their general
definitions, independently of the kernel's shortcuts.

W is built explicitly from the CSR (entries with an id outside [0, n) dropped; binary, or each row divided by its sum);
S0 / S1 / S2 come from W's general definitions, each statistic from z^T W z (Moran) or the per-entry sum
w_ij (z_i - z_j)^2 (Geary), and the permutations from oracle.enrichment.permutations (K15's pi_p). It also carries the
variance under the randomisation assumption (Cliff & Ord), which the product does not output."""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp

from . import enrichment as oe

EPS = 2.0 ** -53


def weight_matrix(row_ptr, col, n: int, transformation: bool) -> sp.csr_matrix:
    """float64 [n, n]: w_ij = 1 per in-range entry (duplicates add), or row-normalised (w_ij / row sum)."""
    rp = np.asarray(row_ptr, dtype=np.int64)
    c = np.asarray(col, dtype=np.int64)
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(rp))
    ok = (c >= 0) & (c < n)
    w = sp.csr_matrix((np.ones(int(ok.sum())), (rows[ok], c[ok])), shape=(n, n))
    if transformation:
        s = np.asarray(w.sum(axis=1)).ravel()
        inv = np.divide(1.0, s, out=np.zeros_like(s), where=s > 0)
        w = sp.diags(inv) @ w
    return sp.csr_matrix(w)


def weight_sums(w: sp.spmatrix) -> tuple[float, float, float]:
    """S0 = sum w_ij, S1 = 1/2 sum (w_ij + w_ji)^2, S2 = sum_i (w_i. + w_.i)^2."""
    s0 = float(w.sum())
    sym = w + w.T
    s1 = 0.5 * float(sym.multiply(sym).sum())
    s2 = float(((np.asarray(w.sum(axis=1)).ravel() + np.asarray(w.sum(axis=0)).ravel()) ** 2).sum())
    return s0, s1, s2


def weight_sums_shortcut(row_ptr, col, n: int, transformation: bool) -> tuple[float, float, float]:
    """The degree formulas the kernel uses for a symmetric CSR: binary S0 = sum d_i, S1 = 2 S0, S2 = 4 sum d_i^2 (exact
    integers); row-standardised S0 = non-isolated nodes, S1 = 1/2 sum over entries (1/d_i + 1/d_j)^2,
    S2 = sum_i (1 + sum_{j in N(i)} 1/d_j)^2."""
    rp = np.asarray(row_ptr, dtype=np.int64)
    c = np.asarray(col, dtype=np.int64)
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(rp))
    ok = (c >= 0) & (c < n)
    rows, c = rows[ok], c[ok]
    d = np.bincount(rows, minlength=n).astype(np.int64)
    if not transformation:
        s0 = int(d.sum())
        return float(s0), float(2 * s0), float(4 * int((d * d).sum()))
    inv = np.divide(1.0, d, out=np.zeros(n), where=d > 0)
    s1 = 0.5 * float(((inv[rows] + inv[c]) ** 2).sum())
    a = np.bincount(rows, weights=inv[c], minlength=n)
    s2 = float(((1.0 + a[d > 0]) ** 2).sum())
    return float((d > 0).sum()), s1, s2


def centred(x) -> np.ndarray:
    """z = x - mean(x) per column of x [n, F]."""
    x = np.asarray(x, dtype=np.float64)
    return x - x.mean(axis=0) if x.shape[0] else x.copy()


def statistic(mode: str, w: sp.csr_matrix, z) -> np.ndarray:
    """Moran's I or Geary's C of every column of the centred values z [n, F] (NaN where m2 = 0 or S0 = 0)."""
    z = np.asarray(z, dtype=np.float64)
    n = z.shape[0]
    s0 = float(w.sum())
    m2 = (z * z).sum(axis=0)
    with np.errstate(divide="ignore", invalid="ignore"):
        if mode == "moran":
            out = n * (z * (w @ z)).sum(axis=0) / (s0 * m2)
        else:
            coo = w.tocoo()
            d = z[coo.row] - z[coo.col]
            out = (n - 1.0) * (coo.data[:, None] * d * d).sum(axis=0) / (2.0 * s0 * m2)
    out = np.asarray(out, dtype=np.float64)
    out[(m2 == 0) | (s0 == 0)] = np.nan
    return out


def bound(mode: str, w: sp.csr_matrix, z) -> np.ndarray:
    """Per column, the agreement bound of a fixed-order float64 evaluation: 8 (E_dir + n) 2^-53 x the statistic of
    |terms| (Moran: sum |w z_i z_j| n / (S0 m2); Geary: the statistic itself, whose terms are >= 0)."""
    z = np.asarray(z, dtype=np.float64)
    n = z.shape[0]
    scale = 8.0 * (w.nnz + n) * EPS
    if mode == "moran":
        s0 = float(w.sum())
        m2 = (z * z).sum(axis=0)
        with np.errstate(divide="ignore", invalid="ignore"):
            return scale * n * (np.abs(z) * (abs(w) @ np.abs(z))).sum(axis=0) / (s0 * m2)
    return scale * np.abs(statistic(mode, w, z))


def permuted(mode: str, w: sp.csr_matrix, z, seed: int, perms, with_bound: bool = False):
    """[len(perms), F] statistics of z[pi_p] (every column shuffled by the same pi_p), and the bounds with
    ``with_bound``."""
    z = np.asarray(z, dtype=np.float64)
    n, f = z.shape
    perms = list(perms)
    sims = np.empty((len(perms), f))
    bnd = np.empty((len(perms), f))
    step = max(1, (1 << 22) // max(n, 1))
    for s in range(0, len(perms), step):
        pis = oe.permutations(n, seed, perms[s:s + step]) if n else np.zeros((len(perms[s:s + step]), 0), np.int64)
        for k, pi in enumerate(pis):
            sims[s + k] = statistic(mode, w, z[pi])
            if with_bound:
                bnd[s + k] = bound(mode, w, z[pi])
    return (sims, bnd) if with_bound else sims


def spatial_autocorr(row_ptr, col, x, mode: str = "moran", transformation: bool = True, n_perms: int = 0,
                     seed: int = 0) -> dict:
    """The outputs of pg_spatial_autocorr for x [n, F], with their bounds: stat, sims [P, F], perm_mean, perm_var,
    s012, and bound / sims_bound."""
    x = np.asarray(x, dtype=np.float64)
    n = x.shape[0]
    w = weight_matrix(row_ptr, col, n, transformation)
    z = centred(x)
    sims, sb = permuted(mode, w, z, seed, range(n_perms), with_bound=True)
    with np.errstate(invalid="ignore"):
        mean = sims.mean(axis=0) if n_perms else np.full(x.shape[1], np.nan)
        var = sims.var(axis=0) if n_perms else np.full(x.shape[1], np.nan)
    return {"stat": statistic(mode, w, z), "bound": bound(mode, w, z), "sims": sims, "sims_bound": sb,
            "perm_mean": mean, "perm_var": var, "s012": np.array(weight_sums(w)), "w": w}


def randomisation_variance(mode: str, w: sp.spmatrix, z) -> np.ndarray:
    """Variance of I / C under the randomisation assumption (Cliff & Ord 1981; PySAL esda's VI_rand / VC_rand), per
    column of the centred values z [n, F]."""
    z = np.asarray(z, dtype=np.float64)
    n = float(z.shape[0])
    s0, s1, s2 = weight_sums(w)
    m2 = (z ** 2).sum(axis=0) / n
    k = ((z ** 4).sum(axis=0) / n) / (m2 * m2)
    if mode == "moran":
        e = -1.0 / (n - 1.0)
        a = n * ((n * n - 3 * n + 3) * s1 - n * s2 + 3 * s0 * s0)
        b = k * ((n * n - n) * s1 - 2 * n * s2 + 6 * s0 * s0)
        return (a - b) / ((n - 1) * (n - 2) * (n - 3) * s0 * s0) - e * e
    a = (n - 1) * s1 * (n * n - 3 * n + 3 - (n - 1) * k)
    b = 0.25 * (n - 1) * s2 * (n * n + 3 * n - 6 - (n * n - n + 2) * k)
    c = s0 * s0 * (n * n - 3 - (n - 1) ** 2 * k)
    return (a - b + c) / (n * (n - 2) * (n - 3) * s0 * s0)
