"""Oracle of K15 (pg_nhood_enrichment): the keyed Feistel permutations restated in numpy uint64 arithmetic, the
per-labelling type-pair counts (bincount), and the statistics in Python integers, each output rounded once.

The definition is the one include/pathgraph.h states: pi_p is 8 Feistel rounds over 4^h >= max(n, 4) values split
into two h-bit halves, round function splitmix64(R ^ k_{p,r}) & (2^h - 1), k_{p,r} = splitmix64(seed ^ (64 p + r)),
cycle-walked into [0, n)."""
from __future__ import annotations

import math

import numpy as np

ROUNDS = 8
_U = np.uint64


def splitmix64(x):
    with np.errstate(over="ignore"):
        z = np.asarray(x, dtype=np.uint64) + _U(0x9E3779B97F4A7C15)
        z = (z ^ (z >> _U(30))) * _U(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> _U(27))) * _U(0x94D049BB133111EB)
        return z ^ (z >> _U(31))


def half_bits(n: int) -> int:
    h = 1
    while (1 << (2 * h)) < n:
        h += 1
    return h


def permutations(n: int, seed: int, perms) -> np.ndarray:
    """int64 [len(perms), n]: row k is pi_{perms[k]} (node i takes the label of node pi(i))."""
    perms = np.asarray(perms, dtype=np.uint64).reshape(-1)
    h = half_bits(n)
    mask, sh = _U((1 << h) - 1), _U(h)
    r = np.arange(ROUNDS, dtype=np.uint64)
    with np.errstate(over="ignore"):
        keys = splitmix64(_U(seed) ^ (_U(64) * perms[:, None] + r[None, :]))  # [P, ROUNDS]
    out = np.empty((len(perms), n), dtype=np.uint64)
    cur = np.broadcast_to(np.arange(n, dtype=np.uint64), out.shape).copy()
    todo = np.ones(out.shape, dtype=bool)
    while todo.any():
        rows, cols = np.nonzero(todo)
        v = cur[rows, cols]
        lo, ro = v >> sh, v & mask
        for k in range(ROUNDS):
            f = splitmix64(ro ^ keys[rows, k]) & mask
            lo, ro = ro, lo ^ f
        v = (lo << sh) | ro
        cur[rows, cols] = v
        ok = v < _U(n)
        out[rows[ok], cols[ok]] = v[ok]
        todo[rows[ok], cols[ok]] = False
    return out.astype(np.int64)


def labels(types, n_types: int) -> np.ndarray:
    """int64 labels with everything outside 1..n_types as 0."""
    t = np.asarray(types, dtype=np.int64)
    return np.where((t >= 1) & (t <= n_types), t, 0)


def pair_counts(lab, edges, n_types: int) -> np.ndarray:
    """int64 [L, T, T] directed counts of labellings lab [L, n]: each edge row (i, j) adds (t_i, t_j) and (t_j, t_i);
    rows with an id outside [0, n) or a label 0 count nowhere."""
    lab = np.atleast_2d(lab)
    n_lab, n = lab.shape
    t2 = n_types * n_types
    e = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
    e = e[(e >= 0).all(axis=1) & (e < n).all(axis=1)]
    a, b = lab[:, e[:, 0]], lab[:, e[:, 1]]
    ok = (a > 0) & (b > 0)
    base = (np.arange(n_lab, dtype=np.int64) * t2)[:, None]
    ab = (base + (a - 1) * n_types + (b - 1))[ok]
    ba = (base + (b - 1) * n_types + (a - 1))[ok]
    c = np.bincount(ab, minlength=n_lab * t2) + np.bincount(ba, minlength=n_lab * t2)
    return c.reshape(n_lab, n_types, n_types).astype(np.int64)


def permuted_counts(edges, types, n_types: int, seed: int, perms, chunk: int = 64) -> np.ndarray:
    """int64 [len(perms), T, T]: pair_counts under pi_p for every p in perms."""
    lab = labels(types, n_types)
    n = lab.shape[0]
    perms = list(perms)
    out = np.zeros((len(perms), n_types, n_types), dtype=np.int64)
    if n == 0:
        return out
    step = max(1, min(chunk, (1 << 22) // max(n, len(np.asarray(edges).reshape(-1, 2)))))
    for s in range(0, len(perms), step):
        pi = permutations(n, seed, perms[s:s + step])
        out[s:s + step] = pair_counts(lab[pi], edges, n_types)
    return out


def statistics(count, perm_counts) -> dict:
    """count [T,T] and per-permutation counts [P,T,T] -> zscore / perm_mean / perm_std float64 [T,T], from the exact
    integers S1 = sum c_p and S2 = sum c_p^2, each converted to float once (the zscore is NaN / +-inf where
    P S2 - S1^2 = 0)."""
    pc = np.asarray(perm_counts)
    p = pc.shape[0]
    t = pc.shape[1:]
    z, mean, std = (np.empty(t, dtype=np.float64) for _ in range(3))
    for idx in np.ndindex(*t):
        col = [int(v) for v in pc[(slice(None),) + idx]]
        s1, s2 = sum(col), sum(v * v for v in col)
        sd = math.sqrt(float(p * s2 - s1 * s1))
        mean[idx] = s1 / p
        std[idx] = sd / p
        with np.errstate(divide="ignore", invalid="ignore"):
            z[idx] = np.float64(float(p * int(count[idx]) - s1)) / np.float64(sd)
    return {"count": np.asarray(count, dtype=np.int64), "zscore": z, "perm_mean": mean, "perm_std": std}


def nhood_enrichment(edges, types, n_types: int = 5, n_perms: int = 1000, seed: int = 0) -> dict:
    """The four outputs of pg_nhood_enrichment."""
    lab = labels(types, n_types)
    count = pair_counts(lab[None, :], edges, n_types)[0]
    return statistics(count, permuted_counts(edges, types, n_types, seed, range(n_perms)))
