"""Numpy restatement of the oriented-normal rule of include/ldp_b200.h (ldp_estimate_normals).

* ``knn_lex``              brute force: the k_eff points with the smallest (d^2, index) of every query row, ascending
* ``knn_lex_exact``        the same rows, with scipy's cKDTree proposing candidates; rows whose k-th distance ties beyond
                           the candidates fall back to brute force, so the result equals ``knn_lex``
* ``normals_from_neighbors``  covariance in the stated order, ``numpy.linalg.eigh``, the undefined rule, canonical sign,
                           orientation and curvature
* ``estimate_normals``     both steps
"""
from __future__ import annotations

import numpy as np

from tests.outlier_oracle import _d2

LINE = 1e-12         # lambda1 <= LINE * lambda2: the plane is not determined


def _lex_rows(d2: np.ndarray, cols: np.ndarray, k: int) -> np.ndarray:
    """Per row of d2 [m, c] (candidate indices cols [m, c] or [c]): the k candidates with the smallest (d^2, index)."""
    cols = np.broadcast_to(cols, d2.shape)
    order = np.lexsort((cols, d2), axis=1)[:, :k]
    return np.take_along_axis(cols, order, axis=1)


def knn_lex(xyz: np.ndarray, k: int, rows=None, chunk: int = 256) -> np.ndarray:
    """int64 [m, k_eff]: brute force over every point; ties at the k-th d^2 are taken by ascending index."""
    x = np.asarray(xyz, np.float32).astype(np.float64)
    n = x.shape[0]
    rows = np.arange(n) if rows is None else np.asarray(rows)
    k = min(k, n)
    out = np.empty((rows.shape[0], k), np.int64)
    all_idx = np.arange(n)
    for a in range(0, rows.shape[0], chunk):
        d2 = _d2(x[rows[a:a + chunk]], x)
        if k == n:
            out[a:a + chunk] = _lex_rows(d2, all_idx, k)
            continue
        kth = np.partition(d2, k - 1, axis=1)[:, k - 1]
        r, c = np.nonzero(d2 <= kth[:, None])                 # every candidate, ties at the k-th value included
        o = np.lexsort((c, d2[r, c], r))                       # by row, then (d^2, index)
        r, c = r[o], c[o]
        start = np.searchsorted(r, np.arange(d2.shape[0]))
        out[a:a + chunk] = c[start[:, None] + np.arange(k)[None, :]]
    return out


def knn_lex_exact(xyz: np.ndarray, k: int, extra: int = 16, workers: int = -1) -> np.ndarray:
    """``knn_lex`` (n >= 1) without the quadratic cost on clouds without massive ties."""
    from scipy.spatial import cKDTree
    x = np.asarray(xyz, np.float32).astype(np.float64)
    n = x.shape[0]
    k = min(k, n)
    kq = min(n, k + extra)
    if kq == n:
        return knn_lex(xyz, k)
    dist, idx = cKDTree(x).query(x, k=kq, workers=workers)
    dist, idx = dist.reshape(n, kq), idx.reshape(n, kq)
    # every point outside the candidates is at least dist[:, -1] away (up to the tree's rounding): the candidates hold
    # every point tied with the k-th when that is clearly beyond the k-th candidate distance
    ok = dist[:, -1] > dist[:, k - 1] * (1 + 1e-9) + 1e-300
    out = np.empty((n, k), np.int64)
    step = 1 << 18
    for a in range(0, n, step):
        ia = idx[a:a + step]
        dx, dy, dz = (x[ia, c] - x[a:a + step, None, c] for c in range(3))
        out[a:a + step] = _lex_rows((dx * dx + dy * dy) + dz * dz, ia, k)
    bad = np.nonzero(~ok)[0]
    if bad.size:
        out[bad] = knn_lex(xyz, k, rows=bad)
    return out


def covariances(xyz: np.ndarray, idx: np.ndarray) -> np.ndarray:
    """f64 [m, 3, 3]: mu and C of the rule, sums sequential over the neighbours in the given order, no FMA."""
    x = np.asarray(xyz, np.float32).astype(np.float64)
    m, k = idx.shape
    p = x[idx]                                                 # [m, k, 3]
    s = np.zeros((m, 3))
    for j in range(k):
        s = s + p[:, j]
    mu = s / np.float64(k)
    d = p - mu[:, None, :]
    c = np.zeros((m, 6))
    pairs = ((0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2))
    for j in range(k):
        dj = d[:, j]
        c = c + np.stack([dj[:, a] * dj[:, b] for a, b in pairs], axis=1)
    c = c / np.float64(k)
    cov = np.empty((m, 3, 3))
    for e, (a, b) in enumerate(pairs):
        cov[:, a, b] = cov[:, b, a] = c[:, e]
    return cov


def normals_from_neighbors(xyz: np.ndarray, idx: np.ndarray, centers=None, center_idx=None, chunk: int = 1 << 18):
    """(normals f64 [m,3], curvature f64 [m], undefined bool [m], eigenvalues f64 [m,3]) for the query rows 0..m-1 of
    xyz with neighbourhoods idx [m, k_eff] (ascending (d^2, index))."""
    x = np.asarray(xyz, np.float32).astype(np.float64)
    m, k = idx.shape
    nrm = np.zeros((m, 3))
    curv = np.full((m,), np.nan)
    und = np.ones((m,), bool)
    lam = np.zeros((m, 3))
    if k < 3:
        return nrm, curv, und, lam
    for a in range(0, m, chunk):
        b = min(m, a + chunk)
        cov = covariances(xyz, idx[a:b])
        tr = (cov[:, 0, 0] + cov[:, 1, 1]) + cov[:, 2, 2]
        w, v = np.linalg.eigh(cov)
        lam[a:b] = w
        u = (tr == 0) | ~(w[:, 1] > LINE * w[:, 2])
        n = v[:, :, 0]
        n = n / np.linalg.norm(n, axis=1, keepdims=True)
        big = np.argmax(np.abs(n), axis=1)                     # first maximum: the lowest axis on ties
        sgn = np.where(n[np.arange(b - a), big] < 0, -1.0, 1.0)
        if centers is not None:
            cen = np.asarray(centers, np.float32).astype(np.float64)
            ci = np.zeros((b - a,), np.int64) if center_idx is None else np.asarray(center_idx)[a:b]
            dc = cen[ci] - x[a:b]
            dot = (n[:, 0] * dc[:, 0] + n[:, 1] * dc[:, 1]) + n[:, 2] * dc[:, 2]
            sgn = np.where(sgn * dot < 0, -sgn, sgn)
        n = n * sgn[:, None]
        with np.errstate(invalid="ignore", divide="ignore"):
            cv = w[:, 0] / ((w[:, 0] + w[:, 1]) + w[:, 2])
        nrm[a:b] = np.where(u[:, None], 0.0, n)
        curv[a:b] = np.where(u, np.nan, cv)
        und[a:b] = u
    return nrm, curv, und, lam


def estimate_normals(xyz: np.ndarray, k: int, centers=None, center_idx=None, exact_knn=knn_lex):
    """(neighbours int64 [n, k_eff], normals, curvature, undefined, eigenvalues)."""
    if not 3 <= k <= 64:
        raise ValueError("k must lie in [3, 64]")
    x = np.asarray(xyz, np.float32)
    if x.shape[0] == 0:
        return (np.zeros((0, 0), np.int64), np.zeros((0, 3)), np.zeros((0,)), np.zeros((0,), bool), np.zeros((0, 3)))
    idx = exact_knn(x, k)
    return (idx,) + normals_from_neighbors(x, idx, centers, center_idx)


def noisy_sphere(n: int, seed: int = 0, noise: float = 0.002) -> np.ndarray:
    """n points on the unit sphere, radius jittered by ``noise`` (no floaters)."""
    rng = np.random.default_rng(seed)
    v = rng.normal(size=(n, 3))
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    return (v * (1.0 + noise * rng.normal(size=(n, 1)))).astype(np.float32)


def angle(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """Angle in radians between the rows of a and b (both unit or nearly so)."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    c = np.sum(a * b, axis=1) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))
    # arctan2 of |a x b| and a . b keeps the precision near 0 that arccos loses
    s = np.linalg.norm(np.cross(a, b), axis=1) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))
    return np.arctan2(s, c)
