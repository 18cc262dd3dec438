"""Numpy restatement of the statistical outlier rule of include/ldp_b200.h (Open3D's RemoveStatisticalOutliers, restated;
parity with Open3D itself is unpinned), with the device's fixed order of the two threshold sums.

* ``mean_distances``        chunked brute-force k-NN, the exact f64 distance formula: the reference for the kernel's ``m_i``
* ``mean_distances_exact``  the same values, with scipy's cKDTree proposing candidates; rows whose k-th distance ties
                            beyond the candidates fall back to brute force, so the result equals ``mean_distances``
* ``mean_distances_kdtree`` distances recomputed from cKDTree's own neighbour indices (equal within float rounding)
* ``threshold_stats`` / ``statistical_outliers``  steps 3 and 4
"""
from __future__ import annotations

import numpy as np

CHUNK = 256          # consecutive points per first-stage partial sum
FINAL = 1024         # second-stage threads


def _d2(q: np.ndarray, x: np.ndarray) -> np.ndarray:
    """(dx*dx + dy*dy) + dz*dz in f64 for every (query row, point) pair; numpy does not contract to FMA."""
    dx = x[None, :, 0] - q[:, None, 0]
    dy = x[None, :, 1] - q[:, None, 1]
    dz = x[None, :, 2] - q[:, None, 2]
    return (dx * dx + dy * dy) + dz * dz


def means_from_sorted_d2(d2_sorted: np.ndarray, k: int) -> np.ndarray:
    """m_i from the ascending d^2 rows: sqrt, then the first k added sequentially, divided by k."""
    d = np.sqrt(d2_sorted[:, :k])
    s = np.zeros(d.shape[0], np.float64)
    for j in range(k):                    # sequential, ascending
        s = s + d[:, j]
    return s / np.float64(k)


def sorted_knn_d2(xyz: np.ndarray, k: int, rows=None, chunk: int = 512) -> np.ndarray:
    """Brute force: the k smallest d^2 of every query row (ascending), the point itself included."""
    x = np.asarray(xyz, np.float32).astype(np.float64)
    rows = np.arange(x.shape[0]) if rows is None else np.asarray(rows)
    k = min(k, x.shape[0])
    out = np.empty((rows.shape[0], k), np.float64)
    for a in range(0, rows.shape[0], chunk):
        d2 = _d2(x[rows[a:a + chunk]], x)
        part = np.partition(d2, k - 1, axis=1)[:, :k] if k < x.shape[0] else d2
        out[a:a + chunk] = np.sort(part, axis=1)
    return out


def mean_distances(xyz: np.ndarray, k: int) -> np.ndarray:
    n = int(np.asarray(xyz).shape[0])
    if n == 0:
        return np.zeros((0,), np.float64)
    return means_from_sorted_d2(sorted_knn_d2(xyz, k), min(k, n))


def mean_distances_exact(xyz: np.ndarray, k: int, extra: int = 16) -> np.ndarray:
    """``mean_distances`` without the quadratic cost on clouds without massive ties."""
    n = int(np.asarray(xyz).shape[0])
    if n == 0:
        return np.zeros((0,), np.float64)
    return means_from_sorted_d2(sorted_knn_d2_exact(xyz, k, extra), min(k, n))


def sorted_knn_d2_exact(xyz: np.ndarray, k: int, extra: int = 16) -> np.ndarray:
    """``sorted_knn_d2`` (n >= 1), with cKDTree proposing the candidates."""
    from scipy.spatial import cKDTree
    x = np.asarray(xyz, np.float32).astype(np.float64)
    n = x.shape[0]
    k = min(k, n)
    kq = min(n, k + extra)
    if kq == n:
        return sorted_knn_d2(xyz, k)
    dist, idx = cKDTree(x).query(x, k=kq)
    dist, idx = dist.reshape(n, kq), idx.reshape(n, kq)
    # every point outside the candidates is at least dist[:, -1] away (up to the tree's rounding): the candidates hold
    # the k nearest when that is clearly beyond the k-th candidate distance
    ok = dist[:, -1] > dist[:, k - 1] * (1 + 1e-9) + 1e-300
    dx, dy, dz = (x[idx, c] - x[:, None, c] for c in range(3))
    d2 = (dx * dx + dy * dy) + dz * dz
    d2 = np.sort(d2, axis=1)[:, :k]
    bad = np.nonzero(~ok)[0]
    if bad.size:
        d2[bad] = sorted_knn_d2(xyz, k, rows=bad)
    return d2


def mean_distances_kdtree(xyz: np.ndarray, k: int, workers: int = -1) -> np.ndarray:
    """m_i from cKDTree's k neighbour indices, distances recomputed with the exact formula (ties may pick other points)."""
    from scipy.spatial import cKDTree
    x = np.asarray(xyz, np.float32).astype(np.float64)
    n = x.shape[0]
    k = min(k, n)
    _, idx = cKDTree(x).query(x, k=k, workers=workers)
    idx = idx.reshape(n, k)
    out = np.empty((n,), np.float64)
    for a in range(0, n, 1 << 18):
        xi = x[a:a + (1 << 18)]
        dx, dy, dz = (x[idx[a:a + (1 << 18)], c] - xi[:, None, c] for c in range(3))
        out[a:a + (1 << 18)] = means_from_sorted_d2(np.sort((dx * dx + dy * dy) + dz * dz, axis=1), k)
    return out


def fixed_order_sum(terms: np.ndarray) -> np.float64:
    """The device's order: sequential sums of CHUNK consecutive terms; thread t of FINAL sums partials t, t + FINAL, ...
    sequentially; then v[t] += v[t + s] for s = FINAL/2, ..., 1.  Zero padding changes nothing (x + 0.0 == x)."""
    t = np.asarray(terms, np.float64)
    n_part = max(1, -(-t.size // CHUNK))
    t = np.concatenate([t, np.zeros(n_part * CHUNK - t.size)]).reshape(n_part, CHUNK)
    part = np.cumsum(t, axis=1)[:, -1]
    rows = -(-n_part // FINAL)
    part = np.concatenate([part, np.zeros(rows * FINAL - n_part)]).reshape(rows, FINAL)
    v = np.cumsum(part, axis=0)[-1].copy()
    s = FINAL // 2
    while s >= 1:
        v[:s] = v[:s] + v[s:2 * s]
        s //= 2
    return np.float64(v[0])


def threshold_stats(m: np.ndarray, std_ratio: float):
    """(mean, std, threshold) of step 3."""
    m = np.asarray(m, np.float64)
    n = m.size
    pos = m > 0
    with np.errstate(invalid="ignore", divide="ignore"):
        mean = fixed_order_sum(np.where(pos, m, 0.0)) / np.float64(n)
        dev = np.where(pos, m - mean, 0.0)
        q = fixed_order_sum(dev * dev)
        std = np.sqrt(q / np.float64(n - 1))
        thr = mean + np.float64(std_ratio) * std
    return np.float64(mean), np.float64(std), np.float64(thr)


def statistical_outliers(xyz: np.ndarray, nb_neighbors: int, std_ratio: float, means=None):
    """(kept indices ascending, m, (mean, std, threshold))."""
    if not 1 <= nb_neighbors <= 64 or not std_ratio > 0:
        raise ValueError("nb_neighbors must lie in [1, 64] and std_ratio must be positive")
    x = np.asarray(xyz, np.float32)
    if not np.isfinite(x).all():
        raise ValueError("a coordinate is not finite")
    if x.shape[0] == 0:
        return np.zeros((0,), np.int64), np.zeros((0,), np.float64), (np.nan, np.nan, np.nan)
    m = mean_distances(x, nb_neighbors) if means is None else means
    st = threshold_stats(m, std_ratio)
    with np.errstate(invalid="ignore"):
        keep = np.nonzero((m > 0) & (m < st[2]))[0].astype(np.int64)
    return keep, m, st


# ---- test clouds ---------------------------------------------------------------------------------------------------------
def sphere_with_floaters(n: int, seed: int = 0, noise: float = 0.002, floater_frac: float = 0.01):
    """A noisy unit sphere plus uniform floaters in its bounding box; returns (xyz f32, is_floater)."""
    rng = np.random.default_rng(seed)
    nf = int(round(n * floater_frac))
    ns = n - nf
    v = rng.normal(size=(ns, 3))
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    v *= 1.0 + noise * rng.normal(size=(ns, 1))
    f = rng.uniform(-1.0, 1.0, size=(nf, 3))
    xyz = np.concatenate([v, f]).astype(np.float32)
    is_f = np.concatenate([np.zeros(ns, bool), np.ones(nf, bool)])
    perm = rng.permutation(n)
    return xyz[perm], is_f[perm]


def make_cloud(kind: str, n: int, seed: int = 0) -> np.ndarray:
    rng = np.random.default_rng(seed)
    if kind == "cube":
        return rng.uniform(-1, 1, size=(n, 3)).astype(np.float32)
    if kind == "sphere_floaters":
        return sphere_with_floaters(n, seed)[0]
    if kind == "plane":
        p = rng.uniform(-2, 2, size=(n, 3))
        p[:, 2] = 0.5
        return p.astype(np.float32)
    if kind == "lattice":
        s = int(np.ceil(n ** (1 / 3)))
        g = np.stack(np.meshgrid(np.arange(s), np.arange(s), np.arange(s), indexing="ij"), -1).reshape(-1, 3)
        return g[rng.permutation(g.shape[0])[:n]].astype(np.float32)
    if kind == "duplicates":
        centres = rng.uniform(-1, 1, size=(max(1, n // 400) + 1, 3))
        lab = rng.integers(0, centres.shape[0], size=n)
        p = centres[lab]
        jitter = rng.random(n) < 0.3                          # 70 % exact duplicates of their cluster centre
        p[jitter] += 0.01 * rng.normal(size=(int(jitter.sum()), 3))
        return p.astype(np.float32)
    if kind == "line":
        t = rng.uniform(0, 10, size=n)
        return np.stack([t, 0.5 * t + 1e-4 * rng.normal(size=n), np.full(n, -3.0)], -1).astype(np.float32)
    if kind == "two_clusters":
        p = rng.normal(size=(n, 3))
        p[: n // 2, 0] += 1e6
        return p.astype(np.float32)
    raise ValueError(kind)


CLOUDS = ("cube", "sphere_floaters", "plane", "lattice", "duplicates", "line", "two_clusters")
