"""numpy restatement of the cross-view depth consistency rule (include/ldp_b200.h: ldp_depth_consistency).

Every product of two f32 values is exact in f64 and numpy does not contract, so the projection, the map pixel and the depth
test are the kernels' bit for bit on pinhole views.  The lens forward model is restated from the same formula; the kernels'
f64 arithmetic there may contract into FMAs, so ``edge`` reports how close each point's map coordinate came to a pixel edge."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

NONE, CONSISTENT, VIOLATION, OCCLUDED = 0, 1, 2, 3


@dataclass
class ConsistencyOracle:
    n_consistent: np.ndarray    # int32 [n]
    n_violations: np.ndarray    # int32 [n]
    kept_idx: np.ndarray        # int64 [m], ascending
    edge: np.ndarray            # f64 [n]: smallest distance of a map coordinate u * ax, v * ay (views in front) to an integer
    verdict: Optional[np.ndarray] = None   # uint8 [n, V] (detail=True): NONE, CONSISTENT, VIOLATION, OCCLUDED


def lens_distort(model: int, k: Sequence[float], x: np.ndarray, y: np.ndarray):
    """The forward lens of include/ldp_b200.h: ldp_lens (1 OpenCV, 2 fisheye), normalised coordinates, f64."""
    k = [float(c) for c in k]
    r2 = x * x + y * y
    if model == 2:
        r = np.sqrt(r2)
        th = np.arctan(r)
        t2 = th * th
        thd = th * (1.0 + t2 * (k[0] + t2 * (k[1] + t2 * (k[2] + t2 * k[3]))))
        with np.errstate(invalid="ignore", divide="ignore"):
            s = np.where(r > 0.0, thd / np.where(r > 0.0, r, 1.0), 1.0)
        return x * s, y * s
    radial = (1.0 + r2 * (k[0] + r2 * (k[1] + r2 * k[4]))) / (1.0 + r2 * (k[5] + r2 * (k[6] + r2 * k[7])))
    return (x * radial + 2.0 * k[2] * x * y + k[3] * (r2 + 2.0 * x * x),
            y * radial + k[2] * (r2 + 2.0 * y * y) + 2.0 * k[3] * x * y)


def project(P: np.ndarray, xyz: np.ndarray):
    """q_r = ((P[r,0] X + P[r,1] Y) + P[r,2] Z) + P[r,3] in f64 (P f32 [12] or [3, 4], xyz f32 [n, 3])."""
    P = np.asarray(P, dtype=np.float32).reshape(3, 4).astype(np.float64)
    X = np.asarray(xyz, dtype=np.float32).astype(np.float64)
    return [((P[r, 0] * X[:, 0] + P[r, 1] * X[:, 1]) + P[r, 2] * X[:, 2]) + P[r, 3] for r in range(3)]


def check(xyz: np.ndarray, maps: np.ndarray, P: np.ndarray, scales: np.ndarray, *, owner: Optional[np.ndarray] = None,
          lenses: Optional[Sequence[Optional[tuple]]] = None, rel_tol: float = 0.01, min_views: int = 1, max_violations: int = 0,
          detail: bool = False) -> ConsistencyOracle:
    """xyz f32 [n, 3]; maps f32 [V, H, W]; P f32 [V, 12]; scales f64 [V, 2] (engine.depth_map_scales); owner int [n] or
    None; lenses: per view None (pinhole) or (model, k[8], fx, fy, cx, cy) with the f32 intrinsics."""
    xyz = np.asarray(xyz, dtype=np.float32)
    n = xyz.shape[0]
    V, H, W = maps.shape
    nc = np.zeros(n, np.int32)
    nv = np.zeros(n, np.int32)
    edge = np.full(n, np.inf)
    verdict = np.zeros((n, V), np.uint8) if detail else None
    own = np.full(n, -1, np.int64) if owner is None else np.asarray(owner, dtype=np.int64)
    flat = maps.reshape(V, -1)
    for v in range(V):
        q0, q1, z = project(P[v], xyz)
        with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
            u, w = q0 / z, q1 / z
            L = lenses[v] if lenses is not None else None
            if L is not None and L[0] != 0:
                fx, fy, cx, cy = (float(np.float32(c)) for c in L[2:6])
                xd, yd = lens_distort(L[0], L[1], (u - cx) / fx, (w - cy) / fy)
                u, w = fx * xd + cx, fy * yd + cy
            mx, my = u * scales[v, 0], w * scales[v, 1]
            fx_, fy_ = np.floor(mx), np.floor(my)
        sees = (z > 0.0) & (own != v)
        e = np.minimum(np.abs(mx - np.round(mx)), np.abs(my - np.round(my)))
        edge = np.where(sees & np.isfinite(e), np.minimum(edge, e), edge)
        inside = sees & (fx_ >= 0) & (fx_ < W) & (fy_ >= 0) & (fy_ < H)
        idx = np.nonzero(inside)[0]
        D = flat[v][fy_[idx].astype(np.int64) * W + fx_[idx].astype(np.int64)].astype(np.float64)
        ok = D > 0.0
        idx, D = idx[ok], D[ok]
        d = z[idx] - D
        t = rel_tol * D
        cons = np.abs(d) <= t
        viol = ~cons & (d < -t)
        nc[idx[cons]] += 1
        nv[idx[viol]] += 1
        if detail:
            verdict[idx, v] = OCCLUDED
            verdict[idx[cons], v] = CONSISTENT
            verdict[idx[viol], v] = VIOLATION
    kept = np.nonzero((nc >= min_views) & (nv <= max_violations))[0].astype(np.int64)
    return ConsistencyOracle(nc, nv, kept, edge, verdict)


def lens_tuple(cam) -> Optional[tuple]:
    """(model, k[8], fx, fy, cx, cy) of a CameraRecord, as engine.lens_of fills ldp_lens; None for a pinhole."""
    from lichtfeld_densification_plugin_b200.engine import lens_of
    L = lens_of(cam)
    if L.model == 0:
        return None
    return (int(L.model), [float(c) for c in L.k], L.fx, L.fy, L.cx, L.cy)


def sphere_map(cam, H: int, W: int, w_match: int, h_match: int, radius: float) -> np.ndarray:
    """f32 [H, W] depth map of a pinhole camera looking at the sphere of ``radius`` about the origin, in f64: camera z of the
    first hit of the ray through each map pixel's centre (u = (x + 1/2) / W * (w_match - 1) * width / w_match); NaN where the
    ray misses."""
    xs = (np.arange(W) + 0.5) / W * (w_match - 1) * (cam.width / w_match)
    ys = (np.arange(H) + 0.5) / H * (h_match - 1) * (cam.height / h_match)
    u, v = np.meshgrid(xs, ys)
    K = np.asarray(cam.K, np.float64)
    ray = np.stack([(u - K[0, 2]) / K[0, 0], (v - K[1, 2]) / K[1, 1], np.ones_like(u)], -1)      # camera, z = 1
    d = ray @ np.asarray(cam.R, np.float64)                                                     # world direction
    C = np.asarray(cam.C, np.float64).reshape(3)
    a, b, c = (d * d).sum(-1), d @ C, C @ C - radius * radius
    disc = b * b - a * c
    with np.errstate(invalid="ignore"):
        t = (-b - np.sqrt(disc)) / a
    return np.where(disc >= 0, t, np.nan).astype(np.float32)
