"""numpy restatement of the normal maps and the oriented fusion (include/ldp_b200.h: ldp_depth_normals,
ldp_fuse_depth_maps_oriented).

* ``window_neighbors``   the depth-continuous window of every pixel, in the rule's row-major order
* ``depth_normals``      the normals of one view's map: the windows grouped by their size k, each group through
                         ``tests/normals_oracle.normals_from_neighbors`` (covariance in the stated order, eigh, the undefined
                         rule, canonical sign, orientation)
* ``fuse_oriented``      the oriented fusion rule on top of ``tests/fusion_oracle`` and ``tests/consistency_oracle``: the
                         depth verdicts are theirs, the normal test and the sums are explicit loops in ascending view order,
                         each term added in f64 and each result rounded once, as the kernels do
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from tests import consistency_oracle as CO
from tests import fusion_oracle as FO
from tests import normals_oracle as NO


def window_neighbors(depth: np.ndarray, radius: int, rel_tol: float):
    """(idx int64 [H*W, (2r+1)^2], valid bool [H*W, (2r+1)^2]) for a map f32 [H, W]: entry j of pixel p is the flat index
    of the window pixel (dy, dx) = divmod(j, 2r + 1) - r, valid iff it lies in the map, has a finite depth and
    |D_q - D_p| <= rel_tol * D_p in f64 (each operation rounded once).  Rows of pixels without a depth are all invalid."""
    H, W = depth.shape
    D = np.asarray(depth, np.float32).astype(np.float64)
    ys, xs = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    ys, xs = ys.reshape(-1), xs.reshape(-1)
    Dp = D.reshape(-1)
    t = np.float64(rel_tol) * Dp
    idx, valid = [], []
    for dy in range(-radius, radius + 1):
        for dx in range(-radius, radius + 1):
            qy, qx = ys + dy, xs + dx
            inside = (qy >= 0) & (qy < H) & (qx >= 0) & (qx < W)
            q = np.where(inside, qy * W + qx, 0)
            Dq = np.where(inside, D.reshape(-1)[q], np.nan)
            with np.errstate(invalid="ignore"):
                ok = inside & np.isfinite(Dq) & np.isfinite(Dp) & (np.abs(Dq - Dp) <= t)
            idx.append(q)
            valid.append(ok)
    return np.stack(idx, 1), np.stack(valid, 1)


@dataclass
class DepthNormalsOracle:
    normals: np.ndarray         # f64 [H, W, 3], NaN where there is no depth or no normal
    curvature: np.ndarray       # f64 [H, W], NaN likewise
    undefined: np.ndarray       # bool [H, W]: a depth and no normal
    eigenvalues: np.ndarray     # f64 [H, W, 3] ascending (0 where k < 3 or there is no depth)
    k: np.ndarray               # int [H, W]: window size (0 where there is no depth)


def depth_normals(depth: np.ndarray, xyz: np.ndarray, centre, radius: int = 2, rel_tol: float = 0.05) -> DepthNormalsOracle:
    """One view: depth f32 [H, W], xyz f32 [H, W, 3], centre f32 [3] (the camera centre)."""
    H, W = depth.shape
    n = H * W
    x = np.asarray(xyz, np.float32).reshape(n, 3)
    idx, valid = window_neighbors(depth, radius, rel_tol)
    k = valid.sum(1)
    has = np.isfinite(np.asarray(depth, np.float32).reshape(-1))
    nrm = np.full((n, 3), np.nan)
    curv = np.full((n,), np.nan)
    und = np.zeros((n,), bool)
    lam = np.zeros((n, 3))
    cen = np.asarray(centre, np.float32).reshape(1, 3)
    for kk in np.unique(k[has]):
        q = np.nonzero(has & (k == kk))[0]
        rows = idx[q][valid[q]].reshape(len(q), kk)        # row-major window order kept by the boolean selection
        # the queries first: normals_from_neighbors orients row i from xyz row i
        ext = np.concatenate([x[q], x], 0)
        rn, rc, ru, rl = NO.normals_from_neighbors(ext, rows + len(q), centers=cen, center_idx=np.zeros(len(q), np.int64))
        nrm[q] = np.where(ru[:, None], np.nan, rn)
        curv[q] = rc
        und[q] = ru
        lam[q] = rl
    return DepthNormalsOracle(normals=nrm.reshape(H, W, 3), curvature=curv.reshape(H, W), undefined=und.reshape(H, W),
                              eigenvalues=lam.reshape(H, W, 3), k=np.where(has, k, 0).reshape(H, W))


def _dot(n: np.ndarray, m: np.ndarray) -> np.ndarray:
    """((n0 m0 + n1 m1) + n2 m2) in f64 of f32 rows: the products are exact, each sum rounded once."""
    n, m = np.asarray(n, np.float32).astype(np.float64), np.asarray(m, np.float32).astype(np.float64)
    return (n[:, 0] * m[:, 0] + n[:, 1] * m[:, 1]) + n[:, 2] * m[:, 2]


@dataclass
class OrientedFusionOracle(FO.FusionOracle):
    normals: Optional[np.ndarray] = None     # f32 [m, 3]


def fuse_oriented(depth: np.ndarray, xyz: np.ndarray, rgb: np.ndarray, err: np.ndarray, normals: np.ndarray, P: np.ndarray,
                  scales: np.ndarray, *, cos_max: float, lenses: Optional[Sequence[Optional[tuple]]] = None,
                  rel_tol: float = 0.01, min_views: int = 1, max_violations: int = 0) -> OrientedFusionOracle:
    """As ``fusion_oracle.fuse`` with normals f32 [V, H, W, 3] and the normal test at ``cos_max``."""
    V, H, W = depth.shape
    N = H * W
    xyz_f = np.asarray(xyz, np.float32).reshape(V, N, 3)
    rgb_f = np.asarray(rgb, np.float32).reshape(V, N, 3)
    err_f = np.asarray(err, np.float32).reshape(V, N)
    nrm_f = np.asarray(normals, np.float32).reshape(V, N, 3)
    nrm_ok = np.isfinite(nrm_f).all(2)
    pts = [np.nonzero(np.isfinite(depth[v].reshape(-1)))[0] for v in range(V)]
    kept = np.zeros((V, N), bool)
    ncm = np.zeros((V, N), np.int32)
    edge = np.full((V, N), np.inf)
    agrees, pixels = [], []
    for r in range(V):                                   # pass 1
        X = xyz_f[r, pts[r]]
        own = nrm_f[r, pts[r]]
        own_ok = nrm_ok[r, pts[r]]
        o = CO.check(X, depth, P, scales, owner=np.full(len(X), r), lenses=lenses, rel_tol=rel_tol, min_views=0,
                     max_violations=1 << 30, detail=True)
        edge[r, pts[r]] = o.edge
        pix = np.zeros((len(X), V), np.int64)
        agree = np.zeros((len(X), V), bool)
        for v in range(V):
            mx, my = FO.map_pixel(P[v], scales[v], None if lenses is None else lenses[v], X)
            cons = o.verdict[:, v] == CO.CONSISTENT
            pix[cons, v] = my[cons].astype(np.int64) * W + mx[cons].astype(np.int64)
            c = np.nonzero(cons)[0]
            m = nrm_f[v, pix[c, v]]
            with np.errstate(invalid="ignore"):
                agree[c, v] = nrm_ok[v, pix[c, v]] & (_dot(own[c], m) >= cos_max)
        agree &= own_ok[:, None]
        nc = agree.sum(1).astype(np.int32)
        nv = (o.verdict == CO.VIOLATION).sum(1)
        kept[r, pts[r]] = own_ok & (nc >= min_views) & (nv <= max_violations)
        ncm[r, pts[r]] = nc
        agrees.append(agree)
        pixels.append(pix)
    src, out_xyz, out_rgb, out_nrm, out_err, out_nv, out_nc = [], [], [], [], [], [], []
    for r in range(V):                                   # pass 2
        sel = np.nonzero(kept[r, pts[r]])[0]
        ag, pix = agrees[r][sel], pixels[r][sel]
        member = np.zeros((len(sel), V), bool)
        for v in range(V):
            if v == r:
                continue
            m = ag[:, v]
            member[m, v] = kept[v, pix[m, v]]
        emitted = ~member[:, :r].any(axis=1)
        sel, pix, member = sel[emitted], pix[emitted], member[emitted]
        i = pts[r][sel]
        sx = xyz_f[r, i].astype(np.float64)
        sc = rgb_f[r, i].astype(np.float64)
        sn = nrm_f[r, i].astype(np.float64)
        cnt = np.zeros(len(i), np.int64)
        for v in range(r + 1, V):
            m = member[:, v]
            sx[m] = sx[m] + xyz_f[v, pix[m, v]].astype(np.float64)
            sc[m] = sc[m] + rgb_f[v, pix[m, v]].astype(np.float64)
            sn[m] = sn[m] + nrm_f[v, pix[m, v]].astype(np.float64)
            cnt[m] += 1
        d = (cnt + 1).astype(np.float64)[:, None]
        length = np.sqrt((sn[:, 0] * sn[:, 0] + sn[:, 1] * sn[:, 1]) + sn[:, 2] * sn[:, 2])[:, None]
        src.append(r * N + i.astype(np.int64))
        out_xyz.append((sx / d).astype(np.float32))
        out_rgb.append((sc / d).astype(np.float32))
        out_nrm.append((sn / length).astype(np.float32))
        out_err.append(err_f[r, i])
        out_nv.append((cnt + 1).astype(np.int32))
        out_nc.append(ncm[r, i])
    cat = lambda parts, shape, dt: np.concatenate(parts) if parts else np.zeros(shape, dt)  # noqa: E731
    return OrientedFusionOracle(source=cat(src, (0,), np.int64), xyz=cat(out_xyz, (0, 3), np.float32),
                                rgb=cat(out_rgb, (0, 3), np.float32), err=cat(out_err, (0,), np.float32),
                                n_views=cat(out_nv, (0,), np.int32), n_consistent=cat(out_nc, (0,), np.int32), kept=kept,
                                n_consistent_map=ncm, edge=edge, normals=cat(out_nrm, (0, 3), np.float32))
