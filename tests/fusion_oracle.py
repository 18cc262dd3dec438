"""numpy restatement of depth-map fusion (include/ldp_b200.h: ldp_depth_colors, ldp_fuse_depth_maps).

The per-view test is tests/consistency_oracle.py's (the verdicts of ``check(detail=True)``), so pinhole views are the kernels'
bit for bit.  The sums are explicit loops over the views in ascending order (np.sum is pairwise beyond 8 terms), each term
added in f64, divided once and rounded to f32 once, as the kernels do."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from tests import consistency_oracle as CO


@dataclass
class FusionOracle:
    source: np.ndarray          # int64 [m], ascending
    xyz: np.ndarray             # f32 [m, 3]
    rgb: np.ndarray             # f32 [m, 3]
    err: np.ndarray             # f32 [m]
    n_views: np.ndarray         # int32 [m]
    n_consistent: np.ndarray    # int32 [m]
    kept: np.ndarray            # bool [V, H * W]: pass 1
    n_consistent_map: np.ndarray  # int32 [V, H * W]: pass 1's count (0 where the depth is not finite)
    edge: np.ndarray            # f64 [V, H * W]: consistency_oracle's edge distance of each tested pixel (inf elsewhere)


def map_pixel(P, scales, lens, xyz: np.ndarray) -> np.ndarray:
    """Step 2 of the consistency rule: the map pixel (floor(u * ax), floor(v * ay)) of each point in one view, f64, with
    consistency_oracle's projection and lens model (only meaningful where the view's verdict is not NONE)."""
    q0, q1, z = CO.project(P, xyz)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        u, w = q0 / z, q1 / z
        if lens is not None and lens[0] != 0:
            fx, fy, cx, cy = (float(np.float32(c)) for c in lens[2:6])
            xd, yd = CO.lens_distort(lens[0], lens[1], (u - cx) / fx, (w - cy) / fy)
            u, w = fx * xd + cx, fy * yd + cy
        mx, my = np.floor(u * scales[0]), np.floor(w * scales[1])
    return mx, my


def fuse(depth: np.ndarray, xyz: np.ndarray, rgb: np.ndarray, err: np.ndarray, P: np.ndarray, scales: np.ndarray, *,
         lenses: Optional[Sequence[Optional[tuple]]] = None, rel_tol: float = 0.01, min_views: int = 1,
         max_violations: int = 0) -> FusionOracle:
    """depth f32 [V, H, W]; xyz, rgb f32 [V, H, W, 3]; err f32 [V, H, W]; P f32 [V, 12]; scales f64 [V, 2]; lenses as
    consistency_oracle.check takes them."""
    V, H, W = depth.shape
    N = H * W
    xyz_f = np.asarray(xyz, np.float32).reshape(V, N, 3)
    rgb_f = np.asarray(rgb, np.float32).reshape(V, N, 3)
    err_f = np.asarray(err, np.float32).reshape(V, N)
    pts = [np.nonzero(np.isfinite(depth[v].reshape(-1)))[0] for v in range(V)]
    kept = np.zeros((V, N), bool)
    ncm = np.zeros((V, N), np.int32)
    edge = np.full((V, N), np.inf)
    verdicts, pixels = [], []
    for r in range(V):                                   # pass 1
        X = xyz_f[r, pts[r]]
        o = CO.check(X, depth, P, scales, owner=np.full(len(X), r), lenses=lenses, rel_tol=rel_tol, min_views=min_views,
                     max_violations=max_violations, detail=True)
        kept[r, pts[r][o.kept_idx]] = True
        ncm[r, pts[r]] = o.n_consistent
        edge[r, pts[r]] = o.edge
        verdicts.append(o.verdict)
        pix = np.zeros((len(X), V), np.int64)
        for v in range(V):
            mx, my = map_pixel(P[v], scales[v], None if lenses is None else lenses[v], X)
            cons = o.verdict[:, v] == CO.CONSISTENT
            pix[cons, v] = my[cons].astype(np.int64) * W + mx[cons].astype(np.int64)
        pixels.append(pix)
    src, out_xyz, out_rgb, out_err, out_nv, out_nc = [], [], [], [], [], []
    for r in range(V):                                   # pass 2
        sel = np.nonzero(kept[r, pts[r]])[0]             # kept pixels of view r, ascending
        ver, pix = verdicts[r][sel], pixels[r][sel]
        member = np.zeros((len(sel), V), bool)
        for v in range(V):
            if v == r:
                continue
            m = ver[:, v] == CO.CONSISTENT
            member[m, v] = kept[v, pix[m, v]]
        emitted = ~member[:, :r].any(axis=1)
        sel, pix, member = sel[emitted], pix[emitted], member[emitted]
        i = pts[r][sel]
        sx = xyz_f[r, i].astype(np.float64)              # the sums: the own pixel first, then members in ascending view order
        sc = rgb_f[r, i].astype(np.float64)
        cnt = np.zeros(len(i), np.int64)
        for v in range(r + 1, V):
            m = member[:, v]
            sx[m] = sx[m] + xyz_f[v, pix[m, v]].astype(np.float64)
            sc[m] = sc[m] + rgb_f[v, pix[m, v]].astype(np.float64)
            cnt[m] += 1
        d = (cnt + 1).astype(np.float64)[:, None]
        src.append(r * N + i.astype(np.int64))
        out_xyz.append((sx / d).astype(np.float32))
        out_rgb.append((sc / d).astype(np.float32))
        out_err.append(err_f[r, i])
        out_nv.append((cnt + 1).astype(np.int32))
        out_nc.append(ncm[r, i])
    cat = lambda parts, shape, dt: np.concatenate(parts) if parts else np.zeros(shape, dt)  # noqa: E731
    return FusionOracle(source=cat(src, (0,), np.int64), xyz=cat(out_xyz, (0, 3), np.float32), rgb=cat(out_rgb, (0, 3), np.float32),
                        err=cat(out_err, (0,), np.float32), n_views=cat(out_nv, (0,), np.int32),
                        n_consistent=cat(out_nc, (0,), np.int32), kept=kept, n_consistent_map=ncm, edge=edge)


def color_maps(flags: np.ndarray, warps: np.ndarray, image: np.ndarray, nn: int, w_match: int, h_match: int) -> np.ndarray:
    """The colour map of one view (ldp_depth_colors): flags u8 [H, W]; warps f32 [nn, H, W, 4]; image u8 [ih, iw, 3].
    The bilinear blend of core/pipeline.py:661-679 at the kept pixels' winner rows (f32 decode, f64 weights, clipped
    corners, acc / 255 rounded to f32); NaN elsewhere.  f32 [H, W, 3]."""
    H, W = flags.shape
    ih, iw = image.shape[:2]
    out = np.full((H, W, 3), np.nan, np.float32)
    f = flags.astype(np.int64)
    k = f >> 4
    sel = ((f & 4) != 0) & (k < nn)
    ys, xs = np.nonzero(sel)
    wv = warps[k[ys, xs], ys, xs]
    f32 = np.float32
    xA = ((wv[:, 0].astype(f32) + f32(1.0)) * f32(0.5)) * f32(w_match - 1)
    yA = ((wv[:, 1].astype(f32) + f32(1.0)) * f32(0.5)) * f32(h_match - 1)
    fx = (xA * f32(iw / w_match)).astype(f32)
    fy = (yA * f32(ih / h_match)).astype(f32)
    x0 = np.clip(np.clip(np.floor(fx), -1, iw).astype(np.int64), 0, iw - 1)
    y0 = np.clip(np.clip(np.floor(fy), -1, ih).astype(np.int64), 0, ih - 1)
    x1, y1 = np.minimum(x0 + 1, iw - 1), np.minimum(y0 + 1, ih - 1)
    dfx, dfy = fx.astype(np.float64), fy.astype(np.float64)
    ax, bx, ay, by = x1 - dfx, dfx - x0, y1 - dfy, dfy - y0
    img = image.astype(np.float64)
    acc = img[y0, x0] * (ax * ay)[:, None]
    acc = acc + img[y0, x1] * (bx * ay)[:, None]
    acc = acc + img[y1, x0] * (ax * by)[:, None]
    acc = acc + img[y1, x1] * (bx * by)[:, None]
    out[ys, xs] = (acc / 255.0).astype(np.float32)
    return out
