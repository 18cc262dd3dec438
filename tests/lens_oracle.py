"""TEST INFRASTRUCTURE ONLY -- numpy f64 restatement of the lens models of the device path (include/ldp_b200.h: ldp_lens).

The reference ignores lens distortion, so there is no reference behaviour to pin: this module states the models
(OpenCV rational, fisheye) and their inversion by the same rule as csrc/ldp_geometry.cu -- Newton's method from the
distorted point, the 2x2 analytic Jacobian for OpenCV, 1-D on theta for the fisheye, a step tolerance and an iteration cap
(below, shared with the kernel and checked against its source by tests/test_oracle_lens.py; the fisheye iteration starts at
min(r_d, pi/2 - 1e-6), as cv2.fisheye clamps its start) -- and is itself checked
against OpenCV's cv2.projectPoints / cv2.undistortPointsIter / cv2.fisheye.

``triangulate_ref_lens`` is oracle/densify_oracle.py's ``triangulate_ref`` with lens cameras: the observed pixels are
undistorted before the Sampson gate and the DLT, and a lens camera's reprojection error is measured in its distorted
image.  Everything else is the pinned oracle's own functions.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np

from oracle import densify_oracle as O

LENS_MAX_ITERS = 20            # csrc/ldp_geometry.cu LENS_MAX_ITERS
LENS_STEP_TOL = 1e-12          # csrc/ldp_geometry.cu LENS_STEP_TOL (normalised units)
HALF_PI = 1.5707963267948966
FISHEYE_THETA0_MAX = 1.5707963267948966 - 1e-6   # csrc/ldp_geometry.cu LENS_FISHEYE_THETA0_MAX: first iterate inside [0, pi/2)


@dataclass
class Lens:
    model: str                 # "opencv" | "fisheye"
    k: np.ndarray              # f64 [8]
    fx: float                  # the record's f32 K entries, held as f64
    fy: float
    cx: float
    cy: float


def lens_of(rec) -> Optional[Lens]:
    if getattr(rec, "lens_model", None) is None:
        return None
    K = np.asarray(rec.K, dtype=np.float32)
    return Lens(rec.lens_model, np.asarray(rec.lens_coeffs, dtype=np.float64).copy(),
                float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2]))


def distort(L: Lens, x: np.ndarray, y: np.ndarray):
    """Forward model on normalised coordinates (f64)."""
    k = L.k
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    r2 = x * x + y * y
    if L.model == "fisheye":
        r = np.sqrt(r2)
        th = np.arctan(r)
        t2 = th * th
        thd = th * (1.0 + t2 * (k[0] + t2 * (k[1] + t2 * (k[2] + t2 * k[3]))))
        with np.errstate(divide="ignore", invalid="ignore"):
            s = np.where(r > 0.0, thd / np.where(r > 0.0, r, 1.0), 1.0)
        return x * s, y * s
    radial = (1.0 + r2 * (k[0] + r2 * (k[1] + r2 * k[4]))) / (1.0 + r2 * (k[5] + r2 * (k[6] + r2 * k[7])))
    xd = x * radial + 2.0 * k[2] * x * y + k[3] * (r2 + 2.0 * x * x)
    yd = y * radial + k[2] * (r2 + 2.0 * y * y) + 2.0 * k[3] * x * y
    return xd, yd


def undistort(L: Lens, xd: np.ndarray, yd: np.ndarray):
    """Inverse of ``distort`` by the kernel's rule; NaN where there is no valid inverse."""
    k = L.k
    xd = np.asarray(xd, dtype=np.float64).reshape(-1)
    yd = np.asarray(yd, dtype=np.float64).reshape(-1)
    n = xd.size
    x = np.full(n, np.nan)
    y = np.full(n, np.nan)
    with np.errstate(all="ignore"):
        if L.model == "fisheye":
            rd = np.sqrt(xd * xd + yd * yd)
            zero = rd == 0.0
            x[zero], y[zero] = xd[zero], yd[zero]
            th = np.minimum(rd, FISHEYE_THETA0_MAX)
            active = ~zero
            ok = np.zeros(n, dtype=bool)
            for _ in range(LENS_MAX_ITERS):
                if not active.any():
                    break
                t2 = th * th
                f = th * (1.0 + t2 * (k[0] + t2 * (k[1] + t2 * (k[2] + t2 * k[3])))) - rd
                d = 1.0 + t2 * (3.0 * k[0] + t2 * (5.0 * k[1] + t2 * (7.0 * k[2] + t2 * 9.0 * k[3])))
                active &= d > 0.0
                step = np.where(active, f / d, 0.0)
                th = np.where(active, th - step, th)
                done = active & (np.abs(step) < LENS_STEP_TOL)
                ok |= done & (th >= 0.0) & (th < HALF_PI)
                active &= ~done
            s = np.tan(th[ok]) / rd[ok]
            x[ok], y[ok] = xd[ok] * s, yd[ok] * s
            return x, y
        u, v = xd.copy(), yd.copy()
        active = np.ones(n, dtype=bool)
        for _ in range(LENS_MAX_ITERS):
            if not active.any():
                break
            r2 = u * u + v * v
            a = 1.0 + r2 * (k[0] + r2 * (k[1] + r2 * k[4]))
            b = 1.0 + r2 * (k[5] + r2 * (k[6] + r2 * k[7]))
            da = k[0] + r2 * (2.0 * k[1] + r2 * 3.0 * k[4])
            db = k[5] + r2 * (2.0 * k[6] + r2 * 3.0 * k[7])
            radial = a / b
            drad = (da * b - a * db) / (b * b)
            fx = u * radial + 2.0 * k[2] * u * v + k[3] * (r2 + 2.0 * u * u) - xd
            fy = v * radial + k[2] * (r2 + 2.0 * v * v) + 2.0 * k[3] * u * v - yd
            j00 = radial + 2.0 * u * u * drad + 2.0 * k[2] * v + 6.0 * k[3] * u
            j01 = 2.0 * u * v * drad + 2.0 * k[2] * u + 2.0 * k[3] * v
            j10 = j01
            j11 = radial + 2.0 * v * v * drad + 6.0 * k[2] * v + 2.0 * k[3] * u
            det = j00 * j11 - j01 * j10
            active &= det > 0.0
            du = np.where(active, (j11 * fx - j01 * fy) / det, 0.0)
            dv = np.where(active, (j00 * fy - j10 * fx) / det, 0.0)
            u = np.where(active, u - du, u)
            v = np.where(active, v - dv, v)
            done = active & (du * du + dv * dv < LENS_STEP_TOL * LENS_STEP_TOL)
            x[done], y[done] = u[done], v[done]
            active &= ~done
    return x, y


def undistort_px(L: Optional[Lens], uv: np.ndarray) -> np.ndarray:
    """f32 observed pixels [n,2] -> f32 ideal pinhole pixels (the kernel's lens_undistort_px)."""
    uv = np.asarray(uv, dtype=np.float32)
    if L is None:
        return uv.copy()
    x, y = undistort(L, (uv[:, 0].astype(np.float64) - L.cx) / L.fx, (uv[:, 1].astype(np.float64) - L.cy) / L.fy)
    return np.stack([(L.fx * x + L.cx).astype(np.float32), (L.fy * y + L.cy).astype(np.float32)], axis=1)


def distort_px(L: Lens, uv: np.ndarray) -> np.ndarray:
    """f64 ideal pixels -> f64 distorted pixels."""
    uv = np.asarray(uv, dtype=np.float64)
    xd, yd = distort(L, (uv[:, 0] - L.cx) / L.fx, (uv[:, 1] - L.cy) / L.fy)
    return np.stack([L.fx * xd + L.cx, L.fy * yd + L.cy], axis=1)


def reprojection_error(P: np.ndarray, X: np.ndarray, uv_obs: np.ndarray, L: Optional[Lens]) -> np.ndarray:
    """Pinhole camera: the oracle's f32 error.  Lens camera: the f32 projection through the forward lens in f64, distance to
    the observed pixel rounded to f32."""
    if L is None:
        return O.reprojection_error(P, X, uv_obs)
    q = X @ P.T
    z = np.maximum(q[:, 2], np.float32(1e-12)).astype(np.float64)
    uv = np.stack([q[:, 0].astype(np.float64) / z, q[:, 1].astype(np.float64) / z], axis=1)
    d = distort_px(L, uv) - np.asarray(uv_obs, dtype=np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        return np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]).astype(np.float32)


def triangulate_ref_lens(cert_list, warp_list, img_u8: np.ndarray, ref_cam: O.OracleCamera,
                         nbr_cams: Sequence[O.OracleCamera], cfg: O.OracleConfig, ref_lens: Optional[Lens],
                         nbr_lenses: Sequence[Optional[Lens]], uniforms: Optional[np.ndarray] = None,
                         keep_taps: bool = True) -> Optional[O.OracleResult]:
    """densify_oracle.triangulate_ref with lens cameras (see the module docstring).  Taps: ``uvA`` / ``uvB`` are the ideal
    pixels the DLT saw, ``uvA_obs`` / ``uvB_obs`` the observed ones."""
    taps: dict = {}
    best_cert, best_k = O.best_neighbour(cert_list)
    sel_idx = O.select_samples(best_cert, cfg.matches_per_ref, cap=cfg.sample_cap, border=cfg.border, tiles=cfg.tiles,
                               no_filter=cfg.no_filter, uniforms=uniforms, taps=taps if keep_taps else None)
    if sel_idx.size == 0:
        return None
    wm, hm = cfg.w_match, cfg.h_match
    k_sel, xA, yA, xBn, yBn = O.decode_samples(warp_list, best_k, sel_idx, wm, hm)
    rgb_all = O.bilinear_colour(img_u8, xA, yA, wm, hm)
    uvA_obs_all = np.stack([xA * (ref_cam.width / float(wm)), yA * (ref_cam.height / float(hm))], axis=1)
    uvA_all = undistort_px(ref_lens, uvA_obs_all)
    members: Dict[int, List[int]] = {}
    slot_of: Dict[int, int] = {}
    for pos, kk in enumerate(k_sel):
        cam = nbr_cams[int(kk)]
        members.setdefault(cam.uid, []).append(pos)
        slot_of.setdefault(cam.uid, int(kk))
    out_xyz, out_rgb, out_err, group_taps = [], [], [], []
    for uid, pos_list in members.items():
        pos = np.asarray(pos_list, dtype=np.int64)
        cam, lensB = nbr_cams[slot_of[uid]], nbr_lenses[slot_of[uid]]
        xB = (xBn[pos] + 1.0) * 0.5 * (wm - 1)
        yB = (yBn[pos] + 1.0) * 0.5 * (hm - 1)
        uvB_obs = np.stack([xB * (cam.width / float(wm)), yB * (cam.height / float(hm))], axis=1)
        uvB = undistort_px(lensB, uvB_obs)
        gt = {"uid": uid, "pos_all": pos.copy()}
        if (not cfg.no_filter) and cfg.sampson_thresh > 0:
            F = O.fundamental_matrix(ref_cam.K, ref_cam.R, ref_cam.t, cam.K, cam.R, cam.t)
            with np.errstate(invalid="ignore"):
                se = O.sampson_distance(F, uvA_all[pos], uvB)
                ok = se < float(cfg.sampson_thresh)
            if not np.any(ok):
                group_taps.append(gt)
                continue
            pos, uvB, uvB_obs = pos[ok], uvB[ok], uvB_obs[ok]
        uvA, uvA_obs = uvA_all[pos], uvA_obs_all[pos]
        finite = np.isfinite(uvA).all(axis=1) & np.isfinite(uvB).all(axis=1)
        X = np.full((pos.size, 4), np.nan, dtype=np.float32)   # LAPACK refuses NaN rows; the kernel's NaN point is never kept
        if finite.any():
            X[finite] = O.dlt_points(ref_cam.P, cam.P, uvA[finite], uvB[finite])
        with np.errstate(invalid="ignore"):
            e = np.maximum(reprojection_error(ref_cam.P, X, uvA_obs, ref_lens), reprojection_error(cam.P, X, uvB_obs, lensB))
            if cfg.no_filter:
                keep = np.isfinite(X).all(axis=1) & np.isfinite(e)
            else:
                keep = e <= float(cfg.reproj_thresh)
                keep &= O.in_front(ref_cam.P, X)
                keep &= O.in_front(cam.P, X)
                if cfg.min_parallax_deg > 0:
                    keep &= O.parallax_ok(ref_cam.C, cam.C, X, cfg.min_parallax_deg)
        gt.update(pos=pos, X=X, err=e, keep=keep, uvA=uvA, uvB=uvB, uvA_obs=uvA_obs, uvB_obs=uvB_obs, P1=ref_cam.P, P2=cam.P,
                  lensB=lensB)
        group_taps.append(gt)
        if not np.any(keep):
            continue
        out_xyz.append(X[keep][:, :3].astype(np.float32))
        out_rgb.append(rgb_all[pos][keep].astype(np.float32))
        out_err.append(e[keep].astype(np.float32))
    if not out_xyz:
        return None
    if keep_taps:
        taps.update(ref_uid=ref_cam.uid, best_k=best_k.numpy(), best_cert=best_cert.numpy(), k_sel=k_sel, groups=group_taps,
                    ref_lens=ref_lens)
    return O.OracleResult(xyz=np.concatenate(out_xyz, axis=0), rgb=np.concatenate(out_rgb, axis=0),
                          err=np.concatenate(out_err, axis=0), sel_idx=sel_idx, taps=taps)
