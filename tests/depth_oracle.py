"""numpy restatement of the depth-map rule (include/ldp_b200.h: ldp_depth_maps) for pinhole cameras and post-processed
certainty planes: the candidate set, then oracle.densify_oracle's own per-sample geometry on it, group by group exactly as
``triangulate_ref`` evaluates its samples (decode, Sampson gate, DLT by f32 SVD, reprojection, cheirality, parallax or
no_filter's finiteness test).  The multi-view refinement is not restated here."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Sequence

import numpy as np

from oracle import densify_oracle as O


@dataclass
class DepthOracle:
    cand: np.ndarray      # bool [H*W]
    good: np.ndarray      # bool [H*W]: Sampson pass (candidates only)
    keep: np.ndarray      # bool [H*W]
    winner: np.ndarray    # int [H*W]
    depth: np.ndarray     # f32 [H*W], NaN where not kept
    err: np.ndarray       # f32 [H*W], NaN where not triangulated
    xyz: np.ndarray       # f32 [H*W, 3], NaN where not kept
    margin: np.ndarray    # f64 [H*W]: distance of the keep verdict's closest quantity to its threshold (relative), inf if none


def depth_maps(cert_list, warp_list, ref_cam: O.OracleCamera, nbr_cams: Sequence[O.OracleCamera], cfg: O.OracleConfig,
               min_certainty: float) -> DepthOracle:
    best_cert, best_k = O.best_neighbour(cert_list)
    H, W = best_cert.shape
    n = H * W
    bc = best_cert.reshape(-1).numpy()
    cand = bc >= np.float32(min_certainty)
    idx = np.nonzero(cand)[0]
    nan = np.float32(np.nan)
    good = np.zeros(n, bool)
    keep = np.zeros(n, bool)
    depth = np.full(n, nan, np.float32)
    err = np.full(n, nan, np.float32)
    xyz = np.full((n, 3), nan, np.float32)
    margin = np.full(n, np.inf)
    winner = best_k.reshape(-1).numpy().astype(np.int64)
    if idx.size == 0:
        return DepthOracle(cand, good, keep, winner, depth, err, xyz, margin)
    wm, hm = cfg.w_match, cfg.h_match
    k_sel, xA, yA, xBn, yBn = O.decode_samples(warp_list, best_k, idx, wm, hm)
    uvA_all = np.stack([xA * (ref_cam.width / float(wm)), yA * (ref_cam.height / float(hm))], axis=1)
    for k in np.unique(k_sel):
        cam = nbr_cams[int(k)]
        pos = np.nonzero(k_sel == k)[0]
        xB = (xBn[pos] + 1.0) * 0.5 * (wm - 1)
        yB = (yBn[pos] + 1.0) * 0.5 * (hm - 1)
        uvB = np.stack([xB * (cam.width / float(wm)), yB * (cam.height / float(hm))], axis=1)
        if (not cfg.no_filter) and cfg.sampson_thresh > 0:
            F = O.fundamental_matrix(ref_cam.K, ref_cam.R, ref_cam.t, cam.K, cam.R, cam.t)
            se = O.sampson_distance(F, uvA_all[pos], uvB)
            ok = se < float(cfg.sampson_thresh)
            m = np.abs(se / float(cfg.sampson_thresh) - 1.0)
            margin[idx[pos]] = np.minimum(margin[idx[pos]], np.where(np.isfinite(m), m, np.inf))
            pos, uvB = pos[ok], uvB[ok]
        if pos.size == 0:
            continue
        uvA = uvA_all[pos]
        X = O.dlt_points(ref_cam.P, cam.P, uvA, uvB)
        e = np.maximum(O.reprojection_error(ref_cam.P, X, uvA), O.reprojection_error(cam.P, X, uvB))
        if cfg.no_filter:
            kp = np.isfinite(X).all(axis=1) & np.isfinite(e)
        else:
            kp = e <= float(cfg.reproj_thresh)
            kp &= O.in_front(ref_cam.P, X)
            kp &= O.in_front(cam.P, X)
            m = np.abs(e / float(cfg.reproj_thresh) - 1.0)
            margin[idx[pos]] = np.minimum(margin[idx[pos]], np.where(np.isfinite(m), m, np.inf))
            if cfg.min_parallax_deg > 0:
                kp &= O.parallax_ok(ref_cam.C, cam.C, X, cfg.min_parallax_deg)
        z = (X @ ref_cam.P.T)[:, 2]
        i = idx[pos]
        good[i] = True
        err[i] = e.astype(np.float32)
        keep[i] = kp
        depth[i[kp]] = z[kp].astype(np.float32)
        xyz[i[kp]] = X[kp][:, :3].astype(np.float32)
    return DepthOracle(cand, good, keep, winner, depth, err, xyz, margin)
