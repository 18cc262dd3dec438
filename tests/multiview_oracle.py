"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the multi-view refinement of the device path (ldp_params.multiview;
the semantics are stated in include/ldp_b200.h).

The reference triangulates every sample from its winning neighbour alone, so there is no reference behaviour to pin.  This
module applies the stated rule to the per-sample taps of ``lens_oracle.triangulate_ref_lens`` (the pinned oracle's two-view
path with lens cameras): for every kept sample it gathers the candidates, builds the same float32 DLT rows, solves them by
a float64 SVD, trims once and accepts or falls back.  ``oracle/densify_oracle.py`` is not touched.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np

from oracle import densify_oracle as O
from tests import lens_oracle as LO


@dataclass
class Refined:
    """Per oracle sample position (``res.sel_idx`` order); meaningful where ``keep``."""
    keep: np.ndarray           # bool [S]: the two-view verdict
    xyz: np.ndarray            # f32 [S,3] the point to emit
    err: np.ndarray            # f32 [S]
    mask: np.ndarray           # int64 [S] view mask (bit = neighbour slot)
    margin: np.ndarray         # f64 [S] smallest |error - reproj_thresh| over the trimming / acceptance decisions (inf: none)
    two_xyz: np.ndarray        # f32 [S,3] the two-view point


def dlt_rows(P: np.ndarray, uv: np.ndarray) -> np.ndarray:
    """The two DLT rows of camera P at pixel uv = (u, v), in the dtype of P and uv (float32 in the path)."""
    return np.stack([uv[0] * P[2] - P[0], uv[1] * P[2] - P[1]])


def solve(rows: np.ndarray) -> np.ndarray:
    """Null vector of the stacked rows by a float64 SVD, dehomogenised (f64 [3])."""
    v = np.linalg.svd(np.asarray(rows, dtype=np.float64))[2][-1]
    w = v[3] if abs(v[3]) >= 1e-12 else 1e-12
    return v[:3] / w


def _decode_b(warp_q, idx: int, cam, wm: int, hm: int) -> np.ndarray:
    """Neighbour pixel (observed) of warp plane ``warp_q`` [H,W,4] at flat pixel idx, float32 like the path."""
    row = np.asarray(warp_q).reshape(-1, 4)[idx].astype(np.float32)
    xB = (row[2] + np.float32(1.0)) * np.float32(0.5) * np.float32(wm - 1)
    yB = (row[3] + np.float32(1.0)) * np.float32(0.5) * np.float32(hm - 1)
    return np.array([xB * np.float32(cam.width / float(wm)), yB * np.float32(cam.height / float(hm))], dtype=np.float32)


def _view_err(P, X3: np.ndarray, uv_obs: np.ndarray, L) -> tuple:
    X = np.concatenate([X3.astype(np.float32), np.ones(1, dtype=np.float32)])[None, :]
    X = np.repeat(X, 4, axis=0)                  # a batch, like the oracle's group-wise projection
    e = float(LO.reprojection_error(P, X, np.repeat(uv_obs[None, :], 4, axis=0), L)[0])
    z = float((X @ P.T)[0, 2])
    return e, z


def refine(res: O.OracleResult, cert_list, warp_list, ref_cam: O.OracleCamera, nbr_cams: Sequence[O.OracleCamera],
           cfg: O.OracleConfig, groups: Sequence[int], min_cert: float,
           ref_lens: Optional[LO.Lens] = None, nbr_lenses: Optional[Sequence[Optional[LO.Lens]]] = None) -> Refined:
    """The multi-view refinement of every kept sample of ``res`` (a ``triangulate_ref_lens`` result with taps).
    ``cert_list``: the certainty planes AFTER post-processing; ``groups[q]``: the descriptor's group of slot q."""
    nn = len(nbr_cams)
    nbr_lenses = list(nbr_lenses) if nbr_lenses is not None else [None] * nn
    wm, hm = cfg.w_match, cfg.h_match
    thr = np.float32(cfg.reproj_thresh)
    S = res.sel_idx.size
    keep = np.zeros(S, dtype=bool)
    xyz = np.full((S, 3), np.nan, dtype=np.float32)
    two = np.full((S, 3), np.nan, dtype=np.float32)
    err = np.full(S, np.nan, dtype=np.float32)
    mask = np.zeros(S, dtype=np.int64)
    margin = np.full(S, np.inf)
    certs = [np.asarray(c, dtype=np.float32).reshape(-1) for c in cert_list]
    P = [np.asarray(c.P, dtype=np.float32) for c in nbr_cams]
    P1 = np.asarray(ref_cam.P, dtype=np.float32)
    F = [O.fundamental_matrix(ref_cam.K, ref_cam.R, ref_cam.t, c.K, c.R, c.t) for c in nbr_cams]
    k_sel = res.taps["k_sel"]
    mc = np.float32(min_cert)
    for gt in res.taps["groups"]:
        if "pos" not in gt:
            continue
        for j, pos in enumerate(gt["pos"]):
            if not gt["keep"][j]:
                continue
            pos = int(pos)
            k = int(k_sel[pos])
            idx = int(res.sel_idx[pos])
            keep[pos] = True
            X2 = gt["X"][j, :3].astype(np.float32)
            two[pos] = X2
            xyz[pos], err[pos], mask[pos] = X2, gt["err"][j], 1 << k
            uvA, uvA_obs = gt["uvA"][j], gt["uvA_obs"][j]
            uvB, uvB_obs = gt["uvB"][j], gt["uvB_obs"][j]
            cand: Dict[int, tuple] = {}
            for q in range(nn):
                if groups[q] != q or q == groups[k]:
                    continue
                if not certs[q][idx] >= mc:
                    continue
                b_obs = _decode_b(warp_list[q], idx, nbr_cams[q], wm, hm)
                b = LO.undistort_px(nbr_lenses[q], b_obs[None, :])[0]
                if not np.isfinite(b).all():
                    continue
                if (not cfg.no_filter) and cfg.sampson_thresh > 0:
                    with np.errstate(invalid="ignore"):
                        se = O.sampson_distance(F[q], uvA[None, :].astype(np.float64), b[None, :].astype(np.float64))[0]
                    if not se < float(cfg.sampson_thresh):
                        continue
                cand[q] = (b, b_obs)
            if not cand:
                continue
            base = [dlt_rows(P1, uvA), dlt_rows(P[k], uvB)]
            Y = solve(np.concatenate(base + [dlt_rows(P[q], cand[q][0]) for q in cand]))
            used = []
            for q, (b, b_obs) in cand.items():
                e, z = _view_err(P[q], Y, b_obs, nbr_lenses[q])
                margin[pos] = min(margin[pos], abs(e - float(thr)))
                if np.float32(e) <= thr and z > 0:
                    used.append(q)
            if not used:
                continue
            if len(used) != len(cand):
                Y = solve(np.concatenate(base + [dlt_rows(P[q], cand[q][0]) for q in used]))
            views = [(P1, uvA_obs, ref_lens), (P[k], uvB_obs, nbr_lenses[k])] + [(P[q], cand[q][1], nbr_lenses[q]) for q in used]
            ok, emax = True, 0.0
            for Pv, uv_obs, L in views:
                e, z = _view_err(Pv, Y, uv_obs, L)
                margin[pos] = min(margin[pos], abs(e - float(thr)))
                ok = ok and bool(np.float32(e) <= thr) and z > 0
                emax = max(emax, e)
            if ok and cfg.min_parallax_deg > 0:
                Xp = np.concatenate([Y.astype(np.float32), np.ones(1, dtype=np.float32)])[None, :]
                ok = bool(O.parallax_ok(np.asarray(ref_cam.C, dtype=np.float32), np.asarray(nbr_cams[k].C, dtype=np.float32),
                                        Xp, cfg.min_parallax_deg)[0])
            if ok:
                xyz[pos], err[pos] = Y.astype(np.float32), np.float32(emax)
                mask[pos] = (1 << k) | sum(1 << q for q in used)
    return Refined(keep=keep, xyz=xyz, err=err, mask=mask, margin=margin, two_xyz=two)


def groups_of(uids: Sequence[int]) -> List[int]:
    """The descriptor's group table: smallest slot with the same uid."""
    uids = list(uids)
    return [uids.index(u) for u in uids]


def run(scene, inp: dict, cfg: O.OracleConfig, min_cert: float = 0.5, uniforms=None):
    """Two-view oracle + refinement for one synthetic reference view.  Returns (two-view result, Refined)."""
    from tests.helpers import oracle_cam
    cams = scene.cameras
    nn = len(inp["nbr_indices"])
    ref = cams[inp["ref_index"]]
    nbrs = [cams[j] for j in inp["nbr_indices"]]
    certs = [inp["cert"][k] for k in range(nn)]
    warps = [inp["warp"][k] for k in range(nn)]
    res = LO.triangulate_ref_lens(certs, warps, inp["image"].numpy(), oracle_cam(ref), [oracle_cam(c) for c in nbrs], cfg,
                                  LO.lens_of(ref), [LO.lens_of(c) for c in nbrs], uniforms=uniforms)
    if res is None:
        return None, None
    ref_o, nbr_o = oracle_cam(ref), [oracle_cam(c) for c in nbrs]
    mv = refine(res, [c.numpy() for c in certs], [w.numpy() for w in warps], ref_o, nbr_o, cfg,
                groups_of([c.uid for c in nbrs]), min_cert, LO.lens_of(ref), [LO.lens_of(c) for c in nbrs])
    return res, mv
