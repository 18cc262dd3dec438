"""Numpy restatement of the 3DGS initialisation rule of include/ldp_b200.h (ldp_gaussian_init / output.init_gaussians).

* ``dist2``            step 1: the k_eff smallest non-self f64 d^2 (``outlier_oracle``'s exact k-NN over k_eff + 1 entries,
                       the point itself first at 0), summed sequentially, over k_eff, clamped in f32
* ``scales`` / ``sh_dc`` / ``opacity_logit`` / ``rotations``   steps 2-4
* ``init_gaussians``   every step
* ``build_rotation`` / ``covariance``   graphdeco 3DGS's own ``build_rotation`` and ``R S S^T R^T``, restated in f64
"""
from __future__ import annotations

import numpy as np

from tests import outlier_oracle as OO

C0 = 0.28209479177387814                 # 3DGS's SH band-0 constant (utils/sh_utils.py)
FLOOR = np.float32(1e-7)                 # 3DGS's clamp_min(dist2, 0.0000001) on an f32 tensor
ARC_MIN = 1e-12                          # 1 + u_z at or below this: half a turn about x


def dist2(xyz: np.ndarray, k: int) -> np.ndarray:
    """f32 [n]: max(f32(mean of the k_eff smallest d^2 over j != i), 1e-7), k_eff = min(k, n - 1); brute force on small
    clouds, cKDTree candidates otherwise (the same values)."""
    x = np.asarray(xyz, np.float32)
    n = x.shape[0]
    if n == 0:
        return np.zeros((0,), np.float32)
    kk = min(k + 1, n)
    d2 = OO.sorted_knn_d2_exact(x, kk) if n > 4096 else OO.sorted_knn_d2(x, kk)
    ke = kk - 1
    m = np.zeros(n, np.float64)
    for j in range(1, kk):                # sequential, ascending; entry 0 is the point itself (d^2 = 0)
        m = m + d2[:, j]
    if ke > 0:
        m = m / np.float64(ke)
    return np.maximum(m.astype(np.float32), FLOOR)


def sh_dc(rgb: np.ndarray) -> np.ndarray:
    """3DGS's RGB2SH in f32: (rgb - 0.5) / C0, each operation correctly rounded."""
    r = np.asarray(rgb, np.float32)
    return (r - np.float32(0.5)) / np.float32(C0)


def opacity_logit(alpha: float) -> np.float32:
    a = np.float64(alpha)
    return np.float32(np.log(a / (1.0 - a)))


def _unit_normals(normals, n: int):
    """(u f64 [n,3], defined bool [n]): the normals renormalised in f64; undefined for a zero or non-finite length."""
    if normals is None:
        return np.zeros((n, 3)), np.zeros(n, bool)
    v = np.asarray(normals, np.float32).astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        ln = np.sqrt((v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1]) + v[:, 2] * v[:, 2])
        ok = (ln > 0) & np.isfinite(ln)
        u = np.where(ok[:, None], v / np.where(ok, ln, 1.0)[:, None], 0.0)
    return u, ok


def rotations(normals, n: int):
    """(f32 [n,4] (w, x, y, z), defined bool [n]) of step 4."""
    u, ok = _unit_normals(normals, n)
    q = np.zeros((n, 4))
    q[:, 0] = 1.0
    w = 1.0 + u[:, 2]
    arc = ok & (w > ARC_MIN)
    qa = np.stack([w, -u[:, 1], u[:, 0], np.zeros(n)], axis=1)[arc]
    qn = np.sqrt((qa[:, 0] * qa[:, 0] + qa[:, 1] * qa[:, 1]) + qa[:, 2] * qa[:, 2])
    q[arc] = qa / qn[:, None]
    q[ok & ~arc] = (0.0, 1.0, 0.0, 0.0)
    return q.astype(np.float32), ok


def scales(d2: np.ndarray, defined: np.ndarray, flatten: float) -> np.ndarray:
    ls = np.log(np.sqrt(np.asarray(d2, np.float32).astype(np.float64)))
    s = np.repeat(ls.astype(np.float32)[:, None], 3, axis=1)
    s[defined, 2] = (ls[defined] + np.log(np.float64(flatten))).astype(np.float32)
    return s


def init_gaussians(xyz, rgb, normals=None, k: int = 3, opacity: float = 0.1, flatten: float = 1.0) -> dict:
    """Every output of ldp_gaussian_init: sh_dc, opacity, scales, rotations, dist2 and the undefined count."""
    x = np.asarray(xyz, np.float32)
    if not np.isfinite(x).all():
        raise ValueError("a coordinate is not finite")
    n = x.shape[0]
    d2 = dist2(x, k)
    q, ok = rotations(normals, n)
    return dict(sh_dc=sh_dc(rgb), opacity=np.full(n, opacity_logit(opacity), np.float32), scales=scales(d2, ok, flatten),
                rotations=q, dist2=d2, undefined=int(n - ok.sum()))


def build_rotation(q: np.ndarray) -> np.ndarray:
    """graphdeco 3DGS utils/general_utils.build_rotation in f64: q / |q|, then the rotation matrix [n,3,3]."""
    q = np.asarray(q, np.float64)
    q = q / np.linalg.norm(q, axis=1, keepdims=True)
    r, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    R = np.empty((q.shape[0], 3, 3))
    R[:, 0, 0] = 1 - 2 * (y * y + z * z); R[:, 0, 1] = 2 * (x * y - r * z); R[:, 0, 2] = 2 * (x * z + r * y)
    R[:, 1, 0] = 2 * (x * y + r * z); R[:, 1, 1] = 1 - 2 * (x * x + z * z); R[:, 1, 2] = 2 * (y * z - r * x)
    R[:, 2, 0] = 2 * (x * z - r * y); R[:, 2, 1] = 2 * (y * z + r * x); R[:, 2, 2] = 1 - 2 * (x * x + y * y)
    return R


def covariance(scales_log: np.ndarray, q: np.ndarray) -> np.ndarray:
    """3DGS's build_covariance_from_scaling_rotation: L = R S, Sigma = L L^T, in f64."""
    L = build_rotation(q) * np.exp(np.asarray(scales_log, np.float64))[:, None, :]
    return L @ np.transpose(L, (0, 2, 1))
