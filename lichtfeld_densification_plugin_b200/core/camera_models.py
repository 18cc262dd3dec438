"""Camera records and the packed per-launch camera tables.

``CameraRecord`` keeps the reference's field names and dtypes (reference core/camera_models.py:10-21:
K,R [3,3] f32; t [3,1] f32; P [3,4] f32; C [3] f32; width/height = full-resolution camera size).

A record may also carry a lens model (``lens_model`` / ``lens_coeffs``, built by ``from_colmap``); the device path then
triangulates through it (include/ldp_b200.h: ldp_lens).  The reference drops distortion coefficients (reference
core/geometry.py:10-30, SURVEY F2): its records, and every record ``from_KRt`` builds, carry no lens and are triangulated
exactly as the reference does.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np


@dataclass
class CameraRecord:
    uid: int
    image_path: str
    width: int
    height: int
    K: np.ndarray
    R: np.ndarray
    t: np.ndarray
    P: np.ndarray
    C: np.ndarray
    mask_path: Optional[str] = None
    lens_model: Optional[str] = None           # None (pinhole), "opencv" or "fisheye"
    lens_coeffs: Optional[np.ndarray] = None   # f64 [8]: opencv k1 k2 p1 p2 k3 k4 k5 k6; fisheye k1 k2 k3 k4 0 0 0 0

    def __post_init__(self) -> None:
        check_lens(self)

    @classmethod
    def from_KRt(cls, uid: int, width: int, height: int, K, R, t, image_path: str = "",
                 mask_path: Optional[str] = None) -> "CameraRecord":
        """Build P and C from K,R,t with the reference's float32 arithmetic
        (reference densify.py:226-230, core/geometry.py:45-50)."""
        K = np.asarray(K, dtype=np.float32).reshape(3, 3)
        R = np.asarray(R, dtype=np.float32).reshape(3, 3)
        t = np.asarray(t, dtype=np.float32).reshape(3, 1)
        P = K @ np.concatenate([R, t], axis=1)
        C = (-R.T @ t).reshape(3)
        return cls(uid=int(uid), image_path=image_path, width=int(width), height=int(height),
                   K=K, R=R, t=t, P=P, C=C, mask_path=mask_path)

    @classmethod
    def from_colmap(cls, uid: int, model_name: str, params, width: int, height: int, R, t, image_path: str = "",
                    mask_path: Optional[str] = None) -> "CameraRecord":
        """A record from a COLMAP camera: ``model_name`` / ``params`` as ``pycolmap.Camera.model.name`` / ``.params`` give
        them.  K is built like the reference's ``K_from_camera`` (f32 fx, fy, cx, cy; the SIMPLE_* models use f for both),
        P and C like ``from_KRt``; the distortion coefficients become the record's lens (none if they are all zero)."""
        name = str(model_name).upper()
        if name not in COLMAP_MODELS:
            raise ValueError(f"unsupported COLMAP camera model {model_name!r} (supported: {', '.join(COLMAP_MODELS)})")
        family, n_focal, slots = COLMAP_MODELS[name]
        params = np.asarray(params, dtype=np.float64).reshape(-1)
        if params.size != n_focal + 2 + len(slots):
            raise ValueError(f"{name} takes {n_focal + 2 + len(slots)} parameters, got {params.size}")
        fx = params[0]
        fy = params[1] if n_focal == 2 else params[0]
        cx, cy = params[n_focal], params[n_focal + 1]
        K = np.array([[fx, 0.0, cx], [0.0, fy, cy], [0.0, 0.0, 1.0]], dtype=np.float32)
        rec = cls.from_KRt(uid, width, height, K, R, t, image_path=image_path, mask_path=mask_path)
        coeffs = np.zeros(8, dtype=np.float64)
        coeffs[list(slots)] = params[n_focal + 2:]
        if family is not None and np.any(coeffs != 0.0):
            rec.lens_model, rec.lens_coeffs = family, coeffs
            check_lens(rec)
        return rec

    def flat_pose(self) -> np.ndarray:
        """Row-major 4x4 world-to-camera transform, used for clustering / nearest neighbours."""
        T = np.eye(4)
        T[:3, :3] = self.R
        T[:3, 3] = self.t.reshape(3)
        return T.reshape(-1)


# COLMAP model name -> (lens family, focal parameters, slot in lens_coeffs of each distortion parameter)
COLMAP_MODELS = {
    "SIMPLE_PINHOLE": (None, 1, ()),
    "PINHOLE": (None, 2, ()),
    "SIMPLE_RADIAL": ("opencv", 1, (0,)),
    "RADIAL": ("opencv", 1, (0, 1)),
    "OPENCV": ("opencv", 2, (0, 1, 2, 3)),
    "FULL_OPENCV": ("opencv", 2, (0, 1, 2, 3, 4, 5, 6, 7)),
    "OPENCV_FISHEYE": ("fisheye", 2, (0, 1, 2, 3)),
    "SIMPLE_RADIAL_FISHEYE": ("fisheye", 1, (0,)),
    "RADIAL_FISHEYE": ("fisheye", 1, (0, 1)),
}
LENS_FAMILIES = ("opencv", "fisheye")


def check_lens(rec: CameraRecord) -> None:
    """A lens record must name a known family, carry 8 finite coefficients and have no skew (the lens normalises pixels
    with fx, fy, cx, cy alone)."""
    if rec.lens_model is None:
        return
    if rec.lens_model not in LENS_FAMILIES:
        raise ValueError(f"unknown lens model {rec.lens_model!r} (expected one of {LENS_FAMILIES})")
    k = np.asarray(rec.lens_coeffs, dtype=np.float64)
    if k.shape != (8,) or not np.all(np.isfinite(k)):
        raise ValueError("lens_coeffs must be 8 finite float64 values")
    if float(np.asarray(rec.K, dtype=np.float32)[0, 1]) != 0.0:
        raise ValueError("a camera with a lens model must have zero skew (K[0,1])")


def stack_flat_poses(records: Sequence[CameraRecord]) -> np.ndarray:
    return np.stack([r.flat_pose() for r in records], axis=0)
