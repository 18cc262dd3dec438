"""Stored OpenCV results for tests/test_oracle_lens.py, so that the lens oracle is checked against OpenCV also where cv2 is
not installed: tests/golden/lens/cv2_lens.npz (a subdirectory: the *.npz files directly under tests/golden are pipeline
cases).

For every supported COLMAP model with a distortion (coefficients below), on a grid of ideal pixels covering a 1297 x 840
image and a grid of observed pixels over the same image:
  fwd_<model>  cv2.projectPoints (8 coefficients) / cv2.fisheye.distortPoints of the ideal grid, pixels
  und_<model>  cv2.undistortPointsIter / cv2.fisheye.undistortPoints (P = K) of the observed grid, run to tight criteria

    python tests/golden/make_lens_golden.py
"""
from __future__ import annotations

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
GOLDEN = os.path.join(HERE, "lens", "cv2_lens.npz")

WIDTH, HEIGHT = 1297, 840
FOCAL = 0.74 * WIDTH
# COLMAP model -> distortion parameters (COLMAP's order)
CASES = {
    "SIMPLE_RADIAL": [-0.12],
    "RADIAL": [-0.1, 0.02],
    "OPENCV": [-0.12, 0.03, 4e-4, -3e-4],
    "FULL_OPENCV": [0.2, -0.05, 4e-4, -3e-4, 0.01, 0.25, -0.03, 0.01],
    "OPENCV_FISHEYE": [0.05, -0.01, 0.003, -0.0005],
    "SIMPLE_RADIAL_FISHEYE": [0.04],
    "RADIAL_FISHEYE": [0.04, -0.008],
}


def record(name: str):
    """The CameraRecord of a case (identity pose)."""
    sys.path.insert(0, ROOT)
    from lichtfeld_densification_plugin_b200.core.camera_models import COLMAP_MODELS, CameraRecord
    focal = [FOCAL] * COLMAP_MODELS[name][1]
    return CameraRecord.from_colmap(0, name, focal + [WIDTH / 2.0, HEIGHT / 2.0] + CASES[name], WIDTH, HEIGHT,
                                    np.eye(3), np.zeros(3))


def pixel_grid(n: int = 25) -> np.ndarray:
    """[n*n, 2] f64 pixels over the whole image, edges and corners included."""
    u, v = np.meshgrid(np.linspace(0.0, WIDTH, n), np.linspace(0.0, HEIGHT, n))
    return np.stack([u.reshape(-1), v.reshape(-1)], axis=1)


def cv2_results(cv2, rec):
    K = np.asarray(rec.K, dtype=np.float64)
    k = np.asarray(rec.lens_coeffs, dtype=np.float64)
    ideal = pixel_grid()
    obs = pixel_grid().astype(np.float32).astype(np.float64)
    crit = (cv2.TERM_CRITERIA_COUNT | cv2.TERM_CRITERIA_EPS, 1000, 1e-15)
    xn = np.stack([(ideal[:, 0] - K[0, 2]) / K[0, 0], (ideal[:, 1] - K[1, 2]) / K[1, 1]], axis=1)
    if rec.lens_model == "fisheye":
        fwd = cv2.fisheye.distortPoints(xn[:, None, :], K, k[:4])[:, 0, :]
        und = cv2.fisheye.undistortPoints(obs[:, None, :], K, k[:4], R=np.eye(3), P=K, criteria=crit)[:, 0, :]
    else:
        obj = np.concatenate([xn, np.ones((xn.shape[0], 1))], axis=1)
        fwd = cv2.projectPoints(obj[:, None, :], np.zeros(3), np.zeros(3), K, k)[0][:, 0, :]
        und = cv2.undistortPointsIter(obs[:, None, :], K, k, np.eye(3), K, crit)[:, 0, :]
    return ideal, obs, fwd.astype(np.float64), und.astype(np.float64)


def main() -> None:
    import cv2
    out = {"cv2_version": np.array(cv2.__version__)}
    for name in CASES:
        ideal, obs, fwd, und = cv2_results(cv2, record(name))
        out[f"fwd_{name}"], out[f"und_{name}"] = fwd, und
    out["ideal"], out["obs"] = ideal, obs
    os.makedirs(os.path.dirname(GOLDEN), exist_ok=True)
    np.savez_compressed(GOLDEN, **out)
    print(GOLDEN, os.path.getsize(GOLDEN), "bytes")


if __name__ == "__main__":
    main()
