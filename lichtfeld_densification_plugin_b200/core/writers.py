"""Point-cloud writers: the reference's on-disk contract, vectorised.

Byte-for-byte the files reference core/writers.py:15-46 produces (a per-point ``struct.pack`` loop there),
written here as one structured-array ``tofile``:

* ``write_ply``            binary little-endian PLY: header (core/writers.py:31-41) then per vertex ``<fff`` + ``BBB``;
                           with ``normals`` (not in the reference) ``nx ny nz`` floats between ``z`` and ``red``, 27 bytes
* ``write_points3D_bin``   ``<Q n`` then per point ``<Q id=i+1``, ``<ddd xyz``, ``<BBB rgb``, ``<d err`` (no track list)
* ``to_uint8_rgb``         ``clip(round(x * 255), 0, 255)`` with round-half-to-even (core/image_utils.py:24-26)
"""
from __future__ import annotations

import os
from typing import Optional

import numpy as np

_PLY_VERTEX = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("r", "u1"), ("g", "u1"), ("b", "u1")])
_BIN_POINT = np.dtype([("id", "<u8"), ("x", "<f8"), ("y", "<f8"), ("z", "<f8"),
                       ("r", "u1"), ("g", "u1"), ("b", "u1"), ("err", "<f8")])
_PLY_NORMAL_VERTEX = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("nx", "<f4"), ("ny", "<f4"), ("nz", "<f4"),
                               ("r", "u1"), ("g", "u1"), ("b", "u1")])
assert _PLY_VERTEX.itemsize == 15 and _BIN_POINT.itemsize == 43 and _PLY_NORMAL_VERTEX.itemsize == 27


def ensure_dir(path: str) -> None:
    os.makedirs(os.path.dirname(path), exist_ok=True)


def to_uint8_rgb(arr_float01: np.ndarray) -> np.ndarray:
    """Float RGB in [0, 1] -> uint8 (numpy's round is half-to-even, like the reference's)."""
    return np.clip(np.round(arr_float01 * 255.0), 0, 255).astype(np.uint8)


def ply_header(n: int, normals: bool = False) -> bytes:
    return (f"ply\nformat binary_little_endian 1.0\nelement vertex {n}\n"
            "property float x\nproperty float y\nproperty float z\n"
            + ("property float nx\nproperty float ny\nproperty float nz\n" if normals else "")
            + "property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n").encode("ascii")


def write_ply(path_out: str, xyz: np.ndarray, rgb_uint8: np.ndarray, normals: Optional[np.ndarray] = None) -> None:
    """``normals`` [n,3] (e.g. ``output.estimate_normals``) adds the nx / ny / nz vertex properties."""
    n = int(xyz.shape[0])
    rec = np.empty(n, dtype=_PLY_VERTEX if normals is None else _PLY_NORMAL_VERTEX)
    rec["x"], rec["y"], rec["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]          # float(xyz[i, j]) packed as <f
    if normals is not None:
        rec["nx"], rec["ny"], rec["nz"] = normals[:, 0], normals[:, 1], normals[:, 2]
    rec["r"], rec["g"], rec["b"] = rgb_uint8[:, 0], rgb_uint8[:, 1], rgb_uint8[:, 2]
    with open(path_out, "wb") as f:
        f.write(ply_header(n, normals is not None))
        rec.tofile(f)


def write_points3D_bin(path_out: str, xyz: np.ndarray, rgb_uint8: np.ndarray,
                       errors: Optional[np.ndarray] = None) -> None:
    n = int(xyz.shape[0])
    if errors is None:
        errors = np.zeros((n,), dtype=np.float32)
    rec = np.empty(n, dtype=_BIN_POINT)
    rec["id"] = np.arange(1, n + 1, dtype=np.uint64)
    rec["x"], rec["y"], rec["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]          # widened to f64 like float(x) -> <d
    rec["r"], rec["g"], rec["b"] = rgb_uint8[:, 0], rgb_uint8[:, 1], rgb_uint8[:, 2]
    rec["err"] = errors
    with open(path_out, "wb") as f:
        f.write(np.uint64(n).tobytes())
        rec.tofile(f)
