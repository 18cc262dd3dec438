"""Point-cloud writers: the reference's on-disk contract, vectorised.

Byte-for-byte the files reference core/writers.py:15-46 produces (a per-point ``struct.pack`` loop there),
written here as one structured-array ``tofile``:

* ``write_ply``            binary little-endian PLY: header (core/writers.py:31-41) then per vertex ``<fff`` + ``BBB``;
                           with ``normals`` (not in the reference) ``nx ny nz`` floats between ``z`` and ``red``, 27 bytes
* ``write_points3D_bin``   ``<Q n`` then per point ``<Q id=i+1``, ``<ddd xyz``, ``<BBB rgb``, ``<d err`` (no track list)
* ``to_uint8_rgb``         ``clip(round(x * 255), 0, 255)`` with round-half-to-even (core/image_utils.py:24-26)
* ``write_gaussian_ply``   not in the reference: the 3DGS PLY of initialised splats (graphdeco 3DGS ``save_ply``), the
                           byte reference for ``output.write_gaussian_ply``
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


def gaussian_ply_attributes(sh_degree: int) -> list:
    """Vertex property names of graphdeco 3DGS's ``construct_list_of_attributes`` for SH degree ``sh_degree``, in order."""
    if not 0 <= int(sh_degree) <= 3:
        raise ValueError("sh_degree must lie in [0, 3]")
    n_rest = 3 * ((int(sh_degree) + 1) ** 2 - 1)
    return (["x", "y", "z", "nx", "ny", "nz"] + [f"f_dc_{i}" for i in range(3)] + [f"f_rest_{i}" for i in range(n_rest)]
            + ["opacity"] + [f"scale_{i}" for i in range(3)] + [f"rot_{i}" for i in range(4)])


def gaussian_ply_header(n: int, sh_degree: int = 3) -> bytes:
    return (f"ply\nformat binary_little_endian 1.0\nelement vertex {n}\n"
            + "".join(f"property float {a}\n" for a in gaussian_ply_attributes(sh_degree)) + "end_header\n").encode("ascii")


def gaussian_ply_vertices(xyz: np.ndarray, sh_dc: np.ndarray, opacity: np.ndarray, scales: np.ndarray,
                          rotations: np.ndarray, normals: Optional[np.ndarray] = None, sh_degree: int = 3) -> np.ndarray:
    """f32 [n, 17 + 3((d+1)^2 - 1)]: one row per vertex in ``gaussian_ply_attributes`` order (f_rest zeros, normals zeros
    when None)."""
    n = int(xyz.shape[0])
    n_rest = 3 * ((int(sh_degree) + 1) ** 2 - 1)
    f32 = lambda a, c: np.asarray(a, np.float32).reshape(n, c)          # noqa: E731
    nrm = np.zeros((n, 3), np.float32) if normals is None else f32(normals, 3)
    return np.concatenate([f32(xyz, 3), nrm, f32(sh_dc, 3), np.zeros((n, n_rest), np.float32), f32(opacity, 1),
                           f32(scales, 3), f32(rotations, 4)], axis=1)


def write_gaussian_ply(path_out: str, xyz: np.ndarray, sh_dc: np.ndarray, opacity: np.ndarray, scales: np.ndarray,
                       rotations: np.ndarray, normals: Optional[np.ndarray] = None, sh_degree: int = 3) -> None:
    """The 3DGS PLY (``save_ply``) of initialised splats: sh_dc [n,3], opacity [n] (logit), scales [n,3] (log),
    rotations [n,4] (w, x, y, z), e.g. from ``output.init_gaussians``; every property ``<f4``."""
    rec = gaussian_ply_vertices(xyz, sh_dc, opacity, scales, rotations, normals, sh_degree)
    with open(path_out, "wb") as f:
        f.write(gaussian_ply_header(int(xyz.shape[0]), sh_degree))
        rec.astype("<f4").tofile(f)
