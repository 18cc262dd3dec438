"""Device side of the reference's output contract and of the reducers that follow the path.

Mirrors, on tensors that stay on the GPU (SURVEY.md 8a row a15, 8f rows 2 and 4):

* ``to_uint8_rgb``                     reference core/image_utils.py:24-26
* ``write_ply`` / ``write_points3D_bin``   reference core/writers.py:15-46 (files byte-identical; the records are built by
  ``ldp_pack_ply_records`` / ``ldp_pack_points3d_records`` and reach the host as one copy of 15 / 43 bytes per point)
* ``voxel_downsample``                 reference densify.py:29-50 (Open3D voxel grid mean; parity unpinned, see the function)
* ``remove_statistical_outliers``      not in the reference: Open3D's ``remove_statistical_outlier`` (parity unpinned)
* ``estimate_normals``                 not in the reference: oriented normals by PCA over the exact k nearest neighbours
* ``init_gaussians`` / ``write_gaussian_ply``   not in the reference: 3DGS's ``create_from_pcd`` initialisation (scales from
  the exact nearest neighbours, optionally flattened along the normals) and its ``save_ply`` layout
* ``check_depth_consistency``          not in the reference: MVS fusion's visibility test of a cloud against the reference
  views' depth maps (``engine.DepthViews``)
* ``fuse_depth_maps``                  not in the reference: MVS fusion of the reference views' depth maps into one dense
  coloured cloud, each surface point emitted once and averaged over the views that agree with it (optionally in depth and
  normal, with the fused normals)
* ``estimate_depth_normals``           not in the reference: oriented normal maps of the reference views, PCA over each
  pixel's depth-continuous map window
* ``apply_point_cap``                  reference densify.py:110-120 (the indices are numpy's own
  ``default_rng(seed).choice`` on the host - PCG64 + a sequential shuffle, microseconds; only the gather is device work)
* ``subsample_preview_matches``        reference core/pipeline.py:573-582 (debug preview subsample of the kept matches)
* ``IncrementalPly``                   reference core/pipeline.py:508-532: the reference re-concatenates and re-packs EVERY
  point each time it emits an intermediate PLY (O(refs^2) struct.pack calls); here each point is packed once, on the
  device, and an emission is header + one bulk write of the records gathered so far.

No CPU fallback: every function needs the CUDA library (``NativeLibraryError`` otherwise).
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np
import torch

from . import _native as N
from .core.writers import gaussian_ply_header, ply_header

PLY_RECORD_BYTES = 15
PLY_NORMAL_RECORD_BYTES = 27
POINTS3D_RECORD_BYTES = 43


class PackedCloud:
    """A point cloud in ONE device allocation: 16-byte header (int64 point count) | xyz [cap,3] | rgb [cap,3] | err [cap],
    all float32 - so that a rank's whole cloud goes into a single collective (``distributed.all_gather_points``) and a
    launch sequence can append to it without the host learning any count."""
    HEADER_BYTES = 16

    def __init__(self, capacity: int, device, storage: Optional[torch.Tensor] = None) -> None:
        self.capacity = cap = self.round_capacity(capacity)
        nbytes = self.nbytes(cap)
        self.packed = storage if storage is not None else torch.zeros((nbytes,), dtype=torch.uint8, device=device)
        if self.packed.numel() != nbytes or self.packed.dtype != torch.uint8:
            raise ValueError("storage must be a uint8 tensor of PackedCloud.nbytes(capacity) bytes")
        h = self.HEADER_BYTES
        self.count = self.packed[:8].view(torch.int64)                       # [1], stays on the device
        self.xyz = self.packed[h:h + 12 * cap].view(torch.float32).view(cap, 3)
        self.rgb = self.packed[h + 12 * cap:h + 24 * cap].view(torch.float32).view(cap, 3)
        self.err = self.packed[h + 24 * cap:h + 28 * cap].view(torch.float32)

    @staticmethod
    def round_capacity(capacity: int) -> int:
        return (max(1, int(capacity)) + 3) // 4 * 4          # blocks of a gathered [world, nbytes] buffer stay 16-byte aligned

    @classmethod
    def nbytes(cls, capacity: int) -> int:
        return cls.HEADER_BYTES + 28 * cls.round_capacity(capacity)

    def total_points(self) -> int:
        """Synchronises."""
        return int(self.count.item())


class ConcatPlan:
    """``ldp_concat_points`` with its pointer tables built once: concatenates the first ``*count[q]`` rows of every segment
    (the outputs of a launch, or a rank's block of an all-gather) into a ``PackedCloud``, in segment order - the
    reference's final ``np.concatenate`` (core/pipeline.py:914-928) without a host round trip."""

    def __init__(self, xyz, rgb, err, counts, seg_cap: int) -> None:
        n = len(xyz)
        if not (n == len(rgb) == len(err) == len(counts)) or n == 0:
            raise ValueError("one xyz / rgb / err / count tensor per segment")
        dev = xyz[0].device
        if not xyz[0].is_cuda:
            raise N.NativeLibraryError("device tensors required (there is no CPU fallback)")
        for t in list(xyz) + list(rgb) + list(err):
            if t.dtype != torch.float32 or not t.is_contiguous() or t.device != dev:
                raise ValueError("segments must be contiguous float32 tensors on one device")
        for c in counts:
            if c.dtype != torch.int64 or c.device != dev or c.numel() < 1:
                raise ValueError("counts must be int64 device tensors")
        self.n_seg, self.seg_cap, self.device = n, int(seg_cap), dev
        self._keep = (list(xyz), list(rgb), list(err), list(counts))
        tab = np.array([[t.data_ptr() for t in lst] for lst in self._keep], dtype=np.int64)        # [4, n_seg] device pointers
        self.tables = torch.from_numpy(tab).to(dev)
        self.seg_offsets = torch.zeros((n + 1,), dtype=torch.int64, device=dev)

    def run(self, dst: PackedCloud) -> PackedCloud:
        lib = N.load()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        t = self.tables
        N.check(lib.ldp_concat_points(C.c_void_p(t[0].data_ptr()), C.c_void_p(t[1].data_ptr()), C.c_void_p(t[2].data_ptr()),
                                      C.c_void_p(t[3].data_ptr()), self.n_seg, self.seg_cap, C.c_void_p(dst.xyz.data_ptr()),
                                      C.c_void_p(dst.rgb.data_ptr()), C.c_void_p(dst.err.data_ptr()), dst.capacity,
                                      C.c_void_p(self.seg_offsets.data_ptr()), C.c_void_p(dst.count.data_ptr()),
                                      C.c_void_p(stream)), "ldp_concat_points")
        return dst


def concat_launches(outs, dst: Optional[PackedCloud] = None) -> PackedCloud:
    """Kept points of several launches (``DensifyOutputs``, launch order) as one packed cloud."""
    seg_cap = max(int(o.err.shape[0]) for o in outs)
    plan = ConcatPlan([o.xyz for o in outs], [o.rgb for o in outs], [o.err for o in outs],
                      [o.ref_offset[o.n_refs:o.n_refs + 1] for o in outs], seg_cap)
    if dst is None:
        dst = PackedCloud(sum(int(o.err.shape[0]) for o in outs), outs[0].xyz.device)
    plan.run(dst)
    dst._plan = plan                     # keeps the pointer tables alive until the stream is done with them
    return dst


def _lib_and_stream(t: torch.Tensor):
    if not t.is_cuda:
        raise N.NativeLibraryError("device tensors required (there is no CPU fallback)")
    return N.load(), torch.cuda.current_stream(t.device).cuda_stream


def _f32c(t: torch.Tensor, what: str) -> torch.Tensor:
    if t.dtype != torch.float32:
        raise ValueError(f"{what} must be float32")
    return t.contiguous()


def to_uint8_rgb(rgb: torch.Tensor) -> torch.Tensor:
    """``clip(round(rgb * 255), 0, 255).astype(uint8)`` (half to even) of a float32 device tensor."""
    rgb = _f32c(rgb, "rgb")
    lib, stream = _lib_and_stream(rgb)
    out = torch.empty(rgb.shape, dtype=torch.uint8, device=rgb.device)
    N.check(lib.ldp_rgb_to_uint8(C.c_void_p(rgb.data_ptr()), rgb.numel(), C.c_void_p(out.data_ptr()), C.c_void_p(stream)),
            "ldp_rgb_to_uint8")
    return out


def ply_records(xyz: torch.Tensor, rgb: torch.Tensor, n: Optional[int] = None, n_dev: Optional[torch.Tensor] = None,
                out: Optional[torch.Tensor] = None, normals: Optional[torch.Tensor] = None) -> torch.Tensor:
    """uint8 [n * 15] device tensor of PLY vertex records (``<fff`` xyz, ``BBB`` to_uint8_rgb(rgb)); with ``normals``
    [n,3] f32, [n * 27] records (``<fff`` xyz, ``<fff`` normal, ``BBB``).

    ``n`` defaults to all rows.  With ``n_dev`` (an int64 device scalar, e.g. ``outputs.ref_offset[-1:]``) only
    ``min(n, n_dev)`` records are written and nothing synchronises with the host."""
    xyz, rgb = _f32c(xyz, "xyz"), _f32c(rgb, "rgb")
    lib, stream = _lib_and_stream(xyz)
    n = int(xyz.shape[0]) if n is None else int(n)
    rec_bytes = PLY_RECORD_BYTES if normals is None else PLY_NORMAL_RECORD_BYTES
    if out is None:
        out = torch.empty((n * rec_bytes,), dtype=torch.uint8, device=xyz.device)
    n_dev_p = C.c_void_p(n_dev.data_ptr() if n_dev is not None else 0)
    if normals is None:
        N.check(lib.ldp_pack_ply_records(C.c_void_p(xyz.data_ptr()), C.c_void_p(rgb.data_ptr()), n, n_dev_p,
                                         C.c_void_p(out.data_ptr()), C.c_void_p(stream)), "ldp_pack_ply_records")
    else:
        normals = _f32c(normals, "normals")
        if tuple(normals.shape) != tuple(xyz.shape):
            raise ValueError("normals must have the shape of xyz")
        N.check(lib.ldp_pack_ply_normal_records(C.c_void_p(xyz.data_ptr()), C.c_void_p(rgb.data_ptr()),
                                                C.c_void_p(normals.data_ptr()), n, n_dev_p, C.c_void_p(out.data_ptr()),
                                                C.c_void_p(stream)), "ldp_pack_ply_normal_records")
    return out


def points3d_records(xyz: torch.Tensor, rgb: torch.Tensor, err: Optional[torch.Tensor] = None, first_id: int = 1,
                     n: Optional[int] = None, n_dev: Optional[torch.Tensor] = None) -> torch.Tensor:
    """uint8 [n * 43] device tensor of points3D.bin records (``<Q`` id, ``<ddd`` xyz, ``<BBB`` rgb, ``<d`` err)."""
    xyz, rgb = _f32c(xyz, "xyz"), _f32c(rgb, "rgb")
    if err is not None:
        err = _f32c(err, "err")
    lib, stream = _lib_and_stream(xyz)
    n = int(xyz.shape[0]) if n is None else int(n)
    out = torch.empty((n * POINTS3D_RECORD_BYTES,), dtype=torch.uint8, device=xyz.device)
    N.check(lib.ldp_pack_points3d_records(C.c_void_p(xyz.data_ptr()), C.c_void_p(rgb.data_ptr()),
                                          C.c_void_p(err.data_ptr() if err is not None else 0), n,
                                          C.c_void_p(n_dev.data_ptr() if n_dev is not None else 0), C.c_uint64(first_id),
                                          C.c_void_p(out.data_ptr()), C.c_void_p(stream)), "ldp_pack_points3d_records")
    return out


def write_ply(path_out: str, xyz: torch.Tensor, rgb: torch.Tensor, normals: Optional[torch.Tensor] = None) -> None:
    """The reference's ``write_ply(path, xyz, to_uint8_rgb(rgb))`` for device tensors: same bytes.  ``normals`` [n,3] f32
    (``estimate_normals``) adds nx / ny / nz: the bytes of ``core.writers.write_ply(..., normals=)``."""
    n = int(xyz.shape[0])
    rec = ply_records(xyz, rgb, normals=normals).cpu().numpy() if n else np.zeros((0,), np.uint8)
    with open(path_out, "wb") as f:
        f.write(ply_header(n, normals is not None))
        rec.tofile(f)


def write_points3D_bin(path_out: str, xyz: torch.Tensor, rgb: torch.Tensor, errors: Optional[torch.Tensor] = None) -> None:
    """The reference's ``write_points3D_bin(path, xyz, to_uint8_rgb(rgb), errors)`` for device tensors: same bytes."""
    n = int(xyz.shape[0])
    rec = points3d_records(xyz, rgb, errors).cpu().numpy() if n else np.zeros((0,), np.uint8)
    with open(path_out, "wb") as f:
        f.write(np.uint64(n).tobytes())
        rec.tofile(f)


def gather_rows(src: torch.Tensor, sel: torch.Tensor) -> torch.Tensor:
    """``src[sel]`` for a float32 [n] or [n, c] device tensor and int64 device indices."""
    src = _f32c(src, "src")
    lib, stream = _lib_and_stream(src)
    sel = sel.to(device=src.device, dtype=torch.int64).contiguous()
    n, m = int(src.shape[0]), int(sel.numel())
    row = int(src.numel() // max(n, 1)) if n else 1
    out = torch.empty((m,) + tuple(src.shape[1:]), dtype=torch.float32, device=src.device)
    bad = torch.zeros((1,), dtype=torch.int32, device=src.device)
    N.check(lib.ldp_gather_rows(C.c_void_p(src.data_ptr()), row, C.c_void_p(sel.data_ptr()), m, n, C.c_void_p(out.data_ptr()),
                                C.c_void_p(bad.data_ptr()), C.c_void_p(stream)), "ldp_gather_rows")
    if m and int(bad.item()):
        raise IndexError("index out of bounds")
    return out


def apply_point_cap(xyz: torch.Tensor, rgb: torch.Tensor, err: torch.Tensor, max_points: int, seed: int
                    ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """reference densify.py:110-120 on device tensors: keep ``max_points`` rows chosen by
    ``np.random.default_rng(seed).choice(n, size=max_points, replace=False)`` (drawn on the host by numpy itself)."""
    n = int(xyz.shape[0])
    if not (max_points > 0 and n > max_points):
        return xyz, rgb, err
    xyz, rgb, err = _f32c(xyz, "xyz"), _f32c(rgb, "rgb"), _f32c(err, "err")
    lib, stream = _lib_and_stream(xyz)
    sel = np.random.default_rng(seed).choice(n, size=max_points, replace=False)
    sel_dev = torch.from_numpy(np.ascontiguousarray(sel, dtype=np.int64)).to(xyz.device)
    m = int(max_points)
    o_xyz = torch.empty((m, 3), dtype=torch.float32, device=xyz.device)
    o_rgb = torch.empty((m, 3), dtype=torch.float32, device=xyz.device)
    o_err = torch.empty((m,), dtype=torch.float32, device=xyz.device)
    N.check(lib.ldp_gather_points(C.c_void_p(xyz.data_ptr()), C.c_void_p(rgb.data_ptr()), C.c_void_p(err.data_ptr()),
                                  C.c_void_p(sel_dev.data_ptr()), m, n, C.c_void_p(o_xyz.data_ptr()), C.c_void_p(o_rgb.data_ptr()),
                                  C.c_void_p(o_err.data_ptr()), C.c_void_p(0), C.c_void_p(stream)), "ldp_gather_points")
    return o_xyz, o_rgb, o_err


def voxel_downsample(xyz: torch.Tensor, rgb: torch.Tensor, voxel_size: float) -> Tuple[torch.Tensor, torch.Tensor]:
    """reference densify.py:29-50 (Open3D ``voxel_down_sample``) on device tensors: one point per occupied voxel, the f64
    mean of the voxel's points and colours (colours above 1 are taken as 0..255 and scaled), float32 out.
    PARITY UNPINNED (Open3D is not installed here; see include/ldp_b200.h).  Voxels come out in the order of their first
    point.  Synchronises once to learn the voxel count."""
    xyz, rgb = _f32c(xyz, "xyz"), _f32c(rgb[:, :3], "rgb")
    lib, stream = _lib_and_stream(xyz)
    n = int(xyz.shape[0])
    if n == 0:
        return xyz, rgb
    need = C.c_size_t(0)
    N.check(lib.ldp_voxel_workspace_bytes(n, C.byref(need)), "ldp_voxel_workspace_bytes")
    ws = torch.empty((need.value,), dtype=torch.uint8, device=xyz.device)
    o_xyz, o_rgb = torch.empty_like(xyz), torch.empty_like(rgb)
    status = torch.zeros((2,), dtype=torch.int32, device=xyz.device)
    N.check(lib.ldp_voxel_downsample(C.c_void_p(xyz.data_ptr()), C.c_void_p(rgb.data_ptr()), n, C.c_double(float(voxel_size)),
                                     C.c_void_p(o_xyz.data_ptr()), C.c_void_p(o_rgb.data_ptr()), C.c_void_p(status.data_ptr()),
                                     C.c_void_p(ws.data_ptr()), C.c_size_t(need.value), C.c_void_p(stream)), "ldp_voxel_downsample")
    bad, nv = (int(v) for v in status.cpu().tolist())
    if bad:
        raise ValueError("voxel_size is too small for the extent of the cloud (or a coordinate is not finite)")
    return o_xyz[:nv], o_rgb[:nv]


@dataclass
class OutlierResult:
    """What ``remove_statistical_outliers`` returns: the kept rows and the filter's statistics."""
    xyz: torch.Tensor               # [m, 3] f32, kept rows in input order
    rgb: torch.Tensor               # [m, 3] f32
    err: Optional[torch.Tensor]     # [m] f32, None when no err was given
    kept_idx: torch.Tensor          # [m] int64 device, ascending
    mean_dist: torch.Tensor         # [n] f64 device: mean distance of every point to its k nearest (itself included)
    cloud_mean: float
    std_dev: float
    threshold: float


def remove_statistical_outliers(xyz: torch.Tensor, rgb: torch.Tensor, err: Optional[torch.Tensor] = None, *,
                                nb_neighbors: int, std_ratio: float) -> OutlierResult:
    """Open3D's ``remove_statistical_outlier(nb_neighbors, std_ratio)`` on device tensors: a point is kept iff the mean
    distance to its ``nb_neighbors`` nearest points (itself included) is positive and below ``mean + std_ratio * std`` of
    those means over the cloud.  The k-nearest-neighbour search is exact (f64 distances).  PARITY UNPINNED (Open3D is not
    installed here; the rule and the order of its sums are in include/ldp_b200.h).  Synchronises twice: once inside the
    call (the finest grid cell size follows from a trial grid's cell count) and once to learn the kept count."""
    if not 1 <= int(nb_neighbors) <= 64:
        raise ValueError("nb_neighbors must lie in [1, 64]")
    if not float(std_ratio) > 0.0:
        raise ValueError("std_ratio must be positive")
    xyz, rgb = _f32c(xyz, "xyz"), _f32c(rgb, "rgb")
    if err is not None:
        err = _f32c(err, "err")
    lib, stream = _lib_and_stream(xyz)
    dev, n = xyz.device, int(xyz.shape[0])
    need = C.c_size_t(0)
    N.check(lib.ldp_outlier_workspace_bytes(n, int(nb_neighbors), C.byref(need)), "ldp_outlier_workspace_bytes")
    ws = torch.empty((max(1, need.value),), dtype=torch.uint8, device=dev)
    kept = torch.empty((n,), dtype=torch.int64, device=dev)
    mean_dist = torch.empty((n,), dtype=torch.float64, device=dev)
    stats = torch.full((3,), float("nan"), dtype=torch.float64, device=dev)
    status = torch.zeros((3,), dtype=torch.int32, device=dev)
    N.check(lib.ldp_statistical_outliers(C.c_void_p(xyz.data_ptr()), n, int(nb_neighbors), C.c_double(float(std_ratio)),
                                         C.c_void_p(kept.data_ptr()), C.c_void_p(mean_dist.data_ptr()), C.c_void_p(stats.data_ptr()),
                                         C.c_void_p(status.data_ptr()), C.c_void_p(ws.data_ptr()), C.c_size_t(need.value),
                                         C.c_void_p(stream)), "ldp_statistical_outliers")
    status_h, stats_h = status.to("cpu", non_blocking=True), stats.to("cpu", non_blocking=True)
    torch.cuda.current_stream(dev).synchronize()
    bad, m = int(status_h[0]), int(status_h[1])
    if bad:
        raise ValueError("a coordinate is not finite")
    kept = kept[:m]
    o_xyz = torch.empty((m, 3), dtype=torch.float32, device=dev)
    o_rgb = torch.empty((m, 3), dtype=torch.float32, device=dev)
    o_err = torch.empty((m,), dtype=torch.float32, device=dev) if err is not None else None
    N.check(lib.ldp_gather_points(C.c_void_p(xyz.data_ptr()), C.c_void_p(rgb.data_ptr()),
                                  C.c_void_p(err.data_ptr() if err is not None else 0), C.c_void_p(kept.data_ptr()), m, n,
                                  C.c_void_p(o_xyz.data_ptr()), C.c_void_p(o_rgb.data_ptr()),
                                  C.c_void_p(o_err.data_ptr() if o_err is not None else 0), C.c_void_p(0), C.c_void_p(stream)),
            "ldp_gather_points")
    mu, sd, thr = (float(v) for v in stats_h.tolist())
    return OutlierResult(xyz=o_xyz, rgb=o_rgb, err=o_err, kept_idx=kept, mean_dist=mean_dist, cloud_mean=mu, std_dev=sd, threshold=thr)


@dataclass
class NormalResult:
    """What ``estimate_normals`` returns (device tensors, rows in input order)."""
    normals: torch.Tensor               # [n, 3] f32 unit normals; (0, 0, 0) where undefined
    curvature: torch.Tensor             # [n] f32 surface variation l0 / (l0 + l1 + l2); NaN where undefined
    neighbors: Optional[torch.Tensor]   # [n, k_eff] int32 neighbourhoods, ascending (d^2, index); None unless asked for
    undefined: int                      # points whose normal is undefined (fewer than 3 points, duplicates, a line)


def estimate_normals(xyz: torch.Tensor, *, nb_neighbors: int, centers: Optional[torch.Tensor] = None,
                     center_idx: Optional[torch.Tensor] = None, return_neighbors: bool = False) -> NormalResult:
    """Oriented normals of a device cloud: PCA over the exact ``nb_neighbors`` nearest points of every point (itself
    included, ties by index), the eigenvector of the smallest eigenvalue of their f64 covariance.  ``centers`` [c,3]
    (e.g. camera centres) orients every normal toward ``centers[center_idx[i]]`` (``centers[0]`` without ``center_idx``);
    without ``centers`` the sign is canonical (largest component positive).  The rule is in include/ldp_b200.h.
    Synchronises twice: once inside the call (the grid's cell size) and once to read the status."""
    if not 3 <= int(nb_neighbors) <= 64:
        raise ValueError("nb_neighbors must lie in [3, 64]")
    if center_idx is not None and centers is None:
        raise ValueError("center_idx needs centers")
    xyz = _f32c(xyz, "xyz")
    lib, stream = _lib_and_stream(xyz)
    dev, n = xyz.device, int(xyz.shape[0])
    k_eff = min(int(nb_neighbors), n)
    n_centers = 0
    if centers is not None:
        centers = _f32c(centers, "centers").to(dev)
        if centers.dim() != 2 or centers.shape[1] != 3 or centers.shape[0] < 1:
            raise ValueError("centers must be a [c, 3] float32 tensor with c >= 1")
        n_centers = int(centers.shape[0])
    if center_idx is not None:
        center_idx = center_idx.to(device=dev, dtype=torch.int32).contiguous()
        if center_idx.shape != (n,):
            raise ValueError("center_idx must hold one index per point")
    need = C.c_size_t(0)
    N.check(lib.ldp_normals_workspace_bytes(n, int(nb_neighbors), C.byref(need)), "ldp_normals_workspace_bytes")
    ws = torch.empty((max(1, need.value),), dtype=torch.uint8, device=dev)
    normals = torch.empty((n, 3), dtype=torch.float32, device=dev)
    curvature = torch.empty((n,), dtype=torch.float32, device=dev)
    nbrs = torch.empty((n, k_eff), dtype=torch.int32, device=dev) if return_neighbors else None
    status = torch.zeros((3,), dtype=torch.int32, device=dev)
    ptr = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)          # noqa: E731
    N.check(lib.ldp_estimate_normals(ptr(xyz), n, int(nb_neighbors), ptr(centers), n_centers, ptr(center_idx), ptr(normals),
                                     ptr(curvature), ptr(nbrs), ptr(status), ptr(ws), C.c_size_t(need.value),
                                     C.c_void_p(stream)), "ldp_estimate_normals")
    bad, undefined, _ = (int(v) for v in status.cpu().tolist())
    if bad & 1:
        raise ValueError("a coordinate is not finite")
    if bad & 2:
        raise ValueError("a centre index is out of range")
    return NormalResult(normals=normals, curvature=curvature, neighbors=nbrs, undefined=undefined)


@dataclass
class GaussianInit:
    """What ``init_gaussians`` returns: 3DGS's initial parameters (device tensors, rows in input order, all f32)."""
    sh_dc: torch.Tensor                 # [n, 3] (rgb - 0.5) / C0, 3DGS's RGB2SH
    opacity: torch.Tensor               # [n] logit of the initial opacity
    scales: torch.Tensor                # [n, 3] log scales; the third lies along the normal
    rotations: torch.Tensor             # [n, 4] unit quaternions (w, x, y, z)
    dist2: torch.Tensor                 # [n] mean squared distance to the k nearest other points, clamped to 1e-7
    undefined: int                      # points without a usable normal: identity rotation, isotropic scales


def init_gaussians(xyz: torch.Tensor, rgb: torch.Tensor, *, normals: Optional[torch.Tensor] = None, nb_neighbors: int = 3,
                   opacity: float = 0.1, flatten: float = 1.0) -> GaussianInit:
    """graphdeco 3DGS's ``create_from_pcd`` on a device cloud: scale from the mean squared distance to the ``nb_neighbors``
    nearest other points (exact; 3DGS uses simple-knn's ``distCUDA2`` with 3), SH DC from ``rgb`` in [0, 1], opacity
    ``inverse_sigmoid(opacity)``.  With ``normals`` (e.g. ``estimate_normals``) each splat is rotated so that its third axis
    lies along its normal, and ``flatten`` < 1 shrinks that axis by that factor: discs in the surface.  The rule is in
    include/ldp_b200.h.  Synchronises twice: once inside the call (the grid's cell size) and once to read the status."""
    if not 1 <= int(nb_neighbors) <= 63:
        raise ValueError("nb_neighbors must lie in [1, 63]")
    if not 0.0 < float(opacity) < 1.0:
        raise ValueError("opacity must lie in (0, 1)")
    if not 0.0 < float(flatten) <= 1.0:
        raise ValueError("flatten must lie in (0, 1]")
    if float(flatten) < 1.0 and normals is None:
        raise ValueError("flatten < 1 needs normals")
    xyz, rgb = _f32c(xyz, "xyz"), _f32c(rgb, "rgb")
    if tuple(rgb.shape) != tuple(xyz.shape):
        raise ValueError("rgb must have the shape of xyz")
    if normals is not None:
        normals = _f32c(normals, "normals")
        if tuple(normals.shape) != tuple(xyz.shape):
            raise ValueError("normals must have the shape of xyz")
    lib, stream = _lib_and_stream(xyz)
    dev, n = xyz.device, int(xyz.shape[0])
    need = C.c_size_t(0)
    N.check(lib.ldp_gaussian_workspace_bytes(n, int(nb_neighbors), C.byref(need)), "ldp_gaussian_workspace_bytes")
    ws = torch.empty((max(1, need.value),), dtype=torch.uint8, device=dev)
    f32 = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)      # noqa: E731
    g = GaussianInit(sh_dc=f32(n, 3), opacity=f32(n), scales=f32(n, 3), rotations=f32(n, 4), dist2=f32(n), undefined=0)
    status = torch.zeros((3,), dtype=torch.int32, device=dev)
    ptr = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)          # noqa: E731
    N.check(lib.ldp_gaussian_init(ptr(xyz), ptr(rgb), ptr(normals), n, int(nb_neighbors), float(opacity), float(flatten),
                                  ptr(g.sh_dc), ptr(g.opacity), ptr(g.scales), ptr(g.rotations), ptr(g.dist2), ptr(status),
                                  ptr(ws), C.c_size_t(need.value), C.c_void_p(stream)), "ldp_gaussian_init")
    bad, undefined, _ = (int(v) for v in status.cpu().tolist())
    if bad & 1:
        raise ValueError("a coordinate is not finite")
    g.undefined = undefined
    return g


@dataclass
class DepthConsistency:
    """What ``check_depth_consistency`` returns (device tensors)."""
    kept_idx: torch.Tensor              # [m] int64, the kept points in ascending index (apply to every per-point array)
    n_consistent: torch.Tensor          # [n] int32: other views whose depth agrees with the point
    n_violations: torch.Tensor          # [n] int32: other views that see their surface behind the point (look through it)


def check_depth_consistency(xyz: torch.Tensor, views, *, owner=None, rel_tol: float = 0.01, min_views: int = 1,
                            max_violations: int = 0) -> DepthConsistency:
    """MVS fusion's visibility test on a device cloud: every point is projected into every view of ``views``
    (``engine.DepthViews``) but its own (``owner[i]``, the view index it came from, or -1; None = no owner) and compared
    with the depth that view's map holds at the pixel.  A view whose depth agrees within ``rel_tol`` of it supports the
    point; a view whose surface lies clearly behind the point looks through it (a violation).  The point is kept iff at
    least ``min_views`` views support it and at most ``max_violations`` look through it.  The rule (f64 projection without
    FMA, nearest map pixel) is in include/ldp_b200.h.  Raises on a non-finite coordinate or an owner outside [-1, V).
    Synchronises once, to read the kept count."""
    if not 0.0 < float(rel_tol) < 1.0:
        raise ValueError("rel_tol must lie in (0, 1)")
    if int(min_views) < 0 or int(max_violations) < 0:
        raise ValueError("min_views and max_violations must be >= 0")
    xyz = _f32c(xyz, "xyz")
    lib, stream = _lib_and_stream(xyz)
    if xyz.dim() != 2 or xyz.shape[1] != 3:
        raise ValueError("xyz must be [n, 3]")
    dev, n = xyz.device, int(xyz.shape[0])
    if views.device != dev:
        raise ValueError("the cloud and the depth maps must be on one device")
    if owner is not None:
        owner = torch.as_tensor(owner).to(device=dev, dtype=torch.int32).contiguous()
        if tuple(owner.shape) != (n,):
            raise ValueError("owner must hold one view index per point")
    need = C.c_size_t(0)
    N.check(lib.ldp_consistency_workspace_bytes(n, C.byref(need)), "ldp_consistency_workspace_bytes")
    ws = torch.empty((max(1, need.value),), dtype=torch.uint8, device=dev)
    kept = torch.empty((n,), dtype=torch.int64, device=dev)
    nc = torch.empty((n,), dtype=torch.int32, device=dev)
    nv = torch.empty((n,), dtype=torch.int32, device=dev)
    status = torch.zeros((2,), dtype=torch.int32, device=dev)
    ptrs, P, S, lens = views.tables()
    ptr = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)          # noqa: E731
    N.check(lib.ldp_depth_consistency(ptr(xyz), n, ptr(owner), ptr(ptrs), views.H, views.W, ptr(P), ptr(S), ptr(lens), len(views),
                                      float(rel_tol), int(min_views), int(max_violations), ptr(nc), ptr(nv), ptr(kept), ptr(status),
                                      ptr(ws), C.c_size_t(need.value), C.c_void_p(stream)), "ldp_depth_consistency")
    bad, m = (int(v) for v in status.cpu().tolist())
    if bad & 1:
        raise ValueError("a coordinate is not finite")
    if bad & 2:
        raise ValueError("an owner index is out of range")
    return DepthConsistency(kept_idx=kept[:m], n_consistent=nc, n_violations=nv)


@dataclass
class FusedCloud:
    """What ``fuse_depth_maps`` returns (device tensors, one row per emitted point, ascending ``source``).  ``write_ply`` and
    ``write_points3D_bin`` take ``xyz`` / ``rgb`` (/ ``err``) like any other cloud."""
    xyz: torch.Tensor                   # [m, 3] f32: mean of the point and its members
    rgb: torch.Tensor                   # [m, 3] f32: mean colour, in [0, 1]
    err: torch.Tensor                   # [m] f32: reprojection error of the emitting pixel
    n_views: torch.Tensor               # [m] int32: views averaged (members + 1)
    n_consistent: torch.Tensor          # [m] int32: other views whose depth agrees with the emitting pixel
    source: torch.Tensor                # [m] int64: emitting pixel, view * H * W + pixel index
    normals: Optional[torch.Tensor] = None   # [m, 3] f32 unit normals averaged over the point and its members (max_normal_angle)


def fuse_depth_maps(views, *, rel_tol: float = 0.01, min_views: int = 1, max_violations: int = 0,
                    max_normal_angle: Optional[float] = None) -> FusedCloud:
    """MVS fusion of the maps of ``views`` (``engine.DepthViews`` whose views carry xyz and rgb maps) into one cloud in which
    each surface point appears once: a pixel is kept iff at least ``min_views`` other views agree with its depth (within
    ``rel_tol``) and at most ``max_violations`` look through it (``check_depth_consistency``'s test); a kept pixel is
    emitted iff no lower view holds a kept pixel that agrees with it, and its xyz and rgb are averaged over itself and the
    kept pixels of the views that agree with it.  The rule is in include/ldp_b200.h (ldp_fuse_depth_maps).  Raises on a
    view without xyz or rgb maps and on a non-finite xyz where the depth is finite.  Synchronises once, to read the
    emitted count.

    ``max_normal_angle`` (degrees in (0, 90); COLMAP: 10) adds COLMAP fusion's normal test: a view agrees only where its
    normal map (``DepthViews.add(..., normals=)``, e.g. ``estimate_depth_normals``) is within that angle of the pixel's
    normal too, a pixel without a normal is not kept, and ``FusedCloud.normals`` holds the normalised sum of the point's and
    its members' normals (include/ldp_b200.h: ldp_fuse_depth_maps_oriented).  Raises if a view has no normal map.
    None: no normal test and no normals."""
    if not 0.0 < float(rel_tol) < 1.0:
        raise ValueError("rel_tol must lie in (0, 1)")
    if max_normal_angle is not None and not 0.0 < float(max_normal_angle) < 90.0:
        raise ValueError("max_normal_angle must lie in (0, 90) degrees (None = off)")
    if int(min_views) < 0 or int(max_violations) < 0:
        raise ValueError("min_views and max_violations must be >= 0")
    dev = views.device
    if dev.type != "cuda":
        raise N.NativeLibraryError("fusion runs on a CUDA device (there is no CPU fallback)")
    V, H, W = len(views), views.H, views.W
    if V * H * W >= 2 ** 31:
        raise ValueError("fusion needs n_views * H * W < 2^31")
    xyz_p, rgb_p, err_p = views.fusion_tables()
    nrm_p = views.normal_table() if max_normal_angle is not None else None
    lib, stream = N.load(), torch.cuda.current_stream(dev).cuda_stream
    need = C.c_size_t(0)
    N.check(lib.ldp_fuse_workspace_bytes(V, H, W, C.byref(need)), "ldp_fuse_workspace_bytes")
    ws = torch.empty((max(1, need.value),), dtype=torch.uint8, device=dev)
    cap = max(1, V * H * W)
    f32 = dict(dtype=torch.float32, device=dev)
    xyz, rgb, err = torch.empty((cap, 3), **f32), torch.empty((cap, 3), **f32), torch.empty((cap,), **f32)
    nv, nc = torch.empty((cap,), dtype=torch.int32, device=dev), torch.empty((cap,), dtype=torch.int32, device=dev)
    src = torch.empty((cap,), dtype=torch.int64, device=dev)
    status = torch.zeros((2,), dtype=torch.int32, device=dev)
    ptrs, P, S, lens = views.tables()
    ptr = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)          # noqa: E731
    nrm = None
    if nrm_p is None:
        N.check(lib.ldp_fuse_depth_maps(ptr(ptrs), ptr(xyz_p), ptr(rgb_p), ptr(err_p), V, H, W, ptr(P), ptr(S), ptr(lens),
                                        float(rel_tol), int(min_views), int(max_violations), ptr(xyz), ptr(rgb), ptr(err), ptr(nv),
                                        ptr(nc), ptr(src), ptr(status), ptr(ws), C.c_size_t(need.value), C.c_void_p(stream)),
                "ldp_fuse_depth_maps")
    else:
        nrm = torch.empty((cap, 3), **f32)
        cos_max = math.cos(math.radians(float(max_normal_angle)))
        N.check(lib.ldp_fuse_depth_maps_oriented(ptr(ptrs), ptr(xyz_p), ptr(rgb_p), ptr(err_p), ptr(nrm_p), V, H, W, ptr(P), ptr(S),
                                                 ptr(lens), float(rel_tol), cos_max, int(min_views), int(max_violations), ptr(xyz),
                                                 ptr(rgb), ptr(err), ptr(nrm), ptr(nv), ptr(nc), ptr(src), ptr(status), ptr(ws),
                                                 C.c_size_t(need.value), C.c_void_p(stream)), "ldp_fuse_depth_maps_oriented")
    bad, m = (int(v) for v in status.cpu().tolist())
    if bad & 1:
        raise ValueError("a view's xyz map is not finite where its depth is")
    if bad & 2:
        raise ValueError("a view's map pointer is NULL")
    # copies of the first m rows: the capacity (one row per map pixel) is released
    return FusedCloud(xyz=xyz[:m].clone(), rgb=rgb[:m].clone(), err=err[:m].clone(), n_views=nv[:m].clone(),
                      n_consistent=nc[:m].clone(), source=src[:m].clone(), normals=None if nrm is None else nrm[:m].clone())


@dataclass
class DepthNormals:
    """What ``estimate_depth_normals`` returns (device tensors, one map per view of the ``DepthViews``)."""
    normals: torch.Tensor               # [V, H, W, 3] f32 unit normals facing the view's camera; NaN where there is none
    curvature: torch.Tensor             # [V, H, W] f32 surface variation l0 / (l0 + l1 + l2); NaN where there is no normal
    undefined: int                      # pixels with a depth but no normal (fewer than 3 window pixels, a line)


def estimate_depth_normals(views, *, radius: int = 2, rel_tol: float = 0.05) -> DepthNormals:
    """Oriented normal maps of ``views`` (``engine.DepthViews`` whose views carry xyz maps): for every pixel with a depth,
    PCA over the xyz of the pixels of its (2 radius + 1)^2 map window whose depth lies within ``rel_tol`` of its own (the
    window stops at depth edges), the eigenvector of the smallest eigenvalue of their f64 covariance, facing the view's
    camera centre (``CameraRecord.C``).  A slice ``normals[v]`` is what ``DepthViews.add(..., normals=)`` takes.  The rule
    is in include/ldp_b200.h (ldp_depth_normals).  Raises on a view without an xyz map and on a non-finite xyz where the
    depth is finite.  Synchronises once, to read the status."""
    if not 1 <= int(radius) <= 3:
        raise ValueError("radius must lie in [1, 3]")
    if not 0.0 < float(rel_tol) < 1.0:
        raise ValueError("rel_tol must lie in (0, 1)")
    dev = views.device
    if dev.type != "cuda":
        raise N.NativeLibraryError("normal maps run on a CUDA device (there is no CPU fallback)")
    V, H, W = len(views), views.H, views.W
    if V * H * W >= 2 ** 31:
        raise ValueError("normal maps need n_views * H * W < 2^31")
    xyz_p = views.xyz_table()
    ptrs = views.tables()[0]
    centers = np.zeros((max(V, 1), 3), np.float32)
    for v, cam in enumerate(views.cameras):
        centers[v] = np.asarray(cam.C, np.float64).reshape(3).astype(np.float32)
    centers_dev = torch.from_numpy(centers).to(dev)
    normals = torch.empty((V, H, W, 3), dtype=torch.float32, device=dev)
    curvature = torch.empty((V, H, W), dtype=torch.float32, device=dev)
    status = torch.zeros((2,), dtype=torch.int32, device=dev)
    lib, stream = N.load(), torch.cuda.current_stream(dev).cuda_stream
    ptr = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)          # noqa: E731
    N.check(lib.ldp_depth_normals(ptr(ptrs), ptr(xyz_p), V, H, W, ptr(centers_dev), int(radius), float(rel_tol), ptr(normals),
                                  ptr(curvature), ptr(status), C.c_void_p(stream)), "ldp_depth_normals")
    bad, undefined = (int(v) for v in status.cpu().tolist())
    if bad & 1:
        raise ValueError("a view's xyz map is not finite where its depth is")
    if bad & 2:
        raise ValueError("a view's map pointer is NULL")
    return DepthNormals(normals=normals, curvature=curvature, undefined=undefined)


def gaussian_record_bytes(sh_degree: int) -> int:
    """68, 104, 164 or 248 bytes per vertex of the 3DGS PLY for SH degree 0..3."""
    return 4 * (17 + 3 * ((int(sh_degree) + 1) ** 2 - 1))


def gaussian_ply_records(xyz: torch.Tensor, g: GaussianInit, normals: Optional[torch.Tensor] = None, sh_degree: int = 3,
                         n: Optional[int] = None, n_dev: Optional[torch.Tensor] = None) -> torch.Tensor:
    """uint8 [n * gaussian_record_bytes(sh_degree)] device tensor of 3DGS PLY vertices (``core.writers.gaussian_ply_vertices``
    order: x y z nx ny nz f_dc f_rest opacity scale rot, all ``<f4``; f_rest zeros, normals zeros when None).  ``n`` and
    ``n_dev`` as for ``ply_records``."""
    if not 0 <= int(sh_degree) <= 3:
        raise ValueError("sh_degree must lie in [0, 3]")
    xyz = _f32c(xyz, "xyz")
    arrs = [_f32c(t, name) for t, name in ((g.sh_dc, "sh_dc"), (g.opacity, "opacity"), (g.scales, "scales"),
                                           (g.rotations, "rotations"))]
    if normals is not None:
        normals = _f32c(normals, "normals")
        if tuple(normals.shape) != tuple(xyz.shape):
            raise ValueError("normals must have the shape of xyz")
    lib, stream = _lib_and_stream(xyz)
    n = int(xyz.shape[0]) if n is None else int(n)
    out = torch.empty((n * gaussian_record_bytes(sh_degree),), dtype=torch.uint8, device=xyz.device)
    ptr = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)          # noqa: E731
    N.check(lib.ldp_pack_gaussian_ply_records(ptr(xyz), ptr(normals), *(ptr(t) for t in arrs), n, ptr(n_dev), int(sh_degree),
                                              ptr(out), C.c_void_p(stream)), "ldp_pack_gaussian_ply_records")
    return out


def write_gaussian_ply(path_out: str, xyz: torch.Tensor, g: GaussianInit, normals: Optional[torch.Tensor] = None,
                       sh_degree: int = 3) -> None:
    """The 3DGS PLY of ``init_gaussians``' splats, loadable by 3DGS-style trainers and viewers: the bytes of
    ``core.writers.write_gaussian_ply`` on the same arrays."""
    n = int(xyz.shape[0])
    rec = gaussian_ply_records(xyz, g, normals, sh_degree).cpu().numpy() if n else np.zeros((0,), np.uint8)
    with open(path_out, "wb") as f:
        f.write(gaussian_ply_header(n, sh_degree))
        rec.tofile(f)


PREVIEW_MAX_MATCHES = 10000       # reference core/pipeline.py:50 _PREVIEW_MAX_MATCHES


def preview_seed(ref_id: int, nbr_id: int) -> int:
    """reference core/pipeline.py:574-575"""
    seed = ((int(ref_id) & 0xFFFF_FFFF) * 73856093) ^ ((int(nbr_id) & 0xFFFF_FFFF) * 19349663)
    return seed & 0xFFFF_FFFF


def subsample_preview_matches(matches: torch.Tensor, cert_norm: torch.Tensor, ref_id: int, nbr_id: int,
                              max_matches: int = PREVIEW_MAX_MATCHES) -> Tuple[torch.Tensor, torch.Tensor]:
    """reference core/pipeline.py:573-582 on the device-resident debug outputs of a pair (``dbg_matches`` [K,4],
    ``dbg_cert`` [K]): at most ``max_matches`` rows, chosen by ``default_rng(pair seed).choice`` on the host."""
    k = int(matches.shape[0])
    if not (k > max_matches > 0):
        return matches, cert_norm
    sel = np.random.default_rng(preview_seed(ref_id, nbr_id)).choice(k, size=max_matches, replace=False)
    sel_dev = torch.from_numpy(np.ascontiguousarray(sel, dtype=np.int64)).to(matches.device)
    return gather_rows(matches, sel_dev), gather_rows(cert_norm, sel_dev)


class IncrementalPly:
    """Intermediate PLY emission without the reference's quadratic cost (core/pipeline.py:508-532).

    ``append`` packs the new points' 15-byte records on the device and keeps them on the host; ``emit`` writes
    header + all records so far - the same bytes as ``write_ply(path, concatenate(xyz_parts), to_uint8_rgb(concatenate(rgb_parts)))``."""

    def __init__(self) -> None:
        self._parts = []
        self.n_points = 0

    def append(self, xyz: torch.Tensor, rgb: torch.Tensor) -> None:
        n = int(xyz.shape[0])
        if n == 0:
            return
        self._parts.append(ply_records(xyz, rgb).cpu().numpy())
        self.n_points += n

    def emit(self, path_out: str) -> None:
        with open(path_out, "wb") as f:
            f.write(ply_header(self.n_points))
            for p in self._parts:
                p.tofile(f)


def write_depth_map(path_out: str, depth) -> None:
    """One reference view's depth map (``DensifyEngine.depth_maps(...).depth[r]``, a tensor or array [H, W]) as a float32
    ``.npy`` [H, W]; NaN = no depth.  Pixel (y, x) of the map is map pixel i = y * W + x, indexed like the certainty planes;
    its camera pixel is the decoded ``(uA_obs, vA_obs)`` of its own warp row: ((xA + 1) / 2 * (w_match - 1) * sxA,
    (yA + 1) / 2 * (h_match - 1) * syA) with sxA = width / w_match, syA = height / h_match (the reference camera's full
    resolution over the matcher's), in float32 as the kernels decode it.  The value is that camera's z of the kept point
    (the distance along its optical axis), not a distance along the ray.  For the synthetic grid of ``synth``, whose warp rows
    hold each map pixel's own grid coordinates (gx, gy) in [-1, 1] as (xA, yA), that is
    ((gx + 1) / 2 * (w_match - 1) * sxA, (gy + 1) / 2 * (h_match - 1) * syA)."""
    if isinstance(depth, torch.Tensor):
        depth = depth.detach().cpu().numpy()
    a = np.asarray(depth)
    if a.ndim != 2:
        raise ValueError(f"a depth map is [H, W], got shape {a.shape}")
    np.save(path_out, np.ascontiguousarray(a, dtype=np.float32), allow_pickle=False)
