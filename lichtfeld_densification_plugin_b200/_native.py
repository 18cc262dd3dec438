"""ctypes binding of csrc/libldp_b200.so (C ABI: include/ldp_b200.h).

There is no fallback: if the shared library is missing or does not match the header, every product
entry point raises ``NativeLibraryError``.  The library is built in-tree by ``build.py`` (nvcc, sm_100a).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

from . import build as _build

LDP_ABI_VERSION = 16
LDP_MAX_NN = 16
LDP_MAX_BINS = 4096

LDP_OK = 0
LDP_REF_OK = 0
LDP_REF_EMPTY = 1
LDP_REF_FEWER_NONZERO = 2
LDP_REF_BAD_WEIGHTS = 3
LDP_REF_PSUM = 4
LDP_REF_UNIFORMS_EXHAUSTED = 5
LDP_REF_ROUNDS_EXCEEDED = 6
LDP_REF_NO_NEIGHBOURS = 7
LDP_REF_INEXACT_SCAN = 0x100
LDP_REF_CODE_MASK = 0xFF

LDP_RNG_PHILOX = 0
LDP_RNG_EXPLICIT = 1

LDP_LENS_PINHOLE = 0
LDP_LENS_OPENCV = 1
LDP_LENS_FISHEYE = 2

REF_STATUS_MESSAGES = {
    LDP_REF_EMPTY: "all sampling weights are zero",
    LDP_REF_FEWER_NONZERO: "Fewer non-zero entries in p than size",
    LDP_REF_BAD_WEIGHTS: "probabilities contain NaN or are not non-negative",
    LDP_REF_PSUM: "probabilities do not sum to 1",
    LDP_REF_UNIFORMS_EXHAUSTED: "explicit uniform stream exhausted",
    LDP_REF_ROUNDS_EXCEEDED: "weighted draw did not terminate",
    LDP_REF_NO_NEIGHBOURS: "reference view has no neighbours",
}


class NativeLibraryError(RuntimeError):
    pass


class LdpParams(C.Structure):
    _fields_ = [
        ("n_refs", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
        ("w_match", C.c_int32), ("h_match", C.c_int32),
        ("matches_per_ref", C.c_int32), ("border", C.c_int32), ("tiles", C.c_int32),
        ("sample_cap", C.c_float), ("reproj_thresh", C.c_float), ("min_parallax_deg", C.c_float),
        ("sampson_thresh", C.c_double),
        ("no_filter", C.c_int32), ("collect_debug", C.c_int32), ("rng_mode", C.c_int32), ("scalar_loads", C.c_int32),
        ("nn_max", C.c_int32), ("prologue", C.c_int32),
        ("certainty_floor", C.c_float), ("no_warped_masks", C.c_int32),
        ("seed", C.c_uint64), ("uniforms_per_ref", C.c_int64),
        ("sm_reserve", C.c_int32), ("lens", C.c_int32),
        ("multiview", C.c_int32), ("multiview_min_cert", C.c_float),
    ]


class LdpLens(C.Structure):
    _fields_ = [
        ("model", C.c_int32), ("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float),
        ("pad", C.c_int32), ("k", C.c_double * 8),
    ]


class LdpRefDesc(C.Structure):
    _fields_ = [
        ("cert", C.c_uint64 * LDP_MAX_NN),
        ("warp", C.c_uint64 * LDP_MAX_NN),
        ("image", C.c_uint64),
        ("nn", C.c_int32), ("img_w", C.c_int32), ("img_h", C.c_int32), ("rng_stream", C.c_uint32),
        ("weight_sum_override", C.c_float),
        ("sxA", C.c_float), ("syA", C.c_float), ("sx_img", C.c_float), ("sy_img", C.c_float),
        ("P1", C.c_float * 12), ("C1", C.c_float * 3),
        ("P2", (C.c_float * 12) * LDP_MAX_NN), ("C2", (C.c_float * 3) * LDP_MAX_NN),
        ("F", (C.c_float * 9) * LDP_MAX_NN),
        ("sxB", C.c_float * LDP_MAX_NN), ("syB", C.c_float * LDP_MAX_NN),
        ("group", C.c_int32 * LDP_MAX_NN),
        ("mask_a", C.c_uint64), ("mask_b", C.c_uint64 * LDP_MAX_NN),
        ("mask_w", C.c_int32), ("mask_h", C.c_int32), ("mask_sx", C.c_float), ("mask_sy", C.c_float),
        ("lens_a", LdpLens), ("lens_b", LdpLens * LDP_MAX_NN),
    ]


class LdpOutputs(C.Structure):
    _fields_ = [
        ("xyz", C.c_uint64), ("rgb", C.c_uint64), ("err", C.c_uint64), ("capacity", C.c_int64),
        ("ref_offset", C.c_uint64), ("status", C.c_uint64), ("n_samples", C.c_uint64),
        ("group_count", C.c_uint64), ("group_order", C.c_uint64),
        ("dbg_matches", C.c_uint64), ("dbg_cert", C.c_uint64), ("sel_idx", C.c_uint64),
        ("sample_flags", C.c_uint64), ("sample_xyzerr", C.c_uint64),
        ("uniforms_used", C.c_uint64), ("rounds", C.c_uint64), ("weight_sum", C.c_uint64),
        ("view_mask", C.c_uint64),
    ]


REF_DESC_DTYPE = np.dtype(LdpRefDesc)

EXPORTS = [
    "ldp_abi_version", "ldp_last_error_string", "ldp_sel_capacity", "ldp_workspace_bytes",
    "ldp_densify_refs", "ldp_sample_refs", "ldp_triangulate_samples", "ldp_postprocess_certainty", "ldp_last_launch_count",
    "ldp_struct_size", "ldp_profile_enable", "ldp_profile_read", "ldp_profile_name", "ldp_debug_set_cluster", "ldp_debug_last_cluster", "ldp_debug_set_subbatches", "ldp_debug_read_clocks", "ldp_debug_launch_stream",
    "ldp_pack_ply_records", "ldp_pack_points3d_records", "ldp_rgb_to_uint8", "ldp_gather_points", "ldp_gather_rows", "ldp_concat_points", "ldp_scatter_points",
    "ldp_select_kcenters", "ldp_nearest_neighbors", "ldp_voxel_workspace_bytes", "ldp_voxel_downsample", "ldp_set_sm_reserve",
    "ldp_undistort_points", "ldp_debug_force_fixup", "ldp_debug_read_fixups",
    "ldp_outlier_workspace_bytes", "ldp_statistical_outliers", "ldp_debug_outlier_max_shells",
    "ldp_normals_workspace_bytes", "ldp_estimate_normals", "ldp_pack_ply_normal_records",
]

_lock = threading.Lock()
_lib = None


def library_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = False):
    """Load (once) and return the ctypes handle.  Raises NativeLibraryError when unavailable."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = library_path()
        if not os.path.isfile(path):
            if build_if_missing:
                _build.build()
            else:
                raise NativeLibraryError(
                    f"{path} is missing: build it with `python -m lichtfeld_densification_plugin_b200.build` "
                    "(there is no CPU fallback)")
        try:
            lib = C.CDLL(path)
        except OSError as exc:
            raise NativeLibraryError(f"cannot load {path}: {exc}") from exc
        for name in EXPORTS:
            if not hasattr(lib, name):
                raise NativeLibraryError(f"{path} does not export {name}")
        lib.ldp_abi_version.restype = C.c_int
        lib.ldp_last_error_string.restype = C.c_char_p
        lib.ldp_sel_capacity.restype = C.c_int64
        lib.ldp_sel_capacity.argtypes = [C.c_int32]
        lib.ldp_struct_size.restype = C.c_int64
        lib.ldp_struct_size.argtypes = [C.c_int]
        lib.ldp_last_launch_count.restype = C.c_int
        lib.ldp_profile_enable.restype = C.c_int
        lib.ldp_profile_enable.argtypes = [C.c_int]
        lib.ldp_profile_read.restype = C.c_int
        lib.ldp_debug_last_cluster.restype = C.c_int
        lib.ldp_debug_set_cluster.restype = C.c_int
        lib.ldp_debug_set_cluster.argtypes = [C.c_int]
        lib.ldp_profile_name.restype = C.c_char_p
        lib.ldp_profile_name.argtypes = [C.c_int]
        lib.ldp_profile_read.argtypes = [C.POINTER(C.c_float), C.c_int]
        lib.ldp_workspace_bytes.restype = C.c_int
        lib.ldp_workspace_bytes.argtypes = [C.POINTER(LdpParams), C.POINTER(C.c_size_t)]
        for fn in (lib.ldp_densify_refs, lib.ldp_sample_refs):
            fn.restype = C.c_int
            fn.argtypes = [C.POINTER(LdpParams), C.c_void_p, C.c_void_p, C.POINTER(LdpOutputs), C.c_void_p,
                           C.c_size_t, C.c_void_p]
        lib.ldp_triangulate_samples.restype = C.c_int
        lib.ldp_triangulate_samples.argtypes = [C.POINTER(LdpParams), C.c_void_p, C.POINTER(LdpOutputs), C.c_void_p,
                                                C.c_size_t, C.c_void_p]
        lib.ldp_debug_launch_stream.restype = C.c_int
        lib.ldp_debug_launch_stream.argtypes = [C.POINTER(LdpParams), C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int]
        lib.ldp_postprocess_certainty.restype = C.c_int
        lib.ldp_postprocess_certainty.argtypes = [C.POINTER(LdpParams), C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p]
        lib.ldp_pack_ply_records.restype = C.c_int
        lib.ldp_pack_ply_records.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.ldp_pack_points3d_records.restype = C.c_int
        lib.ldp_pack_points3d_records.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_uint64,
                                                  C.c_void_p, C.c_void_p]
        lib.ldp_rgb_to_uint8.restype = C.c_int
        lib.ldp_rgb_to_uint8.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
        lib.ldp_gather_points.restype = C.c_int
        lib.ldp_gather_points.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.ldp_gather_rows.restype = C.c_int
        lib.ldp_gather_rows.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.ldp_concat_points.restype = C.c_int
        lib.ldp_concat_points.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.ldp_scatter_points.restype = C.c_int
        lib.ldp_scatter_points.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int64,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.ldp_select_kcenters.restype = C.c_int
        lib.ldp_select_kcenters.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.ldp_nearest_neighbors.restype = C.c_int
        lib.ldp_nearest_neighbors.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
        lib.ldp_voxel_workspace_bytes.restype = C.c_int
        lib.ldp_voxel_workspace_bytes.argtypes = [C.c_int64, C.POINTER(C.c_size_t)]
        lib.ldp_voxel_downsample.restype = C.c_int
        lib.ldp_voxel_downsample.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_size_t, C.c_void_p]
        lib.ldp_set_sm_reserve.restype = C.c_int
        lib.ldp_set_sm_reserve.argtypes = [C.c_int]
        lib.ldp_undistort_points.restype = C.c_int
        lib.ldp_undistort_points.argtypes = [C.POINTER(LdpLens), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.ldp_debug_force_fixup.restype = C.c_int
        lib.ldp_debug_force_fixup.argtypes = [C.c_int, C.c_int]
        lib.ldp_debug_read_fixups.restype = C.c_int
        lib.ldp_debug_read_fixups.argtypes = [C.POINTER(LdpParams), C.c_void_p, C.POINTER(C.c_int32)]
        lib.ldp_outlier_workspace_bytes.restype = C.c_int
        lib.ldp_outlier_workspace_bytes.argtypes = [C.c_int64, C.c_int32, C.POINTER(C.c_size_t)]
        lib.ldp_statistical_outliers.restype = C.c_int
        lib.ldp_statistical_outliers.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        lib.ldp_debug_outlier_max_shells.restype = C.c_int
        lib.ldp_debug_outlier_max_shells.argtypes = [C.c_int]
        lib.ldp_normals_workspace_bytes.restype = C.c_int
        lib.ldp_normals_workspace_bytes.argtypes = [C.c_int64, C.c_int32, C.POINTER(C.c_size_t)]
        lib.ldp_estimate_normals.restype = C.c_int
        lib.ldp_estimate_normals.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        lib.ldp_pack_ply_normal_records.restype = C.c_int
        lib.ldp_pack_ply_normal_records.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                                    C.c_void_p]
        if lib.ldp_abi_version() != LDP_ABI_VERSION:
            raise NativeLibraryError(f"ABI version mismatch: library {lib.ldp_abi_version()}, binding {LDP_ABI_VERSION}")
        for which, struct in enumerate((LdpParams, LdpRefDesc, LdpOutputs, LdpLens)):
            if lib.ldp_struct_size(which) != C.sizeof(struct):
                raise NativeLibraryError(f"struct layout mismatch for {struct.__name__}: "
                                         f"library {lib.ldp_struct_size(which)}, binding {C.sizeof(struct)}")
        _lib = lib
        return _lib


def check(rc: int, what: str) -> None:
    if rc != LDP_OK:
        msg = load().ldp_last_error_string()
        raise NativeLibraryError(f"{what} failed with code {rc}: {msg.decode() if msg else ''}")
