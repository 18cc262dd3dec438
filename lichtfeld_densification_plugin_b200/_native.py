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

LDP_ABI_VERSION = 22
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

_P, _I32, _I64, _SZ = C.c_void_p, C.c_int32, C.c_int64, C.c_size_t
_PARAMS, _OUTPUTS, _SZ_OUT = C.POINTER(LdpParams), C.POINTER(LdpOutputs), C.POINTER(C.c_size_t)

# The C ABI, in include/ldp_b200.h's order: name -> (restype, argtypes).  Device pointers and streams are c_void_p.
SIGNATURES = {
    "ldp_abi_version": (C.c_int, []),
    "ldp_last_error_string": (C.c_char_p, []),
    "ldp_sel_capacity": (_I64, [_I32]),
    "ldp_workspace_bytes": (C.c_int, [_PARAMS, _SZ_OUT]),
    "ldp_densify_refs": (C.c_int, [_PARAMS, _P, _P, _OUTPUTS, _P, _SZ, _P]),
    "ldp_sample_refs": (C.c_int, [_PARAMS, _P, _P, _OUTPUTS, _P, _SZ, _P]),
    "ldp_triangulate_samples": (C.c_int, [_PARAMS, _P, _OUTPUTS, _P, _SZ, _P]),
    "ldp_undistort_points": (C.c_int, [C.POINTER(LdpLens), _I64, _P, _P, _P]),
    "ldp_postprocess_certainty": (C.c_int, [_PARAMS, _P, _P, _SZ, _SZ, _P]),
    "ldp_depth_workspace_bytes": (C.c_int, [_PARAMS, _SZ_OUT]),
    "ldp_depth_maps": (C.c_int, [_PARAMS, _P, C.c_double, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "ldp_pack_ply_records": (C.c_int, [_P, _P, _I64, _P, _P, _P]),
    "ldp_pack_ply_normal_records": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P]),
    "ldp_pack_points3d_records": (C.c_int, [_P, _P, _P, _I64, _P, C.c_uint64, _P, _P]),
    "ldp_rgb_to_uint8": (C.c_int, [_P, _I64, _P, _P]),
    "ldp_gather_points": (C.c_int, [_P, _P, _P, _P, _I64, _I64, _P, _P, _P, _P, _P]),
    "ldp_gather_rows": (C.c_int, [_P, _I32, _P, _I64, _I64, _P, _P, _P]),
    "ldp_concat_points": (C.c_int, [_P, _P, _P, _P, _I32, _I64, _P, _P, _P, _I64, _P, _P, _P]),
    "ldp_scatter_points": (C.c_int, [_P, _P, _P, _P, _I32, _I32, _I64, _P, _P, _P, _I64, _P, _P, _P]),
    "ldp_select_kcenters": (C.c_int, [_P, _I32, _I32, _P, _P, _P, _P]),
    "ldp_nearest_neighbors": (C.c_int, [_P, _I32, _I32, _P, _P]),
    "ldp_voxel_workspace_bytes": (C.c_int, [_I64, _SZ_OUT]),
    "ldp_voxel_downsample": (C.c_int, [_P, _P, _I64, C.c_double, _P, _P, _P, _P, _SZ, _P]),
    "ldp_outlier_workspace_bytes": (C.c_int, [_I64, _I32, _SZ_OUT]),
    "ldp_statistical_outliers": (C.c_int, [_P, _I64, _I32, C.c_double, _P, _P, _P, _P, _P, _SZ, _P]),
    "ldp_debug_outlier_max_shells": (C.c_int, [C.c_int]),
    "ldp_normals_workspace_bytes": (C.c_int, [_I64, _I32, _SZ_OUT]),
    "ldp_estimate_normals": (C.c_int, [_P, _I64, _I32, _P, _I32, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "ldp_gaussian_workspace_bytes": (C.c_int, [_I64, _I32, _SZ_OUT]),
    "ldp_gaussian_init": (C.c_int, [_P, _P, _P, _I64, _I32, C.c_double, C.c_double, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "ldp_pack_gaussian_ply_records": (C.c_int, [_P, _P, _P, _P, _P, _P, _I64, _P, _I32, _P, _P]),
    "ldp_consistency_workspace_bytes": (C.c_int, [_I64, _SZ_OUT]),
    "ldp_depth_consistency": (C.c_int, [_P, _I64, _P, _P, _I32, _I32, _P, _P, _P, _I32, C.c_double, _I32, _I32, _P, _P, _P, _P, _P, _SZ, _P]),
    "ldp_depth_colors": (C.c_int, [_P, _P, _P, _P, _P]),
    "ldp_fuse_workspace_bytes": (C.c_int, [_I32, _I32, _I32, _SZ_OUT]),
    "ldp_fuse_depth_maps": (C.c_int, [_P, _P, _P, _P, _I32, _I32, _I32, _P, _P, _P, C.c_double, _I32, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "ldp_depth_normals": (C.c_int, [_P, _P, _I32, _I32, _I32, _P, _I32, C.c_double, _P, _P, _P, _P]),
    "ldp_fuse_depth_maps_oriented": (C.c_int, [_P, _P, _P, _P, _P, _I32, _I32, _I32, _P, _P, _P, C.c_double, C.c_double, _I32, _I32,
                                               _P, _P, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "ldp_set_sm_reserve": (C.c_int, [C.c_int]),
    "ldp_last_launch_count": (C.c_int, []),
    "ldp_profile_enable": (C.c_int, [C.c_int]),
    "ldp_profile_read": (C.c_int, [C.POINTER(C.c_float), C.c_int]),
    "ldp_profile_name": (C.c_char_p, [C.c_int]),
    "ldp_debug_set_cluster": (C.c_int, [C.c_int]),
    "ldp_debug_last_cluster": (C.c_int, []),
    "ldp_debug_read_clocks": (C.c_int, [_PARAMS, _P, C.POINTER(C.c_longlong)]),
    "ldp_debug_force_fixup": (C.c_int, [C.c_int, C.c_int]),
    "ldp_debug_read_fixups": (C.c_int, [_PARAMS, _P, C.POINTER(C.c_int32)]),
    "ldp_debug_launch_stream": (C.c_int, [_PARAMS, _P, _P, _SZ, _P, C.c_int]),
    "ldp_struct_size": (_I64, [C.c_int]),
}
EXPORTS = list(SIGNATURES)

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
        for name, (restype, argtypes) in SIGNATURES.items():
            if not hasattr(lib, name):
                raise NativeLibraryError(f"{path} does not export {name}")
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = restype, argtypes
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
