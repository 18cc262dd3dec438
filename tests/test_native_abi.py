"""CPU: the C-ABI library loads and exports every symbol include/ldp_b200.h declares (no compute calls)."""
import ctypes
import os
import re

import pytest

from lichtfeld_densification_plugin_b200 import _native, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    build.build()          # no-op when csrc/libldp_b200.so is up to date
    return _native.load()


def test_header_symbols_exported(lib):
    header = open(os.path.join(ROOT, "include", "ldp_b200.h")).read()
    declared = set(re.findall(r"^\s*(?:int|int64_t|const char\*)\s+(ldp_[a-z_0-9]+)\s*\(", header, flags=re.M))
    assert declared == set(_native.EXPORTS), declared ^ set(_native.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name


SCALARS = {"int": ctypes.c_int, "int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "uint64_t": ctypes.c_uint64,
           "size_t": ctypes.c_size_t, "double": ctypes.c_double, "const char*": ctypes.c_char_p}


def test_binding_signatures_match_the_header(lib):
    """Every prototype's return type and parameter list against the binding's restype / argtypes (a missing argtypes lets
    ctypes pass a Python int as a 32-bit C int, which truncates a pointer)."""
    header = open(os.path.join(ROOT, "include", "ldp_b200.h")).read()
    protos = re.findall(r"^\s*(int|int64_t|const char\*)\s+(ldp_[a-z_0-9]+)\s*\(([^)]*)\)\s*;", header, flags=re.M)
    assert [name for _, name, _ in protos] == list(_native.SIGNATURES)
    for ret, name, params in protos:
        fn = getattr(lib, name)
        assert fn.restype is SCALARS[ret], name
        params = [] if params.strip() == "void" else [" ".join(p.split()) for p in params.split(",")]
        assert fn.argtypes is not None and len(fn.argtypes) == len(params), name
        for decl, t in zip(params, fn.argtypes):
            if "*" in decl:
                assert t is ctypes.c_void_p or issubclass(t, ctypes._Pointer), (name, decl, t)
            else:
                assert t is SCALARS[decl.rsplit(" ", 1)[0]], (name, decl, t)


def test_abi_version_and_struct_layout(lib):
    header = open(os.path.join(ROOT, "include", "ldp_b200.h")).read()
    assert int(re.search(r"#define LDP_ABI_VERSION (\d+)", header).group(1)) == lib.ldp_abi_version() == _native.LDP_ABI_VERSION
    assert int(re.search(r"#define LDP_MAX_NN (\d+)", header).group(1)) == _native.LDP_MAX_NN
    for which, struct in enumerate((_native.LdpParams, _native.LdpRefDesc, _native.LdpOutputs, _native.LdpLens)):
        assert lib.ldp_struct_size(which) == ctypes.sizeof(struct)
    assert lib.ldp_struct_size(4) == -1
    assert _native.REF_DESC_DTYPE.itemsize == ctypes.sizeof(_native.LdpRefDesc)


def test_host_only_entry_points(lib):
    assert lib.ldp_sel_capacity(10000) == 10000
    assert lib.ldp_sel_capacity(1) == 4
    p = _native.LdpParams()
    p.n_refs, p.H, p.W, p.w_match, p.h_match, p.matches_per_ref, p.border, p.tiles = 46, 512, 512, 512, 512, 10000, 2, 24
    need = ctypes.c_size_t(0)
    assert lib.ldp_workspace_bytes(ctypes.byref(p), ctypes.byref(need)) == 0
    assert 46 * 512 * 512 * 5 < need.value < 46 * 512 * 512 * 16
    p.H = 0
    assert lib.ldp_workspace_bytes(ctypes.byref(p), ctypes.byref(need)) == -1
    assert b"bad" in lib.ldp_last_error_string()


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from lichtfeld_densification_plugin_b200.engine import DensifyEngine
    with pytest.raises(_native.NativeLibraryError):
        DensifyEngine()


def test_no_cpu_fallback_around_the_path():
    """The device output contract and pair generation refuse to run without a GPU as well."""
    import numpy as np
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from lichtfeld_densification_plugin_b200 import output
    from lichtfeld_densification_plugin_b200.core import selection
    with pytest.raises(_native.NativeLibraryError):
        output.ply_records(torch.zeros((4, 3)), torch.zeros((4, 3)))
    with pytest.raises(_native.NativeLibraryError):
        output.apply_point_cap(torch.zeros((4, 3)), torch.zeros((4, 3)), torch.zeros((4,)), 2, 0)
    with pytest.raises(_native.NativeLibraryError):
        selection.select_cameras_kcenters(np.zeros((4, 16), np.float32), 2)
    with pytest.raises(_native.NativeLibraryError):
        selection.nearest_neighbors(np.zeros((4, 16), np.float32), 2)
