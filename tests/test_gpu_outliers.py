"""GPU: statistical outlier removal (ldp_statistical_outliers / output.remove_statistical_outliers) against the numpy
oracle of tests/outlier_oracle.py, bit for bit."""
import ctypes as C

import numpy as np
import pytest
import torch

from lichtfeld_densification_plugin_b200 import _native as N
from lichtfeld_densification_plugin_b200 import build, output, synth
from tests import outlier_oracle as OO

pytestmark = pytest.mark.gpu

KS = (1, 2, 8, 20, 64)


@pytest.fixture(scope="module")
def lib():
    build.build()
    return N.load()


def _raw(lib, xyz: torch.Tensor, k: int, ratio: float = 2.0, stream=None):
    """The C entry point: (kept indices, m, (mean, std, threshold), status) on the host."""
    dev, n = xyz.device, int(xyz.shape[0])
    need = C.c_size_t(0)
    N.check(lib.ldp_outlier_workspace_bytes(n, k, C.byref(need)), "ldp_outlier_workspace_bytes")
    ws = torch.empty((max(1, need.value),), dtype=torch.uint8, device=dev)
    kept = torch.full((n,), -1, dtype=torch.int64, device=dev)
    m = torch.full((n,), -1.0, dtype=torch.float64, device=dev)
    stats = torch.full((3,), -1.0, dtype=torch.float64, device=dev)
    status = torch.full((3,), -1, dtype=torch.int32, device=dev)
    st = stream if stream is not None else torch.cuda.current_stream(dev)
    with torch.cuda.stream(st):
        N.check(lib.ldp_statistical_outliers(C.c_void_p(xyz.data_ptr()), n, k, C.c_double(ratio), C.c_void_p(kept.data_ptr()),
                                             C.c_void_p(m.data_ptr()), C.c_void_p(stats.data_ptr()), C.c_void_p(status.data_ptr()),
                                             C.c_void_p(ws.data_ptr()), C.c_size_t(need.value), C.c_void_p(st.cuda_stream)),
                "ldp_statistical_outliers")
    st.synchronize()
    s = status.cpu().numpy()
    return kept.cpu().numpy()[:s[1]], m.cpu().numpy(), stats.cpu().numpy(), s


def _bits(x) -> bytes:
    return np.asarray(x, np.float64).tobytes()


@pytest.mark.parametrize("kind", OO.CLOUDS)
@pytest.mark.parametrize("n", [1, 2, 17, 1000, 50_000])
def test_kernel_vs_oracle(lib, kind, n):
    xyz = OO.make_cloud(kind, n, seed=n)
    d2 = OO.sorted_knn_d2_exact(xyz, 64)
    dev = torch.from_numpy(xyz).cuda()
    for k in KS:
        m_ref = OO.means_from_sorted_d2(d2, min(k, n))
        keep_ref, _, st_ref = OO.statistical_outliers(xyz, k, 2.0, means=m_ref)
        kept, m, stats, status = _raw(lib, dev, k)
        assert status[0] == 0
        assert _bits(m) == _bits(m_ref), (kind, n, k, int(np.sum(m != m_ref)))
        assert _bits(stats) == _bits(st_ref), (kind, n, k, stats, st_ref)
        assert np.array_equal(kept, keep_ref), (kind, n, k)
        if n == 50_000:
            print(f"{kind} n={n} k={k}: kept {kept.size}, left the finest grid {status[2]}")


@pytest.mark.parametrize("kind", ["sphere_floaters", "duplicates", "two_clusters", "lattice"])
def test_shells_do_not_change_results(lib, kind):
    xyz = torch.from_numpy(OO.make_cloud(kind, 20_000, seed=7)).cuda()
    try:
        N.check(lib.ldp_debug_outlier_max_shells(1), "max_shells")
        a = _raw(lib, xyz, 20)
        N.check(lib.ldp_debug_outlier_max_shells(0), "max_shells")
        b = _raw(lib, xyz, 20)
    finally:
        lib.ldp_debug_outlier_max_shells(0)
    assert a[3][2] >= b[3][2]
    assert np.array_equal(a[0], b[0]) and _bits(a[1]) == _bits(b[1]) and _bits(a[2]) == _bits(b[2])


def test_large_sphere_vs_kdtree(lib):
    """2.3 M points (the config-5 cloud size): sphere + 1 % floaters against cKDTree's neighbours."""
    xyz, is_f = OO.sphere_with_floaters(2_300_000, seed=1)
    kept, m, stats, status = _raw(lib, torch.from_numpy(xyz).cuda(), 20)
    ref = OO.mean_distances_kdtree(xyz, 20)
    np.testing.assert_allclose(m, ref, rtol=1e-12, atol=0)
    thr = stats[2]
    near = np.nonzero(np.abs(ref - thr) <= 1e-9 * thr)[0]
    keep_ref = np.nonzero((ref > 0) & (ref < thr))[0]
    diff = np.setxor1d(kept, keep_ref)
    print(f"2.3M: kept {kept.size}, within 1e-9 of the threshold {near.tolist()}, left the finest grid {status[2]} "
          f"({status[2] / xyz.shape[0]:.2%}); floaters removed {1 - np.isin(np.nonzero(is_f)[0], kept).mean():.3f}")
    assert np.isin(diff, near).all()
    assert np.isin(np.nonzero(~is_f)[0], kept).all()


def test_rejections(lib):
    xyz = torch.from_numpy(OO.make_cloud("cube", 1000)).cuda()
    rgb = torch.zeros_like(xyz)
    for k, r in ((0, 2.0), (65, 2.0), (8, 0.0), (8, -1.0)):
        with pytest.raises(ValueError):
            output.remove_statistical_outliers(xyz, rgb, nb_neighbors=k, std_ratio=r)
    need = C.c_size_t(0)
    assert lib.ldp_outlier_workspace_bytes(10, 65, C.byref(need)) == -1
    for bad in (float("nan"), float("inf"), -float("inf")):
        x = xyz.clone()
        x[17, 2] = bad
        with pytest.raises(ValueError):
            output.remove_statistical_outliers(x, rgb, nb_neighbors=8, std_ratio=2.0)
        assert _raw(lib, x, 8)[3][0] == 1


def test_repeatable_streams_and_input_untouched(lib):
    xyz_np = OO.make_cloud("sphere_floaters", 100_000, seed=9)
    xyz = torch.from_numpy(xyz_np).cuda()
    rgb = torch.rand((xyz.shape[0], 3), device="cuda")
    err = torch.rand((xyz.shape[0],), device="cuda")
    a = _raw(lib, xyz, 20)
    b = _raw(lib, xyz, 20, stream=torch.cuda.Stream())
    assert np.array_equal(a[0], b[0]) and _bits(a[1]) == _bits(b[1]) and _bits(a[2]) == _bits(b[2])
    r = output.remove_statistical_outliers(xyz, rgb, err, nb_neighbors=20, std_ratio=2.0)
    torch.cuda.synchronize()
    assert xyz.cpu().numpy().tobytes() == xyz_np.tobytes()
    assert np.array_equal(r.kept_idx.cpu().numpy(), a[0]) and _bits(r.mean_dist.cpu().numpy()) == _bits(a[1])
    assert (r.cloud_mean, r.std_dev, r.threshold) == tuple(float(v) for v in a[2])
    sel = r.kept_idx
    assert torch.equal(r.xyz, xyz[sel]) and torch.equal(r.rgb, rgb[sel]) and torch.equal(r.err, err[sel])
    assert output.remove_statistical_outliers(xyz, rgb, nb_neighbors=20, std_ratio=2.0).err is None
    e = output.remove_statistical_outliers(xyz[:0], rgb[:0], nb_neighbors=20, std_ratio=2.0)
    assert e.xyz.shape == (0, 3) and e.kept_idx.numel() == 0


def test_run_dense_pipeline_filters_the_final_cloud(tmp_path):
    from lichtfeld_densification_plugin_b200.core import pipeline as P
    from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig
    scene = synth.make_scene(24, "turbo", ref_fraction=0.5, nn=4)
    cams = scene.cameras
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=12) for rp in range(scene.n_refs)]

    def match_source(rp):
        inp = inputs[rp]
        ri, nb = inp["ref_index"], inp["nbr_indices"]
        packed = P._PackedReferenceBatch(ref_id=cams[ri].uid, ref_path="", imA_np=inp["image"].numpy(), maskA_np=None,
                                         wA_cam=cams[ri].width, hA_cam=cams[ri].height, nn_ids=[cams[j].uid for j in nb],
                                         nn_masks=[None] * len(nb), nn_arrays=[None] * len(nb))
        return P._MatchedReference(packed=packed, warp_list_cpu=[inp["warp"][k] for k in range(len(nb))],
                                   cert_list_cpu=[inp["cert"][k] for k in range(len(nb))], pair_index_by_nbr={}, image_by_nbr={})
    refs = list(range(scene.n_refs))
    kw = dict(output_path=str(tmp_path / "dense.ply"), matches_per_ref=4000, refs_per_launch=4, multiview=True)
    steps = []
    on = P.run_dense_pipeline(cams, refs, None, DensePipelineConfig(outlier_neighbors=20, **kw), match_source=match_source,
                              w_match=scene.w_match, h_match=scene.h_match, progress_callback=lambda p, s: steps.append(s))
    off = P.run_dense_pipeline(cams, refs, None, DensePipelineConfig(**kw), match_source=match_source,
                               w_match=scene.w_match, h_match=scene.h_match)
    assert "Removing outliers..." in steps
    keep, _, _ = OO.statistical_outliers(off.xyz, 20, 2.0, means=OO.mean_distances_exact(off.xyz, 20))
    assert 0 < keep.size < off.xyz.shape[0]
    assert on.xyz.tobytes() == off.xyz[keep].tobytes() and on.rgb.tobytes() == off.rgb[keep].tobytes()
    assert on.err.tobytes() == off.err[keep].tobytes() and on.n_views.tobytes() == off.n_views[keep].tobytes()
