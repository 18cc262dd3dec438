"""CPU: the oracle restatement vs the unmodified reference.  Where the reference is installed (oracle/ref_import.py) the
comparison is live and bit for bit; elsewhere it is against the stored vectors of tests/golden/make_reference_golden.py."""
import numpy as np
import pytest
import torch

from oracle import densify_oracle as O
from oracle import ref_import
from lichtfeld_densification_plugin_b200 import synth
from tests.helpers import load_reference_golden, oracle_cam

TRIANGULATE_CASES = [("T", False, 3), ("R", False, 2), ("T", True, 3), ("R", True, 1)]


@pytest.fixture(scope="module")
def ref():
    return ref_import.import_reference(full_pipeline=True) if ref_import.reference_available() else None


@pytest.fixture(scope="module")
def stored():
    return load_reference_golden()


def random_configuration(seed):
    """Random map / match sizes, neighbour count, draw size, certainty family and filters of one configuration."""
    rs = np.random.RandomState(500 + seed)
    H, W = int(rs.randint(24, 110)), int(rs.randint(24, 110))
    hm, wm = (H, W) if rs.rand() < 0.5 else (int(rs.randint(16, 100)), int(rs.randint(16, 100)))
    nn, M = int(rs.randint(1, 5)), int(rs.randint(1, min(2500, H * W // 3)))
    return dict(H=H, W=W, hm=hm, wm=wm, nn=nn, M=M, fam="T" if rs.rand() < 0.5 else "R", no_filter=bool(rs.rand() < 0.2),
                seed=int(rs.randint(1, 10000)), sampson=float(rs.choice([5.0, 0.0, 1.0])), parallax=float(rs.choice([0.5, 0.0, 2.0])))


@pytest.mark.parametrize("fam,no_filter,nn", TRIANGULATE_CASES)
def test_triangulate_ref_bit_identical(ref, stored, fam, no_filter, nn):
    scene = synth.make_scene(10, "turbo", ref_fraction=0.2, nn=nn)
    scene.H = scene.W = 128
    scene.h_match = scene.w_match = 96
    cams = scene.cameras
    for rp in range(scene.n_refs):
        inp = synth.synth_ref_inputs(scene, rp, cert_family=fam, seed=3)
        ri, nb = inp["ref_index"], inp["nbr_indices"]
        ocfg = O.OracleConfig(matches_per_ref=5000, no_filter=no_filter, w_match=scene.w_match, h_match=scene.h_match)
        got = O.triangulate_ref([inp["cert"][k] for k in range(len(nb))], [inp["warp"][k] for k in range(len(nb))],
                                inp["image"].numpy(), oracle_cam(cams[ri]), [oracle_cam(cams[j]) for j in nb], ocfg,
                                rng=np.random.RandomState(40 + rp), collect_debug=True)
        if ref is None:
            key = f"tri/{fam}/{int(no_filter)}/{nn}/{rp}"
            stored.check(f"{key}/xyz", got.xyz, rtol=1e-5, atol=1e-6)
            stored.check(f"{key}/rgb", got.rgb, atol=1e-7)
            stored.check(f"{key}/err", got.err, rtol=1e-3, atol=2e-4)
            assert list(got.debug_matches_by_nbr.keys()) == [int(u) for u in stored.z[f"{key}/dbg_uids"]]
            for uid in got.debug_matches_by_nbr:
                stored.check(f"{key}/dbg_matches/{uid}", got.debug_matches_by_nbr[uid], atol=1e-4)
                stored.check(f"{key}/dbg_cert/{uid}", got.debug_cert_by_nbr[uid], atol=1e-7)
            continue
        P = ref.pipeline
        cfg = ref.config.DensePipelineConfig(output_path="unused.ply", no_filter=no_filter, matches_per_ref=5000)
        ctx = P._TriangulationContext(cameras=P._build_camera_lookup(cams), config=cfg, matcher_sample_cap=0.9,
                                      w_match=scene.w_match, h_match=scene.h_match)
        packed = P._PackedReferenceBatch(ref_id=cams[ri].uid, ref_path="", imA_np=inp["image"].numpy(), maskA_np=None,
                                         wA_cam=cams[ri].width, hA_cam=cams[ri].height,
                                         nn_ids=[cams[j].uid for j in nb], nn_masks=[None] * len(nb),
                                         nn_arrays=[None] * len(nb))
        mr = P._MatchedReference(packed=packed, warp_list_cpu=[inp["warp"][k] for k in range(len(nb))],
                                 cert_list_cpu=[inp["cert"][k] for k in range(len(nb))],
                                 pair_index_by_nbr={}, image_by_nbr={})
        np.random.seed(40 + rp)
        want = P._triangulate_ref(mr, ctx, collect_debug_matches=True)
        assert np.array_equal(want.xyz, got.xyz)
        assert np.array_equal(want.rgb, got.rgb)
        assert np.array_equal(want.err, got.err)
        assert list(want.debug_matches_by_nbr.keys()) == list(got.debug_matches_by_nbr.keys())
        for uid in want.debug_matches_by_nbr:
            assert np.array_equal(want.debug_matches_by_nbr[uid], got.debug_matches_by_nbr[uid])
            assert np.array_equal(want.debug_cert_by_nbr[uid], got.debug_cert_by_nbr[uid])


def test_sampler_and_geometry_functions(ref, stored):
    rs = np.random.RandomState(0)
    cert = torch.from_numpy(rs.random_sample((90, 120)).astype(np.float32))
    got = O.select_samples(cert, 2000, rng=np.random.RandomState(5))
    cams = synth.make_orbit_cameras(5)
    a, b = cams[0], cams[1]
    F2 = O.fundamental_matrix(a.K, a.R, a.t, b.K, b.R, b.t)
    uv1 = (rs.random_sample((500, 2)) * 800).astype(np.float32)
    uv2 = (uv1 + rs.standard_normal((500, 2)) * 5).astype(np.float32)
    X2 = O.dlt_points(a.P, b.P, uv1, uv2)
    if ref is None:
        stored.check("fn/select_samples", got)
        F1 = stored.z["fn/F"]
        assert F1.dtype == F2.dtype and np.allclose(F1, F2, rtol=1e-12, atol=0)
        stored.check("fn/sampson", O.sampson_distance(F2, uv1, uv2), rtol=1e-3, atol=2e-4)
        stored.check("fn/dlt", X2, rtol=1e-5, atol=1e-6)
        stored.check("fn/dlt1", O.dlt_points(a.P, b.P, uv1[:1], uv2[:1]), rtol=1e-5, atol=1e-6)
        stored.check("fn/reproj", O.reprojection_error(a.P, X2, uv1), rtol=1e-3, atol=2e-4)
        stored.check("fn/cheirality", O.in_front(b.P, X2))
        stored.check("fn/parallax", O.parallax_ok(a.C, b.C, X2, 0.5))
        return
    np.random.seed(5)
    want = ref.sampling.select_samples_with_coverage(cert, 2000)
    assert np.array_equal(want, got)
    F1 = ref.geometry.fundamental_from_world2cam(a.K, a.R, a.t, b.K, b.R, b.t)
    assert np.array_equal(F1, F2) and F1.dtype == F2.dtype
    assert np.array_equal(ref.geometry.sampson_error(F1, uv1, uv2), O.sampson_distance(F2, uv1, uv2))
    X1 = ref.geometry.dlt_triangulate_batch(a.P, b.P, uv1, uv2)
    assert np.array_equal(X1, X2)
    assert np.array_equal(ref.geometry.dlt_triangulate_batch(a.P, b.P, uv1[:1], uv2[:1]), O.dlt_points(a.P, b.P, uv1[:1], uv2[:1]))
    assert np.array_equal(ref.geometry.reprojection_errors(a.P, X1, uv1), O.reprojection_error(a.P, X2, uv1))
    assert np.array_equal(ref.geometry.cheirality_mask(b.P, X1), O.in_front(b.P, X2))
    assert np.array_equal(ref.geometry.parallax_mask(a.C, b.C, X1, 0.5), O.parallax_ok(a.C, b.C, X2, 0.5))


@pytest.mark.parametrize("seed", range(12))
def test_random_configurations_bit_identical(ref, stored, seed):
    """Random map / match sizes (down to maps narrower than 48 px: one-pixel coverage tiles), 1-4 neighbours, draw sizes, both
    certainty families, filters on / partly off / off: outputs - or the exception raised - identical to the reference
    (a slice of scratch/oracle_fuzz.py, which ran 360 such configurations against the live reference)."""
    from tests import gpu_harness as G
    from tests.golden.make_golden import build_scene
    c = random_configuration(seed)
    scene = build_scene(c)
    inp = synth.synth_ref_inputs(scene, 0, cert_family=c["fam"], seed=c["seed"])
    cams = scene.cameras
    ri, nb = inp["ref_index"], inp["nbr_indices"]

    def run(f):
        np.random.seed(c["seed"])
        try:
            return f(), None
        except Exception as exc:
            return None, f"{type(exc).__name__}: {exc}"
    got, err_g = run(lambda: G.run_oracle_ref(scene, inp, c))
    if ref is None:
        key = f"rand/{seed}"
        assert (err_g or "") == str(stored.z[f"{key}/error"]), c
        if err_g is None:
            stored.check(f"{key}/xyz", got.xyz, rtol=1e-5, atol=1e-6)
            stored.check(f"{key}/rgb", got.rgb, atol=1e-7)
            stored.check(f"{key}/err", got.err, rtol=1e-3, atol=2e-4)
        return
    P = ref.pipeline
    cfg = ref.config.DensePipelineConfig(output_path="unused.ply", matches_per_ref=c["M"], no_filter=c["no_filter"],
                                         sampson_thresh=c["sampson"], min_parallax_deg=c["parallax"])
    ctx = P._TriangulationContext(cameras=P._build_camera_lookup(cams), config=cfg, matcher_sample_cap=0.9, w_match=c["wm"],
                                  h_match=c["hm"])
    packed = P._PackedReferenceBatch(ref_id=cams[ri].uid, ref_path="", imA_np=inp["image"].numpy(), maskA_np=None,
                                     wA_cam=cams[ri].width, hA_cam=cams[ri].height, nn_ids=[cams[j].uid for j in nb],
                                     nn_masks=[None] * len(nb), nn_arrays=[None] * len(nb))
    mr = P._MatchedReference(packed=packed, warp_list_cpu=[inp["warp"][k] for k in range(len(nb))],
                             cert_list_cpu=[inp["cert"][k] for k in range(len(nb))], pair_index_by_nbr={}, image_by_nbr={})
    want, err_w = run(lambda: P._triangulate_ref(mr, ctx, collect_debug_matches=False))
    assert err_w == err_g, c
    if want is None or got is None:
        assert want is None and (got is None or got.xyz.shape[0] == 0), c
        return
    assert np.array_equal(want.xyz, got.xyz) and np.array_equal(want.rgb, got.rgb), c
    assert np.array_equal(want.err, got.err, equal_nan=True), c
