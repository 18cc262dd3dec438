"""GPU: cross-view depth consistency (ldp_depth_consistency, output.check_depth_consistency) against its numpy restatement
(tests/consistency_oracle.py), on the device's own depth maps, through the pipeline, and on bad input and side streams."""
import ctypes as C

import numpy as np
import pytest
import torch

from lichtfeld_densification_plugin_b200 import _native as N
from lichtfeld_densification_plugin_b200 import synth
from lichtfeld_densification_plugin_b200.engine import DepthViews, PathConfig, depth_map_scales
from lichtfeld_densification_plugin_b200.output import check_depth_consistency
from tests import consistency_oracle as CO

pytestmark = pytest.mark.gpu

OPENCV = ("OPENCV", [-0.12, 0.03, 4e-4, -3e-4])
FISHEYE = ("OPENCV_FISHEYE", [0.05, -0.01, 0.003, -0.0005])


def _setup(n_views, H, W, wm, hm, lens=None, holes=0.05, seed=0):
    """Orbit cameras, each with the analytic map of the sphere of synth.SPHERE_RADIUS (pinhole ray cast: for lens views the
    maps are simply inputs), with NaN holes."""
    cams = synth.make_orbit_cameras(n_views, lens=lens)
    rs = np.random.RandomState(seed)
    maps = np.stack([CO.sphere_map(c, H, W, wm, hm, synth.SPHERE_RADIUS) for c in cams])
    maps[rs.random_sample(maps.shape) < holes] = np.nan
    views = DepthViews(H, W, wm, hm)
    for m, c in zip(maps, cams):
        views.add(m, c)
    P = np.stack([np.asarray(c.P, np.float32).reshape(12) for c in cams])
    S = np.array([depth_map_scales(c.width, c.height, H, W, wm, hm) for c in cams])
    lenses = [CO.lens_tuple(c) for c in cams]
    return cams, maps, views, P, S, (lenses if any(l is not None for l in lenses) else None)


def _points(n, seed=1):
    """Points on the sphere, moved radially by up to 5 %, plus 1 % scattered through and far outside the scene."""
    rs = np.random.RandomState(seed)
    d = rs.normal(size=(n, 3))
    X = synth.SPHERE_RADIUS * d / np.linalg.norm(d, axis=1, keepdims=True) * rs.uniform(0.95, 1.05, size=(n, 1))
    k = max(1, n // 100)
    X[:k] = rs.uniform(-50, 50, size=(k, 3))
    return X.astype(np.float32)


def _run(xyz, views, **kw):
    dev = views.device
    owner = kw.pop("owner", None)
    r = check_depth_consistency(torch.from_numpy(xyz).to(dev), views, owner=None if owner is None else torch.from_numpy(owner), **kw)
    return r.n_consistent.cpu().numpy(), r.n_violations.cpu().numpy(), r.kept_idx.cpu().numpy()


def _compare(xyz, views, maps, P, S, lenses, tag, **kw):
    nc, nv, kept = _run(xyz, views, **kw)
    o = CO.check(xyz, maps, P, S, lenses=lenses, **kw)
    if lenses is None:
        assert np.array_equal(nc, o.n_consistent) and np.array_equal(nv, o.n_violations), tag
        assert np.array_equal(kept, o.kept_idx), tag
        return nc, nv
    diff = (nc != o.n_consistent) | (nv != o.n_violations)
    listed = np.nonzero(diff)[0]
    print(f"[lens] {tag}: {len(xyz)} points, differing {listed.size} (edge distances {o.edge[listed][:10].tolist()})")
    assert (o.edge[listed] < 1e-9).all(), tag
    assert np.isin(np.setxor1d(kept, o.kept_idx), listed).all(), tag
    return nc, nv


@pytest.mark.parametrize("with_owner", [False, True])
@pytest.mark.parametrize("rel_tol", [0.002, 0.01, 0.05])
def test_pinhole_vs_oracle(with_owner, rel_tol):
    cams, maps, views, P, S, lenses = _setup(12, 128, 128, 320, 320)
    xyz = _points(40000)
    owner = np.random.RandomState(2).randint(-1, 12, size=len(xyz)).astype(np.int32) if with_owner else None
    seen = set()
    for mv, mx in ((1, 0), (0, 0), (2, 1), (3, 5)):
        nc, nv = _compare(xyz, views, maps, P, S, None, (with_owner, rel_tol, mv, mx), owner=owner, rel_tol=rel_tol, min_views=mv,
                          max_violations=mx)
        seen.add((int((nc > 0).sum() > 100), int((nv > 0).sum() > 100)))
    assert seen == {(1, 1)}                               # the points give both kinds of evidence


def test_lens_vs_oracle():
    cams, maps, views, P, S, lenses = _setup(12, 128, 128, 320, 320, lens=[[OPENCV, None, FISHEYE][v % 3] for v in range(12)])
    assert views.has_lens and lenses is not None
    xyz = _points(40000, seed=5)
    owner = np.random.RandomState(3).randint(-1, 12, size=len(xyz)).astype(np.int32)
    for kw in (dict(), dict(owner=owner, rel_tol=0.03, min_views=2, max_violations=1)):
        _compare(xyz, views, maps, P, S, lenses, f"lens {sorted(kw)}", **kw)


def test_tiny_and_outside():
    cams, maps, views, P, S, lenses = _setup(4, 64, 64, 64, 64)
    nc, nv, kept = _run(np.zeros((0, 3), np.float32), views)
    assert nc.size == nv.size == kept.size == 0
    for x in ([[0.0, 0.0, synth.SPHERE_RADIUS]], [[1e4, 1e4, 1e4]], [[0.0, 0.0, 0.0]]):
        xyz = np.asarray(x, np.float32)
        for mv in (0, 1):
            _compare(xyz, views, maps, P, S, None, ("n=1", x, mv), min_views=mv)
    far = np.array([[1e5, 0, 0], [0, -1e5, 0], [3e4, 3e4, -3e4]], np.float32)      # outside every map / behind every camera
    nc, nv, kept = _run(far, views, min_views=0)
    assert (nc == 0).all() and (nv == 0).all() and kept.tolist() == [0, 1, 2]


@pytest.mark.parametrize("lens", [False, True])
def test_many_views(lens):
    """More views than one staging chunk (128 pinhole, 64 lens), millions of points in the pinhole case."""
    V = 150
    spec = [[OPENCV, None, FISHEYE][v % 3] for v in range(V)] if lens else None
    cams, maps, views, P, S, lenses = _setup(V, 96, 96, 320, 320, lens=spec, seed=7)
    xyz = _points(300000 if lens else 2500000, seed=8)
    owner = np.random.RandomState(9).randint(-1, V, size=len(xyz)).astype(np.int32)
    nc, nv = _compare(xyz, views, maps, P, S, lenses, f"many views lens={lens}", owner=owner, min_views=2, max_violations=2)
    print(f"[many] V={V} n={len(xyz)}: supported by >= 1 view {np.mean(nc > 0):.3f}, violated {np.mean(nv > 0):.3f}, "
          f"max support {nc.max()}")
    assert nc.max() > 5


def _batch(engine, scene, inputs):
    b = engine.new_batch(scene.H, scene.W, scene.w_match, scene.h_match)
    dev = engine.device
    for inp in inputs:
        nb = inp["nbr_indices"]
        cert, warp = inp["cert"].to(dev), inp["warp"].to(dev)
        b.add([cert[k] for k in range(len(nb))], [warp[k] for k in range(len(nb))], inp["image"].to(dev),
              scene.cameras[inp["ref_index"]], [scene.cameras[j] for j in nb], rng_stream=inp["ref_index"])
    return b


def test_device_depth_maps():
    """Maps of DensifyEngine.depth_maps on the sphere scene: a view's own kept points, checked against its own map alone,
    agree wherever they land on their own pixel; the other reference views (60 degrees apart on the ring) support many."""
    from lichtfeld_densification_plugin_b200.engine import DensifyEngine
    engine = DensifyEngine()
    scene = synth.make_scene(24, "turbo", ref_fraction=0.25, nn=4)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=4, surface="sphere") for rp in range(scene.n_refs)]
    dm = engine.depth_maps(_batch(engine, scene, inputs), PathConfig(matches_per_ref=4000), 0.3, want_xyz=True)
    torch.cuda.synchronize()
    H, W = scene.H, scene.W
    all_views = DepthViews(H, W, scene.w_match, scene.h_match)
    for r, inp in enumerate(inputs):
        all_views.add(dm.depth[r], scene.cameras[inp["ref_index"]])
    on_own = supported = total = 0
    for r, inp in enumerate(inputs):
        cam = scene.cameras[inp["ref_index"]]
        own = DepthViews(H, W, scene.w_match, scene.h_match)
        own.add(dm.depth[r], cam)
        xyz_map = dm.xyz[r].reshape(-1, 3)
        pix = torch.nonzero(torch.isfinite(dm.depth[r].reshape(-1))).reshape(-1)
        xyz = xyz_map[pix].contiguous()
        res = check_depth_consistency(xyz, own, min_views=0)
        nc = res.n_consistent.cpu().numpy()
        q0, q1, z = CO.project(np.asarray(cam.P, np.float32), xyz.cpu().numpy())
        ax, ay = depth_map_scales(cam.width, cam.height, H, W, scene.w_match, scene.h_match)
        lands = (np.floor(q1 / z * ay) * W + np.floor(q0 / z * ax)) == pix.cpu().numpy()
        assert lands.mean() > 0.5, r
        assert (nc[lands] == 1).all(), r
        cross = check_depth_consistency(xyz, all_views, owner=torch.full((xyz.shape[0],), r, dtype=torch.int32))
        supported += int((cross.n_consistent > 0).sum())
        on_own += int(lands.sum())
        total += int(xyz.shape[0])
    print(f"[device maps] {total} kept pixels, on their own pixel {on_own}, supported by another view {supported}")
    assert supported > 0.15 * total


def _pipeline(tmp_path, n_views=24, lens=None):
    from lichtfeld_densification_plugin_b200.core import pipeline as P
    scene = synth.make_scene(n_views, "turbo", ref_fraction=0.5, nn=4, lens=lens)
    cams = scene.cameras
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=12, surface="sphere") for rp in range(scene.n_refs)]

    def match_source(rp):
        inp = inputs[rp]
        ri, nb = inp["ref_index"], inp["nbr_indices"]
        packed = P._PackedReferenceBatch(ref_id=cams[ri].uid, ref_path="", imA_np=inp["image"].numpy(), maskA_np=None,
                                         wA_cam=cams[ri].width, hA_cam=cams[ri].height, nn_ids=[cams[j].uid for j in nb],
                                         nn_masks=[None] * len(nb), nn_arrays=[None] * len(nb))
        return P._MatchedReference(packed=packed, warp_list_cpu=[inp["warp"][k] for k in range(len(nb))],
                                   cert_list_cpu=[inp["cert"][k] for k in range(len(nb))], pair_index_by_nbr={}, image_by_nbr={})

    def run(**kw):
        from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig
        cfg = DensePipelineConfig(output_path=str(tmp_path / "dense.ply"), matches_per_ref=4000, depth_min_certainty=0.3, **kw)
        return P.run_dense_pipeline(cams, list(range(scene.n_refs)), None, cfg.validate(), match_source=match_source,
                                    w_match=scene.w_match, h_match=scene.h_match)
    return cams, run


def _unfiltered_then_check(tmp_path, cams, run, tag, **kw):
    """The unfiltered run (its maps written to disk), then check_depth_consistency on those maps with the owners."""
    import json
    ddir = tmp_path / f"maps_{tag}"
    base = run(depth_dir=str(ddir), **kw)
    views = DepthViews.from_depth_dir(str(ddir), cams)
    uids = [e["camera_uid"] for e in json.load(open(ddir / "depth_maps.json"))["maps"]]
    return base, views, uids


@pytest.mark.parametrize("rng_mode", ["philox", "numpy"])
def test_pipeline_equals_check_on_the_same_maps(tmp_path, rng_mode):
    from lichtfeld_densification_plugin_b200.core import pipeline as P
    cams, run = _pipeline(tmp_path)
    kw = dict(rng_mode=rng_mode, refs_per_launch=0)
    seen = []
    orig = P._check_consistency

    def spy(xyz, ref_uid, depth_kept, tri_ctx):          # the owners the pipeline used, for the restatement below
        seen.append(ref_uid.copy())
        return orig(xyz, ref_uid, depth_kept, tri_ctx)
    P._check_consistency = spy
    try:
        res = run(depth_consistency=True, consistency_min_views=1, **kw)
    finally:
        P._check_consistency = orig
    base, views, uids = _unfiltered_then_check(tmp_path, cams, run, rng_mode, **kw)
    assert seen[0].shape[0] == base.xyz.shape[0]
    owner = np.array([uids.index(int(u)) for u in seen[0]], np.int32)
    r = check_depth_consistency(torch.from_numpy(base.xyz).cuda(), views, owner=torch.from_numpy(owner))
    kept = r.kept_idx.cpu().numpy()
    print(f"[pipeline {rng_mode}] {base.xyz.shape[0]} points, {kept.size} consistent")
    assert 0 < kept.size < base.xyz.shape[0]
    assert res.xyz.tobytes() == base.xyz[kept].tobytes() and res.rgb.tobytes() == base.rgb[kept].tobytes()
    assert res.err.tobytes() == base.err[kept].tobytes()
    assert res.consistent_views.dtype == np.int32 and np.array_equal(res.consistent_views, r.n_consistent.cpu().numpy()[kept])
    assert base.consistent_views is None


def test_pipeline_launch_cuts_and_composition(tmp_path):
    from lichtfeld_densification_plugin_b200.output import remove_statistical_outliers
    cams, run = _pipeline(tmp_path)
    one = run(depth_consistency=True, refs_per_launch=0)
    ring = run(depth_consistency=True, refs_per_launch=4)              # several launches in flight on the ring
    assert ring.xyz.tobytes() == one.xyz.tobytes() and np.array_equal(ring.consistent_views, one.consistent_views)
    full = run(depth_consistency=True, refs_per_launch=4, outlier_neighbors=16, normal_neighbors=8, gaussian_neighbors=3,
               consistency_max_violations=1)
    loose = run(depth_consistency=True, refs_per_launch=4, consistency_max_violations=1)
    dev = torch.device("cuda")
    xyz = torch.from_numpy(loose.xyz).to(dev)
    keep = remove_statistical_outliers(xyz, xyz, nb_neighbors=16, std_ratio=2.0).kept_idx.cpu().numpy()
    assert full.xyz.tobytes() == loose.xyz[keep].tobytes()
    assert np.array_equal(full.consistent_views, loose.consistent_views[keep])
    assert full.normals.shape == full.xyz.shape and full.gaussians["scales"].shape == full.xyz.shape
    assert loose.xyz.shape[0] >= one.xyz.shape[0]


def test_invalid_inputs_and_streams():
    cams, maps, views, P, S, lenses = _setup(6, 64, 64, 64, 64)
    dev = views.device
    xyz = torch.from_numpy(_points(5000, seed=3)).to(dev)
    for bad in (dict(rel_tol=0.0), dict(rel_tol=1.0), dict(min_views=-1), dict(max_violations=-1)):
        with pytest.raises(ValueError):
            check_depth_consistency(xyz, views, **bad)
    nan = xyz.clone()
    nan[17, 1] = float("nan")
    with pytest.raises(ValueError, match="not finite"):
        check_depth_consistency(nan, views)
    for o in (6, -2):
        owner = torch.zeros((xyz.shape[0],), dtype=torch.int32)
        owner[3] = o
        with pytest.raises(ValueError, match="owner"):
            check_depth_consistency(xyz, views, owner=owner)
    with pytest.raises(ValueError):
        check_depth_consistency(xyz, views, owner=torch.zeros((4,), dtype=torch.int32))
    with pytest.raises(ValueError):
        views.add(np.zeros((32, 64), np.float32), cams[0])
    # the C entry point's own checks
    lib = N.load()
    need = C.c_size_t(0)
    n = int(xyz.shape[0])
    N.check(lib.ldp_consistency_workspace_bytes(n, C.byref(need)), "ldp_consistency_workspace_bytes")
    ws = torch.empty((need.value,), dtype=torch.uint8, device=dev)
    kept = torch.empty((n,), dtype=torch.int64, device=dev)
    status = torch.zeros((2,), dtype=torch.int32, device=dev)
    ptrs, Pt, St, _ = views.tables()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: C.c_void_p(t.data_ptr())                                                     # noqa: E731

    def call(tol=0.01, H=64, ws_bytes=need.value, mv=1):
        return lib.ldp_depth_consistency(p(xyz), n, None, p(ptrs), H, 64, p(Pt), p(St), None, len(views), tol, mv, 0, None, None,
                                         p(kept), p(status), p(ws), C.c_size_t(ws_bytes), st)
    assert call(tol=1.5) == -1 and call(H=0) == -1 and call(mv=-1) == -1
    assert call(ws_bytes=need.value - 1) == -3
    assert call() == 0
    ref = check_depth_consistency(xyz, views)
    ref_kept = ref.kept_idx.cpu().numpy()
    assert int(status[1]) == ref_kept.size and kept[:ref_kept.size].cpu().numpy().tolist() == ref_kept.tolist()
    # enqueued on the current stream: the side stream first rewrites the cloud, then the check reads it
    moved = xyz * 1.2
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        target = xyz.clone()
        torch.cuda._sleep(100_000_000)
        target.copy_(moved)
        got = check_depth_consistency(target, views)
    torch.cuda.synchronize()
    want = check_depth_consistency(moved, views)
    assert torch.equal(got.n_consistent, want.n_consistent) and torch.equal(got.kept_idx, want.kept_idx)
    assert not torch.equal(want.n_consistent, ref.n_consistent)
