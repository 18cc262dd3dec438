"""GPU: normal maps (ldp_depth_normals, output.estimate_depth_normals) against their numpy restatement
(tests/depth_normals_oracle.py), judged as tests/test_gpu_normals.py judges point normals; the oriented fusion
(ldp_fuse_depth_maps_oriented) against its restatement for equality; the thin-structure case the normal test is for; the
pipeline; bad input and side streams."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from lichtfeld_densification_plugin_b200 import _native as N
from lichtfeld_densification_plugin_b200 import synth
from lichtfeld_densification_plugin_b200.engine import DepthViews, PathConfig
from lichtfeld_densification_plugin_b200.output import estimate_depth_normals, fuse_depth_maps, init_gaussians
from tests import depth_normals_oracle as DN
from tests import normals_oracle as NO
from tests.test_gpu_fusion import FISHEYE, OPENCV, _batch, _lens_tuples, _pipeline
from tests.test_gpu_normals import COND, GRAZING
from tests.test_oracle_depth_normals import plane_view
from tests.test_oracle_fusion import sphere_views

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from lichtfeld_densification_plugin_b200.engine import DensifyEngine
    return DensifyEngine()


def _views(depth, xyz, cams, wm=64, hm=64, rgb=None, err=None, normals=None):
    V, H, W = depth.shape[:3]
    views = DepthViews(H, W, wm, hm)
    for v in range(V):
        views.add(depth[v], cams[v], xyz=xyz[v], rgb=None if rgb is None else rgb[v], err=None if err is None else err[v],
                  normals=None if normals is None else normals[v])
    return views


def _judge(views, res, radius, rel_tol, tag):
    """Every view's map against the oracle: undefined sets equal outside the l1/l2 band [1e-13, 1e-11] (listed, not
    judged), angles within 2e-7 + COND * l2 / (l1 - l0), sign ties only where the camera is grazing, curvature within 1e-6
    relative, NaN where there is no depth.  Returns the largest angle * gap / l2."""
    got_n, got_c = res.normals.cpu().numpy(), res.curvature.cpu().numpy()
    worst, n_und = 0.0, 0
    for v in range(len(views)):
        depth, xyz = views.maps[v].cpu().numpy(), views.xyz[v].cpu().numpy()
        cen = np.asarray(views.cameras[v].C, np.float64).reshape(3).astype(np.float32)
        o = DN.depth_normals(depth, xyz, cen, radius=radius, rel_tol=rel_tol)
        has = np.isfinite(depth)
        gn, gc = got_n[v], got_c[v]
        assert np.isnan(gn[~has]).all() and np.isnan(gc[~has]).all(), tag
        gu = has & np.isnan(gn[..., 0])
        assert np.isnan(gn[gu]).all() and np.isnan(gc[gu]).all(), tag
        n_und += int(gu.sum())
        lam = o.eigenvalues
        with np.errstate(invalid="ignore", divide="ignore"):
            ratio = lam[..., 1] / lam[..., 2]
        listed = has & (ratio >= 1e-13) & (ratio <= 1e-11)
        if listed.any():
            print(f"{tag} view {v}: {int(listed.sum())} pixels with l1/l2 in [1e-13, 1e-11] not judged")
        assert np.array_equal(gu[~listed], o.undefined[~listed]), (tag, v, int(np.sum(gu[~listed] != o.undefined[~listed])))
        d = has & ~gu & ~o.undefined
        if not d.any():
            continue
        l = lam[d]
        with np.errstate(divide="ignore"):
            tol = 2e-7 + COND * l[:, 2] / (l[:, 1] - l[:, 0])
        rn = o.normals[d]
        ang = NO.angle(gn[d], rn)
        dc = cen.astype(np.float64) - xyz[d].astype(np.float64)
        dot = np.abs(np.sum(rn * dc, axis=1)) / np.linalg.norm(dc, axis=1)
        amb = dot <= np.maximum(GRAZING, 2 * tol)
        ang = np.where(amb, np.minimum(ang, np.pi - ang), ang)
        bad = ang > tol
        assert not bad.any(), (tag, v, int(bad.sum()), ang[bad][:5], tol[bad][:5])
        cerr = np.abs(gc[d].astype(np.float64) - o.curvature[d])
        assert np.all(cerr <= np.maximum(1e-6 * np.abs(o.curvature[d]), 1e-12)), (tag, v, cerr.max())
        worst = max(worst, float(np.max(ang * (l[:, 1] - l[:, 0]) / l[:, 2])))
    assert res.undefined == n_und, tag
    return worst


@pytest.mark.parametrize("case", ["pinhole", "lens", "narrow"])
def test_normal_maps_vs_oracle(engine, case):
    """The engine's own maps of the sphere scene, at radius 1, 2 and 3."""
    lens = [[OPENCV, None, FISHEYE][v % 3] for v in range(24)] if case == "lens" else None
    scene = synth.make_scene(24, "fast", ref_fraction=0.25, nn=4, lens=lens)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=31, surface="sphere") for rp in range(scene.n_refs)]
    W, H = (40, 64) if case == "narrow" else (None, None)
    b = _batch(engine, scene, inputs, W, H)
    dm = engine.depth_maps(b, PathConfig(matches_per_ref=6000, sampson_thresh=5.0), 0.2, want_xyz=True)
    cams = [scene.cameras[inp["ref_index"]] for inp in inputs]
    views = _views(dm.depth, dm.xyz, cams, scene.w_match, scene.h_match)
    assert views.has_lens == (case == "lens")
    for radius in (1, 2, 3):
        for rel_tol in (0.05, 0.01):
            res = estimate_depth_normals(views, radius=radius, rel_tol=rel_tol)
            worst = _judge(views, res, radius, rel_tol, f"{case} r={radius} tol={rel_tol}")
            print(f"[normal maps] {case} r={radius} rel_tol={rel_tol}: undefined {res.undefined}, "
                  f"largest angle * gap / l2 {worst:.2e}")


def _fuse_compare(views, depth, xyz, rgb, err, nrm, P, S, lenses, tag, angle, **kw):
    f = fuse_depth_maps(views, max_normal_angle=angle, **kw)
    o = DN.fuse_oriented(depth, xyz, rgb, err, nrm, P, S, cos_max=math.cos(math.radians(angle)), lenses=lenses, **kw)
    got = {k: getattr(f, k).cpu().numpy() for k in ("source", "xyz", "rgb", "err", "n_views", "n_consistent", "normals")}
    if lenses is not None:
        near = np.argwhere(o.edge < 1e-9)
        print(f"[lens] {tag}: pixels within 1e-9 of a map pixel edge: {near[:10].tolist()}")
        if near.size:                                     # only those may differ: compare the rest
            flat = near[:, 0] * depth.shape[1] * depth.shape[2] + near[:, 1]
            assert np.isin(np.setxor1d(got["source"], o.source), flat).all(), tag
            return f, o
    assert np.array_equal(got["source"], o.source), tag
    for k in ("xyz", "rgb", "err", "n_views", "n_consistent", "normals"):
        assert got[k].tobytes() == getattr(o, k).tobytes(), (tag, k)
    return f, o


def _sphere_with_normals(n_views, H, W, noise, seed, cams=None, radius=2, nan_view=None):
    c0, depth, xyz, rgb, err, P, S = sphere_views(n_views=n_views, H=H, W=W, noise=noise, seed=seed)
    cams = c0 if cams is None else cams
    if nan_view is not None:
        depth[nan_view] = np.nan
        xyz[nan_view] = np.nan
        rgb[nan_view] = np.nan
    nrm = estimate_depth_normals(_views(depth, xyz, cams), radius=radius).normals
    views = _views(depth, xyz, cams, rgb=rgb, err=err, normals=nrm)
    P = np.stack([np.asarray(c.P, np.float32).reshape(12) for c in cams])
    return cams, views, depth, xyz, rgb, err, nrm.cpu().numpy(), P, S


@pytest.mark.parametrize("angle,rel_tol,min_views,max_violations", [(10.0, 0.01, 1, 0), (30.0, 0.02, 2, 1), (3.0, 0.01, 0, 0),
                                                                    (60.0, 0.05, 1, 3)])
def test_oriented_fusion_vs_oracle(angle, rel_tol, min_views, max_violations):
    cams, views, depth, xyz, rgb, err, nrm, P, S = _sphere_with_normals(24, 40, 56, 2e-3, 11, nan_view=5)
    kw = dict(rel_tol=rel_tol, min_views=min_views, max_violations=max_violations)
    f, o = _fuse_compare(views, depth, xyz, rgb, err, nrm, P, S, None, f"angle {angle} {kw}", angle, **kw)
    plain = fuse_depth_maps(views, **kw)
    print(f"[oriented] {angle} deg {kw}: emitted {o.source.size} (without the normal test {plain.source.numel()}), "
          f"views per point max {o.n_views.max() if o.source.size else 0}")
    assert o.source.size > 0 and not (o.source // (40 * 56) == 5).any()
    assert np.allclose(np.linalg.norm(o.normals.astype(np.float64), axis=1), 1.0, atol=1e-6)


def test_oriented_fusion_many_views():
    """More views than one staging chunk (128 pinhole): the normal pointers are staged over two chunks."""
    cams, views, depth, xyz, rgb, err, nrm, P, S = _sphere_with_normals(150, 20, 28, 1e-3, 13, radius=1)
    f, o = _fuse_compare(views, depth, xyz, rgb, err, nrm, P, S, None, "V=150", 20.0, min_views=2, max_violations=1)
    print(f"[many] V=150: emitted {o.source.size}, views per point max {o.n_views.max()}")
    assert o.n_views.max() > 10 and (o.source // (20 * 28)).max() >= 128


def test_oriented_fusion_lens_vs_oracle():
    cams = synth.make_orbit_cameras(12, lens=[[OPENCV, None, FISHEYE][v % 3] for v in range(12)])
    cams, views, depth, xyz, rgb, err, nrm, P, S = _sphere_with_normals(12, 40, 56, 2e-3, 14, cams=cams)
    assert views.has_lens
    for kw in (dict(), dict(rel_tol=0.03, min_views=2, max_violations=1)):
        _fuse_compare(views, depth, xyz, rgb, err, nrm, P, S, _lens_tuples(cams), f"lens {sorted(kw)}", 15.0, **kw)


def test_no_angle_is_the_plain_fusion():
    """max_normal_angle=None: ldp_fuse_depth_maps itself, bit for bit, and no normals, although the views carry normal maps."""
    cams, views, depth, xyz, rgb, err, nrm, P, S = _sphere_with_normals(12, 32, 32, 1e-3, 16)
    f = fuse_depth_maps(views, min_views=1)
    assert f.normals is None
    lib, dev = N.load(), views.device
    need = C.c_size_t(0)
    N.check(lib.ldp_fuse_workspace_bytes(12, 32, 32, C.byref(need)), "ldp_fuse_workspace_bytes")
    cap = 12 * 32 * 32
    ws = torch.empty((need.value,), dtype=torch.uint8, device=dev)
    outs = [torch.empty((cap, 3), device=dev), torch.empty((cap, 3), device=dev), torch.empty((cap,), device=dev),
            torch.empty((cap,), dtype=torch.int32, device=dev), torch.empty((cap,), dtype=torch.int32, device=dev),
            torch.empty((cap,), dtype=torch.int64, device=dev)]
    status = torch.zeros((2,), dtype=torch.int32, device=dev)
    ptrs, Pt, St, _ = views.tables()
    xp, rp, ep = views.fusion_tables()
    p = lambda t: C.c_void_p(t.data_ptr())                                                     # noqa: E731
    N.check(lib.ldp_fuse_depth_maps(p(ptrs), p(xp), p(rp), p(ep), 12, 32, 32, p(Pt), p(St), None, 0.01, 1, 0, *[p(t) for t in outs],
                                    p(status), p(ws), C.c_size_t(need.value), C.c_void_p(torch.cuda.current_stream().cuda_stream)),
            "ldp_fuse_depth_maps")
    m = int(status[1])
    assert m == f.source.numel() > 0
    for t, g in zip(outs, (f.xyz, f.rgb, f.err, f.n_views, f.n_consistent, f.source)):
        assert t[:m].cpu().numpy().tobytes() == g.cpu().numpy().tobytes()


def test_thin_structure():
    """Two parallel sheets 2g apart (closer than rel_tol * depth), each seen from its own side.  Without the normal test
    the depth test lets pixels of opposite sheets become members and their average lies between the sheets; with it every
    fused point stays on its sheet and its normal faces its source camera."""
    g = 0.005
    allc = synth.make_orbit_cameras(16)
    cams = [c for c in allc if abs(float(np.asarray(c.C).reshape(3)[2])) > 2.0]      # no grazing view of the sheets
    H = W = 48
    depth, xyz = [], []
    for c in cams:
        side = 1.0 if float(np.asarray(c.C).reshape(3)[2]) > 0 else -1.0
        d, x = plane_view(c, H, W, [((0.0, 0.0, 1.0), side * g)])
        out = (np.abs(x[..., 0]) > 1.0) | (np.abs(x[..., 1]) > 1.0)
        d[out] = np.nan
        x[out] = np.nan
        depth.append(d)
        xyz.append(x)
    depth, xyz = np.stack(depth), np.stack(xyz)
    rs = np.random.RandomState(3)
    rgb = rs.uniform(0, 1, size=xyz.shape).astype(np.float32)
    err = rs.uniform(0, 1, size=depth.shape).astype(np.float32)
    nrm = estimate_depth_normals(_views(depth, xyz, cams), radius=2).normals
    views = _views(depth, xyz, cams, rgb=rgb, err=err, normals=nrm)
    plain = fuse_depth_maps(views, rel_tol=0.01, min_views=1)
    orient = fuse_depth_maps(views, rel_tol=0.01, min_views=1, max_normal_angle=10.0)
    zp, zo = plain.xyz[:, 2].cpu().numpy().astype(np.float64), orient.xyz[:, 2].cpu().numpy().astype(np.float64)
    between = np.abs(np.abs(zp) - g) > 1e-6
    print(f"[thin] {len(cams)} views, sheets {2 * g} apart: plain {zp.size} points, {int(between.sum())} between the sheets; "
          f"oriented {zo.size} points, largest distance from a sheet {np.max(np.abs(np.abs(zo) - g)):.2e}")
    assert between.any()                                          # members crossed without the normal test
    assert orient.source.numel() > 0 and np.all(np.abs(np.abs(zo) - g) <= 1e-6)
    src = (orient.source // (H * W)).cpu().numpy()
    cen = np.stack([np.asarray(cams[v].C, np.float64).reshape(3) for v in src])
    n = orient.normals.cpu().numpy().astype(np.float64)
    assert np.all(np.sum(n * (cen - orient.xyz.cpu().numpy()), axis=1) > 0)
    assert np.all(np.abs(n[:, 2]) > math.cos(math.radians(1.0)))


def test_pipeline_normal_files_and_launch_cuts(tmp_path):
    from lichtfeld_densification_plugin_b200.core import pipeline as P
    import json
    import os
    cams, run = _pipeline(tmp_path)
    seen = []
    orig = P._fuse_depth_maps

    def spy(depth_kept, tri_ctx, normals=None):
        seen.append((list(depth_kept), normals, tri_ctx.w_match, tri_ctx.h_match))
        return orig(depth_kept, tri_ctx, normals=normals) if normals is not None else orig(depth_kept, tri_ctx)
    opts = dict(depth_fusion=True, depth_normal_radius=2, depth_fusion_max_normal_angle=20.0)
    ddir = tmp_path / "maps"
    P._fuse_depth_maps = spy
    try:
        one = run(refs_per_launch=0, depth_dir=str(ddir), **opts)
    finally:
        P._fuse_depth_maps = orig
    dk, nk, wm, hm = seen[0]
    assert nk is not None and len(nk) == len(dk)
    m0 = dk[0][1]
    views = DepthViews(int(m0.shape[0]), int(m0.shape[1]), wm, hm)
    for uid, depth, cam, xyz, rgb, err in dk:
        views.add(depth, cam, xyz=xyz, rgb=rgb, err=err)
    ref = estimate_depth_normals(views, radius=2, rel_tol=0.05).normals.cpu().numpy()
    index = json.load(open(ddir / "depth_maps.json"))
    by_uid = {m["camera_uid"]: m for m in index["maps"]}
    for v, (uid, *_rest) in enumerate(dk):
        entry = by_uid[uid]
        assert entry["normals_file"] == "normals/" + entry["file"]
        on_disk = np.load(os.path.join(ddir, entry["normals_file"]))
        assert on_disk.dtype == np.float32 and on_disk.tobytes() == ref[v].tobytes()
        assert nk[v].cpu().numpy().tobytes() == ref[v].tobytes()
    assert one.normals is not None and one.normals.shape == one.xyz.shape
    ring = run(refs_per_launch=4, **opts)
    mt = run(refs_per_launch=0, rng_mode="numpy", **opts)
    for other in (ring, mt):
        assert other.xyz.tobytes() == one.xyz.tobytes() and other.rgb.tobytes() == one.rgb.tobytes()
        assert other.normals.tobytes() == one.normals.tobytes()
        assert np.array_equal(other.fused_views, one.fused_views)
    plain = run(refs_per_launch=4, depth_fusion=True, depth_dir=str(tmp_path / "plain"))
    assert "normals_file" not in json.load(open(tmp_path / "plain" / "depth_maps.json"))["maps"][0]
    assert not os.path.exists(tmp_path / "plain" / "normals") and plain.normals is None


def test_pipeline_sphere_normals_and_composition(tmp_path):
    cams, run = _pipeline(tmp_path)
    opts = dict(depth_fusion=True, depth_normal_radius=2, depth_fusion_max_normal_angle=20.0, refs_per_launch=4)
    loose = run(**opts)
    knn = run(normal_neighbors=8, **opts)                        # normal_neighbors keeps the k-NN normals
    assert knn.xyz.tobytes() == loose.xyz.tobytes() and knn.normals.tobytes() != loose.normals.tobytes()
    radial = loose.xyz.astype(np.float64) / np.linalg.norm(loose.xyz.astype(np.float64), axis=1, keepdims=True)
    n = loose.normals.astype(np.float64)
    out = np.mean((n * radial).sum(1) > 0)
    ang = lambda a: np.degrees(NO.angle(a, radial))                 # noqa: E731
    kn = knn.normals.astype(np.float64)
    kd = np.linalg.norm(kn, axis=1) > 0.5
    print(f"[sphere] {n.shape[0]} fused points, {out:.4f} outward; angle to the analytic normal: fused median "
          f"{np.median(ang(n)):.3f} deg, p95 {np.percentile(ang(n), 95):.3f}; k-NN (8) median {np.median(ang(kn[kd])):.3f} deg, "
          f"p95 {np.percentile(ang(kn[kd]), 95):.3f}")
    assert out > 0.95
    full = run(outlier_neighbors=16, gaussian_neighbors=3, gaussian_flatten=0.3, **opts)
    from lichtfeld_densification_plugin_b200.output import remove_statistical_outliers
    xyz = torch.from_numpy(loose.xyz).cuda()
    keep = remove_statistical_outliers(xyz, xyz, nb_neighbors=16, std_ratio=2.0).kept_idx.cpu().numpy()
    assert full.xyz.tobytes() == loose.xyz[keep].tobytes() and full.normals.tobytes() == loose.normals[keep].tobytes()
    g = init_gaussians(torch.from_numpy(full.xyz).cuda(), torch.from_numpy(full.rgb).cuda(),
                       normals=torch.from_numpy(full.normals).cuda(), nb_neighbors=3, flatten=0.3)
    assert g.undefined == 0
    for name in ("scales", "rotations"):
        assert full.gaussians[name].tobytes() == getattr(g, name).cpu().numpy().tobytes(), name


def test_invalid_inputs_and_streams():
    cams, depth, xyz, rgb, err, P, S = sphere_views(n_views=12, H=32, W=32, noise=1e-3, seed=16)
    views = _views(depth, xyz, cams, rgb=rgb, err=err)
    for bad in (dict(radius=0), dict(radius=4), dict(rel_tol=0.0), dict(rel_tol=1.0)):
        with pytest.raises(ValueError):
            estimate_depth_normals(views, **bad)
    depth_only = DepthViews(32, 32, 64, 64)
    for v in range(12):
        depth_only.add(depth[v], cams[v])
    with pytest.raises(ValueError, match="no xyz map"):
        estimate_depth_normals(depth_only)
    with pytest.raises(ValueError, match="no normal map"):
        fuse_depth_maps(views, max_normal_angle=10.0)
    with pytest.raises(ValueError):
        views.add(depth[0], cams[0], normals=xyz[0][:, :16])
    nan_xyz = xyz.copy()
    nan_xyz[2, 5, 7] = np.nan
    with pytest.raises(ValueError, match="not finite"):
        estimate_depth_normals(_views(depth, nan_xyz, cams))
    # the C entry point's own checks
    lib, dev = N.load(), views.device
    ptrs, _, _, _ = views.tables()
    xp = views.xyz_table()
    cen = torch.from_numpy(np.stack([np.asarray(c.C, np.float64).reshape(3) for c in cams]).astype(np.float32)).to(dev)
    nrm = torch.full((12, 32, 32, 3), -7.0, device=dev)
    curv = torch.full((12, 32, 32), -7.0, device=dev)
    status = torch.full((2,), -1, dtype=torch.int32, device=dev)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)                             # noqa: E731

    def call(V=12, H=32, radius=2, tol=0.05, depth_table=ptrs, xyz_table=xp, centers=cen):
        return lib.ldp_depth_normals(p(depth_table), p(xyz_table), V, H, 32, p(centers), radius, tol, p(nrm), p(curv), p(status), st)
    assert call(radius=0) == -1 and call(radius=4) == -1 and call(tol=0.0) == -1 and call(tol=1.0) == -1
    assert call(V=32768, H=65536) == -1 and call(H=0) == -1 and call(centers=None) == -1
    nulls = xp.clone()
    nulls[3] = 0
    assert call(xyz_table=nulls) == 0
    assert status.cpu().tolist() == [2, 0] and (nrm == -7.0).all() and (curv == -7.0).all()      # nothing else written
    bad_views = _views(depth, nan_xyz, cams)
    assert call(xyz_table=bad_views.xyz_table()) == 0
    assert status.cpu().tolist() == [1, 0] and (nrm == -7.0).all()
    assert call() == 0
    ref = estimate_depth_normals(views)
    assert status.cpu().tolist() == [0, ref.undefined] and torch.equal(nrm.nan_to_num(5.0), ref.normals.nan_to_num(5.0))
    # the oriented fusion's checks: a NULL normal map pointer, cos_max outside (0, 1)
    views = _views(depth, xyz, cams, rgb=rgb, err=err, normals=ref.normals)
    ptrs = views.tables()[0]
    need = C.c_size_t(0)
    N.check(lib.ldp_fuse_workspace_bytes(12, 32, 32, C.byref(need)), "ldp_fuse_workspace_bytes")
    cap = 12 * 32 * 32
    ws = torch.empty((need.value,), dtype=torch.uint8, device=dev)
    outs = [torch.empty((cap, 3), device=dev), torch.empty((cap, 3), device=dev), torch.empty((cap,), device=dev),
            torch.empty((cap, 3), device=dev), torch.empty((cap,), dtype=torch.int32, device=dev),
            torch.empty((cap,), dtype=torch.int32, device=dev), torch.empty((cap,), dtype=torch.int64, device=dev)]
    fstatus = torch.zeros((2,), dtype=torch.int32, device=dev)
    _, Pt, St, _ = views.tables()
    fxp, rp, ep = views.fusion_tables()

    angle = 25.0
    cos_max = math.cos(math.radians(angle))                      # what fuse_depth_maps passes for 25 degrees

    def fuse(cos_max=cos_max, table=views.normal_table()):
        return lib.ldp_fuse_depth_maps_oriented(p(ptrs), p(fxp), p(rp), p(ep), p(table), 12, 32, 32, p(Pt), p(St), None, 0.01, cos_max,
                                                1, 0, *[p(t) for t in outs], p(fstatus), p(ws), C.c_size_t(need.value), st)
    assert fuse(cos_max=0.0) == -1 and fuse(cos_max=1.0) == -1 and fuse(table=None) == -1
    nt = views.normal_table().clone()
    nt[4] = 0
    assert fuse(table=nt) == 0 and fstatus.cpu().tolist() == [2, 0]
    assert fuse() == 0
    want = fuse_depth_maps(views, max_normal_angle=angle)
    m = int(fstatus[1])
    assert m == want.source.numel() > 0 and torch.equal(outs[3][:m], want.normals) and torch.equal(outs[6][:m], want.source)
    # enqueued on the current stream: the side stream first rewrites the xyz maps, then the normal maps read them
    moved = np.ascontiguousarray(xyz[:, :, ::-1])                 # another surface: the columns mirrored
    moved_depth = np.ascontiguousarray(depth[:, :, ::-1])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        target = [torch.from_numpy(xyz[v]).cuda() for v in range(12)]
        tdepth = [torch.from_numpy(depth[v]).cuda() for v in range(12)]
        sv = DepthViews(32, 32, 64, 64)
        for v in range(12):
            sv.add(tdepth[v], cams[v], xyz=target[v])
        torch.cuda._sleep(100_000_000)
        for v in range(12):
            target[v].copy_(torch.from_numpy(moved[v]).cuda())
            tdepth[v].copy_(torch.from_numpy(moved_depth[v]).cuda())
        got = estimate_depth_normals(sv)
    torch.cuda.synchronize()
    want = estimate_depth_normals(_views(moved_depth, moved, cams))
    assert torch.equal(got.normals.nan_to_num(5.0), want.normals.nan_to_num(5.0))
    assert not torch.equal(want.normals.nan_to_num(5.0), ref.normals.nan_to_num(5.0))
