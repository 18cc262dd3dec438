"""GPU: colour maps (ldp_depth_colors) against the sampled path and their restatement, and depth-map fusion
(ldp_fuse_depth_maps, output.fuse_depth_maps) against its numpy restatement (tests/fusion_oracle.py), against the consistency
check, on the engine's own maps through the pipeline, and on bad input and side streams."""
import ctypes as C

import numpy as np
import pytest
import torch

from lichtfeld_densification_plugin_b200 import _native as N
from lichtfeld_densification_plugin_b200 import synth
from lichtfeld_densification_plugin_b200.engine import DepthViews, PathConfig
from lichtfeld_densification_plugin_b200.output import check_depth_consistency, fuse_depth_maps
from tests import consistency_oracle as CO
from tests import fusion_oracle as FO
from tests import gpu_harness as G
from tests.test_oracle_fusion import sphere_views

pytestmark = pytest.mark.gpu

OPENCV = ("OPENCV", [-0.12, 0.03, 4e-4, -3e-4])
FISHEYE = ("OPENCV_FISHEYE", [0.05, -0.01, 0.003, -0.0005])


@pytest.fixture(scope="module")
def engine():
    from lichtfeld_densification_plugin_b200.engine import DensifyEngine
    return DensifyEngine()


def _batch(engine, scene, inputs, W=None, H=None):
    dev = engine.device
    W, H = W or scene.W, H or scene.H
    b = engine.new_batch(H, W, scene.w_match, scene.h_match)
    to_dev = lambda m: None if m is None else torch.as_tensor(np.ascontiguousarray(m), dtype=torch.uint8).to(dev)  # noqa: E731
    for inp in inputs:
        nb = inp["nbr_indices"]
        cert = inp["cert"][:, :H, :W].contiguous().to(dev)
        warp = inp["warp"][:, :H, :W, :].contiguous().to(dev)
        b.add([cert[k] for k in range(len(nb))], [warp[k] for k in range(len(nb))], inp["image"].to(dev),
              scene.cameras[inp["ref_index"]], [scene.cameras[j] for j in nb], rng_stream=inp["ref_index"],
              mask_a=to_dev(inp.get("mask_a")),
              masks_b=[to_dev(m) for m in inp["masks_b"]] if inp.get("masks_b") is not None else None)
    return b


@pytest.mark.parametrize("case", ["pinhole", "lens", "raw_masks", "multiview", "narrow"])
def test_colour_maps_equal_the_sampled_rgb(engine, case):
    nn = 4
    lens = [[OPENCV, None, FISHEYE][v % 3] for v in range(24)] if case == "lens" else None
    scene = synth.make_scene(24, "fast", ref_fraction=0.125, nn=nn, lens=lens)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=21) for rp in range(scene.n_refs)]
    cfg = PathConfig(matches_per_ref=1000 if case == "narrow" else 6000, sampson_thresh=5.0, multiview=case == "multiview")
    min_cert = 0.2
    if case == "raw_masks":
        cfg.certainty_floor = 0.3
        min_cert = 0.3
        rs = np.random.RandomState(9)
        for inp in inputs:
            inp["mask_a"] = (rs.random_sample((64, 64)) > 0.1).astype(np.uint8)
            inp["masks_b"] = [(rs.random_sample((64, 64)) > 0.2).astype(np.uint8) if k % 2 else None for k in range(nn)]
    W, H = (40, 64) if case == "narrow" else (None, None)
    b = _batch(engine, scene, inputs, W, H)
    out = engine.prepare(b, cfg, taps=True).launch()
    dm = engine.depth_maps(b, cfg, min_cert, want_rgb=True)
    assert dm.flags is not None                           # allocated for the colours although not asked for
    torch.cuda.synchronize()
    off, S = out.ref_offset.cpu().numpy(), out.n_samples.cpu().numpy()
    flags, rgb = dm.flags.cpu().numpy(), dm.rgb.cpu().numpy()
    n_cmp = 0
    for r, inp in enumerate(inputs):
        sel = out.sel_idx[r, :S[r]].cpu().numpy().astype(np.int64)
        sf = out.sample_flags[r, :S[r]].cpu().numpy().astype(np.int64)
        order = G.expected_pack_order(sf)
        packed = out.rgb[off[r]:off[r + 1]].cpu().numpy()
        f = flags[r].reshape(-1)[sel].astype(np.int64)
        in_maps = ((f[order] >> 2) & 1) == 1              # kept by the sampled path and in the maps
        both, pos = order[in_maps], np.nonzero(in_maps)[0]
        assert both.size > 0.5 * order.size, (case, r)
        got = rgb[r].reshape(-1, 3)[sel[both]]
        assert got.tobytes() == packed[pos].tobytes(), (case, r)
        n_cmp += both.size
        # the whole map against the restated blend; NaN wherever the pixel is not kept
        Hm, Wm = flags.shape[1:]
        o = FO.color_maps(flags[r], inp["warp"][:, :Hm, :Wm, :].numpy(), inp["image"].numpy(), len(inp["nbr_indices"]),
                          scene.w_match, scene.h_match)
        assert o.tobytes() == rgb[r].tobytes(), (case, r)
    print(f"[colour] {case}: {n_cmp} sampled kept pixels bit-identical to the packed rgb")


def _device_views(depth, xyz, rgb, err, cams, wm, hm):
    V, H, W = depth.shape
    views = DepthViews(H, W, wm, hm)
    for v in range(V):
        views.add(depth[v], cams[v], xyz=xyz[v], rgb=rgb[v], err=err[v])
    return views


def _lens_tuples(cams):
    t = [CO.lens_tuple(c) for c in cams]
    return t if any(x is not None for x in t) else None


def _compare(views, depth, xyz, rgb, err, P, S, lenses, tag, **kw):
    f = fuse_depth_maps(views, **kw)
    o = FO.fuse(depth, xyz, rgb, err, P, S, lenses=lenses, **kw)
    got = {k: getattr(f, k).cpu().numpy() for k in ("source", "xyz", "rgb", "err", "n_views", "n_consistent")}
    if lenses is not None:
        near = np.argwhere(o.edge < 1e-9)
        print(f"[lens] {tag}: pixels within 1e-9 of a map pixel edge: {near[:10].tolist()}")
        if near.size:                                     # only those may differ: compare the rest
            flat = near[:, 0] * depth.shape[1] * depth.shape[2] + near[:, 1]
            assert np.isin(np.setxor1d(got["source"], o.source), flat).all(), tag
            return f, o
    assert np.array_equal(got["source"], o.source), tag
    for k in ("xyz", "rgb", "err", "n_views", "n_consistent"):
        assert got[k].tobytes() == getattr(o, k).tobytes(), (tag, k)
    return f, o


@pytest.mark.parametrize("rel_tol,min_views,max_violations", [(0.01, 1, 0), (0.002, 0, 0), (0.05, 2, 1), (0.01, 3, 5)])
def test_pinhole_vs_oracle(rel_tol, min_views, max_violations):
    cams, depth, xyz, rgb, err, P, S = sphere_views(n_views=24, H=40, W=56, noise=2e-3, seed=11)    # 15 degrees apart
    rs = np.random.RandomState(12)
    depth[rs.random_sample(depth.shape) < 0.05] = np.nan
    depth[5] = np.nan                                     # an all-NaN view
    xyz[~np.isfinite(depth)] = np.nan
    views = _device_views(depth, xyz, rgb, err, cams, 64, 64)
    f, o = _compare(views, depth, xyz, rgb, err, P, S, None, (rel_tol, min_views, max_violations), rel_tol=rel_tol,
                    min_views=min_views, max_violations=max_violations)
    src_view = o.source // (40 * 56)
    print(f"[pinhole] {(rel_tol, min_views, max_violations)}: kept {int(o.kept.sum())}, emitted {o.source.size}, "
          f"views per point max {o.n_views.max() if o.source.size else 0}")
    assert o.source.size > 0 and not (src_view == 5).any()
    if min_views <= 1:
        assert o.n_views.max() > 2


def test_many_views():
    """More views than one staging chunk (128 pinhole)."""
    cams, depth, xyz, rgb, err, P, S = sphere_views(n_views=150, H=20, W=28, noise=1e-3, seed=13)
    views = _device_views(depth, xyz, rgb, err, cams, 64, 64)
    f, o = _compare(views, depth, xyz, rgb, err, P, S, None, "V=150", min_views=2, max_violations=1)
    print(f"[many] V=150: emitted {o.source.size}, views per point max {o.n_views.max()}, last source view "
          f"{int(o.source[-1]) // (20 * 28)}")
    assert o.n_views.max() > 10


def test_lens_vs_oracle():
    cams, depth, xyz, rgb, err, P, S = sphere_views(n_views=12, H=40, W=56, noise=2e-3, seed=14)
    cams = synth.make_orbit_cameras(12, lens=[[OPENCV, None, FISHEYE][v % 3] for v in range(12)])
    views = _device_views(depth, xyz, rgb, err, cams, 64, 64)
    assert views.has_lens
    lenses = _lens_tuples(cams)
    P = np.stack([np.asarray(c.P, np.float32).reshape(12) for c in cams])
    for kw in (dict(), dict(rel_tol=0.03, min_views=2, max_violations=1)):
        _compare(views, depth, xyz, rgb, err, P, S, lenses, f"lens {sorted(kw)}", **kw)


def test_pass_one_equals_the_consistency_check():
    cams, depth, xyz, rgb, err, P, S = sphere_views(n_views=12, H=40, W=56, noise=3e-3, seed=15)
    views = _device_views(depth, xyz, rgb, err, cams, 64, 64)
    V, HW = depth.shape[0], depth.shape[1] * depth.shape[2]
    for kw in (dict(min_views=0, max_violations=1000), dict(min_views=1, max_violations=0), dict(rel_tol=0.003, min_views=2)):
        f = fuse_depth_maps(views, **kw)
        src, nc = f.source.cpu().numpy(), f.n_consistent.cpu().numpy()
        for r in range(V):
            pix = np.nonzero(np.isfinite(depth[r].reshape(-1)))[0]
            pts = torch.from_numpy(xyz[r].reshape(-1, 3)[pix]).cuda()
            c = check_depth_consistency(pts, views, owner=torch.full((pix.size,), r, dtype=torch.int32), **kw)
            kept = pix[c.kept_idx.cpu().numpy()]
            mine = src[src // HW == r] % HW
            assert np.isin(mine, kept).all(), (kw, r)               # emitted pixels are kept by the check
            at = np.searchsorted(pix, mine)
            assert np.array_equal(nc[src // HW == r], c.n_consistent.cpu().numpy()[at]), (kw, r)
            if r == 0:                                               # nothing lies below view 0: all its kept pixels emit
                assert np.array_equal(mine, kept), kw


def _pipeline(tmp_path, n_views=24):
    from lichtfeld_densification_plugin_b200.core import pipeline as P
    scene = synth.make_scene(n_views, "turbo", ref_fraction=0.5, nn=4)
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


def test_pipeline_launch_cuts_and_rng_paths(tmp_path):
    from lichtfeld_densification_plugin_b200.core import pipeline as P
    cams, run = _pipeline(tmp_path)
    seen = []
    orig = P._fuse_depth_maps

    def spy(depth_kept, tri_ctx):                          # the maps the pipeline fused, for the restatement below
        seen.append(list(depth_kept))
        return orig(depth_kept, tri_ctx)
    P._fuse_depth_maps = spy
    try:
        one = run(depth_fusion=True, refs_per_launch=0)
    finally:
        P._fuse_depth_maps = orig
    dk = seen[0]
    uids = [e[0] for e in dk]
    assert len(uids) == len(set(uids))
    sample = run(refs_per_launch=0)
    assert one.consistent_views is not None and one.fused_views is not None and sample.fused_views is None
    ring = run(depth_fusion=True, refs_per_launch=4)                    # several launches in flight
    mt = run(depth_fusion=True, refs_per_launch=0, rng_mode="numpy")    # the maps do not depend on the sampler's RNG
    both = run(depth_fusion=True, depth_consistency=True, refs_per_launch=4)
    for other in (ring, mt, both):
        assert other.xyz.tobytes() == one.xyz.tobytes() and other.rgb.tobytes() == one.rgb.tobytes()
        assert other.err.tobytes() == one.err.tobytes()
        assert np.array_equal(other.fused_views, one.fused_views) and np.array_equal(other.consistent_views, one.consistent_views)
    finite = torch.cat([e[3].reshape(-1, 3)[torch.isfinite(e[1].reshape(-1))] for e in dk]).double()
    rms = lambda x: float(torch.sqrt(((x.norm(dim=1) - synth.SPHERE_RADIUS) ** 2).mean()))          # noqa: E731
    r_fused, r_maps = rms(torch.from_numpy(one.xyz).double()), rms(finite)
    print(f"[pipeline] sampled {sample.xyz.shape[0]} points, kept map pixels {finite.shape[0]}, fused {one.xyz.shape[0]}; "
          f"rms radial error fused {r_fused:.3e}, maps {r_maps:.3e}; views per point max {one.fused_views.max()}")
    assert one.xyz.shape[0] > sample.xyz.shape[0] and r_fused < r_maps


def test_pipeline_matches_the_public_entry_point(tmp_path):
    from lichtfeld_densification_plugin_b200.core import pipeline as P
    cams, run = _pipeline(tmp_path)
    seen = []
    orig = P._fuse_depth_maps

    def spy(depth_kept, tri_ctx):
        seen.append((list(depth_kept), tri_ctx.w_match, tri_ctx.h_match))
        return orig(depth_kept, tri_ctx)
    P._fuse_depth_maps = spy
    try:
        res = run(depth_fusion=True, refs_per_launch=4, consistency_min_views=2, consistency_max_violations=1)
    finally:
        P._fuse_depth_maps = orig
    dk, wm, hm = seen[0]
    m0 = dk[0][1]
    views = DepthViews(int(m0.shape[0]), int(m0.shape[1]), wm, hm)
    for uid, depth, cam, xyz, rgb, err in dk:
        views.add(depth, cam, xyz=xyz, rgb=rgb, err=err)
    f = fuse_depth_maps(views, min_views=2, max_violations=1)
    assert res.xyz.tobytes() == f.xyz.cpu().numpy().tobytes() and res.rgb.tobytes() == f.rgb.cpu().numpy().tobytes()
    assert res.err.tobytes() == f.err.cpu().numpy().tobytes()
    assert np.array_equal(res.fused_views, f.n_views.cpu().numpy()) and np.array_equal(res.consistent_views, f.n_consistent.cpu().numpy())


def test_pipeline_composition(tmp_path):
    from lichtfeld_densification_plugin_b200.output import remove_statistical_outliers
    cams, run = _pipeline(tmp_path)
    loose = run(depth_fusion=True, refs_per_launch=4)
    full = run(depth_fusion=True, refs_per_launch=4, outlier_neighbors=16, normal_neighbors=8, gaussian_neighbors=3)
    xyz = torch.from_numpy(loose.xyz).cuda()
    keep = remove_statistical_outliers(xyz, xyz, nb_neighbors=16, std_ratio=2.0).kept_idx.cpu().numpy()
    assert full.xyz.tobytes() == loose.xyz[keep].tobytes()
    assert np.array_equal(full.fused_views, loose.fused_views[keep]) and np.array_equal(full.consistent_views, loose.consistent_views[keep])
    assert full.normals.shape == full.xyz.shape and full.gaussians["scales"].shape == full.xyz.shape
    # every normal faces the camera of its point's source view: the sphere's outward normal, seen from outside
    n = full.normals.astype(np.float64)
    defined = np.linalg.norm(n, axis=1) > 0.5
    radial = full.xyz.astype(np.float64) / np.linalg.norm(full.xyz.astype(np.float64), axis=1, keepdims=True)
    assert np.mean((n[defined] * radial[defined]).sum(1) > 0) > 0.95


def test_invalid_inputs_and_streams(engine):
    cams, depth, xyz, rgb, err, P, S = sphere_views(n_views=12, H=32, W=32, noise=1e-3, seed=16)
    views = _device_views(depth, xyz, rgb, err, cams, 64, 64)
    for bad in (dict(rel_tol=0.0), dict(rel_tol=1.0), dict(min_views=-1), dict(max_violations=-1)):
        with pytest.raises(ValueError):
            fuse_depth_maps(views, **bad)
    depth_only = DepthViews(32, 32, 64, 64)
    for v in range(12):
        depth_only.add(depth[v], cams[v])
    with pytest.raises(ValueError, match="depth only"):
        fuse_depth_maps(depth_only)
    with pytest.raises(ValueError):
        views.add(depth[0], cams[0], xyz=xyz[0][:, :16])
    nan_xyz = xyz.copy()
    nan_xyz[2, 5, 7] = np.nan
    with pytest.raises(ValueError, match="not finite"):
        fuse_depth_maps(_device_views(depth, nan_xyz, rgb, err, cams, 64, 64))
    # the C entry point's own checks
    lib = N.load()
    need = C.c_size_t(0)
    assert lib.ldp_fuse_workspace_bytes(40000, 256, 256, C.byref(need)) == -1       # n_views * H * W >= 2^31
    assert lib.ldp_fuse_workspace_bytes(32768, 256, 256, C.byref(need)) == -1       # exactly 2^31
    assert lib.ldp_fuse_workspace_bytes(12, 0, 32, C.byref(need)) == -1
    N.check(lib.ldp_fuse_workspace_bytes(12, 32, 32, C.byref(need)), "ldp_fuse_workspace_bytes")
    dev = views.device
    cap = 12 * 32 * 32
    ws = torch.empty((need.value,), dtype=torch.uint8, device=dev)
    outs = [torch.empty((cap, 3), device=dev), torch.empty((cap, 3), device=dev), torch.empty((cap,), device=dev),
            torch.empty((cap,), dtype=torch.int32, device=dev), torch.empty((cap,), dtype=torch.int32, device=dev),
            torch.empty((cap,), dtype=torch.int64, device=dev)]
    status = torch.zeros((2,), dtype=torch.int32, device=dev)
    ptrs, Pt, St, _ = views.tables()
    xp, rp, ep = views.fusion_tables()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: C.c_void_p(t.data_ptr())                                                     # noqa: E731

    def call(tol=0.01, H=32, V=12, ws_bytes=need.value, rgb_table=rp):
        return lib.ldp_fuse_depth_maps(p(ptrs), p(xp), p(rgb_table), p(ep), V, H, 32, p(Pt), p(St), None, tol, 1, 0,
                                       *[p(t) for t in outs], p(status), p(ws), C.c_size_t(ws_bytes), st)
    assert call(tol=1.5) == -1 and call(H=0) == -1 and call(V=300000, H=256) == -1
    assert call(ws_bytes=need.value - 1) == -3
    nulls = rp.clone()
    nulls[3] = 0
    assert call(rgb_table=nulls) == 0
    assert status.cpu().tolist() == [2, 0]                       # a NULL map pointer: nothing emitted
    assert call() == 0
    ref = fuse_depth_maps(views)
    m = int(status[1])
    assert m > 0 and m == ref.source.numel() and torch.equal(outs[5][:m], ref.source) and torch.equal(outs[0][:m], ref.xyz)
    # enqueued on the current stream: the side stream first rewrites the xyz maps, then fusion reads them
    moved = torch.from_numpy(xyz * np.float32(1.001)).cuda()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        target = [torch.from_numpy(xyz[v]).cuda() for v in range(12)]
        sv = DepthViews(32, 32, 64, 64)
        for v in range(12):
            sv.add(views.maps[v], cams[v], xyz=target[v], rgb=rgb[v], err=err[v])
        torch.cuda._sleep(100_000_000)
        for v in range(12):
            target[v].copy_(moved[v])
        got = fuse_depth_maps(sv)
    torch.cuda.synchronize()
    want = fuse_depth_maps(_device_views(depth, moved.cpu().numpy(), rgb, err, cams, 64, 64))
    assert torch.equal(got.source, want.source) and torch.equal(got.xyz, want.xyz)
    assert not torch.equal(want.xyz, ref.xyz)
