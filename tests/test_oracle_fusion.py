"""CPU: the depth-map fusion rule's numpy restatement (tests/fusion_oracle.py) on analytic sphere maps, the pipeline's
validation, and that nothing falls back to the CPU."""
import numpy as np
import pytest
import torch

from lichtfeld_densification_plugin_b200 import _native as N
from lichtfeld_densification_plugin_b200 import synth
from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig
from lichtfeld_densification_plugin_b200.engine import depth_map_scales
from tests import consistency_oracle as CO
from tests import fusion_oracle as FO


def sphere_views(n_views=12, H=48, W=48, wm=64, hm=64, noise=0.0, seed=0):
    """Orbit cameras with the analytic sphere map each, the world point of every pixel (ray cast in f64, moved along its ray
    by a relative ``noise``), a colour map and an error map."""
    cams = synth.make_orbit_cameras(n_views)
    rs = np.random.RandomState(seed)
    depth, xyz = [], []
    for c in cams:
        d = CO.sphere_map(c, H, W, wm, hm, synth.SPHERE_RADIUS).astype(np.float64)
        d = d * (1.0 + noise * rs.standard_normal(d.shape))
        xs = (np.arange(W) + 0.5) / W * (wm - 1) * (c.width / wm)
        ys = (np.arange(H) + 0.5) / H * (hm - 1) * (c.height / hm)
        u, v = np.meshgrid(xs, ys)
        K = np.asarray(c.K, np.float64)
        cam_pts = np.stack([(u - K[0, 2]) / K[0, 0] * d, (v - K[1, 2]) / K[1, 1] * d, d], -1)
        world = (cam_pts - np.asarray(c.t, np.float64).reshape(3)) @ np.asarray(c.R, np.float64)
        depth.append(d.astype(np.float32))
        xyz.append(world.astype(np.float32))
    depth, xyz = np.stack(depth), np.stack(xyz)
    rgb = rs.uniform(0, 1, size=xyz.shape).astype(np.float32)
    err = rs.uniform(0, 2, size=depth.shape).astype(np.float32)
    rgb[~np.isfinite(depth)] = np.nan
    P = np.stack([np.asarray(c.P, np.float32).reshape(12) for c in cams])
    S = np.array([depth_map_scales(c.width, c.height, H, W, wm, hm) for c in cams])
    return cams, depth, xyz, rgb, err, P, S


def test_fused_points_lie_on_the_sphere():
    cams, depth, xyz, rgb, err, P, S = sphere_views(noise=2e-3, seed=1)
    o = FO.fuse(depth, xyz, rgb, err, P, S, rel_tol=0.01, min_views=1)
    assert o.source.size > 100 and (np.diff(o.source) > 0).all()
    r_fused = np.linalg.norm(o.xyz.astype(np.float64), axis=1)
    finite = np.isfinite(depth)
    r_maps = np.linalg.norm(xyz[finite].astype(np.float64), axis=1)
    rms = lambda r: float(np.sqrt(np.mean((r - synth.SPHERE_RADIUS) ** 2)))      # noqa: E731
    print(f"[sphere] emitted {o.source.size} of {int(o.kept.sum())} kept; rms radial error fused {rms(r_fused):.2e}, "
          f"maps {rms(r_maps):.2e}; mean views per point {o.n_views.mean():.2f}")
    assert np.abs(r_fused - synth.SPHERE_RADIUS).max() < 5 * 2e-3 * 8.0
    assert (o.n_views >= 1).all() and o.n_views.max() > 1
    assert rms(r_fused) < rms(r_maps)


def test_no_emitted_pixel_has_a_lower_member():
    cams, depth, xyz, rgb, err, P, S = sphere_views(noise=1e-3, seed=2)
    o = FO.fuse(depth, xyz, rgb, err, P, S, rel_tol=0.01, min_views=1)
    V, H, W = depth.shape
    for s in o.source[:: max(1, o.source.size // 300)]:
        r, i = divmod(int(s), H * W)
        X = xyz[r].reshape(-1, 3)[i:i + 1]
        c = CO.check(X, depth, P, S, owner=np.array([r]), detail=True)
        for v in range(r):
            if c.verdict[0, v] == CO.CONSISTENT:
                mx, my = FO.map_pixel(P[v], S[v], None, X)
                assert not o.kept[v, int(my[0]) * W + int(mx[0])], (s, v)


def test_two_identical_views():
    cams, depth, xyz, rgb, err, P, S = sphere_views(n_views=1, seed=3)
    d2, x2, c2, e2 = (np.concatenate([a, a]) for a in (depth, xyz, rgb, err))
    P2, S2 = np.concatenate([P, P]), np.concatenate([S, S])
    o = FO.fuse(d2, x2, c2, e2, P2, S2, min_views=1)
    N = depth.shape[1] * depth.shape[2]
    assert (o.source < N).all()                                  # view 1 contributes nothing of its own
    kept0 = np.nonzero(o.kept[0])[0]
    assert np.array_equal(o.source, kept0) and kept0.size > 0.5 * np.isfinite(depth).sum()
    assert o.xyz.tobytes() == xyz[0].reshape(-1, 3)[kept0].tobytes()      # (x + x) / 2 == x exactly
    assert o.rgb.tobytes() == rgb[0].reshape(-1, 3)[kept0].tobytes()
    assert (o.n_views == 2).all()


def test_one_view_min_views_zero():
    cams, depth, xyz, rgb, err, P, S = sphere_views(n_views=1, seed=4)
    o = FO.fuse(depth, xyz, rgb, err, P, S, min_views=0)
    finite = np.nonzero(np.isfinite(depth[0].reshape(-1)))[0]
    assert np.array_equal(o.source, finite)
    assert o.xyz.tobytes() == xyz[0].reshape(-1, 3)[finite].tobytes()
    assert o.rgb.tobytes() == rgb[0].reshape(-1, 3)[finite].tobytes()
    assert o.err.tobytes() == err[0].reshape(-1)[finite].tobytes()
    assert (o.n_views == 1).all() and (o.n_consistent == 0).all()


def test_config_validation():
    assert DensePipelineConfig(output_path="x.ply").depth_fusion is False
    DensePipelineConfig(output_path="x.ply", depth_fusion=True).validate()
    for bad in (dict(consistency_rel_tol=0.0), dict(consistency_rel_tol=1.0), dict(consistency_min_views=-1),
                dict(consistency_max_violations=-1)):
        with pytest.raises(ValueError):
            DensePipelineConfig(output_path="x.ply", depth_fusion=True, **bad).validate()


def test_no_cpu_fallback_fusion(monkeypatch):
    from lichtfeld_densification_plugin_b200 import output
    from lichtfeld_densification_plugin_b200.engine import DepthViews
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    with pytest.raises(N.NativeLibraryError):
        DepthViews(8, 8, 8, 8)

    class CpuViews:
        device = torch.device("cpu")
    with pytest.raises(N.NativeLibraryError):
        output.fuse_depth_maps(CpuViews())
