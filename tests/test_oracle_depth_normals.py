"""CPU: the normal-map rule (tests/depth_normals_oracle.py) on analytic maps, the oriented fusion rule against the plain one,
config validation of the three options and that there is no CPU fallback."""
import numpy as np
import pytest
import torch

from lichtfeld_densification_plugin_b200 import _native as N
from lichtfeld_densification_plugin_b200 import synth
from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig
from tests import depth_normals_oracle as DN
from tests import fusion_oracle as FO
from tests import normals_oracle as NO
from tests.test_oracle_fusion import sphere_views


def plane_view(cam, H, W, planes, side=None, wm=64, hm=64):
    """Depth f32 [H, W] and xyz f32 [H, W, 3] of the world planes n . X = c (``planes``: list of (n, c)) seen by ``cam``;
    pixel (y, x) sees plane ``side[y, x]`` (default 0).  The map pixel's camera pixel is decoded as sphere_views does."""
    K, R = np.asarray(cam.K, np.float64), np.asarray(cam.R, np.float64)
    C = np.asarray(cam.C, np.float64).reshape(3)
    xs = (np.arange(W) + 0.5) / W * (wm - 1) * (cam.width / wm)
    ys = (np.arange(H) + 0.5) / H * (hm - 1) * (cam.height / hm)
    u, v = np.meshgrid(xs, ys)
    d_cam = np.stack([(u - K[0, 2]) / K[0, 0], (v - K[1, 2]) / K[1, 1], np.ones_like(u)], -1)
    d_world = d_cam @ R                                  # R^T d per pixel
    side = np.zeros((H, W), np.int64) if side is None else side
    z = np.empty((H, W))
    for s, (n, c) in enumerate(planes):
        n = np.asarray(n, np.float64)
        zs = (c - n @ C) / (d_world @ n)
        z = np.where(side == s, zs, z)
    X = C + z[..., None] * d_world
    return z.astype(np.float32), X.astype(np.float32)


def _unit(v):
    v = np.asarray(v, np.float64)
    return v / np.linalg.norm(v)


TILT = _unit([0.3, -0.2, 1.0])


@pytest.mark.parametrize("radius", [1, 2, 3])
def test_tilted_plane_gets_the_plane_normal_facing_the_camera(radius):
    cam = synth.make_orbit_cameras(1)[0]
    n = _unit(-np.asarray(cam.C, np.float64).reshape(3) + 0.6 * TILT)       # a plane through the origin, tilted to the camera
    depth, xyz = plane_view(cam, 40, 48, [(n, 0.0)])
    o = DN.depth_normals(depth, xyz, np.asarray(cam.C, np.float32), radius=radius, rel_tol=0.05)
    full = (2 * radius + 1) ** 2
    interior = np.zeros_like(o.undefined)
    interior[radius:-radius, radius:-radius] = True
    assert (o.k[interior] == full).all() and not o.undefined.any()
    facing = n if n @ (np.asarray(cam.C, np.float64).reshape(3)) > 0 else -n
    ang = NO.angle(o.normals.reshape(-1, 3), np.broadcast_to(facing, (40 * 48, 3)))
    print(f"r={radius}: largest angle to the plane normal {ang.max():.2e} rad")
    assert ang.max() < 1e-3                              # f32 coordinates of a plane a few units away
    assert np.all(o.curvature < 1e-5)


def test_two_planes_edge_pixels_use_their_own_plane():
    cam = synth.make_orbit_cameras(1)[0]
    C = np.asarray(cam.C, np.float64).reshape(3)
    back = -C / np.linalg.norm(C)
    na, nb = _unit(back + 0.4 * TILT), _unit(back - 0.5 * TILT)
    H, W = 32, 40
    side = (np.arange(W)[None, :] >= W // 2).astype(np.int64).repeat(H, 0)
    depth, xyz = plane_view(cam, H, W, [(na, 0.0), (nb, -1.5)], side)        # plane b 1.5 units further away
    o = DN.depth_normals(depth, xyz, np.asarray(cam.C, np.float32), radius=2, rel_tol=0.05)
    idx, valid = DN.window_neighbors(depth, 2, 0.05)
    s = side.reshape(-1)
    assert np.all(~valid | (s[idx] == s[:, None])), "a window crossed the depth edge"
    for label, n in ((0, na), (1, nb)):
        facing = n if n @ C > (n @ np.zeros(3)) else -n
        m = (side == label).reshape(-1)
        ang = NO.angle(o.normals.reshape(-1, 3)[m], np.broadcast_to(facing, (int(m.sum()), 3)))
        assert ang.max() < 1e-3, (label, ang.max())


def test_window_matches_a_loop_with_holes_and_borders():
    cams, depth, xyz, *_ = sphere_views(n_views=1, H=17, W=23, noise=3e-3, seed=3)
    d = depth[0].copy()
    rs = np.random.RandomState(4)
    d[rs.random_sample(d.shape) < 0.2] = np.nan
    for radius in (1, 2, 3):
        idx, valid = DN.window_neighbors(d, radius, 0.01)
        H, W = d.shape
        for p in range(H * W):
            y, x = divmod(p, W)
            want = []
            if np.isfinite(d[y, x]):
                for dy in range(-radius, radius + 1):
                    for dx in range(-radius, radius + 1):
                        qy, qx = y + dy, x + dx
                        if 0 <= qy < H and 0 <= qx < W and np.isfinite(d[qy, qx]) and \
                                abs(float(d[qy, qx]) - float(d[y, x])) <= 0.01 * float(d[y, x]):
                            want.append(qy * W + qx)
            assert idx[p][valid[p]].tolist() == want, (radius, p)
        o = DN.depth_normals(d, xyz[0], np.asarray(cams[0].C, np.float32), radius=radius, rel_tol=0.01)
        assert np.isnan(o.normals[~np.isfinite(d)]).all() and np.isnan(o.curvature[~np.isfinite(d)]).all()
        assert (o.k[0, 0] <= (radius + 1) ** 2) and np.all(o.undefined == (np.isfinite(d) & np.isnan(o.normals[..., 0])))


def test_one_pixel_wide_strip_is_undefined():
    H, W = 12, 9
    depth = np.full((H, W), np.nan, np.float32)
    xyz = np.full((H, W, 3), np.nan, np.float32)
    depth[:, 4] = 4.0 + 0.01 * np.arange(H)
    xyz[:, 4] = np.stack([np.full(H, 0.5), np.full(H, 0.25), depth[:, 4]], -1)      # a line along z, exactly
    o = DN.depth_normals(depth, xyz, np.zeros(3, np.float32), radius=2, rel_tol=0.05)
    assert o.undefined[:, 4].all() and np.isnan(o.normals).all()


def test_oriented_fusion_with_agreeing_normals_is_the_plain_fusion():
    """Every normal equal: the normal test passes wherever the depth test does, so the fused cloud is the plain one."""
    cams, depth, xyz, rgb, err, P, S = sphere_views(n_views=8, H=24, W=32, noise=2e-3, seed=5)
    nrm = np.zeros(xyz.shape, np.float32)
    nrm[..., 2] = 1.0
    nrm[~np.isfinite(depth)] = np.nan
    a = FO.fuse(depth, xyz, rgb, err, P, S, rel_tol=0.01, min_views=1)
    b = DN.fuse_oriented(depth, xyz, rgb, err, nrm, P, S, cos_max=0.9, rel_tol=0.01, min_views=1)
    assert np.array_equal(a.source, b.source) and a.source.size > 0
    for k in ("xyz", "rgb", "err", "n_views", "n_consistent"):
        assert getattr(a, k).tobytes() == getattr(b, k).tobytes(), k
    assert np.array_equal(b.normals, np.broadcast_to(np.float32([0, 0, 1]), b.normals.shape))
    # opposite normals in views 4..7: across the halves a view counts for nothing, so a pixel has fewer consistent views
    nrm[4:] = -nrm[4:]
    c = DN.fuse_oriented(depth, xyz, rgb, err, nrm, P, S, cos_max=0.9, rel_tol=0.01, min_views=1)
    print(f"emitted {a.source.size} plain, {c.source.size} with the halves opposed")
    assert c.source.size > 0 and (c.n_consistent_map <= a.n_consistent_map).all()
    assert (c.n_consistent_map < a.n_consistent_map).any() and not (c.kept & ~a.kept).any()


def test_config_validation():
    base = dict(output_path="x.ply")
    c = DensePipelineConfig(**base)
    assert c.depth_normal_radius == 0 and c.depth_fusion_max_normal_angle == 0.0 and c.depth_normal_rel_tol == 0.05
    DensePipelineConfig(**base, depth_dir="d", depth_normal_radius=2).validate()
    DensePipelineConfig(**base, depth_fusion=True, depth_normal_radius=3, depth_fusion_max_normal_angle=10.0).validate()
    DensePipelineConfig(**base, depth_fusion=True, depth_normal_radius=1, depth_fusion_max_normal_angle=10.0,
                        gaussian_neighbors=3, gaussian_flatten=0.2).validate()
    for bad in (dict(depth_dir="d", depth_normal_radius=4), dict(depth_dir="d", depth_normal_radius=-1),
                dict(depth_normal_radius=2),                                            # nothing consumes the maps
                dict(depth_dir="d", depth_normal_radius=2, depth_normal_rel_tol=0.0),
                dict(depth_dir="d", depth_normal_radius=2, depth_normal_rel_tol=1.0),
                dict(depth_fusion=True, depth_normal_radius=2, depth_fusion_max_normal_angle=90.0),
                dict(depth_fusion=True, depth_normal_radius=2, depth_fusion_max_normal_angle=-1.0),
                dict(depth_fusion=True, depth_fusion_max_normal_angle=10.0),            # no normal maps
                dict(depth_dir="d", depth_normal_radius=2, depth_fusion_max_normal_angle=10.0),   # no fusion
                dict(depth_fusion=True, depth_normal_radius=2, gaussian_neighbors=3, gaussian_flatten=0.2)):  # no normals
        with pytest.raises(ValueError):
            DensePipelineConfig(**base, **bad).validate()


def test_no_cpu_fallback(monkeypatch):
    from lichtfeld_densification_plugin_b200 import output

    class CpuViews:
        device = torch.device("cpu")
    with pytest.raises(N.NativeLibraryError):
        output.estimate_depth_normals(CpuViews())
    with pytest.raises(N.NativeLibraryError):
        output.fuse_depth_maps(CpuViews(), max_normal_angle=10.0)
    for bad in (dict(radius=0), dict(radius=4), dict(rel_tol=0.0), dict(rel_tol=1.0)):
        with pytest.raises(ValueError):
            output.estimate_depth_normals(CpuViews(), **bad)
    for bad in (0.0, 90.0, -5.0):
        with pytest.raises(ValueError):
            output.fuse_depth_maps(CpuViews(), max_normal_angle=bad)
