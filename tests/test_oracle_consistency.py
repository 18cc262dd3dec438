"""CPU: the cross-view depth consistency rule's numpy restatement (tests/consistency_oracle.py): the pixel convention of the
map scales, the verdicts on an analytic sphere, the pipeline's validation, and that nothing falls back to the CPU."""
import numpy as np
import pytest
import torch

from lichtfeld_densification_plugin_b200 import _native as N
from lichtfeld_densification_plugin_b200 import synth
from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig
from lichtfeld_densification_plugin_b200.engine import depth_map_scales
from tests import consistency_oracle as CO


@pytest.mark.parametrize("H,W,w_match,h_match", [(512, 512, 512, 512), (512, 512, 320, 320), (640, 640, 640, 640),
                                                 (1280, 1280, 800, 800), (40, 64, 320, 320), (40, 64, 64, 40)])
@pytest.mark.parametrize("size", [(1297, 840), (1920, 1080), (640, 480), (4032, 3024)])
def test_every_map_pixel_maps_back_to_itself(H, W, w_match, h_match, size):
    """The matcher's grid (linspace(-1 + 1/W, 1 - 1/W, W), f32 as torch makes it), decoded by the kernels' f32 chain
    ((g + 1) * 0.5 * (w_match - 1), then * f32(width / w_match)), lands on its own map pixel: floor(f64(u) * ax) = x."""
    width, height = size
    ax, ay = depth_map_scales(width, height, H, W, w_match, h_match)
    for n, m, s, a in ((W, w_match, width, ax), (H, h_match, height, ay)):
        g = torch.linspace(-1 + 1 / n, 1 - 1 / n, n).numpy()
        sc = np.float32(s / float(m))
        px = ((g + np.float32(1.0)) * np.float32(0.5)) * np.float32(m - 1)
        u = (px.astype(np.float32) * sc).astype(np.float32)
        back = np.floor(u.astype(np.float64) * a)
        assert np.array_equal(back, np.arange(n)), (n, m, s)
        frac = u.astype(np.float64) * a - np.arange(n)
        assert np.abs(frac - 0.5).max() < 1e-3                       # every decoded pixel sits at its pixel's centre


def _sphere_setup(n_views=8, H=512, W=512, wm=512, hm=512, radius=2.6):
    cams = synth.make_orbit_cameras(n_views)
    maps = np.stack([CO.sphere_map(c, H, W, wm, hm, radius) for c in cams])
    P = np.stack([np.asarray(c.P, np.float32).reshape(12) for c in cams])
    S = np.array([depth_map_scales(c.width, c.height, H, W, wm, hm) for c in cams])
    return cams, maps, P, S


def _facing(cams, X, cos_min=0.5):
    """[n, V]: the sphere's outward normal at X makes an angle with the direction to camera v of cosine > cos_min."""
    nrm = X / np.linalg.norm(X, axis=1, keepdims=True)
    out = np.zeros((X.shape[0], len(cams)), bool)
    for v, c in enumerate(cams):
        to_c = np.asarray(c.C, np.float64).reshape(1, 3) - X
        out[:, v] = (nrm * to_c).sum(1) / np.linalg.norm(to_c, axis=1) > cos_min
    return out


def _in_frame(cams, X, margin=0.05):
    out = np.zeros((X.shape[0], len(cams)), bool)
    for v, c in enumerate(cams):
        q0, q1, z = CO.project(np.asarray(c.P, np.float32), X.astype(np.float32))
        u, w = q0 / z, q1 / z
        out[:, v] = (z > 0) & (u > margin * c.width) & (u < (1 - margin) * c.width) & (w > margin * c.height) & \
                    (w < (1 - margin) * c.height)
    return out


def _sphere_points(n, radius, seed):
    d = np.random.RandomState(seed).normal(size=(n, 3))
    return radius * d / np.linalg.norm(d, axis=1, keepdims=True)


def test_sphere_verdicts():
    cams, maps, P, S = _sphere_setup()
    X = _sphere_points(20000, 2.6, 0)
    seen = _facing(cams, X) & _in_frame(cams, X)
    assert seen.sum() > 3000
    o = CO.check(X.astype(np.float32), maps, P, S, detail=True)
    assert (o.verdict[seen] == CO.CONSISTENT).all()                 # on the surface: every view that sees it agrees
    assert o.n_violations[seen.any(1)].max() == 0
    for v in (0, 3):                                                # moved along view v's ray: toward it, then away
        rows = np.nonzero(seen[:, v])[0]
        C = np.asarray(cams[v].C, np.float64).reshape(1, 3)
        front = (C + 0.9 * (X[rows] - C)).astype(np.float32)
        back = (C + 1.1 * (X[rows] - C)).astype(np.float32)
        of = CO.check(front, maps, P, S, detail=True)
        ob = CO.check(back, maps, P, S, detail=True)
        assert (of.verdict[:, v] == CO.VIOLATION).all()             # in front of the surface view v sees: it looks through
        assert (ob.verdict[:, v] == CO.OCCLUDED).all()              # behind it: hidden, no evidence either way
        assert (ob.n_violations == 0).all() or (ob.verdict == CO.VIOLATION).sum() < 0.01 * rows.size
    own = np.argmax(seen, axis=1)
    with_owner = CO.check(X.astype(np.float32), maps, P, S, owner=own, detail=True)
    assert (with_owner.verdict[np.arange(len(X)), own] == CO.NONE).all()
    assert (with_owner.n_consistent == o.n_consistent - (o.verdict[np.arange(len(X)), own] == CO.CONSISTENT)).all()


def test_no_evidence_cases():
    cams, maps, P, S = _sphere_setup(n_views=4, H=64, W=64, wm=64, hm=64)
    holes = maps.copy()
    holes[:, :, :] = np.nan
    X = _sphere_points(500, 2.6, 1).astype(np.float32)
    o = CO.check(X, holes, P, S)
    assert (o.n_consistent == 0).all() and (o.n_violations == 0).all() and o.kept_idx.size == 0
    far = np.array([[1e4, 0, 0], [0, 1e4, 0], [0, 0, -1e4]], np.float32)          # outside every map or behind cameras
    o = CO.check(far, maps, P, S, min_views=0)
    assert (o.n_consistent == 0).all() and (o.n_violations == 0).all() and o.kept_idx.tolist() == [0, 1, 2]


def test_synth_sphere_surface_is_shared():
    """surface="sphere": every reference view's points lie on the one sphere; the default surface is untouched."""
    scene = synth.make_scene(12, "turbo", ref_fraction=0.17, nn=2)
    a = synth.synth_ref_inputs(scene, 0, seed=3, return_points=True, surface="sphere")
    r = a["points"].reshape(-1, 3).norm(dim=1)
    ok = torch.isfinite(r)
    assert ok.float().mean() > 0.99 and (r[ok] - synth.SPHERE_RADIUS).abs().max() < 1e-9
    d1 = synth.synth_ref_inputs(scene, 0, seed=3, return_points=True)
    d2 = synth.synth_ref_inputs(scene, 0, seed=3, return_points=True, surface="field")
    for k in ("cert", "warp", "image", "points"):
        assert torch.equal(d1[k], d2[k]) or torch.allclose(d1[k], d2[k], equal_nan=True), k
    with pytest.raises(ValueError):
        synth.synth_ref_inputs(scene, 0, surface="cube")


def test_config_validation():
    base = dict(output_path="x.ply")
    DensePipelineConfig(depth_consistency=True, **base).validate()
    for bad in (dict(consistency_rel_tol=0.0), dict(consistency_rel_tol=1.0), dict(consistency_rel_tol=-0.1),
                dict(consistency_min_views=-1), dict(consistency_max_violations=-1)):
        with pytest.raises(ValueError):
            DensePipelineConfig(depth_consistency=True, **base, **bad).validate()
    c = DensePipelineConfig(**base)
    assert (c.depth_consistency, c.consistency_rel_tol, c.consistency_min_views, c.consistency_max_violations) == (False, 0.01, 1, 0)


def test_scales_reject_a_degenerate_matcher():
    with pytest.raises(ValueError):
        depth_map_scales(1297, 840, 512, 512, 1, 512)


def test_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from lichtfeld_densification_plugin_b200.engine import DepthViews
    from lichtfeld_densification_plugin_b200.output import check_depth_consistency
    with pytest.raises(N.NativeLibraryError):
        DepthViews(64, 64, 64, 64)

    class _Views:
        device = torch.device("cpu")
    with pytest.raises(N.NativeLibraryError):
        check_depth_consistency(torch.zeros((4, 3)), _Views())
