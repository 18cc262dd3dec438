"""CPU: the depth-map rule's numpy restatement (tests/depth_oracle.py) against the oracle's sampled path and against the
synthetic scenes' ground truth; validation of the pipeline's depth-map fields."""
import numpy as np
import pytest

from lichtfeld_densification_plugin_b200 import synth
from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig
from oracle import densify_oracle as O
from tests import depth_oracle as D
from tests.helpers import oracle_cam


def _scene(nn=2, seed=1, **kw):
    scene = synth.make_scene(12, "turbo", ref_fraction=0.17, nn=nn)
    inp = synth.synth_ref_inputs(scene, 0, cert_family="R", seed=seed, return_points=True, **kw)
    return scene, inp


def _oracle_args(scene, inp, no_filter=False, sampson=5.0):
    cams = scene.cameras
    nb = inp["nbr_indices"]
    cfg = O.OracleConfig(matches_per_ref=4000, no_filter=no_filter, sampson_thresh=sampson, min_parallax_deg=0.5,
                         w_match=scene.w_match, h_match=scene.h_match)
    return ([inp["cert"][k] for k in range(len(nb))], [inp["warp"][k] for k in range(len(nb))],
            oracle_cam(cams[inp["ref_index"]]), [oracle_cam(cams[j]) for j in nb], cfg)


@pytest.mark.parametrize("no_filter,sampson", [(False, 5.0), (False, 0.0), (True, 5.0)])
def test_maps_equal_the_sampled_path_at_its_samples(no_filter, sampson):
    """At every pixel triangulate_ref samples (and that is a candidate), the map's verdict, point and error are the sampled
    path's own: the same geometry on the same inputs."""
    scene, inp = _scene()
    certs, warps, ref, nbrs, cfg = _oracle_args(scene, inp, no_filter, sampson)
    m = D.depth_maps(certs, warps, ref, nbrs, cfg, min_certainty=0.2)
    res = O.triangulate_ref(certs, warps, inp["image"].numpy(), ref, nbrs, cfg, uniforms=np.random.RandomState(3).random_sample(20000),
                            keep_taps=True)
    assert m.cand[res.sel_idx].all()                    # the floor of the synthetic planes is 0.2: every pixel is a candidate
    n_exact = n = 0
    for gt in res.taps["groups"]:
        if "pos" not in gt:
            continue
        i = res.sel_idx[gt["pos"]]
        assert np.array_equal(m.keep[i], gt["keep"])
        assert m.good[i].all()
        X = gt["X"][:, :3].astype(np.float32)
        k = gt["keep"]
        np.testing.assert_allclose(m.xyz[i[k]], X[k], rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(m.err[i], gt["err"].astype(np.float32), rtol=1e-5, atol=1e-6)
        z = (gt["X"] @ ref.P.T)[:, 2].astype(np.float32)
        np.testing.assert_allclose(m.depth[i[k]], z[k], rtol=1e-6)
        n_exact += int((m.xyz[i[k]] == X[k]).all(axis=1).sum())
        n += int(k.sum())
    print(f"[sampled pixels] kept {n}, bit-identical points {n_exact}")
    assert n > 500


def test_kept_depths_follow_the_ground_truth():
    scene, inp = _scene(seed=5)
    certs, warps, ref, nbrs, cfg = _oracle_args(scene, inp)
    # at the synthetic planes' floor every pixel is a candidate, the injected outliers (certainty halved) too
    m = D.depth_maps(certs, warps, ref, nbrs, cfg, min_certainty=0.2)
    H, W = scene.H, scene.W
    Xw = inp["points"].reshape(-1, 3).numpy()
    cam = scene.cameras[inp["ref_index"]]
    z_true = (Xw @ cam.R.astype(np.float64).T + cam.t.astype(np.float64).reshape(1, 3))[:, 2]
    # outliers: the winner's match lies far from the true point's projection (the synthetic noise is 1e-3 grid units)
    wk = inp["warp"].numpy().reshape(len(inp["nbr_indices"]), H * W, 4)[m.winner, np.arange(H * W)]
    PB = np.stack([scene.cameras[j].P.astype(np.float64) for j in inp["nbr_indices"]])[m.winner]
    q = np.einsum("nij,nj->ni", PB, np.concatenate([Xw, np.ones((H * W, 1))], axis=1))
    camB = [scene.cameras[j] for j in inp["nbr_indices"]]
    sx = np.array([c.width / float(scene.w_match) for c in camB])[m.winner]
    sy = np.array([c.height / float(scene.h_match) for c in camB])[m.winner]
    xBn = q[:, 0] / q[:, 2] / sx / (0.5 * (scene.w_match - 1)) - 1.0
    yBn = q[:, 1] / q[:, 2] / sy / (0.5 * (scene.h_match - 1)) - 1.0
    outlier = np.hypot(wk[:, 2] - xBn, wk[:, 3] - yBn) > 0.02
    cand = m.cand
    rel = np.abs(m.depth[m.keep].astype(np.float64) - z_true[m.keep]) / z_true[m.keep]
    rejected = 1.0 - m.keep[cand & outlier].mean()
    kept_inliers = m.keep[cand & ~outlier].mean()
    print(f"[ground truth] candidates {int(cand.sum())} of {H * W}, kept {int(m.keep.sum())}: median relative depth error "
          f"{np.median(rel):.2e} (max {rel.max():.2e}); outliers among candidates {int((cand & outlier).sum())}, rejected "
          f"{rejected:.4f}; inliers kept {kept_inliers:.4f}")
    assert np.median(rel) < 2e-3
    assert (cand & outlier).sum() > 1000
    assert rejected > 0.97
    assert kept_inliers > 0.99


def test_threshold_selects_the_candidates():
    scene, inp = _scene()
    certs, warps, ref, nbrs, cfg = _oracle_args(scene, inp)
    lo = D.depth_maps(certs, warps, ref, nbrs, cfg, min_certainty=0.3)
    hi = D.depth_maps(certs, warps, ref, nbrs, cfg, min_certainty=0.7)
    assert (hi.cand <= lo.cand).all() and hi.cand.sum() < lo.cand.sum()
    # a pixel's verdict does not depend on the threshold that made it a candidate
    both = hi.cand
    assert np.array_equal(hi.keep[both], lo.keep[both])
    assert np.array_equal(hi.depth[both], lo.depth[both], equal_nan=True)
    assert np.isnan(hi.depth[~hi.cand]).all() and np.isnan(hi.err[~hi.cand]).all()


def test_config_fields_are_validated():
    DensePipelineConfig(output_path="x.ply", depth_dir="maps", depth_min_certainty=1.0).validate()
    assert DensePipelineConfig(output_path="x.ply").depth_dir == ""
    for bad in (0.0, -0.1, 1.5, float("nan")):
        with pytest.raises(ValueError):
            DensePipelineConfig(output_path="x.ply", depth_min_certainty=bad).validate()
    with pytest.raises(ValueError):
        DensePipelineConfig(output_path="x.ply", depth_dir=None).validate()


def test_write_depth_map_round_trip(tmp_path):
    from lichtfeld_densification_plugin_b200.output import write_depth_map
    a = np.full((3, 5), np.nan, np.float32)
    a[1, 2] = 3.25
    write_depth_map(str(tmp_path / "v.npy"), a.astype(np.float64))
    b = np.load(tmp_path / "v.npy")
    assert b.dtype == np.float32 and b.shape == (3, 5) and np.array_equal(a, b, equal_nan=True)
    with pytest.raises(ValueError):
        write_depth_map(str(tmp_path / "w.npy"), np.zeros((2, 2, 2)))
