"""The multi-view refinement restated in numpy (tests/multiview_oracle.py): exactness of its solve, the accuracy it buys on the
synthetic scenes against their ground-truth points, and the configuration that switches it on.  CPU only."""
from __future__ import annotations

import numpy as np
import pytest

from lichtfeld_densification_plugin_b200 import synth
from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig
from lichtfeld_densification_plugin_b200.engine import PathConfig
from oracle import densify_oracle as O
from tests import multiview_oracle as MV


def _cfg(scene, M):
    return O.OracleConfig(matches_per_ref=M, no_filter=False, sampson_thresh=5.0, min_parallax_deg=0.5, reproj_thresh=0.8,
                          w_match=scene.w_match, h_match=scene.h_match)


def _gt_errors(scene, nn_refs, **kw):
    """Distance to the ground-truth point of the two-view and the refined point of every kept sample, and the mask sizes."""
    two, mv, nv = [], [], []
    for rp in nn_refs:
        inp = synth.synth_ref_inputs(scene, rp, cert_family="R", return_points=True, **kw)
        res, ref = MV.run(scene, inp, _cfg(scene, 4000))
        pts = inp["points"].numpy().reshape(-1, 3)
        k = ref.keep
        gt = pts[res.sel_idx[k]]
        two.append(np.linalg.norm(ref.two_xyz[k].astype(np.float64) - gt, axis=1))
        mv.append(np.linalg.norm(ref.xyz[k].astype(np.float64) - gt, axis=1))
        nv.append(np.array([bin(int(m)).count("1") + 1 for m in ref.mask[k]]))
    return np.concatenate(two), np.concatenate(mv), np.concatenate(nv)


def test_solve_is_exact_on_exact_projections():
    """The N-view DLT solve recovers a point from its exact float64 projections to 1e-9 relative."""
    scene = synth.make_scene(40, "turbo", nn=8)
    cams = scene.cameras
    rng = np.random.default_rng(1)
    for _ in range(50):
        views = rng.choice(len(cams), size=int(rng.integers(2, 9)), replace=False)
        X = rng.normal(size=3) * 0.8
        rows = []
        for v in views:
            P = cams[v].P.astype(np.float64)
            q = P @ np.append(X, 1.0)
            rows.append(MV.dlt_rows(P, q[:2] / q[2]))
        Y = MV.solve(np.concatenate(rows))
        assert np.linalg.norm(Y - X) <= 1e-9 * np.linalg.norm(X)


def test_refined_points_on_noise_free_scene():
    """Without noise or outliers the refined point is the ground-truth one up to the float32 warp coordinates, and a
    point joins every neighbour that sees it confidently."""
    scene = synth.make_scene(40, "turbo", nn=4)
    two, mv, nv = _gt_errors(scene, [0], noise_sigma=0.0, outlier_frac=0.0)
    assert mv.size > 1000
    assert np.median(mv) <= np.median(two)
    # f32 warp coordinates: one ulp of a normalised coordinate is ~6e-8, ~1e-5 px.  Measured (scene units, depths about 3.6):
    # largest distance 8.7e-6 (~2.4e-6 of the depth), median 2.7e-7 against 4.8e-7 for the two-view points
    assert np.max(mv) < 2e-5
    assert np.median(mv) < 5e-7
    assert (nv >= 3).mean() > 0.5


@pytest.mark.parametrize("nn,ratio", [(4, 0.8), (8, 0.7)])
def test_refinement_reduces_the_ground_truth_error(nn, ratio):
    """The default noisy scene (warp noise 1e-3, 10 % gross outliers): the median distance of the kept points to the
    ground truth shrinks to at most ``ratio`` of the two-view median (measured 0.72 at nn = 4, 0.63 at nn = 8)."""
    scene = synth.make_scene(40, "turbo", nn=nn)
    two, mv, nv = _gt_errors(scene, [0, 1, 2])
    r = np.median(mv) / np.median(two)
    print(f"nn={nn}: two-view median {np.median(two):.3e}, multi-view {np.median(mv):.3e}, ratio {r:.3f}, "
          f"cameras per point {np.bincount(nv)[2:].tolist()}")
    assert r <= ratio
    assert nv.min() >= 2 and nv.max() <= nn + 1


def test_config_validation():
    DensePipelineConfig(output_path="x", multiview=True).validate()
    with pytest.raises(ValueError):
        DensePipelineConfig(output_path="x", multiview=True, no_filter=True).validate()
    for bad in (0.0, -0.1, 1.5, float("nan")):
        with pytest.raises(ValueError):
            DensePipelineConfig(output_path="x", multiview=True, multiview_min_certainty=bad).validate()
    cfg = DensePipelineConfig(output_path="x", multiview=True, multiview_min_certainty=0.7)
    pc = PathConfig.from_pipeline_config(cfg)
    assert pc.multiview and pc.multiview_min_certainty == 0.7
    pc.check_multiview()
    assert not PathConfig.from_pipeline_config(DensePipelineConfig(output_path="x")).multiview
    with pytest.raises(ValueError):
        PathConfig(multiview=True, no_filter=True).check_multiview()
    with pytest.raises(ValueError):
        PathConfig(multiview=True, multiview_min_certainty=0.0).check_multiview()
