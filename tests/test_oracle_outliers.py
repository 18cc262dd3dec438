"""CPU: the statistical outlier oracle (tests/outlier_oracle.py) against scipy, on edge cases, and on the property users
want from it; the pipeline config fields."""
import numpy as np
import pytest

from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig
from tests import outlier_oracle as OO


@pytest.mark.parametrize("kind", ["cube", "sphere_floaters", "plane", "line"])
@pytest.mark.parametrize("k", [1, 5, 20, 64])
def test_oracle_agrees_with_kdtree(kind, k):
    xyz = OO.make_cloud(kind, 3000, seed=k)
    m = OO.mean_distances(xyz, k)
    ref = OO.mean_distances_kdtree(xyz, k)
    np.testing.assert_allclose(m, ref, rtol=1e-12, atol=0)


@pytest.mark.parametrize("kind", OO.CLOUDS)
@pytest.mark.parametrize("k", [2, 20])
def test_exact_tree_variant_equals_brute_force(kind, k):
    xyz = OO.make_cloud(kind, 2500, seed=3)
    assert OO.mean_distances_exact(xyz, k).tobytes() == OO.mean_distances(xyz, k).tobytes()


def test_distance_formula_and_self_inclusion():
    xyz = np.array([[0, 0, 0], [3, 4, 0], [0, 0, 12]], np.float32)
    m = OO.mean_distances(xyz, 2)
    assert m.tolist() == [2.5, 2.5, 6.0]                       # the point itself at 0, then its nearest
    assert OO.mean_distances(xyz, 3).tolist() == [(0 + 5 + 12) / 3, (0 + 5 + 13) / 3, (0 + 12 + 13) / 3]


def test_fixed_order_sum_is_the_documented_order():
    rng = np.random.default_rng(0)
    t = rng.random(300_007) * 1e3
    partials = []
    for a in range(0, t.size, OO.CHUNK):
        s = 0.0
        for v in t[a:a + OO.CHUNK]:
            s += float(v)
        partials.append(s)
    v = []
    for th in range(OO.FINAL):
        s = 0.0
        for j in range(th, len(partials), OO.FINAL):
            s += partials[j]
        v.append(s)
    s = OO.FINAL // 2
    while s >= 1:
        for th in range(s):
            v[th] = v[th] + v[th + s]
        s //= 2
    assert OO.fixed_order_sum(t) == v[0]
    assert abs(OO.fixed_order_sum(t) - t.sum()) < 1e-6 * t.sum()


def test_edge_cases():
    keep, m, st = OO.statistical_outliers(np.zeros((0, 3), np.float32), 20, 2.0)
    assert keep.size == 0 and m.size == 0
    keep, m, st = OO.statistical_outliers(np.array([[1, 2, 3]], np.float32), 20, 2.0)          # n = 1: std = NaN
    assert keep.size == 0 and m.tolist() == [0.0] and np.isnan(st[1])
    keep, m, st = OO.statistical_outliers(np.array([[0, 0, 0], [1, 0, 0]], np.float32), 20, 2.0)  # k >= n: k_eff = 2
    assert m.tolist() == [0.5, 0.5] and st[1] == 0.0 and keep.size == 0                           # m < mean + 0 fails
    xyz = OO.make_cloud("cube", 500, seed=1)
    keep, m, st = OO.statistical_outliers(xyz, 1, 2.0)                                            # k = 1 keeps nothing
    assert keep.size == 0 and (m == 0).all()
    keep, m, st = OO.statistical_outliers(np.tile(np.float32([[1, 2, 3]]), (100, 1)), 8, 2.0)   # all duplicates
    assert keep.size == 0 and (m == 0).all() and st[0] == 0.0


def test_duplicate_clusters_are_dropped_and_left_out_of_the_sums():
    rng = np.random.default_rng(5)
    base = rng.uniform(-1, 1, size=(400, 3)).astype(np.float32)
    dup = np.repeat(base[:3], 30, axis=0)                      # three clusters of 31 identical points
    xyz = np.concatenate([base, dup])
    keep, m, (mean, std, thr) = OO.statistical_outliers(xyz, 10, 2.0)
    zero = m == 0
    assert zero.sum() == 93 and not np.isin(np.nonzero(zero)[0], keep).any()
    assert mean == OO.fixed_order_sum(np.where(zero, 0.0, m)) / xyz.shape[0]      # V = n
    assert keep.tolist() == sorted(keep.tolist())


def test_rejections():
    xyz = OO.make_cloud("cube", 50)
    for k, r in ((0, 2.0), (65, 2.0), (8, 0.0), (8, -1.0)):
        with pytest.raises(ValueError):
            OO.statistical_outliers(xyz, k, r)
    bad = xyz.copy()
    bad[3, 1] = np.nan
    with pytest.raises(ValueError):
        OO.statistical_outliers(bad, 8, 2.0)


@pytest.mark.parametrize("n, removed", [(50_000, 0.78), (200_000, 0.84)])
def test_sphere_floaters_property(n, removed):
    """No surface point is lost and most floaters go (k = 20, std_ratio = 2).  With floaters uniform in [-1, 1]^3 this
    cloud loses 81 % of them at n = 50 000 and 86 % at 200 000: the ones that stay lie within a few mean spacings of the
    sphere, where no distance statistic can tell them from the surface."""
    xyz, is_f = OO.sphere_with_floaters(n, seed=0)
    m = OO.mean_distances_exact(xyz, 20)
    keep, _, _ = OO.statistical_outliers(xyz, 20, 2.0, means=m)
    kept = np.zeros(xyz.shape[0], bool)
    kept[keep] = True
    assert kept[~is_f].all()
    assert (~kept[is_f]).mean() >= removed


def test_config_fields():
    cfg = DensePipelineConfig(output_path="x.ply")
    assert cfg.outlier_neighbors == 0 and cfg.outlier_std_ratio == 2.0
    cfg.validate()
    DensePipelineConfig(output_path="x.ply", outlier_neighbors=64).validate()
    for kw in (dict(outlier_neighbors=-1), dict(outlier_neighbors=65), dict(outlier_neighbors=20, outlier_std_ratio=0.0),
               dict(outlier_std_ratio=-2.0)):
        with pytest.raises(ValueError):
            DensePipelineConfig(output_path="x.ply", **kw).validate()
