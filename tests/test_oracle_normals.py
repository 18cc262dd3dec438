"""CPU: the oriented-normal oracle (tests/normals_oracle.py), the configuration switch and the PLY writer with normals."""
import numpy as np
import pytest

from lichtfeld_densification_plugin_b200.core import writers
from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig
from tests import normals_oracle as NO
from tests import outlier_oracle as OO

# The noisy unit sphere of test_sphere_normals_are_radial (20 000 points, radius noise 0.002, seed 3), per-point centres
# 3 x: angle between the normal and the radial direction, in degrees, as measured with this oracle (median, p99 =
# 3.153, 12.58 at k = 8 and 1.102, 3.157 at k = 20).  tests/test_gpu_normals.py holds the kernel to the same bounds.
SPHERE_N, SPHERE_SEED = 20_000, 3
SPHERE_BOUND_DEG = {8: (3.2, 12.7), 20: (1.15, 3.2)}


@pytest.mark.parametrize("kind", ["lattice", "duplicates", "plane", "cube"])
@pytest.mark.parametrize("k", [3, 8, 20, 64])
def test_brute_force_equals_kdtree_candidates(kind, k):
    x = OO.make_cloud(kind, 3000, seed=k)
    a = NO.knn_lex(x, k)
    b = NO.knn_lex_exact(x, k)
    assert np.array_equal(a, b)
    # the rule's order: ascending d^2, ties by ascending index, the point itself first unless it has a lower-index duplicate
    xd = x.astype(np.float64)
    d2 = np.sum((xd[a] - xd[:, None, :]) ** 2, axis=2)
    assert np.all(np.diff(d2, axis=1) >= 0)
    tie = np.diff(d2, axis=1) == 0
    assert np.all(np.diff(a, axis=1)[tie] > 0)
    assert np.all(d2[:, 0] == 0)


def test_ties_are_broken_by_index():
    # a point with six lattice neighbours at the same distance: k = 4 takes itself and the three lowest indices
    x = np.array([[0, 0, 0], [1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]], np.float32)
    perm = np.array([3, 6, 0, 5, 1, 4, 2])
    xp = x[perm]
    idx = NO.knn_lex(xp, 4)
    centre = int(np.nonzero(perm == 0)[0][0])
    assert idx[centre].tolist() == [centre] + sorted(set(range(7)) - {centre})[:3]


def test_plane_gives_z():
    x = OO.make_cloud("plane", 2000, seed=1)
    for k in (3, 8, 20):
        _, nrm, curv, und, _ = NO.estimate_normals(x, k, exact_knn=NO.knn_lex_exact)
        assert not und.any()
        assert np.array_equal(nrm, np.tile([0.0, 0.0, 1.0], (x.shape[0], 1)))        # canonical sign: +z
        assert np.all(curv == 0)
        # one centre below the plane turns every normal to -z
        _, nrm2, _, _, _ = NO.estimate_normals(x, k, centers=np.array([[0, 0, -5]], np.float32), exact_knn=NO.knn_lex_exact)
        assert np.array_equal(nrm2, -nrm)


@pytest.mark.parametrize("k", [8, 20])
def test_sphere_normals_are_radial(k):
    x = NO.noisy_sphere(SPHERE_N, seed=SPHERE_SEED)
    _, nrm, _, und, _ = NO.estimate_normals(x, k, centers=3 * x, center_idx=np.arange(SPHERE_N), exact_knn=NO.knn_lex_exact)
    assert not und.any()
    radial = x / np.linalg.norm(x, axis=1, keepdims=True)
    ang = np.degrees(NO.angle(nrm, radial))
    med, p99 = np.median(ang), np.percentile(ang, 99)
    print(f"sphere k={k}: median {med:.3f} deg, p99 {p99:.3f} deg")
    assert med <= SPHERE_BOUND_DEG[k][0] and p99 <= SPHERE_BOUND_DEG[k][1]
    assert np.all(np.sum(nrm * x, axis=1) > 0)                 # outward: every centre lies outside


def test_undefined_rule():
    t = np.random.default_rng(2).uniform(0, 10, size=500).astype(np.float32)
    _, nrm, curv, und, _ = NO.estimate_normals(np.stack([t, t, t], 1), 8)          # exactly collinear
    assert und.all() and np.all(nrm == 0) and np.isnan(curv).all()
    dup = np.zeros((10, 3), np.float32)
    _, nrm, curv, und, _ = NO.estimate_normals(dup, 8)
    assert und.all() and np.all(nrm == 0)
    _, _, _, und, _ = NO.estimate_normals(OO.make_cloud("cube", 2, seed=0), 8)      # k_eff = 2 < 3
    assert und.all()
    with pytest.raises(ValueError):
        NO.estimate_normals(dup, 2)


@pytest.mark.parametrize("value", [-1, 1, 2, 65])
def test_config_rejects(value):
    with pytest.raises(ValueError):
        DensePipelineConfig(output_path="x.ply", normal_neighbors=value).validate()


@pytest.mark.parametrize("value", [0, 3, 64])
def test_config_accepts(value):
    assert DensePipelineConfig(output_path="x.ply", normal_neighbors=value).validate().normal_neighbors == value


def test_write_ply_with_normals(tmp_path):
    rng = np.random.default_rng(0)
    n = 37
    xyz = rng.normal(size=(n, 3)).astype(np.float32)
    nrm = rng.normal(size=(n, 3)).astype(np.float32)
    rgb = rng.integers(0, 256, size=(n, 3)).astype(np.uint8)
    p = tmp_path / "n.ply"
    writers.write_ply(str(p), xyz, rgb, normals=nrm)
    data = p.read_bytes()
    header = (f"ply\nformat binary_little_endian 1.0\nelement vertex {n}\n"
              "property float x\nproperty float y\nproperty float z\n"
              "property float nx\nproperty float ny\nproperty float nz\n"
              "property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n").encode("ascii")
    assert data.startswith(header) and len(data) == len(header) + 27 * n
    rec = np.frombuffer(data[len(header):], dtype=np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("nx", "<f4"),
                                                            ("ny", "<f4"), ("nz", "<f4"), ("r", "u1"), ("g", "u1"), ("b", "u1")]))
    assert np.array_equal(np.stack([rec["x"], rec["y"], rec["z"]], 1), xyz)
    assert np.array_equal(np.stack([rec["nx"], rec["ny"], rec["nz"]], 1), nrm)
    assert np.array_equal(np.stack([rec["r"], rec["g"], rec["b"]], 1), rgb)
    # without normals: the reference's bytes, unchanged
    q = tmp_path / "p.ply"
    writers.write_ply(str(q), xyz, rgb)
    assert q.read_bytes() == writers.ply_header(n) + np.frombuffer(data[len(header):], np.uint8).reshape(n, 27)[
        :, np.r_[0:12, 24:27]].tobytes()
