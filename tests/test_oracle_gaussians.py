"""CPU: the 3DGS initialisation oracle (tests/gaussian_oracle.py) against 3DGS's own torch expressions, the rotation rule,
the host 3DGS PLY writer and the pipeline config."""
import numpy as np
import pytest
import torch

from lichtfeld_densification_plugin_b200.core import writers
from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig
from tests import gaussian_oracle as GO
from tests import outlier_oracle as OO


def _ulps(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """Distance in f32 ulps of finite values (across zero too)."""
    def ordered(x):
        i = np.asarray(x, np.float32).view(np.int32).astype(np.int64)
        return np.where(i < 0, -(2 ** 31) - i, i)
    return np.abs(ordered(a) - ordered(b))


def _construct_list_of_attributes(sh_degree: int) -> list:
    """graphdeco 3DGS GaussianModel.construct_list_of_attributes, restated on the shapes it reads (features_dc [n,1,3],
    features_rest [n,(d+1)^2-1,3], scaling [n,3], rotation [n,4])."""
    l = ["x", "y", "z", "nx", "ny", "nz"]
    for i in range(1 * 3):
        l.append("f_dc_{}".format(i))
    for i in range(((sh_degree + 1) ** 2 - 1) * 3):
        l.append("f_rest_{}".format(i))
    l.append("opacity")
    for i in range(3):
        l.append("scale_{}".format(i))
    for i in range(4):
        l.append("rot_{}".format(i))
    return l


@pytest.mark.parametrize("kind", ["sphere_floaters", "lattice", "duplicates"])
@pytest.mark.parametrize("k", [1, 3, 8])
def test_dist2_is_the_mean_of_the_nearest_other_points(kind, k):
    """The oracle's k_eff + 1 list with the point itself first equals an explicit j != i brute force."""
    x = OO.make_cloud(kind, 600, seed=k)
    xd = x.astype(np.float64)
    d2 = OO._d2(xd, xd)
    np.fill_diagonal(d2, np.inf)
    near = np.sort(d2, axis=1)[:, :k]
    m = np.zeros(x.shape[0])
    for j in range(k):
        m = m + near[:, j]
    ref = np.maximum((m / k).astype(np.float32), np.float32(1e-7))
    assert GO.dist2(x, k).tobytes() == ref.tobytes()


def test_dist2_small_clouds():
    x = np.array([[0, 0, 0], [3, 0, 0], [0, 4, 0], [0, 0, 0]], np.float32)
    assert GO.dist2(x[:1], 3).tolist() == [np.float32(1e-7)]
    assert GO.dist2(x[:2], 3).tolist() == [9.0, 9.0]
    assert GO.dist2(x[:3], 1).tolist() == [9.0, 9.0, 16.0]
    assert GO.dist2(x, 1)[[0, 3]].tolist() == [np.float32(1e-7)] * 2          # exact duplicates: 0, then the floor
    assert GO.dist2(x, 3)[0] == np.float32((0.0 + 9.0 + 16.0) / 3)


def test_formulas_match_3dgs_torch():
    """RGB2SH bit-exact; inverse_sigmoid and log(sqrt(clamp_min(dist2, 1e-7))) within 1 f32 ulp of torch on the CPU (the
    latter up to torch's own f32 rounding of the sqrt)."""
    rng = np.random.default_rng(3)
    rgb = np.concatenate([rng.random((200_000, 3)), np.linspace(0, 1, 3 * 4097).reshape(-1, 3)]).astype(np.float32)
    t = torch.from_numpy(rgb)
    assert ((t - 0.5) / GO.C0).numpy().tobytes() == GO.sh_dc(rgb).tobytes()
    # 3DGS's own value, 0.1 (far from 0 and 1 torch's f32 x / (1 - x) of the f32-rounded alpha loses more; the rule is f64)
    for a in (0.1, 0.5):
        ones = torch.ones((4, 1), dtype=torch.float32)
        x = a * ones
        inv = torch.log(x / (1 - x))                          # 3DGS utils/general_utils.inverse_sigmoid
        assert _ulps(inv.numpy().ravel(), np.full(4, GO.opacity_logit(a))).max() <= 1, a
    d2 = np.concatenate([10.0 ** rng.uniform(-12, 4, 100_000), [0.0, 1e-7, 1e-8]]).astype(np.float32)
    ref = torch.log(torch.sqrt(torch.clamp_min(torch.from_numpy(d2), 0.0000001))).numpy()
    ours = GO.scales(np.maximum(d2, GO.FLOOR), np.zeros(d2.size, bool), 1.0)[:, 0]
    # torch rounds sqrt to f32 before the log: an absolute error up to 2^-24 that dominates where the log is near 0
    # (dist2 near 1); elsewhere the two agree within 1 ulp
    ok = (_ulps(ref, ours) <= 1) | (np.abs(ref.astype(np.float64) - ours) <= 1.5 * 2.0 ** -24)
    assert ok.all() and (_ulps(ref, ours)[np.abs(ref) >= 1.0] <= 1).all()


def _unit(v):
    v = np.asarray(v, np.float64)
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def test_rotation_takes_e_z_to_the_normal():
    rng = np.random.default_rng(5)
    nrm = np.concatenate([_unit(rng.normal(size=(100_000, 3))),
                          [[0, 0, 1], [0, 0, -1], [1, 0, 0], [0, -1, 0], [1e-7, -2e-7, -1], [1e-5, 0, -1],
                           [-3e-4, 2e-4, -1], [0, 0, -5], [2, 2, 1]]]).astype(np.float32)
    q, ok = GO.rotations(nrm, nrm.shape[0])
    assert ok.all()
    assert np.all(np.abs(np.linalg.norm(q.astype(np.float64), axis=1) - 1) <= 1e-6)
    ez = GO.build_rotation(q)[:, :, 2]
    err = np.abs(ez - _unit(nrm.astype(np.float64))).max(axis=1)
    assert err.max() <= 1e-6, (err.max(), nrm[np.argmax(err)])
    assert q[-8].tolist() == q[-5].tolist() == q[-2].tolist() == [0.0, 1.0, 0.0, 0.0]          # half a turn about x


def test_undefined_normals():
    nrm = np.array([[0, 0, 0], [np.nan, 0, 1], [np.inf, 0, 0], [0, 0, 2]], np.float32)
    q, ok = GO.rotations(nrm, 4)
    assert ok.tolist() == [False, False, False, True]
    assert q[:3].tolist() == [[1, 0, 0, 0]] * 3
    q0, ok0 = GO.rotations(None, 3)
    assert not ok0.any() and q0.tolist() == [[1, 0, 0, 0]] * 3
    g = GO.init_gaussians(OO.make_cloud("cube", 4), np.full((4, 3), 0.5, np.float32), normals=nrm, flatten=0.25)
    assert g["undefined"] == 3
    assert np.all(g["scales"][:3, 2] == g["scales"][:3, 0]) and g["scales"][3, 2] < g["scales"][3, 0]
    with pytest.raises(ValueError):
        GO.init_gaussians(np.array([[0, 0, np.nan]], np.float32), np.zeros((1, 3), np.float32))


def test_flattened_covariance_has_the_normal_as_its_smallest_axis():
    rng = np.random.default_rng(9)
    x = OO.make_cloud("sphere_floaters", 2000, seed=9)
    nrm = _unit(rng.normal(size=(2000, 3))).astype(np.float32)
    nrm[:3] = [[0, 0, -1], [0, 0, 1], [1e-7, 0, -1]]
    g = GO.init_gaussians(x, rng.random((2000, 3)).astype(np.float32), normals=nrm, k=3, flatten=0.1)
    cov = GO.covariance(g["scales"], g["rotations"])
    lam, vec = np.linalg.eigh(cov)
    small = vec[:, :, 0]
    assert np.all(np.abs(np.abs(np.sum(small * _unit(nrm.astype(np.float64)), axis=1)) - 1) <= 1e-6)
    assert np.allclose(lam[:, 0] / lam[:, 1], 0.01, rtol=1e-5)
    assert np.allclose(lam[:, 1], lam[:, 2], rtol=1e-5)


@pytest.mark.parametrize("d,size", [(0, 68), (1, 104), (2, 164), (3, 248)])
@pytest.mark.parametrize("with_normals", [False, True])
def test_write_gaussian_ply_layout(tmp_path, d, size, with_normals):
    rng = np.random.default_rng(d)
    n = 37
    x = rng.normal(size=(n, 3)).astype(np.float32)
    nrm = _unit(rng.normal(size=(n, 3))).astype(np.float32) if with_normals else None
    g = GO.init_gaussians(x, rng.random((n, 3)).astype(np.float32), normals=nrm, flatten=0.5 if with_normals else 1.0)
    p = tmp_path / "g.ply"
    writers.write_gaussian_ply(str(p), x, g["sh_dc"], g["opacity"], g["scales"], g["rotations"], normals=nrm, sh_degree=d)
    raw = p.read_bytes()
    head, body = raw.split(b"end_header\n", 1)
    lines = head.decode("ascii").splitlines()
    assert lines[:3] == ["ply", "format binary_little_endian 1.0", f"element vertex {n}"]
    props = [ln.split() for ln in lines[3:]]
    assert all(p_[:2] == ["property", "float"] for p_ in props)
    names = [p_[2] for p_ in props]
    assert names == _construct_list_of_attributes(d) == writers.gaussian_ply_attributes(d)
    assert len(body) == n * size == n * 4 * len(names)
    v = np.frombuffer(body, dtype=np.dtype([(a, "<f4") for a in names]))
    col = lambda *a: np.stack([v[c] for c in a], axis=1)            # noqa: E731
    assert col("x", "y", "z").tobytes() == x.tobytes()
    assert col("nx", "ny", "nz").tobytes() == (nrm if with_normals else np.zeros((n, 3), np.float32)).tobytes()
    assert col("f_dc_0", "f_dc_1", "f_dc_2").tobytes() == g["sh_dc"].tobytes()
    rest = [a for a in names if a.startswith("f_rest_")]
    assert len(rest) == 3 * ((d + 1) ** 2 - 1) and all(np.all(v[a] == 0) for a in rest)
    assert v["opacity"].tobytes() == g["opacity"].tobytes()
    assert col("scale_0", "scale_1", "scale_2").tobytes() == g["scales"].tobytes()
    assert col("rot_0", "rot_1", "rot_2", "rot_3").tobytes() == g["rotations"].tobytes()


def test_gaussian_config_validation():
    DensePipelineConfig(output_path="d.ply", gaussian_neighbors=3).validate()
    DensePipelineConfig(output_path="d.ply", gaussian_neighbors=63, normal_neighbors=20, gaussian_flatten=0.1,
                        gaussian_opacity=0.5).validate()
    for bad in (dict(gaussian_neighbors=-1), dict(gaussian_neighbors=64), dict(gaussian_neighbors=3, gaussian_opacity=0.0),
                dict(gaussian_neighbors=3, gaussian_opacity=1.0), dict(gaussian_neighbors=3, gaussian_flatten=0.0),
                dict(gaussian_neighbors=3, gaussian_flatten=1.5), dict(gaussian_neighbors=3, gaussian_flatten=0.5)):
        with pytest.raises(ValueError):
            DensePipelineConfig(output_path="d.ply", **bad).validate()
    assert DensePipelineConfig(output_path="d.ply").gaussian_neighbors == 0
